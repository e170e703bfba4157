"""GPU: level-1 deflate output pinned byte for byte around the walk's match-start screen.

At level 1 (a chain budget of one, greedy parse) the walk first marks every position of a block where the search would
find a match and then searches only there.  That must not change a single token, so these cases pin the SHA-256 of
level-1 streams recorded on a B200 from the walk that searched at every token start, and check that each stream decodes
to its input with the system zlib.  They cover the screen's edges: matches that end 1-4 bytes before a block ends,
match starts in the last 1-5 bytes of a block (where the block end caps the length), inputs that end 1-5 bytes after a
block boundary, runs and period-d repeats whose matches cross sub-units and blocks, noise (no match start) and zeros
(one at nearly every position), windowBits 9 and 12 (heads beyond the window's reach must be screened out), job mode
with short jobs at odd offsets, and the strategies that keep the old walk at level 1 (Z_RLE, Z_HUFFMAN_ONLY) or take
the screened one (Z_FILTERED, Z_FIXED).
"""
import hashlib
import random
import zlib

import pytest

from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

BLOCK = 32768                                                # input bytes of one walk block
Z_FILTERED, Z_HUFFMAN_ONLY, Z_RLE, Z_FIXED = 1, 2, 3, 4


def noise(n, seed):
    return random.Random(seed).randbytes(n)


def block_edge_inputs():
    """Noise with copies of earlier bytes placed against the block ends."""
    buf = bytearray(noise(12 * BLOCK, 41))
    for k in (1, 2, 3, 4):                                   # a 16-byte match ends k bytes before block k's end
        end = (k + 1) * BLOCK - k
        buf[end - 16:end] = buf[end - 16 - 1000 * k:end - 1000 * k]
    for j in (1, 2, 3, 4, 5):                                # a match starts j bytes before block 5 + j's end
        at = (6 + j) * BLOCK - j
        buf[at:at + 12] = buf[at - 777:at - 765]
    yield "edges", bytes(buf)
    text = (b"the quick brown fox jumps over the lazy dog; " * 3000)
    for t in (1, 2, 3, 4, 5):                                # ends t bytes after a block boundary
        yield f"tail{t}", text[:2 * BLOCK + t]
    for n in (1, 2, 3, 4, 5, 7):
        yield f"short{n}", text[:n]


def repeat_inputs():
    """Runs and period-d repeats: matches run over sub-units (64 bytes) and blocks."""
    yield "zeros", bytes(300000)
    yield "noise", noise(300000, 42)
    for d in (1, 2, 3, 5, 31, 64, 65, 300, 4000, 32000):
        pat = noise(d, 43 + d)
        yield f"period{d}", (pat * (250000 // d + 1))[:250000 + d % 7]
    half = noise(BLOCK // 2 + 5, 44)
    yield "noise-copy", half + bytes(100) + half + half[:999]


def stream_cases(lib):
    """compress2 at level 1 (stream mode) on the constructed inputs and on corpus samples."""
    for gen in (block_edge_inputs, repeat_inputs):
        for name, data in gen():
            rc, z = lib.compress2(data, 1)
            assert rc == zb.Z_OK, (name, rc, lib.last_error())
            yield name, data, z
    for kind, seed in ((0, 51), (1, 52)):
        data = lib.synth((2 << 20) + 321, kind=kind, seed=seed).tobytes()
        rc, z = lib.compress2(data, 1)
        assert rc == zb.Z_OK, (kind, rc, lib.last_error())
        yield f"corpus{kind}", data, z


def option_cases(lib):
    """The streaming API at level 1 with small windows and with every strategy."""
    data = lib.synth(1 << 20, kind=1, seed=53).tobytes()
    per600 = (noise(600, 54) * 500)[:300000]                 # distance 600: beyond the reach of windowBits 9 (250)
    per5k = (noise(5000, 55) * 60)[:300000]                  # distance 5000: beyond the reach of windowBits 12 (3834)
    for wbits in (9, 12):
        for name, src in (("mixed", data), ("per600", per600), ("per5k", per5k)):
            rc, z = lib.deflate_stream(src, level=1, wbits=wbits, in_chunk=len(src), out_chunk=lib.compress_bound(len(src)) + 64)
            assert rc == zb.Z_OK, (wbits, name, rc, lib.last_error())
            yield f"w{wbits}-{name}", src, z
    for strategy, name in ((Z_FILTERED, "filtered"), (Z_HUFFMAN_ONLY, "huffman"), (Z_RLE, "rle"), (Z_FIXED, "fixed")):
        rc, z = lib.deflate_stream(data, level=1, in_chunk=len(data), out_chunk=lib.compress_bound(len(data)) + 64,
                                   strategy=strategy)
        assert rc == zb.Z_OK, (name, rc, lib.last_error())
        yield f"s-{name}", data, z


def batch_cases(lib):
    """zb200_deflate_batch at level 1: jobs of 1-300 bytes, each after an odd number of bytes, then larger ones."""
    sizes = list(range(1, 301, 13)) + [300, 2, 1, 40001, 131077]
    src = lib.synth(sum(sizes), kind=1, seed=56).tobytes()
    jobs, at = [], 0
    for size in sizes:
        jobs.append(src[at:at + size])
        at += size
    outs, st, _, _ = lib.deflate_batch(jobs, 1, zb.WRAP_ZLIB)
    assert st == [0] * len(jobs), st
    for i, (job, z) in enumerate(zip(jobs, outs)):
        yield f"job{i}", job, z


GROUPS = {"stream": stream_cases, "options": option_cases, "batch": batch_cases}


def digests(lib, group):
    """{case: sha256 of the stream} of one group, after checking that every stream decodes to its input."""
    out = {}
    for case, data, z in GROUPS[group](lib):
        assert zlib.decompress(z) == data, case
        out[case] = hashlib.sha256(z).hexdigest()
    return out


# recorded on one B200 (1000 W) from the walk that searched at every token start, before the screen
EXPECTED = {
    "batch": {
        "job0": "f2367b8e398dac8a7dfa1a032b8bdee241c568e9fde82617a64c43342b5a292d",
        "job1": "22ae46d7c5e1ba791d42ebe87c34d6cd28e8ed44feb440fc93cd8d31edc70677",
        "job10": "3a1f54dddce8cd151586a4fc27d3f888c63e757ed8bedeaba0e000db78172ff9",
        "job11": "b8f1820706a601f51f05c5411875b8609a7e4622dca4a09b3c518d31ec5a589e",
        "job12": "b52756474d86443913da49bed839629a0dd9c718f8d82f006458a5a748937f03",
        "job13": "2354e8de62d15b943e0b87faedc8fabe3d6db039715ad43825d9941f19164033",
        "job14": "91230a30ca2d5756cfd02b61d95c422458cc35220aa4e050534e680161cc042b",
        "job15": "da2a6fc8110ba20363a7bded71ce31a9a21ccbe1e5c4fdfa553863f9a3bed53a",
        "job16": "083d723f55dfbd4e8b7731c2aeb18b5a61251f06d954799bd42c4ed59495e7a5",
        "job17": "d94a1f0683251907b6d521715606fd3e219f3c0a87557a89ca5934b856daafab",
        "job18": "5d144234d2d2fbd33e5cd069791694bb46bb5f049255242aa31e82d70f8a6acd",
        "job19": "0b0bfc280fc70cec659d969d0609652eb404d7e1a81bcd1f83e6a25c11be88fd",
        "job2": "6005f7d1d8a2486bc15dec29417027d228842016d73de02ed109dd49622766c8",
        "job20": "91b4573cb0514f60aa59502d8b3344e6cca92876516551a4b7ffe5e905d70347",
        "job21": "9db9ba51c0655326cff050a1f9451b47c71f7ae888fbd25038da7c5beb95727a",
        "job22": "622e4c30bb1e0b7d2e71ea4e879de4b850f5ff00ac560feae7dce10ca001ab9a",
        "job23": "8d6671236be5a3de5299dfd15d4ffe03c3a05f3fbbebb8f6af1edf0f44376fcf",
        "job24": "464b747a548816eb06c1963adbef7556dd9ddb0f27f5c22e8c6a6d8036eb1879",
        "job25": "87b31ce9535cc0642d0cc97e0f5907a074205f7a69b29930cb7edf44321a5496",
        "job26": "abe9c813a5442cc4df3c0fa9ff206fa3f7565dc5b668e9c5d9fa5b19fd308b88",
        "job27": "45c837d03f3af14d763192557f52e44b84344946e32c5f555b328199d0ae7754",
        "job28": "020a5b441cdfb6b7587785007eb4bae54ed8369772c04588e6ea8c6f459c8689",
        "job3": "cababd41e8c727f5280f42249d0a2957be473ce49daa1a1433b811158929fcdf",
        "job4": "1320ec6856554cb74bce0b3e455c360186bc717f30bcf14ca9981f59be3f5678",
        "job5": "01d96f2d640f8a461c3b908eb498d492d570fa632956a85eba6fd25701563b6d",
        "job6": "e7a94a388c5a797be2ca6b991afd94a2b87785889f1a51d926f9b1ab3babd8bb",
        "job7": "a8a29329a7182428a3d50a6bf178facd1d383c38256117c491e756b0e621ca2d",
        "job8": "ca07936f050a09a41ddaf2da322bb3c5b72bed996e107b735da16f0b84209153",
        "job9": "f047777bda713ee7846b8c6d9888e8e37cc06fe3c4890fdd4e4f071a7d32b73d",
    },
    "options": {
        "s-filtered": "76e00a50cfe822f949bba3a2fad130070acfa18ad4a51553eeecacf4e5d7bc7f",
        "s-fixed": "59479701bff10137a31b66fab2ceb3253974b3390e71192ac81758ffecccef64",
        "s-huffman": "4d88e0d59def00cf67f9554512016467bdc784aa1c18f8629ed13d74acf9f120",
        "s-rle": "bcb3ca22dd9d723653215f716ef47dd6b0f95d2a5abf23586cb17760db2291fa",
        "w12-mixed": "7b0255c39851d766d2c2bb7506eae2875606842089a3d15cc92492a5bf793326",
        "w12-per5k": "29bff59918d94adbbf8312a96c476d68911dd3e3be423b7dd7211189154c380d",
        "w12-per600": "5ee920f170136bad1331c202b15fae3072636a9ccf760ac47a6d934bb032c961",
        "w9-mixed": "5c7ee37e6b5bd0f9cb95f31bc79e2a8e010a87e6e44c7c1b7c78ba0a9912d92f",
        "w9-per5k": "51fd0bcb2e7e65d5caf021a89c1fb5ee18215ff3fd68d7b68ac699beb9ab8bd2",
        "w9-per600": "4a4de9f986bc2fca6fbce8310292776d5a082b5fed9c0a5ef021219f48a62167",
    },
    "stream": {
        "corpus0": "8903d5b2c599fc5f08956f8bd9efe9fa154cd064e2655244c79e42f2aab62201",
        "corpus1": "493d594a782c6f3bcb590e5a2486f45f60a3d50a32148ec24246c7fa8f1d2025",
        "edges": "7eae6cae68b9b076a09f9a3221d1a1b130d09bc7eb89031f0b92ae05e87cdfef",
        "noise": "efd969334cef0dfcd33fe4143f16c7bfc747b7e975f11cc45a238ec381ce379e",
        "noise-copy": "d82069b8d34fa5c34e787fe3f34ba21df51d14c59f8fcf15cf1dc5035d2e6a79",
        "period1": "281bda298363490e4b17471b9c14da7b302d4ca9b91e061967aa63d9e8b32ed0",
        "period2": "c654629b7d5591cc53bf1a243fc41646fffce3e91a5ddf91f338c9b89c1cb037",
        "period3": "6878c7d90411112b2f1d4f4f383752ac2d83b6d51f404412c80ae1dea107a042",
        "period300": "1f0117fc188566b2793d773b492d4a88f93bd7f8318d30f973b7fe0adafc59e1",
        "period31": "0fe1f4c3f46dbe3cd9ecec4d08228506e254d4734594486cfd0993705c56722b",
        "period32000": "f90ee0dbaf725cb730002c2bc02599391ce9d6210e0f662d84855507c329cf1e",
        "period4000": "a74d5b880731db5c37ac39d161661601f67bb3810fe04eddf5c600fc79ba3599",
        "period5": "bc450c316759038484a1b0a9cb43b0d8d7c30b0f9fb49e41a4b63199fb790a6e",
        "period64": "894ec655c48d43cef433b74d9d3ef97b700f7aba642511eff0da6e03a8896586",
        "period65": "3cc99600bdd8c2f0d87114f50811d3a91d5352b98e5db43c76131cd1971ef970",
        "short1": "9eb89a1d22a98731240746e0a2142b1e42af61f31f7b41a2bbcaa925baf1c108",
        "short2": "cc0201989e45c46a5eac7689a2c89f1859e40627d705a9bde6e03ce67d957ff2",
        "short3": "547c30f53ea2c31278e17bf055e39a1c950ac0fb2c6081af09b8be8cdba645d6",
        "short4": "bab93790720db494077a557b8f2418ce3d4d861cb803622ed3a738eeee8c1734",
        "short5": "1d5b27b171189414b10f86f3037643163e626622a5b7324c5f5b13b85d5ace62",
        "short7": "f5a81800c9c40a26af436fce4f710b5fe452090ce52e9b2af46cf79434951934",
        "tail1": "768d9c473e70513368fd34ef3de72539f8a2ca9b8edfa278d65c62a05ae150ed",
        "tail2": "995417b4f5c82fece700430429f29f09fefbb06d220ca64b31cb2d61f088a2f4",
        "tail3": "626e5000f7b87d4eb2d6d69a873fc3e3098f300738771ce898633e85721d33d0",
        "tail4": "79f97028ccc6e3cf9698fd98df0c60c4a44d0cc2d582ee66b52139f5bfefe1b1",
        "tail5": "9d44467c2b3dfbd51e387094f49b12a7c8f7d1bf783c67cf727b01f2c7f3146a",
        "zeros": "4096fe4792ebe2884e7515a465480564215091e098bc9abecf2e23ac4a614d8d",
    },
}


@pytest.mark.parametrize("group", sorted(GROUPS))
def test_level1_streams_match_recorded_hashes(gpu_lib, group):
    got = digests(gpu_lib, group)
    want = EXPECTED[group]
    assert sorted(got) == sorted(want)
    assert [case for case in got if got[case] != want[case]] == []
