"""GPU: deflate output pinned byte for byte.

The hash-chain links (k_lz_link) are a pure function of the input, the segment partition, the tile alignment and the
lane of each position within its 32-position step; in the relaxed mode of levels 1-6 the write that wins for positions
sharing a hash within a step is whichever the hardware keeps within one store instruction.  Any change to those makes
the walk see other candidates and changes the stream.  These cases cover both link modes (relaxed: levels 1 and 6;
exact: level 9 and Z_FIXED from level 4 on), stream mode at 4-byte aligned and misaligned starts, and job mode, and
compare each stream's SHA-256 with the value recorded on a B200 before the kernel was restructured.  Every stream must
also decode to its input.
"""
import ctypes as C
import hashlib
import zlib

import pytest

from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

Z_FIXED = 4
SAMPLE = 8 << 20                                              # bytes of each corpus sample
CORPORA = {"text": (0, 31), "mixed": (1, 32)}                # name: (synth kind, seed)
MISALIGNED = 3 * (1 << 20) + 12345                           # crosses segment and chunk edges, ragged end
BATCH_SIZES = [0, 1, 3, 4, 100, 4099, 32768, 40000, 131072, 131077, 300000, 1 << 20]


def corpus_streams(lib):
    """compress2 at levels 1, 6, 9 and the streaming API with Z_FIXED at levels 1 and 6 (host buffers)."""
    for name, (kind, seed) in CORPORA.items():
        data = lib.synth(SAMPLE, kind=kind, seed=seed).tobytes()
        for level in (1, 6, 9):
            rc, z = lib.compress2(data, level)
            assert rc == zb.Z_OK, (name, level, rc, lib.last_error())
            yield f"{name}-L{level}", data, z
        for level in (1, 6):
            rc, z = lib.deflate_stream(data, level=level, in_chunk=len(data), out_chunk=lib.compress_bound(len(data)) + 64,
                                       strategy=Z_FIXED)
            assert rc == zb.Z_OK, (name, level, rc, lib.last_error())
            yield f"{name}-L{level}-fixed", data, z


def misaligned_streams(lib):
    """zb200_deflate on device buffers that start 1, 2 and 3 bytes past a 4-byte boundary."""
    data = lib.synth(MISALIGNED, kind=1, seed=33).tobytes()
    n, cap = len(data), lib.compress_bound(len(data)) + 64
    d_src, d_dst = lib.dll.zb200_alloc_device(n + 8), lib.dll.zb200_alloc_device(cap)
    assert d_src and d_dst
    try:
        for off in (1, 2, 3):
            assert lib.dll.zb200_copy(C.c_void_p(d_src + off), data, n, None) == 0
            for level in (1, 9):
                m = lib.deflate(d_src + off, n, d_dst, cap, level, zb.WRAP_ZLIB)
                out = C.create_string_buffer(m)
                assert lib.dll.zb200_copy(out, C.c_void_p(d_dst), m, None) == 0
                yield f"offset{off}-L{level}", data, out.raw
    finally:
        lib.dll.zb200_free_device(d_src)
        lib.dll.zb200_free_device(d_dst)


def batch_streams(lib):
    """zb200_deflate_batch (job mode: one link segment per 128 KiB chunk of a job) at levels 1, 6, 9."""
    src = lib.synth(sum(BATCH_SIZES), kind=0, seed=34).tobytes()
    jobs, at = [], 0
    for size in BATCH_SIZES:
        jobs.append(src[at:at + size])
        at += size
    for level in (1, 6, 9):
        outs, st, _, _ = lib.deflate_batch(jobs, level, zb.WRAP_ZLIB)
        assert st == [0] * len(jobs), (level, st)
        for i, (job, z) in enumerate(zip(jobs, outs)):
            yield f"batch-L{level}-{i}", job, z


GROUPS = {"corpus": corpus_streams, "misaligned": misaligned_streams, "batch": batch_streams}


def digests(lib, group):
    """{case: sha256 of the stream} of one group, after checking that every stream decodes to its input."""
    out = {}
    for case, data, z in GROUPS[group](lib):
        assert zlib.decompress(z) == data, case
        out[case] = hashlib.sha256(z).hexdigest()
    return out


# recorded on one B200 (1000 W) from the link kernel of four steps per ring turn, before the turns were widened
EXPECTED = {
    "batch": {
        "batch-L1-0": "09d469dfeeaf4c436fd3f80ba7e168bcc34e5050993b5da3c8416fbae680f18f",
        "batch-L1-1": "f2367b8e398dac8a7dfa1a032b8bdee241c568e9fde82617a64c43342b5a292d",
        "batch-L1-10": "ec985d5eae4f1c66a78117c9ff9cc329cc43919273694b2218e3c0686f8b7c49",
        "batch-L1-11": "5641771ec27921fe053a9855ef5065fa14ad3c7af70f2238363b02f3ee980903",
        "batch-L1-2": "46eaad96d2bbce32b25e7cfd3b94c876a15bf4de73e537f5c299cbaa3116b9cc",
        "batch-L1-3": "7ec88c0235b58fb8ad1e8ef9915a7e8f2c06b77cc7e9735ecb5cf128c71d0889",
        "batch-L1-4": "936a6e11327e09aed4e9366f558d320155670fadc985da6d43ebff6204f335d5",
        "batch-L1-5": "b4b10c189999af2f00a217c2bd6b793a9bcc66af6ca5e3991ea9524e440147f4",
        "batch-L1-6": "53eafb06ba3ceec31b2eaa3504192bd05942468f80b22d4ca03efadb4102ed8a",
        "batch-L1-7": "eb4b6b1028ed0126ad56bf468cc97bbf328370bb723d2b041b2efa5df05a3b18",
        "batch-L1-8": "bacea2b36c3366005cc6e468d84f5d4e37990efec35f82d50fd57d2d66e0330c",
        "batch-L1-9": "d9e6fa52bf3cc840d91635a7712ddad5c92ddb752df3a21482264c71070875e7",
        "batch-L6-0": "aca503def43dc086a5aaa5c3d6f86bcbbc2aa6a80007ddea4a81bce2b376fceb",
        "batch-L6-1": "6c9488314027e12b58610510bb7b2a17873dbb12d7166e18c4e611b039db0921",
        "batch-L6-10": "df8437f5930f769da56fdcc4214322af6d392fa5b124ff5284ab84bd47ed6edd",
        "batch-L6-11": "06225d16a9c015b3b7f530e2717f457c2f24511b0fc6a7d094c2743c87ac87bb",
        "batch-L6-2": "ad4208035bb436077cd9c6ef8f275a8c6e9cf207bee6280c0ffaec20d8d78c38",
        "batch-L6-3": "c51515e149af91456963e5e158e941f3ebb9c52f6ea3d124c6bda59fbf1b538c",
        "batch-L6-4": "cc762312c77f922c0dc46db9bb058fa4d4027980fc0e21e29e573ca6ff3b81cb",
        "batch-L6-5": "451bdcea82b1af7530191f5bf0881b5630eec3bb16075135a8e14b90eead3b82",
        "batch-L6-6": "6e7f7246c44af55cb11a9a4aab0fcecb7fa5d45e21fa634e86675e9230ba9e10",
        "batch-L6-7": "f58b3d67aa78e7aaeed12f3a9742cafe337a2b69b644b845c0ae7f448d38ddab",
        "batch-L6-8": "2d0d803618025b97e2beae292878d5b7f008b8ea2cfa1299ce93fc3a9281f9e7",
        "batch-L6-9": "f8f2b30c636769a8fbaa96dc97b1be2682ba4a4418f114b91ff69f6430ea00b4",
        "batch-L9-0": "b171e283c6145acf2b923098dbbc40ffc39b4f1db0212928f9869747376c4ac8",
        "batch-L9-1": "144b5195a6e990b47447050b9573b99a03e8493c7a97a0a69db8cf1fd6ec8d4c",
        "batch-L9-10": "805d2d129fbca41ff7d411807adaa9cc7a74f7094d9a8db2aeaad5670cce04ea",
        "batch-L9-11": "6786980958cd14d508fbf0fa7888a0626eb2468f30bdc8b0b787ee5f168167e8",
        "batch-L9-2": "83575b7d99fc437e4b0230f61cd076bdf1bb23ee793ff9aadf121f54df5f2caa",
        "batch-L9-3": "4b80593e4c473f88698b048a2fbdf2c40fd91b6be2a23799abc0f217eddc6bbc",
        "batch-L9-4": "2322a770fbe88c79d5d7572997230edfd4f5e906f3812234e39067d197a33f49",
        "batch-L9-5": "5f0bf5a567b1bb457ef6969dae9bb81d4652ba5e866f84373a5e58b439de339a",
        "batch-L9-6": "ddc3fa1649abdba2438ba45fe5a451a164823cbf41442581224c900bb6148764",
        "batch-L9-7": "1e69c37e29e85ff24a21afc23688431ca360155625a5f130cd810c887ca5fadb",
        "batch-L9-8": "602f3238f403d05f3ae9a5aa1dd46c9b88d9756d44c38f8134caf938aa50dfdf",
        "batch-L9-9": "14dd7a3d58fa86069cb5995a72c0475559d0f0935209b616ce73aa1a94b7d51c",
    },
    "corpus": {
        "mixed-L1": "9ccb10f7496863bad101811cca29d7bf60d8f399b5a215ced50c5ad35cf464c3",
        "mixed-L1-fixed": "c5309e981b8790d8ddf14ada9f58529708cc72187b65ab2e5f78ebe209b279d6",
        "mixed-L6": "a2a10d990631a43f29490cc552fa9eb3cecf0c58ca3f4407b0e38c876a2c4e05",
        "mixed-L6-fixed": "b14c3d7a76b931cecae5c57a44fcfb7f1877abf92e9e8d12203ef376511ef38b",
        "mixed-L9": "593f747af0d86e13daff402ab8be1bcbd26ab5e62a8e95c62b414d47b2d7e662",
        "text-L1": "d996157976ca16102ed0da6dd3e0382587d9f6e7eb111fa5ac0d4c7452e14287",
        "text-L1-fixed": "bdcccf072cab87b31fabe4983171cef63969202b72ddf432620aa3e7405e3be6",
        "text-L6": "dc1d3ca23541dc6890f6a2e5dfaf56ed614b571ece779a90be07f15068cde744",
        "text-L6-fixed": "e32caebf5a28ad79379a8e6cb1f4573dc2ee3cf9c8797f8b03a06855e9b9594e",
        "text-L9": "0277e81c7ad70671d7deba954ea2f0cce58eca355945605a600f86ad57013004",
    },
    "misaligned": {
        "offset1-L1": "e222b1850e15d96e810227138fcca24021d583bf948de7e462495f4b01dcf8be",
        "offset1-L9": "2f3cd7d47148a68026348fe8e7a4ba74a4effa3d5bd52e894bcd6fd1222c84b4",
        "offset2-L1": "7ecb02c003b3bc9b52be0564fa8973e38aec4eae60a6ba174fcb252e70dc3f4c",
        "offset2-L9": "2f3cd7d47148a68026348fe8e7a4ba74a4effa3d5bd52e894bcd6fd1222c84b4",
        "offset3-L1": "97d72aaeb8796cf7e6f54578d464b2ff057ff3d06587751625e96cb1871a649c",
        "offset3-L9": "2f3cd7d47148a68026348fe8e7a4ba74a4effa3d5bd52e894bcd6fd1222c84b4",
    },
}


@pytest.mark.parametrize("group", sorted(GROUPS))
def test_streams_match_recorded_hashes(gpu_lib, group):
    got = digests(gpu_lib, group)
    want = EXPECTED[group]
    assert sorted(got) == sorted(want)
    assert [case for case in got if got[case] != want[case]] == []
