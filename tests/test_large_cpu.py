"""CPU: the plain-Python CRC-32 / Adler-32 algebra that the 64-bit GPU tests use as their reference, checked against
the system zlib; and the library's host crc32_combine / adler32_combine at lengths up to 2^40 against that algebra."""
import random
import zlib

import zhelpers


def _pieces(rng):
    out = [b"", b"\x00", bytes([0xFF]) * 5553]
    for _ in range(12):
        out.append(rng.randbytes(rng.choice((1, 3, 16, 511, 512, 513, 4096, 65537, rng.randrange(200000)))))
    return out


def test_cat_and_drop_prefix_match_zlib():
    rng = random.Random(5)
    ps = _pieces(rng)
    for _ in range(60):
        a, b = rng.choice(ps), rng.choice(ps)
        ca, cb, cab = zlib.crc32(a), zlib.crc32(b), zlib.crc32(a + b)
        aa, ab, aab = zlib.adler32(a), zlib.adler32(b), zlib.adler32(a + b)
        assert zhelpers.crc32_cat(ca, cb, len(b)) == cab
        assert zhelpers.crc32_drop_prefix(cab, ca, len(b)) == cb
        assert zhelpers.adler32_cat(aa, ab, len(b)) == aab
        assert zhelpers.adler32_drop_prefix(aab, aa, len(b)) == ab


def test_cat_over_long_zero_runs():
    """crc / adler of n zeros built by doubling agree with zlib run over the bytes (n past 2^24 and odd)."""
    for n in (1, 7, 4096 + 3, (1 << 24) + 5):
        z = bytes(n)
        c, a, m = 0, 1, 0
        cz, az = zlib.crc32(b"\0"), zlib.adler32(b"\0")     # k zeros, k doubling
        k, left = 1, n
        while left:
            if left & 1:
                c, a, m = zhelpers.crc32_cat(c, cz, k), zhelpers.adler32_cat(a, az, k), m + k
            cz, az, k = zhelpers.crc32_cat(cz, cz, k), zhelpers.adler32_cat(az, az, k), 2 * k
            left >>= 1
        assert m == n
        assert c == zlib.crc32(z) and a == zlib.adler32(z), n


def test_library_combine_to_2_40(lib):
    rng = random.Random(9)
    lens = [1, 511, 512, 65520, 65521, 65522, (1 << 32) - 1, 1 << 32, (1 << 32) + 1, (1 << 34) + 17,
            14_898_168_320, 1 << 40, (1 << 40) - 1] + [rng.randrange(1 << 40) for _ in range(40)]
    for n in lens:
        c1, c2 = rng.getrandbits(32), rng.getrandbits(32)
        a1 = (rng.randrange(65521) << 16) | rng.randrange(65521)
        a2 = (rng.randrange(65521) << 16) | rng.randrange(65521)
        assert lib.crc32_combine(c1, c2, n) == zhelpers.crc32_cat(c1, c2, n), n
        assert lib.adler32_combine(a1, a2, n) == zhelpers.adler32_cat(a1, a2, n), n
