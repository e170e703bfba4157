"""A DEFLATE bit writer for tests (RFC 1951), pure Python: streams built token by token, including constructs that the
zlib family of encoders never emits (length code 284 with 31 extra bits, incomplete and empty codes, 15-bit codes, any
code-length sequence) and constructs that are invalid on purpose.  The writer computes the plaintext a stream means
from its tokens; it never asks a decoder.  Test infrastructure only.

Tokens of a compressed block:
    int 0..255           a literal
    (length, distance)   a match, coded with the usual symbol and extra bits
    Raw(...)             a literal/length symbol and, optionally, a distance symbol, each with chosen extra bits
    RawBits(v, n)        n bits written as they are (a bit pattern that is no code of the block)

`plain` is what the tokens mean.  Header-level damage the caller asks for (counts, code lengths, LEN / NLEN) does not
change it -- it is what a decoder that missed the damage would produce, and what the wrappers' checksums cover -- but a
token without a meaning (an invalid symbol, raw bits, a distance beyond the output) ends it: `plain` is then None.
"""
import struct
import zlib

# RFC 1951 3.2.5
LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [i // 2 for i in range(2, 28)]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32


def len_symbol(length):
    """(symbol, extra value, extra bit count) for a match length 3..258; 258 is symbol 285."""
    assert 3 <= length <= 258, length
    if length == 258:
        return 285, 0, 0
    c = max(i for i in range(28) if LEN_BASE[i] <= length)
    return 257 + c, length - LEN_BASE[c], LEN_EXTRA[c]


def dist_symbol(dist):
    assert 1 <= dist <= 32768, dist
    c = max(i for i in range(30) if DIST_BASE[i] <= dist)
    return c, dist - DIST_BASE[c], DIST_EXTRA[c]


def canonical(lens):
    """Bit-reversed canonical codes (RFC 1951 3.2.2) for a list of code lengths: codes[s] is ready for LSB-first output."""
    count = [0] * 16
    for n in lens:
        count[n] += 1
    count[0] = 0
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    codes = [0] * len(lens)
    for s, n in enumerate(lens):
        if n:
            c = nxt[n]
            nxt[n] += 1
            codes[s] = int(format(c, "0%db" % n)[::-1], 2)
    return codes


def flat_lengths(n):
    """Complete code lengths for n >= 2 symbols, all of length d - 1 or d."""
    d = max(1, (n - 1).bit_length())
    short = (1 << d) - n
    return [d - 1] * short + [d] * (n - short)


class Raw:
    """A literal/length symbol with `lextra` in `lbits` extra bits (default: the symbol's own count, 0 for 286/287), then,
    when dsym is given, a distance symbol with `dextra` in `dbits` bits (default: its own count, 0 for 30/31)."""
    __slots__ = ("lsym", "lextra", "lbits", "dsym", "dextra", "dbits")

    def __init__(self, lsym, lextra=0, dsym=None, dextra=0, lbits=None, dbits=None):
        self.lsym, self.lextra, self.dsym, self.dextra = lsym, lextra, dsym, dextra
        self.lbits = lbits if lbits is not None else (LEN_EXTRA[lsym - 257] if 257 <= lsym <= 285 else 0)
        self.dbits = dbits if dbits is not None else (DIST_EXTRA[dsym] if dsym is not None and dsym < 30 else 0)

    def meaning(self):
        """A literal, a (length, distance) pair, or None for a symbol that has no meaning."""
        if self.lsym < 256:
            return self.lsym
        if not 257 <= self.lsym <= 285 or self.dsym is None or self.dsym > 29:
            return None
        if self.lbits != LEN_EXTRA[self.lsym - 257] or self.dbits != DIST_EXTRA[self.dsym]:
            return None
        return LEN_BASE[self.lsym - 257] + self.lextra, DIST_BASE[self.dsym] + self.dextra


class RawBits:
    __slots__ = ("v", "n")

    def __init__(self, v, n):
        self.v, self.n = v, n


class Deflate:
    """Raw DEFLATE data and the plaintext its tokens mean."""

    def __init__(self):
        self.buf = bytearray()
        self.acc = 0                                            # bits not yet in buf, LSB first
        self.n = 0
        self.plain = bytearray()
        self.valid = True
        self.pos = 0                                            # output the tokens ask for, meaningful or not
        self.zero_history = False                               # True: bytes in front of the output read as zeros
        self.copies = []                                        # (position, length, distance) of every match

    # ---- bits ----
    def bits(self, v, n):
        self.acc |= (v & ((1 << n) - 1)) << self.n
        self.n += n
        while self.n >= 8:
            self.buf.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    @property
    def bitpos(self):
        return len(self.buf) * 8 + self.n

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)

    def data(self):
        """The stream so far, a partial last byte padded with zero bits."""
        return bytes(self.buf) + (bytes([self.acc & 0xFF]) if self.n else b"")

    def result(self):
        return self.data(), (bytes(self.plain) if self.valid else None)

    def mark(self):
        return len(self.buf), self.acc, self.n, len(self.plain), self.valid, self.pos, len(self.copies)

    def rewind(self, m):
        """Back to what mark() returned: everything written since is gone."""
        nb, self.acc, self.n, npl, self.valid, self.pos, nc = m
        del self.buf[nb:]
        del self.plain[npl:]
        del self.copies[nc:]

    # ---- plaintext ----
    def _copy(self, length, dist):
        self.copies.append((self.pos, length, dist))
        self.pos += length
        if not self.valid:
            return
        p = self.plain
        if dist > len(p):
            if not self.zero_history:
                self.valid = False
                return
            # a distance past the output, meant as what a decoder that took the missing history for zeros would produce
            missing = dist - len(p)
            p[:0] = bytes(missing)
            self._copy_in(p, length, dist)
            del p[:missing]
            return
        self._copy_in(p, length, dist)

    @staticmethod
    def _copy_in(p, length, dist):
        s = len(p) - dist
        if dist >= length:
            p += p[s:s + length]
        else:
            chunk = bytes(p[s:])
            p += (chunk * (length // dist + 1))[:length]

    # ---- blocks ----
    def header(self, final, btype):
        self.bits(1 if final else 0, 1)
        self.bits(btype, 2)

    def stored(self, data, final=False, len_=None, nlen=None):
        """A stored block; len_ / nlen override the LEN and NLEN fields."""
        self.header(final, 0)
        self.align()
        ln = len(data) if len_ is None else len_
        nl = (ln ^ 0xFFFF) if nlen is None else nlen
        self.bits(ln, 16)
        self.bits(nl, 16)
        self.buf += data
        self.pos += len(data)
        if self.valid:
            self.plain += data

    def sync(self):
        """The empty stored block of a flush point: 00 00 FF FF on a byte boundary."""
        self.stored(b"")

    def _symbols(self, tokens, lcodes, llens, dcodes, dlens, eob=True):
        bits = self.bits
        for t in tokens:
            if isinstance(t, int):
                assert llens[t], ("literal without a code", t)
                bits(lcodes[t], llens[t])
                self.pos += 1
                if self.valid:
                    self.plain.append(t)
            elif isinstance(t, tuple):
                length, dist = t
                s, e, n = len_symbol(length)
                assert llens[s], ("length symbol without a code", s)
                bits(lcodes[s], llens[s])
                bits(e, n)
                s, e, n = dist_symbol(dist)
                assert dlens[s], ("distance symbol without a code", s)
                bits(dcodes[s], dlens[s])
                bits(e, n)
                self._copy(length, dist)
            elif isinstance(t, RawBits):
                bits(t.v, t.n)
                self.valid = False
            else:
                bits(lcodes[t.lsym], llens[t.lsym])
                bits(t.lextra, t.lbits)
                if t.dsym is not None:
                    bits(dcodes[t.dsym], dlens[t.dsym])
                    bits(t.dextra, t.dbits)
                m = t.meaning()
                if m is None:
                    self.valid = False
                elif isinstance(m, int):
                    self.pos += 1
                    if self.valid:
                        self.plain.append(m)
                else:
                    self._copy(*m)
        if eob:
            bits(lcodes[256], llens[256])

    def fixed(self, tokens, final=False, eob=True):
        self.header(final, 1)
        self._symbols(tokens, _FIXED_LC, FIXED_LIT, _FIXED_DC, FIXED_DIST, eob)

    def dynamic(self, tokens, lit_lens, dist_lens, final=False, hlit=None, hdist=None, hclen=None, cl_lens=None,
                cl_seq=None, eob=True):
        """A dynamic block.  lit_lens / dist_lens: code lengths by symbol (lists or {symbol: length}).  Overrides: the
        HLIT / HDIST / HCLEN counts (as numbers of codes, 257.. / 1.. / 4..), the code-length code's lengths (by symbol
        0..18), and the raw code-length sequence cl_seq of (symbol, extra value) pairs.  Without cl_seq the lengths are
        run-length coded with 16 / 17 / 18 where that is shorter."""
        ll = as_list(lit_lens, 288)
        dl = as_list(dist_lens, 32)
        nl = hlit if hlit is not None else max(257, max((i + 1 for i, n in enumerate(ll) if n), default=0))
        nd = hdist if hdist is not None else max(1, max((i + 1 for i, n in enumerate(dl) if n), default=0))
        seq = cl_seq if cl_seq is not None else rle(ll[:nl] + dl[:nd])
        if cl_lens is None:
            used = sorted({s for s, _ in seq})
            if len(used) == 1:
                used.append(0 if used[0] else 1)
            cl_lens = [0] * 19
            for s, n in zip(used, flat_lengths(len(used))):
                cl_lens[s] = n
        cl_lens = list(cl_lens)
        nc = hclen if hclen is not None else max(4, max(i + 1 for i, s in enumerate(CL_ORDER) if cl_lens[s]))
        self.header(final, 2)
        self.bits(nl - 257, 5)
        self.bits(nd - 1, 5)
        self.bits(nc - 4, 4)
        for i in range(nc):
            self.bits(cl_lens[CL_ORDER[i]], 3)
        clc = canonical(cl_lens)
        for s, e in seq:
            assert cl_lens[s], ("code-length symbol without a code", s)
            self.bits(clc[s], cl_lens[s])
            if s >= 16:
                self.bits(e, (2, 3, 7)[s - 16])
        self._symbols(tokens, canonical(ll), ll, canonical(dl), dl, eob)


_FIXED_LC = canonical(FIXED_LIT)
_FIXED_DC = canonical(FIXED_DIST)


def as_list(lens, n):
    if isinstance(lens, dict):
        out = [0] * n
        for s, v in lens.items():
            out[s] = v
        return out
    return list(lens) + [0] * (n - len(lens))


def rle(lens):
    """Code lengths as a code-length sequence of (symbol, extra value): 16 repeats the previous length 3-6 times, 17 and
    18 give 3-10 and 11-138 zeros (RFC 1951 3.2.7)."""
    out, i = [], 0
    while i < len(lens):
        v, j = lens[i], i
        while j < len(lens) and lens[j] == v:
            j += 1
        run = j - i
        if v == 0:
            while run >= 11:
                k = min(run, 138)
                out.append((18, k - 11))
                run -= k
            if run >= 3:
                out.append((17, run - 3))
                run = 0
            out += [(0, 0)] * run
        else:
            out.append((v, 0))
            run -= 1
            while run >= 3:
                k = min(run, 6)
                out.append((16, k - 3))
                run -= k
            out += [(v, 0)] * run
        i = j
    return out


def fixed_bits(tokens):
    """Bits a list of tokens takes in a fixed-code block (without header and end-of-block code)."""
    n = 0
    for t in tokens:
        if isinstance(t, int):
            n += FIXED_LIT[t]
        else:
            s, _, e = len_symbol(t[0])
            d, _, de = dist_symbol(t[1])
            n += FIXED_LIT[s] + e + 5 + de
    return n


def phase_literals(now, target, mod=32):
    """Literals (8-bit 'a' and 9-bit 0xC0 codes of the fixed code) that move bit position `now` to `target` modulo `mod`
    (a multiple of 8 up to 32)."""
    want = (target - now) % mod
    nine = want % 8
    eight = ((want - 9 * nine) // 8) % (mod // 8)
    return [0xC0] * nine + [ord("a")] * eight


# ---- wrappers ----
def zlib_wrap(raw, plain, trailer=True):
    """78 9C, the raw data, Adler-32 of the plaintext (of nothing when it is None); trailer=False for a cut stream."""
    return b"\x78\x9c" + raw + (struct.pack(">I", zlib.adler32(plain or b"")) if trailer else b"")


def gzip_wrap(raw, plain, trailer=True):
    p = plain or b""
    h = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"
    return h + raw + (struct.pack("<II", zlib.crc32(p), len(p) & 0xFFFFFFFF) if trailer else b"")


def zip_archive(members):
    """A minimal ZIP32 archive: members are (name, raw deflate data, plaintext for CRC-32 and size).  Returns the archive
    bytes and the offset of every member's data."""
    out = bytearray()
    cd = bytearray()
    offs = []
    for name, raw, plain in members:
        nm = name.encode()
        crc, size = zlib.crc32(plain), len(plain)
        lo = len(out)
        out += struct.pack("<IHHHHHIIIHH", 0x04034B50, 20, 0, 8, 0, 0x21, crc, len(raw), size, len(nm), 0) + nm
        offs.append(len(out))
        out += raw
        cd += struct.pack("<IHHHHHHIIIHHHHHII", 0x02014B50, 20, 20, 0, 8, 0, 0x21, crc, len(raw), size, len(nm), 0, 0, 0, 0,
                          0, lo) + nm
    cd_off = len(out)
    out += cd
    out += struct.pack("<IHHHHIIH", 0x06054B50, 0, 0, len(members), len(members), len(cd), cd_off, 0)
    return bytes(out), offs
