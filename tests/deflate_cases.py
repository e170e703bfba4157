"""Hand-built DEFLATE streams at the edges of RFC 1951, written by tests/deflate_writer.py: the catalogue of short cases
(valid constructs that zlib-family encoders never emit, the hand-over points of the decoders' lean loops, and invalid
constructs placed on purpose) and long streams whose segment starts, markers and window references are chosen, for the
segment-parallel decoder.  Shared by the CPU check of the catalogue and the GPU tests.  Test infrastructure only."""
import random
from collections import namedtuple

from deflate_writer import (DIST_BASE, DIST_EXTRA, LEN_BASE, LEN_EXTRA, Deflate, Raw, RawBits, as_list, dist_symbol,
                            fixed_bits, flat_lengths, len_symbol, phase_literals, rle)

# kind: "ok" (plain is what it decodes to), "bad" (refused with msg), "cut" (the data end early: refused, no message)
Case = namedtuple("Case", "name raw plain kind msg")

CHUNK = 128 << 10                                               # output between sync markers in this library's streams
MARKER = b"\x00\x00\xff\xff"                                     # an empty stored block on a byte boundary

FLAT_LIT = flat_lengths(286)                                    # every literal/length symbol, lengths 8 and 9
FLAT_DIST = flat_lengths(30)                                    # every distance code, lengths 4 and 5
# a complete code with lengths 1..14, 15, 15: the two 15-bit codes go to a literal and to length 258 / distance code 29
DEEP_LIT = dict(zip([97, 98, 99, 100, 101, 102, 103, 104, 105, 106, 257, 265, 256, 284, 122, 285], list(range(1, 15)) + [15, 15]))
DEEP_DIST = dict(zip([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 28, 29], list(range(1, 15)) + [15, 15]))


def _one(build):
    d = Deflate()
    build(d)
    return d.result()


def ok(name, build):
    raw, plain = _one(build)
    assert plain is not None, name
    return Case(name, raw, plain, "ok", None)


def bad(name, msg, build):
    raw, plain = _one(build)
    return Case(name, raw, plain, "bad", msg)


def cut(name, build, keep):
    """The stream `build` writes, ending after byte `keep` (a negative value counts from the end)."""
    raw, plain = _one(build)
    return Case(name, raw[:keep], None, "cut", None)


def m284(dist):
    """Length 258 written as symbol 284 with 31 extra bits."""
    c, e, _ = dist_symbol(dist)
    return Raw(284, 31, dsym=c, dextra=e)


def lens_for(tokens, extra_lit=(256,)):
    """Code lengths covering exactly the symbols the tokens use (one symbol: a single one-bit code)."""
    ls, ds = set(extra_lit), set()
    for t in tokens:
        if isinstance(t, int):
            ls.add(t)
        elif isinstance(t, tuple):
            ls.add(len_symbol(t[0])[0])
            ds.add(dist_symbol(t[1])[0])
        elif isinstance(t, Raw):
            ls.add(t.lsym)
            if t.dsym is not None:
                ds.add(t.dsym)

    def code(syms):
        syms = sorted(syms)
        return {} if not syms else {syms[0]: 1} if len(syms) == 1 else dict(zip(syms, flat_lengths(len(syms))))
    return code(ls), code(ds)


def seven_bit_cl(lit_lens, dist_lens):
    """Lengths of a code-length code that holds a 7-bit code: 1, 2, ..., 7, 7 over the symbols the lengths need."""
    ll, dl = as_list(lit_lens, 288), as_list(dist_lens, 32)
    nl = max(257, max((i + 1 for i, n in enumerate(ll) if n), default=0))
    nd = max(1, max((i + 1 for i, n in enumerate(dl) if n), default=0))
    used = sorted({s for s, _ in rle(ll[:nl] + dl[:nd])})
    assert len(used) <= 8
    used += [s for s in range(19) if s not in used][:8 - len(used)]
    cl = [0] * 19
    for s, n in zip(used, [1, 2, 3, 4, 5, 6, 7, 7]):
        cl[s] = n
    return cl


def rand_tokens(rng, lit_lens, dist_lens, budget, back, far=32768):
    """Random tokens over the symbols that have codes: literals, and matches with random extra bits whose distances stay
    within `back` bytes of history (grown by what the tokens produce) and `far`.  Stops before `budget` bytes of output."""
    ll, dl = as_list(lit_lens, 288), as_list(dist_lens, 32)
    lits = [s for s in range(256) if ll[s]]
    lsyms = [s for s in range(257, 286) if ll[s]]
    dsyms = [s for s in range(30) if dl[s]]
    out, made = [], 0
    while True:
        if lsyms and dsyms and rng.random() < 0.5:
            s = rng.choice(lsyms)
            length = LEN_BASE[s - 257] + rng.randrange(1 << LEN_EXTRA[s - 257])
            reach = min(back + made, far)
            ds = [c for c in dsyms if DIST_BASE[c] <= reach]
            if ds and made + length <= budget:
                c = rng.choice(ds)
                e = rng.randrange(min(1 << DIST_EXTRA[c], reach - DIST_BASE[c] + 1))
                out.append(Raw(s, length - LEN_BASE[s - 257], dsym=c, dextra=e))
                made += length
                continue
        if not lits or made + 1 > budget:
            return out
        n = rng.randint(1, 40)
        for _ in range(min(n, budget - made)):
            out.append(rng.choice(lits))
            made += 1


# ------------------------------------------------------------------------------------------------------------------
# the catalogue
# ------------------------------------------------------------------------------------------------------------------
def valid_cases():
    rng = random.Random(1951)
    noise = rng.randbytes(32768)
    cases = []
    # length 258 as 284 + 31, in a fixed and in a dynamic block, next to 285
    cases.append(ok("len284_extra31_fixed", lambda d: d.fixed([120, m284(1), 121, m284(2), (258, 3)], final=True)))
    toks = [120, 121, m284(1), (258, 2), m284(3), 122]
    lit, dist = lens_for(toks)
    cases.append(ok("len284_extra31_dynamic", lambda d: d.dynamic(toks, lit, dist, final=True)))
    # a single one-bit distance code (an incomplete code zlib accepts), for distance code 0 and for code 3
    for dc in (0, 3):
        toks = [97, 98, 99, 100] + [(L, DIST_BASE[dc]) for L in (3, 4, 10, 258, 57)] + [101]
        lit, dist = lens_for(toks)
        assert dist == {dc: 1}
        cases.append(ok("dist_single_one_bit_code%d" % dc, lambda d, toks=toks, lit=lit, dist=dist: d.dynamic(toks, lit, dist, final=True)))
    # a block without distance codes (HDIST 1, its length 0), and a single one-bit literal/length code (end-of-block only)
    toks = list(b"no distance codes at all")
    lit, _ = lens_for(toks)
    cases.append(ok("no_dist_codes", lambda d: d.dynamic(toks, lit, {}, final=True)))
    cases.append(ok("lit_single_one_bit_eob_only", lambda d: (d.dynamic([], {256: 1}, {}), d.fixed([65], final=True))))
    # HLIT 286 / HDIST 30: every length symbol with every distance code; the code-length code holds a 7-bit code
    toks = list(range(256)) + [(LEN_BASE[c] + (1 << LEN_EXTRA[c]) - 1, DIST_BASE[k] + (1 << DIST_EXTRA[k]) - 1)
                               for c in range(29) for k in range(30)]
    cases.append(ok("hlit286_hdist30", lambda d: (d.stored(noise), d.dynamic(toks, FLAT_LIT, FLAT_DIST, final=True))))
    cases.append(ok("cl_code_7bit", lambda d: (d.stored(noise), d.dynamic(toks[:300], FLAT_LIT, FLAT_DIST, final=True,
                                                                         cl_lens=seven_bit_cl(FLAT_LIT, FLAT_DIST)))))
    # 15-bit codes in both trees, used: literal 'z', length 258 (285) and distance code 29
    toks = [97] + [(258, 1)] * 130 + [122, (258, 32768), 122, (3, 24577), m284(25000), 98, (11, 16385), (258, 30000), 122]
    cases.append(ok("codes_15bit", lambda d: d.dynamic(toks, DEEP_LIT, DEEP_DIST, final=True)))
    # 16 / 17 / 18 at their minimum and maximum repeats; a 16 that runs from the literal/length into the distance lengths
    seq = [(18, 127), (17, 0), (17, 7), (18, 0), (4, 0), (16, 0), (16, 3), (18, 73), (4, 0), (16, 3), (16, 3), (16, 3), (16, 0)]
    rl = {s: 4 for s in list(range(162, 172)) + list(range(256, 262))}
    rd = {s: 4 for s in range(16)}
    toks = [162 + i % 10 for i in range(260)] + [162, 163, 171, (3, 1), 170, (7, 2), (5, 200), 165, (6, 256), 164]
    cases.append(ok("repeat_codes_min_max", lambda d: d.dynamic(toks, rl, rd, final=True, hlit=262, hdist=16, cl_seq=seq)))
    # distances at the edges of their codes, with every length 3..258 (dist < len: overlapping copies)
    for dist in (1, 2, 3, 31, 32, 33, 258, 32767, 32768):
        toks = [(L, dist) for L in range(3, 259)]
        pre = noise if dist > 64 else noise[:64]
        cases.append(ok("dist%d_len3_258" % dist, lambda d, pre=pre, toks=toks: (d.stored(pre), d.fixed(toks, final=True))))
    # a distance that reaches exactly the first byte of the output
    for n in (1, 100, 32768):
        cases.append(ok("dist_to_first_byte_%d" % n,
                        lambda d, n=n: (d.stored(noise[:n]), d.fixed([(258, n)] + [(3, n + 258)] * (n + 258 <= 32768), final=True))))
    # stored blocks of 0, 1 and 65535 bytes at every bit phase of the block header: 9-bit literals in front move the phase
    big = (noise * 2)[:65535]
    for size in (0, 1, 65535):
        for phase in range(8):
            k = (phase - 2) % 8                                 # a fixed block of k 9-bit literals takes 3 + 9k + 7 bits
            cases.append(ok("stored%d_phase%d" % (size, phase),
                            lambda d, k=k, size=size: (d.fixed([0xC0] * k), d.stored(big[:size], final=True))))
    # empty fixed and empty dynamic blocks, an empty final block, many sync markers in a row
    cases.append(ok("empty_fixed_block", lambda d: (d.fixed([]), d.fixed([]), d.fixed([66, 67], final=True))))
    cases.append(ok("empty_dynamic_block", lambda d: (d.dynamic([], FLAT_LIT, FLAT_DIST), d.fixed([68], final=True))))
    cases.append(ok("empty_final_fixed", lambda d: d.fixed([], final=True)))
    cases.append(ok("empty_final_stored", lambda d: d.stored(b"", final=True)))

    def syncs(d):
        d.fixed([120])
        for _ in range(300):
            d.sync()
        d.fixed([121, (10, 1)])
        for _ in range(7):
            d.sync()
        d.stored(b"z", final=True)
    cases.append(ok("many_sync_markers", syncs))
    return cases


def deferred_store_cases():
    """The lean loops keep the bytes of a short copy (length <= 32, dist >= len) in registers and store them when the
    next match comes: per distance 1..64, such a match, 0-2 literals, then a match whose source overlaps the first one's
    destination.  Long matches at the end keep the lean loop's room."""
    rng = random.Random(64)
    cases = []
    for dist in range(1, 65):
        toks = list(rng.randbytes(70))
        for L in sorted({3, min(max(dist, 3), 32), min(dist, 16), min(dist, 7), 32}):
            if L < 3:
                continue
            for j in (0, 1, 2):
                for d2 in {L + j, j + 1} if L + j > j + 1 else {L + j}:
                    for L2 in (3, 12, 40):
                        toks += [(L, dist)] + list(rng.randbytes(j)) + [(L2, d2)] + list(rng.randbytes(3))
        toks += [(258, 1), (258, 5)] + list(rng.randbytes(40))
        cases.append(ok("deferred_store_dist%d" % dist, lambda d, toks=toks: d.fixed(toks, final=True)))
    return cases


def straddle(toks, L, p, mod=32):
    """Literals that put the end of the length symbol (and extra bits) of a match of length L at bit p modulo `mod`,
    counted from the start of a first fixed-code block holding toks."""
    s, _, e = len_symbol(L)
    return phase_literals(3 + fixed_bits(toks), p - (7 if s < 280 else 8) - e, mod)


def handover_cases():
    """Where the lean loops hand over to the careful ones: a length and its distance on two sides of a 32-bit word (every
    bit phase of the crossing, so every placement of the stream in memory meets one), a stream ending 1-8 words after
    such a match, and 316-335 bytes of room after it (the loops need 324)."""
    rng = random.Random(32)
    cases = []
    for p in range(32):
        def crossing(d, p=p):
            toks = list(rng.randbytes(80))
            for L, dist in ((13, 40), (258, 7), (3, 80), (100, 1)):
                toks += straddle(toks, L, p) + [(L, dist)] + list(rng.randbytes(9))
            toks += [(258, 1), (258, 2)] + list(rng.randbytes(30))
            d.fixed(toks, final=True)
        cases.append(ok("straddle_phase%d" % p, crossing))
    for t in range(24):
        def ends(d, t=t):
            toks = list(rng.randbytes(80))
            toks += straddle(toks, 20, 0) + [(20, 30)] + [0xC0] * t + [(258, 1), (258, 1), (100, 1)]
            d.fixed(toks, final=True)
        cases.append(ok("ends_after_match_%d" % t, ends))
    for room in range(316, 336):
        def roomy(d, room=room):
            toks = list(rng.randbytes(80))
            toks += straddle(toks, 30, 0) + [(30, 17)] + list(rng.randbytes(room))
            d.fixed(toks, final=True)
        cases.append(ok("room_after_match_%d" % room, roomy))
    return cases


def invalid_cases():
    rng = random.Random(3)
    pre = list(b"prefix")
    cases = []
    cases.append(bad("block_type_3", "invalid block type", lambda d: (d.fixed(pre), d.header(True, 3), d.bits(0, 16))))
    cases.append(bad("block_type_3_first", "invalid block type", lambda d: (d.header(False, 3), d.bits(0, 16))))
    cases.append(bad("stored_len_nlen", "invalid stored block lengths",
                     lambda d: (d.fixed(pre), d.stored(b"abc", final=True, nlen=0x1234))))
    for hl in (287, 288):
        cases.append(bad("hlit_%d" % hl, "too many length or distance symbols",
                         lambda d, hl=hl: d.dynamic([65], FLAT_LIT, FLAT_DIST, final=True, hlit=hl)))
    for hd in (31, 32):
        cases.append(bad("hdist_%d" % hd, "too many length or distance symbols",
                         lambda d, hd=hd: d.dynamic([65], FLAT_LIT, FLAT_DIST, final=True, hdist=hd)))
    two = {97: 1, 256: 1}
    cases.append(bad("cl_oversubscribed", "invalid code lengths set",
                     lambda d: d.dynamic([97], two, {}, final=True, cl_lens=[1] * 19)))
    cases.append(bad("cl_incomplete", "invalid code lengths set",
                     lambda d: d.dynamic([97], two, {}, final=True, cl_lens=[3, 3] + [0] * 16 + [1])))
    cases.append(bad("cl_single_one_bit", "invalid code lengths set",
                     lambda d: d.dynamic([], {256: 1}, {}, final=True, cl_lens=[0] * 18 + [1],
                                         cl_seq=[(18, 127), (18, 127), (18, 3)])))
    cases.append(bad("repeat16_first", "invalid bit length repeat", _repeat16_first))
    seq = [(18, 86), (1, 0), (18, 127), (18, 9), (1, 0), (17, 0)]         # 258 lengths asked for, 260 given
    cases.append(bad("repeat_past_end", "invalid bit length repeat",
                     lambda d: d.dynamic([97], two, {}, final=True, cl_seq=seq)))
    seq16 = rle([0] * 97 + [1] + [0] * 158 + [1]) + [(16, 3)]           # a 16 that runs past the end
    cases.append(bad("repeat16_past_end", "invalid bit length repeat",
                     lambda d: d.dynamic([97], two, {}, final=True, hdist=4, cl_seq=seq16)))
    cases.append(bad("lit_oversubscribed", "invalid literal/lengths set", lambda d: d.dynamic([97], {97: 1, 98: 1, 256: 1}, {}, final=True)))
    cases.append(bad("lit_incomplete", "invalid literal/lengths set", lambda d: d.dynamic([97], {97: 2, 256: 1}, {}, final=True)))
    cases.append(bad("dist_oversubscribed", "invalid distances set",
                     lambda d: d.dynamic([97, (3, 1)], {97: 2, 256: 2, 257: 1}, {0: 1, 1: 1, 2: 1}, final=True)))
    cases.append(bad("dist_incomplete", "invalid distances set",
                     lambda d: d.dynamic([97, (3, 1)], {97: 2, 256: 2, 257: 1}, {0: 2, 1: 2, 2: 2}, final=True)))
    for s in (286, 287):
        cases.append(bad("fixed_symbol_%d" % s, "invalid literal/length code", lambda d, s=s: d.fixed(pre + [Raw(s)], final=True)))
    for s in (30, 31):
        cases.append(bad("fixed_dist_code_%d" % s, "invalid distance code",
                         lambda d, s=s: d.fixed(pre + [Raw(257, dsym=s)], final=True)))
    cases.append(bad("dynamic_dist_without_codes", "invalid distance code",
                     lambda d: d.dynamic(pre + [Raw(257, dsym=0)], lens_for(pre + [(3, 1)])[0], {}, final=True)))
    cases.append(bad("dist_single_one_bit_other_pattern", "invalid distance code",
                     lambda d: d.dynamic([97, Raw(257), RawBits(1, 1)], {97: 1, 256: 2, 257: 2}, {0: 1}, final=True)))
    cases.append(bad("lit_single_one_bit_other_pattern", "invalid literal/length code",
                     lambda d: (d.fixed(pre), d.dynamic([RawBits(1, 1)], {256: 1}, {}, final=True, eob=False))))
    cases.append(bad("dist_one_past_output", "invalid distance too far back", lambda d: d.fixed(pre + [(3, len(pre) + 1)], final=True)))
    noise = rng.randbytes(32767)
    cases.append(bad("dist_32768_one_past_output", "invalid distance too far back",
                     lambda d: (d.stored(noise), d.fixed([(258, 32768)], final=True))))
    # the data end early: inside a dynamic header, inside stored data, between a length and its distance
    cases.append(cut("cut_in_dynamic_header", lambda d: (d.fixed(pre), d.dynamic([65], FLAT_LIT, FLAT_DIST, final=True)), 12))
    cases.append(cut("cut_in_stored_data", lambda d: (d.fixed(pre), d.stored(noise[:100], final=True)), -50))

    def len_then_end(d):
        toks = pre + phase_literals(3 + fixed_bits(pre), -7, mod=8) + [(10, 2)]
        d.fixed(toks, final=True)
        assert (3 + fixed_bits(toks) - 5) % 8 == 0
    cut_at = (3 + fixed_bits(pre + phase_literals(3 + fixed_bits(pre), -7, mod=8)) + 7) // 8
    cases.append(cut("cut_between_length_and_distance", len_then_end, cut_at))
    return cases


def _repeat16_first(d, final=True, opening=((16, 0),)):
    """A code-length sequence that opens with 16.  The rest is a consistent header for lengths whose first three are
    zero: a decoder that took the 16 for three zeros would decode the block (and its check values) as written."""
    lit = {s: 4 for s in list(range(97, 111)) + [256, 257]}
    seq = list(opening) + rle(as_list(lit, 288)[3:258] + [1])  # HLIT 258, then the one distance length
    d.dynamic([97, 98, (3, 1), 110, (3, 1), 100], lit, {0: 1}, final=final, cl_seq=seq)


def catalogue():
    return valid_cases() + deferred_store_cases() + handover_cases() + invalid_cases()


# ------------------------------------------------------------------------------------------------------------------
# long streams for the segment-parallel decoder
# ------------------------------------------------------------------------------------------------------------------
def _fill(d, rng, n, final):
    """Exactly n more bytes of output as stored blocks of noise (at least one block, so a final flag has a home)."""
    while True:
        k = min(n, 65535)
        n -= k
        d.stored(rng.randbytes(k), final=final and n == 0)
        if n == 0:
            return


def piece(d, rng, size, lead, final, base):
    """`size` bytes of output in blocks that carry the catalogue's valid constructs, closed by a sync marker (or as the
    final block).  lead: "far" opens with a match of distance 32768, "run" with a dist-1 run of 258 (both reach in front
    of the piece), "none" keeps every distance inside the piece (its tail then holds no window symbols).  `base` is where
    the piece's output starts."""
    start = d.pos
    back = start if lead != "none" else start - base

    def made():
        return d.pos - start
    if lead == "far":
        d.fixed([(258, 32768)])
    elif lead == "run":
        d.fixed([(258, 1)])
    d.stored(rng.randbytes(rng.randint(size // 64, size // 32)))
    reach = lambda: back + made()
    d.dynamic(rand_tokens(rng, FLAT_LIT, FLAT_DIST, size // 8, reach()) + [m284(min(reach(), 32768))], FLAT_LIT, FLAT_DIST,
              cl_lens=seven_bit_cl(FLAT_LIT, FLAT_DIST))
    d.dynamic(rand_tokens(rng, DEEP_LIT, DEEP_DIST, size // 8, reach()), DEEP_LIT, DEEP_DIST)
    d.dynamic(rand_tokens(rng, {97: 2, 98: 2, 256: 2, 285: 3, 258: 3}, {0: 1}, size // 16, reach()), {97: 2, 98: 2, 256: 2, 285: 3, 258: 3}, {0: 1})
    d.dynamic(list(rng.randbytes(500)), lens_for(list(range(256)))[0], {})
    d.fixed(rand_tokens(rng, [8] * 288, [5] * 30, size // 8, reach()))
    assert made() < size, (made(), size)
    _fill(d, rng, size - made(), final)
    if not final:
        d.sync()


def period_piece(d, rng, size, final):
    """Output that repeats with a period of 32 KiB, written as distance-32768 matches only (noise first, if there is no
    history yet): every window reference of a segment is to the one in front, so the dependent tails form one chain."""
    toks = []
    n = size
    if not d.pos:
        d.stored(rng.randbytes(32768))
        n -= 32768
    while n:
        L = 258 if n >= 261 or n == 258 else n - 3 if n > 258 else n
        toks.append((L, 32768))
        n -= L
    d.fixed(toks, final=final)
    if not final:
        d.sync()


def chain_piece(d, rng, size, final):
    """Like period_piece, but the output has no period: matches of random length from 30000-32768 bytes back, and now
    and then a fresh literal.  Every byte of a segment but those literals still comes from the segment in front (a copy
    of a window symbol is one), so every tail depends on the one in front; and a byte read from the wrong place -- a
    slot of a 32 KiB ring that holds another generation, say -- is the wrong byte."""
    toks = []
    n = size
    if not d.pos:
        d.stored(rng.randbytes(32768))
        n -= 32768
    while n:
        if n >= 6 and rng.random() < 0.01:
            toks.append(rng.randrange(256))
            n -= 1
            continue
        L = min(rng.randint(100, 258), n)
        if 0 < n - L < 3:
            L = n - 3 if n - 3 >= 3 else n
        toks.append((L, rng.randint(30000, 32768)))
        n -= L
    d.fixed(toks, final=final)
    if not final:
        d.sync()


def long_stream(*args, **kw):
    """(raw, plain) of long_writer(...)."""
    return long_writer(*args, **kw).result()


def long_writer(seed, sizes, lead="none", bad_at=None, bad_block=None, markers=True):
    """The Deflate writer of a stream of pieces with the given output sizes (16 KiB or more), each ended by a sync marker (markers=False:
    nothing between them; the dynamic blocks are then found by the block finder).  lead "period" / "chain": pieces of
    period_piece / chain_piece, else of piece() with that lead.  bad_block(d) writes an invalid construct at the start
    of piece bad_at."""
    rng = random.Random(seed)
    d = Deflate()
    for i, size in enumerate(sizes):
        last = i == len(sizes) - 1
        base = d.pos
        if not markers:
            blockfinder_piece(d, rng, size, last)
            continue
        while True:
            # the marker pattern may turn up in coded data (a run of 1-bit codes, then 15-bit ones): such a piece is
            # written again, so that the markers of the stream are exactly the sync points
            m = d.mark()
            if lead == "period":
                period_piece(d, rng, size, last)
            elif lead == "chain":
                chain_piece(d, rng, size, last)
            else:
                if i == bad_at:
                    d.fixed([65, 66])
                    bad_block(d)
                piece(d, rng, size - (d.pos - base), lead if i else "none", last, base)
            body = bytes(d.buf[max(m[0] - 3, 0):len(d.buf) - (0 if last else 4)])
            if MARKER not in body:
                break
            d.rewind(m)
    return d


def tails_with_window_symbols(copies, seg_starts, total):
    """Indices j of the segments [seg_starts[j], seg_starts[j + 1]) whose last 32 KiB hold a byte that comes, through
    copies inside the segment, from in front of it -- the tails that depend on the segment in front.  `copies` is
    Deflate.copies."""
    import numpy as np
    win = np.zeros(total, dtype=bool)                           # byte p is a window symbol of its segment
    bounds = list(seg_starts) + [total]
    seg = np.zeros(total, dtype=np.int64)
    for j in range(len(seg_starts)):
        seg[bounds[j]:bounds[j + 1]] = bounds[j]
    for pos0, length0, dist in copies:
        for off in range(0, length0, dist):                     # an overlapping copy: pieces of at most dist bytes
            pos, length = pos0 + off, min(dist, length0 - off)
            start = seg[pos]
            src = pos - dist
            k = min(max(start - src, 0), length)                # the part in front of the segment
            win[pos:pos + k] = True
            win[pos + k:pos + length] = win[src + k:src + length]
    return [j for j in range(len(seg_starts)) if win[max(bounds[j + 1] - 32768, bounds[j]):bounds[j + 1]].any()]


def blockfinder_piece(d, rng, size, final):
    """Non-final dynamic blocks only (the block finder's candidates), the last one closing at `size` bytes of output."""
    start = len(d.plain)
    while True:
        left = size - (len(d.plain) - start)
        toks = rand_tokens(rng, FLAT_LIT, FLAT_DIST, min(left, 40000), len(d.plain))
        got = sum(1 if isinstance(t, int) else t.meaning()[0] for t in toks)
        if got == left:
            d.dynamic(toks, FLAT_LIT, FLAT_DIST, final=final)
            return
        if left - got < 300:                                    # close with literals
            toks += list(rng.randbytes(left - got))
            d.dynamic(toks, FLAT_LIT, FLAT_DIST, final=final)
            return
        d.dynamic(toks, FLAT_LIT, FLAT_DIST)


def chunked_sizes(total):
    """Piece sizes of this library's own layout: CHUNK bytes each, the last one what is left."""
    return [CHUNK] * (total // CHUNK) + ([total % CHUNK] if total % CHUNK else [])


# invalid constructs that fit anywhere inside a stream (after some output)
def long_invalid_blocks():
    two = {97: 1, 256: 1}
    seq = [(18, 86), (1, 0), (18, 127), (18, 9), (1, 0), (17, 0)]
    return {
        "block_type_3": lambda d: (d.header(False, 3), d.bits(0, 16)),
        "stored_len_nlen": lambda d: d.stored(b"abc", nlen=0x1234),
        "hlit_287": lambda d: d.dynamic([65], FLAT_LIT, FLAT_DIST, hlit=287),
        "hdist_31": lambda d: d.dynamic([65], FLAT_LIT, FLAT_DIST, hdist=31),
        "cl_oversubscribed": lambda d: d.dynamic([97], two, {}, cl_lens=[1] * 19),
        "cl_incomplete": lambda d: d.dynamic([97], two, {}, cl_lens=[3, 3] + [0] * 16 + [1]),
        "repeat16_first": lambda d: _repeat16_first(d, final=False),
        "repeat_past_end": lambda d: d.dynamic([97], two, {}, cl_seq=seq),
        "lit_oversubscribed": lambda d: d.dynamic([97], {97: 1, 98: 1, 256: 1}, {}),
        "dist_incomplete": lambda d: d.dynamic([97, (3, 1)], {97: 2, 256: 2, 257: 1}, {0: 2, 1: 2, 2: 2}),
        "fixed_symbol_286": lambda d: d.fixed([Raw(286)]),
        "fixed_dist_code_30": lambda d: d.fixed([Raw(257, dsym=30)]),
        "dist_single_one_bit_other_pattern": lambda d: d.dynamic([97, Raw(257), RawBits(1, 1)], {97: 1, 256: 2, 257: 2}, {0: 1}),
        "lit_single_one_bit_other_pattern": lambda d: d.dynamic([RawBits(1, 1)], {256: 1}, {}, eob=False),
        "lit_incomplete": lambda d: d.dynamic([97], {97: 2, 256: 1}, {}),
        "dist_oversubscribed": lambda d: d.dynamic([97, (3, 1)], {97: 2, 256: 2, 257: 1}, {0: 1, 1: 1, 2: 1}),
        "dynamic_dist_without_codes": lambda d: d.dynamic([97, Raw(257, dsym=0)], {97: 2, 256: 2, 257: 1}, {}),
        "cl_single_one_bit": lambda d: d.dynamic([], {256: 1}, {}, cl_lens=[0] * 18 + [1], cl_seq=[(18, 127), (18, 107)]),
        "repeat16_past_end": lambda d: d.dynamic([97], {97: 1, 256: 1}, {}, hdist=4,
                                                 cl_seq=rle([0] * 97 + [1] + [0] * 158 + [1]) + [(16, 3)]),
    }


def far_in_first_segment(d):
    """A distance past the output inside the first segment (the segment decoder's own rule for it).  The writer takes the
    missing history for zeros, so the check values are those of a decoder that read zeros there."""
    d.zero_history = True
    d.stored(bytes(range(256)) * 80)
    d.fixed([(258, d.pos + 100)])
