// zb_inflate.cu -- K4: many independent DEFLATE streams decoded in parallel, one warp each.
//
// Replaces the reference's inflate() state machine (qcsrc/inflate.c:554-1153), its table
// builder inflate_table() (qcsrc/inftrees.c:32-329) and the inner loop inflate_fast()
// (qcsrc/inffast.c:67-302) for the case the GPU is good at: a batch of complete streams
// (uncompress() semantics, qcsrc/uncompr.c:26-61), and -- through the same code with a
// saved state -- one z_stream fed piecewise (zapi_stream.c).
//
// Shape.  DEFLATE decoding is serial inside a stream (the bit position of symbol i+1 depends
// on symbol i; copies depend on earlier output), so the parallel axis is the stream.  A warp
// owns a stream: all 32 lanes run the same bit-level decode on warp-uniform values (no
// divergence), and the lanes split the two things that are wide: building the Huffman tables
// of a dynamic block and copying matches (lane i moves byte i; overlapping copies read
// modulo the distance, so nothing depends on bytes written by the same copy).
// Tables live in shared memory, per warp: a 10-bit primary table for literal/length codes and
// an 8-bit primary for distances, each entry carrying {code bits, extra bits, kind, base}; codes
// longer than the primary width (rare) fall back to canonical first-code decoding over the
// sorted symbol list, which is also what rejects bit patterns that are not codes.
//
// Validity rules follow the reference: over-subscribed sets and incomplete sets (other than a
// single one-bit code) are rejected (inftrees.c:130-138), nlen > 286 / ndist > 30
// (inflate.c:846), stored LEN/NLEN (inflate.c:810), distance beyond the produced output
// (inflate.c:1039), zlib header (inflate.c:589-632) and Adler-32 trailer (inflate.c:1077-1098).
//
// Roofline: HBM (algorithmic bytes = compressed in + plain out), but the kernel is
// latency/issue bound by construction; see DESIGN.md.
#include "zb_inflate.cuh"
#include "zb200_internal.h"
#include <cooperative_groups.h>
#include <vector>
#include <algorithm>
#include <string.h>
#include <stdlib.h>

namespace zb {

constexpr int kInfWarps = 4;                     // warps (= streams in flight) per CTA
constexpr int kLitBits = 10, kDistBits = 8, kClBits = 7;
constexpr int kLitSize = 1 << kLitBits, kDistSize = 1 << kDistBits;
constexpr uint32_t kFull = 0xffffffffu;
constexpr uint32_t kWindow32 = 32768;

__constant__ uint8_t c_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// entry: bits 0-4 code length (0 = not in the primary table), 5-9 code length + extra-bit count (what the symbol
// consumes), 10-11 kind, 15 set for a length / distance base that is in the table, 16-30 literal value / symbol, or
// base of a length or distance, 31 set for a literal that is in the table.  Bits 15 and 31 are what the lean loop
// tests: one sign test for "literal", one bit test for "base", anything else goes to the careful decoder.
enum { kLit = 0, kBase = 1, kEob = 2, kBad = 3 };
__device__ __forceinline__ uint32_t mk_entry(uint32_t len, uint32_t extra, uint32_t kind, uint32_t val)
{
    const uint32_t flags = len == 0 ? 0u : kind == kBase ? 0x8000u : kind == kLit ? 0x80000000u : 0u;
    return len | ((len + extra) << 5) | (kind << 10) | (val << 16) | flags;
}
__device__ __forceinline__ uint32_t ent_len(uint32_t e) { return e & 31u; }
__device__ __forceinline__ uint32_t ent_extra(uint32_t e) { return ((e >> 5) & 31u) - (e & 31u); }
__device__ __forceinline__ uint32_t ent_kind(uint32_t e) { return (e >> 10) & 3u; }
__device__ __forceinline__ uint32_t ent_val(uint32_t e) { return (e >> 16) & 0x7fffu; }
__device__ __forceinline__ uint32_t litlen_entry(uint32_t s, uint32_t len)
{
    if (s < 256) return mk_entry(len, 0, kLit, s);
    if (s == 256) return mk_entry(len, 0, kEob, 0);
    if (s > 285) return mk_entry(len, 0, kBad, 0);
    uint32_t c = s - 257;
    if (c < 8) return mk_entry(len, 0, kBase, 3 + c);
    if (c == 28) return mk_entry(len, 0, kBase, 258);
    uint32_t e = (c >> 2) - 1;
    return mk_entry(len, e, kBase, 3 + ((4 + (c & 3)) << e));
}
__device__ __forceinline__ uint32_t dist_entry(uint32_t s, uint32_t len)
{
    if (s > 29) return mk_entry(len, 0, kBad, 0);
    if (s < 4) return mk_entry(len, 0, kBase, 1 + s);
    uint32_t e = (s >> 1) - 1;
    return mk_entry(len, e, kBase, 1 + ((2 + (s & 1)) << e));
}

struct WarpTables {
    uint32_t lit[kLitSize];
    uint32_t dist[kDistSize];                    // also hosts the code-length code while a header is read
    uint32_t lit_count[16], dist_count[16];      // symbols per code length
    uint32_t first[16], offs[16], run[16];       // scratch while building
    uint16_t lit_sorted[288];
    uint16_t dist_sorted[32];
    uint8_t  lens[320];
    uint8_t  cl_lens[20];
    int      lit_max, dist_max;                  // longest code present (0 = no codes at all)
};

struct Bits {
    const uint32_t* words;                       // 4-byte aligned base at the last seek (see seek_bits)
    uint32_t nwords, nextw;                      // words from that base to the end of the stream (at most 2^32 - 1) / next to load
    uint64_t buf;
    int cnt;
    uint64_t used, total;                        // bits consumed so far / bits in the stream
};

__device__ __forceinline__ void refill(Bits& b)
{
    if (b.cnt <= 32) {
        uint32_t w = b.nextw < b.nwords ? __ldg(b.words + b.nextw) : 0u;
        b.nextw++;
        b.buf |= (uint64_t)w << b.cnt;
        b.cnt += 32;
    }
}
__device__ __forceinline__ uint32_t peek(const Bits& b, int n) { return (uint32_t)b.buf & ((1u << n) - 1u); }
__device__ __forceinline__ void drop(Bits& b, int n) { b.buf >>= n; b.cnt -= n; b.used += n; }
__device__ __forceinline__ bool have(const Bits& b, int n) { return b.used + (uint64_t)n <= b.total; }

// Every seek moves the word base to the word holding `bitpos`, so the 32-bit word indices (nextw here, wi in the lean
// loops) count from a recent seek, not from the start of the stream: a stream of 2^32 words (16 GiB) or more would wrap
// them.  The lean loops seek whenever they stop, and they stop before nwords, so no index wraps between two seeks.
__device__ void seek_bits(Bits& b, const uint8_t* in, uint64_t bitpos)
{
    const uintptr_t a = (uintptr_t)in + (bitpos >> 3);
    const uintptr_t base = a & ~(uintptr_t)3;
    const uintptr_t end = ((uintptr_t)in + (b.total >> 3) + 3) & ~(uintptr_t)3;
    const uint64_t left = end > base ? (end - base) >> 2 : 0;
    const int skip = (int)((a & 3) * 8 + (bitpos & 7));
    b.words = reinterpret_cast<const uint32_t*>(base);
    b.nwords = left > 0xffffffffu ? 0xffffffffu : (uint32_t)left;
    b.nextw = 0;
    b.buf = 0; b.cnt = 0;
    refill(b);
    b.buf >>= skip; b.cnt -= skip;
    refill(b);
    b.used = bitpos;
}

// ---- table construction, all lanes of the warp cooperate (inftrees.c:32-329) ----
// kind 0 = code-length code, 1 = literal/length, 2 = distance.  Returns 0 ok, -1 invalid set.
__device__ int build_table(const uint8_t* lens, int n, int kind, uint32_t* tab, int tab_bits,
                           uint16_t* sorted, uint32_t* count, WarpTables* t, int* max_out)
{
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    __syncwarp();
    if (lane < 16) { count[lane] = 0; t->run[lane] = 0; }
    for (int i = lane; i < (1 << tab_bits); i += 32) tab[i] = 0;
    __syncwarp();
    for (int s = lane; s < n; s += 32) atomicAdd(&count[lens[s]], 1u);
    __syncwarp();
    int maxlen = 15;
    while (maxlen >= 1 && count[maxlen] == 0) maxlen--;
    if (lane == 0) *max_out = maxlen;
    if (maxlen == 0) { __syncwarp(); return 0; }  // no codes: an error only if a symbol is needed (inftrees.c:116-124)
    int left = 1;
    for (int len = 1; len <= 15; len++) {
        left = (left << 1) - (int)count[len];
        if (left < 0) return -1;                 // over-subscribed
    }
    if (left > 0 && (kind == 0 || maxlen != 1)) return -1;   // incomplete
    if (lane == 0) {
        uint32_t code = 0, o = 0;
        for (int len = 1; len <= 15; len++) {
            code = (code + (len > 1 ? count[len - 1] : 0u)) << 1;
            t->first[len] = code;
            t->offs[len] = o;
            o += count[len];
        }
    }
    __syncwarp();
    for (int base = 0; base < n; base += 32) {
        const int s = base + lane;
        const uint32_t L = s < n ? lens[s] : 0u;
        const uint32_t grp = __match_any_sync(kFull, L);
        const uint32_t rank = t->run[L] + __popc(grp & lt);
        __syncwarp();
        if ((grp & lt) == 0) t->run[L] += __popc(grp);       // first lane of each length group
        __syncwarp();
        if (L != 0) {
            if (sorted) sorted[t->offs[L] + rank] = (uint16_t)s;
            if ((int)L <= tab_bits) {
                const uint32_t code = t->first[L] + rank;
                const uint32_t rc = __brev(code) >> (32 - L);
                const uint32_t e = kind == 1 ? litlen_entry((uint32_t)s, L)
                                 : kind == 2 ? dist_entry((uint32_t)s, L) : mk_entry(L, 0, kLit, (uint32_t)s);
                for (uint32_t j = rc; j < (1u << tab_bits); j += 1u << L) tab[j] = e;
            }
        }
    }
    __syncwarp();
    return 0;
}

// Canonical decode for codes that are not in the primary table.  Returns the symbol, -1 if the
// input ends inside the code, -2 if the bits are not a code of this set.  Consumes on success.
__device__ int slow_symbol(Bits& b, const uint32_t* count, const uint16_t* sorted, int maxlen)
{
    if (maxlen == 0) return have(b, 1) ? -2 : -1;
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= maxlen; len++) {
        if (!have(b, len)) return -1;
        code |= (int)((b.buf >> (len - 1)) & 1u);
        const int c = (int)count[len];
        if (code - c < first) {
            drop(b, len);
            return sorted[index + (code - first)];
        }
        index += c; first += c; first <<= 1; code <<= 1;
    }
    return -2;
}

__device__ __forceinline__ void store_lens(WarpTables* t, int at, int n, uint8_t v)
{
    const int lane = threadIdx.x & 31;
    for (int i = lane; i < n; i += 32) t->lens[at + i] = v;
}

enum Stop { kRunning = 0, kDone, kShortIn, kShortOut, kError, kWantDict };

// Output cursor: positions are relative to p; bytes at negative offsets down to -hist are history.
// Count mode (kCount, zb200_inflate_batch_size): p is null, nothing is stored, pos only counts; cap is the caller's limit.
struct Out { uint8_t* p; uint64_t pos, cap, hist; };

template <bool kCount>
__device__ __forceinline__ uint32_t copy_match(Out& o, uint32_t len, uint32_t dist)
{
    const int lane = threadIdx.x & 31;
    uint32_t n = len;
    if (o.pos + n > o.cap) n = (uint32_t)(o.cap - o.pos);
    if (kCount) { o.pos += n; return n; }
    __syncwarp();
    uint8_t* dst = o.p + o.pos;
    const uint8_t* src = dst - dist;
    if (dist >= n) {
        for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i];
    } else {
        for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i % dist];
    }
    __syncwarp();
    o.pos += n;
    return n;
}

// Decodes symbols of the current block until end-of-block or a stop condition (the work of
// inflate_fast, inffast.c:67-302, plus the careful tail of inflate.c:951-1076).  Count mode decodes and checks the same
// symbols and stops at the same ones; it only leaves out the stores.
template <bool kCount>
__device__ Stop decode_block(Bits& b, Out& o, const WarpTables* t, InfState* st, bool streaming, bool one)
{
    const int lane = threadIdx.x & 31;
    for (;;) {
        const uint64_t mark = b.used;
        refill(b);
        uint32_t e = t->lit[peek(b, kLitBits)];
        const uint32_t len = ent_len(e);
        if (len != 0) {
            if (!have(b, (int)len)) { b.used = mark; return kShortIn; }
            drop(b, (int)len);
        } else {
            int s = slow_symbol(b, t->lit_count, t->lit_sorted, t->lit_max);
            if (s == -1) { b.used = mark; return kShortIn; }
            if (s == -2) { st->msg = kMsgBadLit; return kError; }
            e = litlen_entry((uint32_t)s, 1);
        }
        const uint32_t kind = ent_kind(e);
        if (kind == kLit) {
            if (o.pos >= o.cap) { if (streaming) b.used = mark; return kShortOut; }
            if (!kCount && lane == 0) o.p[o.pos] = (uint8_t)ent_val(e);
            o.pos++;
            if (one) return kRunning;
            continue;
        }
        if (kind == kEob) return kDone;
        if (kind == kBad) { st->msg = kMsgBadLit; return kError; }
        const int xl = (int)ent_extra(e);
        if (!have(b, xl)) { b.used = mark; return kShortIn; }
        const uint32_t mlen = ent_val(e) + peek(b, xl);
        drop(b, xl);
        refill(b);
        uint32_t de = t->dist[peek(b, kDistBits)];
        const uint32_t dl = ent_len(de);
        if (dl != 0) {
            if (!have(b, (int)dl)) { b.used = mark; return kShortIn; }
            drop(b, (int)dl);
        } else {
            int s = slow_symbol(b, t->dist_count, t->dist_sorted, t->dist_max);
            if (s == -1) { b.used = mark; return kShortIn; }
            if (s == -2) { st->msg = kMsgBadDist; return kError; }
            de = dist_entry((uint32_t)s, 1);
        }
        if (ent_kind(de) == kBad) { st->msg = kMsgBadDist; return kError; }
        const int xd = (int)ent_extra(de);
        refill(b);
        if (!have(b, xd)) { b.used = mark; return kShortIn; }
        const uint32_t dist = ent_val(de) + peek(b, xd);
        drop(b, xd);
        if ((uint64_t)dist > o.pos + o.hist) { st->msg = kMsgFar; return kError; }
        const uint32_t done = copy_match<kCount>(o, mlen, dist);
        if (done < mlen) {
            st->copy_len = mlen - done; st->copy_dist = dist;
            return kShortOut;
        }
        if (one) return kRunning;
    }
}

// The same decode without the bookkeeping, for the stretch of a block where neither buffer can run out: a symbol
// starts only while five whole input words lie ahead (it takes at most 48 bits) and 260 bytes of room are left (the
// reference's inflate_fast makes the same deal, inffast.c:24-30,67-70).  Every lane executes this loop, so its cost is
// its instruction count: the bit position is a word index plus an offset below 64 into a register pair (lo, hi) with
// the following word already loaded (its latency hides behind the symbols in between), a code is looked up in the 32
// bits at the offset (one funnel shift), a field is "bits below the total, shifted by the code length", and the only
// tests on an entry are its sign (literal) and bit 15 (length / distance base).  Anything else -- a code longer than
// the primary table, end of block, an invalid symbol, a distance beyond the history -- leaves the loop at the start
// of that symbol and the careful decoder above deals with it (and produces the error, if it is one).
// Returns kDone after an end-of-block code, kRunning otherwise.
// Count mode is the same loop without the stores and the deferred copy: a literal is its code length and one count, a
// match its length and distance codes, the distance check against what was counted, and one add.
template <bool kCount>
__device__ Stop decode_fast(Bits& b, Out& o, const WarpTables* t, const uint8_t* in)
{
    const int lane = threadIdx.x & 31;
    const uint32_t nwords = b.nwords;
    const uint32_t* words = b.words;
    const uint64_t room64 = o.cap - o.pos, back64 = o.pos + o.hist;
    const uint32_t room = room64 > 0x7fffffffu ? 0x7fffffffu : (uint32_t)room64;
    const uint32_t back = back64 > 0x7fffffffu ? 0x7fffffffu : (uint32_t)back64;   // bytes behind p at entry
    if (room < 324 || nwords < 6) return kRunning;
    // Limits are tested where the word index moves and after a match (not per literal): between two tests at most 32
    // bits go by, i.e. at most 64 bytes of literals -- the 64 on top of the 260 bytes a symbol may need.
    const uint32_t w_lim = nwords - 5, p_lim = room - 324;
    const uint64_t pos0 = (uint64_t)b.nextw * 32u - (uint64_t)b.cnt;              // bit position from the word base
    const uint32_t wi0 = (uint32_t)(pos0 >> 5), off0 = (uint32_t)pos0 & 31u;
    if (wi0 > w_lim) return kRunning;
    uint32_t wi = wi0, off = off0;
    uint32_t lo = __ldg(words + wi), hi = __ldg(words + wi + 1), nxt = __ldg(words + wi + 2);
    uint8_t* p = kCount ? nullptr : o.p + o.pos;
    if constexpr (!kCount) {
        asm volatile("" : "+l"(p));                             // one register pair; not re-derived from its parts at every use
        __builtin_assume(__isGlobal(p));
    }
    const uint32_t* const lit = t->lit;
    const uint32_t* const dtab = t->dist;
    uint32_t produced = 0;
    uint32_t end_wi, end_off;                                   // where the careful decoder takes over
    bool pend = false;                                          // this lane holds a byte of the last copy that is still to be stored
    uint32_t pend_v = 0;
    uint8_t* pend_d = p;
    Stop result = kRunning;
    for (;;) {
        if (off >= 32) {
            off -= 32; lo = hi; hi = nxt; wi++;
            nxt = __ldg(words + wi + 2);
            asm volatile("");                                   // keep this a branch: it runs once per 32 bits, not per symbol
            if (wi > w_lim || produced > p_lim) { end_wi = wi; end_off = off; break; }
        }
        const uint32_t win = __funnelshift_r(lo, hi, off);
        const uint32_t e = lit[win & (kLitSize - 1)];
        if ((int32_t)e < 0) {
            // literals come in runs: try the next symbol too -- at least 17 bits of the window are left, enough for any
            // code.  Every lane stores the (same) byte: cheaper than electing one.
            const uint32_t e2 = lit[__funnelshift_r(win, 0u, e) & (kLitSize - 1)];
            uint8_t* q = p + produced;
            if (!kCount) q[0] = (uint8_t)(e >> 16);
            off += e & 31u; produced++;
            if ((int32_t)e2 < 0) { if (!kCount) q[1] = (uint8_t)(e2 >> 16); off += e2 & 31u; produced++; }
            continue;
        }
        end_wi = wi; end_off = off;                             // start of this symbol
        if (!(e & 0x8000u)) {
            if (ent_kind(e) == kEob && ent_len(e) != 0) { end_off = off + ent_len(e); result = kDone; }
            break;
        }
        const uint32_t tot = (e >> 5) & 31u;
        const uint32_t mlen = (e >> 16) + __funnelshift_r(win & ((1u << tot) - 1u), 0u, e);   // bit 31 is clear: not a literal
        off += tot;
        if (off >= 32) {
            // the word index moves here too: without this test a stream whose every word crossing falls between a length
            // and its distance (one-bit codes at an odd phase) would never meet the limit at the top of the loop
            off -= 32; lo = hi; hi = nxt; wi++;
            if (wi > w_lim) break;                              // back to the start of this symbol (end_wi / end_off)
            nxt = __ldg(words + wi + 2);
        }
        const uint32_t dwin = __funnelshift_r(lo, hi, off);
        const uint32_t de = dtab[dwin & (kDistSize - 1)];
        const uint32_t dtot = (de >> 5) & 31u;
        const uint32_t dist = (de >> 16) + __funnelshift_r(dwin & ((1u << dtot) - 1u), 0u, de);
        if (!(de & 0x8000u) || dist > back + produced) break;
        off += dtot;
        if (kCount) {
            produced += mlen;
            if (produced > p_lim) { end_wi = wi; end_off = off; break; }
            continue;
        }
        uint8_t* d = p + produced + lane;
        const uint8_t* s = d - dist;
        produced += mlen;
        // The bytes of a short copy are loaded now and stored when the next match arrives (or the loop ends): the trip
        // to L2 -- the output was written moments ago and is not in L1 -- overlaps the decoding of the symbols in between
        // instead of stalling the warp at the store.  Literal stores in between go to other addresses.
        if (pend) *pend_d = (uint8_t)pend_v;
        __syncwarp();
        if (mlen <= 32u && dist >= mlen) {
            pend = (uint32_t)lane < mlen;
            if (pend) pend_v = *s;
            pend_d = d;
        } else {
            pend = false;
            if (dist >= 32u || dist >= mlen) {
                // a pass of 32 bytes never reads what the same pass writes; later passes may read earlier ones
#pragma unroll 1
                for (uint32_t i0 = 0; i0 < mlen; i0 += 32) { if (i0 + lane < mlen) d[i0] = s[i0]; __syncwarp(); }
            } else {
                const uint8_t* s0 = s - lane;
#pragma unroll 1
                for (uint32_t i = lane; i < mlen; i += 32) d[i - lane] = s0[i % dist];
                __syncwarp();
            }
        }
        if (produced > p_lim) { end_wi = wi; end_off = off; break; }
    }
    if (!kCount && pend) *pend_d = (uint8_t)pend_v;
    __syncwarp();
    o.pos += produced;
    seek_bits(b, in, b.used + ((uint64_t)(end_wi - wi0) * 32u + end_off - off0));
    return result;
}

// Adds out[0..n) to the running Adler-32 (s1, s2) of the stream; all lanes cooperate.
__device__ void adler_fold(uint32_t& s1, uint32_t& s2, const uint8_t* p, uint64_t n)
{
    const int lane = threadIdx.x & 31;
    while (n) {
        const uint32_t m = n > (1u << 20) ? (1u << 20) : (uint32_t)n;
        uint64_t a = 0, w = 0;
        for (uint32_t i = lane; i < m; i += 32) {
            const uint32_t v = p[i];
            a += v; w += (uint64_t)(m - i) * v;
        }
#pragma unroll
        for (int k = 16; k; k >>= 1) {
            a += __shfl_xor_sync(kFull, a, k);
            w += __shfl_xor_sync(kFull, w, k);
        }
        s2 = (uint32_t)((s2 + (uint64_t)m % kAdlerBase * s1 + w % kAdlerBase) % kAdlerBase);
        s1 = (uint32_t)((s1 + a) % kAdlerBase);
        p += m; n -= m;
    }
}

// Whole-stream driver for one warp.  `st` is this stream's state (shared memory for the batch
// path, global memory for a z_stream, where it carries the position between calls).
// kCount: the sizing pass of zb200_inflate_batch_size (never streaming, out == nullptr, out_cap = the limit).  Headers,
// tables, symbols, distances and stops are those of the decode; stored bytes are skipped, the Adler-32 is not computed,
// and a gzip ISIZE is compared here (the decode leaves it to the k_checksum_batch launch behind it).
template <bool kCount>
__device__ void inflate_warp(const uint8_t* in, uint64_t in_len, uint8_t* out, uint64_t out_cap,
                             bool streaming, InfState* st, WarpTables* t,
                             uint64_t* out_len_p, uint64_t* in_used_p, int32_t* status_p, int32_t* msg_p)
{
    const int lane = threadIdx.x & 31;
    Bits b;
    b.total = in_len * 8;
    seek_bits(b, in, st->bit_off);
    Out o{out, 0, out_cap, st->hist};
    int wrap = st->wrap;                                        // 3 = zlib or gzip, decided by the first two bytes
    int mode = st->mode;
    int last = st->last;
    uint32_t s1 = st->s1, s2 = st->s2;
    uint64_t folded = 0;
    Stop stop = kRunning;

    if (streaming && (mode == kModeCodes || mode == kModeCopy)) {   // resume inside a compressed block: rebuild its tables
        for (int i = lane; i < 320; i += 32) t->lens[i] = st->lens[i];
        __syncwarp();
        build_table(t->lens, st->nlen, 1, t->lit, kLitBits, t->lit_sorted, t->lit_count, t, &t->lit_max);
        build_table(t->lens + st->nlen, st->ndist, 2, t->dist, kDistBits, t->dist_sorted, t->dist_count, t, &t->dist_max);
    }

    while (stop == kRunning) {
        const uint64_t mark = b.used;
        if (mode == kModeHead) {
            if (wrap == kWrapAuto) {                  // inflate.c:596: gzip if the stream opens with 1f 8b
                if (!have(b, 16)) { stop = kShortIn; continue; }
                refill(b);
                wrap = peek(b, 16) == 0x8b1fu ? ZB200_WRAP_GZIP : ZB200_WRAP_ZLIB;
                if (lane == 0) st->wrap = wrap;
            }
            if (wrap == ZB200_WRAP_ZLIB) {           // inflate.c:589-632
                if (!have(b, 16)) { stop = kShortIn; continue; }
                refill(b);
                const uint32_t cmf = peek(b, 8); drop(b, 8);
                const uint32_t flg = peek(b, 8); drop(b, 8);
                if (((cmf << 8) + flg) % 31u) { st->msg = kMsgHeader; stop = kError; continue; }
                if ((cmf & 15u) != 8u) { st->msg = kMsgMethod; stop = kError; continue; }
                {   // inflate.c:622: a stream that declares a larger window than the caller opened is refused
                    const uint32_t wb = (st->flags >> 8) & 15u;
                    if ((cmf >> 4) + 8u > (wb ? wb : 15u)) { st->msg = kMsgWindow; stop = kError; continue; }
                }
                s1 = 1; s2 = 0;
                if (flg & 0x20u) {                    // preset dictionary, inflate.c:630, 761-770
                    if (!streaming) { st->msg = kMsgNeedDict; stop = kError; continue; }
                    if (!have(b, 32)) { b.used = mark; stop = kShortIn; continue; }
                    uint32_t id = 0;
                    for (int i = 0; i < 4; i++) { refill(b); id = (id << 8) | peek(b, 8); drop(b, 8); }
                    st->dict_id = id;
                    mode = kModeDict; stop = kWantDict; continue;
                }
            } else if (wrap == ZB200_WRAP_GZIP) {    // inflate.c:596-602, 634-759; nothing is kept of the header fields
                // bytes are read straight from the input: the header starts on a byte boundary
                const uint64_t h0 = b.used >> 3;
                const uint64_t avail = in_len - h0;
                const uint8_t* hp = in + h0;
                uint64_t need = 10;
                int bad = 0;
                bool shortin = avail < need;
                uint32_t flg = 0;
                if (!shortin) {
                    if (hp[0] != 0x1f || hp[1] != 0x8b) bad = kMsgHeader;
                    else if (hp[2] != 8) bad = kMsgMethod;
                    else if (hp[3] & 0xe0) bad = kMsgFlags;
                    flg = hp[3];
                }
                if (!shortin && !bad && (flg & 4)) {                          // FEXTRA: two length bytes, then the field
                    if (avail < need + 2) shortin = true;
                    else { need += 2 + ((uint64_t)hp[need] | ((uint64_t)hp[need + 1] << 8)); shortin = avail < need; }
                }
                for (int f = 8; f <= 16 && !shortin && !bad; f <<= 1) {       // FNAME, FCOMMENT: zero-terminated
                    if (!(flg & f)) continue;
                    while (need < avail && hp[need] != 0) need++;
                    if (need >= avail) shortin = true; else need++;
                }
                if (!shortin && !bad && (flg & 2)) {                          // FHCRC: low 16 bits of the CRC-32 of the header so far
                    if (avail < need + 2) shortin = true;
                    else {
                        uint32_t c = 0xffffffffu;
                        for (uint64_t k = 0; k < need; k++) {
                            c ^= hp[k];
                            for (int j = 0; j < 8; j++) c = (c >> 1) ^ (kCrcPoly & (0u - (c & 1u)));
                        }
                        c = ~c;
                        if ((c & 0xffffu) != ((uint32_t)hp[need] | ((uint32_t)hp[need + 1] << 8))) bad = kMsgHcrc;
                        need += 2;
                    }
                }
                if (bad) { st->msg = bad; stop = kError; continue; }
                if (shortin) { stop = kShortIn; continue; }
                seek_bits(b, in, (h0 + need) * 8);
            } else if (wrap != ZB200_WRAP_RAW) { st->msg = kMsgHeader; stop = kError; continue; }
            mode = kModeBlock;
        } else if (mode == kModeBlock) {
            if (last) { mode = kModeTrailer; continue; }
            if (!have(b, 3)) { stop = kShortIn; continue; }
            refill(b);
            const int blast = (int)peek(b, 1); drop(b, 1);
            const uint32_t type = peek(b, 2); drop(b, 2);
            if (type == 0) {                          // stored, inflate.c:807-836
                const int pad = (int)((8 - (b.used & 7)) & 7);
                if (!have(b, pad + 32)) { b.used = mark; stop = kShortIn; continue; }
                drop(b, pad);
                refill(b);
                const uint32_t len = peek(b, 16); drop(b, 16);
                refill(b);
                const uint32_t nlen = peek(b, 16); drop(b, 16);
                if (len != (nlen ^ 0xffffu)) { st->msg = kMsgStored; stop = kError; continue; }
                st->stored_left = len;
                last = blast;
                mode = kModeStored;
            } else if (type == 1) {                   // fixed code, inflate.c:205-246
                store_lens(t, 0, 144, 8); store_lens(t, 144, 112, 9); store_lens(t, 256, 24, 7);
                store_lens(t, 280, 8, 8); store_lens(t, 288, 32, 5);
                __syncwarp();
                build_table(t->lens, 288, 1, t->lit, kLitBits, t->lit_sorted, t->lit_count, t, &t->lit_max);
                build_table(t->lens + 288, 32, 2, t->dist, kDistBits, t->dist_sorted, t->dist_count, t, &t->dist_max);
                st->nlen = 288; st->ndist = 32;
                if (streaming) { for (int i = lane; i < 320; i += 32) st->lens[i] = t->lens[i]; }
                last = blast;
                mode = kModeCodes;
            } else if (type == 2) {                   // dynamic, inflate.c:837-949
                if (!have(b, 14)) { b.used = mark; stop = kShortIn; continue; }
                refill(b);
                const int nlen = (int)peek(b, 5) + 257; drop(b, 5);
                const int ndist = (int)peek(b, 5) + 1; drop(b, 5);
                const int ncode = (int)peek(b, 4) + 4; drop(b, 4);
                if (nlen > 286 || ndist > 30) { st->msg = kMsgTooMany; stop = kError; continue; }
                if (lane < 20) t->cl_lens[lane] = 0;
                __syncwarp();
                bool shortin = false;
                for (int i = 0; i < ncode; i++) {
                    if (!have(b, 3)) { shortin = true; break; }
                    refill(b);
                    const uint32_t v = peek(b, 3); drop(b, 3);
                    if (lane == 0) t->cl_lens[c_cl_order[i]] = (uint8_t)v;
                }
                if (shortin) { b.used = mark; stop = kShortIn; continue; }
                __syncwarp();
                int cl_max;
                if (build_table(t->cl_lens, 19, 0, t->dist, kClBits, nullptr, t->dist_count, t, &t->dist_max)) {
                    st->msg = kMsgCodeLens; stop = kError; continue;
                }
                __syncwarp();
                cl_max = t->dist_max;
                const int total = nlen + ndist;
                int idx = 0, err = 0;
                uint32_t prev = 0;
                while (idx < total) {
                    refill(b);
                    uint32_t sym;
                    if (cl_max == 0) {                // empty code-length code: the reference's marker table
                        if (!have(b, 1)) { shortin = true; break; }   // yields symbol 0 for one bit
                        drop(b, 1); sym = 0;
                    } else {
                        const uint32_t e = t->dist[peek(b, kClBits)];
                        const int l = (int)ent_len(e);
                        if (!have(b, l)) { shortin = true; break; }
                        drop(b, l); sym = ent_val(e);
                    }
                    if (sym < 16) {
                        if (lane == 0) t->lens[idx] = (uint8_t)sym;
                        prev = sym; idx++;
                        continue;
                    }
                    uint32_t rep, val = 0;
                    if (sym == 16) {
                        if (!have(b, 2)) { shortin = true; break; }
                        if (idx == 0) { err = 1; break; }
                        val = prev; rep = 3 + peek(b, 2); drop(b, 2);
                    } else if (sym == 17) {
                        if (!have(b, 3)) { shortin = true; break; }
                        rep = 3 + peek(b, 3); drop(b, 3);
                    } else {
                        if (!have(b, 7)) { shortin = true; break; }
                        rep = 11 + peek(b, 7); drop(b, 7);
                    }
                    if (idx + (int)rep > total) { err = 1; break; }
                    store_lens(t, idx, (int)rep, (uint8_t)val);
                    idx += (int)rep; prev = val;
                }
                if (shortin) { b.used = mark; stop = kShortIn; continue; }
                if (err) { st->msg = kMsgRepeat; stop = kError; continue; }
                __syncwarp();
                if (build_table(t->lens, nlen, 1, t->lit, kLitBits, t->lit_sorted, t->lit_count, t, &t->lit_max)) {
                    st->msg = kMsgLitSet; stop = kError; continue;
                }
                if (build_table(t->lens + nlen, ndist, 2, t->dist, kDistBits, t->dist_sorted, t->dist_count, t, &t->dist_max)) {
                    st->msg = kMsgDistSet; stop = kError; continue;
                }
                st->nlen = nlen; st->ndist = ndist;
                if (streaming) { for (int i = lane; i < 320; i += 32) st->lens[i] = t->lens[i]; }
                last = blast;
                mode = kModeCodes;
            } else { st->msg = kMsgBlockType; stop = kError; }
        } else if (mode == kModeStored) {
            const uint64_t bytepos = b.used >> 3;
            const uint64_t ain = in_len - bytepos, aout = o.cap - o.pos;
            uint64_t c = st->stored_left;
            if (c > ain) c = ain;
            if (c > aout) c = aout;
            if (!kCount) {
                __syncwarp();
                for (uint64_t i = lane; i < c; i += 32) o.p[o.pos + i] = in[bytepos + i];
                __syncwarp();
            }
            o.pos += c; b.used += c * 8;
            st->stored_left -= (uint32_t)c;
            if (st->stored_left == 0) { seek_bits(b, in, b.used); mode = kModeBlock; }
            else stop = (c == ain) ? kShortIn : kShortOut;
        } else if (mode == kModeCodes) {
            // lean loop while both buffers have room, one careful symbol whenever it stops short (it leaves at symbol
            // boundaries with the position and the output count up to date, so a z_stream fed piecewise can use it too)
            if (decode_fast<kCount>(b, o, t, in) == kDone) { mode = kModeBlock; continue; }
            stop = decode_block<kCount>(b, o, t, st, streaming, true);
            if (stop == kDone) { stop = kRunning; mode = kModeBlock; }
            else if (stop == kShortOut && st->copy_len) mode = kModeCopy;
        } else if (mode == kModeCopy) {
            const uint32_t done = copy_match<kCount>(o, st->copy_len, st->copy_dist);
            st->copy_len -= done;
            if (st->copy_len) stop = kShortOut; else mode = kModeCodes;
        } else if (mode == kModeTrailer) {
            const int pad = (int)((8 - (b.used & 7)) & 7);
            if (wrap == ZB200_WRAP_ZLIB) {            // inflate.c:1077-1098
                if (!have(b, pad + 32)) { stop = kShortIn; continue; }
                drop(b, pad);
                uint32_t want = 0;
                for (int i = 0; i < 4; i++) { refill(b); want = (want << 8) | peek(b, 8); drop(b, 8); }
                if (!kCount) {
                    __syncwarp();
                    adler_fold(s1, s2, o.p + folded, o.pos - folded);
                    folded = o.pos;
                    if (want != ((s2 << 16) | s1)) { st->msg = kMsgCheck; stop = kError; continue; }
                }
            } else if (wrap == ZB200_WRAP_GZIP) {     // inflate.c:1099-1112; the caller checks CRC-32 and length of the output
                if (!have(b, pad + 64)) { stop = kShortIn; continue; }
                drop(b, pad);
                uint32_t w[2];
                for (int k = 0; k < 2; k++) {
                    w[k] = 0;
                    for (int i = 0; i < 4; i++) { refill(b); w[k] |= peek(b, 8) << (8 * i); drop(b, 8); }
                }
                if (lane == 0) { st->crc = w[0]; st->isize = w[1]; st->flags |= kFlagGzipTrailer; }
            } else {
                if (!have(b, pad)) { stop = kShortIn; continue; }
                drop(b, pad);
            }
            mode = kModeDone;
            stop = kDone;
        } else if (mode == kModeDict) {
            stop = kWantDict;
        } else {
            stop = mode == kModeDone ? kDone : kError;
        }
    }

    if (wrap == ZB200_WRAP_ZLIB && streaming && folded < o.pos) {
        __syncwarp();
        adler_fold(s1, s2, o.p + folded, o.pos - folded);
    }
    int32_t status;
    if (streaming) {
        status = stop == kDone ? ZB_STREAM_END : stop == kShortIn ? kNeedInput : stop == kShortOut ? kNeedOutput
               : stop == kWantDict ? ZB_NEED_DICT : ZB_DATA_ERROR;
        if (stop == kError) mode = kModeBad;
    } else {
        // uncompress() mapping, uncompr.c:53-55: out of input is a data error, out of room with input left a buffer error
        if (stop == kDone) status = ZB_OK;
        else if (stop == kShortOut && ((b.used + 7) >> 3) < in_len) status = ZB_BUF_ERROR;
        else status = ZB_DATA_ERROR;
    }
    __syncwarp();
    if (lane == 0) {
        // inflate.c:1106-1110: the length check of a gzip member (its CRC-32 would need the output); lane 0 wrote the trailer
        if (kCount && status == ZB_OK && (st->flags & kFlagGzipTrailer) && st->isize != (uint32_t)o.pos) {
            status = ZB_DATA_ERROR;
            st->msg = kMsgLength;
        }
        st->mode = mode; st->last = last; st->s1 = s1; st->s2 = s2;
        st->bit_off = (uint32_t)(b.used & 7);
        uint64_t h = st->hist + o.pos;
        st->hist = h > 32768 ? 32768 : h;
        st->total_out += o.pos;
        *out_len_p = o.pos;
        if (in_used_p) *in_used_p = stop == kDone ? ((b.used + 7) >> 3) : (b.used >> 3);
        *status_p = status;
        if (msg_p) *msg_p = st->msg;
    }
}

__global__ void __launch_bounds__(kInfWarps * 32)
k_inflate_batch(const uint8_t* __restrict__ src, const uint64_t* __restrict__ src_off, uint64_t n,
                uint8_t* __restrict__ dst, const uint64_t* __restrict__ dst_off,
                uint64_t* __restrict__ dst_len, int32_t* __restrict__ status, int wrap, uint32_t* __restrict__ expect,
                const uint32_t* __restrict__ ids, const uint64_t* __restrict__ src_end, const uint64_t* __restrict__ dst_end,
                uint64_t* __restrict__ in_used)
{
    __shared__ WarpTables s_tab[kInfWarps];
    __shared__ InfState s_state[kInfWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t k = (uint64_t)blockIdx.x * kInfWarps + warp;
    if (k >= n) return;
    // ids == nullptr: stream k is [src_off[k], src_off[k + 1]); otherwise stream ids[k], whose ranges end at src_end / dst_end
    // (members of an archive: any subset, each with its own slot)
    const uint64_t i = ids ? ids[k] : k;
    InfState* st = &s_state[warp];
    for (int k = lane; k < (int)(sizeof(InfState) / 4); k += 32) reinterpret_cast<uint32_t*>(st)[k] = 0;
    __syncwarp();
    if (lane == 0) st->wrap = wrap;
    __syncwarp();
    const uint64_t a = src_off[i], e = ids ? src_end[i] : src_off[i + 1], oa = dst_off[i], oe = ids ? dst_end[i] : dst_off[i + 1];
    inflate_warp<false>(src + a, e - a, dst + oa, oe - oa, false, st, &s_tab[warp], &dst_len[i], in_used ? &in_used[i] : nullptr, &status[i], nullptr);
    __syncwarp();
    if (expect && lane == 0) {                                  // gzip members: {crc32, isize, 1} for the check that follows
        const bool gz = (st->flags & kFlagGzipTrailer) != 0;
        expect[3 * i] = st->crc; expect[3 * i + 1] = st->isize; expect[3 * i + 2] = gz ? 1u : 0u;
    }
}

// One z_stream: a single warp continues from *st.
__global__ void __launch_bounds__(32)
k_inflate_stream(const uint8_t* __restrict__ in, uint64_t in_len, uint8_t* __restrict__ out, uint64_t out_cap,
                 InfState* __restrict__ st, InfCallResult* __restrict__ res)
{
    __shared__ WarpTables s_tab;
    inflate_warp<false>(in, in_len, out, out_cap, true, st, &s_tab, &res->out_len, &res->in_used, &res->status, &res->msg);
}

// zb200_inflate_batch_size: k_inflate_batch's warp per stream in count mode.  limit == 0: no limit.
__global__ void __launch_bounds__(kInfWarps * 32)
k_inflate_count(const uint8_t* __restrict__ src, const uint64_t* __restrict__ src_off, uint64_t n, uint64_t limit,
                uint64_t* __restrict__ out_len, uint64_t* __restrict__ src_used, int32_t* __restrict__ status, int wrap)
{
    __shared__ WarpTables s_tab[kInfWarps];
    __shared__ InfState s_state[kInfWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t i = (uint64_t)blockIdx.x * kInfWarps + warp;
    if (i >= n) return;
    InfState* st = &s_state[warp];
    for (int k = lane; k < (int)(sizeof(InfState) / 4); k += 32) reinterpret_cast<uint32_t*>(st)[k] = 0;
    __syncwarp();
    if (lane == 0) st->wrap = wrap;
    __syncwarp();
    const uint64_t a = src_off[i], e = src_off[i + 1];
    inflate_warp<true>(src + a, e - a, nullptr, limit ? limit : ~0ull, false, st, &s_tab[warp], &out_len[i],
                       src_used ? &src_used[i] : nullptr, &status[i], nullptr);
}

// off[i] = len[0] + ... + len[i - 1] for i = 0 .. n (a d_dst_off from the sizes).  One CTA, tiles of 4096 entries.
__global__ void __launch_bounds__(1024) k_size_scan(const uint64_t* __restrict__ len, uint64_t n, uint64_t* __restrict__ off)
{
    constexpr int kPer = 4;
    __shared__ uint64_t s_warp[32];
    __shared__ uint64_t s_carry;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) s_carry = 0;
    __syncthreads();
    for (uint64_t base = 0; base < n; base += 1024 * kPer) {
        uint64_t v[kPer], sum = 0;
#pragma unroll
        for (int k = 0; k < kPer; k++) {
            const uint64_t j = base + (uint64_t)t * kPer + k;
            v[k] = j < n ? len[j] : 0;
            sum += v[k];
        }
        uint64_t x = sum;                                       // inclusive scan over the warp
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint64_t y = __shfl_up_sync(kFull, x, d); if (lane >= d) x += y; }
        if (lane == 31) s_warp[w] = x;
        __syncthreads();
        if (w == 0) {
            uint64_t y = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint64_t z = __shfl_up_sync(kFull, y, d); if (lane >= d) y += z; }
            s_warp[lane] = y;
        }
        __syncthreads();
        uint64_t ex = s_carry + (w ? s_warp[w - 1] : 0) + x - sum;
#pragma unroll
        for (int k = 0; k < kPer; k++) {
            const uint64_t j = base + (uint64_t)t * kPer + k;
            if (j < n) off[j] = ex;
            ex += v[k];
        }
        __syncthreads();
        if (t == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (t == 0) off[n] = s_carry;
}

static int inflate_count_launch(const uint8_t* d_src, const uint64_t* d_src_off, size_t n, uint64_t limit, uint64_t* d_out_len,
                                uint64_t* d_src_used, int32_t* d_status, int wrap, cudaStream_t s)
{
    if (n == 0) return 0;
    ZB_LAUNCH(k_inflate_count, (unsigned)((n + kInfWarps - 1) / kInfWarps), kInfWarps * 32, 0, s, d_src, d_src_off, (uint64_t)n, limit,
              d_out_len, d_src_used, d_status, wrap);
    ZB_CHECK_LAUNCH();
    return 0;
}

// d_expect: n x 3 words of scratch, needed when wrap is gzip or auto (the CRC-32 / length check runs as a second launch)
int inflate_batch_launch(const uint8_t* d_src, const uint64_t* d_src_off, size_t n, uint8_t* d_dst,
                         const uint64_t* d_dst_off, uint64_t* d_dst_len, int32_t* d_status, int wrap, uint32_t* d_expect,
                         cudaStream_t s)
{
    if (n == 0) return 0;
    if (wrap < 0 || wrap > kWrapAuto) { set_error("inflate batch: wrap %d not supported", wrap); return ZB_STREAM_ERROR; }
    const bool gz = wrap == ZB200_WRAP_GZIP || wrap == kWrapAuto;
    if (gz && !d_expect) { set_error("inflate batch: gzip needs check scratch"); return ZB_STREAM_ERROR; }
    const unsigned blocks = (unsigned)((n + kInfWarps - 1) / kInfWarps);
    ZB_LAUNCH(k_inflate_batch, blocks, kInfWarps * 32, 0, s, d_src, d_src_off, (uint64_t)n, d_dst, d_dst_off, d_dst_len, d_status, wrap,
              gz ? d_expect : nullptr, (const uint32_t*)nullptr, (const uint64_t*)nullptr, (const uint64_t*)nullptr, (uint64_t*)nullptr);
    ZB_CHECK_LAUNCH();
    // gzip trailer (inflate.c:1099-1112): CRC-32 and length of what was produced, for every member that decoded
    if (gz) return checksum_batch_launch(d_dst, d_dst_off, d_dst_len, n, nullptr, nullptr, d_expect, d_status, s);
    return 0;
}

int inflate_members_launch(const uint8_t* d_src, const uint64_t* d_beg, const uint64_t* d_end, uint8_t* d_dst, const uint64_t* d_dst_beg,
                           const uint64_t* d_dst_end, const uint32_t* d_ids, size_t nids, uint64_t* d_dst_len, int32_t* d_status,
                           cudaStream_t s, uint64_t* d_in_used)
{
    if (nids == 0) return 0;
    ZB_LAUNCH(k_inflate_batch, (unsigned)((nids + kInfWarps - 1) / kInfWarps), kInfWarps * 32, 0, s, d_src, d_beg, (uint64_t)nids, d_dst,
              d_dst_beg, d_dst_len, d_status, (int)ZB200_WRAP_RAW, (uint32_t*)nullptr, d_ids, d_end, d_dst_end, d_in_used);
    ZB_CHECK_LAUNCH();
    return 0;
}

int inflate_stream_launch(const uint8_t* d_in, uint64_t in_len, uint8_t* d_out, uint64_t out_cap, InfState* d_state,
                          InfCallResult* d_res, cudaStream_t s)
{
    ZB_LAUNCH(k_inflate_stream, 1, 32, 0, s, d_in, in_len, d_out, out_cap, d_state, d_res);
    ZB_CHECK_LAUNCH();
    return 0;
}

// After a streaming call: keep the last 32 KiB of (history + new output) right-aligned in front of the
// output region (the reference's updatewindow, inflate.c:323-371).  One CTA; loads complete before stores.
__global__ void __launch_bounds__(1024) k_slide_history(uint8_t* arena, uint64_t hist_before, uint64_t out_len)
{
    const uint64_t valid = hist_before + out_len;
    const uint32_t keep = (uint32_t)(valid > kWindow32 ? kWindow32 : valid);
    const uint8_t* src = arena + kWindow32 + out_len - keep;
    uint8_t* dst = arena + kWindow32 - keep;
    uint8_t r[32];
    const uint32_t base = threadIdx.x * 32;
#pragma unroll
    for (int i = 0; i < 32; i++) r[i] = base + i < keep ? src[base + i] : 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 32; i++) if (base + i < keep) dst[base + i] = r[i];
}

// ------------------------------------------------------------------------------------------
// One long stream, decoded in parallel wherever it offers a byte-aligned block boundary
// ------------------------------------------------------------------------------------------
// A single DEFLATE stream is serial, and one warp decodes it at some 15 MB/s.  But streams written by this library
// end every 128 KiB chunk with an empty stored block (00 00 FF FF on a byte boundary), and so does any stream written
// with Z_SYNC_FLUSH / Z_FULL_FLUSH points (deflate.c:808-825): after such a marker a new block starts on a byte
// boundary.  Only the 32 KiB of history are missing there.  So (the scheme of two-stage parallel gzip decoders):
//   find     every 00 00 FF FF in the compressed bytes is a candidate boundary;
//   count    one warp per segment decodes from its candidate without producing output: the segment is valid if the
//            decoder arrives EXACTLY at the next candidate at the end of a block (or at the final block, for the last
//            one); this also yields every segment's output size, hence its place.  Any failure -- a pattern that was
//            data, a damaged stream -- makes the whole call fall back to the serial decoder, which reports it;
//   decode   the same decode again, now into 16-bit symbols: a byte, or 0x8000 | w for "byte w of the 32 KiB in front
//            of this segment", which is what a match reaching back over the segment start becomes (later copies
//            propagate such symbols unchanged);
//   tails    one CTA walks the segments in order and resolves the last 32 KiB of each against the 32 KiB in front of it
//            (already final by then): the only sequential part, ~64 KiB of traffic per segment;
//   rest     every other symbol of every segment resolves in parallel against the final bytes in front of its segment.
//
// The same kernels decode the segments of MANY streams in one set of launches (the members of a ZIP archive, whose lengths
// the central directory states): a segment carries a "first segment of its stream" mark, and its symbols live at sym_off
// of the scratch, which need not follow the output layout (one stream: sym_off == out_off).  sym_off == out_off mod 8.
struct SegDesc {
    uint64_t start, stop, out_off, out_len;                     // BIT range of the segment's blocks; its place in the output
    uint64_t sym_off;                                           // its 16-bit symbols in the scratch
    uint32_t flags, pad;                                        // kSegFirst / kSegLast: first / last segment of its stream
};
constexpr uint32_t kSegFirst = 1, kSegLast = 2;
struct SegResult { uint64_t out_len, end_bit; int32_t status, final; uint32_t arrive, pad; };   // status 0 = ok, 1 = missed, 2 = invalid data
constexpr uint64_t kSegMinOut = 128u << 10;                     // accepted segments are merged up to this much output (less for short streams)
constexpr size_t kParFewStreams = 8;                            // with more streams than this in a call, only the really long ones are tried
constexpr size_t kParLongStream = 32u << 20;
constexpr size_t kParMinInput = 64u << 10;                      // shorter streams are not worth the extra passes (one warp: ~15 MB/s)

__global__ void k_find_markers(const uint8_t* __restrict__ in, uint64_t first, uint64_t len, uint32_t* __restrict__ count,
                               uint64_t* __restrict__ pos, uint32_t cap)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t p = first + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p + 4 <= len; p += stride) {
        if (in[p] == 0 && in[p + 1] == 0 && in[p + 2] == 0xff && in[p + 3] == 0xff) {
            const uint32_t k = atomicAdd(count, 1u);
            if (k < cap) pos[k] = p + 4;
        }
    }
}

// Header of a dynamic block (inflate.c:837-949) into t->lens: HLIT / HDIST / HCLEN, the code-length code, the run-length
// coded lengths.  All lanes run it; false on anything the reference rejects (or on running out of input).
__device__ bool seg_read_dynamic(Bits& b, WarpTables* t, int& nlen, int& ndist)
{
    const int lane = threadIdx.x & 31;
    if (!have(b, 14)) return false;
    refill(b);
    nlen = (int)peek(b, 5) + 257; drop(b, 5);
    ndist = (int)peek(b, 5) + 1; drop(b, 5);
    const int ncode = (int)peek(b, 4) + 4; drop(b, 4);
    if (nlen > 286 || ndist > 30) return false;
    if (lane < 20) t->cl_lens[lane] = 0;
    __syncwarp();
    if (!have(b, 3 * ncode)) return false;
    for (int i = 0; i < ncode; i++) {
        refill(b);
        const uint32_t v = peek(b, 3); drop(b, 3);
        if (lane == 0) t->cl_lens[c_cl_order[i]] = (uint8_t)v;
    }
    __syncwarp();
    if (build_table(t->cl_lens, 19, 0, t->dist, kClBits, nullptr, t->dist_count, t, &t->dist_max)) return false;
    __syncwarp();
    const int cl_max = t->dist_max, total = nlen + ndist;
    int idx = 0;
    uint32_t prev = 0;
    while (idx < total) {
        refill(b);
        uint32_t s;
        if (cl_max == 0) { if (!have(b, 1)) return false; drop(b, 1); s = 0; }
        else {
            const uint32_t e = t->dist[peek(b, kClBits)];
            const int l = (int)ent_len(e);
            if (l == 0 || !have(b, l)) return false;
            drop(b, l); s = ent_val(e);
        }
        if (s < 16) { if (lane == 0) t->lens[idx] = (uint8_t)s; prev = s; idx++; continue; }
        uint32_t rep, val = 0;
        if (s == 16) { if (!have(b, 2) || idx == 0) return false; val = prev; rep = 3 + peek(b, 2); drop(b, 2); }
        else if (s == 17) { if (!have(b, 3)) return false; rep = 3 + peek(b, 3); drop(b, 3); }
        else { if (!have(b, 7)) return false; rep = 11 + peek(b, 7); drop(b, 7); }
        if (idx + (int)rep > total) return false;
        store_lens(t, idx, (int)rep, (uint8_t)val);
        idx += (int)rep; prev = val;
    }
    __syncwarp();
    return true;
}

// The lean in-bounds loop of decode_fast for a segment: same bit handling, but the output is counted (kEmit == false)
// or written as 16-bit symbols, where a source in front of the segment becomes a window symbol.  Returns true after an
// end-of-block code; otherwise the careful loop of seg_decode continues at the symbol where this one stopped.
template <bool kEmit>
__device__ bool seg_fast(Bits& b, const WarpTables* t, const uint8_t* in, uint16_t* __restrict__ out, uint64_t& produced_io,
                         uint64_t out_len, bool first_seg)
{
    const int lane = threadIdx.x & 31;
    const uint32_t nwords = b.nwords;
    const uint32_t* words = b.words;
    const uint64_t produced0 = produced_io;
    uint32_t p_lim = 0x70000000u;
    if (kEmit) {
        const uint64_t room = out_len - produced0;
        if (room < 324) return false;
        p_lim = (uint32_t)min(room - 324, (uint64_t)0x70000000u);
    }
    if (nwords < 6) return false;
    const uint32_t w_lim = nwords - 5;
    const uint64_t pos0 = (uint64_t)b.nextw * 32u - (uint64_t)b.cnt;
    const uint32_t wi0 = (uint32_t)(pos0 >> 5), off0 = (uint32_t)pos0 & 31u;
    if (wi0 > w_lim) return false;
    uint32_t wi = wi0, off = off0;
    uint32_t lo = __ldg(words + wi), hi = __ldg(words + wi + 1), nxt = __ldg(words + wi + 2);
    uint16_t* const o16 = kEmit ? out + produced0 : nullptr;
    const uint32_t* const lit = t->lit;
    const uint32_t* const dtab = t->dist;
    const uint64_t back_known = first_seg ? produced0 : produced0 + kWindow32;   // how far a distance may reach at produced == 0
    uint32_t produced = 0, end_wi, end_off;
    bool eob = false;
    for (;;) {
        if (off >= 32) {
            off -= 32; lo = hi; hi = nxt; wi++;
            nxt = __ldg(words + wi + 2);
            asm volatile("");
            if (wi > w_lim || produced > p_lim) { end_wi = wi; end_off = off; break; }
        }
        const uint32_t win = __funnelshift_r(lo, hi, off);
        const uint32_t e = lit[win & (kLitSize - 1)];
        if ((int32_t)e < 0) {
            const uint32_t e2 = lit[__funnelshift_r(win, 0u, e) & (kLitSize - 1)];
            if (kEmit) o16[produced] = (uint16_t)((e >> 16) & 0xffu);
            off += e & 31u; produced++;
            if ((int32_t)e2 < 0) { if (kEmit) o16[produced] = (uint16_t)((e2 >> 16) & 0xffu); off += e2 & 31u; produced++; }
            continue;
        }
        end_wi = wi; end_off = off;
        if (!(e & 0x8000u)) {
            if (ent_kind(e) == kEob && ent_len(e) != 0) { end_off = off + ent_len(e); eob = true; }
            break;
        }
        const uint32_t tot = (e >> 5) & 31u;
        const uint32_t mlen = (e >> 16) + __funnelshift_r(win & ((1u << tot) - 1u), 0u, e);
        off += tot;
        if (off >= 32) {
            off -= 32; lo = hi; hi = nxt; wi++;
            if (wi > w_lim) break;                              // same bound as in decode_fast: the symbol is redone by the careful loop
            nxt = __ldg(words + wi + 2);
        }
        const uint32_t dwin = __funnelshift_r(lo, hi, off);
        const uint32_t de = dtab[dwin & (kDistSize - 1)];
        const uint32_t dtot = (de >> 5) & 31u;
        const uint32_t dist = (de >> 16) + __funnelshift_r(dwin & ((1u << dtot) - 1u), 0u, de);
        if (!(de & 0x8000u) || (uint64_t)dist > back_known + produced) break;
        off += dtot;
        if (kEmit) {
            __syncwarp();
            const int64_t src0 = (int64_t)(produced0 + produced) - (int64_t)dist;      // relative to the segment start
            uint16_t* d = o16 + produced;
            if (dist >= mlen) {
                for (uint32_t i = lane; i < mlen; i += 32) {
                    const int64_t q = src0 + i;
                    d[i] = q >= 0 ? out[q] : (uint16_t)(0x8000u | (uint32_t)(q + (int64_t)kWindow32));
                }
            } else {
                for (uint32_t i = lane; i < mlen; i += 32) {
                    const int64_t q = src0 + (i % dist);
                    d[i] = q >= 0 ? out[q] : (uint16_t)(0x8000u | (uint32_t)(q + (int64_t)kWindow32));
                }
            }
            __syncwarp();
        }
        produced += mlen;
        if (produced > p_lim) { end_wi = wi; end_off = off; break; }
    }
    produced_io = produced0 + produced;
    seek_bits(b, in, b.used + ((uint64_t)(end_wi - wi0) * 32u + end_off - off0));
    return eob;
}

// kEmit == false: count only.  kEmit == true: 16-bit symbols to sym[sd.out_off ...), exactly sd.out_len of them.
// Count mode also gets the sorted list of ALL candidate positions: the decoder stops at the first one it arrives at (at the
// end of a block) and reports its index -- a candidate that is not a block boundary of the true decode is simply never
// arrived at.  Emit mode stops at sd.stop.
template <bool kEmit>
__device__ void seg_decode(const uint8_t* in, uint64_t in_len, const SegDesc sd, bool first_seg, bool last_seg,
                           uint16_t* __restrict__ sym, WarpTables* t, SegResult* res, const uint64_t* __restrict__ cand,
                           uint32_t ncand, uint32_t self)
{
    const int lane = threadIdx.x & 31;
    Bits b;
    b.total = in_len * 8;
    seek_bits(b, in, sd.start);
    uint16_t* out = kEmit ? sym + sd.sym_off : nullptr;
    uint64_t produced = 0;
    int status = 2, last = 0;
    uint32_t nx = self + 1, arrive = 0xffffffffu;
    for (;;) {
        // ---- at a block boundary ----
        if (last) { status = (kEmit && !last_seg) ? 1 : 0; break; }
        if (kEmit) {
            if (!last_seg) {
                if (b.used == sd.stop) { status = 0; break; }
                if (b.used > sd.stop) { status = 1; break; }
            }
        } else if (b.used != sd.start) {
            while (nx < ncand && cand[nx] < b.used) nx++;
            if (nx < ncand && cand[nx] == b.used) { arrive = nx; status = 0; break; }
        }
        if (!have(b, 3)) break;
        refill(b);
        last = (int)peek(b, 1); drop(b, 1);
        const uint32_t type = peek(b, 2); drop(b, 2);
        if (type == 0) {                                        // stored, inflate.c:807-836
            const int pad = (int)((8 - (b.used & 7)) & 7);
            if (!have(b, pad + 32)) break;
            drop(b, pad);
            refill(b);
            const uint32_t len = peek(b, 16); drop(b, 16);
            refill(b);
            const uint32_t nlen = peek(b, 16); drop(b, 16);
            if (len != (nlen ^ 0xffffu)) break;
            const uint64_t bytepos = b.used >> 3;
            if (bytepos + len > in_len) break;
            if (kEmit) {
                if (produced + len > sd.out_len) break;
                __syncwarp();
                for (uint32_t i = lane; i < len; i += 32) out[produced + i] = in[bytepos + i];
                __syncwarp();
            }
            produced += len;
            seek_bits(b, in, (bytepos + len) * 8);
            continue;
        }
        if (type == 3) break;
        int nlen = 288, ndist = 32;
        if (type == 1) {                                        // fixed code, inflate.c:205-246
            store_lens(t, 0, 144, 8); store_lens(t, 144, 112, 9); store_lens(t, 256, 24, 7);
            store_lens(t, 280, 8, 8); store_lens(t, 288, 32, 5);
            __syncwarp();
        } else if (!seg_read_dynamic(b, t, nlen, ndist)) break;     // dynamic, inflate.c:837-949
        if (build_table(t->lens, nlen, 1, t->lit, kLitBits, t->lit_sorted, t->lit_count, t, &t->lit_max)) break;
        if (build_table(t->lens + nlen, ndist, 2, t->dist, kDistBits, t->dist_sorted, t->dist_count, t, &t->dist_max)) break;
        // ---- symbols of the block: the lean loop while both buffers have room, one careful symbol whenever it stops ----
        bool bad = false;
        for (;;) {
            if (seg_fast<kEmit>(b, t, in, out, produced, sd.out_len, first_seg)) break;
            refill(b);
            uint32_t e = t->lit[peek(b, kLitBits)];
            const uint32_t len = ent_len(e);
            if (len != 0) { if (!have(b, (int)len)) { bad = true; break; } drop(b, (int)len); }
            else {
                const int s = slow_symbol(b, t->lit_count, t->lit_sorted, t->lit_max);
                if (s < 0) { bad = true; break; }
                e = litlen_entry((uint32_t)s, 1);
            }
            const uint32_t kind = ent_kind(e);
            if (kind == kLit) {
                if (kEmit) {
                    if (produced >= sd.out_len) { bad = true; break; }
                    if (lane == 0) out[produced] = (uint16_t)ent_val(e);
                }
                produced++;
                continue;
            }
            if (kind == kEob) break;
            if (kind == kBad) { bad = true; break; }
            const int xl = (int)ent_extra(e);
            if (!have(b, xl)) { bad = true; break; }
            const uint32_t mlen = ent_val(e) + peek(b, xl);
            drop(b, xl);
            refill(b);
            uint32_t de = t->dist[peek(b, kDistBits)];
            const uint32_t dl = ent_len(de);
            if (dl != 0) { if (!have(b, (int)dl)) { bad = true; break; } drop(b, (int)dl); }
            else {
                const int s = slow_symbol(b, t->dist_count, t->dist_sorted, t->dist_max);
                if (s < 0) { bad = true; break; }
                de = dist_entry((uint32_t)s, 1);
            }
            if (ent_kind(de) == kBad) { bad = true; break; }
            const int xd = (int)ent_extra(de);
            refill(b);
            if (!have(b, xd)) { bad = true; break; }
            const uint32_t dist = ent_val(de) + peek(b, xd);
            drop(b, xd);
            if (dist > produced && (first_seg || dist - produced > kWindow32)) { bad = true; break; }   // beyond the history
            if (kEmit) {
                if (produced + mlen > sd.out_len) { bad = true; break; }
                __syncwarp();
                const int64_t src0 = (int64_t)produced - (int64_t)dist;    // may lie in front of the segment
                for (uint32_t i = lane; i < mlen; i += 32) {
                    const int64_t q = src0 + (int64_t)(dist < mlen ? i % dist : i);
                    out[produced + i] = q >= 0 ? out[q] : (uint16_t)(0x8000u | (uint32_t)(q + (int64_t)kWindow32));
                }
                __syncwarp();
            }
            produced += mlen;
        }
        if (bad) break;
    }
    if (kEmit && produced < sd.out_len) {
        // a segment that stopped short: the symbols it did not write are plain zero bytes, not whatever an earlier call left
        // in the scratch -- the tail and rest kernels then read no window for them (the call falls back on it anyway)
        __syncwarp();
        for (uint64_t i = produced + lane; i < sd.out_len; i += 32) out[i] = 0;
    }
    if (lane == 0) { res->out_len = produced; res->end_bit = b.used; res->status = status; res->final = last; res->arrive = arrive; res->pad = 0; }
}

// Emit mode decodes segments [j_lo, j_hi) of the nseg the stream has (the one-stream decoder runs in a few phases so that
// the output of one phase travels to the host while the next is decoded); count mode takes all candidates at once.
template <bool kEmit>
__global__ void __launch_bounds__(kInfWarps * 32)
k_inflate_segments(const uint8_t* __restrict__ in, uint64_t in_len, const SegDesc* __restrict__ segs, uint32_t nseg,
                   uint16_t* __restrict__ sym, SegResult* __restrict__ res, const uint64_t* __restrict__ cand,
                   uint32_t j_lo, uint32_t j_hi)
{
    __shared__ WarpTables s_tab[kInfWarps];
    const uint32_t j = j_lo + blockIdx.x * kInfWarps + (threadIdx.x >> 5);
    if (j >= j_hi) return;
    if (kEmit) {
        const SegDesc sd = segs[j];
        seg_decode<true>(in, in_len, sd, (sd.flags & kSegFirst) != 0, (sd.flags & kSegLast) != 0, sym, &s_tab[threadIdx.x >> 5], &res[j], nullptr, 0, 0);
    }
    else seg_decode<false>(in, in_len, SegDesc{cand[j], 0, 0, 0, 0, 0, 0}, j == 0, false, nullptr, &s_tab[threadIdx.x >> 5], &res[j], cand, nseg, j);
}

// Tails in parallel.  The last 32 KiB of a segment only depend on the segment in front of it where they still hold
// window symbols -- and after 96 KiB and more of its own output a tail rarely does (a copy chain has to carry a symbol
// all the way).  So: round 0 turns every tail WITHOUT window symbols into bytes at once; round r >= 1 resolves the tails
// whose predecessor was finished in an earlier round.  done[j] = (round it was finished in) + 1.  Whatever is still open
// after the rounds (a chain of dependent tails longer than the number of rounds) is left to the sequential walk below,
// which starts at the first open segment.  One CTA per segment.
constexpr int kTailRounds = 4;

__global__ void __launch_bounds__(256)
k_tails_round(const uint16_t* __restrict__ sym, uint8_t* __restrict__ out, const SegDesc* __restrict__ segs, uint32_t j_lo,
              uint32_t* __restrict__ done, uint32_t round, uint32_t* __restrict__ err)
{
    __shared__ uint32_t s_any;
    const uint32_t j = j_lo + blockIdx.x;
    const SegDesc sd = segs[j];
    const uint64_t t = min(sd.out_len, (uint64_t)kWindow32), lo = sd.out_off + sd.out_len - t, slo = sd.sym_off + sd.out_len - t;
    if (round == 0) {
        if (threadIdx.x == 0) s_any = 0;
        __syncthreads();
        uint32_t any = 0;
        for (uint64_t i = threadIdx.x; i < t; i += 256) any |= sym[slo + i] & 0x8000u;
        if (any) s_any = 1;                                     // benign race: every writer stores 1
        __syncthreads();
        if (s_any) { if (threadIdx.x == 0) done[j] = 0; return; }
        for (uint64_t i = threadIdx.x; i < t; i += 256) out[lo + i] = (uint8_t)sym[slo + i];
        if (threadIdx.x == 0) done[j] = 1;
        return;
    }
    if (done[j] != 0) return;
    // the window must be final since an EARLIER launch; a first segment has no window (it holds no window symbols, so round 0
    // has finished it) and never waits on the segment in front of it, which belongs to another stream
    if (!(sd.flags & kSegFirst)) { const uint32_t d = done[j - 1]; if (d == 0 || d > round) return; }
    const int64_t wbase = (int64_t)sd.out_off - (int64_t)kWindow32;
    uint32_t bad = 0;
    for (uint64_t i = threadIdx.x; i < t; i += 256) {
        uint32_t v = sym[slo + i];
        if (v & 0x8000u) {
            const int64_t q = wbase + (int64_t)(v & 0x7fffu);
            if (q < 0) { bad++; v = 0; }
            else v = __ldcg(out + q);
        }
        out[lo + i] = (uint8_t)v;
    }
    if (bad) atomicAdd(err, bad);
    if (threadIdx.x == 0) done[j] = round + 1;
}

// first_open[0] = the first segment of [j_lo, j_hi) whose tail is still open, or 0xffffffff
__global__ void k_tails_first_open(const uint32_t* __restrict__ done, uint32_t j_lo, uint32_t j_hi, uint32_t* __restrict__ first_open)
{
    __shared__ uint32_t s_min;
    if (threadIdx.x == 0) s_min = 0xffffffffu;
    __syncthreads();
    uint32_t m = 0xffffffffu;
    for (uint32_t j = j_lo + threadIdx.x; j < j_hi; j += blockDim.x) if (done[j] == 0) { m = j; break; }
    if (m != 0xffffffffu) atomicMin(&s_min, m);
    __syncthreads();
    if (threadIdx.x == 0) first_open[0] = s_min;
}

// The sequential part: segment by segment, the last 32 KiB of symbols become bytes; a window symbol reads the 32 KiB in
// front of the segment, which the earlier trips of this loop (same CTA) have made final.
// One cluster of eight CTAs.  The 32 KiB in front of a segment are exactly what the previous trips resolved last, so they
// are kept on chip: a ring indexed by output position mod 32 KiB, distributed over the cluster -- CTA r owns the
// positions whose 4 KiB block number is r mod 8, resolves exactly those symbols of every tail, and serves them to the
// other CTAs through distributed shared memory.  A trip (one segment's tail) is then 4 K symbols per SM instead of 32 K
// on one (the single-CTA form was bound by that one SM's instruction issue: 7 us per trip), two cluster barriers, and no
// scattered L2 gathers; the symbols of the NEXT trip are requested before this trip's work.
// Many streams in one walk need nothing else here: the ring runs on across a stream boundary, which is safe only because a
// first segment holds no window symbols (seg_decode refuses them), so the bytes of another stream that the ring holds in
// front of it are never read; every other segment's window is the end of its own stream's previous segment, the trip
// before.  The symbols are read at sym_off, which keeps the output position's residue mod 8 (the 16-byte loads).
constexpr int kTailCtas = 8, kTailThreads = 512;
constexpr uint32_t kTailSlice = kWindow32 / kTailCtas;          // 4096 positions per CTA and trip

struct TailWork { uint64_t grp[2]; uint4 v[2]; };               // up to two groups of 8 symbols per thread and trip

__global__ void __cluster_dims__(kTailCtas, 1, 1) __launch_bounds__(kTailThreads)
k_resolve_tails(const uint16_t* __restrict__ sym, uint8_t* __restrict__ out, const SegDesc* __restrict__ segs, uint32_t j0, uint32_t nseg,
                uint32_t* __restrict__ err, const uint32_t* __restrict__ first_open, uint32_t* __restrict__ done)
{
    if (first_open) {                                           // after the parallel rounds: only what they left open (usually nothing)
        j0 = first_open[0];
        if (j0 >= nseg) return;                                 // every CTA of the cluster reads the same word and leaves together
    }
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const uint32_t r = cluster.block_rank();
    __shared__ __align__(16) uint8_t ring[kTailSlice];
    const uint8_t* rings[kTailCtas];
#pragma unroll
    for (int k = 0; k < kTailCtas; k++) rings[k] = cluster.map_shared_rank(ring, k);
    const bool out_aligned = ((uintptr_t)out & 7) == 0;
    constexpr uint64_t kNone = ~0ull;

    // this CTA's share of a tail: the 4 KiB blocks (by absolute output position) with block number = r mod 8; thread t takes
    // the t-th group of 8 positions of such a block
    auto fetch = [&](const SegDesc& d, TailWork& w) {
        const uint64_t t = min(d.out_len, (uint64_t)kWindow32), lo = d.out_off + d.out_len - t, hi = lo + t;
        w.grp[0] = w.grp[1] = kNone;
        int n = 0;
        if (t == 0) return;
        for (uint64_t m = lo >> 12; m <= (hi - 1) >> 12; m++) {
            if ((m & (kTailCtas - 1)) != r) continue;
            const uint64_t g = m * (kTailSlice / 8) + threadIdx.x;
            if (g * 8 + 8 > lo && g * 8 < hi && n < 2) {
                w.grp[n] = g;
                w.v[n] = *reinterpret_cast<const uint4*>(sym + (g * 8 - d.out_off + d.sym_off));
                n++;
            }
        }
    };
    // the ring from the 32 KiB of final output in front of a segment
    auto load_ring = [&](const SegDesc& d) {
        const uint64_t hi = d.out_off, lo = hi > kWindow32 ? hi - kWindow32 : 0;
        for (uint64_t m = lo >> 12; hi && m <= (hi - 1) >> 12; m++) {
            if ((m & (kTailCtas - 1)) != r) continue;
            for (uint64_t p = max(lo, m << 12) + threadIdx.x; p < min(hi, (m + 1) << 12); p += kTailThreads)
                ring[(uint32_t)p & (kTailSlice - 1)] = __ldcg(out + p);
        }
        cluster.sync();
    };
    TailWork cur, nxt;
    SegDesc sd = segs[j0], sn = sd;
    fetch(sd, nxt);
    bool stale = j0 > 0;                                        // a later launch of the same walk: the ring comes from the output
    uint32_t bad = 0;
    for (uint32_t j = j0; j < nseg; j++) {
        sd = sn; cur = nxt;
        if (j + 1 < nseg) { sn = segs[j + 1]; fetch(sn, nxt); }
        // A tail the parallel rounds finished is final in the output already: no trip (every CTA reads the same word, written
        // by an earlier launch), and the ring is reloaded in front of the next open one.  With many segments -- the members
        // of an archive -- one long chain of dependent tails otherwise costs a trip for every segment behind it.
        if (first_open && j > j0 && done[j] != 0) { stale = true; continue; }
        if (stale && !(sd.flags & kSegFirst)) load_ring(sd);   // a first segment has no window to load
        stale = false;
        const uint64_t t = min(sd.out_len, (uint64_t)kWindow32), lo = sd.out_off + sd.out_len - t, hi = lo + t;
        const int64_t wbase = (int64_t)sd.out_off - (int64_t)kWindow32;
        uint32_t bytes[2][8];
#pragma unroll
        for (int n = 0; n < 2; n++) {
            if (cur.grp[n] == kNone) continue;
            const uint32_t w4[4] = {cur.v[n].x, cur.v[n].y, cur.v[n].z, cur.v[n].w};
#pragma unroll
            for (int e = 0; e < 8; e++) {
                uint32_t v = (w4[e >> 1] >> (16 * (e & 1))) & 0xffffu;
                const uint64_t pos = cur.grp[n] * 8 + e;
                if ((v & 0x8000u) && pos >= lo && pos < hi) {
                    const int64_t q = wbase + (int64_t)(v & 0x7fffu);
                    if (q < 0) { bad++; v = 0; }
                    else v = rings[((uint64_t)q >> 12) & (kTailCtas - 1)][(uint32_t)q & (kTailSlice - 1)];
                }
                bytes[n][e] = v;
            }
        }
        cluster.sync();                                         // every window read of this trip is done: the ring may move on
#pragma unroll
        for (int n = 0; n < 2; n++) {
            if (cur.grp[n] == kNone) continue;
            const uint64_t p0 = cur.grp[n] * 8;
            const uint32_t w0 = bytes[n][0] | (bytes[n][1] << 8) | (bytes[n][2] << 16) | (bytes[n][3] << 24);
            const uint32_t w1 = bytes[n][4] | (bytes[n][5] << 8) | (bytes[n][6] << 16) | (bytes[n][7] << 24);
            if (p0 >= lo && p0 + 8 <= hi) {
                *reinterpret_cast<uint2*>(ring + ((uint32_t)p0 & (kTailSlice - 1))) = make_uint2(w0, w1);
                if (out_aligned) *reinterpret_cast<uint2*>(out + p0) = make_uint2(w0, w1);
                else {
#pragma unroll
                    for (int e = 0; e < 8; e++) out[p0 + e] = (uint8_t)bytes[n][e];
                }
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++)
                    if (p0 + e >= lo && p0 + e < hi) { out[p0 + e] = (uint8_t)bytes[n][e]; ring[(uint32_t)(p0 + e) & (kTailSlice - 1)] = (uint8_t)bytes[n][e]; }
            }
        }
        cluster.sync();
        if (done && r == 0 && threadIdx.x == 0) done[j] = 1;     // final since this launch: the next phase's rounds may build on it
    }
    if (bad) atomicAdd(err, bad);
}

// Everything in front of the tails, all segments at once.
__global__ void __launch_bounds__(256) k_resolve_rest(const uint16_t* __restrict__ sym, uint8_t* __restrict__ out,
                                                      const SegDesc* __restrict__ segs, uint32_t* __restrict__ err)
{
    const SegDesc sd = segs[blockIdx.x];
    const uint64_t t = min(sd.out_len, (uint64_t)kWindow32), n = sd.out_len - t;
    for (uint64_t i = threadIdx.x; i < n; i += 256) {
        const uint32_t v = sym[sd.sym_off + i];
        uint32_t byte = v;
        if (v & 0x8000u) {
            const int64_t q = (int64_t)sd.out_off - (int64_t)kWindow32 + (int64_t)(v & 0x7fffu);
            if (q < 0) { atomicAdd(err, 1u); byte = 0; }
            else byte = __ldcg(out + q);
        }
        out[sd.out_off + i] = (uint8_t)byte;
    }
}

// ---- block finder: for streams without markers (the reference's own one-shot output) ----
// Stage 1, a thread per BIT position: could a non-final dynamic block start here?  BFINAL = 0, BTYPE = 10, HLIT <= 29,
// HDIST <= 29, and the code-length code complete (Kraft sum exactly one: inftrees.c:130-138 rejects anything else).
// Stage 2, a warp per survivor: the whole header the way the decoder reads it -- both codes must build and the block
// must be able to end (a length for symbol 256).  What passes both is almost always a real block start; what is not is
// never ARRIVED AT by the counting pass and drops out there.
__global__ void k_find_blocks_probe(const uint8_t* __restrict__ in, uint64_t in_len, uint64_t first_bit, uint64_t last_bit,
                                    uint32_t* __restrict__ count, uint64_t* __restrict__ pos, uint32_t cap)
{
    const uint32_t* words = reinterpret_cast<const uint32_t*>((uintptr_t)in & ~(uintptr_t)3);
    const uint64_t skew = ((uintptr_t)in & 3) * 8;
    const uint64_t nwords = ((((uintptr_t)in + in_len + 3) & ~(uintptr_t)3) - (uintptr_t)words) >> 2;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t p = first_bit + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < last_bit; p += stride) {
        const uint64_t q = p + skew, wi = q >> 5;
        const uint32_t sh = (uint32_t)q & 31;
        if (wi + 3 >= nwords) continue;
        const uint32_t w0 = __ldg(words + wi), w1 = __ldg(words + wi + 1);
        const uint32_t lo = __funnelshift_r(w0, w1, sh);
        if ((lo & 7u) != 4u) continue;                          // BFINAL 0, BTYPE 2
        if (((lo >> 3) & 31u) > 29u || ((lo >> 8) & 31u) > 29u) continue;
        const uint32_t w2 = __ldg(words + wi + 2), w3 = __ldg(words + wi + 3);
        const uint64_t mid = ((uint64_t)__funnelshift_r(w2, w3, sh) << 32) | __funnelshift_r(w1, w2, sh);   // bits 32..95
        const int ncode = (int)((lo >> 13) & 15u) + 4;
        uint64_t bits = ((uint64_t)(lo >> 17)) | (mid << 15);   // from bit 17 on: 15 bits of lo, then mid (64 - 15 = 49 more)
        uint32_t kraft = 0;
        // 3 * 19 = 57 bits <= 64 available
#pragma unroll
        for (int i = 0; i < 19; i++) {
            const uint32_t l = (uint32_t)(bits >> (3 * i)) & 7u;
            if (i < ncode && l) kraft += 128u >> l;
        }
        if (kraft != 128u) continue;
        const uint32_t k = atomicAdd(count, 1u);
        if (k < cap) pos[k] = p;
    }
}

__global__ void __launch_bounds__(kInfWarps * 32)
k_find_blocks_check(const uint8_t* __restrict__ in, uint64_t in_len, const uint64_t* __restrict__ probe, uint32_t nprobe,
                    uint32_t* __restrict__ count, uint64_t* __restrict__ pos, uint32_t cap)
{
    __shared__ WarpTables s_tab[kInfWarps];
    const uint32_t j = blockIdx.x * kInfWarps + (threadIdx.x >> 5);
    if (j >= nprobe) return;
    WarpTables* t = &s_tab[threadIdx.x >> 5];
    Bits b;
    b.total = in_len * 8;
    seek_bits(b, in, probe[j]);
    refill(b);
    drop(b, 3);
    int nlen = 0, ndist = 0;
    if (!seg_read_dynamic(b, t, nlen, ndist)) return;
    if (t->lens[256] == 0) return;                              // no end-of-block code: not a block a compressor wrote
    if (build_table(t->lens, nlen, 1, t->lit, kLitBits, t->lit_sorted, t->lit_count, t, &t->lit_max)) return;
    if (build_table(t->lens + nlen, ndist, 2, t->dist, kDistBits, t->dist_sorted, t->dist_count, t, &t->dist_max)) return;
    if ((threadIdx.x & 31) == 0) {
        const uint32_t k = atomicAdd(count, 1u);
        if (k < cap) pos[k] = probe[j];
    }
}

// Segments [j0, j1) of a list: emit (16-bit symbols), tails (parallel rounds, then the sequential walk for what they left
// open), rest.  One stream or many: the launch shape does not depend on it, but for the number of tail rounds.
static int launch_segment_phase(const uint8_t* d_src, uint64_t len, uint8_t* d_dst, const SegDesc* d_segs, uint32_t nseg,
                                uint16_t* d_sym, SegResult* d_res, uint32_t* d_done, uint32_t* d_err, uint32_t* d_first_open,
                                uint32_t j0, uint32_t j1, cudaStream_t s, int rounds = kTailRounds)
{
    ZB_LAUNCH((k_inflate_segments<true>), (j1 - j0 + kInfWarps - 1) / kInfWarps, kInfWarps * 32, 0, s, d_src, len, d_segs, nseg, d_sym, d_res,
              (const uint64_t*)nullptr, j0, j1);
    for (int r = 0; r < rounds; r++)
        ZB_LAUNCH(k_tails_round, j1 - j0, 256, 0, s, d_sym, d_dst, d_segs, j0, d_done, (uint32_t)r, d_err);
    ZB_LAUNCH(k_tails_first_open, 1, 1024, 0, s, d_done, j0, j1, d_first_open);
    ZB_LAUNCH(k_resolve_tails, kTailCtas, kTailThreads, 0, s, d_sym, d_dst, d_segs, j0, j1, d_err, d_first_open, d_done);
    ZB_LAUNCH(k_resolve_rest, j1 - j0, 256, 0, s, d_sym, d_dst, d_segs + j0, d_err);
    ZB_CHECK_LAUNCH();
    return 0;
}

// Second half of the one-stream decoder: emit (16-bit symbols), tails, rest, trailer check -- for a list of segments whose
// sizes are known (counted) or assumed (speculative: every segment but the last is exactly out_len bytes, the last one at
// most out_len; used for streams that look like this library's own, see inflate_single_parallel).  In speculative mode
// `final_end` and the total are learnt from the last segment.  Returns 0 = decoded, 1 = not taken, negative = CUDA error.
static int emit_segments(Ctx* c, const uint8_t* d_src, uint64_t len, uint8_t* d_dst, std::vector<SegDesc> segs, uint64_t total,
                         uint64_t final_end, bool speculative, int wrap, cudaStream_t s, void* h_dst, uint64_t* total_out,
                         uint64_t* used_out, uint32_t* check_out)
{
    const uint32_t nseg = (uint32_t)segs.size();
    for (uint32_t j = 0; j < nseg; j++) {                       // one stream: symbols laid out like the output
        segs[j].sym_off = segs[j].out_off;
        segs[j].flags = (j == 0 ? kSegFirst : 0u) | (j == nseg - 1 ? kSegLast : 0u);
    }
    const uint64_t sym_len = segs.back().out_off + segs.back().out_len;
    const uint64_t trailer_len = wrap == ZB200_WRAP_ZLIB ? 4 : wrap == ZB200_WRAP_GZIP ? 8 : 0;
    int rc;
    if ((rc = c->small.ensure(256)) != 0) return rc;
    if ((rc = c->ws[2].ensure((size_t)nseg * sizeof(SegDesc))) != 0) return rc;
    if ((rc = c->ws[3].ensure((size_t)nseg * sizeof(SegResult))) != 0) return rc;
    if ((rc = c->ws[4].ensure((size_t)sym_len * 2 + 64)) != 0) return rc;
    if ((rc = c->ws[6].ensure((size_t)nseg * 4 + 64)) != 0) return rc;
    uint32_t* d_err = c->small.as<uint32_t>() + 17;
    uint32_t* d_first_open = c->small.as<uint32_t>() + 18;
    SegDesc* d_segs = c->ws[2].as<SegDesc>();
    SegResult* d_res = c->ws[3].as<SegResult>();
    uint16_t* d_sym = c->ws[4].as<uint16_t>();
    uint32_t* d_done = c->ws[6].as<uint32_t>();
    ZB_CUDA(cudaMemsetAsync(d_err, 0, 4, s));
    ZB_CUDA(cudaMemcpyAsync(d_segs, segs.data(), (size_t)nseg * sizeof(SegDesc), cudaMemcpyHostToDevice, s));
    // A few phases, each a contiguous range of segments: emit, tails (parallel rounds, then the sequential walk for what they
    // left open), rest -- and, with a pinned host destination, the phase's output on its way while the next phase is decoded.
    const uint32_t nphase = (h_dst && nseg >= 4096) ? 2 : 1;
    if (h_dst && (rc = c->ensure_aux(nphase + 2)) != 0) return rc;
    for (uint32_t k = 0; k < nphase; k++) {
        const uint32_t j0 = (uint32_t)((uint64_t)nseg * k / nphase), j1 = (uint32_t)((uint64_t)nseg * (k + 1) / nphase);
        if (j1 == j0) continue;
        if ((rc = launch_segment_phase(d_src, len, d_dst, d_segs, nseg, d_sym, d_res, d_done, d_err, d_first_open, j0, j1, s)) != 0) return rc;
        if (h_dst && !(speculative && k == nphase - 1)) {       // (the last speculative phase is copied once its true length is known)
            const uint64_t a = segs[j0].out_off, b = segs[j1 - 1].out_off + segs[j1 - 1].out_len;
            ZB_CUDA(cudaEventRecord(c->evs[k], s));
            ZB_CUDA(cudaStreamWaitEvent(c->aux[1], c->evs[k], 0));
            if (b > a) ZB_CUDA(cudaMemcpyAsync((uint8_t*)h_dst + a, d_dst + a, b - a, cudaMemcpyDeviceToHost, c->aux[1]));
        }
    }
    ZB_CHECK_LAUNCH();
    std::vector<SegResult> res(nseg);
    uint32_t nerr = 0;
    ZB_CUDA(cudaMemcpyAsync(res.data(), d_res, (size_t)nseg * sizeof(SegResult), cudaMemcpyDeviceToHost, s));
    ZB_CUDA(cudaMemcpyAsync(&nerr, d_err, 4, cudaMemcpyDeviceToHost, s));
    ZB_CUDA(cudaStreamSynchronize(s));
    bool ok = nerr == 0;
    for (uint32_t j = 0; j < nseg && ok; j++) {
        if (res[j].status != 0) ok = false;
        else if (speculative && j == nseg - 1) ok = res[j].final != 0 && res[j].out_len <= segs[j].out_len;
        else ok = res[j].out_len == segs[j].out_len;
    }
    if (ok && speculative) {
        total = segs.back().out_off + res[nseg - 1].out_len;
        final_end = res[nseg - 1].end_bit;
        if (h_dst) {                                            // the last phase, now that its length is known
            const uint32_t j0 = (uint32_t)((uint64_t)nseg * (nphase - 1) / nphase);
            const uint64_t a = segs[j0].out_off;
            if (total > a) ZB_CUDA(cudaMemcpyAsync((uint8_t*)h_dst + a, d_dst + a, total - a, cudaMemcpyDeviceToHost, c->aux[1]));
        }
    }
    const uint64_t trailer_at = (final_end + 7) >> 3;
    if (ok && trailer_at + trailer_len > len) ok = false;
    uint32_t sums[2] = {0, 1};
    uint8_t tr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (ok && trailer_len) {
        if ((rc = checksum_launch(c, d_dst, (size_t)total, c->small.as<uint32_t>(), s)) != 0) { if (h_dst) cudaStreamSynchronize(c->aux[1]); return rc; }
        ZB_CUDA(cudaMemcpyAsync(sums, c->small.p, 8, cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaMemcpyAsync(tr, d_src + trailer_at, trailer_len, cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaStreamSynchronize(s));
        if (wrap == ZB200_WRAP_ZLIB) {                          // inflate.c:1077-1098
            const uint32_t want = ((uint32_t)tr[0] << 24) | ((uint32_t)tr[1] << 16) | ((uint32_t)tr[2] << 8) | tr[3];
            if (want != sums[1]) ok = false;                    // let the serial decoder find and name the damage
        } else if (wrap == ZB200_WRAP_GZIP) {                   // inflate.c:1099-1112: CRC-32, then the length mod 2^32
            const uint32_t want = (uint32_t)tr[0] | ((uint32_t)tr[1] << 8) | ((uint32_t)tr[2] << 16) | ((uint32_t)tr[3] << 24);
            const uint32_t isize = (uint32_t)tr[4] | ((uint32_t)tr[5] << 8) | ((uint32_t)tr[6] << 16) | ((uint32_t)tr[7] << 24);
            if (want != sums[0] || isize != (uint32_t)total) ok = false;
        }
    }
    if (h_dst) ZB_CUDA(cudaStreamSynchronize(c->aux[1]));
    if (!ok) return 1;
    *total_out = total;
    *used_out = trailer_at + trailer_len;
    *check_out = wrap == ZB200_WRAP_GZIP ? sums[0] : sums[1];   // what strm->adler holds at the end: CRC-32 for gzip
    return 0;
}

// Returns 0 when the stream was decoded here (*status, *out_len set), 1 when the caller should use the serial decoder
// (no usable boundaries, output that does not fit, damaged data), negative on CUDA errors.
int inflate_single_parallel(Ctx* c, const uint8_t* d_src, uint64_t len, uint8_t* d_dst, uint64_t cap, int wrap,
                            uint64_t* out_len, int32_t* status, cudaStream_t s, uint64_t* in_used, uint32_t* adler,
                            int* wrap_found, void* h_dst, uint64_t* need, bool count_only)
{
    if (len < kParMinInput || wrap < 0 || wrap > kWrapAuto) return 1;
    uint64_t hdr = 0;
    if (wrap != ZB200_WRAP_RAW) {
        // the wrapper's header is read on the host; anything unusual about it goes the serial way, which names the problem
        uint8_t hb[4096];
        const size_t hn = (size_t)std::min<uint64_t>(len, sizeof(hb));
        ZB_CUDA(cudaMemcpyAsync(hb, d_src, hn, cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaStreamSynchronize(s));
        if (wrap == kWrapAuto) wrap = (hb[0] == 0x1f && hb[1] == 0x8b) ? ZB200_WRAP_GZIP : ZB200_WRAP_ZLIB;   // inflate.c:596
        if (wrap == ZB200_WRAP_ZLIB) {                          // inflate.c:589-632; a preset dictionary goes the serial way
            if (((hb[0] << 8) + hb[1]) % 31 || (hb[0] & 15) != 8 || (hb[0] >> 4) + 8 > 15 || (hb[1] & 0x20)) return 1;
            hdr = 2;
        } else {                                                // gzip, inflate.c:634-759
            if (hb[0] != 0x1f || hb[1] != 0x8b || hb[2] != 8 || (hb[3] & 0xe0)) return 1;
            const unsigned flg = hb[3];
            size_t need = 10;
            if (flg & 4) { if (need + 2 > hn) return 1; need += 2 + ((size_t)hb[need] | ((size_t)hb[need + 1] << 8)); }
            for (unsigned f = 8; f <= 16; f <<= 1) {
                if (!(flg & f)) continue;
                while (need < hn && hb[need] != 0) need++;
                need++;
            }
            if (flg & 2) need += 2;                             // FHCRC: left unchecked here; a mismatch there is the serial decoder's to report
            if (need + 64 > hn || (flg & 2)) return 1;
            hdr = need;
        }
    }
    const uint32_t cand_cap = (uint32_t)std::min<uint64_t>(len / 32 + 4096, 1u << 26);
    int rc;
    if ((rc = c->small.ensure(256)) != 0) return rc;
    if ((rc = c->ws[1].ensure((size_t)cand_cap * 8 + 64)) != 0) return rc;
    if ((rc = c->ws[5].ensure((size_t)cand_cap * 8 + 64)) != 0) return rc;
    uint32_t* d_count = c->small.as<uint32_t>() + 16;
    uint32_t* d_err = d_count + 1;
    uint64_t* d_pos = c->ws[1].as<uint64_t>();
    uint64_t* d_probe = c->ws[5].as<uint64_t>();
    std::vector<uint64_t> cand;
    std::vector<SegResult> res;
    std::vector<SegDesc> segs;
    uint64_t total = 0, final_end = 0;
    // enough segments to fill the GPU with warps, not more than the sequential tail pass likes (3 us per segment)
    const uint64_t seg_min = std::min<uint64_t>(kSegMinOut, std::max<uint64_t>(32768, len * 2 / 4096));
    // Two sources of candidates, the cheap one first: sync markers (bytes), then block headers (bits).
    for (int source = 0; source < 2 && segs.empty(); source++) {
        uint32_t ncand = 0;
        ZB_CUDA(cudaMemsetAsync(d_count, 0, 8, s));
        if (source == 0) {
            ZB_LAUNCH(k_find_markers, device_sms() * 8, 256, 0, s, d_src, hdr, len, d_count, d_pos, cand_cap);
        } else {
            uint32_t nprobe = 0;
            ZB_LAUNCH(k_find_blocks_probe, device_sms() * 16, 256, 0, s, d_src, len, hdr * 8 + 1, len * 8, d_count, d_probe, cand_cap);
            ZB_CUDA(cudaMemcpyAsync(&nprobe, d_count, 4, cudaMemcpyDeviceToHost, s));
            ZB_CUDA(cudaStreamSynchronize(s));
            if (nprobe == 0 || nprobe > cand_cap) return 1;
            ZB_CUDA(cudaMemsetAsync(d_count, 0, 8, s));
            ZB_LAUNCH(k_find_blocks_check, (nprobe + kInfWarps - 1) / kInfWarps, kInfWarps * 32, 0, s, d_src, len, d_probe, nprobe, d_count,
                      d_pos, cand_cap);
        }
        ZB_CUDA(cudaMemcpyAsync(&ncand, d_count, 4, cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaStreamSynchronize(s));
        if (ncand == 0 || ncand > cand_cap) continue;
        cand.assign((size_t)ncand + 1, 0);
        ZB_CUDA(cudaMemcpyAsync(cand.data() + 1, d_pos, (size_t)ncand * 8, cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaStreamSynchronize(s));
        if (source == 0) for (size_t k = 1; k < cand.size(); k++) cand[k] *= 8;       // marker positions are bytes
        cand[0] = hdr * 8;                                      // the stream's first block: the one certain boundary
        std::sort(cand.begin() + 1, cand.end());
        cand.erase(std::unique(cand.begin(), cand.end()), cand.end());
        while (!cand.empty() && cand.back() + 64 > len * 8) cand.pop_back();
        const uint32_t nc = (uint32_t)cand.size();
        if (nc < 2) continue;
        // ---- streams of this library end every ZB200_CHUNK bytes of input with a marker: assume exactly that (segment j
        // holds bytes [j, j + 1) * ZB200_CHUNK of the output) and go straight to the emit pass, which checks every
        // segment's length and arrival; if the assumption fails anywhere, the counting pass below takes over.  (Sizing
        // skips this: the assumption is only checked by decoding) ----
        if (!count_only && source == 0 && (uint64_t)(nc - 1) * ZB200_CHUNK < cap) {
            std::vector<SegDesc> guess(nc);
            for (uint32_t j = 0; j < nc; j++)
                guess[j] = SegDesc{cand[j], j + 1 < nc ? cand[j + 1] : 0, (uint64_t)j * ZB200_CHUNK,
                                   j + 1 < nc ? (uint64_t)ZB200_CHUNK : std::min<uint64_t>(ZB200_CHUNK, cap - (uint64_t)j * ZB200_CHUNK)};
            uint64_t g_total = 0, g_used = 0;
            uint32_t g_check = 1;
            rc = emit_segments(c, d_src, len, d_dst, guess, 0, 0, true, wrap, s, h_dst, &g_total, &g_used, &g_check);
            if (rc < 0) return rc;
            if (rc == 0) {
                *out_len = g_total;
                *status = ZB_OK;
                if (in_used) *in_used = g_used;
                if (adler) *adler = g_check;
                if (wrap_found) *wrap_found = wrap;
                return 0;
            }
        }
        // ---- count: every candidate decodes to the first candidate it arrives at ----
        if ((rc = c->ws[3].ensure((size_t)nc * sizeof(SegResult))) != 0) return rc;
        SegResult* d_res = c->ws[3].as<SegResult>();
        ZB_CUDA(cudaMemcpyAsync(d_pos, cand.data(), (size_t)nc * 8, cudaMemcpyHostToDevice, s));
        ZB_LAUNCH((k_inflate_segments<false>), (nc + kInfWarps - 1) / kInfWarps, kInfWarps * 32, 0, s, d_src, len, (const SegDesc*)nullptr, nc,
                  (uint16_t*)nullptr, d_res, d_pos, 0u, nc);
        res.resize(nc);
        ZB_CUDA(cudaMemcpyAsync(res.data(), d_res, (size_t)nc * sizeof(SegResult), cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaStreamSynchronize(s));
        // ---- the true decode's path through the candidates; short hops merge ----
        bool ok = true;
        uint64_t seg_out = 0, seg_start = cand[0];
        total = 0;
        for (uint32_t j = 0;;) {
            const SegResult& r = res[j];
            if (r.status != 0) { ok = false; break; }
            seg_out += r.out_len;
            if (r.final) { segs.push_back(SegDesc{seg_start, r.end_bit, total, seg_out}); total += seg_out; final_end = r.end_bit; break; }
            if (r.arrive <= j || r.arrive >= nc) { ok = false; break; }
            if (seg_out >= seg_min) {
                segs.push_back(SegDesc{seg_start, cand[r.arrive], total, seg_out});
                total += seg_out; seg_out = 0; seg_start = cand[r.arrive];
            }
            // the counting pass lets a segment reach 32 KiB in front of it; where less than that lies in front, only the
            // emit pass (or the serial decoder) can tell "too far back", so sizing leaves such a stream to the count kernel
            if (count_only && total + seg_out < kWindow32) { ok = false; break; }
            j = r.arrive;
        }
        if (!ok) return 1;                                      // damage on the true path: the serial decoder names it
        if (segs.size() < 2) segs.clear();                      // nothing gained; try the other source
    }
    if (segs.empty()) return 1;
    if (total > cap) {                                          // the serial decoder reports Z_BUF_ERROR the reference's way
        if (need) *need = total;
        return 1;
    }
    if (count_only) {
        // the stream ends at the final block's end and its trailer; a trailer cut short, or a gzip ISIZE that differs from
        // the count (inflate.c:1106-1110), is declined: the count kernel names it
        const uint64_t trailer_len = wrap == ZB200_WRAP_ZLIB ? 4 : wrap == ZB200_WRAP_GZIP ? 8 : 0, trailer_at = (final_end + 7) >> 3;
        if (trailer_at + trailer_len > len) return 1;
        if (wrap == ZB200_WRAP_GZIP) {
            uint8_t tr[8];
            ZB_CUDA(cudaMemcpyAsync(tr, d_src + trailer_at, 8, cudaMemcpyDeviceToHost, s));
            ZB_CUDA(cudaStreamSynchronize(s));
            const uint32_t isize = (uint32_t)tr[4] | ((uint32_t)tr[5] << 8) | ((uint32_t)tr[6] << 16) | ((uint32_t)tr[7] << 24);
            if (isize != (uint32_t)total) return 1;
        }
        *out_len = total;
        *status = ZB_OK;
        if (in_used) *in_used = trailer_at + trailer_len;
        if (wrap_found) *wrap_found = wrap;
        return 0;
    }
    uint64_t used = 0;
    uint32_t check = 1;
    rc = emit_segments(c, d_src, len, d_dst, segs, total, final_end, false, wrap, s, h_dst, &total, &used, &check);
    if (rc) return rc;
    *out_len = total;
    *status = ZB_OK;
    if (in_used) *in_used = used;
    if (adler) *adler = check;
    if (wrap_found) *wrap_found = wrap;
    return 0;
}

// ---- many raw streams of known output length in one segment decode (the large members of a ZIP archive) ----
// A ZIP central directory states every member's uncompressed length, and a member this library wrote ends each ZB200_CHUNK
// bytes of its input with a marker.  So a stream with exactly ceil(out_len / ZB200_CHUNK) - 1 markers has its segments
// planned before anything is decoded -- segment j is output [j, j + 1) * ZB200_CHUNK, starting behind marker j - 1 -- and
// no counting pass is needed: the non-speculative form of emit_segments, for all such streams at once.  The emit pass checks
// every segment's length and arrival; a stream that misses either (a marker pattern that was data stands in for a real one)
// leaves the plan with ok[i] = 0 and its output undefined, for the caller to decode another way.  Streams are taken in groups
// of about kPlanGroupBytes of output, which bounds the symbol scratch (2 bytes per output byte).
// Tails: a chain of dependent tails runs through a stream, and each round of k_tails_round finishes one more link of it in
// EVERY stream at once, where the sequential walk would take the chains of all streams one after the other (text: most
// tails hold window symbols, so the chain is most of a member; 2280 long members of the config-5 archive took 92 ms in the
// walk with four rounds).  So the plan runs as many rounds as its longest stream has segments, up to kPlanTailRounds.
constexpr uint64_t kPlanGroupBytes = 1ull << 30;
constexpr uint32_t kPlanTailRounds = 64;

int find_markers_launch(const uint8_t* d_src, uint64_t first, uint64_t last, uint32_t* d_count, uint64_t* d_pos, uint32_t cap, cudaStream_t s)
{
    ZB_LAUNCH(k_find_markers, device_sms() * 8, 256, 0, s, d_src, first, last, d_count, d_pos, cap);
    ZB_CHECK_LAUNCH();
    return 0;
}

int inflate_planned(Ctx* c, const uint8_t* d_src, uint64_t src_len, uint8_t* d_dst, const PlannedStream* ps, size_t np,
                    const uint64_t* marks, uint8_t* ok, cudaStream_t s, bool exact_end)
{
    int rc;
    if ((rc = c->small.ensure(256)) != 0) return rc;
    uint32_t* d_err = c->small.as<uint32_t>() + 17;
    uint32_t* d_first_open = c->small.as<uint32_t>() + 18;
    std::vector<SegDesc> segs;
    std::vector<SegResult> res;
    std::vector<uint32_t> seg0;                                 // first segment of each stream of the group
    for (size_t g0 = 0; g0 < np;) {
        size_t g1 = g0;
        uint64_t out = 0;
        while (g1 < np && (g1 == g0 || out + ps[g1].out_len <= kPlanGroupBytes)) out += ps[g1++].out_len;
        segs.clear(); seg0.clear();
        uint64_t sym = 16;                                      // k_resolve_tails reads whole groups of 8 around a segment's ends
        for (size_t i = g0; i < g1; i++) {
            const PlannedStream& p = ps[i];
            sym += (p.out_off - sym) & 7;                       // the scratch keeps the output's residue mod 8
            seg0.push_back((uint32_t)segs.size());
            const uint32_t nseg = p.nmarks + 1;
            for (uint32_t j = 0; j < nseg; j++) {
                SegDesc d;
                d.start = 8 * (j == 0 ? p.in_beg : marks[p.first_mark + j - 1]);
                d.stop = j + 1 < nseg ? 8 * marks[p.first_mark + j] : 0;
                d.out_off = p.out_off + (uint64_t)j * ZB200_CHUNK;
                d.out_len = std::min<uint64_t>(ZB200_CHUNK, p.out_len - (uint64_t)j * ZB200_CHUNK);
                d.sym_off = sym + (uint64_t)j * ZB200_CHUNK;
                d.flags = (j == 0 ? kSegFirst : 0u) | (j + 1 == nseg ? kSegLast : 0u);
                d.pad = 0;
                segs.push_back(d);
            }
            sym += p.out_len + 8;
        }
        seg0.push_back((uint32_t)segs.size());
        const uint32_t nseg = (uint32_t)segs.size();
        uint32_t longest = 0;
        for (size_t i = g0; i < g1; i++) longest = std::max(longest, ps[i].nmarks + 1);
        const int rounds = (int)std::min(kPlanTailRounds, std::max<uint32_t>(longest, kTailRounds));
        if ((rc = c->ws[2].ensure((size_t)nseg * sizeof(SegDesc))) != 0) return rc;
        if ((rc = c->ws[3].ensure((size_t)nseg * sizeof(SegResult))) != 0) return rc;
        if ((rc = c->ws[4].ensure((size_t)sym * 2 + 64)) != 0) return rc;
        if ((rc = c->ws[6].ensure((size_t)nseg * 4 + 64)) != 0) return rc;
        SegDesc* d_segs = c->ws[2].as<SegDesc>();
        SegResult* d_res = c->ws[3].as<SegResult>();
        ZB_CUDA(cudaMemsetAsync(d_err, 0, 4, s));
        ZB_CUDA(cudaMemcpyAsync(d_segs, segs.data(), (size_t)nseg * sizeof(SegDesc), cudaMemcpyHostToDevice, s));
        if ((rc = launch_segment_phase(d_src, src_len, d_dst, d_segs, nseg, c->ws[4].as<uint16_t>(), d_res, c->ws[6].as<uint32_t>(), d_err,
                                       d_first_open, 0, nseg, s, rounds)) != 0) return rc;
        res.resize(nseg);
        ZB_CUDA(cudaMemcpyAsync(res.data(), d_res, (size_t)nseg * sizeof(SegResult), cudaMemcpyDeviceToHost, s));
        ZB_CUDA(cudaStreamSynchronize(s));
        // The window-error count of the tail and rest kernels is not consulted, and each stream is judged by its own
        // segments: a stream whose segments all pass holds no window symbol in its first segment (seg_decode refuses them
        // there) and starts every other segment ZB200_CHUNK or more into its own output, so none of its window references
        // reaches in front of that output; a segment that failed wrote zeros where it stopped (seg_decode), so one damaged
        // or foreign member neither reads outside its slot nor takes the other members of its group off the plan.
        for (size_t i = g0; i < g1; i++) {
            bool good = true;
            for (uint32_t j = seg0[i - g0]; j < seg0[i - g0 + 1] && good; j++) {
                const SegResult& r = res[j];
                good = r.status == 0 && r.out_len == segs[j].out_len;
                if (good && (segs[j].flags & kSegLast))
                    good = r.final != 0 && (exact_end ? (r.end_bit + 7) / 8 == ps[i].in_end : r.end_bit <= 8 * ps[i].in_end);
            }
            ok[i] = good ? 1 : 0;
        }
        g0 = g1;
    }
    return 0;
}

}  // namespace zb

using namespace zb;

// inflate(strm, Z_FINISH) with the whole stream and the whole output buffer in one call -- what uncompress() is in the
// reference (uncompr.c:26-61) -- may take the segment-parallel decoder.  0 = decoded, 1 = use the streaming decoder.
extern "C" int zb200i_inflate_try_parallel(const uint8_t* in, size_t in_len, uint8_t* out, size_t cap, int wrap,
                                           size_t* in_used, size_t* out_len, uint32_t* check)
{
    if (ensure_init() != 0 || in_len < kParMinInput) return 1;
    Ctx* c = ctx_acquire_own();
    if (!c) return 1;
    cudaStream_t s = c->own_stream;
    int r = 1;
    do {
        if (c->in.ensure(in_len + 64) != 0 || c->out.ensure(cap + 16) != 0) break;
        if (cudaMemcpyAsync(c->in.p, in, in_len, cudaMemcpyHostToDevice, s) != cudaSuccess) { cudaGetLastError(); break; }
        uint64_t got = 0, used = 0;
        int32_t st = 0;
        uint32_t adl = 1;
        r = inflate_single_parallel(c, c->in.as<uint8_t>(), in_len, c->out.as<uint8_t>(), cap, wrap, &got, &st, s, &used, &adl);
        if (r != 0) { cudaStreamSynchronize(s); r = 1; break; }
        if (got && cudaMemcpyAsync(out, c->out.p, got, cudaMemcpyDeviceToHost, s) != cudaSuccess) { cudaGetLastError(); r = 1; break; }
        if (cudaStreamSynchronize(s) != cudaSuccess) { cudaGetLastError(); r = 1; break; }
        *in_used = (size_t)used; *out_len = (size_t)got; *check = adl;
    } while (0);
    ctx_release(c, s);
    return r;
}

// ---- one resumable stream behind zlib.h's inflate() ----
struct zb200i_inflater {
    int wrap = 1, wbits = 0;
    InfState* d_state = nullptr;
    InfCallResult* d_res = nullptr;
    uint8_t* d_arena = nullptr;                  // [32 KiB history][output window]
    size_t out_window = 0;
    uint8_t* d_in = nullptr; size_t d_in_cap = 0;
    uint8_t* h_pin = nullptr; size_t h_pin_cap = 0;
    std::vector<uint8_t> carry;                  // input the decoder has been handed but could not finish
    cudaStream_t s = nullptr;
    uint64_t hist = 0;
    int mode = kModeHead;
    uint32_t check = 1;
    uint32_t crc = 0;                            // gzip: running CRC-32 and length of everything produced
    uint64_t produced = 0;
};

extern "C" unsigned long crc32_combine(unsigned long crc1, unsigned long crc2, long len2);   // zapi_checksum.c

static const char* const kInfMsgs[] = {
    nullptr, "incorrect header check", "unknown compression method", "invalid window size", "need dictionary",
    "invalid block type", "invalid stored block lengths", "too many length or distance symbols",
    "invalid code lengths set", "invalid bit length repeat", "invalid literal/lengths set", "invalid distances set",
    "invalid literal/length code", "invalid distance code", "invalid distance too far back", "incorrect data check",
    "incorrect length check", "unknown header flags set", "header crc mismatch"};

extern "C" const char* zb200i_inflate_msg(int msg)
{
    return (msg > 0 && msg < (int)(sizeof(kInfMsgs) / sizeof(kInfMsgs[0]))) ? kInfMsgs[msg] : nullptr;
}

static int inflater_write_state(zb200i_inflater* h, int wrap)
{
    InfState st;
    memset(&st, 0, sizeof(st));
    const int wbits = (wrap >> 8) & 15;                          // 0 = 15 (inflateInit2's windowBits, inflate.c:622)
    wrap &= 0xff;
    st.wrap = wrap; st.mode = kModeHead; st.s1 = 1;
    st.flags = (uint32_t)wbits << 8;
    ZB_CUDA(cudaMemcpyAsync(h->d_state, &st, sizeof(st), cudaMemcpyHostToDevice, h->s));
    ZB_CUDA(cudaStreamSynchronize(h->s));
    h->wrap = wrap; h->wbits = wbits; h->hist = 0; h->mode = kModeHead; h->check = wrap >= ZB200_WRAP_GZIP ? 0u : 1u; h->carry.clear();
    h->crc = 0; h->produced = 0;
    return 0;
}

extern "C" int zb200i_inflate_open(zb200i_inflater** out, int wrap)
{
    int rc = ensure_init();
    if (rc) return rc;
    zb200i_inflater* h = new zb200i_inflater();
    h->out_window = 1u << 20;
    bool ok = cudaStreamCreateWithFlags(&h->s, cudaStreamNonBlocking) == cudaSuccess &&
              cudaMalloc(&h->d_state, sizeof(InfState)) == cudaSuccess &&
              cudaMalloc(&h->d_res, sizeof(InfCallResult)) == cudaSuccess &&
              cudaMalloc(&h->d_arena, kWindow32 + h->out_window + 64) == cudaSuccess;
    if (!ok) { cudaGetLastError(); zb200i_inflate_close(h); set_error("inflate state allocation failed"); return ZB_MEM_ERROR; }
    if ((rc = inflater_write_state(h, wrap)) != 0) { zb200i_inflate_close(h); return rc; }
    *out = h;
    return 0;
}

extern "C" int zb200i_inflate_reset(zb200i_inflater* h, int wrap) { return inflater_write_state(h, wrap); }

extern "C" void zb200i_inflate_close(zb200i_inflater* h)
{
    if (!h) return;
    if (h->d_state) cudaFree(h->d_state);
    if (h->d_res) cudaFree(h->d_res);
    if (h->d_arena) cudaFree(h->d_arena);
    if (h->d_in) cudaFree(h->d_in);
    if (h->h_pin) cudaFreeHost(h->h_pin);
    if (h->s) cudaStreamDestroy(h->s);
    delete h;
}

extern "C" int zb200i_inflate_clone(zb200i_inflater** out, const zb200i_inflater* src)
{
    zb200i_inflater* h = nullptr;
    int rc = zb200i_inflate_open(&h, src->wrap | (src->wbits << 8));
    if (rc) return rc;
    cudaError_t e = cudaMemcpy(h->d_state, src->d_state, sizeof(InfState), cudaMemcpyDeviceToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(h->d_arena, src->d_arena, kWindow32, cudaMemcpyDeviceToDevice);
    if (e != cudaSuccess) { zb200i_inflate_close(h); set_error("inflate state copy failed"); return ZB_MEM_ERROR; }
    h->carry = src->carry; h->hist = src->hist; h->mode = src->mode; h->check = src->check;
    h->crc = src->crc; h->produced = src->produced;
    *out = h;
    return 0;
}

extern "C" int zb200i_inflate_mode(const zb200i_inflater* h) { return h->mode; }
extern "C" size_t zb200i_inflate_pending_input(const zb200i_inflater* h) { return h->carry.size(); }
extern "C" const uint8_t* zb200i_inflate_pending_bytes(const zb200i_inflater* h) { return h->carry.data(); }

extern "C" int zb200i_inflate_set_dict(zb200i_inflater* h, const uint8_t* dict, size_t n)
{
    if (n > kWindow32) { dict += n - kWindow32; n = kWindow32; }
    ZB_CUDA(cudaMemcpyAsync(h->d_arena + kWindow32 - n, dict, n, cudaMemcpyDefault, h->s));
    const uint64_t hist = n;
    ZB_CUDA(cudaMemcpyAsync((uint8_t*)h->d_state + offsetof(InfState, hist), &hist, 8, cudaMemcpyHostToDevice, h->s));
    if (h->mode == kModeDict) {
        const int32_t mode = kModeBlock;
        ZB_CUDA(cudaMemcpyAsync((uint8_t*)h->d_state + offsetof(InfState, mode), &mode, 4, cudaMemcpyHostToDevice, h->s));
        h->mode = kModeBlock;
    }
    ZB_CUDA(cudaStreamSynchronize(h->s));
    h->hist = n;
    return 0;
}

extern "C" int zb200i_inflate_resync_keep(zb200i_inflater* h, size_t drop)
{
    // as below, but the marker was found INSIDE bytes the stream already holds: what follows it stays queued
    std::vector<uint8_t> rest;
    if (drop < h->carry.size()) rest.assign(h->carry.begin() + drop, h->carry.end());
    const int rc = zb200i_inflate_resync(h);
    if (rc == 0) h->carry.swap(rest);
    return rc;
}

extern "C" int zb200i_inflate_resync(zb200i_inflater* h)
{
    // inflate.c:1294-1301: keep totals, restart at a block boundary with an empty bit buffer
    InfState st;
    ZB_CUDA(cudaMemcpy(&st, h->d_state, sizeof(st), cudaMemcpyDeviceToHost));
    st.mode = kModeBlock; st.last = 0; st.bit_off = 0; st.stored_left = 0; st.copy_len = 0; st.msg = 0;
    ZB_CUDA(cudaMemcpy(h->d_state, &st, sizeof(st), cudaMemcpyHostToDevice));
    h->mode = kModeBlock;
    h->carry.clear();
    return 0;
}

// inflatePrime (inflate.c:128-142): `bits` bits of `value` are to be decoded ahead of the next input byte.  The decoder
// already knows how to start inside a byte (bit_off = bits of the first byte that are spent), so the primed bits become
// one or two bytes at the front of the pending input with the unused low bits marked as spent.
extern "C" int zb200i_inflate_prime(zb200i_inflater* h, int bits, int value)
{
    if (bits < 0 || bits > 16) return ZB_STREAM_ERROR;
    if (bits == 0) return 0;
    InfState st;
    ZB_CUDA(cudaMemcpy(&st, h->d_state, sizeof(InfState) - sizeof(st.lens), cudaMemcpyDeviceToHost));
    if (!h->carry.empty() || st.bit_off != 0) { set_error("inflatePrime: only on a byte boundary with no input pending"); return ZB_STREAM_ERROR; }
    const int nbytes = (bits + 7) / 8, pad = nbytes * 8 - bits;
    const uint32_t v = ((uint32_t)value & ((1u << bits) - 1u)) << pad;
    for (int i = 0; i < nbytes; i++) h->carry.push_back((uint8_t)(v >> (8 * i)));
    st.bit_off = (uint32_t)pad;
    ZB_CUDA(cudaMemcpy(h->d_state, &st, sizeof(InfState) - sizeof(st.lens), cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int zb200i_inflate_run(zb200i_inflater* h, const uint8_t* in, size_t in_len, uint8_t* out, size_t out_cap,
                                  size_t* in_used, size_t* out_len, int* status, int* msg, uint32_t* check)
{
    size_t taken = 0, produced = 0;
    int st = ZB200I_NEED_INPUT, m = 0;
    for (;;) {
        const size_t window = out_cap - produced < h->out_window ? out_cap - produced : h->out_window;
        size_t feed = in_len - taken;
        const size_t feed_cap = window + (window >> 3) + 4096;        // enough compressed bytes for one output window
        if (feed > feed_cap) feed = feed_cap;
        const size_t total_in = h->carry.size() + feed;
        if (total_in + 64 > h->h_pin_cap) {
            if (h->h_pin) cudaFreeHost(h->h_pin);
            h->h_pin_cap = (total_in + 64) * 2;
            if (cudaMallocHost(&h->h_pin, h->h_pin_cap) != cudaSuccess) { h->h_pin = nullptr; h->h_pin_cap = 0; set_error("pinned allocation failed"); return ZB_MEM_ERROR; }
        }
        if (total_in + 64 > h->d_in_cap) {
            if (h->d_in) cudaFree(h->d_in);
            h->d_in_cap = (total_in + 64) * 2;
            if (cudaMalloc(&h->d_in, h->d_in_cap) != cudaSuccess) { h->d_in = nullptr; h->d_in_cap = 0; set_error("device allocation failed"); return ZB_MEM_ERROR; }
        }
        if (!h->carry.empty()) memcpy(h->h_pin, h->carry.data(), h->carry.size());
        if (feed) memcpy(h->h_pin + h->carry.size(), in + taken, feed);
        memset(h->h_pin + total_in, 0, 8);
        ZB_CUDA(cudaMemcpyAsync(h->d_in, h->h_pin, total_in + 8, cudaMemcpyHostToDevice, h->s));
        int rc = inflate_stream_launch(h->d_in, total_in, h->d_arena + kWindow32, window, h->d_state, h->d_res, h->s);
        if (rc) return rc;
        InfCallResult res;
        ZB_CUDA(cudaMemcpyAsync(&res, h->d_res, sizeof(res), cudaMemcpyDeviceToHost, h->s));
        ZB_CUDA(cudaStreamSynchronize(h->s));
        if (res.out_len && h->wrap >= ZB200_WRAP_GZIP) {         // gzip (or undecided): CRC-32 of this window joins the running value
            Ctx* c = ctx_acquire(h->s);
            if (!c) return ZB_MEM_ERROR;
            uint32_t piece[2] = {0, 0};
            int rc2 = c->small.ensure(256);
            if (!rc2) rc2 = checksum_launch(c, h->d_arena + kWindow32, res.out_len, c->small.as<uint32_t>(), h->s);
            if (!rc2 && (cudaMemcpyAsync(piece, c->small.p, 8, cudaMemcpyDeviceToHost, h->s) != cudaSuccess ||
                         cudaStreamSynchronize(h->s) != cudaSuccess)) { set_error("checksum readback failed"); rc2 = ZB_STREAM_ERROR; }
            ctx_release(c, h->s);
            if (rc2) return rc2;
            h->crc = (uint32_t)crc32_combine(h->crc, piece[0], (long)res.out_len);
            h->produced += res.out_len;
        }
        if (res.out_len) {
            ZB_CUDA(cudaMemcpyAsync(out + produced, h->d_arena + kWindow32, res.out_len, cudaMemcpyDeviceToHost, h->s));
            ZB_LAUNCH(k_slide_history, 1, 1024, 0, h->s, h->d_arena, h->hist, res.out_len);
            ZB_CUDA(cudaStreamSynchronize(h->s));
            const uint64_t v = h->hist + res.out_len;
            h->hist = v > kWindow32 ? kWindow32 : v;
        }
        produced += res.out_len;
        st = res.status; m = res.msg;
        if (res.in_used > total_in) {                                  // the decoder may never run past what it was given
            set_error("internal error: inflate consumed %llu of %zu input bytes", (unsigned long long)res.in_used, total_in);
            return ZB_STREAM_ERROR;
        }
        // account for the input: the decoder consumed res.in_used bytes of [carry | feed]
        const size_t carry_n = h->carry.size();
        size_t from_new = res.in_used > carry_n ? res.in_used - carry_n : 0;
        if (st == ZB200I_NEED_INPUT || st == ZB_NEED_DICT || st == ZB_STREAM_END || st == ZB_DATA_ERROR) {
            // whatever is left of this call's window of input stays with the stream
            std::vector<uint8_t> rest(h->h_pin + res.in_used, h->h_pin + total_in);
            if (st == ZB_STREAM_END || st == ZB_DATA_ERROR || st == ZB_NEED_DICT) {
                // bytes after the end of the stream, or after the dictionary id (inflate.c:1138 stops there too), belong to
                // the caller again; bytes taken by an earlier call stay queued for the decode behind the dictionary
                // The carry holds bytes only after a NEED_INPUT stop, which the decoder makes only when those bytes do not
                // complete the item it must read next (a code and its extra bits, a header field, a stored length, the
                // trailer): so a stream cannot end inside them.  They were counted into an earlier call's total_in and could
                // not be handed back; should that ever happen, say so rather than drop the start of what follows.
                if (st == ZB_STREAM_END && res.in_used < carry_n) {
                    set_error("internal error: the stream ended inside %zu bytes held from an earlier call", carry_n - (size_t)res.in_used);
                    return ZB_STREAM_ERROR;
                }
                rest.clear();
                taken += from_new;
                if (st == ZB_NEED_DICT && res.in_used < carry_n) rest.assign(h->h_pin + res.in_used, h->h_pin + carry_n);
            } else {
                taken += feed;
            }
            h->carry.swap(rest);
        } else {                                                       // output window full
            if (res.in_used >= carry_n) { h->carry.clear(); taken += from_new; }
            else h->carry.erase(h->carry.begin(), h->carry.begin() + res.in_used);
        }
        if (st == ZB200I_NEED_INPUT && taken < in_len) continue;       // more caller input to hand over
        if (st == ZB200I_NEED_OUTPUT && produced < out_cap) continue;  // more room in the caller's buffer
        break;
    }
    InfState dst;
    ZB_CUDA(cudaMemcpy(&dst, h->d_state, sizeof(InfState) - sizeof(dst.lens), cudaMemcpyDeviceToHost));
    h->mode = dst.mode;
    if (h->wrap == kWrapAuto && dst.wrap != kWrapAuto) h->wrap = dst.wrap;      // the header settled zlib vs gzip
    h->check = st == ZB_NEED_DICT ? dst.dict_id : h->wrap >= ZB200_WRAP_GZIP ? h->crc : ((dst.s2 << 16) | dst.s1);
    if (st == ZB_STREAM_END && (dst.flags & kFlagGzipTrailer)) {                // inflate.c:1099-1112
        if (dst.crc != h->crc) { st = ZB_DATA_ERROR; m = kMsgCheck; }
        else if (dst.isize != (uint32_t)h->produced) { st = ZB_DATA_ERROR; m = kMsgLength; }
        if (st == ZB_DATA_ERROR) h->mode = kModeBad;
    }
    *in_used = taken; *out_len = produced; *status = st; *msg = m; *check = h->check;
    return 0;
}


ZB_API int zb200_inflate_batch_dev(const void* d_src, const uint64_t* d_src_off, size_t n, void* d_dst,
                                   const uint64_t* d_dst_off, uint64_t* d_dst_len, int32_t* d_status, int wrap,
                                   void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (wrap != ZB200_WRAP_GZIP && wrap != kWrapAuto)
        return inflate_batch_launch((const uint8_t*)d_src, d_src_off, n, (uint8_t*)d_dst, d_dst_off, d_dst_len, d_status,
                                    wrap, nullptr, (cudaStream_t)stream);
    Ctx* c = ctx_acquire((cudaStream_t)stream);                  // scratch for the trailer values
    if (!c) return ZB_MEM_ERROR;
    if ((rc = c->ws[0].ensure(n * 12 + 16)) == 0)
        rc = inflate_batch_launch((const uint8_t*)d_src, d_src_off, n, (uint8_t*)d_dst, d_dst_off, d_dst_len, d_status,
                                  wrap, c->ws[0].as<uint32_t>(), (cudaStream_t)stream);
    ctx_release(c, (cudaStream_t)stream);
    return rc;
}

// Host arenas: the streams are taken in groups of about kInfGroupBytes of output; the H2D copy of group k+1 and the D2H
// copy of group k-1 run on the context's two copy streams while group k decodes (the batch is PCIe-bound end to end:
// about 0.47 bytes in and 1 byte out per byte decoded).  Groups alternate between two streams, because one group's warps
// (one per stream) do not fill the GPU and kernels on one stream do not overlap.  Device arenas: one launch, no copies.
constexpr uint64_t kInfGroupBytes = 192ull << 20;

ZB_API int zb200_inflate_batch(const void* src, const uint64_t* src_off, size_t n, void* dst, const uint64_t* dst_off,
                               uint64_t* dst_len, int32_t* status, int wrap, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (n == 0) return 0;
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    Ctx* c2 = nullptr;                                           // odd groups decode on a second stream
    HostStager stager;                                           // pageable arenas of 64 MiB and more
    HostDrainer drainer;
    do {
        const size_t src_total = (size_t)src_off[n], dst_total = (size_t)dst_off[n];
        const bool src_on_host = src_total != 0 && classify(src) != kDevice;
        const bool dst_on_host = classify(dst) != kDevice;
        const uint8_t* d_src = (const uint8_t*)src;
        if (src_on_host || src_total == 0) {
            if ((rc = c->in.ensure(src_total + 64)) != 0) break;
            d_src = c->in.as<uint8_t>();
        }
        uint8_t* d_dst = (uint8_t*)dst;
        if (dst_on_host) {
            if ((rc = c->out.ensure(dst_total + 16)) != 0) break;
            d_dst = c->out.as<uint8_t>();
        }
        cudaError_t e = cudaSuccess;
        // ---- long streams first: a stream of its own is serial (one warp, ~15 MB/s), so the few long ones of a call --
        // uncompress() of a big buffer is the case n == 1 -- try the segment-parallel decoder; whatever it does not take
        // stays in the batch below.  Many medium streams are better off side by side in the batch kernel.
        std::vector<uint8_t> handled(n, 0);
        size_t nhandled = 0;
        {
            for (size_t i = 0; i < n && !rc; i++) {
                const uint64_t a = src_off[i], len = src_off[i + 1] - a;
                if (len < kParMinInput || (n > kParFewStreams && len < kParLongStream)) continue;
                if (src_on_host && len >= HostStager::kMinBytes && classify(src) == kHostPageable) {
                    HostStager stager;                          // pageable and long: host threads feed pinned slots
                    if ((rc = stager.start((const uint8_t*)src + a, (uint8_t*)d_src + a, len, s)) != 0) break;
                    if ((rc = stager.wait_range(0, len, s)) != 0) break;
                    stager.finish();
                } else if (src_on_host) {
                    e = cudaMemcpyAsync((uint8_t*)d_src + a, (const uint8_t*)src + a, len, cudaMemcpyHostToDevice, s);
                    if (e != cudaSuccess) { set_error("input staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
                }
                uint64_t got = 0;
                int32_t st = ZB_OK;
                void* h_out = dst_on_host && classify(dst) == kHostPinned ? (uint8_t*)dst + dst_off[i] : nullptr;   // receives the output as it is finished
                const int pr = inflate_single_parallel(c, d_src + a, len, d_dst + dst_off[i], dst_off[i + 1] - dst_off[i], wrap, &got, &st, s,
                                                       nullptr, nullptr, nullptr, h_out);
                if (pr < 0) { rc = pr; break; }
                if (pr != 0) { if (h_out && c->aux[1]) cudaStreamSynchronize(c->aux[1]); continue; }
                if (h_out) {                                    // already there: copied phase by phase behind the walk
                } else if (dst_on_host && got >= HostStager::kMinBytes && classify(dst) == kHostPageable) {
                    HostDrainer drainer;                        // the decoder has synchronised: the output is complete
                    if ((rc = drainer.drain((uint8_t*)dst + dst_off[i], d_dst + dst_off[i], got)) != 0) break;
                } else if (dst_on_host && got) e = cudaMemcpyAsync((uint8_t*)dst + dst_off[i], d_dst + dst_off[i], got, cudaMemcpyDeviceToHost, s);
                if (e != cudaSuccess) { set_error("inflate readback failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
                dst_len[i] = got; status[i] = st;
                handled[i] = 1; nhandled++;
            }
            if (rc) { cudaStreamSynchronize(s); break; }
        }
        if (nhandled == n) {
            if (cudaStreamSynchronize(s) != cudaSuccess) { set_error("inflate readback failed: %s", cudaGetErrorString(cudaGetLastError())); rc = ZB_STREAM_ERROR; }
            break;
        }
        // ---- groups of consecutive streams that are still to do ----
        std::vector<size_t> g0, g1;                              // group k = streams [g0[k], g1[k])
        const bool pipelined = src_on_host || dst_on_host;
        for (size_t i = 0; i < n;) {
            if (handled[i]) { i++; continue; }
            size_t j = i + 1;
            while (j < n && !handled[j] && !(pipelined && dst_off[j] - dst_off[i] >= kInfGroupBytes)) j++;
            g0.push_back(i); g1.push_back(j);
            i = j;
        }
        const size_t ng = g0.size();
        if (ng > 1 && (c2 = ctx_acquire_own()) == nullptr) { rc = ZB_MEM_ERROR; break; }
        if ((rc = c->ensure_aux((int)(2 * ng + 4))) != 0) break;
        cudaStream_t s_in = c->aux[0], s_out = c->aux[1];
        cudaEvent_t* ev_in = c->evs;
        cudaEvent_t* ev_done = c->evs + ng;
        // descriptors: [src_off n+1][dst_off n+1][dst_len n][status n][gzip trailer values 3n]
        const size_t desc_bytes = (size_t)(3 * n + 2) * 8 + n * 4 + n * 12;
        if ((rc = c->ws[0].ensure(desc_bytes)) != 0) break;
        uint64_t* d_src_off = c->ws[0].as<uint64_t>();
        uint64_t* d_dst_off = d_src_off + (n + 1);
        uint64_t* d_len = d_dst_off + (n + 1);
        int32_t* d_status = (int32_t*)(d_len + n);
        uint32_t* d_expect = (uint32_t*)(d_status + n);
        if ((rc = c->ensure_pinned(n * 12 + 16)) != 0) break;
        uint64_t* h_len = (uint64_t*)c->pinned;
        int32_t* h_status = (int32_t*)(h_len + n);
        e = cudaMemcpyAsync(d_src_off, src_off, (n + 1) * 8, cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_dst_off, dst_off, (n + 1) * 8, cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) {                                  // the copy streams and the second decode stream start here
            e = cudaEventRecord(c->evs[2 * ng], s);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(s_in, c->evs[2 * ng], 0);
            if (e == cudaSuccess && c2) e = cudaStreamWaitEvent(c2->own_stream, c->evs[2 * ng], 0);
        }
        if (e != cudaSuccess) { set_error("descriptor upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        const bool threaded = src_on_host && src_total >= HostStager::kMinBytes && classify(src) == kHostPageable;
        const bool drain_threads = dst_on_host && dst_total >= HostStager::kMinBytes && classify(dst) == kHostPageable;
        if (threaded && (rc = stager.start(src, (uint8_t*)d_src, src_total, s_in)) != 0) break;
        cudaStream_t s_main = s;
        for (size_t k = 0; k < ng && !rc; k++) {
            const size_t i0 = g0[k], i1 = g1[k];
            const uint64_t a = src_off[i0], b = src_off[i1];
            cudaStream_t s = (c2 && (k & 1)) ? c2->own_stream : s_main;
            if (src_on_host && b > a && threaded) {              // pageable arena: pieces arrive from the staging threads
                if ((rc = stager.wait_range(a, b - a, s)) != 0) break;
            } else if (src_on_host && b > a) {
                e = cudaMemcpyAsync((uint8_t*)d_src + a, (const uint8_t*)src + a, b - a, cudaMemcpyHostToDevice, s_in);
                if (e == cudaSuccess) e = cudaEventRecord(ev_in[k], s_in);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s, ev_in[k], 0);
                if (e != cudaSuccess) { set_error("input staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
            if ((rc = inflate_batch_launch(d_src, d_src_off + i0, i1 - i0, d_dst, d_dst_off + i0, d_len + i0, d_status + i0, wrap,
                                           d_expect + 3 * i0, s)) != 0) break;
            // results go to pinned memory (a copy to the caller's pageable arrays would block the host until this group is done)
            e = cudaMemcpyAsync(h_len + i0, d_len + i0, (i1 - i0) * 8, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaMemcpyAsync(h_status + i0, d_status + i0, (i1 - i0) * 4, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && dst_on_host && dst_off[i1] > dst_off[i0]) {
                e = cudaEventRecord(ev_done[k], s);
                if (e == cudaSuccess && !drain_threads) {
                    e = cudaStreamWaitEvent(s_out, ev_done[k], 0);
                    if (e == cudaSuccess) e = cudaMemcpyAsync((uint8_t*)dst + dst_off[i0], d_dst + dst_off[i0], dst_off[i1] - dst_off[i0], cudaMemcpyDeviceToHost, s_out);
                }
            }
            if (e != cudaSuccess) { set_error("output copy failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        }
        if (c2) {                                                // join the second stream
            cudaEventRecord(c->evs[2 * ng + 1], c2->own_stream);
            cudaStreamWaitEvent(s, c->evs[2 * ng + 1], 0);
        }
        if (rc) { cudaStreamSynchronize(s); cudaStreamSynchronize(s_in); cudaStreamSynchronize(s_out); break; }
        if (drain_threads) {                                    // malloc'ed output arena: drain group by group while later groups decode
            for (size_t k = 0; k < ng && !rc; k++) {
                if (dst_off[g1[k]] == dst_off[g0[k]]) continue;
                if (cudaEventSynchronize(ev_done[k]) != cudaSuccess) { set_error("inflate batch failed: %s", cudaGetErrorString(cudaGetLastError())); rc = ZB_STREAM_ERROR; break; }
                rc = drainer.drain((uint8_t*)dst + dst_off[g0[k]], d_dst + dst_off[g0[k]], dst_off[g1[k]] - dst_off[g0[k]]);
            }
            if (rc) { cudaStreamSynchronize(s); break; }
        }
        e = cudaStreamSynchronize(s);
        if (e == cudaSuccess && dst_on_host) e = cudaStreamSynchronize(s_out);
        if (e != cudaSuccess) { set_error("inflate batch readback failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        for (size_t k = 0; k < ng; k++)
            for (size_t i = g0[k]; i < g1[k]; i++) { dst_len[i] = h_len[i]; status[i] = h_status[i]; }
    } while (0);
    stager.finish();
    drainer.finish();
    if (c2) ctx_release(c2, c2->own_stream);
    ctx_release(c, s);
    return rc;
}

// ---- sizing: zb200_inflate_batch_size ----
// The streams zb200_inflate_batch would send to the one-stream segment decoder (same rule) get its search and counting
// pass alone; the rest, and whatever that pass declines, go to k_inflate_count.  Only compressed bytes travel: a host
// arena moves in groups of about kInfGroupBytes on the copy stream while earlier groups are counted, the groups alternate
// between two streams (one group's warps do not fill the GPU), and the results come back through the context's pinned
// words, 20 bytes per stream.
static int size_args(const char* who, const uint64_t* src_off, size_t n, const void* out_len, const void* status, int wrap)
{
    if (wrap < 0 || wrap > kWrapAuto) { set_error("%s: wrap %d not supported", who, wrap); return ZB_STREAM_ERROR; }
    if (n && (!src_off || !out_len || !status)) { set_error("%s: src_off, out_len and status are required", who); return ZB_STREAM_ERROR; }
    return 0;
}

ZB_API int zb200_inflate_batch_size(const void* src, const uint64_t* src_off, size_t n, uint64_t* out_len, uint64_t* src_used,
                                    int32_t* status, int wrap, uint64_t limit, void* stream)
{
    int rc = size_args("zb200_inflate_batch_size", src_off, n, out_len, status, wrap);
    if (rc) return rc;
    for (size_t i = 0; i < n; i++)
        if (src_off[i + 1] < src_off[i]) { set_error("zb200_inflate_batch_size: src_off must not decrease"); return ZB_STREAM_ERROR; }
    if ((rc = ensure_init()) != 0) return rc;
    if (n == 0) return 0;
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    Ctx* c2 = nullptr;
    HostStager stager;
    const uint64_t cap = limit ? limit : ~0ull;
    do {
        const size_t src_total = (size_t)src_off[n];
        const bool src_on_host = src_total != 0 && classify(src) != kDevice;
        const uint8_t* d_src = (const uint8_t*)src;
        if (src_on_host || src_total == 0) {
            if ((rc = c->in.ensure(src_total + 64)) != 0) break;
            d_src = c->in.as<uint8_t>();
        }
        cudaError_t e = cudaSuccess;
        // ---- long streams: the counting pass of the segment decoder ----
        std::vector<uint8_t> handled(n, 0);
        size_t nhandled = 0;
        for (size_t i = 0; i < n && !rc; i++) {
            const uint64_t a = src_off[i], len = src_off[i + 1] - a;
            if (len < kParMinInput || (n > kParFewStreams && len < kParLongStream)) continue;
            if (src_on_host && len >= HostStager::kMinBytes && classify(src) == kHostPageable) {
                HostStager one;
                if ((rc = one.start((const uint8_t*)src + a, (uint8_t*)d_src + a, len, s)) != 0) break;
                if ((rc = one.wait_range(0, len, s)) != 0) break;
                one.finish();
            } else if (src_on_host) {
                e = cudaMemcpyAsync((uint8_t*)d_src + a, (const uint8_t*)src + a, len, cudaMemcpyHostToDevice, s);
                if (e != cudaSuccess) { set_error("input staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
            uint64_t got = 0, used = 0;
            int32_t st = ZB_OK;
            const int pr = inflate_single_parallel(c, d_src + a, len, nullptr, cap, wrap, &got, &st, s, &used, nullptr, nullptr, nullptr,
                                                   nullptr, true);
            if (pr < 0) { rc = pr; break; }
            if (pr != 0) continue;
            out_len[i] = got; status[i] = st;
            if (src_used) src_used[i] = used;
            handled[i] = 1; nhandled++;
        }
        if (rc) { cudaStreamSynchronize(s); break; }
        if (nhandled == n) {
            if (cudaStreamSynchronize(s) != cudaSuccess) { set_error("inflate size failed: %s", cudaGetErrorString(cudaGetLastError())); rc = ZB_STREAM_ERROR; }
            break;
        }
        // ---- groups of consecutive streams still to do, by compressed bytes ----
        std::vector<size_t> g0, g1;
        for (size_t i = 0; i < n;) {
            if (handled[i]) { i++; continue; }
            size_t j = i + 1;
            while (j < n && !handled[j] && !(src_on_host && src_off[j] - src_off[i] >= kInfGroupBytes)) j++;
            g0.push_back(i); g1.push_back(j);
            i = j;
        }
        const size_t ng = g0.size();
        if (ng > 1 && (c2 = ctx_acquire_own()) == nullptr) { rc = ZB_MEM_ERROR; break; }
        if ((rc = c->ensure_aux((int)(ng + 2))) != 0) break;
        cudaStream_t s_in = c->aux[0];
        // descriptors: [src_off n+1][out_len n][src_used n][status n]; results: [out_len n][src_used n][status n] pinned
        if ((rc = c->ws[0].ensure((size_t)(3 * n + 1) * 8 + n * 4)) != 0) break;
        uint64_t* d_src_off = c->ws[0].as<uint64_t>();
        uint64_t* d_len = d_src_off + (n + 1);
        uint64_t* d_used = d_len + n;
        int32_t* d_status = (int32_t*)(d_used + n);
        if ((rc = c->ensure_pinned(n * 20 + 16)) != 0) break;
        uint64_t* h_len = (uint64_t*)c->pinned;
        uint64_t* h_used = h_len + n;
        int32_t* h_status = (int32_t*)(h_used + n);
        e = cudaMemcpyAsync(d_src_off, src_off, (n + 1) * 8, cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) {
            e = cudaEventRecord(c->evs[ng], s);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(s_in, c->evs[ng], 0);
            if (e == cudaSuccess && c2) e = cudaStreamWaitEvent(c2->own_stream, c->evs[ng], 0);
        }
        if (e != cudaSuccess) { set_error("descriptor upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        const bool threaded = src_on_host && src_total >= HostStager::kMinBytes && classify(src) == kHostPageable;
        if (threaded && (rc = stager.start(src, (uint8_t*)d_src, src_total, s_in)) != 0) break;
        cudaStream_t s_main = s;
        for (size_t k = 0; k < ng && !rc; k++) {
            const size_t i0 = g0[k], i1 = g1[k];
            const uint64_t a = src_off[i0], b = src_off[i1];
            cudaStream_t s = (c2 && (k & 1)) ? c2->own_stream : s_main;
            if (src_on_host && b > a && threaded) {
                if ((rc = stager.wait_range(a, b - a, s)) != 0) break;
            } else if (src_on_host && b > a) {
                e = cudaMemcpyAsync((uint8_t*)d_src + a, (const uint8_t*)src + a, b - a, cudaMemcpyHostToDevice, s_in);
                if (e == cudaSuccess) e = cudaEventRecord(c->evs[k], s_in);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(s, c->evs[k], 0);
                if (e != cudaSuccess) { set_error("input staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
            if ((rc = inflate_count_launch(d_src, d_src_off + i0, i1 - i0, limit, d_len + i0, src_used ? d_used + i0 : nullptr,
                                           d_status + i0, wrap, s)) != 0) break;
            e = cudaMemcpyAsync(h_len + i0, d_len + i0, (i1 - i0) * 8, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && src_used) e = cudaMemcpyAsync(h_used + i0, d_used + i0, (i1 - i0) * 8, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaMemcpyAsync(h_status + i0, d_status + i0, (i1 - i0) * 4, cudaMemcpyDeviceToHost, s);
            if (e != cudaSuccess) { set_error("result copy failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        }
        if (c2) {
            cudaEventRecord(c->evs[ng + 1], c2->own_stream);
            cudaStreamWaitEvent(s, c->evs[ng + 1], 0);
        }
        if (rc) { cudaStreamSynchronize(s); cudaStreamSynchronize(s_in); break; }
        e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { set_error("inflate size readback failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        for (size_t k = 0; k < ng; k++)
            for (size_t i = g0[k]; i < g1[k]; i++) {
                out_len[i] = h_len[i]; status[i] = h_status[i];
                if (src_used) src_used[i] = h_used[i];
            }
    } while (0);
    stager.finish();
    if (c2) ctx_release(c2, c2->own_stream);
    ctx_release(c, s);
    return rc;
}

ZB_API int zb200_inflate_batch_size_dev(const void* d_src, const uint64_t* d_src_off, size_t n, uint64_t* d_out_len,
                                        uint64_t* d_src_used, int32_t* d_status, uint64_t* d_dst_off, int wrap, uint64_t limit,
                                        void* stream)
{
    int rc = size_args("zb200_inflate_batch_size_dev", d_src_off, n, d_out_len, d_status, wrap);
    if (rc) return rc;
    if ((rc = ensure_init()) != 0) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if ((rc = inflate_count_launch((const uint8_t*)d_src, d_src_off, n, limit, d_out_len, d_src_used, d_status, wrap, s)) != 0) return rc;
    if (d_dst_off) {
        ZB_LAUNCH(k_size_scan, 1, 1024, 0, s, d_out_len, (uint64_t)n, d_dst_off);
        ZB_CHECK_LAUNCH();
    }
    return 0;
}
