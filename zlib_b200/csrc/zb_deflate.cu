// zb_deflate.cu -- K1..K3: the DEFLATE compressor as a pipeline of data-parallel kernels.
//
// Replaces, in the reference: fill_window/INSERT_STRING/longest_match/deflate_fast/deflate_slow
// (qcsrc/deflate.c:1266,189,1027,1448,1554) and _tr_tally/_tr_flush_block/build_tree/gen_bitlen/
// gen_codes/send_all_trees/compress_block/send_bits (qcsrc/trees.c:1022,921,619,490,577,838,1072,217).
//
// The reference interleaves these per input byte inside one sequential loop.  Here the same
// decisions are taken in passes over HBM-resident arrays, each with its own parallel axis:
//
//   K1a link   one CTA (8 warps) per 256 KiB segment shares a 15-bit hash -> last position table in
//              shared memory (the reference's head[]).  The warps take 128-position tiles round robin; only
//              the table accesses of a tile are serial and the turn is handed from warp to warp with named
//              barriers.  Output: for every position the distance to the previous position with the same
//              4-byte hash (the reference's prev[] chain, stored as deltas so chains cross chunk boundaries
//              and the 32 KiB of history in front of a chunk needs no copy -- it is simply there).
//   K1b walk   one CTA per 32 KiB block, window staged in shared memory, one thread per 64-byte sub-unit
//              running the reference's own search-emit-skip loop (deflate_fast, or deflate_slow with max_lazy,
//              good_match and TOO_FAR, deflate.c:1448-1674): chain candidates up to max_chain
//              (configuration_table, deflate.c:137-149), quick reject on the word a longer match must reach,
//              nice_match.  Sub-unit boundaries are reconciled afterwards (prefix maximum of end positions);
//              tokens are compacted per block and tallied into the block histogram.
//   K2 codes   one warp per block (32 KiB of input) builds the three length-limited canonical
//              codes (sort + two-queue merge, the reference's overflow repair), prices stored / fixed /
//              dynamic with the reference's rule (trees.c:955-1001) and serialises the dynamic header.
//   plan+scan  exact compressed size of every chunk -> exclusive prefix sum -> byte offsets.
//   K3 pack    one CTA per chunk: per-symbol (code, length) -> prefix sum of lengths -> bits OR-ed into a
//              shared-memory staging window -> bytes to their final place.  Chunks end byte-aligned (empty
//              stored block, i.e. what Z_SYNC_FLUSH emits, deflate.c:808-819), so shards from several
//              GPUs concatenate by byte copy.
//
// A call is cut into slabs of kSlabChunks chunks that run back to back on one stream and share one set of
// scratch buffers; with host buffers the H2D copy of slab i+1 and the D2H copy of slab i-1 overlap the
// kernels of slab i (separate copy streams).
//
// Output is a valid DEFLATE stream, not the reference's bytes: parity is "reference inflate decodes
// it bit-exact" plus a size bound (<= 1.02 x reference at the same level), see tests/.
#include "zb_deflate.cuh"
#include "zb200_internal.h"
#include <stdlib.h>
#include <algorithm>
#include <type_traits>
#include <vector>

namespace zb {

// configuration_table (deflate.c:137-149): good / lazy / nice as in the reference, and the same two parsers (greedy for
// levels 1..3, lazy for 4..9), but NOT its chain budgets, because the chains are not the reference's: k_lz_link enters
// every position (the reference's fast levels only enter token starts) and hashes FOUR bytes where the reference's
// UPDATE_HASH covers MIN_MATCH = 3.  A chain over three bytes is mostly other strings that share three bytes: at level 1
// two steps down such a chain found less than ONE step down a four-byte chain finds (256 MiB mixed: 134.8 MB at 3.40 ms
// against 127.2 MB at 3.32 ms; the reference's level 1 writes 136.3 MB, its level 9 129.1 MB), and at level 6 eight
// candidates of a four-byte chain beat 32 of a three-byte one (124.5 MB at 5.76 ms against 126.6 MB at 9.19 ms; reference
// level 6: 129.5 MB).  What four bytes give up are the matches of exactly three bytes (found only where hashes collide);
// the tables of profiles/r2_sweeps.md show what that costs: nothing, on these corpora.  The budgets below are the knees of
// those sweeps -- every level writes less than the reference's level 9 on both corpora, sizes fall and times rise with
// the level.  Z_FIXED and windowBits < 15 use the same chains.
static const LevelCfg h_levels[10] = {
    {0, 0, 0, 0, 0},      {4, 4, 8, 1, 1},       {4, 5, 16, 2, 1},     {4, 6, 32, 3, 1},
    {4, 4, 16, 4, 2},     {8, 16, 32, 5, 2},     {8, 16, 128, 8, 2},   {8, 32, 128, 16, 2},
    {32, 128, 258, 48, 2}, {32, 258, 258, 192, 2}};

constexpr uint32_t kFullMask = 0xffffffffu;
constexpr int kHashBits = 15;

// ------------------------------------------------------------------------------------------
// K1a: hash-chain links
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hash4(uint32_t v) { return (v * 0x9E3779B1u) >> (32 - kHashBits); }   // four bytes, see h_levels

// Ring version: kLinkWarps warps share one segment and one head[] table.  Warp w owns tiles
// w, w+W, w+2W, ... (a tile = kLinkSteps steps of 32 consecutive positions).  Everything that does not touch head[]
// -- loads, hashes, the intra-step same-hash groups, the dist16 stores -- runs concurrently in all
// warps; only the short "read head[], then write head[]" section of a tile is serial, and it is
// passed from warp to warp in position order with named barriers (producer bar.arrive, consumer
// bar.sync, 64 threads each).  The links are exactly those of the one-warp version.
constexpr int kLinkWarps = 8;
// Stream mode: one CTA links two chunks.  The 32 KiB of priming in front of a segment is redundant work; 1 / 2 / 4 chunks per
// segment measured 13.50 / 13.31 / 13.56 ms per step.
constexpr uint32_t kLinkSegBytes = 2 * kChunk;
// A segment's CTA is one serial chain of ring turns, and the kernel runs as one wave, so its time is turns per segment x
// the latency of a turn.  A hand-off costs far more than a step's read and write of head[], so a turn takes many steps.
constexpr int kLinkSteps = 16;
constexpr int kLinkTile = 32 * kLinkSteps;                      // positions per tile
constexpr int kLinkRegs = kLinkSteps / 4;                       // words of the tile per lane (a step covers eight)
// head[], then one slot per lane that positions whose hash is not entered read and write instead
constexpr uint32_t kLinkSmem = (1u << kHashBits) * 2 + 32 * 2;

__device__ __forceinline__ void ring_wait(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void ring_pass(int id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }

struct LinkAddrs { uint32_t a[kLinkSteps]; };                   // per step: the shared-memory address of the lane's head[] slot
struct LinkHeads { uint32_t h[kLinkSteps]; };                   // per step: what that slot held before the step

// One warp's turn: wait for the token, then for each of the tile's steps read head[] (every lane, the caller ignores what
// it does not need) and write the lane's position -- in exact mode only where bit k of wmask is set: the step's group
// leaders; pass the token on.  Each step is one warp-wide read and one warp-wide write, so same-hash positions of a
// relaxed step resolve within one store instruction.  Shared-memory accesses of one warp execute in program order, which
// is all the steps need from each other.  A real call, so that the compiler schedules nothing else between the barriers.
template <bool kExact>
__device__ __noinline__ LinkHeads ring_turn(LinkAddrs a, uint32_t q, uint32_t wmask, int bar_in, int bar_out)
{
    LinkHeads t;
    asm volatile("bar.sync %0, 64;" ::"r"(bar_in) : "memory");
#pragma unroll
    for (int k = 0; k < kLinkSteps; ++k) {
        if (kExact)
            asm volatile("{\n.reg .pred w;\n.reg .b32 x;\nand.b32 x, %3, %4; setp.ne.u32 w, x, 0;\n"
                         "ld.shared.u16 %0, [%1];\n@w st.shared.u16 [%1], %2;\n}"
                         : "=r"(t.h[k]) : "r"(a.a[k]), "r"(q + 32 * k), "r"(wmask), "r"(1u << k) : "memory");
        else
            asm volatile("ld.shared.u16 %0, [%1];\nst.shared.u16 [%1], %2;"
                         : "=r"(t.h[k]) : "r"(a.a[k]), "r"(q + 32 * k) : "memory");
    }
    asm volatile("bar.arrive %0, 64;" ::"r"(bar_out) : "memory");
    return t;
}

template <bool kExact>
__global__ void __launch_bounds__(kLinkWarps * 32, 3)          // 3 CTAs per SM: the 64 KiB head[] tables fill shared memory
k_lz_link(const uint8_t* __restrict__ buf, uint64_t total, uint16_t* __restrict__ dist16, const ChunkDesc* __restrict__ cd)
{
    extern __shared__ uint16_t s_head[];                       // 2^15 entries: low 16 bits of the last position
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    for (int i = threadIdx.x; i < (1 << kHashBits) / 2; i += kLinkWarps * 32) reinterpret_cast<uint32_t*>(s_head)[i] = 0;
    __syncthreads();

    // the segment, the first position whose hash is entered (priming), the end of hashable data, position zero of the stream
    uint64_t seg_beg, seg_end, prime_beg, lim, origin;
    if (cd) {                                                   // job mode: the segment is a chunk of some job
        const ChunkDesc d = cd[blockIdx.x];
        seg_beg = d.beg; seg_end = (uint64_t)d.beg + d.len; origin = d.job_beg; lim = d.job_end;
        prime_beg = seg_beg - origin > kWindow ? seg_beg - kWindow : origin;
    } else {
        seg_beg = (uint64_t)blockIdx.x * kLinkSegBytes;         // stream mode: a CTA links kLinkSegBytes
        seg_end = min(total, seg_beg + kLinkSegBytes);
        prime_beg = seg_beg > kWindow ? seg_beg - kWindow : 0;
        origin = 0; lim = total;
    }
    const uint32_t mis = (uint32_t)((uintptr_t)buf & 3);
    // q = p + mis indexes bytes from the 4-byte aligned base; tiles start at q0, the 128-aligned q in front of the first
    // position to insert.  Everything below is relative to q0, so it fits 32 bits (a segment spans <= 288 KiB + 128).
    const uint64_t tile_beg = (prime_beg + mis) >> 7;
    const uint64_t q0 = tile_beg * 128;
    const uint32_t* words = reinterpret_cast<const uint32_t*>(buf - mis) + tile_beg * 32;
    const uint32_t nwords = (uint32_t)min((uint64_t)0x7fffffffu, ((mis + total + 3) >> 2) - tile_beg * 32);
    uint16_t* dout = dist16 + q0 - mis;                         // dout[q - q0] = link of position q - mis (never dereferenced below q_seg)
    const int q_lo = (int)(prime_beg + mis - q0);               // first position to insert
    // one past the last hashable position: a position is entered only if all four bytes of its hash are the stream's own
    const int q_hi = (int)(min(seg_end, lim >= origin + 3 ? lim - 3 : origin) + mis) - (int)q0;
    const int q_seg = (int)(seg_beg + mis - q0), q_end = (int)(seg_end + mis - q0);   // positions whose link is stored
    const int p_cap = (int)min((uint64_t)0x40000000u, q0 - mis + 128 - origin) - 128;   // stream position of q0, saturated (only "dd > p" uses it)
    const uint32_t ntiles = (uint32_t)((q_end + kLinkTile - 1) / kLinkTile);
    const uint32_t iters = (ntiles + kLinkWarps - 1) / kLinkWarps;
    const uint32_t head_base = (uint32_t)__cvta_generic_to_shared(s_head);
    const uint32_t spare = head_base + (1u << kHashBits) * 2 + lane * 2;   // the slot of a position that is not entered
    const int bar_in = 1 + warp, bar_out = 1 + (warp + 1) % kLinkWarps;
    // A tile's 8 * kLinkSteps words: word 32 i + lane of the tile in w[i], the word behind the tile in e (every lane).
    auto load = [&](uint32_t t, uint32_t (&w)[kLinkRegs], uint32_t& e) {
        const uint32_t w0 = t * (kLinkTile / 4);
#pragma unroll
        for (int i = 0; i < kLinkRegs; ++i) w[i] = w0 + 32 * i + lane < nwords ? __ldg(words + w0 + 32 * i + lane) : 0u;
        e = w0 + kLinkTile / 4 < nwords ? __ldg(words + w0 + kLinkTile / 4) : 0u;
    };
    // Step k's position 32 k + lane hashes the four bytes that start in word 8 k + lane / 4: that word (from lane
    // 8 (k % 4) + lane / 4 of w[k / 4]) and the next one (from the next lane, where lane 0 stands for the following
    // register, which only the last lanes of every fourth step read).
    const uint32_t src = lane >> 2, shift = (lane & 3) * 8;

    if (warp == kLinkWarps - 1) ring_pass(bar_out);            // lets warp 0 take the first turn
    uint32_t tile = warp;
    uint32_t cur[kLinkRegs], ext;
    load(tile, cur, ext);
    for (uint32_t it = 0; it < iters; ++it, tile += kLinkWarps) {
        uint32_t nxt[kLinkRegs], ext_n;
        load(tile + kLinkWarps, nxt, ext_n);
        const int qb = (int)tile * kLinkTile;
        uint32_t v[kLinkSteps];                                  // the four bytes at each of the lane's positions
#pragma unroll
        for (int i = 0; i < kLinkRegs; ++i) {
            const uint32_t succ = lane == 0 ? (i + 1 < kLinkRegs ? cur[i + 1] : ext) : cur[i];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const uint32_t wa = __shfl_sync(kFullMask, cur[i], src + 8 * r);
                const uint32_t wb = __shfl_sync(kFullMask, succ, (src + 8 * r + 1) & 31);
                v[4 * i + r] = __funnelshift_r(wa, wb, shift);
            }
        }
        // Most tiles lie inside [q_lo, q_hi), are not cut by q_seg, and are more than a window from the stream's start:
        // every position is entered, all or none are stored, and no link can reach in front of the stream.
        const bool inner = qb >= q_lo && qb + kLinkTile <= q_hi &&
                           (qb + kLinkTile <= q_seg || (qb >= q_seg && p_cap + qb >= (int)kWindow));
        auto link = [&](auto edge_tag) {
            constexpr bool kEdge = decltype(edge_tag)::value;
            LinkAddrs ha;
            uint32_t d[kLinkSteps], rd = 0, wmask = 0;
#pragma unroll
            for (int k = 0; k < kLinkSteps; ++k) {
                const int q = qb + 32 * k + lane;
                const bool valid = !kEdge || (q >= q_lo && q < q_hi);
                const uint32_t h = hash4(v[k]);
                ha.a[k] = valid ? head_base + h * 2 : spare;
                if (kExact) {
                    const uint32_t grp = __match_any_sync(kFullMask, valid ? h : 0x10000u + lane);
                    const uint32_t lower = grp & lt;
                    wmask |= (valid && (grp >> lane) == 1u) ? 1u << k : 0u;    // highest lane of its group writes head[]
                    rd |= (valid && lower == 0) ? 1u << k : 0u;                // lowest lane of its group reads head[]
                    d[k] = (valid && lower) ? (uint32_t)(lane - (31 - __clz(lower))) : 0u;
                } else {
                    // Relaxed: positions of one 32-wide step that share a hash all link to the entry from before the
                    // step (a valid, merely older, chain member) and the table keeps whichever of them the hardware
                    // writes last.  No cross-lane grouping (MATCH.ANY saturates the ADU pipe), ~0.1 % larger output.
                    rd |= valid ? 1u << k : 0u;
                    d[k] = 0;
                }
            }
            const LinkHeads hv = ring_turn<kExact>(ha, (uint32_t)(qb + lane), wmask, bar_in, bar_out);
            if (!kEdge && qb < q_seg) return;                    // priming: nothing to store
#pragma unroll
            for (int k = 0; k < kLinkSteps; ++k) {
                const int q = qb + 32 * k + lane;
                if (rd >> k & 1) {
                    if (kEdge) {
                        uint32_t dd = ((uint32_t)q - hv.h[k]) & 0xffffu;
                        if (dd == 0) dd = 0x10000u;
                        d[k] = (dd > kWindow || (int)dd > p_cap + q) ? 0u : dd;
                    } else {                                     // the same test: (dd - 1) mod 2^16 < kWindow
                        const uint32_t dd = (uint32_t)q - hv.h[k];
                        d[k] = (dd - 1u) & kWindow ? 0u : dd;
                    }
                }
                if (!kEdge || (q >= q_seg && q < q_end)) dout[q] = (uint16_t)d[k];
            }
        };
        if (inner) link(std::false_type{});
        else link(std::true_type{});
#pragma unroll
        for (int i = 0; i < kLinkRegs; ++i) cur[i] = nxt[i];
        ext = ext_n;
    }
    if (warp == 0) ring_wait(bar_in);                            // absorb the last hand-off
}

// ------------------------------------------------------------------------------------------
// K1b: match search + parse, one thread per 64-byte sub-unit, window staged in shared memory
// ------------------------------------------------------------------------------------------
// A parse only needs a match where a token starts (one position in three on text), and a kernel with one thread per
// position both searches everywhere and leaves lanes idle while a neighbour extends a match (round 1 measured it:
// 4x the instructions of this kernel).  This kernel works the way deflate_fast / deflate_slow do -- search, emit,
// skip the matched bytes (deflate.c:1448-1674) -- with one thread per 64-byte sub-unit, so every lane is always
// searching a position that matters.
//   * One CTA per 32 KiB block (3 CTAs per SM): the block, the 32 KiB in front of it and 272 bytes of lookahead are staged in
//     shared memory once (16-byte loads); every candidate comparison then reads shared memory.  Only the chain
//     links (dist16) come from global memory; they are L2 hits because the CTAs in flight cover a few tens of MiB.
//   * Sub-units start parsing at their boundary without knowing where the previous sub-unit's last token ends.
//     A match may run past the end of its sub-unit; afterwards a prefix maximum over the threads' end positions
//     gives every thread the frontier it really starts at, and it drops the tokens in front of it -- a match that
//     straddles the frontier is shortened (the tail of a match is a match at the same distance) or, below three
//     bytes, turned into literals.
//   * Tokens go to a private region per thread, then each warp copies its 32 regions into the block's contiguous
//     token array with coalesced stores and tallies the block histogram on the way (dense shared-memory atomics).
// Two shapes: greedy levels run 512 threads (64-byte sub-units) at 3 CTAs per SM with the chain links read from
// global memory (L2); lazy levels walk up to 4096 candidates per search, where every link is a dependent load, so
// they also stage the links of the window (128 KiB more shared memory, one CTA per SM) and run 1024 threads
// (32-byte sub-units).
constexpr int kWalkThreadsFast = 512, kWalkThreadsLazy = 1024;
constexpr uint32_t kSubSlotsMax = 68;                           // token slots per sub-unit incl. four in front (two spare, 16-byte alignment): max over both shapes
constexpr uint32_t kTmpPerBlock = 1024 * 36 > 512 * 68 ? 1024 * 36 : 512 * 68;   // private token slots per block
constexpr uint32_t kWalkPad = 272;                              // lookahead behind the block (kMaxMatch + word slack)
// Shared-memory image of the window: rows of 128 bytes followed by one pad word that repeats the first word of
// the next row.  The lanes of a warp sit 64 bytes apart (one sub-unit each): without the skew they would share two
// banks; with 132-byte rows a pair of lanes shifts by one bank per row and the 32 lanes cover all 32 banks.  An unaligned 4-byte read that starts in the last bytes of a row still finds its continuation in the pad word.
constexpr uint32_t kWalkRows = (kWindow + kBlockBytes + kWalkPad + 16 + 127) / 128 + 1;
constexpr uint32_t kWalkSmem = kWalkRows * 132;
constexpr uint32_t kWalkLinkSmem = (kWindow + kBlockBytes + 16) * 2;   // image of dist16 over the window and the block
__device__ __forceinline__ uint32_t smap(uint32_t off) { return off + ((off >> 7) << 2); }

__device__ __forceinline__ uint32_t lds32u(const uint8_t* s_mem, uint32_t off)   // 4 bytes at any window-image offset
{
    const uint32_t m = smap(off);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(s_mem + (m & ~3u));
    return __funnelshift_r(w[0], w[1], (m & 3u) * 8);
}

struct Found { uint32_t len, dist; };

// longest_match (deflate.c:1027-1168) at window offset `o` (= absolute position gp): candidates from the dist16 chain,
// quick reject on the word that ends at the byte a better match must reach, strictly longer wins, stop at nice.
template <bool kSkipLast>                                       // links in global memory: no load for the last candidate the budget allows
__device__ __forceinline__ Found walk_search(const uint8_t* s_mem, uint32_t o, const uint16_t* dp, uint32_t head, uint32_t maxlen,
                                             int chain, uint32_t nice_eff, uint32_t prev_len, uint32_t max_dist)
{
    Found f{kMinMatch - 1, 0};
    if (prev_len > f.len) f.len = prev_len;                     // deflate_slow: only a longer match is of interest
    uint32_t acc = head;                                        // = dp[0]: the caller may have it cached
    if (acc == 0 || f.len >= maxlen) return f;
    uint32_t qoff = f.len >= 4 ? f.len - 3 : 0u, qmask = f.len >= 3 ? 0xffffffffu : 0xffffffu;
    uint32_t hq = lds32u(s_mem, o + qoff);
    do {
        if (acc > max_dist) break;
        const uint32_t d = (!kSkipLast || chain > 1) ? *(dp - acc) : 0u;   // next link: issued before the compare so that its trip overlaps it
        const uint32_t co = o - acc;
        const uint32_t x = lds32u(s_mem, co + qoff) ^ hq;
        if ((x & qmask) == 0) {
            uint32_t len;
            if (qoff == 0 && x != 0) len = 3;                   // first three agree, the fourth does not
            else {
                len = qoff == 0 ? 4u : 0u;
                while (len < maxlen) {
                    const uint32_t y = lds32u(s_mem, o + len) ^ lds32u(s_mem, co + len);
                    if (y) { len += (uint32_t)(__ffs(y) - 1) >> 3; break; }
                    len += 4;
                }
                len = min(len, maxlen);
            }
            if (len > f.len) {
                f.len = len; f.dist = acc;
                if (len >= nice_eff) break;
                qoff = len >= 4 ? len - 3 : 0u;
                qmask = 0xffffffffu;
                hq = lds32u(s_mem, o + qoff);
            }
        }
        if (d == 0) break;
        acc += d;
    } while (--chain > 0);
    return f;
}

// Z_RLE (deflate.c:1485-1494, 1594-1598): the only candidate is the previous byte, i.e. a match is a run.
__device__ __forceinline__ Found walk_search_rle(const uint8_t* s_mem, uint32_t o, bool has_prev, uint32_t maxlen, uint32_t prev_len)
{
    Found f{kMinMatch - 1, 0};
    if (prev_len > f.len) f.len = prev_len;
    if (!has_prev) return f;
    uint32_t len = 0;
    while (len < maxlen) {
        const uint32_t y = lds32u(s_mem, o + len) ^ lds32u(s_mem, o - 1 + len);
        if (y) { len += (uint32_t)(__ffs(y) - 1) >> 3; break; }
        len += 4;
    }
    len = min(len, maxlen);
    if (len > f.len) { f.len = len; f.dist = 1; }
    return f;
}

template <int kT, bool kSmemLinks>
__global__ void __launch_bounds__(kT, kSmemLinks ? 1 : 3)
k_lz_walk(const uint8_t* __restrict__ buf, uint32_t total, uint32_t dict, const uint16_t* __restrict__ dist16,
          uint32_t* __restrict__ tok_tmp, uint32_t* __restrict__ tok, uint32_t* __restrict__ blk_ntok,
          uint32_t* __restrict__ blk_hist, int kind, int max_chain, uint32_t nice, uint32_t max_lazy, uint32_t good,
          int strategy, uint32_t max_dist, const ChunkDesc* __restrict__ cd, uint32_t nblocks, uint32_t* __restrict__ next_block)
{
    extern __shared__ __align__(16) uint8_t s_mem[];
    __shared__ uint32_t s_hist[kHistSize];
    constexpr uint32_t kFront = kSmemLinks ? 2 : 4;             // spare slots in front of a region; four keep the greedy shape's regions 16-byte aligned
    constexpr uint32_t kSub = kBlockBytes / kT, kSubSlots = kSub + kFront;   // input bytes / private token slots per thread
    __shared__ uint32_t s_end[kT];                    // end position of each thread's walk, then its prefix maximum
    __shared__ uint32_t s_cnt[kT];                    // kept tokens per thread, then their exclusive prefix sum
    __shared__ uint32_t s_first[kT];
    __shared__ uint32_t s_wsum[kT / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // Persistent CTAs: the grid is one CTA per resident slot and every CTA takes the next unclaimed block from a device
    // counter.  The private token regions are indexed by SLOT, not by block: a few tens of MB that are rewritten every
    // ~100 us and stay in L2, instead of one region per block of the slab (half a GB per slab that went out to HBM and
    // came back).
    __shared__ uint32_t s_claim;
    const uint32_t slot = blockIdx.x;
  for (;;) {
    __syncthreads();                                            // the previous block's shared memory is no longer read
    if (tid == 0) s_claim = atomicAdd(next_block, 1u);
    __syncthreads();
    const uint32_t b = s_claim;
    if (b >= nblocks) return;
    uint32_t blk_beg, blk_end, win_beg;                         // absolute positions in buf
    if (cd) {                                                   // job mode: block b is the (b % 4)-th block of a chunk of some job
        const ChunkDesc d = cd[b / kBlocksPerChunk];
        const uint32_t rel = (b % kBlocksPerChunk) * kBlockBytes;
        if (rel >= d.len) continue;                             // short chunk: this block slot is unused (nobody reads it)
        blk_beg = d.beg + rel;
        blk_end = d.beg + min(d.len, rel + kBlockBytes);
        win_beg = blk_beg - d.job_beg > kWindow ? blk_beg - kWindow : d.job_beg;
    } else {
        blk_beg = dict + b * kBlockBytes;
        blk_end = min(total, blk_beg + kBlockBytes);
        win_beg = blk_beg > kWindow ? blk_beg - kWindow : 0u;
    }
    const uint32_t stage_end = min(total, blk_end + kWalkPad);
    // ---- stage [win_beg, stage_end) ----
    const uintptr_t g_lo = (uintptr_t)(buf + win_beg) & ~(uintptr_t)15;
    const uint32_t mis = (uint32_t)((uintptr_t)(buf + win_beg) - g_lo);     // window offset w lives at s_mem[w + mis]
    const uint32_t nvec = (mis + (stage_end - win_beg) + 15) >> 4;
    for (uint32_t i = tid; i < nvec; i += kT) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(g_lo) + i);
        uint32_t* d = reinterpret_cast<uint32_t*>(s_mem + smap(i * 16));    // a 16-byte vector never straddles a row
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    for (int i = tid; i < (int)kHistSize; i += kT) s_hist[i] = 0;
    __syncthreads();
    for (uint32_t r = tid; r + 1 < kWalkRows; r += kT)            // pad word = first word of the next row
        reinterpret_cast<uint32_t*>(s_mem)[r * 33 + 32] = reinterpret_cast<const uint32_t*>(s_mem)[(r + 1) * 33];
    __syncthreads();
    const uint32_t sm_off = mis;                                 // image offset of window offset 0
    const uint16_t* links = dist16 + win_beg;                    // links[q - win_beg] = dist16[q]
    if (kSmemLinks) {
        uint16_t* sl = reinterpret_cast<uint16_t*>(s_mem + kWalkSmem);
        const uintptr_t l_lo = (uintptr_t)(dist16 + win_beg) & ~(uintptr_t)15;
        const uint32_t lmis = (uint32_t)(((uintptr_t)(dist16 + win_beg) - l_lo) >> 1);
        const uint32_t lvec = (lmis + (blk_end - win_beg) + 7) >> 3;
        for (uint32_t i = tid; i < lvec; i += kT)
            reinterpret_cast<uint4*>(sl)[i] = __ldg(reinterpret_cast<const uint4*>(l_lo) + i);
        __syncthreads();
        links = sl + lmis;
    }
    auto byte_at = [&](uint32_t q) { return (uint32_t)s_mem[smap(sm_off + q - win_beg)]; };   // buf[q]

    // ---- level 1: screen every position of the block for a match start ----
    // With a chain budget of one, the search at p is a pure function of p: the head dist16[p] and one 3-byte test.  Four
    // tokens in five are literals at level 1, and in the walk below every lane of a warp pays for the search whenever one
    // lane needs it.  So each warp first tests the 2048 positions of its own 32 sub-units, 32 consecutive positions per
    // ballot (coalesced head loads, every lane busy), and bit r of a thread's 64-bit word is set exactly where the search
    // at s0 + r finds a match.  The walk then emits the literals in front of the next set bit without searching.
    const bool screened = !kSmemLinks && kind == 1 && max_chain == 1 && strategy != 3;
    if constexpr (!kSmemLinks) {
        static_assert(kSub == 64, "one 64-bit word of match starts per sub-unit");
        if (screened) {
            constexpr uint32_t kBatch = 8;                      // head loads in flight per lane
            const uint32_t wbeg = blk_beg + (uint32_t)warp * 32u * kSub;
            for (uint32_t k = 0; k < kSub; k += kBatch) {
                uint32_t hd[kBatch];
#pragma unroll
                for (uint32_t j = 0; j < kBatch; j++) {
                    const uint32_t p = wbeg + 32u * (k + j) + lane;
                    hd[j] = p + kMinMatch <= blk_end ? __ldg(dist16 + p) : 0u;
                }
#pragma unroll
                for (uint32_t j = 0; j < kBatch; j++) {
                    const uint32_t o = sm_off + wbeg + 32u * (k + j) + lane - win_beg;
                    const uint32_t d = hd[j] <= max_dist ? hd[j] : 0u;
                    const bool hit = d != 0 && ((lds32u(s_mem, o) ^ lds32u(s_mem, o - d)) & 0xffffffu) == 0;
                    const uint32_t word = __ballot_sync(kFullMask, hit);
                    if (lane == 0) {                            // the bitmap borrows s_end / s_cnt, idle until the frontier
                        const uint32_t t = warp * 32 + (k + j) / 2;
                        ((k + j) & 1 ? s_cnt : s_end)[t] = word;     // thread t: positions s0..s0+31 in s_end, the rest in s_cnt
                    }
                }
            }
            __syncwarp();
        }
    }

    // ---- walk this thread's sub-unit ----
    const uint32_t s0 = blk_beg + tid * kSub, s1 = min(s0 + kSub, blk_end);
    uint32_t* mine = tok_tmp + (size_t)slot * kTmpPerBlock + (size_t)tid * kSubSlots + kFront;
    uint32_t ntok = 0, pos = s0;
    if (s0 < blk_end) {
        if (kind == 1) {                                        // deflate_fast, deflate.c:1448-1546
            uint32_t held0 = 0, held1 = 0, held2 = 0;           // tokens waiting for the fourth of their group
            // tokens leave four at a time (the private region is 16-byte aligned): a quarter of the store requests to L2
            // (selects, not branches: the lanes of a warp are at different phases)
            auto put = [&](uint32_t tk) {
                const uint32_t ph = ntok & 3u;
                if (ph == 3u) *reinterpret_cast<uint4*>(mine + ntok - 3) = make_uint4(held0, held1, held2, tk);
                held0 = ph == 0u ? tk : held0;
                held1 = ph == 1u ? tk : held1;
                held2 = ph == 2u ? tk : held2;
                ntok++;
            };
            if (screened) {
                // One turn per match: the literals up to the next match start, then the match.  The head of that start is
                // loaded before the literals go out, so its trip to L2 overlaps them.  The screen had that head in a register
                // of another lane; reloading it (0.08 loads per byte) is deliberate: keeping it needs room the 40 registers
                // of three CTAs per SM do not leave.
                const uint32_t n = s1 - s0;
                auto next_start = [&](uint32_t r) -> uint32_t {    // first match start at or after offset r, else n
                    const uint64_t m = r < 64u ? ((uint64_t)s_cnt[tid] << 32 | s_end[tid]) >> r : 0u;
                    return m ? r + (uint32_t)__ffsll((long long)m) - 1u : n;
                };
                uint32_t r = 0, q = next_start(0);
                while (r < n) {
                    const uint32_t head = q < n ? __ldg(dist16 + s0 + q) : 0u;
#pragma unroll 1                                        // unrolled, the literal loop makes the kernel spill
                    for (; r < q; r++) put(byte_at(s0 + r));
                    if (q >= n) break;
                    const uint32_t at = s0 + q, maxlen = min(kMaxMatch, blk_end - at);
                    const Found f = walk_search<true>(s_mem, sm_off + at - win_beg, links + (at - win_beg), head, maxlen, 1,
                                                      min(nice, maxlen), 0, max_dist);
                    put((f.dist << 16) | (f.len - kMinMatch));
                    r = q + f.len;
                    q = next_start(r);
                }
                pos = s0 + r;
            } else {
                // Chain heads of neighbouring positions share a 32-byte sector that L1 (3 % hits: the window image leaves it
                // ~30 KB) has lost by the time the next token starts.  Four of them are kept per thread in the shared arrays
                // of the later phases, which are idle during the walk: one 8-byte load serves up to four token starts.
                s_first[tid] = 0xffffffffu;
                auto head_of = [&](uint32_t q) -> uint32_t {        // dist16[q]
                    const uint32_t g = q >> 2;
                    if (s_first[tid] != g) {
                        const uint2 v = __ldg(reinterpret_cast<const uint2*>(dist16) + g);
                        s_end[tid] = v.x; s_cnt[tid] = v.y; s_first[tid] = g;
                    }
                    const uint32_t w = (q & 2u) ? s_cnt[tid] : s_end[tid];
                    return (q & 1u) ? w >> 16 : w & 0xffffu;
                };
                while (pos < s1) {
                    const uint32_t maxlen = min(kMaxMatch, blk_end - pos);
                    Found f{0, 0};
                    if (maxlen >= kMinMatch && max_chain > 0) {
                        if (strategy == 3) f = walk_search_rle(s_mem, sm_off + pos - win_beg, pos > win_beg, maxlen, 0);
                        else f = walk_search<!kSmemLinks>(s_mem, sm_off + pos - win_beg, links + (pos - win_beg), kSmemLinks ? links[pos - win_beg] : head_of(pos), maxlen, max_chain, min(nice, maxlen), 0, max_dist);
                    }
                    uint32_t tk;
                    if (f.len >= kMinMatch) { tk = (f.dist << 16) | (f.len - kMinMatch); pos += f.len; }
                    else { tk = byte_at(pos); pos++; }
                    put(tk);
                }
            }
            {
                const uint32_t ph = ntok & 3u, at = ntok - ph;
                if (ph > 0) mine[at] = held0;
                if (ph > 1) mine[at + 1] = held1;
                if (ph > 2) mine[at + 2] = held2;
            }
        } else {                                                // deflate_slow, deflate.c:1554-1674
            uint32_t prev_len = kMinMatch - 1, prev_dist = 0;
            bool avail = false;                                 // position pos-1 is pending (as a literal or as prev match)
            for (;;) {
                if (!avail && pos >= s1) break;
                if (avail && pos - 1 >= s1) { pos--; break; }   // the pending position belongs to the next sub-unit: leave it
                Found f{kMinMatch - 1, 0};
                if (pos < blk_end) {
                    const uint32_t maxlen = blk_end - pos < kMaxMatch ? blk_end - pos : kMaxMatch;
                    if (maxlen >= kMinMatch && prev_len < max_lazy) {
                        const int chain = prev_len >= good ? max(max_chain >> 2, 1) : max_chain;
                        if (strategy == 3) f = walk_search_rle(s_mem, sm_off + pos - win_beg, pos > win_beg, maxlen, prev_len);
                        else f = walk_search<!kSmemLinks>(s_mem, sm_off + pos - win_beg, links + (pos - win_beg), links[pos - win_beg], maxlen, chain, min(nice, maxlen), prev_len, max_dist);
                        if (f.dist == 0) f.len = kMinMatch - 1;                  // nothing longer than the pending match
                        if (f.len <= 5 && (strategy == 1 || (f.len == kMinMatch && f.dist > kTooFar))) f.len = kMinMatch - 1;   // Z_FILTERED, TOO_FAR
                    }
                }
                if (prev_len >= kMinMatch && f.len <= prev_len) {               // the pending match wins
                    mine[ntok++] = (prev_dist << 16) | (prev_len - kMinMatch);
                    pos += prev_len - 1;
                    avail = false; prev_len = kMinMatch - 1;
                } else if (avail) {                                             // pending literal goes out, the new match waits
                    mine[ntok++] = byte_at(pos - 1);
                    prev_len = f.len; prev_dist = f.dist;
                    pos++;
                } else {
                    avail = true;
                    prev_len = f.len; prev_dist = f.dist;
                    pos++;
                }
            }
        }
    } else {
        pos = blk_end;
    }
    // ---- frontier: where the tokens of the threads before this one end ----
    {
        uint32_t m = pos;                                       // inclusive prefix maximum: warp scan, then across warps
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) { const uint32_t y = __shfl_up_sync(kFullMask, m, k); if (lane >= k && y > m) m = y; }
        if (lane == 31) s_wsum[warp] = m;
        __syncthreads();
        uint32_t prevmax = 0;
#pragma unroll
        for (int w = 0; w < kT / 32; w++) { const uint32_t v = s_wsum[w]; if (w < warp && v > prevmax) prevmax = v; }
        s_end[tid] = m > prevmax ? m : prevmax;
        __syncthreads();
    }
    const uint32_t front = tid ? s_end[tid - 1] : blk_beg;
    int first = 0;                                              // index of the first kept token (may go to -2)
    if (front > s0) {
        uint32_t q = s0;
        uint32_t i = 0;
        while (i < ntok) {
            const uint32_t t = mine[i];
            const uint32_t l = (t >> 16) ? (t & 0xffffu) + kMinMatch : 1u;
            if (q + l > front) break;
            q += l; i++;
        }
        first = (int)i;
        if (i < ntok && q < front) {                            // a match straddles the frontier: keep its tail
            const uint32_t t = mine[i];
            const uint32_t l = (t & 0xffffu) + kMinMatch, rem = q + l - front;
            if (rem >= kMinMatch) mine[i] = (t & 0xffff0000u) | (rem - kMinMatch);
            else {
                for (uint32_t k = 0; k < rem; k++) mine[(int)i - (int)k] = byte_at(front + (rem - 1 - k));
                first = (int)i - (int)(rem - 1);
            }
        }
    }
    const uint32_t keep = (uint32_t)((int)ntok - first);
    // ---- compact: exclusive prefix sum of the kept counts ----
    uint32_t x = keep;
#pragma unroll
    for (int k = 1; k < 32; k <<= 1) { const uint32_t y = __shfl_up_sync(kFullMask, x, k); if (lane >= k) x += y; }
    if (lane == 31) s_wsum[warp] = x;
    __syncthreads();
    uint32_t before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < kT / 32; w++) { const uint32_t v = s_wsum[w]; if (w < warp) before += v; all += v; }
    // region descriptor for the copy: {first kept slot (index into this block's private slots), output offset | count << 16}
    s_first[tid] = (uint32_t)tid * kSubSlots + (uint32_t)(first + (int)kFront);
    s_cnt[tid] = (before + x - keep) | (keep << 16);             // a block holds at most 32768 tokens, a sub-unit at most 66
    __syncthreads();
    // ---- each warp moves its 32 regions, coalesced, and tallies ----
    uint32_t* out = tok + (size_t)b * kBlockBytes;
    const uint32_t* tmp_blk = tok_tmp + (size_t)slot * kTmpPerBlock;
    auto tally = [&](uint32_t v) {
        const bool is_match = (v >> 16) != 0;
        atomicAdd(&s_hist[is_match ? 257 + len_code(v & 0xffffu) : v], 1u);
        if (is_match) atomicAdd(&s_hist[288 + dist_code((v >> 16) - 1)], 1u);
    };
    for (int r0 = 0; r0 < 32; r0 += 4) {                         // four regions at a time: their loads are in flight together
        uint32_t cnt[4], off[4], src0[4], v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int t = warp * 32 + r0 + j;
            const uint32_t dsc = s_cnt[t];
            cnt[j] = dsc >> 16; off[j] = dsc & 0xffffu; src0[j] = s_first[t];
        }
#pragma unroll
        for (int j = 0; j < 4; j++) v[j] = (uint32_t)lane < cnt[j] ? tmp_blk[src0[j] + lane] : 0u;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if ((uint32_t)lane < cnt[j]) { out[off[j] + lane] = v[j]; tally(v[j]); }
            for (uint32_t k = lane + 32; k < cnt[j]; k += 32) {  // a region holds at most 66 tokens
                const uint32_t w = tmp_blk[src0[j] + k];
                out[off[j] + k] = w; tally(w);
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < (int)kHistSize; i += kT) blk_hist[(size_t)b * kHistSize + i] = s_hist[i];
    if (tid == 0) blk_ntok[b] = all;
  }
}

// ------------------------------------------------------------------------------------------
// K2: length-limited canonical codes per block (trees.c:490-860), block pricing (trees.c:921-1001)
// ------------------------------------------------------------------------------------------
constexpr int kCodeWarps = 4;

__constant__ uint8_t c_bl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct TreeScratch {
    uint32_t hsum[kHistSize];                                   // block histogram
    uint32_t freq[288];                                         // input of the code under construction
    uint32_t key[512];                                          // freq << 9 | symbol, ascending
    uint32_t wint[288];                                         // weights of internal nodes, in creation order
    uint16_t parent[2 * 288];                                   // leaves [0,m) in sorted order, then internal nodes
    uint8_t  idepth[288];
    uint32_t run[16], next_code[16];
    uint16_t bl_count[16];
    uint16_t llen[288 + 2], dlen[32 + 2];                       // +sentinel slot for the run-length scan
    uint16_t blfreq[20], bllen[20], blcode[20];
    uint16_t lcode[288], dcode[32];
    uint16_t items[320];                                        // run-length items of both length arrays, in sending order
    int nitems;
};

struct BitSink {                                                // serial bit writer into global words
    uint32_t* w; uint64_t acc; int n; uint32_t count, total;
    __device__ void put(uint32_t v, int bits)
    {
        acc |= (uint64_t)v << n; n += bits; total += bits;
        if (n >= 32) { w[count++] = (uint32_t)acc; acc >>= 32; n -= 32; }
    }
    __device__ void finish() { if (n > 0) w[count++] = (uint32_t)acc; }
};

__device__ __forceinline__ uint32_t bit_reverse(uint32_t v, int n) { return __brev(v) >> (32 - n); }


// Warp-cooperative replacement for make_code: same optimal total cost (a Huffman tree), built the way a
// GPU likes it -- (1) compact the used symbols with ballots, (2) bitonic sort of (freq, symbol) keys in
// shared memory, (3) the two-queue merge (leaves in sorted order + internal nodes in creation order are
// both already sorted, so each step picks the two smallest heads: O(m), no heap), (4) depths top-down,
// (5) the reference's overflow repair on the length histogram (trees.c:527-545) and lengths handed out
// in frequency order, (6) canonical codes with ranks from match_any.  Steps 3, 4 are one lane; the rest
// uses all 32.  Returns max_code.  All lanes must call it.
__device__ int warp_make_code(TreeScratch* t, int nsym, int max_length, uint16_t* out_len, uint16_t* out_code)
{
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    // (1) used symbols -> keys
    int m = 0, max_code = -1;
    for (int base = 0; base < nsym; base += 32) {
        const int s = base + lane;
        const uint32_t f = s < nsym ? t->freq[s] : 0u;
        const uint32_t used = __ballot_sync(kFullMask, f != 0);
        if (f) t->key[m + __popc(used & lt)] = (f << 9) | (uint32_t)s;
        if (used) max_code = base + 31 - __clz(used);
        m += __popc(used);
        if (s < nsym) out_len[s] = 0;
    }
    while (m < 2) {                                             // force two codes (trees.c:650-656)
        const int n = (max_code < 2 ? ++max_code : 0);
        if (lane == 0) t->key[m] = (1u << 9) | (uint32_t)n;
        m++;
    }
    int P = 32;
    while (P < m) P <<= 1;
    for (int i = m + lane; i < P; i += 32) t->key[i] = 0xffffffffu;
    __syncwarp();
    // (2) bitonic sort, ascending
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = lane; i < P / 2; i += 32) {
                const int a = ((i & ~(j - 1)) << 1) | (i & (j - 1)), b = a | j;
                const uint32_t x = t->key[a], y = t->key[b];
                const bool up = (a & k) == 0;
                if ((x > y) == up) { t->key[a] = y; t->key[b] = x; }
            }
            __syncwarp();
        }
    }
    // (3) two-queue merge, (4) depths of the internal nodes
    if (lane == 0) {
        int i = 0, j = 0;
        uint32_t lw = t->key[0] >> 9, iw = 0xffffffffu;
        for (int ni = 0; ni < m - 1; ni++) {
            uint32_t w = 0;
#pragma unroll
            for (int r = 0; r < 2; r++) {
                if (i < m && (j >= ni || lw <= iw)) {
                    w += lw; t->parent[i] = (uint16_t)(m + ni);
                    i++; lw = i < m ? t->key[i] >> 9 : 0xffffffffu;
                } else {
                    w += iw; t->parent[m + j] = (uint16_t)(m + ni);
                    j++; iw = j < ni ? t->wint[j] : 0xffffffffu;
                }
            }
            t->wint[ni] = w;
            if (j == ni) iw = w;                                 // the node just made is now the head of its queue
        }
        t->idepth[m - 2] = 0;
        for (int q = m - 3; q >= 0; q--) t->idepth[q] = (uint8_t)(t->idepth[t->parent[m + q] - m] + 1);
    }
    if (lane < 16) { t->bl_count[lane] = 0; t->run[lane] = 0; }
    __syncwarp();
    // (5) length histogram, overflow repair, lengths in frequency order
    uint32_t over = 0;
    for (int i = lane; i < m; i += 32) {
        int bits = t->idepth[t->parent[i] - m] + 1;
        if (bits > max_length) { bits = max_length; over++; }
        atomicAdd(&t->run[bits], 1u);
    }
    // the reference counts every node below the limit, internal ones included (their clamped length is what
    // their children see, trees.c:506-512)
    for (int q = lane; q < m - 1; q += 32) over += t->idepth[q] > max_length ? 1u : 0u;
#pragma unroll
    for (int k = 16; k; k >>= 1) over += __shfl_xor_sync(kFullMask, over, k);
    __syncwarp();
    if (lane == 0) {
        uint32_t cnt[16];
        for (int b = 0; b < 16; b++) { cnt[b] = t->run[b]; t->run[b] = 0; }
        int overflow = (int)over;
        while (overflow > 0) {
            int bits = max_length - 1;
            while (cnt[bits] == 0) bits--;
            cnt[bits]--; cnt[bits + 1] += 2; cnt[max_length]--;
            overflow -= 2;
        }
        uint32_t code = 0;
        for (int b = 0; b < 16; b++) t->bl_count[b] = (uint16_t)cnt[b];
        t->next_code[0] = 0;
        for (int b = 1; b <= 15; b++) { code = (code + cnt[b - 1]) << 1; t->next_code[b] = code; }
    }
    __syncwarp();
    for (int i = lane; i < m; i += 32) {                        // leaf i (ascending frequency) gets the i-th longest length
        int L = max_length, cum = t->bl_count[max_length];
        while (cum <= i) { L--; cum += t->bl_count[L]; }
        out_len[t->key[i] & 511u] = (uint16_t)L;
    }
    __syncwarp();
    // (6) canonical codes (trees.c:577-609): code = next_code[len] + rank among symbols of that length
    for (int base = 0; base < nsym; base += 32) {
        const int s = base + lane;
        const uint32_t L = s < nsym ? out_len[s] : 0u;
        const uint32_t grp = __match_any_sync(kFullMask, L);
        const uint32_t rank = t->run[L] + __popc(grp & lt);
        __syncwarp();
        if ((grp & lt) == 0) t->run[L] += __popc(grp);
        __syncwarp();
        if (s < nsym) out_code[s] = L ? (uint16_t)bit_reverse(t->next_code[L] + rank, (int)L) : 0;
    }
    __syncwarp();
    return max_code;
}

// Run-length coding of the code lengths (scan_tree, trees.c:707-748), by the whole warp.  The reference walks the
// lengths once with a little state machine; its output for a maximal run of equal lengths depends on nothing but the
// run itself (the length in front of a maximal run always differs from it, and the limits 7/4, 6/3, 138/3 are set from
// the run's own value), so runs are coded independently: ballots find the run starts, then a lane per run counts its
// items -- zeros: groups of up to 138 (17: 3..10, 18: 11..138, fewer than 3 as literals); others: the length itself
// and "repeat 3..6" for the first group of up to 7 (fewer than 4 as literals), then groups of up to 6 (fewer than 3 as
// literals) -- a warp prefix sum places them, and every lane writes its own.  Items (code-length symbol | extra value
// << 5) are kept so that sending the trees (send_tree, trees.c:752-797) is a loop over them.  ~19 K of the kernel's
// 30 K warp instructions per block were the one-lane form of this walk.
__device__ __forceinline__ uint32_t rl_tail_items(uint32_t r, uint32_t minc) { return r == 0 ? 0u : r < minc ? r : 1u; }

__device__ void warp_walk_lengths(TreeScratch* t, const uint16_t* lens, int max_code, uint32_t* blf /* 19 counters, shared */)
{
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    uint16_t* starts = reinterpret_cast<uint16_t*>(t->key);     // run starts (the sort keys are idle between two codes)
    int nruns = 0;
    for (int base = 0; base <= max_code; base += 32) {
        const int s = base + lane;
        const bool st = s <= max_code && (s == 0 || lens[s] != lens[s - 1]);
        const uint32_t m = __ballot_sync(kFullMask, st);
        if (st) starts[nruns + __popc(m & lt)] = (uint16_t)s;
        nruns += __popc(m);
    }
    __syncwarp();
    int ni = t->nitems;
    for (int r0 = 0; r0 < nruns; r0 += 32) {
        const int r = r0 + lane;
        uint32_t v = 0, L = 0, n_items = 0, first = 0;
        if (r < nruns) {
            const uint32_t a = starts[r], b = r + 1 < nruns ? starts[r + 1] : (uint32_t)max_code + 1u;
            v = lens[a]; L = b - a;
            if (v == 0) n_items = L / 138u + rl_tail_items(L % 138u, 3u);
            else {
                first = L < 7u ? L : 7u;
                const uint32_t rest = L - first;
                n_items = (first < 4u ? first : 2u) + rest / 6u + rl_tail_items(rest % 6u, 3u);
            }
        }
        uint32_t x = n_items;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) { const uint32_t y = __shfl_up_sync(kFullMask, x, k); if (lane >= k) x += y; }
        uint16_t* out = t->items + ni + (x - n_items);
        if (n_items) {
            uint32_t o = 0;
            if (v == 0) {
                uint32_t left = L;
                while (left) {
                    const uint32_t g = left < 138u ? left : 138u;
                    if (g < 3u) { for (uint32_t k = 0; k < g; k++) out[o++] = 0; atomicAdd(&blf[0], g); }
                    else if (g <= 10u) { out[o++] = (uint16_t)(17u | ((g - 3u) << 5)); atomicAdd(&blf[17], 1u); }
                    else { out[o++] = (uint16_t)(18u | ((g - 11u) << 5)); atomicAdd(&blf[18], 1u); }
                    left -= g;
                }
            } else {
                uint32_t lits = 0, reps = 0;
                if (first < 4u) { for (uint32_t k = 0; k < first; k++) out[o++] = (uint16_t)v; lits += first; }
                else { out[o++] = (uint16_t)v; out[o++] = (uint16_t)(16u | ((first - 4u) << 5)); lits++; reps++; }   // the length, then repeat first - 1 times
                uint32_t left = L - first;
                while (left) {
                    const uint32_t g = left < 6u ? left : 6u;
                    if (g < 3u) { for (uint32_t k = 0; k < g; k++) out[o++] = (uint16_t)v; lits += g; }
                    else { out[o++] = (uint16_t)(16u | ((g - 3u) << 5)); reps++; }
                    left -= g;
                }
                atomicAdd(&blf[v], lits);
                if (reps) atomicAdd(&blf[16], reps);
            }
        }
        ni += (int)__shfl_sync(kFullMask, x, 31);
    }
    __syncwarp();
    if (lane == 0) t->nitems = ni;
    __syncwarp();
}

__device__ void send_items(const TreeScratch* t, BitSink* sink)
{
    for (int i = 0; i < t->nitems; i++) {
        const uint32_t it = t->items[i], sym = it & 31u;
        sink->put(t->blcode[sym], t->bllen[sym]);
        if (sym >= 16) sink->put(it >> 5, sym == 16 ? 2 : sym == 17 ? 3 : 7);
    }
}

__device__ __forceinline__ uint32_t fixed_lit_len(uint32_t s) { return s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8; }
__device__ __forceinline__ uint32_t fixed_lit_code(uint32_t s)
{
    const uint32_t c = s < 144 ? 0x30 + s : s < 256 ? 0x190 + (s - 144) : s < 280 ? (s - 256) : 0xC0 + (s - 280);
    return bit_reverse(c, (int)fixed_lit_len(s));
}

__global__ void __launch_bounds__(kCodeWarps * 32)
k_huff_build(uint64_t n, BlockMeta* __restrict__ blk, const uint32_t* __restrict__ blk_hist,
             uint32_t* __restrict__ blk_codes, uint32_t* __restrict__ blk_hdr, int force_fixed,
             const ChunkDesc* __restrict__ cd, uint64_t nslots)
{
    __shared__ TreeScratch s_t[kCodeWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t nblocks = cd ? nslots : (n + kBlockBytes - 1) / kBlockBytes;
    const uint64_t b = (uint64_t)blockIdx.x * kCodeWarps + warp;
    if (b >= nblocks) return;
    TreeScratch* t = &s_t[warp];
    uint32_t* codes = blk_codes + b * kHistSize;
    uint32_t in_len;
    if (cd) {                                                   // job mode: four block slots per chunk, short chunks leave some unused
        const uint32_t clen = cd[b / kBlocksPerChunk].len, rel = (uint32_t)(b % kBlocksPerChunk) * kBlockBytes;
        if (rel >= clen) return;
        in_len = min(kBlockBytes, clen - rel);
    } else {
        in_len = (uint32_t)min((uint64_t)kBlockBytes, n - b * kBlockBytes);
    }

    // ---- block histogram (+ the end-of-block symbol) ----
    for (int i = lane; i < (int)kHistSize; i += 32) t->hsum[i] = blk_hist[b * kHistSize + i] + (i == 256 ? 1u : 0u);
    __syncwarp();
    // ---- literal/length and distance codes ----
    for (int i = lane; i < 286; i += 32) t->freq[i] = t->hsum[i];
    __syncwarp();
    const int lmax = warp_make_code(t, 286, 15, t->llen, t->lcode);
    if (lane < 30) t->freq[lane] = t->hsum[288 + lane];
    __syncwarp();
    const int dmax = warp_make_code(t, 30, 15, t->dlen, t->dcode);

    // ---- cost of the data under the dynamic and the fixed code (all lanes) ----
    uint32_t dyn = 0, fix = 0;
    for (int s = lane; s < 286; s += 32) {
        const uint32_t f = t->hsum[s];
        const uint32_t x = s >= 257 ? len_extra_bits((uint32_t)s - 257) : 0;
        dyn += f * (t->llen[s] + x); fix += f * (fixed_lit_len((uint32_t)s) + x);
    }
    if (lane < 30) {
        const uint32_t f = t->hsum[288 + lane], x = dist_extra_bits((uint32_t)lane);
        dyn += f * (t->dlen[lane] + x); fix += f * (5 + x);
    }
#pragma unroll
    for (int k = 16; k; k >>= 1) { dyn += __shfl_xor_sync(kFullMask, dyn, k); fix += __shfl_xor_sync(kFullMask, fix, k); }

    // ---- code-length code and header ----
    uint32_t* blf = t->wint;                                    // 19 counters (the internal-node weights are idle here)
    if (lane < 19) blf[lane] = 0;
    if (lane == 0) t->nitems = 0;
    __syncwarp();
    warp_walk_lengths(t, t->llen, lmax, blf);
    warp_walk_lengths(t, t->dlen, dmax, blf);
    if (lane < 19) { t->blfreq[lane] = (uint16_t)blf[lane]; t->freq[lane] = blf[lane]; }
    __syncwarp();
    warp_make_code(t, 19, 7, t->bllen, t->blcode);
    uint32_t type = 0;
    if (lane == 0) {
        uint32_t body = 0, hdr_bits = 0;
        int max_bl = 18;
        while (max_bl >= 3 && t->bllen[c_bl_order[max_bl]] == 0) max_bl--;
        uint32_t tree_bits = 14 + 3 * (max_bl + 1);
        for (int i = 0; i < 19; i++) tree_bits += t->blfreq[i] * (t->bllen[i] + (i == 16 ? 2 : i == 17 ? 3 : i == 18 ? 7 : 0));
        const uint32_t opt_len = dyn + tree_bits, static_len = fix;
        uint32_t opt_lenb = (opt_len + 3 + 7) >> 3;
        const uint32_t static_lenb = (static_len + 3 + 7) >> 3;
        if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
        // a stored block holds at most 65535 bytes: a block of 64 KiB or more would go out as two (5 more bytes)
        if (in_len + 4 + (in_len > 65535u ? 5u : 0u) <= opt_lenb && !force_fixed) { type = 0; body = 0; }
        else if (static_lenb == opt_lenb || force_fixed) { type = 1; body = static_len; }
        else {
            type = 2; body = opt_len;
            BitSink sink{blk_hdr + b * kHdrWords, 0, 0, 0, 0};
            sink.put((uint32_t)lmax + 1 - 257, 5); sink.put((uint32_t)dmax + 1 - 1, 5); sink.put((uint32_t)max_bl + 1 - 4, 4);
            for (int r = 0; r <= max_bl; r++) sink.put(t->bllen[c_bl_order[r]], 3);
            send_items(t, &sink);
            sink.finish();
            hdr_bits = sink.total;
        }
        blk[b] = BlockMeta{in_len, type, body, hdr_bits};
    }
    type = __shfl_sync(kFullMask, type, 0);
    __syncwarp();
    // ---- code tables for the packer: code | len << 16 ----
    for (int s = lane; s < 288; s += 32) {
        uint32_t v;
        if (type == 1) v = fixed_lit_code((uint32_t)s) | (fixed_lit_len((uint32_t)s) << 16);
        else v = s < 286 ? (t->lcode[s] | ((uint32_t)(t->llen[s] & 0xff) << 16)) : 0;
        codes[s] = v;
    }
    {
        uint32_t v;
        if (type == 1) v = bit_reverse((uint32_t)lane, 5) | (5u << 16);
        else v = lane < 30 ? (t->dcode[lane] | ((uint32_t)(t->dlen[lane] & 0xff) << 16)) : 0;
        codes[288 + lane] = v;
    }
}

// ------------------------------------------------------------------------------------------
// plan + scan: exact chunk sizes and offsets
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t stored_chunk_bytes(uint32_t len) { return (uint64_t)len + 5ull * ((len + 65534u) / 65535u); }

// bits: low byte = bits pending in front of chunk 0 (deflatePrime, or what a Z_PARTIAL_FLUSH left over), bit 8 = the last
// chunk ends with the ten bits of _tr_align (trees.c:892) instead of the byte-aligning marker and keeps its last bits.
__global__ void k_plan(uint64_t nchunks, uint64_t n, ChunkMeta* __restrict__ chunks, const BlockMeta* __restrict__ blk,
                       int last_is_final, int force_stored, int force_mark, const ChunkDesc* __restrict__ cd, uint32_t bitmode)
{
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchunks) return;
    ChunkMeta cm;
    const uint32_t clen = cd ? cd[c].len : (uint32_t)min((uint64_t)kChunk, n - c * kChunk);
    cm.nblocks = (clen + kBlockBytes - 1) / kBlockBytes;
    cm.offset = 0;
    const bool final_chunk = cd ? cd[c].last != 0 : (last_is_final && c == nchunks - 1);
    const bool mark = !cd && force_mark && !last_is_final && c == nchunks - 1;   // Z_SYNC_FLUSH marker wanted regardless
    const uint32_t prime = (!cd && c == 0) ? (bitmode & 7u) : 0u;
    const bool partial = !cd && (bitmode & 0x100u) && !last_is_final && c == nchunks - 1;
    uint64_t bytes;
    if (force_stored) {
        cm.stored = 1; bytes = stored_chunk_bytes(clen) + (mark ? 5 : 0);
    } else {
        uint64_t bits = prime;
        bool ends_stored = false;
        for (uint32_t j = 0; j < cm.nblocks; j++) {
            const BlockMeta bm = blk[c * kBlocksPerChunk + j];
            if (bm.type == 0) {
                bits = ((bits + 3 + 7) & ~7ull) + 32 + 8ull * bm.in_len; ends_stored = true;
                if (bm.in_len > 65535u) bits += 8 + 32;         // second stored block: header byte, LEN, NLEN
            }
            else { bits += 3 + bm.body_bits; ends_stored = false; }
        }
        if (partial) bytes = (bits + 10) >> 3;                  // empty static block; the last (bits + 10) & 7 bits stay pending
        else if (final_chunk || (ends_stored && !mark)) bytes = (bits + 7) >> 3;
        else bytes = ((bits + 3 + 7) >> 3) + 4;                 // empty stored block: 000, pad, 00 00 FF FF
        const uint64_t sb = stored_chunk_bytes(clen) + (mark ? 5 : 0);
        cm.stored = (sb <= bytes && !prime && !partial) ? 1u : 0u;   // the all-stored shortcut writes whole bytes only
        if (cm.stored) bytes = sb;
    }
    cm.bytes = bytes;
    chunks[c] = cm;
}

// single CTA: exclusive prefix sum of chunk sizes starting at (*start_ptr or 0) + start_add; end[0] = where
// the next slab starts
__global__ void __launch_bounds__(1024) k_scan(uint64_t nchunks, ChunkMeta* __restrict__ chunks,
                                               const uint64_t* __restrict__ start_ptr, uint64_t start_add,
                                               uint64_t* __restrict__ end)
{
    __shared__ uint64_t s_w[32];
    __shared__ uint64_t s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = (start_ptr ? start_ptr[0] : 0) + start_add;
    __syncthreads();
    for (uint64_t i0 = 0; i0 < nchunks; i0 += 1024) {
        const uint64_t i = i0 + threadIdx.x;
        const uint64_t v = i < nchunks ? chunks[i].bytes : 0;
        uint64_t x = v;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) { const uint64_t y = __shfl_up_sync(kFullMask, x, k); if (lane >= k) x += y; }
        if (lane == 31) s_w[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = s_w[lane];
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) { const uint64_t y = __shfl_up_sync(kFullMask, w, k); if (lane >= k) w += y; }
            s_w[lane] = w;
        }
        __syncthreads();
        const uint64_t carry = s_carry;
        const uint64_t incl = x + (warp ? s_w[warp - 1] : 0);
        if (i < nchunks) chunks[i].offset = carry + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) end[0] = s_carry;
}

// Job mode: the chunks of a slab belong to many independent streams, each with its own output slot.  Single CTA:
// (1) exclusive prefix sum of the chunk sizes over the slab, (2) per job: payload size = span of its chunks, total =
// header + payload + trailer, (3) chunk offset = slot + header + (prefix - prefix of the job's first chunk).
__global__ void __launch_bounds__(1024) k_scan_jobs(uint32_t nchunks, ChunkMeta* __restrict__ chunks,
                                                    const ChunkDesc* __restrict__ cd, const JobDesc* __restrict__ jobs,
                                                    uint32_t njobs, uint32_t hdr_len, uint32_t trailer_len,
                                                    JobResult* __restrict__ jres)
{
    __shared__ uint64_t s_w[32];
    __shared__ uint64_t s_carry;
    __shared__ uint64_t s_base[kSlabChunks];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t i0 = 0; i0 < nchunks; i0 += 1024) {
        const uint32_t i = i0 + threadIdx.x;
        const uint64_t v = i < nchunks ? chunks[i].bytes : 0;
        uint64_t x = v;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) { const uint64_t y = __shfl_up_sync(kFullMask, x, k); if (lane >= k) x += y; }
        if (lane == 31) s_w[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = s_w[lane];
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) { const uint64_t y = __shfl_up_sync(kFullMask, w, k); if (lane >= k) w += y; }
            s_w[lane] = w;
        }
        __syncthreads();
        const uint64_t carry = s_carry;
        const uint64_t incl = x + (warp ? s_w[warp - 1] : 0);
        if (i < nchunks) chunks[i].offset = carry + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + incl;
        __syncthreads();
    }
    for (uint32_t j = threadIdx.x; j < njobs; j += 1024) {
        const JobDesc jd = jobs[j];
        uint64_t base = 0, payload = 2;                         // empty input: 03 00 (k_frame_jobs writes it)
        if (jd.nchunks) {
            const ChunkMeta last = chunks[jd.first_chunk + jd.nchunks - 1];
            base = chunks[jd.first_chunk].offset;
            payload = last.offset + last.bytes - base;
        }
        s_base[j] = base;
        jres[j].total = hdr_len + payload + trailer_len;
        jres[j].err = 0;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nchunks; i += 1024) {
        const uint32_t j = cd[i].job;
        chunks[i].offset = jobs[j].dst_off + hdr_len + (chunks[i].offset - s_base[j]);
    }
}

// ------------------------------------------------------------------------------------------
// stream framing: header and trailer (deflate.c:577-650, 832-850)
// ------------------------------------------------------------------------------------------
__host__ __device__ constexpr uint32_t frame_header_len(int wrap)
{
    return wrap == ZB200_WRAP_ZLIB ? 2 : wrap == ZB200_WRAP_GZIP ? 10 : wrap == kWrapBgzf ? kBgzfHeader : 0;
}
__host__ __device__ constexpr uint32_t frame_trailer_len(int wrap)
{
    return wrap == ZB200_WRAP_ZLIB ? 4 : (wrap == ZB200_WRAP_GZIP || wrap == kWrapBgzf) ? 8 : 0;
}

// zlib or gzip header (BGZF's is written by k_frame_jobs); Z_HUFFMAN_ONLY and above report the fastest level
__device__ __forceinline__ void write_frame_header(uint8_t* o, int wrap, int level, int strat)
{
    if (wrap == ZB200_WRAP_ZLIB) {
        const uint32_t fl = (level < 2 || strat >= 2) ? 0 : level < 6 ? 1 : level == 6 ? 2 : 3;   // deflate.c:628-636
        uint32_t h = (0x78u << 8) | (fl << 6);
        h += 31 - h % 31;
        o[0] = h >> 8; o[1] = h;
    } else if (wrap == ZB200_WRAP_GZIP) {
        const uint8_t g[10] = {31, 139, 8, 0, 0, 0, 0, 0, (uint8_t)(level == 9 ? 2 : (level < 2 || strat >= 2) ? 4 : 0), 3};   // deflate.c:590-593
        for (int i = 0; i < 10; i++) o[i] = g[i];
    }
}

// The trailer in front of `end`.  zlib: big-endian Adler-32; gzip and BGZF: CRC-32, then the input length mod 2^32.
__device__ __forceinline__ void write_frame_trailer(uint8_t* end, int wrap, uint32_t crc, uint32_t adler, uint64_t len)
{
    if (wrap == ZB200_WRAP_ZLIB) {
        uint8_t* t = end - 4;
        t[0] = adler >> 24; t[1] = adler >> 16; t[2] = adler >> 8; t[3] = adler;
    } else if (wrap == ZB200_WRAP_GZIP || wrap == kWrapBgzf) {
        uint8_t* t = end - 8;
        for (int i = 0; i < 4; i++) t[i] = crc >> (8 * i);
        for (int i = 0; i < 4; i++) t[4 + i] = (uint8_t)(len >> (8 * i));
    }
}

// Job mode: header and trailer of every stream of the slab, one thread per job.
__global__ void k_frame_jobs(uint8_t* __restrict__ out, const JobDesc* __restrict__ jobs, uint32_t njobs,
                             const uint32_t* __restrict__ crc, const uint32_t* __restrict__ adler, int level, int wrap,
                             int strat, JobResult* __restrict__ jres)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= njobs) return;
    const JobDesc jd = jobs[j];
    const uint32_t cr = crc[j], ad = adler[j];
    jres[j].crc = cr; jres[j].adler = ad;
    const uint64_t total = jres[j].total;
    if (total > jd.dst_cap) return;
    uint8_t* o = out + jd.dst_off;
    if (wrap == kWrapBgzf) {                                    // htslib's bgzf.c header bytes; BSIZE is known only here
        const uint8_t g[16] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0};
        for (int i = 0; i < 16; i++) o[i] = g[i];
        o[16] = (uint8_t)(total - 1); o[17] = (uint8_t)((total - 1) >> 8);   // total > 65536 is refused by the caller
    } else {
        write_frame_header(o, wrap, level, strat);
    }
    if (jd.nchunks == 0) { const uint32_t hl = frame_header_len(wrap); o[hl] = 3; o[hl + 1] = 0; }
    write_frame_trailer(o + total, wrap, cr, ad, jd.src_len);
}

// ------------------------------------------------------------------------------------------
// K3: bit packing
// ------------------------------------------------------------------------------------------
constexpr int kPackThreads = 256;
constexpr int kPackRun = 8;                                     // consecutive symbols of a block that one thread encodes per round
constexpr int kStageWords = (kPackThreads * kPackRun * 48 + 64) / 32 + 4;   // kPackRun symbols of <= 48 bits per thread and round

struct Packer {
    uint32_t* stage;                                            // two shared staging windows, used alternately; bit 0 of the
    uint32_t par;                                               // current one (0/1) = first unwritten bit of byte `bytepos`
    uint32_t* warp_sums;                                        // shared, kPackThreads/32 entries
    uint8_t* dst;                                               // chunk output
    uint64_t bytepos;                                           // bytes already written to dst
    uint32_t carry_bits;                                        // bits pending in word 0 of the current window (0..7)
    uint32_t prev_words;                                        // words of the other window that the previous round dirtied

    __device__ __forceinline__ void put(uint32_t* st, uint32_t off, uint64_t value)
    {
        const uint32_t sh = off & 31, wi = off >> 5;
        const uint64_t lo = value << sh;
        atomicOr(&st[wi], (uint32_t)lo);
        const uint32_t mid = (uint32_t)(lo >> 32);
        if (mid) atomicOr(&st[wi + 1], mid);
        if (sh) { const uint32_t hi = (uint32_t)(value >> (64 - sh)); if (hi) atomicOr(&st[wi + 2], hi); }
    }

    // Where this thread's `nbits` start in the current window (bits are appended in thread order) and how many bits the
    // CTA adds in this round.  One barrier.
    __device__ __forceinline__ uint32_t place(uint32_t nbits, uint32_t& total)
    {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        uint32_t x = nbits;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) { const uint32_t y = __shfl_up_sync(kFullMask, x, k); if (lane >= k) x += y; }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        // the eight warp sums: every warp scans them with three shuffles (lanes 0..7 hold one each) instead of reading all eight
        static_assert(kPackThreads / 32 == 8, "the cross-warp scan below is written for eight warps");
        uint32_t ws = warp_sums[lane & 7];
#pragma unroll
        for (int k = 1; k < 8; k <<= 1) { const uint32_t y = __shfl_up_sync(kFullMask, ws, k, 8); if ((lane & 7) >= k) ws += y; }
        total = __shfl_sync(kFullMask, ws, 7);
        const uint32_t upto = __shfl_sync(kFullMask, ws, warp ? warp - 1 : 0);
        return carry_bits + (warp ? upto : 0u) + x - nbits;
    }

    // Second barrier of a round: the window written in this round goes out -- bytes up to the output's next 4-byte
    // boundary, whole words (read across two window words), the last bytes -- and the other window (drained one round
    // ago) is cleared for the next round meanwhile.
    __device__ __forceinline__ void finish(uint32_t total)
    {
        uint32_t* cur = stage + par * kStageWords;
        uint32_t* oth = stage + (par ^ 1u) * kStageWords;
        __syncthreads();
        const uint32_t tbits = carry_bits + total, nbytes = tbits >> 3;
        const uint8_t* sb = reinterpret_cast<const uint8_t*>(cur);
        uint8_t* d = dst + bytepos;
        const uint32_t head = min(nbytes, (0u - (uint32_t)reinterpret_cast<uintptr_t>(d)) & 3u);
        if (threadIdx.x < head) d[threadIdx.x] = sb[threadIdx.x];
        const uint32_t nw = (nbytes - head) >> 2;
        for (uint32_t i = threadIdx.x; i < nw; i += kPackThreads) {
            const uint32_t bo = head + 4 * i;
            *reinterpret_cast<uint32_t*>(d + bo) = __funnelshift_r(cur[bo >> 2], cur[(bo >> 2) + 1], (bo & 3u) * 8);
        }
        const uint32_t done = head + 4 * nw;
        if (threadIdx.x < nbytes - done) d[done + threadIdx.x] = sb[done + threadIdx.x];
        const uint32_t tail = (tbits & 7) ? sb[nbytes] : 0u;
        for (uint32_t i = threadIdx.x; i < prev_words; i += kPackThreads) oth[i] = i == 0 ? tail : 0u;   // word 0 carries the pending bits over
        prev_words = min((tbits + 31) / 32 + 2, (uint32_t)kStageWords);
        bytepos += nbytes; carry_bits = tbits & 7;
        par ^= 1;
    }

    // Every thread contributes two symbols (value, nbits <= 48 each); bits are appended in thread order, a thread's
    // first symbol before its second.  Used for headers, stored blocks and chunk ends.
    __device__ void round(uint64_t v0, uint32_t n0, uint64_t v1 = 0, uint32_t n1 = 0)
    {
        uint32_t* cur = stage + par * kStageWords;
        uint32_t total;
        const uint32_t off = place(n0 + n1, total);
        if (n0) put(cur, off, v0);
        if (n1) put(cur, off + n0, v1);
        finish(total);
    }

    // Every thread contributes kPackRun consecutive symbols (value <= 48 bits, length in the top byte of the word).  The
    // thread strings them together in a 64-bit accumulator and hands out whole words: the first word it touches and the
    // last are shared with its neighbours (shared-memory atomic OR), the words between are its own (plain stores).
    __device__ void round_run(const uint64_t (&sym)[kPackRun])
    {
        uint32_t* cur = stage + par * kStageWords;
        uint32_t nbits = 0;
#pragma unroll
        for (int k = 0; k < kPackRun; k++) nbits += (uint32_t)(sym[k] >> 56);
        uint32_t total;
        const uint32_t off = place(nbits, total);
        uint32_t wi = off >> 5, fill = off & 31;
        uint64_t acc = 0;
        bool shared_word = true;
        auto push = [&](uint32_t val, uint32_t nb) {            // nb <= 24, fill < 32 on entry and on exit
            acc |= (uint64_t)val << fill;
            fill += nb;
            if (fill >= 32) {
                if (shared_word) { atomicOr(&cur[wi], (uint32_t)acc); shared_word = false; }
                else cur[wi] = (uint32_t)acc;
                wi++; acc >>= 32; fill -= 32;
            }
        };
#pragma unroll
        for (int k = 0; k < kPackRun; k++) {
            const uint32_t nb = (uint32_t)(sym[k] >> 56);
            push((uint32_t)sym[k] & 0xffffffu, min(nb, 24u));
            if (nb > 24) push((uint32_t)(sym[k] >> 24) & 0xffffffu, nb - 24);
        }
        if ((uint32_t)acc) atomicOr(&cur[wi], (uint32_t)acc);
        finish(total);
    }
};

__global__ void __launch_bounds__(kPackThreads)
k_huff_pack(const uint8_t* __restrict__ src, uint64_t n, const uint32_t* __restrict__ tok,
            const uint32_t* __restrict__ blk_ntok, const BlockMeta* __restrict__ blk,
            const uint32_t* __restrict__ blk_codes, const uint32_t* __restrict__ blk_hdr,
            const ChunkMeta* __restrict__ chunks, uint8_t* __restrict__ out, uint64_t cap, int last_is_final,
            int force_mark, uint32_t* __restrict__ err, const ChunkDesc* __restrict__ cd, const JobDesc* __restrict__ jobs,
            JobResult* __restrict__ jres, uint32_t bitmode, uint32_t prime_val, uint32_t* __restrict__ tail_out)
{
    __shared__ uint32_t s_stage[2][kStageWords];
    __shared__ uint32_t s_sums[kPackThreads / 32];
    __shared__ uint32_t s_codes[kHistSize];
    __shared__ uint32_t s_len[256];                             // match length - 3 -> code and extra bits | their count << 24
    const uint64_t c = blockIdx.x;
    const uint64_t nchunks = gridDim.x;
    const ChunkMeta cm = chunks[c];
    uint64_t cbeg; uint32_t clen; bool final_chunk, mark, partial = false;
    uint32_t prime = 0;
    if (cd) {                                                   // job mode: the chunk's place and role come from the table
        const ChunkDesc d = cd[c];
        if (jres[d.job].total > jobs[d.job].dst_cap) return;    // the job does not fit its slot: Z_BUF_ERROR from the total
        cbeg = d.beg; clen = d.len; final_chunk = d.last != 0; mark = false;
        err = &jres[d.job].err;
    } else {
        if (cm.offset + cm.bytes > cap) return;                 // caller reports Z_BUF_ERROR from the total
        cbeg = c * kChunk;
        clen = (uint32_t)min((uint64_t)kChunk, n - cbeg);
        final_chunk = last_is_final && c == nchunks - 1;
        mark = force_mark && !last_is_final && c == nchunks - 1;
        prime = c == 0 ? (bitmode & 7u) : 0u;
        partial = (bitmode & 0x100u) && !last_is_final && c == nchunks - 1;
    }
    uint8_t* dst = out + cm.offset;
    const uint8_t* in = src + cbeg;

    if (cm.stored) {                                            // deflate_stored / _tr_stored_block (trees.c:867)
        uint32_t done = 0; uint64_t o = 0;
        while (done < clen) {
            const uint32_t len = min(65535u, clen - done);
            const bool lastb = final_chunk && done + len == clen;
            if (threadIdx.x == 0) {
                dst[o] = lastb ? 1 : 0;
                dst[o + 1] = (uint8_t)len; dst[o + 2] = (uint8_t)(len >> 8);
                dst[o + 3] = (uint8_t)~len; dst[o + 4] = (uint8_t)(~len >> 8);
            }
            for (uint32_t i = threadIdx.x; i < len; i += kPackThreads) dst[o + 5 + i] = in[done + i];
            o += 5 + len; done += len;
        }
        if (mark && threadIdx.x == 0) { dst[o] = 0; dst[o + 1] = 0; dst[o + 2] = 0; dst[o + 3] = 0xff; dst[o + 4] = 0xff; }
        return;
    }

    for (int i = threadIdx.x; i < 2 * kStageWords; i += kPackThreads) (&s_stage[0][0])[i] = 0;
    __syncthreads();
    if (prime && threadIdx.x == 0) s_stage[0][0] = prime_val & ((1u << prime) - 1u);   // bits that precede this shard's first block
    __syncthreads();
    Packer pk{&s_stage[0][0], 0, s_sums, dst, 0, prime, 1};
    bool ends_stored = false;
    for (uint32_t j = 0; j < cm.nblocks; j++) {
        const uint64_t b = c * kBlocksPerChunk + j;
        const BlockMeta bm = blk[b];
        const uint32_t bfinal = (final_chunk && j == cm.nblocks - 1) ? 1u : 0u;
        const uint32_t in_start = j * kBlockBytes;
        if (bm.type == 0) {
            // 3 header bits, pad to a byte, LEN, NLEN, then the raw bytes; at most 65535 bytes per stored block
            for (uint32_t done = 0; done < bm.in_len;) {
                const uint32_t len = min(65535u, bm.in_len - done);
                const uint32_t fin = (bfinal && done + len == bm.in_len) ? 1u : 0u;
                const uint32_t pad = (8 - ((pk.carry_bits + 3) & 7)) & 7;
                uint64_t v = 0; uint32_t nb = 0;
                if (threadIdx.x == 0) { v = fin; nb = 3 + pad; }
                else if (threadIdx.x == 1) { v = (len & 0xffffu) | ((~len & 0xffffu) << 16); nb = 32; }
                pk.round(v, nb);
                for (uint32_t i = threadIdx.x; i < len; i += kPackThreads) dst[pk.bytepos + i] = in[in_start + done + i];
                pk.bytepos += len;
                done += len;
            }
            ends_stored = true;
            continue;
        }
        ends_stored = false;
        for (int i = threadIdx.x; i < (int)kHistSize; i += kPackThreads) s_codes[i] = blk_codes[b * kHistSize + i];
        __syncthreads();
        {   // the length part of a match in one lookup (published by the barriers of the header round)
            static_assert(kPackThreads == 256, "one thread per match length");
            const uint32_t l = threadIdx.x, lc = len_code(l), le = len_extra_bits(lc);
            const uint32_t e = s_codes[257 + lc];
            s_len[l] = (e & 0xffffu) | ((l & ((1u << le) - 1u)) << (e >> 16)) | (((e >> 16) + le) << 24);
        }
        {   // block header: 3 bits, then the serialised trees of a dynamic block
            const uint32_t hw = bm.type == 2 ? (bm.hdr_bits + 31) / 32 : 0;
            const uint32_t* hdr = blk_hdr + b * kHdrWords;
            uint64_t v = 0; uint32_t nb = 0;
            if (threadIdx.x == 0) { v = bfinal | (bm.type << 1); nb = 3; }
            else if (threadIdx.x <= hw) {
                const uint32_t i = threadIdx.x - 1;
                v = hdr[i]; nb = (i == hw - 1 && (bm.hdr_bits & 31)) ? (bm.hdr_bits & 31) : 32;
            }
            pk.round(v, nb);                                    // also publishes s_codes (barrier inside)
        }
        const uint32_t* t = tok + b * kBlockBytes;
        const uint32_t cnt = blk_ntok[b];
        auto encode = [&](uint32_t i, uint32_t tk) -> uint64_t {   // symbol i of the block: token, or end-of-block; bits | count << 56
            if (i < cnt) {
                const uint32_t dist = tk >> 16;
                if (dist == 0) {
                    const uint32_t e = s_codes[tk & 0xff];
                    return (uint64_t)(e & 0xffffu) | ((uint64_t)(e >> 16) << 56);
                }
                // length part (<= 20 bits) from its table, distance part (<= 28 bits) composed in 32 bits, then joined once
                const uint32_t le = s_len[tk & 0xff], lbits = le >> 24;
                const uint32_t d = dist - 1, dc = dist_code(d), de = dist_extra_bits(dc);
                const uint32_t f = s_codes[288 + dc];
                const uint32_t dpart = (f & 0xffffu) | ((d & ((1u << de) - 1u)) << (f >> 16)), dbits = (f >> 16) + de;
                return (uint64_t)(le & 0xffffffu) | ((uint64_t)dpart << lbits) | ((uint64_t)(lbits + dbits) << 56);
            }
            if (i == cnt) {
                const uint32_t e = s_codes[256];                // end of block
                return (uint64_t)(e & 0xffffu) | ((uint64_t)(e >> 16) << 56);
            }
            return 0;
        };
        static_assert(kPackRun == 8, "a thread's run is loaded as two 16-byte groups");
        for (uint32_t i0 = 0; i0 <= cnt; i0 += kPackRun * kPackThreads) {
            const uint32_t i = i0 + kPackRun * threadIdx.x;
            uint4 ta = make_uint4(0, 0, 0, 0), tb = ta;         // the block's token array holds kBlockBytes slots: a group that starts below cnt lies inside it
            if (i < cnt) ta = *reinterpret_cast<const uint4*>(t + i);
            if (i + 4 < cnt) tb = *reinterpret_cast<const uint4*>(t + i + 4);
            uint64_t sym[kPackRun];
            sym[0] = encode(i, ta.x); sym[1] = encode(i + 1, ta.y); sym[2] = encode(i + 2, ta.z); sym[3] = encode(i + 3, ta.w);
            sym[4] = encode(i + 4, tb.x); sym[5] = encode(i + 5, tb.y); sym[6] = encode(i + 6, tb.z); sym[7] = encode(i + 7, tb.w);
            pk.round_run(sym);
        }
    }
    // end of chunk: partial flush -> empty static block, bits left as they fall; final -> pad; otherwise empty stored
    // block unless already byte-aligned by a stored block
    if (partial) {
        pk.round(threadIdx.x == 0 ? 2u : 0u, threadIdx.x == 0 ? 10u : 0u);      // 010 (static, not final) + the 7-bit end-of-block code
        if (threadIdx.x == 0) {
            tail_out[0] = pk.carry_bits | ((pk.stage[pk.par * kStageWords] & ((1u << pk.carry_bits) - 1u)) << 8);
            if (pk.bytepos != cm.bytes) atomicAdd(err, 1u);
        }
        return;
    }
    if (final_chunk || (ends_stored && !mark)) {
        const uint32_t pad = (8 - (pk.carry_bits & 7)) & 7;
        pk.round(0, threadIdx.x == 0 ? pad : 0);
    } else {
        const uint32_t pad = (8 - ((pk.carry_bits + 3) & 7)) & 7;
        uint64_t v = 0; uint32_t nb = 0;
        if (threadIdx.x == 0) nb = 3 + pad;
        else if (threadIdx.x == 1) { v = 0xffff0000u; nb = 32; }
        pk.round(v, nb);
    }
    if (threadIdx.x == 0 && (pk.bytepos != cm.bytes || pk.carry_bits != 0)) atomicAdd(err, 1u);
}

// One stream: header and trailer around the payload that ends at d_end[0].
__global__ void k_frame(uint8_t* __restrict__ out, uint64_t cap, uint64_t hdr_len, const uint64_t* __restrict__ d_end,
                        const uint32_t* __restrict__ sums, uint64_t n, int level, int wrap, int flags, uint64_t* __restrict__ total_out)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const uint64_t pos = d_end[0];                              // header + every slab's payload
    const uint32_t tl = (flags & (ZB200_DEFLATE_NO_TRAILER | ZB200_DEFLATE_NOT_LAST)) ? 0 : frame_trailer_len(wrap);
    const uint32_t crc = sums[0], adler = sums[1];
    total_out[0] = pos + tl;
    if (pos + tl > cap) return;
    if (hdr_len) write_frame_header(out, wrap, level, (flags >> 8) & 7);
    if (tl) write_frame_trailer(out + pos + tl, wrap, crc, adler, n);
}

// empty input: a lone final fixed block with just the end-of-block code = 03 00 (what the reference emits)
__global__ void k_empty_payload(uint8_t* out, uint64_t cap, uint64_t at, int not_last, int force_mark, uint64_t* d_end)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (not_last) {
        d_end[0] = at + (force_mark ? 5 : 0);
        if (force_mark && at + 5 <= cap) { out[at] = 0; out[at + 1] = 0; out[at + 2] = 0; out[at + 3] = 0xff; out[at + 4] = 0xff; }
        return;
    }
    d_end[0] = at + 2;
    if (at + 2 <= cap) { out[at] = 3; out[at + 1] = 0; }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct DeflateParams {
    LevelCfg cfg; int level, strategy, wrap, flags;
    uint32_t max_dist;                                          // kWindow, or the reference's MAX_DIST of a smaller windowBits
};

// exact intra-step links (MATCH.ANY, 8.4 ms per GiB) for the levels that search long chains; levels 1..6 take the relaxed
// links (3.1 ms per GiB, ~0.1 % larger output)
static bool link_exact(int level, int strategy) { return level >= 7 || (level >= 4 && strategy == 4); }
// Lazy levels whose chain budget is at most this run in the greedy shape (links from L2, 64-byte sub-units, 3 CTAs per SM): with
// the short budgets of the four-byte chains the few link loads per search no longer pay for staging the links in shared memory
// (levels 4..7: 5 to 12 % faster and 0.1 % smaller, profiles/r2_sweeps.md).  Longer chains (levels 8, 9) keep the shared-memory links.
constexpr uint32_t kLazyGlobalMax = 16;
constexpr uint64_t kWalkCtasPerSm = 3;                          // greedy shape: three fit (the lazy shape: one)

struct BlockBufs {                                              // what k_plan and k_huff_pack read (all null at level 0)
    BlockMeta* blk = nullptr;
    uint32_t *tok = nullptr, *ntok = nullptr, *codes = nullptr, *hdr = nullptr;
};

// Link, walk and code construction of nblocks blocks: the scratch, then the kernels on s.  Stream mode (d_cd null): d_buf =
// [dict][source], total = dict + source bytes, blocks from d_buf + dict on.  Job mode: d_buf[0, total) holds the jobs of
// the chunk table d_cd, dict = 0, four block slots per chunk.
static int deflate_blocks_launch(Ctx* c, const uint8_t* d_buf, uint64_t total, uint64_t dict, uint64_t nblocks,
                                 const ChunkDesc* d_cd, const DeflateParams& P, cudaStream_t s, BlockBufs* out)
{
    const LevelCfg& cfg = P.cfg;
    if (cfg.kind == 0 || nblocks == 0) return 0;
    const uint64_t slots = std::min<uint64_t>(nblocks, (uint64_t)device_sms() * kWalkCtasPerSm);   // persistent walk CTAs
    int rc;
    if ((rc = c->ws[3].ensure(total * 2 + 64)) != 0) return rc;                          // dist16
    if ((rc = c->ws[4].ensure(slots * kTmpPerBlock * 4 + 64)) != 0) return rc;           // private token regions
    if ((rc = c->ws[5].ensure(nblocks * kBlockBytes * 4 + 64)) != 0) return rc;          // tokens, contiguous per block
    if ((rc = c->ws[6].ensure(nblocks * sizeof(BlockMeta))) != 0) return rc;
    if ((rc = c->ws[7].ensure(nblocks * kHistSize * 4)) != 0) return rc;
    if ((rc = c->ws[8].ensure(nblocks * kHistSize * 4)) != 0) return rc;
    if ((rc = c->ws[9].ensure(nblocks * kHdrWords * 4)) != 0) return rc;
    if ((rc = c->ws[10].ensure(nblocks * 4 + 16)) != 0) return rc;
    uint16_t* d_dist = c->ws[3].as<uint16_t>();
    uint32_t* d_tmp = c->ws[4].as<uint32_t>();
    uint32_t* d_hist = c->ws[7].as<uint32_t>();
    out->tok = c->ws[5].as<uint32_t>();
    out->blk = c->ws[6].as<BlockMeta>();
    out->codes = c->ws[8].as<uint32_t>(); out->hdr = c->ws[9].as<uint32_t>();
    out->ntok = c->ws[10].as<uint32_t>();
    uint32_t* d_next = out->ntok + nblocks;                     // the walk kernel's block counter
    if (cfg.chain != 0 && P.strategy != 3) {                    // Z_RLE needs no chains
        const unsigned nseg = (unsigned)(d_cd ? nblocks / kBlocksPerChunk : (total + kLinkSegBytes - 1) / kLinkSegBytes);
        // levels 1-6 trade the exact intra-step links for speed, like the reference's fast levels trade ratio
        if (link_exact(P.level, P.strategy)) ZB_LAUNCH(k_lz_link<true>, nseg, kLinkWarps * 32, kLinkSmem, s, d_buf, total, d_dist, d_cd);
        else ZB_LAUNCH(k_lz_link<false>, nseg, kLinkWarps * 32, kLinkSmem, s, d_buf, total, d_dist, d_cd);
    }
    ZB_CUDA(cudaMemsetAsync(d_next, 0, 4, s));
    if (cfg.kind == 2 && cfg.chain > kLazyGlobalMax && P.strategy != 3)
        ZB_LAUNCH((k_lz_walk<kWalkThreadsLazy, true>), (unsigned)std::min<uint64_t>(nblocks, device_sms()), kWalkThreadsLazy,
                  kWalkSmem + kWalkLinkSmem, s, d_buf, (uint32_t)total, (uint32_t)dict, d_dist, d_tmp, out->tok, out->ntok, d_hist,
                  cfg.kind, (int)cfg.chain, (uint32_t)cfg.nice, (uint32_t)cfg.lazy, (uint32_t)cfg.good, P.strategy, P.max_dist, d_cd,
                  (uint32_t)nblocks, d_next);
    else
        ZB_LAUNCH((k_lz_walk<kWalkThreadsFast, false>), (unsigned)slots, kWalkThreadsFast, kWalkSmem, s, d_buf, (uint32_t)total,
                  (uint32_t)dict, d_dist, d_tmp, out->tok, out->ntok, d_hist, cfg.kind, (int)cfg.chain, (uint32_t)cfg.nice,
                  (uint32_t)cfg.lazy, (uint32_t)cfg.good, P.strategy, P.max_dist, d_cd, (uint32_t)nblocks, d_next);
    ZB_LAUNCH(k_huff_build, (unsigned)((nblocks + kCodeWarps - 1) / kCodeWarps), kCodeWarps * 32, 0, s, total - dict, out->blk, d_hist,
              out->codes, out->hdr, P.strategy == 4 ? 1 : 0, d_cd, nblocks);
    return 0;
}

// One slab: d_buf = [dict bytes][n source bytes], contiguous in device memory.  The slab's payload starts at
// out[(*d_start or 0) + start_add]; *d_end receives where the next slab starts.  Everything is asynchronous on s.
static int deflate_slab_launch(Ctx* c, const uint8_t* d_buf, uint64_t dict, uint64_t n, uint8_t* d_out, uint64_t cap,
                               const DeflateParams& P, int last_is_final, int force_mark, const uint64_t* d_start,
                               uint64_t start_add, uint64_t* d_end, uint32_t* d_err, cudaStream_t s,
                               cudaEvent_t prev_scanned = nullptr, cudaEvent_t scanned = nullptr, uint32_t bitmode = 0, uint32_t prime_val = 0)
{
    const uint64_t nchunks = (n + kChunk - 1) / kChunk;
    const uint64_t nblocks = (n + kBlockBytes - 1) / kBlockBytes;
    int rc;
    if ((rc = c->ws[2].ensure(nchunks * sizeof(ChunkMeta))) != 0) return rc;
    ChunkMeta* d_chunks = c->ws[2].as<ChunkMeta>();
    BlockBufs bb;
    if ((rc = deflate_blocks_launch(c, d_buf, dict + n, dict, nblocks, nullptr, P, s, &bb)) != 0) return rc;
    ZB_LAUNCH(k_plan, (unsigned)((nchunks + 255) / 256), 256, 0, s, nchunks, n, d_chunks, bb.blk, last_is_final, P.cfg.kind == 0 ? 1 : 0, force_mark, (const ChunkDesc*)nullptr, bitmode);
    // Slabs alternate between two streams; only the running output offset links them: this slab's offsets need the
    // end of the previous slab, everything before this point (link, walk, codes, plan) does not.
    if (prev_scanned) ZB_CUDA(cudaStreamWaitEvent(s, prev_scanned, 0));
    ZB_LAUNCH(k_scan, 1, 1024, 0, s, nchunks, d_chunks, d_start, start_add, d_end);
    if (scanned) ZB_CUDA(cudaEventRecord(scanned, s));
    ZB_LAUNCH(k_huff_pack, (unsigned)nchunks, kPackThreads, 0, s, d_buf + dict, n, bb.tok, bb.ntok, bb.blk, bb.codes, bb.hdr, d_chunks, d_out, cap,
              last_is_final, force_mark, d_err, (const ChunkDesc*)nullptr, (const JobDesc*)nullptr, (JobResult*)nullptr, bitmode, prime_val, d_err + 1);
    ZB_CHECK_LAUNCH();
    return 0;
}

// One slab in job mode: d_base[0, span) holds whole jobs back to back; chunk and job tables are on the device.  Every
// stream lands in its own slot of d_out, complete with header and trailer; d_jres[j] = {length, checksums, error count}.
static int deflate_jobs_launch(Ctx* c, const uint8_t* d_base, uint64_t span, uint32_t nchunks, uint32_t njobs,
                               const ChunkDesc* d_cd, const JobDesc* d_jobs, uint8_t* d_out,
                               const DeflateParams& P, uint32_t* d_crc, uint32_t* d_adler, JobResult* d_jres, cudaStream_t s)
{
    int rc;
    if ((rc = c->ws[2].ensure((uint64_t)(nchunks + 1) * sizeof(ChunkMeta))) != 0) return rc;
    ChunkMeta* d_chunks = c->ws[2].as<ChunkMeta>();
    BlockBufs bb;
    if ((rc = deflate_blocks_launch(c, d_base, span, 0, (uint64_t)nchunks * kBlocksPerChunk, d_cd, P, s, &bb)) != 0) return rc;
    if (nchunks)
        ZB_LAUNCH(k_plan, (nchunks + 255) / 256, 256, 0, s, (uint64_t)nchunks, span, d_chunks, bb.blk, 1, P.cfg.kind == 0 ? 1 : 0, 0, d_cd, 0u);
    ZB_LAUNCH(k_scan_jobs, 1, 1024, 0, s, nchunks, d_chunks, d_cd, d_jobs, njobs, frame_header_len(P.wrap), frame_trailer_len(P.wrap), d_jres);
    if (nchunks)
        ZB_LAUNCH(k_huff_pack, nchunks, kPackThreads, 0, s, d_base, span, bb.tok, bb.ntok, bb.blk, bb.codes, bb.hdr, d_chunks, d_out, (uint64_t)0,
                  1, 0, (uint32_t*)nullptr, d_cd, d_jobs, d_jres, 0u, 0u, (uint32_t*)nullptr);
    if ((rc = checksum_jobs_launch(c, d_base, d_cd, nchunks, d_jobs, njobs, d_crc, d_adler, s)) != 0) return rc;
    ZB_LAUNCH(k_frame_jobs, (njobs + 127) / 128, 128, 0, s, d_out, d_jobs, njobs, d_crc, d_adler, P.level, P.wrap, P.strategy, d_jres);
    ZB_CHECK_LAUNCH();
    return 0;
}

// Slab boundaries (byte offsets, cut[0] = 0 .. cut.back() = n).  Device-resident data: uniform slabs.  Host buffers:
// the first and last slabs are a quarter and a half slab, so that the first kernels start after 28 MiB of H2D instead
// of 111 MiB and only 28 MiB of work and its D2H copy trail the last H2D.
static void plan_slabs(uint64_t n, bool ramp, std::vector<uint64_t>& cut)
{
    cut.assign(1, 0);
    if (n == 0) return;
    const uint64_t C = (n + kChunk - 1) / kChunk, full = kSlabChunks, h = full / 2, q = full / 4;
    std::vector<uint64_t> sizes;
    if (!ramp || C <= 4 * full) {
        // equal slabs, an even number of them: slabs alternate between two streams, and a short last slab would run alone
        uint64_t k = (C + full - 1) / full;
        if (k > 1 && (k & 1)) k++;
        const uint64_t per = (C + k - 1) / k;
        for (uint64_t c = 0; c < C; c += per) sizes.push_back(std::min<uint64_t>(per, C - c));
    } else {
        const uint64_t mid = C - 2 * (q + h);
        sizes.push_back(q); sizes.push_back(h);
        for (uint64_t c = 0; c < mid; c += full) sizes.push_back(std::min<uint64_t>(full, mid - c));
        sizes.push_back(h); sizes.push_back(q);
    }
    uint64_t c = 0;
    for (uint64_t z : sizes) { c += z; cut.push_back(std::min<uint64_t>(n, c * kChunk)); }
}

// A whole device-resident job, asynchronous on s with the scratch of context c: slabs, checksums of the input,
// header and trailer.  d_res (device, 32 bytes): u64 total length, then u32 crc32, adler32, error count.
static int deflate_enqueue_dev(Ctx* c, cudaStream_t s, const uint8_t* d_buf, uint64_t dict_len, uint64_t n, uint8_t* d_out,
                               uint64_t cap, const DeflateParams& P, uint32_t* d_res)
{
    const int force_mark = (P.flags & ZB200I_DEFLATE_FORCE_MARK) ? 1 : 0;
    const int last_is_final = (P.flags & ZB200_DEFLATE_NOT_LAST) ? 0 : 1;
    const uint64_t hdr_len = (P.flags & ZB200_DEFLATE_NO_HEADER) ? 0 : frame_header_len(P.wrap);
    std::vector<uint64_t> cut;
    plan_slabs(n, false, cut);
    const uint64_t nslabs = cut.size() - 1;
    int rc;
    if ((rc = c->ws[1].ensure((nslabs + 2) * 8)) != 0) return rc;
    uint64_t* d_pos = c->ws[1].as<uint64_t>();
    uint64_t* d_total = reinterpret_cast<uint64_t*>(d_res);
    uint32_t* d_sums = d_res + 2;
    uint32_t* d_err = d_res + 4;
    ZB_CUDA(cudaMemsetAsync(d_err, 0, 4, s));
    const uint8_t* d_src = d_buf + dict_len;
    if (n == 0) ZB_LAUNCH(k_empty_payload, 1, 32, 0, s, d_out, cap, hdr_len, !last_is_final, force_mark, d_pos);
    for (uint64_t i = 0; i < nslabs; i++) {
        const uint64_t off = cut[i], len = cut[i + 1] - cut[i];
        const uint64_t dlen = i == 0 ? dict_len : kWindow;
        const bool last = i == nslabs - 1;
        if ((rc = deflate_slab_launch(c, d_src + off - dlen, dlen, len, d_out, cap, P, last && last_is_final, last ? force_mark : 0,
                                      i ? d_pos + i - 1 : nullptr, i ? 0 : hdr_len, d_pos + i, d_err, s)) != 0) return rc;
    }
    if ((rc = checksum_launch(c, d_src, n, d_sums, s)) != 0) return rc;
    ZB_LAUNCH(k_frame, 1, 32, 0, s, d_out, cap, hdr_len, d_pos + (nslabs ? nslabs - 1 : 0), d_sums, n, P.level, P.wrap, P.flags, d_total);
    ZB_CHECK_LAUNCH();
    return 0;
}

int deflate_setup()                                             // once per device, from ensure_init (under its lock)
{
    ZB_CUDA(cudaFuncSetAttribute(k_lz_link<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLinkSmem));
    ZB_CUDA(cudaFuncSetAttribute(k_lz_link<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLinkSmem));
    ZB_CUDA(cudaFuncSetAttribute(k_lz_walk<kWalkThreadsFast, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWalkSmem));
    ZB_CUDA(cudaFuncSetAttribute(k_lz_walk<kWalkThreadsLazy, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWalkSmem + kWalkLinkSmem));
    return 0;
}

static int deflate_params(DeflateParams& P, int level, int wrap, int flags)
{
    if (level < 0) level = 6;
    P.cfg = h_levels[level]; P.level = level; P.wrap = wrap; P.flags = flags;
    P.strategy = (flags >> 8) & 7;                              // Z_FILTERED 1, Z_HUFFMAN_ONLY 2, Z_RLE 3, Z_FIXED 4
    const int wbits = (flags >> 12) & 15;                       // 0 = 15; deflate.c:270-279, h/deflate.h:276
    P.max_dist = (wbits >= 9 && wbits < 15) ? (1u << wbits) - 262u : kWindow;
    if (P.strategy == 2 && P.cfg.kind != 0) { P.cfg.chain = 0; P.cfg.kind = 1; }   // literals only (deflate.c:1490)
    return 0;
}

}  // namespace zb

using namespace zb;

// One shard in two halves.  begin: everything is enqueued (copies in, slab kernels on two streams, checksums, header and
// trailer, the result words on their way to pinned memory); end: wait, copy out what is still on the device, report.
// zb200_deflate_shard is begin + end; a caller with several pieces (the multi-GPU rounds) begins piece j + 1 before it
// ends piece j, so the GPU never waits for the host to read a length.
struct ShardJob {
    Ctx* c = nullptr; Ctx* c2 = nullptr;
    cudaStream_t s = nullptr, s_out = nullptr;
    HostStager stager;                                          // pageable sources of 64 MiB and more
    HostDrainer drainer;                                        // and pageable destinations
    std::vector<uint64_t> cut;
    uint64_t nslabs = 0, hdr_len = 0, n = 0;
    size_t cap = 0;
    void* dst = nullptr; uint8_t* d_out = nullptr;
    bool dst_on_host = false;
    cudaEvent_t* ev_done = nullptr;
    cudaEvent_t ev_result = nullptr;                            // the result words have reached pinned memory
    uint64_t* h_res = nullptr; uint64_t* h_pos = nullptr;
    int rc = 0;
};

static void shard_release(ShardJob* J)
{
    J->stager.finish();
    J->drainer.finish();
    if (J->c2) ctx_release(J->c2, J->c2->own_stream);
    if (J->c) ctx_release(J->c, J->s);
    J->c = J->c2 = nullptr;
}

static int shard_begin(ShardJob* J, const void* src, size_t src_len, const void* dict, size_t dict_len, void* dst, size_t cap,
                       int level, int wrap, int flags, void* stream, uint32_t prime_bits = 0, uint32_t prime_val = 0, bool partial_end = false)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (level < -1 || level > 9 || wrap < 0 || wrap > 2 || (src_len && !src) || dict_len > kWindow || !dst) {
        set_error("zb200_deflate: bad argument");
        return ZB_STREAM_ERROR;
    }
    DeflateParams P;
    if ((rc = deflate_params(P, level, wrap, flags)) != 0) return rc;
    level = P.level;
    const int force_mark = (flags & ZB200I_DEFLATE_FORCE_MARK) ? 1 : 0;
    const int last_is_final = (flags & ZB200_DEFLATE_NOT_LAST) ? 0 : 1;
    const uint64_t hdr_len = (flags & ZB200_DEFLATE_NO_HEADER) ? 0 : frame_header_len(wrap);
    const uint64_t n = src_len;
    if ((prime_bits || partial_end) && (P.cfg.kind == 0 || n == 0 || prime_bits > 7 || hdr_len)) {
        set_error("zb200: pending bits need a raw shard with input at level 1..9");   // the shim handles the other cases on the host
        return ZB_STREAM_ERROR;
    }
    std::vector<uint64_t>& cut = J->cut;
    plan_slabs(n, (n != 0 && classify(src) != kDevice) || classify(dst) != kDevice, cut);
    const uint64_t nslabs = cut.size() - 1;

    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    Ctx* c2 = nullptr;
    cudaStream_t s = pick_stream(c, stream);
    J->c = c; J->s = s; J->cap = cap; J->dst = dst; J->n = n; J->nslabs = nslabs; J->hdr_len = hdr_len;
    HostStager& stager = J->stager;
    do {
        const bool src_on_host = n != 0 && classify(src) != kDevice;
        const bool dst_on_host = classify(dst) != kDevice;
        J->dst_on_host = dst_on_host;
        if ((rc = c->ensure_aux((int)(3 * nslabs + 5))) != 0) break;
        cudaStream_t s_in = c->aux[0];
        J->s_out = c->aux[1];
        J->ev_result = c->evs[3 * nslabs + 3];
        cudaEvent_t* ev_in = c->evs;
        cudaEvent_t* ev_done = c->evs + nslabs;
        cudaEvent_t* ev_scan = c->evs + 2 * nslabs;
        cudaEvent_t ev_start = c->evs[3 * nslabs + 1], ev_join = c->evs[3 * nslabs + 2];
        J->ev_done = ev_done;
        cudaError_t e = cudaSuccess;
        // Odd slabs run on a second context and stream: the walk kernel is latency bound and leaves issue slots and
        // some shared memory free, which the pack / code kernels of the neighbouring slab can use.
        if (nslabs > 1 && !c2 && !g_profile) {                  // per-kernel timing (zb200_profile) wants the slabs serialized
            c2 = ctx_acquire_own();
            if (!c2) { rc = ZB_MEM_ERROR; break; }
            J->c2 = c2;
        }
        // ---- [dict][src] as one contiguous device range ----
        const uint8_t* d_buf;
        bool stage_slabs = false;                               // source slabs still have to be copied in
        if (n == 0) {
            if ((rc = c->in.ensure(64)) != 0) break;
            d_buf = c->in.as<uint8_t>();
            dict_len = 0;
        } else if (!src_on_host && (dict_len == 0 || (classify(dict) == kDevice && (const uint8_t*)dict + dict_len == (const uint8_t*)src))) {
            d_buf = (const uint8_t*)src - dict_len;
        } else {
            if ((rc = c->in.ensure(dict_len + n + 64)) != 0) break;
            d_buf = c->in.as<uint8_t>();
            stage_slabs = true;
            cudaStreamWaitEvent(s_in, c->idle, 0);              // the staging buffer may still be read by the previous borrower
            if (!src_on_host) {                                 // device source produced on the caller's stream
                cudaEventRecord(c->evs[3 * nslabs], s);
                cudaStreamWaitEvent(s_in, c->evs[3 * nslabs], 0);
            }
            if (dict_len) {
                e = cudaMemcpyAsync(c->in.p, dict, dict_len, cudaMemcpyDefault, s_in);
                if (e != cudaSuccess) { set_error("dictionary staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
        }
        uint8_t* d_out = (uint8_t*)dst;
        if (dst_on_host) {
            if ((rc = c->out.ensure(cap + 16)) != 0) break;
            d_out = c->out.as<uint8_t>();
        }
        J->d_out = d_out;
        if ((rc = c->small.ensure(256)) != 0) break;
        if ((rc = c->ws[1].ensure((nslabs + 2) * 8)) != 0) break;
        if ((rc = c->ensure_pinned((nslabs + 8) * 8)) != 0) break;
        uint64_t* d_total = c->small.as<uint64_t>();
        uint32_t* d_sums = c->small.as<uint32_t>() + 2;
        uint32_t* d_err = c->small.as<uint32_t>() + 4;
        uint64_t* d_pos = c->ws[1].as<uint64_t>();              // d_pos[i] = end of slab i in the output
        uint64_t* h_res = (uint64_t*)c->pinned;                 // [0..3] result words, [4..] slab ends
        uint64_t* h_pos = h_res + 4;
        J->h_res = h_res; J->h_pos = h_pos;
        if ((e = cudaMemsetAsync(d_err, 0, 8, s)) != cudaSuccess) { set_error("memset failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }   // error count and pending-bits word
        if (c2) {                                               // the second stream starts where the caller's stream is now
            cudaEventRecord(ev_start, s);
            cudaStreamWaitEvent(c2->own_stream, ev_start, 0);
        }

        // ---- slabs: copy in (own stream) -> kernels (s) -> slab end to the host ----
        const uint8_t* d_src = d_buf + dict_len;
        const bool threaded = stage_slabs && n >= HostStager::kMinBytes && classify(src) == kHostPageable;
        if (threaded && (rc = stager.start(src, (uint8_t*)d_src, n, s_in)) != 0) break;
        if (n == 0) {
            ZB_LAUNCH(k_empty_payload, 1, 32, 0, s, d_out, cap, hdr_len, !last_is_final, force_mark, d_pos);
        }
        for (uint64_t i = 0; i < nslabs; i++) {
            const uint64_t off = cut[i], len = cut[i + 1] - cut[i];
            Ctx* cl = (c2 && (i & 1)) ? c2 : c;
            cudaStream_t sl = (c2 && (i & 1)) ? c2->own_stream : s;
            if (stage_slabs && threaded) {                       // pageable source: pieces arrive from the staging threads
                if ((rc = stager.wait_range(off, len, sl)) != 0) break;
                if (c2 && i + 1 < nslabs && (rc = stager.wait_range(off + len - std::min<uint64_t>(len, kWindow), std::min<uint64_t>(len, kWindow),
                                                                    (i & 1) ? s : c2->own_stream)) != 0) break;   // its tail is the next slab's dictionary
            } else if (stage_slabs) {
                e = cudaMemcpyAsync((uint8_t*)d_src + off, (const uint8_t*)src + off, len, cudaMemcpyDefault, s_in);
                if (e == cudaSuccess) e = cudaEventRecord(ev_in[i], s_in);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(sl, ev_in[i], 0);
                if (e == cudaSuccess && c2 && i + 1 < nslabs) e = cudaStreamWaitEvent((i & 1) ? s : c2->own_stream, ev_in[i], 0);   // its tail is the next slab's dictionary
                if (e != cudaSuccess) { set_error("input staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
            const uint64_t dlen = i == 0 ? dict_len : kWindow;  // later slabs see the tail of the previous one
            const bool last = i == nslabs - 1;
            rc = deflate_slab_launch(cl, d_src + off - dlen, dlen, len, d_out, cap, P, last && last_is_final, last ? force_mark : 0,
                                     i ? d_pos + i - 1 : nullptr, i ? 0 : hdr_len, d_pos + i, d_err, sl,
                                     i ? ev_scan[i - 1] : nullptr, last ? nullptr : ev_scan[i],
                                     (i == 0 ? prime_bits : 0u) | ((last && partial_end) ? 0x100u : 0u), i == 0 ? prime_val : 0u);
            if (rc) break;
            if (dst_on_host && !last) {
                e = cudaMemcpyAsync(h_pos + i, d_pos + i, 8, cudaMemcpyDeviceToHost, sl);
                if (e == cudaSuccess) e = cudaEventRecord(ev_done[i], sl);
                if (e != cudaSuccess) { set_error("slab bookkeeping failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
        }
        if (c2) {                                               // join the second stream
            cudaEventRecord(ev_join, c2->own_stream);
            cudaStreamWaitEvent(s, ev_join, 0);
        }
        if (rc) { cudaStreamSynchronize(s); cudaStreamSynchronize(s_in); break; }
        // ---- checksums of the uncompressed data (read_buf, deflate.c:956-981), header, trailer ----
        if ((rc = checksum_launch(c, d_src, n, d_sums, s)) != 0) { cudaStreamSynchronize(s); break; }
        ZB_LAUNCH(k_frame, 1, 32, 0, s, d_out, cap, hdr_len, d_pos + (nslabs ? nslabs - 1 : 0), d_sums, n, level, wrap, flags, d_total);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_res, c->small.p, 32, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaEventRecord(J->ev_result, s);   // shard_end waits for THIS, not for whatever the caller enqueues behind it
        if (e != cudaSuccess) { set_error("deflate launch failed: %s", cudaGetErrorString(e)); cudaStreamSynchronize(s); rc = ZB_STREAM_ERROR; break; }
    } while (0);
    if (rc) shard_release(J);
    return rc;
}

static int shard_end(ShardJob* J, size_t* dst_len, uint32_t* crc, uint32_t* adler, uint32_t* tail = nullptr)
{
    int rc = 0;
    Ctx* c = J->c;
    cudaStream_t s = J->s, s_out = J->s_out;
    const uint64_t nslabs = J->nslabs, hdr_len = J->hdr_len, n = J->n;
    const size_t cap = J->cap;
    void* dst = J->dst;
    uint8_t* d_out = J->d_out;
    const bool dst_on_host = J->dst_on_host;
    uint64_t* h_res = J->h_res; uint64_t* h_pos = J->h_pos;
    HostDrainer& drainer = J->drainer;
    (void)c;
    do {
        cudaError_t e = cudaSuccess;
        // ---- copy out finished slabs while later ones are still running ----
        uint64_t copied = hdr_len;                              // out[0, hdr_len) is written last, by k_frame
        const bool drain_threads = dst_on_host && n >= HostStager::kMinBytes && classify(dst) == kHostPageable;
        if (dst_on_host) {
            for (uint64_t i = 0; i + 1 < nslabs; i++) {
                if ((e = cudaEventSynchronize(J->ev_done[i])) != cudaSuccess) break;
                const uint64_t end = h_pos[i];
                if (end > cap) break;                           // does not fit: reported below from the total
                if (end > copied) {
                    if (drain_threads) { if ((rc = drainer.drain((uint8_t*)dst + copied, d_out + copied, end - copied)) != 0) break; }
                    else e = cudaMemcpyAsync((uint8_t*)dst + copied, d_out + copied, end - copied, cudaMemcpyDeviceToHost, s_out);
                }
                if (e != cudaSuccess) break;
                copied = end;
            }
        }
        if (rc) { cudaStreamSynchronize(s); cudaStreamSynchronize(s_out); break; }
        if (e == cudaSuccess) e = cudaEventSynchronize(J->ev_result);
        if (e != cudaSuccess) { set_error("deflate failed: %s", cudaGetErrorString(e)); cudaStreamSynchronize(s_out); rc = ZB_STREAM_ERROR; break; }
        const uint64_t total = h_res[0];
        const uint32_t* r32 = (const uint32_t*)h_res;
        if (crc) *crc = r32[2];
        if (adler) *adler = r32[3];
        if (tail) *tail = r32[5];                               // bits a partial flush left pending: count | value << 8
        if (r32[4] != 0) { cudaStreamSynchronize(s_out); set_error("internal error: %u chunks packed to a size other than planned", r32[4]); rc = ZB_STREAM_ERROR; break; }
        *dst_len = (size_t)total;
        if (total > cap) {
            cudaStreamSynchronize(s_out);
            rc = ZB_BUF_ERROR; set_error("output buffer too small: need %llu, have %zu", (unsigned long long)total, cap);
            break;
        }
        if (dst_on_host && total) {
            if (total > copied) {
                if (drain_threads) { if ((rc = drainer.drain((uint8_t*)dst + copied, d_out + copied, total - copied)) != 0) break; }
                else e = cudaMemcpyAsync((uint8_t*)dst + copied, d_out + copied, total - copied, cudaMemcpyDeviceToHost, s_out);
            }
            if (e == cudaSuccess && hdr_len) e = cudaMemcpyAsync(dst, d_out, hdr_len, cudaMemcpyDeviceToHost, s_out);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s_out);
            if (e != cudaSuccess) { set_error("D2H copy failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        }
    } while (0);
    shard_release(J);
    return rc;
}

ZB_API int zb200_deflate_shard(const void* src, size_t src_len, const void* dict, size_t dict_len, void* dst,
                               size_t* dst_len, int level, int wrap, int flags, uint32_t* crc, uint32_t* adler, void* stream)
{
    if (!dst_len) { set_error("zb200_deflate: bad argument"); return ZB_STREAM_ERROR; }
    ShardJob J;
    int rc = shard_begin(&J, src, src_len, dict, dict_len, dst, *dst_len, level, wrap, flags, stream);
    if (rc) return rc;
    return shard_end(&J, dst_len, crc, adler);
}

// deflatePrime / Z_PARTIAL_FLUSH (deflate.c:404-414, trees.c:892): a raw shard that starts with `prime_bits` (< 8) pending
// bits and, when partial_end is set, ends with the ten bits of an empty static block and hands back the bits of its last,
// incomplete byte (*tail = count | value << 8) instead of aligning.  Hidden: the streaming shim (zapi_stream.c) is the caller.
extern "C" int zb200i_deflate_shard_bits(const void* src, size_t src_len, const void* dict, size_t dict_len, void* dst, size_t* dst_len,
                                         int level, int flags, uint32_t prime_bits, uint32_t prime_val, int partial_end,
                                         uint32_t* tail, uint32_t* crc, uint32_t* adler)
{
    if (!dst_len) return ZB_STREAM_ERROR;
    ShardJob J;
    int rc = shard_begin(&J, src, src_len, dict, dict_len, dst, *dst_len, level, ZB200_WRAP_RAW,
                         flags | ZB200_DEFLATE_NO_HEADER | ZB200_DEFLATE_NO_TRAILER | (partial_end ? ZB200_DEFLATE_NOT_LAST : 0), nullptr,
                         prime_bits, prime_val, partial_end != 0);
    if (rc) return rc;
    return shard_end(&J, dst_len, crc, adler, tail);
}

// The two halves as calls of their own (see ShardJob): *job receives a handle that zb200_deflate_shard_end consumes.
ZB_API int zb200_deflate_shard_begin(void** job, const void* src, size_t src_len, const void* dict, size_t dict_len, void* dst,
                                     size_t dst_cap, int level, int wrap, int flags, void* stream)
{
    if (!job) { set_error("zb200_deflate_shard_begin: bad argument"); return ZB_STREAM_ERROR; }
    ShardJob* J = new ShardJob();
    const int rc = shard_begin(J, src, src_len, dict, dict_len, dst, dst_cap, level, wrap, flags, stream);
    if (rc) { delete J; *job = nullptr; return rc; }
    *job = J;
    return 0;
}

ZB_API int zb200_deflate_shard_end(void* job, size_t* dst_len, uint32_t* crc, uint32_t* adler)
{
    if (!job || !dst_len) { set_error("zb200_deflate_shard_end: bad argument"); return ZB_STREAM_ERROR; }
    ShardJob* J = static_cast<ShardJob*>(job);
    const int rc = shard_end(J, dst_len, crc, adler);
    delete J;
    return rc;
}

ZB_API int zb200_deflate(const void* src, size_t src_len, void* dst, size_t* dst_len, int level, int wrap, void* stream)
{
    return zb200_deflate_shard(src, src_len, nullptr, 0, dst, dst_len, level, wrap, 0, nullptr, nullptr, stream);
}

// n independent inputs -> n independent streams (the per-member compressor a ZIP writer needs, zip.c:1034-1128).
// Consecutive jobs are packed into slabs of up to kSlabChunks chunks / jobs that go through the kernels together in job
// mode (chunks never cross a job boundary; each stream lands in its own slot with header and trailer), so ten thousand
// small files cost a few dozen launches instead of ten per file.  Jobs above kBatchBigJob take the single-stream
// pipeline.  Slabs alternate over a few contexts (stream + scratch each); with host arenas the H2D copy of the next
// slab and the D2H copies of finished slabs overlap the kernels.  The host waits once per slab, for its result words.
constexpr uint64_t kBatchBigJob = 32ull << 20;
constexpr uint64_t kBatchGapCopy = 64ull << 10;                 // D2H ranges of neighbouring slots merge across gaps up to this

struct BatchSlab { size_t j0, j1; bool big; uint32_t nchunks; size_t cd_at, job_at; };

ZB_API int zb200_deflate_batch(const void* src, const uint64_t* src_off, size_t n, void* dst, const uint64_t* dst_off,
                               uint64_t* dst_len, uint32_t* crc, uint32_t* adler, int32_t* status, int level, int wrap,
                               void* stream)
{
    if (wrap < 0 || wrap > 2) { set_error("zb200_deflate_batch: bad argument"); return ZB_STREAM_ERROR; }
    return zb::deflate_batch(src, src_off, n, dst, dst_off, dst_len, crc, adler, status, level, wrap, stream);
}

int zb::deflate_batch(const void* src, const uint64_t* src_off, size_t n, void* dst, const uint64_t* dst_off, uint64_t* dst_len,
                      uint32_t* crc, uint32_t* adler, int32_t* status, int level, int wrap, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (level < -1 || level > 9 || (n && (!src_off || !dst_off || !dst || !dst_len))) {
        set_error("zb200_deflate_batch: bad argument");
        return ZB_STREAM_ERROR;
    }
    if (n == 0) return 0;
    for (size_t i = 0; i < n; i++)
        if (src_off[i + 1] < src_off[i] || dst_off[i + 1] < dst_off[i]) { set_error("zb200_deflate_batch: offsets must not decrease"); return ZB_STREAM_ERROR; }
    DeflateParams P;
    if ((rc = deflate_params(P, level, wrap, 0)) != 0) return rc;

    // ---- slabs and their tables ----
    std::vector<BatchSlab> slabs;
    std::vector<ChunkDesc> h_cd;
    std::vector<JobDesc> h_jobs;
    {
        BatchSlab cur{0, 0, false, 0, 0, 0};
        auto flush = [&](size_t upto) {
            if (upto > cur.j0) { cur.j1 = upto; slabs.push_back(cur); }
            cur = BatchSlab{upto, upto, false, 0, h_cd.size(), h_jobs.size()};
        };
        for (size_t i = 0; i < n; i++) {
            const uint64_t len = src_off[i + 1] - src_off[i];
            if (len > kBatchBigJob) {
                flush(i);
                cur.big = true; cur.j0 = i;
                flush(i + 1);
                continue;
            }
            const uint32_t nc = (uint32_t)((len + kChunk - 1) / kChunk);
            if (cur.nchunks + nc > kSlabChunks || i - cur.j0 >= kSlabChunks) flush(i);
            const uint64_t base = src_off[cur.j0];
            const uint32_t jb = (uint32_t)(src_off[i] - base), je = (uint32_t)(src_off[i + 1] - base);
            const uint32_t job = (uint32_t)(i - cur.j0), first = cur.nchunks;
            h_jobs.push_back(JobDesc{dst_off[i], dst_off[i + 1] - dst_off[i], first, nc, jb, (uint32_t)len});
            for (uint32_t k = 0; k < nc; k++) {
                const uint32_t cb = jb + k * kChunk;
                h_cd.push_back(ChunkDesc{cb, std::min<uint32_t>(kChunk, je - cb), jb, je, job, first, k + 1 == nc ? 1u : 0u, 0u});
            }
            cur.nchunks += nc;
        }
        flush(n);
    }
    const size_t nslabs = slabs.size();

    constexpr int kLanes = 3;
    cudaStream_t s0 = (cudaStream_t)stream;
    Ctx* c0 = ctx_acquire(s0);
    if (!c0) return ZB_MEM_ERROR;
    Ctx* lane[kLanes] = {nullptr, nullptr, nullptr};
    int nl = 0;
    HostStager stager;                                          // pageable arenas of 64 MiB and more
    HostDrainer drainer;
    do {
        if ((rc = c0->ensure_aux((int)(2 * nslabs + kLanes + 4))) != 0) break;
        cudaStream_t s_in = c0->aux[0], s_out = c0->aux[1];
        cudaEvent_t* ev_in = c0->evs;
        cudaEvent_t* ev_done = c0->evs + nslabs;
        cudaEvent_t* ev_misc = c0->evs + 2 * nslabs;            // [0] setup, [1..kLanes] lane joins
        const size_t nlanes = g_profile ? 1 : nslabs < (size_t)kLanes ? nslabs : (size_t)kLanes;   // per-kernel timing wants the slabs serialized
        for (; nl < (int)nlanes; nl++) {
            lane[nl] = ctx_acquire_own();
            if (!lane[nl]) { rc = ZB_MEM_ERROR; break; }
        }
        if (rc) break;
        const uint64_t src_total = src_off[n] - src_off[0], dst_total = dst_off[n];
        const bool src_on_host = src_total != 0 && classify(src) != kDevice;
        const bool dst_on_host = classify(dst) != kDevice;
        const uint8_t* d_src = (const uint8_t*)src;             // indexed by absolute src_off
        if (src_on_host || src_total == 0) {
            if ((rc = c0->in.ensure(src_total + 64)) != 0) break;
            d_src = c0->in.as<uint8_t>() - src_off[0];
            cudaStreamWaitEvent(s_in, c0->idle, 0);             // the staging buffer may still be read by the previous borrower
        }
        uint8_t* d_dst = (uint8_t*)dst;
        if (dst_on_host) {
            if ((rc = c0->out.ensure(dst_total + 16)) != 0) break;
            d_dst = c0->out.as<uint8_t>();
        }
        // device tables: results, checksums, chunk / job / offset tables of every job-mode slab
        const size_t at_res = 0, at_crc = at_res + n * sizeof(JobResult), at_adl = at_crc + n * 4;
        const size_t at_cd = (at_adl + n * 4 + 15) & ~(size_t)15, at_job = at_cd + h_cd.size() * sizeof(ChunkDesc);
        const size_t tab_bytes = at_job + h_jobs.size() * sizeof(JobDesc) + 16;
        if ((rc = c0->ws[11].ensure(tab_bytes)) != 0) break;
        if ((rc = c0->ensure_pinned(n * sizeof(JobResult))) != 0) break;
        uint8_t* d_tab = c0->ws[11].as<uint8_t>();
        JobResult* d_jres = reinterpret_cast<JobResult*>(d_tab + at_res);
        uint32_t* d_crc = reinterpret_cast<uint32_t*>(d_tab + at_crc);
        uint32_t* d_adl = reinterpret_cast<uint32_t*>(d_tab + at_adl);
        const ChunkDesc* d_cd = reinterpret_cast<const ChunkDesc*>(d_tab + at_cd);
        const JobDesc* d_jobs = reinterpret_cast<const JobDesc*>(d_tab + at_job);
        cudaError_t e = cudaSuccess;
        if (!h_cd.empty()) e = cudaMemcpyAsync(d_tab + at_cd, h_cd.data(), h_cd.size() * sizeof(ChunkDesc), cudaMemcpyHostToDevice, s0);
        if (e == cudaSuccess && !h_jobs.empty()) e = cudaMemcpyAsync(d_tab + at_job, h_jobs.data(), h_jobs.size() * sizeof(JobDesc), cudaMemcpyHostToDevice, s0);
        if (e == cudaSuccess) e = cudaEventRecord(ev_misc[0], s0);   // tables are up (and the caller's stream has reached us)
        for (int k = 0; k < nl && e == cudaSuccess; k++) e = cudaStreamWaitEvent(lane[k]->own_stream, ev_misc[0], 0);
        if (e == cudaSuccess && !src_on_host) e = cudaStreamWaitEvent(s_in, ev_misc[0], 0);
        if (e != cudaSuccess) { set_error("batch setup failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }

        // ---- enqueue: copy in (s_in) -> kernels (lane) -> result words to the host ----
        const bool threaded = src_on_host && src_total >= HostStager::kMinBytes && classify(src) == kHostPageable;
        const bool drain_threads = dst_on_host && src_total >= HostStager::kMinBytes && classify(dst) == kHostPageable;
        if (threaded && (rc = stager.start(src, (uint8_t*)d_src + src_off[0], src_total, s_in)) != 0) break;
        JobResult* h_res = (JobResult*)c0->pinned;
        size_t enq = 0;
        for (; enq < nslabs; enq++) {
            const BatchSlab& sl = slabs[enq];
            Ctx* ck = lane[enq % nl];
            cudaStream_t sk = ck->own_stream;
            const uint64_t a = src_off[sl.j0], span = src_off[sl.j1] - a;
            if (src_on_host && span && threaded) {               // pageable arena: pieces arrive from the staging threads
                if ((rc = stager.wait_range(a - src_off[0], span, sk)) != 0) break;
            } else if (src_on_host && span) {
                e = cudaMemcpyAsync((uint8_t*)d_src + a, (const uint8_t*)src + (a - src_off[0]), span, cudaMemcpyHostToDevice, s_in);
                if (e == cudaSuccess) e = cudaEventRecord(ev_in[enq], s_in);
                if (e == cudaSuccess) e = cudaStreamWaitEvent(sk, ev_in[enq], 0);
                if (e != cudaSuccess) { set_error("input staging failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            }
            if (sl.big)
                rc = deflate_enqueue_dev(ck, sk, d_src + a, 0, span, d_dst + dst_off[sl.j0], dst_off[sl.j0 + 1] - dst_off[sl.j0], P,
                                         reinterpret_cast<uint32_t*>(d_jres + sl.j0));
            else
                rc = deflate_jobs_launch(ck, d_src + a, span, sl.nchunks, (uint32_t)(sl.j1 - sl.j0), d_cd + sl.cd_at, d_jobs + sl.job_at,
                                         d_dst, P, d_crc + sl.j0, d_adl + sl.j0, d_jres + sl.j0, sk);
            if (rc) break;
            e = cudaMemcpyAsync(h_res + sl.j0, d_jres + sl.j0, (sl.j1 - sl.j0) * sizeof(JobResult), cudaMemcpyDeviceToHost, sk);
            if (e == cudaSuccess) e = cudaEventRecord(ev_done[enq], sk);
            if (e != cudaSuccess) { set_error("batch bookkeeping failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        }
        for (int k = 0; k < nl; k++) {                           // join the lanes (also after a failed enqueue)
            cudaEventRecord(ev_misc[1 + k], lane[k]->own_stream);
            cudaStreamWaitEvent(s0, ev_misc[1 + k], 0);
        }
        if (rc) { cudaStreamSynchronize(s0); cudaStreamSynchronize(s_in); break; }

        // ---- collect: per slab, results -> caller's arrays; finished streams -> host arena while later slabs run ----
        // A copy covers neighbouring slots and the short gaps between them (bytes past a stream's length in its own slot).
        uint64_t ra = 0, rb = 0;
        auto flush_copy = [&]() {
            if (rb > ra) {
                if (drain_threads) { if (drainer.drain((uint8_t*)dst + ra, d_dst + ra, rb - ra) != 0) rc = ZB_STREAM_ERROR; }
                else if (cudaMemcpyAsync((uint8_t*)dst + ra, d_dst + ra, rb - ra, cudaMemcpyDeviceToHost, s_out) != cudaSuccess) rc = ZB_STREAM_ERROR;
            }
            ra = rb = 0;
        };
        for (size_t k = 0; k < nslabs && !rc; k++) {
            if ((e = cudaEventSynchronize(ev_done[k])) != cudaSuccess) { set_error("deflate batch failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
            for (size_t i = slabs[k].j0; i < slabs[k].j1; i++) {
                const JobResult& r = h_res[i];
                const uint64_t cap = dst_off[i + 1] - dst_off[i];
                dst_len[i] = r.total;
                if (crc) crc[i] = r.crc;
                if (adler) adler[i] = r.adler;
                const int32_t st = r.err ? ZB_STREAM_ERROR : r.total > cap ? ZB_BUF_ERROR : ZB_OK;
                if (status) status[i] = st;
                if (!dst_on_host || st != ZB_OK || r.total == 0) continue;
                const uint64_t o = dst_off[i];
                if (rb > ra && o >= rb && o - rb <= kBatchGapCopy) rb = o + r.total;
                else { flush_copy(); ra = o; rb = o + r.total; }
            }
        }
        flush_copy();
        if (cudaStreamSynchronize(s0) != cudaSuccess) rc = ZB_STREAM_ERROR;
        if (dst_on_host && cudaStreamSynchronize(s_out) != cudaSuccess) rc = ZB_STREAM_ERROR;
        if (rc) set_error("deflate batch readback failed: %s", cudaGetErrorString(cudaGetLastError()));
    } while (0);
    stager.finish();
    drainer.finish();
    for (int k = 0; k < nl; k++) if (lane[k]) ctx_release(lane[k], lane[k]->own_stream);
    ctx_release(c0, s0);
    return rc;
}
