// zb_checksum.cu -- K5/K6: CRC-32 and Adler-32 in one pass over device memory.
//
// Replaces the reference's crc32()/crc32_little() (qcsrc/crc32.c:219,262) and adler32()
// (qcsrc/adler32.c:57) plus the GF(2) / modular merges of crc32_combine (crc32.c:370) and
// adler32_combine (adler32.c:128), which here run as an on-device combine tree.
//
// CRC formulation.  Write the raw CRC register (no pre/post inversion) of a message M as
// R(M) = M(x) * x^32 mod P.  R is linear over GF(2), so R(M) is the XOR over all 32-bit
// words W at byte offset o of  W * x^(8*(len-o)) mod P.  A warp owns a contiguous segment
// and reads it 512 bytes at a time (one coalesced 16-byte load per lane); each lane keeps
// FOUR independent registers, one per word of its uint4, advanced by Horner's rule with the
// fixed stride of 512 bytes:      c <- c * x^(8*512) mod P  xor  W.
// Multiplying by the constant x^(8*512) is four byte-indexed table lookups (the same shape
// as the reference's slicing-by-4 step, but for a 512-byte jump).  The four tables live in
// shared memory replicated once per bank (entry v of table t for lane l at word
// (t*256+v)*32 + l), so a warp's 32 lookups always hit 32 distinct banks: one lookup per
// input byte at the full shared-memory rate, no bank conflicts, and no staging of the data
// itself -- it goes global -> registers exactly once.
// At the end of a segment each lane register is moved to the segment end with a modular
// multiply by a per-lane constant, lanes are XOR-reduced, and one partial record per warp
// goes to global memory.  A final one-block kernel moves every partial to the end of the
// buffer (multiply by x^(8*suffix) assembled from precomputed x^(8*2^k)), folds in the
// unaligned head/tail bytes and the 0xffffffff pre/post conditioning.
//
// Adler-32 rides along: per 16 bytes three dp4a-fed accumulators give the plain sum, the
// iteration-weighted sum and the in-piece weighted sum, from which s1/s2 partials follow in
// closed form (the deferred-modulo idea of adler32.c:97-106, with the bound set by u32).
//
// Roofline: HBM.  Algorithmic bytes = len (read once), 8 bytes written.
#include "zb_deflate.cuh"

namespace zb {

constexpr int kStride = 512;               // bytes a warp consumes per iteration
constexpr int kMainThreads = 1024;
constexpr int kMainWarps = kMainThreads / 32;
constexpr uint32_t kMaxIters = 1024;       // keeps the u32 Adler accumulators exact (see below)
constexpr size_t kMainThreshold = 1u << 20;                      // below this the stripe kernel runs alone
constexpr int kStripeThreads = 256;
constexpr uint32_t kMaxStripe = 4096;      // u32 bound for the serial s2 accumulation

struct Partial {
    uint32_t reg;                          // raw CRC register contribution at `end`
    uint32_t a, b;                         // Adler sums (mod 65521) of the covered bytes, relative to `end`
    uint32_t pad;
    uint64_t end;                          // byte offset one past the covered range; 0 = unused record
};

__device__ uint32_t g_tab_stride[4][256];  // v<<(8t) times x^(8*512)
__device__ __align__(128) uint32_t g_tab_image[32768];   // the same four tables in the bank-replicated shared-memory layout of k_checksum_main (128 KiB)
__device__ uint32_t g_tab_byte[256];       // the classic byte table (crc32.h table 0)
__device__ uint32_t g_lane_mul[128];       // x^(8*(512 - 16*lane - 4*k))
__constant__ uint32_t c_pow8[64];          // x^(8*2^k) mod P

static unsigned long h_crc_table[256];
const unsigned long* host_crc_table() { return h_crc_table; }

// ---- GF(2) helpers: reflected representation, bit 31 = x^0, right shift = times x ----
__host__ __device__ inline uint32_t gf2_mul(uint32_t a, uint32_t b)
{
    uint32_t r = 0;
#pragma unroll 4
    for (int i = 31; i >= 0; --i) {
        r ^= a & (0u - ((b >> i) & 1u));
        a = (a >> 1) ^ (kCrcPoly & (0u - (a & 1u)));
    }
    return r;
}

__device__ inline uint32_t pow8(uint64_t nbytes)          // x^(8*nbytes) mod P
{
    uint32_t acc = 0x80000000u;
    bool first = true;
    for (int k = 0; nbytes; ++k, nbytes >>= 1)
        if (nbytes & 1) {
            acc = first ? c_pow8[k] : gf2_mul(acc, c_pow8[k]);
            first = false;
        }
    return acc;
}

static uint32_t host_pow8(uint64_t nbytes)
{
    uint32_t acc = 0x80000000u, p = 0x00800000u;          // x^0, x^8
    for (; nbytes; nbytes >>= 1) {
        if (nbytes & 1) acc = gf2_mul(acc, p);
        p = gf2_mul(p, p);
    }
    return acc;
}

int checksum_setup()
{
    uint32_t tab0[256], tabs[4][256], lane_mul[128], pw[64];
    for (uint32_t n = 0; n < 256; n++) {
        uint32_t c = n;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ kCrcPoly : c >> 1;
        tab0[n] = c;
        h_crc_table[n] = c;
    }
    const uint32_t xs = host_pow8(kStride);
    for (int t = 0; t < 4; t++)
        for (uint32_t v = 0; v < 256; v++) tabs[t][v] = gf2_mul(v << (8 * t), xs);
    for (int lane = 0; lane < 32; lane++)
        for (int k = 0; k < 4; k++) lane_mul[lane * 4 + k] = host_pow8((uint64_t)(kStride - 16 * lane - 4 * k));
    uint32_t p = 0x00800000u;
    for (int k = 0; k < 64; k++) { pw[k] = p; p = gf2_mul(p, p); }
    ZB_CUDA(cudaMemcpyToSymbol(g_tab_stride, tabs, sizeof(tabs)));
    {   // word i of the image: table t = 2 * (i >> 14) + ((i >> 5) & 1), entry v = (i >> 6) & 255, replicated over the 32 banks
        static uint32_t image[32768];
        for (uint32_t i = 0; i < 32768; i++) image[i] = tabs[((i >> 14) << 1) | ((i >> 5) & 1u)][(i >> 6) & 255u];
        ZB_CUDA(cudaMemcpyToSymbol(g_tab_image, image, sizeof(image)));
    }
    ZB_CUDA(cudaMemcpyToSymbol(g_tab_byte, tab0, sizeof(tab0)));
    ZB_CUDA(cudaMemcpyToSymbol(g_lane_mul, lane_mul, sizeof(lane_mul)));
    ZB_CUDA(cudaMemcpyToSymbol(c_pow8, pw, sizeof(pw)));
    return 0;
}

// ---- main kernel: aligned bulk, one segment of `iters_per_warp` x 512 B per warp ----
// Table image in shared memory: entry v of table t for lane l is the word at byte offset
//     (t >> 1) * 65536 + v * 256 + (t & 1) * 128 + l * 4
// from a 64 KiB-aligned shared address, so bank = l (a warp's 32 lookups never conflict) and the address of a lookup
// is ONE byte permute: byte 1 of the address is the index byte of the register, bytes 0, 2, 3 come from a per-lane
// constant (PRMT), instead of extract + scale + add.  The kernel is instruction bound, so this is what moves it.
// The image itself arrives by TMA: one thread issues two 64 KiB bulk copies (cp.async.bulk, SASS UBLKCP) from the
// ready-made image in global memory and everybody waits on the mbarrier -- 32 scattered stores per thread before.
// The combine tree runs in the same launch: the last CTA to publish its record folds all of them (see fold_records).
constexpr uint32_t kPrefetchAhead = 16;                          // iterations (512 B each) between an L2 prefetch and its use
constexpr uint32_t kTabImage = 2 * 65536;                       // bytes of the table image
constexpr size_t kMainSmem = 65536 + kTabImage;                 // 64 KiB of alignment room + image

struct FoldArgs {                                               // per-launch constants of the combine, computed on the host
    uint32_t pw_stride[10];                                     // x^(8 * S * G * 2^k), S = bytes one CTA covers, G = group
    uint32_t pw_cta;                                            // X = x^(8 * S)
    uint32_t group;                                             // G: records one fold thread takes before the tree
    uint32_t pw_warp[5];                                        // x^(8 * W * 2^k), W = bytes one warp covers
    uint32_t pw_last;                                           // x^(8 * D): from the end of the last full CTA to the end of the last CTA
    uint32_t pw_tail;                                           // x^(8 * (len - aligned end)): over the ragged tail
    uint32_t pw_head;                                           // x^(8 * (len - head)): from the end of the head bytes to the end
    uint32_t pw_len;                                            // x^(8 * len): for the 0xffffffff pre-conditioning
    uint64_t cta_bytes;                                         // S
};

__device__ __forceinline__ uint32_t lds32(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

__device__ __forceinline__ uint32_t stride_step(uint32_t c, uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3)
{
    return lds32(__byte_perm(c, k0, 0x7604)) ^ lds32(__byte_perm(c, k1, 0x7614)) ^
           lds32(__byte_perm(c, k2, 0x7624)) ^ lds32(__byte_perm(c, k3, 0x7634));
}

__device__ __forceinline__ uint4 ld_stream(const uint4* p)
{
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// ---- mbarrier / bulk-copy primitives (PTX; SASS: SYNCS.*, UBLKCP) ----
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// One 512-byte iteration of a warp: four Horner steps per lane and the three Adler accumulators.
#define ZB_CK_STEP(W, J)                                                                                              \
    do {                                                                                                              \
        c0 = stride_step(c0, k0, k1, k2, k3) ^ (W).x; c1 = stride_step(c1, k0, k1, k2, k3) ^ (W).y;                    \
        c2 = stride_step(c2, k0, k1, k2, k3) ^ (W).z; c3 = stride_step(c3, k0, k1, k2, k3) ^ (W).w;                    \
        const uint32_t sum_ = __dp4a((W).x, 0x01010101u, __dp4a((W).y, 0x01010101u, __dp4a((W).z, 0x01010101u, __dp4a((W).w, 0x01010101u, 0u)))); \
        s_b = __dp4a((W).x, 0x0d0e0f10u, __dp4a((W).y, 0x090a0b0cu, __dp4a((W).z, 0x05060708u, __dp4a((W).w, 0x01020304u, s_b)))); \
        s_a += sum_; s_j += (J) * sum_;                                                                               \
    } while (0)

// The combine tree, run by the last CTA (1024 threads): record i of the grid covers bytes up to
//   end_i = base + (i + 1) * S   (i < n - 1),      end_{n-1} = base + aligned length,
// so with q counted from the back over the first n - 1 records the register at the aligned end is
//   ( sum_q u_q X^q ) * x^(8 D)  xor  u_last,      X = x^(8 S),
// a polynomial in X evaluated by pairing neighbours: ten levels of ONE modular multiply per thread with the host's
// X^(2^k), instead of one modular power per record.  With more than 1024 + 1 records (seven rounds of resident warps
// and more: from 13.875 GiB with 148 SMs) thread t first folds records q = tG .. tG + G - 1 by Horner's rule in X, and the tree
// then runs in X^G.  Head and tail bytes, the pre-conditioning and the Adler sums (closed form per record) are folded
// in the same pass.
__device__ void fold_records(const Partial* __restrict__ parts, uint32_t n_parts, const uint8_t* __restrict__ buf, uint64_t len,
                             uint64_t head, uint64_t tail_begin, const FoldArgs& fa, uint32_t* __restrict__ out2, uint32_t* s_x)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t m = n_parts - 1;                             // records with the uniform spacing
    // ---- CRC: u_q = record m - 1 - q ----
    uint32_t u = 0, a = 0, b = 0;
    // (the records were published with a fence before the counter moved; volatile loads keep them out of registers cached earlier)
    for (uint32_t i = tid; i < n_parts; i += blockDim.x) {
        const volatile Partial* vp = parts + i;
        const uint32_t pa = vp->a, pb = vp->b;
        const uint64_t end = vp->end;
        if (end == 0) continue;
        const uint64_t suffix = len - end;
        a += pa;
        b = (b + pb + (uint32_t)((suffix % kAdlerBase) * pa % kAdlerBase)) % kAdlerBase;
        a %= kAdlerBase;
    }
    if (fa.group == 1) {
        if ((uint32_t)tid < m) u = ((const volatile Partial*)(parts + (m - 1 - tid)))->reg;
    } else {
        for (uint32_t i = fa.group; i-- > 0;) {                 // u = sum_i u_(tG + i) X^i
            const uint64_t q = (uint64_t)tid * fa.group + i;
            if (q < m) u = gf2_mul(u, fa.pw_cta) ^ ((const volatile Partial*)(parts + (m - 1 - q)))->reg;
        }
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {                               // levels inside a warp: lane q takes lane q + 2^k
        const uint32_t hi = __shfl_down_sync(0xffffffffu, u, 1u << k);
        if ((lane & ((2 << k) - 1)) == 0) u ^= gf2_mul(hi, fa.pw_stride[k]);
    }
    if (lane == 0) s_x[warp] = u;
    __syncthreads();
    uint32_t reg = 0;
    if (warp == 0) {
        uint32_t v = s_x[lane];
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const uint32_t hi = __shfl_down_sync(0xffffffffu, v, 1u << k);
            if ((lane & ((2 << k) - 1)) == 0) v ^= gf2_mul(hi, fa.pw_stride[5 + k]);
        }
        if (lane == 0) {
            const volatile Partial* last = parts + m;
            uint32_t r = (m ? gf2_mul(v, fa.pw_last) : 0u) ^ last->reg;      // at the aligned end
            r = gf2_mul(r, fa.pw_tail);                                       // at the end of the buffer
            // head bytes (< 16): byte-wise on this lane, then moved to the end with the host's power
            uint32_t hreg = 0;
            for (uint64_t o = 0; o < head; o++) hreg = g_tab_byte[(hreg ^ buf[o]) & 0xffu] ^ (hreg >> 8);
            if (head) r ^= gf2_mul(hreg, fa.pw_head);
            r ^= gf2_mul(0xffffffffu, fa.pw_len);                              // 0xffffffff pre-conditioning
            reg = r;
        }
    }
    // ---- ragged edges: Adler over head and tail bytes; CRC of the tail bytes (< 512), one per thread: its byte-table
    // entry moved to the end of the buffer by a short power (the suffix is below 512) ----
    uint32_t treg = 0;
    const uint64_t n_edge = head + (len - tail_begin);
    for (uint64_t e = tid; e < n_edge; e += blockDim.x) {
        const uint64_t o = e < head ? e : tail_begin + (e - head);
        const uint32_t v = buf[o];
        a = (a + v) % kAdlerBase;
        b = (b + (uint32_t)(((len - o) % kAdlerBase) * v % kAdlerBase)) % kAdlerBase;
        if (e >= head) {
            const uint64_t suffix = len - o - 1;
            const uint32_t r1 = g_tab_byte[v];
            treg ^= suffix ? gf2_mul(r1, pow8(suffix)) : r1;
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o);
        treg ^= __shfl_xor_sync(0xffffffffu, treg, o);
    }
    __shared__ uint32_t s_t[32];
    __syncthreads();                                            // s_x is reused
    if (lane == 0) { s_x[warp] = a % kAdlerBase; s_x[32 + warp] = b % kAdlerBase; s_t[warp] = treg; }
    __syncthreads();
    if (warp == 0) {
        a = s_x[lane]; b = s_x[32 + lane]; treg = s_t[lane];
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o);
            treg ^= __shfl_xor_sync(0xffffffffu, treg, o);
        }
        reg ^= treg;                                            // (lane 0 holds the register; the others' value is unused)
        if (lane == 0) {
            const uint32_t s1 = (1u + a) % kAdlerBase;
            const uint32_t s2 = (uint32_t)((len % kAdlerBase + b) % kAdlerBase);
            out2[0] = ~reg;
            out2[1] = (s2 << 16) | s1;
        }
    }
}

__global__ void __launch_bounds__(kMainThreads, 1)
k_checksum_main(const uint8_t* __restrict__ base, uint64_t n_units, uint32_t iters_per_warp,
                uint64_t base_off, Partial* __restrict__ parts, const uint8_t* __restrict__ buf, uint64_t len,
                uint64_t tail_begin, const FoldArgs fa, uint32_t* __restrict__ out2, unsigned int* __restrict__ done_ctas)
{
    extern __shared__ __align__(128) uint8_t s_raw[];
    __shared__ Partial s_part[kMainWarps];
    __shared__ __align__(8) uint64_t s_bar;                   // the table image has landed
    __shared__ uint32_t s_x[64];
    __shared__ uint32_t s_last;
    const uint32_t raw = (uint32_t)__cvta_generic_to_shared(s_raw);
    const uint32_t img = (raw + 65535u) & ~65535u;              // shared address of the image
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&s_bar);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        mbar_init(bar0, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(bar0, kTabImage);
        bulk_g2s(img, g_tab_image, 65536, bar0);
        bulk_g2s(img + 65536, reinterpret_cast<const uint8_t*>(g_tab_image) + 65536, 65536, bar0);
    }
    __syncthreads();

    const uint64_t warp = (uint64_t)blockIdx.x * kMainWarps + wid;
    const uint64_t u0 = warp * iters_per_warp;
    Partial mine{0, 0, 0, 0, 0};
    const uint32_t iters = u0 < n_units ? (uint32_t)min((uint64_t)iters_per_warp, n_units - u0) : 0u;
    const uint8_t* seg = base + u0 * kStride;
    mbar_wait(bar0, 0);                                         // the table image has landed

    if (iters) {
        const uint4* p = reinterpret_cast<const uint4*>(seg) + lane;
        const uint32_t k0 = img + lane * 4, k1 = k0 + 128, k2 = k0 + 65536, k3 = k2 + 128;
        uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
        uint32_t s_a = 0, s_j = 0, s_b = 0;    // sum, iteration-weighted sum, in-piece weighted sum
        uint32_t j = 0;
        // two loads in flight per lane
        for (; j + 2 <= iters; j += 2) {
            // two iterations use 1 KiB per warp; ask L2 for the 1 KiB that is kPrefetchAhead iterations away (registers cap
            // the loads in flight at two per lane, which alone does not cover the HBM latency-bandwidth product)
            if (lane < 8) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const uint8_t*>(p - lane) + (size_t)min(j + kPrefetchAhead, iters - 2) * kStride + (lane * 128) % 1024));
            const uint4 w0 = ld_stream(p + (size_t)j * 32);
            const uint4 w1 = ld_stream(p + (size_t)(j + 1) * 32);
            ZB_CK_STEP(w0, j);
            ZB_CK_STEP(w1, j + 1);
        }
        for (; j < iters; ++j) {
            const uint4 w0 = ld_stream(p + (size_t)j * 32);
            ZB_CK_STEP(w0, j);
        }

        // Move the four lane registers to the end of the segment and reduce across the warp.
        uint32_t reg = gf2_mul(c0, g_lane_mul[lane * 4 + 0]) ^ gf2_mul(c1, g_lane_mul[lane * 4 + 1]) ^
                       gf2_mul(c2, g_lane_mul[lane * 4 + 2]) ^ gf2_mul(c3, g_lane_mul[lane * 4 + 3]);
        // Adler: byte at segment offset o = 512 j + 16 lane + t weighs (L - o).
        const uint64_t L = (uint64_t)iters * kStride;
        uint64_t bw = (L - 16u * lane - 16u) * (uint64_t)s_a + (uint64_t)s_b - (uint64_t)kStride * s_j;
        uint32_t a = s_a % kAdlerBase, b = (uint32_t)(bw % kAdlerBase);
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            reg ^= __shfl_xor_sync(0xffffffffu, reg, o);
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        mine = Partial{reg, a % kAdlerBase, b % kAdlerBase, 0, base_off + (u0 + iters) * kStride};
    }
    // The CTA's warps cover consecutive segments: fold their partials to the end of the last one here (one modular
    // power per warp, all CTAs at once), so the combine sees one record per CTA instead of one per warp.
    if (lane == 0) s_part[wid] = mine;
    __syncthreads();
    if (wid == 0) {
        const Partial p = s_part[lane];
        uint64_t cta_end = p.end;
#pragma unroll
        for (int o = 16; o; o >>= 1) { const uint64_t y = __shfl_xor_sync(0xffffffffu, cta_end, o); cta_end = y > cta_end ? y : cta_end; }
        uint32_t reg = 0, a = 0, b = 0;
        if (p.end) {
            const uint64_t suffix = cta_end - p.end;
            a = p.a;
            b = (p.b + (uint32_t)((suffix % kAdlerBase) * p.a % kAdlerBase)) % kAdlerBase;
        }
        if (blockIdx.x + 1 < gridDim.x) {
            // every warp of this CTA ran the full iters_per_warp: warp w ends (31 - w) * W bytes in front of the CTA's end, so the
            // register at the CTA's end is a polynomial in Y = x^(8 W) -- five levels of one multiply with the host's Y^(2^k)
            uint32_t u = __shfl_sync(0xffffffffu, p.reg, 31 - lane);      // u_q = warp 31 - q
#pragma unroll
            for (int k = 0; k < 5; k++) {
                const uint32_t hi = __shfl_down_sync(0xffffffffu, u, 1u << k);
                if ((lane & ((2 << k) - 1)) == 0) u ^= gf2_mul(hi, fa.pw_warp[k]);
            }
            reg = u;                                            // lane 0 holds it
#pragma unroll
            for (int o = 16; o; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
        } else {                                                // the last CTA: ragged, one modular power per warp
            if (p.end) { const uint64_t suffix = cta_end - p.end; reg = suffix ? gf2_mul(p.reg, pow8(suffix)) : p.reg; }
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                reg ^= __shfl_xor_sync(0xffffffffu, reg, o);
                a += __shfl_xor_sync(0xffffffffu, a, o);
                b += __shfl_xor_sync(0xffffffffu, b, o);
            }
        }
        if (lane == 0) {
            parts[blockIdx.x] = Partial{reg, a % kAdlerBase, b % kAdlerBase, 0, cta_end};
            __threadfence();                                    // the record is visible before the count moves
            s_last = atomicAdd(done_ctas, 1u) == gridDim.x - 1 ? 1u : 0u;
        }
    }
    __syncthreads();
    if (s_last) {                                               // every record of the grid is published: fold them
        __threadfence();
        fold_records(parts, gridDim.x, buf, len, base_off, tail_begin, fa, out2, s_x);
        if (threadIdx.x == 0) *done_ctas = 0;                   // ready for the next launch with this context (a context serves one stream at a time)
    }
}

// ---- stripe kernel: small or ragged ranges, one contiguous stripe per thread ----
__global__ void __launch_bounds__(kStripeThreads)
k_checksum_stripes(const uint8_t* __restrict__ buf, uint64_t len, uint32_t stripe, Partial* __restrict__ parts)
{
    __shared__ uint32_t s_tab[256];
    s_tab[threadIdx.x] = g_tab_byte[threadIdx.x];
    __syncthreads();
    const uint64_t t = (uint64_t)blockIdx.x * kStripeThreads + threadIdx.x;
    const uint64_t beg = t * stripe;
    if (beg >= len) { parts[t] = Partial{0, 0, 0, 0, 0}; return; }
    const uint64_t end = min(len, beg + stripe);
    uint32_t c = 0, a = 0, b = 0;
    for (uint64_t i = beg; i < end; ++i) {
        uint32_t v = buf[i];
        c = s_tab[(c ^ v) & 0xffu] ^ (c >> 8);
        a += v; b += a;
    }
    parts[t] = Partial{c, a % kAdlerBase, b % kAdlerBase, 0, end};
}

// ---- final kernel: combine tree over partial records + ragged edge bytes ----
__global__ void __launch_bounds__(1024, 1)
k_checksum_final(const Partial* __restrict__ parts, uint32_t n_parts, const uint8_t* __restrict__ buf,
                 uint64_t len, uint64_t head, uint64_t tail_begin, uint32_t* __restrict__ out2)
{
    __shared__ uint32_t s_reg[32], s_a[32], s_b[32];
    uint32_t reg = 0, a = 0, b = 0;
    for (uint32_t i = threadIdx.x; i < n_parts; i += blockDim.x) {
        Partial p = parts[i];
        if (p.end == 0) continue;
        uint64_t suffix = len - p.end;
        reg ^= suffix ? gf2_mul(p.reg, pow8(suffix)) : p.reg;
        a += p.a;
        b = (b + p.b + (uint32_t)((suffix % kAdlerBase) * p.a % kAdlerBase)) % kAdlerBase;
        a %= kAdlerBase;
    }
    const uint64_t n_edge = head + (len - tail_begin);
    for (uint64_t e = threadIdx.x; e < n_edge; e += blockDim.x) {
        uint64_t o = e < head ? e : tail_begin + (e - head);
        uint32_t v = buf[o];
        uint64_t suffix = len - o - 1;
        uint32_t r1 = g_tab_byte[v];
        reg ^= suffix ? gf2_mul(r1, pow8(suffix)) : r1;
        a = (a + v) % kAdlerBase;
        b = (b + (uint32_t)(((len - o) % kAdlerBase) * v % kAdlerBase)) % kAdlerBase;
    }
    if (threadIdx.x == 0) reg ^= len ? gf2_mul(0xffffffffu, pow8(len)) : 0xffffffffu;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        reg ^= __shfl_xor_sync(0xffffffffu, reg, o);
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_reg[warp] = reg; s_a[warp] = a % kAdlerBase; s_b[warp] = b % kAdlerBase; }
    __syncthreads();
    if (warp == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        reg = lane < nw ? s_reg[lane] : 0; a = lane < nw ? s_a[lane] : 0; b = lane < nw ? s_b[lane] : 0;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            reg ^= __shfl_xor_sync(0xffffffffu, reg, o);
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (lane == 0) {
            uint32_t s1 = (1u + a) % kAdlerBase;
            uint32_t s2 = (uint32_t)((len % kAdlerBase + b) % kAdlerBase);
            out2[0] = ~reg;
            out2[1] = (s2 << 16) | s1;
        }
    }
}

// ---- batch kernel: one CTA per buffer (per-member CRCs of an archive, per-stream checks after a batch inflate) ----
// Thread t runs the byte table over its contiguous stripe (crc32.c:244-252 DO1, adler32.c:66-70), then the CTA moves
// every stripe's register to the end of the buffer and folds -- the combine tree of k_checksum_final, per buffer.
// len == nullptr: buffer i is [off[i], off[i+1]).  expect != nullptr: out2 is not written; instead ok[i] is cleared
// to Z_DATA_ERROR when the pair differs from expect[3i], expect[3i+1] (crc32, length mod 2^32: a gzip trailer;
// expect[3i+2] == 0 means buffer i has no such trailer).
__global__ void __launch_bounds__(kStripeThreads)
k_checksum_batch(const uint8_t* __restrict__ base, const uint64_t* __restrict__ off, const uint64_t* __restrict__ lens,
                 uint32_t* __restrict__ crc_out, uint32_t* __restrict__ adler_out, const uint32_t* __restrict__ expect,
                 int32_t* __restrict__ ok, const ChunkDesc* __restrict__ cd)
{
    __shared__ uint32_t s_tab[256];
    __shared__ uint32_t s_reg[kStripeThreads / 32], s_a[kStripeThreads / 32], s_b[kStripeThreads / 32];
    s_tab[threadIdx.x] = g_tab_byte[threadIdx.x];
    __syncthreads();
    const uint64_t i = blockIdx.x;
    if (expect && (ok[i] != 0 || expect[3 * i + 2] == 0)) return;   // failed already, or not a gzip member
    const uint8_t* buf = base + (cd ? (uint64_t)cd[i].beg : off[i]);
    const uint64_t len = cd ? (uint64_t)cd[i].len : lens ? lens[i] : off[i + 1] - off[i];
    const uint64_t stripe = (len + kStripeThreads - 1) / kStripeThreads;
    const uint64_t beg = min(len, (uint64_t)threadIdx.x * stripe), end = min(len, beg + stripe);
    uint32_t c = 0, a = 0, b = 0;                             // raw register, byte sum, sum of prefix sums (both mod 65521)
    for (uint64_t p = beg; p < end;) {
        const uint64_t stop = min(end, p + 4096);             // u32 bound for the deferred modulo
        uint32_t aa = 0, bb = 0;
        const uint32_t n = (uint32_t)(stop - p);
        // bytes up to a 16-byte boundary, then 16 bytes per load (a thread's stripe is contiguous, so byte loads would
        // cost a cache wavefront per byte and lane), then the ragged end
        for (; p < stop && ((uintptr_t)(buf + p) & 15u); ++p) {
            const uint32_t v = buf[p];
            c = s_tab[(c ^ v) & 0xffu] ^ (c >> 8);
            aa += v; bb += aa;
        }
        for (; p + 16 <= stop; p += 16) {
            const uint4 q = *reinterpret_cast<const uint4*>(buf + p);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                c ^= w[k];
#pragma unroll
                for (int j = 0; j < 4; j++) c = s_tab[c & 0xffu] ^ (c >> 8);
                bb += 4u * aa + __dp4a(w[k], 0x01020304u, 0u);  // byte 0 of the word comes first: weight 4
                aa += __dp4a(w[k], 0x01010101u, 0u);
            }
        }
        for (; p < stop; ++p) {
            const uint32_t v = buf[p];
            c = s_tab[(c ^ v) & 0xffu] ^ (c >> 8);
            aa += v; bb += aa;
        }
        b = (b + (uint32_t)((uint64_t)n * a % kAdlerBase) + bb % kAdlerBase) % kAdlerBase;
        a = (a + aa) % kAdlerBase;
    }
    // move to the end of the buffer: register times x^(8*suffix); Adler sums shift by suffix * a
    const uint64_t suffix = len - end;
    uint32_t reg = (end > beg && suffix) ? gf2_mul(c, pow8(suffix)) : c;
    if (end == beg) { reg = 0; a = 0; b = 0; }
    b = (b + (uint32_t)((suffix % kAdlerBase) * a % kAdlerBase)) % kAdlerBase;
    if (threadIdx.x == 0) reg ^= len ? gf2_mul(0xffffffffu, pow8(len)) : 0xffffffffu;   // the 0xffffffff pre-conditioning
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        reg ^= __shfl_xor_sync(0xffffffffu, reg, o);
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_reg[warp] = reg; s_a[warp] = a % kAdlerBase; s_b[warp] = b % kAdlerBase; }
    __syncthreads();
    if (threadIdx.x == 0) {
        reg = 0; a = 0; b = 0;
        for (int w = 0; w < kStripeThreads / 32; w++) { reg ^= s_reg[w]; a += s_a[w]; b += s_b[w]; }
        const uint32_t s1 = (1u + a) % kAdlerBase;
        const uint32_t s2 = (uint32_t)((len % kAdlerBase + b) % kAdlerBase);
        const uint32_t crc = ~reg, adl = (s2 << 16) | s1;
        if (expect) {
            if (crc != expect[3 * i] || (uint32_t)len != expect[3 * i + 1]) ok[i] = ZB_DATA_ERROR;
        } else {
            if (crc_out) crc_out[i] = crc;
            if (adler_out) adler_out[i] = adl;
        }
    }
}

int checksum_batch_launch(const uint8_t* d_base, const uint64_t* d_off, const uint64_t* d_lens, size_t n, uint32_t* d_crc,
                          uint32_t* d_adler, const uint32_t* d_expect, int32_t* d_ok, cudaStream_t s)
{
    if (n == 0) return 0;
    ZB_LAUNCH(k_checksum_batch, (unsigned)n, kStripeThreads, 0, s, d_base, d_off, d_lens, d_crc, d_adler, d_expect, d_ok,
              (const ChunkDesc*)nullptr);
    ZB_CHECK_LAUNCH();
    return 0;
}

// Job mode of the deflate batch: checksums per chunk (one CTA each, so a 16 MiB member is 128 CTAs, not one), then one
// thread per job folds its chunks in order with crc32_combine / adler32_combine (crc32.c:370-423, adler32.c:128-149).
__global__ void k_checksum_join_jobs(const uint32_t* __restrict__ ccrc, const uint32_t* __restrict__ cadl,
                                     const ChunkDesc* __restrict__ cd, const JobDesc* __restrict__ jobs, uint32_t njobs,
                                     uint32_t* __restrict__ crc_out, uint32_t* __restrict__ adler_out)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= njobs) return;
    const JobDesc jd = jobs[j];
    uint32_t crc = 0, s1 = 1, s2 = 0;
    const uint32_t xfull = pow8(ZB200_CHUNK);
    for (uint32_t k = 0; k < jd.nchunks; k++) {
        const uint32_t c = jd.first_chunk + k, len = cd[c].len;
        crc = gf2_mul(crc, len == ZB200_CHUNK ? xfull : pow8(len)) ^ ccrc[c];
        const uint32_t a2 = cadl[c], rem = len % kAdlerBase;
        s2 = (s2 + (uint32_t)((uint64_t)rem * s1 % kAdlerBase) + (a2 >> 16) + kAdlerBase - rem) % kAdlerBase;
        s1 = (s1 + (a2 & 0xffffu) + kAdlerBase - 1) % kAdlerBase;
    }
    crc_out[j] = crc;
    adler_out[j] = (s2 << 16) | s1;
}

int checksum_jobs_launch(Ctx* c, const uint8_t* d_base, const ChunkDesc* d_cd, uint32_t nchunks, const JobDesc* d_jobs,
                         uint32_t njobs, uint32_t* d_crc, uint32_t* d_adler, cudaStream_t s)
{
    int rc = c->ws[0].ensure((size_t)(nchunks + 1) * 8);
    if (rc) return rc;
    uint32_t* d_ccrc = c->ws[0].as<uint32_t>();
    uint32_t* d_cadl = d_ccrc + nchunks;
    if (nchunks)
        ZB_LAUNCH(k_checksum_batch, nchunks, kStripeThreads, 0, s, d_base, (const uint64_t*)nullptr, (const uint64_t*)nullptr, d_ccrc,
                  d_cadl, (const uint32_t*)nullptr, (int32_t*)nullptr, d_cd);
    ZB_LAUNCH(k_checksum_join_jobs, (njobs + 127) / 128, 128, 0, s, d_ccrc, d_cadl, d_cd, d_jobs, njobs, d_crc, d_adler);
    ZB_CHECK_LAUNCH();
    return 0;
}

int checksum_attr_setup()                                      // once per device, from ensure_init
{
    ZB_CUDA(cudaFuncSetAttribute(k_checksum_main, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMainSmem));
    return 0;
}

int checksum_launch(Ctx* c, const uint8_t* d_buf, size_t len, uint32_t* d_out2, cudaStream_t s)
{
    if (len < kMainThreshold) {
        // one stripe kernel over everything
        uint32_t threads_wanted = (uint32_t)((len + 63) / 64);
        uint32_t blocks = (threads_wanted + kStripeThreads - 1) / kStripeThreads;
        if (blocks < 1) blocks = 1;
        if (blocks > (uint32_t)device_sms()) blocks = (uint32_t)device_sms();
        uint64_t nthreads = (uint64_t)blocks * kStripeThreads;
        uint32_t stripe = (uint32_t)((len + nthreads - 1) / nthreads);
        if (stripe < 16) stripe = 16;
        int rc = c->ws[0].ensure(nthreads * sizeof(Partial));
        if (rc) return rc;
        ZB_LAUNCH(k_checksum_stripes, blocks, kStripeThreads, 0, s, d_buf, (uint64_t)len, stripe, c->ws[0].as<Partial>());
        ZB_LAUNCH(k_checksum_final, 1, 1024, 0, s, c->ws[0].as<Partial>(), (uint32_t)nthreads, d_buf, (uint64_t)len,
                  (uint64_t)0, (uint64_t)len, d_out2);
        ZB_CHECK_LAUNCH();
        return 0;
    }
    const uint64_t head = (16 - ((uintptr_t)d_buf & 15)) & 15;
    const uint64_t n_units = (len - head) / kStride;
    const uint64_t tail_begin = head + n_units * kStride;
    // every resident warp gets the same number of iterations; several rounds only for huge inputs
    uint64_t warps = (uint64_t)device_sms() * kMainWarps;
    uint64_t rounds = (n_units + warps * kMaxIters - 1) / (warps * kMaxIters);
    uint64_t total_warps = warps * rounds;
    uint32_t iters = (uint32_t)((n_units + total_warps - 1) / total_warps);
    if (iters < 8) iters = 8;
    uint64_t used_warps = (n_units + iters - 1) / iters;
    uint32_t blocks = (uint32_t)((used_warps + kMainWarps - 1) / kMainWarps);
    uint64_t n_parts = blocks;                                  // one record per CTA
    int rc = c->ws[0].ensure(n_parts * sizeof(Partial));
    if (rc) return rc;
    if ((rc = c->ensure_flags()) != 0) return rc;
    unsigned int* done = c->flags.as<unsigned int>();            // zero between launches (the last CTA resets it)
    // constants of the combine (fold_records): powers of x for the uniform spacing of the CTA records and for the edges
    FoldArgs fa;
    const uint64_t S = (uint64_t)kMainWarps * iters * kStride;
    fa.cta_bytes = S;
    fa.group = (uint32_t)((blocks - 1 + 1023) / 1024);             // the tree pairs 1024 values; rounds past 6 give it more records
    if (fa.group == 0) fa.group = 1;
    fa.pw_cta = host_pow8(S);
    for (int k = 0; k < 10; k++) fa.pw_stride[k] = host_pow8((S * fa.group) << k);
    for (int k = 0; k < 5; k++) fa.pw_warp[k] = host_pow8(((uint64_t)iters * kStride) << k);
    const uint64_t aligned = n_units * kStride;
    fa.pw_last = host_pow8(aligned - (uint64_t)(blocks - 1) * S);
    fa.pw_tail = host_pow8(len - tail_begin);
    fa.pw_head = host_pow8(len - head);
    fa.pw_len = host_pow8(len);
    ZB_LAUNCH(k_checksum_main, blocks, kMainThreads, kMainSmem, s, d_buf + head, n_units, iters, head, c->ws[0].as<Partial>(),
              d_buf, (uint64_t)len, tail_begin, fa, d_out2, done);
    ZB_CHECK_LAUNCH();
    return 0;
}

}  // namespace zb

using namespace zb;

ZB_API int zb200_checksum_dev(const void* d_buf, size_t len, uint32_t* d_out2, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    rc = checksum_launch(c, static_cast<const uint8_t*>(d_buf), len, d_out2, s);
    ctx_release(c, s);
    return rc;
}

ZB_API int zb200_checksum(const void* buf, size_t len, uint32_t* crc, uint32_t* adler, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    do {
        const uint8_t* d = to_device(c, buf, len, s, &rc);
        if (rc) break;
        if ((rc = c->small.ensure(256)) != 0) break;
        if ((rc = c->ensure_pinned(256)) != 0) break;
        if ((rc = checksum_launch(c, d, len, c->small.as<uint32_t>(), s)) != 0) break;
        if (cudaMemcpyAsync(c->pinned, c->small.p, 8, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
            cudaStreamSynchronize(s) != cudaSuccess) {
            set_error("checksum readback failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = ZB_STREAM_ERROR;
            break;
        }
        const uint32_t* r = static_cast<const uint32_t*>(c->pinned);
        if (crc) *crc = r[0];
        if (adler) *adler = r[1];
    } while (0);
    ctx_release(c, s);
    return rc;
}

ZB_API int zb200_checksum_batch(const void* base, const uint64_t* offsets, size_t n, uint32_t* crc, uint32_t* adler, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (n == 0) return 0;
    if (!offsets) { set_error("zb200_checksum_batch: bad argument"); return ZB_STREAM_ERROR; }
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    do {
        const uint8_t* d = to_device(c, base, (size_t)offsets[n], s, &rc);
        if (rc) break;
        // [offsets n+1 (u64)][crc n][adler n]
        if ((rc = c->ws[0].ensure((n + 1) * 8 + n * 8)) != 0) break;
        if ((rc = c->ensure_pinned(n * 8)) != 0) break;
        uint64_t* d_off = c->ws[0].as<uint64_t>();
        uint32_t* d_crc = (uint32_t*)(d_off + n + 1);
        uint32_t* d_adl = d_crc + n;
        cudaError_t e = cudaMemcpyAsync(d_off, offsets, (n + 1) * 8, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) { set_error("offset upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        if ((rc = checksum_batch_launch(d, d_off, nullptr, n, d_crc, d_adl, nullptr, nullptr, s)) != 0) break;
        e = cudaMemcpyAsync(c->pinned, d_crc, n * 8, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { set_error("checksum batch failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        const uint32_t* r = static_cast<const uint32_t*>(c->pinned);
        for (size_t i = 0; i < n; i++) {
            if (crc) crc[i] = r[i];
            if (adler) adler[i] = r[n + i];
        }
    } while (0);
    ctx_release(c, s);
    return rc;
}
