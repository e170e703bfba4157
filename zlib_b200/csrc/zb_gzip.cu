// zb_gzip.cu -- gzip files of several members (RFC 1952 2.2) read on the GPU, and BGZF (SAM/BAM specification 4.1) written.
//
// A gzip file is a run of members, and nothing but decoding a member tells where the next one starts.  Instead of decoding
// them one after the other, zb200_gunzip guesses the member table from the bytes and then checks the guess:
//   1. k_gz_scan finds every position that opens a plausible member header (1f 8b 08, no reserved flag bit, a header that
//      ends inside the file) and records its header length, the BGZF block size if the 'BC' subfield is there, and the 8
//      bytes in front of it -- the CRC-32 and ISIZE of the member before it, if the candidate is real.
//   2. The plan: a member starts at offset 0; a BGZF member chains to pos + BSIZE + 1, so only candidates on the chain are
//      taken; any other candidate is taken as a member start.  Member k is the deflate data between its header and the 8
//      bytes in front of member k + 1 (the file's last 8 bytes for the last member), with the CRC-32 and ISIZE found there.
//   3. All members are decoded at once by decode_members (zb_zip.cu, the routes of the ZIP reader) and each must pass every
//      check: decoder status, deflate data ending in the last byte of its span, length = ISIZE, CRC-32.  Compressed data may
//      hold 1f 8b 08 00 (a stored .tar.gz holds its inner .gz files verbatim); a spurious candidate splits a member into
//      two spans, and neither can end exactly at its span's end with a matching trailer, so a wrong plan costs time only.
//   4. The file is then walked from offset 0: a verified member at the walk's position is taken as planned; anywhere else
//      one member is decoded at a time from the position (one-stream parallel decoder, else one warp), which also says
//      where it ends, until the position meets a verified member again or the file ends.  Zero padding between members and
//      every kind of damage land here; the walk names the first member it cannot decode.
// The output of the plan and of the walk are laid out by k_zip_gather pieces (or per-piece D2H copies), never by an
// overlapping copy in place.  When every planned member verifies, the plan's output is the result and nothing moves.
//
// zb200_bgzf_compress runs job-mode deflate (zb_deflate.cu) over 65280-byte jobs with BGZF framing, lays the blocks out
// contiguously with k_zip_gather and appends the BGZF EOF block.
#include "zb_common.cuh"
#include "zb_deflate.cuh"
#include "zb_inflate.cuh"
#include <string.h>
#include <algorithm>
#include <vector>

namespace zb {

constexpr uint64_t kBgzfBlock = 65280;                          // bgzip's BGZF_BLOCK_SIZE: input bytes per block
constexpr uint64_t kBgzfMaxMember = 65536;                      // BSIZE is 16 bits
constexpr uint64_t kBgzfSlot = kBgzfMaxMember + 1024;           // per-block output slot of the batch (above compressBound + framing)
static const uint8_t kBgzfEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
// Bytes of header k_gz_scan reads at one candidate.  Without a bound, every 1f 8b 08 with FNAME set in a file without
// NUL bytes would scan to the end of the file (quadratic).  A real member with a longer header is simply not planned: its
// neighbour fails verification and the walk decodes it, header and all.
constexpr uint32_t kScanHeaderMax = 1024;

struct GzCand {                                                 // 32 bytes
    uint64_t pos;
    uint32_t hdr_len, blen;                                     // blen = BSIZE + 1 of a BGZF header, else 0
    uint32_t crc, isize;                                        // the 8 bytes in front of pos (0 at the start of the file)
    uint32_t hcrc_ok, pad;                                      // 0: FHCRC set and wrong
};

__device__ __forceinline__ uint32_t ld16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__device__ __forceinline__ uint32_t ld32(const uint8_t* p) { return ld16(p) | (ld16(p + 2) << 16); }

// A member header at p (RFC 1952 2.3.1; inflate.c:634-759 for the order of the fields), or nothing.
__device__ void gz_candidate(const uint8_t* __restrict__ in, uint64_t len, uint64_t p, uint32_t* __restrict__ count,
                             GzCand* __restrict__ out, uint32_t cap)
{
    len = min(len, p + kScanHeaderMax);                         // everything below reads in[p .. len)
    if (p + 10 > len || in[p + 1] != 0x8b || in[p + 2] != 8) return;
    const uint32_t flg = in[p + 3];
    if (flg & 0xe0) return;
    uint64_t q = p + 10;
    uint32_t blen = 0;
    if (flg & 4) {                                              // FEXTRA: subfields SI1 SI2 SLEN data
        if (q + 2 > len) return;
        const uint64_t xend = q + 2 + ld16(in + q);
        if (xend > len) return;
        for (uint64_t x = q + 2; x + 4 <= xend;) {
            const uint32_t slen = ld16(in + x + 2);
            if (in[x] == 'B' && in[x + 1] == 'C' && slen == 2 && x + 6 <= xend) blen = ld16(in + x + 4) + 1;
            x += 4 + slen;
        }
        q = xend;
    }
    for (uint32_t f = 8; f <= 16; f <<= 1) {                    // FNAME, FCOMMENT: up to and with their NUL
        if (!(flg & f)) continue;
        while (q < len && in[q] != 0) q++;
        if (q >= len) return;
        q++;
    }
    uint32_t hcrc_ok = 1;
    if (flg & 2) {                                              // FHCRC: low 16 bits of the header's CRC-32 (bitwise: headers are short)
        if (q + 2 > len) return;
        uint32_t c = 0xffffffffu;
        for (uint64_t i = p; i < q; i++) {
            c ^= in[i];
            for (int k = 0; k < 8; k++) c = (c >> 1) ^ (kCrcPoly & (0u - (c & 1u)));
        }
        hcrc_ok = ((~c) & 0xffffu) == ld16(in + q);
        q += 2;
    }
    GzCand r;
    r.pos = p; r.hdr_len = (uint32_t)(q - p); r.blen = blen;
    r.crc = p >= 8 ? ld32(in + p - 8) : 0; r.isize = p >= 8 ? ld32(in + p - 4) : 0;
    r.hcrc_ok = hcrc_ok; r.pad = 0;
    const uint32_t k = atomicAdd(count, 1u);
    if (k < cap) out[k] = r;
}

// Grid-stride over aligned words, like k_find_markers: a word without a 1f byte costs one load and one compare.
__global__ void __launch_bounds__(256) k_gz_scan(const uint8_t* __restrict__ in, uint64_t len, uint32_t* __restrict__ count,
                                                 GzCand* __restrict__ out, uint32_t cap)
{
    const uint32_t mis = (uint32_t)((uintptr_t)in & 3);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(in - mis);
    const uint64_t nw = (len + mis + 3) / 4;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t hit = __vcmpeq4(w[i], 0x1f1f1f1fu);
        while (hit) {
            const int b = __ffs(hit) / 8;                       // byte within the word (0..3)
            hit &= ~(0xffu << (8 * b));
            const int64_t p = (int64_t)(4 * i + b) - mis;
            if (p >= 0 && (uint64_t)p < len) gz_candidate(in, len, (uint64_t)p, count, out, cap);
        }
    }
}

}  // namespace zb

using namespace zb;

static uint32_t host_crc32(uint32_t crc, const uint8_t* p, size_t n)
{
    const unsigned long* t = host_crc_table();
    crc = ~crc;
    for (size_t i = 0; i < n; i++) crc = (uint32_t)t[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
    return ~crc;
}

namespace {

// Device scratch that keeps its contents when it grows (the walk's output).
struct Arena {
    DevBuf buf;
    uint64_t used = 0;
    int reserve(uint64_t more, cudaStream_t s)
    {
        if (used + more <= buf.cap) return 0;
        DevBuf nb;
        int rc = nb.ensure(std::max<uint64_t>(used + more, 2 * (uint64_t)buf.cap));
        if (rc) return rc;
        if (used && cudaMemcpyAsync(nb.p, buf.p, used, cudaMemcpyDeviceToDevice, s) != cudaSuccess) { nb.release(); return ZB_STREAM_ERROR; }
        if (cudaStreamSynchronize(s) != cudaSuccess) { nb.release(); return ZB_STREAM_ERROR; }
        buf.release();
        buf = nb;
        return 0;
    }
    ~Arena() { buf.release(); }
};

struct OutPiece { bool from_plan; uint64_t off, len; };      // a member's output: in the plan's buffer or in the walk's arena

// One member decoded where it stands (step 4): header on the host as Python's gzip reads it plus zlib's checks of the
// reserved flags and FHCRC, deflate data by the one-stream parallel decoder, else one warp, trailer against the output.
struct Walker {
    Ctx* c;
    cudaStream_t s;
    const uint8_t* d_in;
    uint64_t len;
    Arena arena;
    DevBuf tab;                                                 // one-member tables of the warp decoder, CRC result
    std::vector<uint8_t> hb;

    int fetch(uint64_t at, uint64_t n)                          // hb = d_in[at .. at + n)
    {
        hb.resize(n);
        if (n && cudaMemcpyAsync(hb.data(), d_in + at, n, cudaMemcpyDeviceToHost, s) != cudaSuccess) return ZB_STREAM_ERROR;
        return cudaStreamSynchronize(s) == cudaSuccess ? 0 : ZB_STREAM_ERROR;
    }
    // the first non-zero byte at or after p (len if none): zero padding after a member is skipped, as gzip.decompress does
    int skip_zeros(uint64_t* p)
    {
        uint64_t w = 4096;
        while (*p < len) {
            const uint64_t n = std::min<uint64_t>(w, len - *p);
            if (fetch(*p, n)) return ZB_STREAM_ERROR;
            uint64_t k = 0;
            while (k < n && hb[k] == 0) k++;
            *p += k;
            if (k < n) return 0;
            w = std::min<uint64_t>(w * 2, 64u << 20);
        }
        return 0;
    }
    // header at p -> its length, or a reason it is not one
    int header(uint64_t p, uint64_t* hdr, const char** why)
    {
        uint64_t w = 4096;
        for (;;) {
            const uint64_t n = std::min<uint64_t>(w, len - p);
            if (fetch(p, n)) return ZB_STREAM_ERROR;
            *why = nullptr;
            if (n < 2 || hb[0] != 0x1f || hb[1] != 0x8b) { *why = n < 2 ? "truncated header" : "not a gzip member header"; return 0; }
            bool more = false;
            if (n < 10) more = true;
            else if (hb[2] != 8) { *why = "unknown compression method"; return 0; }
            else if (hb[3] & 0xe0) { *why = "unknown header flags set"; return 0; }
            else {
                const uint32_t flg = hb[3];
                uint64_t q = 10;
                if (flg & 4) q = q + 2 <= n ? q + 2 + (hb[q] | (hb[q + 1] << 8)) : n + 1;
                for (uint32_t f = 8; f <= 16 && q <= n; f <<= 1) {
                    if (!(flg & f)) continue;
                    while (q < n && hb[q] != 0) q++;
                    q++;
                }
                if ((flg & 2) && q <= n) q += 2;
                if (q > n) more = true;
                else {
                    if ((flg & 2) && (host_crc32(0, hb.data(), q - 2) & 0xffff) != (uint32_t)(hb[q - 2] | (hb[q - 1] << 8))) {
                        *why = "header crc mismatch";
                        return 0;
                    }
                    *hdr = q;
                    return 0;
                }
            }
            if (n == len - p) { *why = "truncated header"; return 0; }
            w *= 4;
        }
    }
    // decodes the member at p; *next = where the following data starts, *why = the reason it is damaged
    // The decoders are first given the data up to `bound` (the next candidate), so that a member followed by padding does
    // not make them search the rest of the file; if the member does not end before it (a candidate inside its data), the
    // whole rest of the file.  A decode that ends is final either way: the deflate data say where they stop.
    int member(uint64_t p, uint64_t bound, uint64_t guess, OutPiece* out, uint64_t* next, const char** why)
    {
        uint64_t hdr = 0;
        int rc = header(p, &hdr, why);
        if (rc || *why) return rc;
        const uint64_t beg = p + hdr;
        if (bound < beg + 10) bound = len;                      // no room for data and trailer in front of the candidate
        uint64_t cap = std::max<uint64_t>(std::max<uint64_t>(guess, 4 * (bound - beg)), 1u << 20);
        if ((rc = tab.ensure(16 * 8)) != 0) return rc;
        for (;;) {
            if ((rc = arena.reserve(cap + 16, s)) != 0) return rc;
            cap = arena.buf.cap - arena.used - 16;
            uint8_t* o = arena.buf.as<uint8_t>() + arena.used;
            uint64_t got = 0, used = 0, need = 0;
            int32_t st = ZB_OK;
            int pr = inflate_single_parallel(c, d_in + beg, bound - beg, o, cap, ZB200_WRAP_RAW, &got, &st, s, &used, nullptr, nullptr,
                                             nullptr, &need);
            // a long member the parallel decoder declined up to the candidate: once more with the rest of the file before
            // one warp takes it (short members never: their try costs a search over the rest of the file for little)
            if (pr == 1 && need == 0 && bound < len && bound - beg >= (64u << 10))
                pr = inflate_single_parallel(c, d_in + beg, len - beg, o, cap, ZB200_WRAP_RAW, &got, &st, s, &used, nullptr, nullptr,
                                             nullptr, &need);
            if (pr < 0) return pr;
            if (pr == 1 && need > cap) { cap = need; continue; }  // the parallel decoder counted the output: room for exactly that
            if (pr == 1) {                                      // one warp: [beg end dbeg dend len used | status id]
                uint64_t h[8] = {beg, bound, arena.used, arena.used + cap, 0, 0, 0, 0};
                uint64_t* d = tab.as<uint64_t>();
                if (cudaMemcpyAsync(d, h, sizeof(h), cudaMemcpyHostToDevice, s) != cudaSuccess) return ZB_STREAM_ERROR;
                if ((rc = inflate_members_launch(d_in, d, d + 1, arena.buf.as<uint8_t>(), d + 2, d + 3, (const uint32_t*)(d + 7), 1, d + 4,
                                                 (int32_t*)(d + 6), s, d + 5)) != 0) return rc;
                if (cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess)
                    return ZB_STREAM_ERROR;
                got = h[4]; used = h[5]; st = (int32_t)(uint32_t)h[6];
                if (st == ZB_BUF_ERROR) { cap *= 2; continue; }
                if (st != ZB_OK && bound < len) { bound = len; continue; }
                if (st != ZB_OK) { *why = "invalid compressed data"; return 0; }
            }
            const uint64_t t = beg + used;
            if (t + 8 > len) { *why = "truncated member"; return 0; }
            uint32_t* d_sum = tab.as<uint32_t>() + 16;
            if ((rc = checksum_launch(c, o, got, d_sum, s)) != 0) return rc;
            uint32_t crc = 0;
            if (cudaMemcpyAsync(&crc, d_sum, 4, cudaMemcpyDeviceToHost, s) != cudaSuccess) return ZB_STREAM_ERROR;
            if ((rc = fetch(t, 8)) != 0) return rc;
            const uint32_t want_crc = hb[0] | (hb[1] << 8) | (hb[2] << 16) | ((uint32_t)hb[3] << 24);
            const uint32_t want_len = hb[4] | (hb[5] << 8) | (hb[6] << 16) | ((uint32_t)hb[7] << 24);
            if (crc != want_crc) { *why = "incorrect data check"; return 0; }
            if ((uint32_t)got != want_len) { *why = "incorrect length check"; return 0; }
            *out = OutPiece{false, arena.used, got};
            arena.used += got;
            *next = t + 8;
            return 0;
        }
    }
};

}  // namespace

ZB_API int zb200_gunzip(const void* src, size_t src_len, void* dst, size_t* dst_len, size_t* members, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if ((src == nullptr && src_len) || dst_len == nullptr || members == nullptr || (dst == nullptr && *dst_len)) {
        set_error("zb200_gunzip: bad argument");
        return ZB_STREAM_ERROR;
    }
    const uint64_t cap = *dst_len, len = src_len;
    if (len == 0) { *dst_len = 0; *members = 0; return 0; }
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    Walker wk{c, s, nullptr, len};
    do {
        const uint8_t* d_in = to_device(c, src, len, s, &rc);
        if (rc) break;
        wk.d_in = d_in;
        // ---- 1. candidates ----
        // room for the candidates of a file of 1 KiB members; more: one more scan with room for all of them
        const uint32_t kMaxCand = 1u << 26;
        uint32_t ccap = (uint32_t)std::min<uint64_t>(len / 1024 + 4096, kMaxCand);
        if ((rc = c->small.ensure(256)) != 0) break;
        if ((rc = c->ws[11].ensure((size_t)ccap * sizeof(GzCand) + 64)) != 0) break;
        uint32_t* d_count = c->small.as<uint32_t>() + 32;
        GzCand* d_cand = c->ws[11].as<GzCand>();
        uint32_t ncand = 0;
        uint8_t last8[8] = {0};
        cudaError_t e = cudaMemsetAsync(d_count, 0, 4, s);
        if (e == cudaSuccess) ZB_LAUNCH(k_gz_scan, device_sms() * 8, 256, 0, s, d_in, len, d_count, d_cand, ccap);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&ncand, d_count, 4, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess && len >= 8) e = cudaMemcpyAsync(last8, d_in + len - 8, 8, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e == cudaSuccess && ncand > ccap && ncand <= kMaxCand) {
            ccap = ncand;
            if ((rc = c->ws[11].ensure((size_t)ccap * sizeof(GzCand) + 64)) != 0) break;
            d_cand = c->ws[11].as<GzCand>();
            ncand = 0;
            e = cudaMemsetAsync(d_count, 0, 4, s);
            if (e == cudaSuccess) ZB_LAUNCH(k_gz_scan, device_sms() * 8, 256, 0, s, d_in, len, d_count, d_cand, ccap);
            if (e == cudaSuccess) e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaMemcpyAsync(&ncand, d_count, 4, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        }
        std::vector<GzCand> cand;
        if (e == cudaSuccess && ncand <= ccap && ncand) {       // more than kMaxCand: no plan, the walk decodes the file from offset 0
            cand.resize(ncand);
            e = cudaMemcpyAsync(cand.data(), d_cand, (size_t)ncand * sizeof(GzCand), cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
            std::sort(cand.begin(), cand.end(), [](const GzCand& a, const GzCand& b) { return a.pos < b.pos; });
        }
        if (e != cudaSuccess) { set_error("zb200_gunzip: scan failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }

        // ---- 2. the plan ----
        std::vector<GzCand> kept;
        if (!cand.empty() && cand[0].pos == 0) {
            kept.push_back(cand[0]);
            for (size_t i = 1; i < cand.size(); i++) {
                const GzCand& prev = kept.back();
                const uint64_t from = prev.blen ? prev.pos + prev.blen : prev.pos + prev.hdr_len + 10;
                if (cand[i].pos >= from) kept.push_back(cand[i]);
            }
        }
        const size_t np = kept.size();
        std::vector<MemberSpan> ms(np);
        uint64_t planned = 0;
        for (size_t k = 0; k < np; k++) {
            const uint64_t beg = kept[k].pos + kept[k].hdr_len, stop = k + 1 < np ? kept[k + 1].pos : len;
            const uint32_t crc = k + 1 < np ? kept[k + 1].crc : (uint32_t)(last8[0] | last8[1] << 8 | last8[2] << 16 | (uint32_t)last8[3] << 24);
            const uint32_t isz = k + 1 < np ? kept[k + 1].isize : (uint32_t)(last8[4] | last8[5] << 8 | last8[6] << 16 | (uint32_t)last8[7] << 24);
            MemberSpan& m = ms[k];
            m = MemberSpan{beg, beg, planned, isz, crc, kMemberDeflated, ZB_OK, 1};
            // a span too short for a trailer, a length no deflate data of that size can produce (1032:1 at most) or a
            // wrong FHCRC: not decoded, the walk decides
            if (stop < beg + 8 + 2 || isz > (stop - 8 - beg) * 1032 || !kept[k].hcrc_ok) { m.route = kMemberSkip; m.status = ZB_DATA_ERROR; m.raw_len = 0; }
            else m.end = stop - 8;
            planned += m.raw_len;
        }
        // ---- 3. decode and verify every planned member: into the caller's device buffer when it has room, else scratch ----
        const bool dst_dev = dst != nullptr && classify(dst) == kDevice;
        uint8_t* d_plan = nullptr;
        std::vector<uint64_t> p_len(np);
        std::vector<int32_t> p_st(np, ZB_DATA_ERROR);
        if (np) {
            if (dst_dev && planned <= cap) d_plan = (uint8_t*)dst;
            else if (c->out.ensure(planned + 16) == 0) d_plan = c->out.as<uint8_t>();
            else cudaGetLastError();                            // a plan no allocation can hold (lengths of spurious candidates): walk it all
        }
        if (d_plan) {
            if ((rc = decode_members(c, d_in, len, d_plan, ms.data(), np, s)) != 0) break;
            if (cudaStreamSynchronize(s) != cudaSuccess) { set_error("zb200_gunzip: decode failed: %s", cudaGetErrorString(cudaGetLastError())); rc = ZB_STREAM_ERROR; break; }
            memcpy(p_len.data(), c->pinned, np * 8);
            memcpy(p_st.data(), (uint8_t*)c->pinned + np * 8, np * 4);
        }
        // ---- 4. the walk: verified members as planned, everything else one member at a time ----
        std::vector<OutPiece> pieces;
        bool all_planned = true;
        uint64_t p = 0, total = 0;
        size_t k = 0, count = 0;
        const char* why = nullptr;
        while (p < len) {
            while (k < np && kept[k].pos < p) k++;
            if (k < np && kept[k].pos == p && p_st[k] == ZB_OK) {
                pieces.push_back(OutPiece{true, ms[k].dst, ms[k].raw_len});
                p = ms[k].end + 8;
                k++;
            } else {
                all_planned = false;
                // room for the output: what the plan says up to the next verified member, grown as the decoders ask
                uint64_t run_out = 0;
                for (size_t j = k; j < np && !(kept[j].pos > p && p_st[j] == ZB_OK); j++) run_out += ms[j].raw_len;
                size_t nx = k;
                while (nx < np && kept[nx].pos <= p) nx++;
                OutPiece op{};
                uint64_t next = 0;
                if ((rc = wk.member(p, nx < np ? kept[nx].pos : len, run_out, &op, &next, &why)) != 0) break;
                if (why) break;
                pieces.push_back(op);
                p = next;
            }
            total += pieces.back().len;
            count++;
            while (k < np && kept[k].pos < p) k++;
            if (k < np && kept[k].pos == p) continue;           // a candidate starts with 1f: no padding to look for
            if ((rc = wk.skip_zeros(&p)) != 0) break;
        }
        if (rc) break;
        if (why) {
            set_error("zb200_gunzip: member %zu at byte %llu: %s", count, (unsigned long long)p, why);
            *members = count;
            rc = ZB_DATA_ERROR;
            break;
        }
        *members = count;
        if (total > cap) { *dst_len = (size_t)total; set_error("zb200_gunzip: %llu bytes of output, room for %llu", (unsigned long long)total, (unsigned long long)cap); rc = ZB_BUF_ERROR; break; }
        // ---- delivery ----
        const uint8_t* d_walk = wk.arena.buf.as<uint8_t>();
        if (all_planned && d_plan == (uint8_t*)dst) {           // decoded in place
        } else if (dst_dev) {
            // the plan's output may sit in the caller's buffer: take it to scratch first, then gather every piece to its place
            const uint8_t* from = d_plan;
            if (d_plan == (uint8_t*)dst && planned) {
                if ((rc = c->out.ensure(planned + 16)) != 0) break;
                e = cudaMemcpyAsync(c->out.p, d_plan, planned, cudaMemcpyDeviceToDevice, s);
                if (e != cudaSuccess) { set_error("zb200_gunzip: copy failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
                from = c->out.as<uint8_t>();
            }
            std::vector<Piece> gp;
            uint64_t o = 0;
            for (const OutPiece& q : pieces) {
                const uint8_t* b = q.from_plan ? from + q.off : d_walk + q.off;
                for (uint64_t x = 0; x < q.len; x += kPieceBytes)
                    gp.push_back(Piece{b + x, (uint8_t*)dst + o + x, std::min<uint64_t>(kPieceBytes, q.len - x)});
                o += q.len;
            }
            if (!gp.empty()) {
                if ((rc = c->ws[10].ensure(gp.size() * sizeof(Piece))) != 0) break;
                if ((rc = c->ensure_pinned(gp.size() * sizeof(Piece))) != 0) break;
                memcpy(c->pinned, gp.data(), gp.size() * sizeof(Piece));
                e = cudaMemcpyAsync(c->ws[10].p, c->pinned, gp.size() * sizeof(Piece), cudaMemcpyHostToDevice, s);
                if (e != cudaSuccess) { set_error("zb200_gunzip: upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
                if ((rc = gather_launch(c->ws[10].as<const Piece>(), gp.size(), s)) != 0) break;
            }
        } else if (total) {                                     // host memory: one D2H copy per run of consecutive plan output
            const bool drain_threads = total >= HostStager::kMinBytes && classify(dst) == kHostPageable;
            HostDrainer drainer;
            uint64_t o = 0;
            for (size_t i = 0; i < pieces.size() && !rc;) {
                const OutPiece q0 = pieces[i];
                uint64_t n = q0.len;
                size_t j = i + 1;
                while (j < pieces.size() && pieces[j].from_plan == q0.from_plan && pieces[j].off == q0.off + n) n += pieces[j++].len;
                const uint8_t* b = q0.from_plan ? d_plan + q0.off : d_walk + q0.off;
                if (n && drain_threads) { if (cudaStreamSynchronize(s) != cudaSuccess || drainer.drain((uint8_t*)dst + o, b, n) != 0) rc = ZB_STREAM_ERROR; }
                else if (n && cudaMemcpyAsync((uint8_t*)dst + o, b, n, cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = ZB_STREAM_ERROR;
                o += n;
                i = j;
            }
            if (rc) { set_error("zb200_gunzip: D2H copy failed: %s", cudaGetErrorString(cudaGetLastError())); break; }
        }
        if (cudaStreamSynchronize(s) != cudaSuccess) { set_error("zb200_gunzip: failed: %s", cudaGetErrorString(cudaGetLastError())); rc = ZB_STREAM_ERROR; break; }
        *dst_len = (size_t)total;
    } while (0);
    cudaStreamSynchronize(s);
    wk.tab.release();
    ctx_release(c, s);
    return rc;
}

ZB_API size_t zb200_bgzf_bound(size_t src_len)
{
    return (size_t)((src_len + kBgzfBlock - 1) / kBgzfBlock * kBgzfMaxMember + sizeof(kBgzfEof));
}

ZB_API int zb200_bgzf_compress(const void* src, size_t src_len, void* dst, size_t* dst_len, int level, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if ((src == nullptr && src_len) || dst == nullptr || dst_len == nullptr || level < -1 || level > 9) {
        set_error("zb200_bgzf_compress: bad argument");
        return ZB_STREAM_ERROR;
    }
    const size_t nb = (size_t)((src_len + kBgzfBlock - 1) / kBgzfBlock);
    std::vector<uint64_t> src_off(nb + 1), slot(nb + 1), clen(nb);
    std::vector<int32_t> status(nb);
    for (size_t i = 0; i <= nb; i++) { src_off[i] = std::min<uint64_t>(i * kBgzfBlock, src_len); slot[i] = i * kBgzfSlot; }
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    do {
        if ((rc = c->out.ensure(slot[nb] + 64)) != 0) break;
        uint8_t* d_arena = c->out.as<uint8_t>();
        if (nb && (rc = deflate_batch(src, src_off.data(), nb, d_arena, slot.data(), clen.data(), nullptr, nullptr, status.data(), level,
                                      kWrapBgzf, stream)) != 0) break;
        uint64_t total = sizeof(kBgzfEof);
        for (size_t i = 0; i < nb && !rc; i++) {
            // the engine emits at most three stored blocks for 65280 bytes (65280 + 15 + 26 with framing): anything longer
            // would not fit BSIZE and is a defect, never written out
            if (status[i] != ZB_OK || clen[i] > kBgzfMaxMember) {
                set_error("zb200_bgzf_compress: block %zu came out at %llu bytes (status %d)", i, (unsigned long long)clen[i], status[i]);
                rc = ZB_STREAM_ERROR;
            }
            total += clen[i];
        }
        if (rc) break;
        if (total > *dst_len) { *dst_len = (size_t)total; set_error("zb200_bgzf_compress: output buffer too small"); rc = ZB_BUF_ERROR; break; }
        const bool dst_on_host = classify(dst) != kDevice;
        uint8_t* d_out = (uint8_t*)dst;
        if (dst_on_host) {
            if ((rc = c->in.ensure(total + 64)) != 0) break;
            d_out = c->in.as<uint8_t>();
        }
        // pieces: every block to its place, then the EOF block from the upload
        const size_t tab_at = 64, up_bytes = tab_at + (nb + 1) * sizeof(Piece);
        if ((rc = c->ensure_pinned(up_bytes)) != 0) break;
        if ((rc = c->ws[0].ensure(up_bytes + 64)) != 0) break;
        uint8_t* h_up = (uint8_t*)c->pinned;
        uint8_t* d_up = c->ws[0].as<uint8_t>();
        memcpy(h_up, kBgzfEof, sizeof(kBgzfEof));
        Piece* pc = reinterpret_cast<Piece*>(h_up + tab_at);
        uint64_t pos = 0;
        for (size_t i = 0; i < nb; i++) { pc[i] = Piece{d_arena + slot[i], d_out + pos, clen[i]}; pos += clen[i]; }
        pc[nb] = Piece{d_up, d_out + pos, sizeof(kBgzfEof)};
        cudaError_t e = cudaMemcpyAsync(d_up, h_up, up_bytes, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) { set_error("zb200_bgzf_compress: upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        if ((rc = gather_launch(reinterpret_cast<const Piece*>(d_up + tab_at), nb + 1, s)) != 0) break;
        const bool drain_threads = dst_on_host && total >= HostStager::kMinBytes && classify(dst) == kHostPageable;
        if (dst_on_host && !drain_threads) e = cudaMemcpyAsync(dst, d_out, total, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { set_error("zb200_bgzf_compress: failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        if (drain_threads) {
            HostDrainer drainer;
            if ((rc = drainer.drain(dst, d_out, total)) != 0) break;
        }
        *dst_len = (size_t)total;
    } while (0);
    if (rc) cudaStreamSynchronize(s);
    ctx_release(c, s);
    return rc;
}
