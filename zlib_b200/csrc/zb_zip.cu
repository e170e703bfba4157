// zb_zip.cu -- a ZIP32 archive from n files compressed in one GPU batch, assembled on the device.
//
// The reference writes archives member by member through zip.c: local header, deflate() in 16 KiB steps, sizes and
// CRC patched in afterwards, central directory at close (qcsrc/zip.c:902-1128, h/zip.h:157-224).  Here all members
// are compressed by one zb200_deflate_batch() call (raw deflate, windowBits = -15 like zip.c:1005, with the CRC-32 of
// each member from the same pass) into device slots; once every size is known the records are laid out by prefix sum
// and one copy kernel moves headers and member data to their final places, so the archive leaves the GPU as ONE
// contiguous D2H copy.  The records are the ones zip.c emits: local file header (30 bytes + name), central directory
// header (46 bytes + name), end of central directory (22 bytes); the reference's unzip.c checks that local and
// central headers agree (unzlocal_CheckCurrentFileCoherencyHeader, unzip.c:963-1047), which they do by construction.
//
// A *segment* is the run of [local header | name | data] records of some members; segments built on different GPUs
// concatenate (BASELINE config 5: files are dealt to the ranks, the root appends the central directory).
// ZIP32 only: at most 65535 members and 4 GiB - 1 for every size and offset; larger inputs are refused.
//
// Reading (zb200_zip_list / zb200_zip_extract) is the reverse: the central directory is parsed on the host (unzOpen,
// unzip.c), then every member is decoded in one pass over the archive on the device instead of unzOpenCurrentFile /
// unzReadCurrentFile member by member.  k_zip_locate checks every local header against the directory at once; stored
// members are copied by k_zip_gather, short deflated members share one k_inflate_batch launch (a warp each), and the long
// ones -- which a warp would decode at ~15 MB/s -- are cut at their sync markers into 128 KiB segments planned from the
// lengths the directory states and decoded all together by the segment kernels of zb_inflate.cu.  CRC-32 and length of
// every member are checked on the device.
#include "zb_common.cuh"
#include "zb_deflate.cuh"
#include "zb_inflate.cuh"
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <vector>

namespace zb {

constexpr int kGatherThreads = 256;

// One CTA per piece: dst-aligned 4-byte stores fed by two aligned loads and a funnel shift (source and destination
// are misaligned against each other in general), four words per thread in flight; ragged ends byte by byte.
__global__ void __launch_bounds__(kGatherThreads) k_zip_gather(const Piece* __restrict__ pieces)
{
    const Piece pc = pieces[blockIdx.x];
    const uint8_t* s = pc.src;
    uint8_t* d = pc.dst;
    uint64_t n = pc.len;
    const uint32_t head = (uint32_t)min((uint64_t)((4 - ((uintptr_t)d & 3)) & 3), n);
    if (threadIdx.x < head) d[threadIdx.x] = s[threadIdx.x];
    s += head; d += head; n -= head;
    const uint64_t nw = n >> 2;
    const uint32_t sh = (uint32_t)((uintptr_t)s & 3) * 8;
    const uint32_t* sw = reinterpret_cast<const uint32_t*>((uintptr_t)s & ~(uintptr_t)3);
    uint32_t* dw = reinterpret_cast<uint32_t*>(d);
    uint64_t i = threadIdx.x;
    for (; i + 3 * kGatherThreads < nw; i += 4 * kGatherThreads) {
        uint32_t a[4], b[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { a[k] = sw[i + k * kGatherThreads]; b[k] = sh ? sw[i + k * kGatherThreads + 1] : 0u; }
#pragma unroll
        for (int k = 0; k < 4; k++) dw[i + k * kGatherThreads] = __funnelshift_r(a[k], b[k], sh);
    }
    for (; i < nw; i += kGatherThreads) dw[i] = __funnelshift_r(sw[i], sh ? sw[i + 1] : 0u, sh);
    const uint32_t tail = (uint32_t)(n & 3);
    if (threadIdx.x < tail) d[nw * 4 + threadIdx.x] = s[nw * 4 + threadIdx.x];
}

static void put16(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
static void put32(uint8_t* p, uint64_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }
__host__ __device__ static inline uint32_t get16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__host__ __device__ static inline uint32_t get32(const uint8_t* p) { return get16(p) | (get16(p + 2) << 16); }

int gather_launch(const Piece* d_pieces, size_t n, cudaStream_t s)
{
    if (n == 0) return 0;
    ZB_LAUNCH(k_zip_gather, (unsigned)n, kGatherThreads, 0, s, d_pieces);
    ZB_CHECK_LAUNCH();
    return 0;
}

// ---- reading ----
struct ZipLoc { uint64_t data_off; int32_t route, status; };    // 16 bytes per member, read back once

// One thread per member: the local header, byte by byte (headers sit at any alignment), against the directory the way
// unzlocal_CheckCurrentFileCoherencyHeader does it (unzip.c:963-1047): signature, method, name length, and CRC-32 and
// sizes unless the local header's bit 3 says they follow the data.  The data start from the LOCAL name and extra lengths.
__global__ void k_zip_locate(const uint8_t* __restrict__ arc, uint64_t arc_len, const zb200_zip_entry* __restrict__ ent,
                             const uint64_t* __restrict__ dst_off, uint32_t n, ZipLoc* __restrict__ loc)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const zb200_zip_entry e = ent[i];
    ZipLoc r{0, kMemberSkip, ZB_OK};
    const uint64_t lo = e.local_off;
    if (lo > arc_len || arc_len - lo < 30) r.status = ZB200_UNZ_BADZIPFILE;
    else {
        const uint8_t* h = arc + lo;
        const uint32_t lflags = get16(h + 6);
        if (get32(h) != 0x04034b50u || get16(h + 8) != e.method || get16(h + 26) != e.name_len) r.status = ZB200_UNZ_BADZIPFILE;
        else if (e.method != 0 && e.method != 8) r.status = ZB200_UNZ_BADZIPFILE;
        else if (!(lflags & 8) && (get32(h + 14) != e.crc32 || get32(h + 18) != e.comp_len || get32(h + 22) != e.raw_len))
            r.status = ZB200_UNZ_BADZIPFILE;
        else {
            r.data_off = lo + 30 + get16(h + 26) + get16(h + 28);
            if (e.flags & 1) r.status = ZB_STREAM_ERROR;                              // encrypted
            else if (e.method == 0 && e.comp_len != e.raw_len) r.status = ZB200_UNZ_BADZIPFILE;
            else if (r.data_off > arc_len || arc_len - r.data_off < e.comp_len) r.status = ZB200_UNZ_BADZIPFILE;
            else if (dst_off[i + 1] - dst_off[i] < e.raw_len) r.status = ZB_BUF_ERROR;
            else r.route = e.method == 0 ? kMemberStored : kMemberDeflated;
        }
    }
    loc[i] = r;
}

// The last word on every member that reached a decoder: any decoder failure is invalid data, then where the data ended
// (members that must end exactly at their span's end), then the length, then the CRC-32 (crc[slot[i]], computed from the
// output) against what the container states.
__global__ void k_zip_verdict(const MemberSpan* __restrict__ m, const uint32_t* __restrict__ crc, const uint32_t* __restrict__ slot,
                              const uint64_t* __restrict__ len, const uint64_t* __restrict__ used, int32_t* __restrict__ status, uint32_t n)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || m[i].route == kMemberSkip) return;
    int32_t st = status[i];
    if (st != ZB_OK) st = ZB_DATA_ERROR;                        // (the batch's Z_BUF_ERROR: more output than raw_len)
    else if (m[i].exact_end && used[i] != m[i].end - m[i].beg) st = ZB_DATA_ERROR;
    else if (len[i] != m[i].raw_len) st = ZB_DATA_ERROR;
    else if (crc[slot[i]] != m[i].crc32) st = ZB200_UNZ_CRCERROR;
    status[i] = st;
}

// ---- the members' routes (shared by zb200_zip_extract and zb200_gunzip) ----
constexpr uint64_t kShortMember = ZB200_CHUNK;                  // members with at most one chunk of output: a warp each in the batch

int decode_members(Ctx* c, const uint8_t* d_arc, uint64_t arc_len, uint8_t* d_dst, const MemberSpan* m, size_t n, cudaStream_t s)
{
    int rc = 0;
    const uint32_t nn = (uint32_t)n;
    // per-member tables, uploaded in one piece: [spans] [len][status, 8 bytes each][used][beg][end][dst beg][dst end]
    // [crc off][crc len] [slot][ids] | written on the device: [crc][adler]
    const size_t per = sizeof(MemberSpan) + 9 * 8 + 2 * 4;
    if ((rc = c->ws[7].ensure(n * (per + 8) + 64)) != 0) return rc;
    uint8_t* up = c->ws[7].as<uint8_t>();
    MemberSpan* d_m = (MemberSpan*)up;
    uint64_t* d_len = (uint64_t*)(d_m + n);
    int32_t* d_st = (int32_t*)(d_len + n);                      // right behind the lengths: the results come back in one copy
    uint64_t* d_used = d_len + 2 * n;
    uint64_t* d_beg = d_used + n;
    uint64_t* d_end = d_beg + n;
    uint64_t* d_dbeg = d_end + n;
    uint64_t* d_dend = d_dbeg + n;
    uint64_t* d_coff = d_dend + n;
    uint64_t* d_clen = d_coff + n;
    uint32_t* d_slot = (uint32_t*)(d_clen + n);
    uint32_t* d_ids = d_slot + n;
    uint32_t* d_crc = d_ids + n;
    uint32_t* d_adl = d_crc + n;
    const size_t up_bytes = (size_t)((uint8_t*)d_crc - up);

    std::vector<uint8_t> hup(up_bytes, 0);
    memcpy(hup.data(), m, n * sizeof(MemberSpan));
    uint64_t* h_len = (uint64_t*)(hup.data() + n * sizeof(MemberSpan));
    int32_t* h_st = (int32_t*)(h_len + n);
    uint64_t* h_used = h_len + 2 * n;
    uint64_t* h_beg = h_used + n;
    uint64_t* h_end = h_beg + n;
    uint64_t* h_dbeg = h_end + n;
    uint64_t* h_dend = h_dbeg + n;
    uint64_t* h_coff = h_dend + n;
    uint64_t* h_clen = h_coff + n;
    uint32_t* h_slot = (uint32_t*)(h_clen + n);
    uint32_t* h_ids = h_slot + n;
    std::vector<Piece> pieces;
    std::vector<uint32_t> large, batch, one_crc, chunk_crc;  // members by route; CRC by one CTA / by chunks
    for (uint32_t i = 0; i < nn; i++) {
        h_st[i] = m[i].status;
        h_beg[i] = m[i].beg; h_end[i] = m[i].end;
        h_dbeg[i] = m[i].dst; h_dend[i] = m[i].dst + m[i].raw_len;
        if (m[i].route == kMemberStored) {
            for (uint64_t o = 0; o < m[i].raw_len; o += kPieceBytes)
                pieces.push_back(Piece{d_arc + m[i].beg + o, d_dst + m[i].dst + o, std::min<uint64_t>(kPieceBytes, m[i].raw_len - o)});
            h_len[i] = m[i].raw_len;
            h_used[i] = m[i].end - m[i].beg;
            one_crc.push_back(i);
        } else if (m[i].route == kMemberDeflated) {
            if (m[i].raw_len > kShortMember) large.push_back(i); else batch.push_back(i);
        }
    }
    cudaError_t e = cudaSuccess;
    // ---- long members: markers in their data, then the planned segment decode of all that fit the plan ----
    std::vector<uint32_t> fallback;
    if (!large.empty()) {
        std::sort(large.begin(), large.end(), [&](uint32_t a, uint32_t b) { return m[a].beg < m[b].beg; });
        uint64_t lo = ~0ull, hi = 0;
        for (uint32_t i : large) { lo = std::min(lo, h_beg[i]); hi = std::max(hi, h_end[i]); }
        const uint32_t cap = (uint32_t)std::min<uint64_t>((hi - lo) / 32 + 4096, 1u << 26);
        if ((rc = c->small.ensure(256)) != 0) return rc;
        if ((rc = c->ws[9].ensure((size_t)cap * 8 + 64)) != 0) return rc;
        uint32_t* d_count = c->small.as<uint32_t>() + 24;
        uint32_t nmark = 0;
        std::vector<uint64_t> mk;
        e = cudaMemsetAsync(d_count, 0, 4, s);
        if (e == cudaSuccess && (rc = find_markers_launch(d_arc, lo, hi, d_count, c->ws[9].as<uint64_t>(), cap, s)) != 0) return rc;
        if (e == cudaSuccess) e = cudaMemcpyAsync(&nmark, d_count, 4, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e == cudaSuccess && nmark <= cap && nmark) {
            mk.resize(nmark);
            e = cudaMemcpyAsync(mk.data(), c->ws[9].p, (size_t)nmark * 8, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
            std::sort(mk.begin(), mk.end());
        }
        if (e != cudaSuccess) { set_error("member decode: marker search failed: %s", cudaGetErrorString(e)); return ZB_STREAM_ERROR; }
        std::vector<PlannedStream> plan;
        std::vector<uint64_t> marks;
        std::vector<uint32_t> planned;
        bool exact = false;
        for (uint32_t i : large) {
            // a marker ends a chunk and the next one starts behind it: strictly inside the member's data
            const auto a = std::upper_bound(mk.begin(), mk.end(), h_beg[i]), b = std::lower_bound(mk.begin(), mk.end(), h_end[i]);
            const uint64_t have = (uint64_t)(b - a), want = (m[i].raw_len + ZB200_CHUNK - 1) / ZB200_CHUNK - 1;
            if (nmark > cap || have != want) { fallback.push_back(i); continue; }
            plan.push_back(PlannedStream{h_beg[i], h_end[i], m[i].dst, m[i].raw_len, (uint32_t)marks.size(), (uint32_t)have});
            marks.insert(marks.end(), a, b);
            planned.push_back(i);
            exact = exact || m[i].exact_end;                    // one container per call: every member or none
        }
        std::vector<uint8_t> ok(plan.size(), 0);
        if (!plan.empty() && (rc = inflate_planned(c, d_arc, arc_len, d_dst, plan.data(), plan.size(), marks.data(), ok.data(), s, exact)) != 0)
            return rc;
        for (size_t k = 0; k < planned.size(); k++) {
            if (ok[k]) { h_len[planned[k]] = m[planned[k]].raw_len; h_used[planned[k]] = h_end[planned[k]] - h_beg[planned[k]]; chunk_crc.push_back(planned[k]); }
            else fallback.push_back(planned[k]);
        }
        // ---- what does not fit the plan: the one-stream decoder (counting pass, block finder), else the batch ----
        for (uint32_t i : fallback) {
            uint64_t got = 0, used = 0;
            int32_t st = ZB_OK;
            const int pr = inflate_single_parallel(c, d_arc + h_beg[i], h_end[i] - h_beg[i], d_dst + m[i].dst, m[i].raw_len,
                                                   ZB200_WRAP_RAW, &got, &st, s, &used);
            if (pr < 0) return pr;
            if (pr == 0) { h_len[i] = got; h_st[i] = st; h_used[i] = used; chunk_crc.push_back(i); }
            else batch.push_back(i);
        }
    }
    // ---- short members (and declined long ones): one batch launch; stored members: one gather launch ----
    for (size_t k = 0; k < batch.size(); k++) { h_ids[k] = batch[k]; one_crc.push_back(batch[k]); }
    for (size_t k = 0; k < one_crc.size(); k++) { h_slot[one_crc[k]] = (uint32_t)k; h_coff[k] = m[one_crc[k]].dst; h_clen[k] = m[one_crc[k]].raw_len; }
    // long members by output position (ChunkDesc positions are 32-bit: one checksum launch per window below 4 GiB)
    std::sort(chunk_crc.begin(), chunk_crc.end(), [&](uint32_t a, uint32_t b) { return m[a].dst < m[b].dst; });
    for (size_t k = 0; k < chunk_crc.size(); k++) h_slot[chunk_crc[k]] = (uint32_t)(one_crc.size() + k);
    e = cudaMemcpyAsync(up, hup.data(), up_bytes, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && !pieces.empty()) {
        if ((rc = c->ws[10].ensure(pieces.size() * sizeof(Piece))) != 0) return rc;
        e = cudaMemcpyAsync(c->ws[10].p, pieces.data(), pieces.size() * sizeof(Piece), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess && (rc = gather_launch(c->ws[10].as<const Piece>(), pieces.size(), s)) != 0) return rc;
    }
    if (e != cudaSuccess) { set_error("member decode: upload failed: %s", cudaGetErrorString(e)); return ZB_STREAM_ERROR; }
    if ((rc = inflate_members_launch(d_arc, d_beg, d_end, d_dst, d_dbeg, d_dend, d_ids, batch.size(), d_len, d_st, s, d_used)) != 0) return rc;
    // ---- CRC-32 of every decoded member: one CTA per short member, per 128 KiB chunk (joined) for long ones ----
    if ((rc = checksum_batch_launch(d_dst, d_coff, d_clen, one_crc.size(), d_crc, d_adl, nullptr, nullptr, s)) != 0) return rc;
    if (!chunk_crc.empty()) {
        std::vector<ChunkDesc> cd;
        std::vector<JobDesc> jobs;
        for (size_t k0 = 0; k0 < chunk_crc.size();) {
            const uint64_t base = m[chunk_crc[k0]].dst;
            size_t k1 = k0;
            cd.clear(); jobs.clear();
            // the first member always (its ChunkDesc positions must stay below 4 GiB), further ones while the window stays below 3 GiB
            while (k1 < chunk_crc.size() && (k1 == k0 || m[chunk_crc[k1]].dst + m[chunk_crc[k1]].raw_len - base < (3ull << 30))) {
                const uint32_t i = chunk_crc[k1];
                JobDesc jd{};
                jd.first_chunk = (uint32_t)cd.size();
                for (uint64_t o = 0; o < m[i].raw_len; o += ZB200_CHUNK) {
                    ChunkDesc d{};
                    d.beg = (uint32_t)(m[i].dst - base + o);
                    d.len = (uint32_t)std::min<uint64_t>(ZB200_CHUNK, m[i].raw_len - o);
                    cd.push_back(d);
                }
                jd.nchunks = (uint32_t)cd.size() - jd.first_chunk;
                jobs.push_back(jd);
                k1++;
            }
            const size_t cd_bytes = cd.size() * sizeof(ChunkDesc), jb_bytes = jobs.size() * sizeof(JobDesc);
            if ((rc = c->ws[8].ensure(cd_bytes + jb_bytes + jobs.size() * 4 + 64)) != 0) return rc;
            uint8_t* d8 = c->ws[8].as<uint8_t>();
            uint32_t* d_jadl = (uint32_t*)(d8 + cd_bytes + jb_bytes);
            e = cudaMemcpyAsync(d8, cd.data(), cd_bytes, cudaMemcpyHostToDevice, s);
            if (e == cudaSuccess) e = cudaMemcpyAsync(d8 + cd_bytes, jobs.data(), jb_bytes, cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) { set_error("member decode: upload failed: %s", cudaGetErrorString(e)); return ZB_STREAM_ERROR; }
            uint32_t* d_wcrc = d_crc + one_crc.size() + k0;         // this window's slots are consecutive
            if ((rc = checksum_jobs_launch(c, d_dst + base, (const ChunkDesc*)d8, (uint32_t)cd.size(), (const JobDesc*)(d8 + cd_bytes),
                                           (uint32_t)jobs.size(), d_wcrc, d_jadl, s)) != 0) return rc;
            k0 = k1;
        }
    }
    ZB_LAUNCH(k_zip_verdict, (nn + 255) / 256, 256, 0, s, d_m, d_crc, d_slot, d_len, d_used, d_st, nn);
    if ((rc = c->ensure_pinned(n * 12 + 16)) != 0) return rc;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->pinned, d_len, n * 12, cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) { set_error("member decode failed: %s", cudaGetErrorString(e)); return ZB_STREAM_ERROR; }
    return 0;
}

}  // namespace zb

using namespace zb;

extern "C" unsigned long compressBound(unsigned long sourceLen);   // zapi_oneshot.c

// Worst-case archive size for these members (every member at compressBound).
ZB_API size_t zb200_zip_bound(const char* const* names, const uint64_t* src_off, size_t n)
{
    size_t total = 22;
    if (names == nullptr || src_off == nullptr) return 0;
    for (size_t i = 0; i < n; i++) {
        const size_t nl = strlen(names[i]);
        total += 30 + nl + 46 + nl + (size_t)compressBound((unsigned long)(src_off[i + 1] - src_off[i])) + 16;
    }
    return total;
}

ZB_API int zb200_zip_segment(const char* const* names, const void* src, const uint64_t* src_off, size_t n, int level,
                             uint32_t dos_datetime, void* dst, size_t* dst_len, zb200_zip_member* members)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (names == nullptr || src_off == nullptr || dst == nullptr || dst_len == nullptr || members == nullptr || n > 65535u ||
        (level != -1 && (level < 0 || level > 9))) {
        set_error("zb200_zip_segment: bad argument");
        return ZB_STREAM_ERROR;
    }
    for (size_t i = 0; i < n; i++) {
        if (names[i] == nullptr || strlen(names[i]) > 65535u || src_off[i + 1] < src_off[i] || src_off[i + 1] - src_off[i] >= 0xffffffffull) {
            set_error("zb200_zip_segment: member %zu is outside ZIP32", i);
            return ZB_STREAM_ERROR;
        }
    }
    if (n == 0) { *dst_len = 0; return 0; }
    std::vector<uint64_t> slot(n + 1), clen(n);
    std::vector<uint32_t> crc(n);
    std::vector<int32_t> status(n);
    slot[0] = 0;
    for (size_t i = 0; i < n; i++) slot[i + 1] = slot[i] + compressBound((unsigned long)(src_off[i + 1] - src_off[i])) + 16;

    Ctx* c = ctx_acquire_own();
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = c->own_stream;
    do {
        if ((rc = c->out.ensure(slot[n] + 64)) != 0) break;
        uint8_t* d_arena = c->out.as<uint8_t>();
        cudaStreamSynchronize(s);                               // the arena may still be read by the context's previous borrower
        if ((rc = zb200_deflate_batch(src, src_off, n, d_arena, slot.data(), clen.data(), crc.data(), nullptr, status.data(), level,
                                      ZB200_WRAP_RAW, nullptr)) != 0) break;
        // ---- layout by prefix sum; local headers (zip.c:969-1032) into one blob ----
        uint64_t pos = 0, blob_len = 0;
        size_t npieces = 0;
        for (size_t i = 0; i < n; i++) {
            if (status[i] != 0) { rc = status[i]; set_error("zb200_zip_segment: member %zu failed (%d)", i, rc); break; }
            const size_t nl = strlen(names[i]);
            members[i].local_off = pos; members[i].comp_len = clen[i]; members[i].raw_len = src_off[i + 1] - src_off[i];
            members[i].crc32 = crc[i]; members[i].reserved = 0;
            pos += 30 + nl + clen[i];
            blob_len += 30 + nl;
            npieces += 1 + (size_t)((clen[i] + kPieceBytes - 1) / kPieceBytes);
        }
        if (rc) break;
        if (pos >= 0xffffffffull) { set_error("zb200_zip_segment: segment of %llu bytes is outside ZIP32", (unsigned long long)pos); rc = ZB_STREAM_ERROR; break; }
        if (pos > *dst_len) { *dst_len = (size_t)pos; set_error("zb200_zip_segment: output buffer too small"); rc = ZB_BUF_ERROR; break; }
        const bool dst_on_host = classify(dst) != kDevice;
        uint8_t* d_arc = (uint8_t*)dst;
        if (dst_on_host) {
            if ((rc = c->in.ensure(pos + 64)) != 0) break;
            d_arc = c->in.as<uint8_t>();
        }
        const size_t tab_at = (size_t)((blob_len + 15) & ~(uint64_t)15), up_bytes = tab_at + npieces * sizeof(Piece);
        if ((rc = c->ensure_pinned(up_bytes)) != 0) break;
        if ((rc = c->ws[0].ensure(up_bytes + 64)) != 0) break;
        uint8_t* h_up = (uint8_t*)c->pinned;
        uint8_t* d_up = c->ws[0].as<uint8_t>();
        Piece* pieces = reinterpret_cast<Piece*>(h_up + tab_at);
        uint64_t bpos = 0;
        size_t k = 0;
        for (size_t i = 0; i < n; i++) {
            const size_t nl = strlen(names[i]);
            uint8_t* lh = h_up + bpos;
            put32(lh, 0x04034b50ul); put16(lh + 4, 20); put16(lh + 6, 0); put16(lh + 8, 8 /* Z_DEFLATED */);
            put32(lh + 10, dos_datetime); put32(lh + 14, crc[i]); put32(lh + 18, clen[i]); put32(lh + 22, members[i].raw_len);
            put16(lh + 26, (uint32_t)nl); put16(lh + 28, 0);
            memcpy(lh + 30, names[i], nl);
            pieces[k++] = Piece{d_up + bpos, d_arc + members[i].local_off, 30 + nl};
            for (uint64_t o = 0; o < clen[i]; o += kPieceBytes)
                pieces[k++] = Piece{d_arena + slot[i] + o, d_arc + members[i].local_off + 30 + nl + o, std::min<uint64_t>(kPieceBytes, clen[i] - o)};
            bpos += 30 + nl;
        }
        cudaError_t e = cudaMemcpyAsync(d_up, h_up, up_bytes, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) { set_error("zip table upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        ZB_LAUNCH(k_zip_gather, (unsigned)k, kGatherThreads, 0, s, reinterpret_cast<const Piece*>(d_up + tab_at));
        e = cudaGetLastError();
        const bool drain_threads = dst_on_host && pos >= HostStager::kMinBytes && classify(dst) == kHostPageable;
        if (e == cudaSuccess && dst_on_host && !drain_threads) e = cudaMemcpyAsync(dst, d_arc, pos, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { set_error("zip assembly failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        if (drain_threads) {                                    // malloc'ed archive buffer: host threads pull it through pinned slots
            HostDrainer drainer;
            if ((rc = drainer.drain(dst, d_arc, pos)) != 0) break;
        }
        *dst_len = (size_t)pos;
    } while (0);
    ctx_release(c, s);
    return rc;
}

// Central directory (zip.c:940-967) and end record (zip.c:1203-1240) for members whose local headers sit at
// members[i].local_off of the finished archive; the directory itself starts at cd_offset.  Host memory, no GPU work.
ZB_API int zb200_zip_directory(const char* const* names, const zb200_zip_member* members, size_t n, uint32_t dos_datetime,
                               uint64_t cd_offset, void* dst, size_t* dst_len)
{
    if (names == nullptr || members == nullptr || dst == nullptr || dst_len == nullptr || n > 65535u) return ZB_STREAM_ERROR;
    uint64_t need = 22;
    for (size_t i = 0; i < n; i++) need += 46 + strlen(names[i]);
    if (cd_offset + need >= 0xffffffffull) { set_error("zb200_zip_directory: archive is outside ZIP32"); return ZB_STREAM_ERROR; }
    if (need > *dst_len) { *dst_len = (size_t)need; return ZB_BUF_ERROR; }
    uint8_t* ch = (uint8_t*)dst;
    for (size_t i = 0; i < n; i++) {
        const size_t nl = strlen(names[i]);
        put32(ch, 0x02014b50ul); put16(ch + 4, 0); put16(ch + 6, 20); put16(ch + 8, 0); put16(ch + 10, 8);
        put32(ch + 12, dos_datetime); put32(ch + 16, members[i].crc32); put32(ch + 20, members[i].comp_len); put32(ch + 24, members[i].raw_len);
        put16(ch + 28, (uint32_t)nl); put16(ch + 30, 0); put16(ch + 32, 0); put16(ch + 34, 0); put16(ch + 36, 0);
        put32(ch + 38, 0); put32(ch + 42, members[i].local_off);
        memcpy(ch + 46, names[i], nl);
        ch += 46 + nl;
    }
    const uint64_t cd_size = need - 22;
    put32(ch, 0x06054b50ul); put16(ch + 4, 0); put16(ch + 6, 0); put16(ch + 8, (uint32_t)n); put16(ch + 10, (uint32_t)n);
    put32(ch + 12, cd_size); put32(ch + 16, cd_offset); put16(ch + 20, 0);
    *dst_len = (size_t)need;
    return 0;
}

ZB_API int zb200_zip_build(const char* const* names, const void* src, const uint64_t* src_off, size_t n, int level,
                           uint32_t dos_datetime, void* dst, size_t* dst_len)
{
    if (dst == nullptr || dst_len == nullptr || n > 65535u) return ZB_STREAM_ERROR;
    std::vector<zb200_zip_member> members(n ? n : 1);
    size_t cd = 22;
    for (size_t i = 0; i < n; i++) cd += names && names[i] ? 46 + strlen(names[i]) : 0;
    if (*dst_len < cd) { *dst_len = cd; return ZB_BUF_ERROR; }
    size_t seg = *dst_len - cd;                                 // what is left for the members once the directory has its room
    int rc = zb200_zip_segment(names, src, src_off, n, level, dos_datetime, dst, &seg, members.data());
    if (rc == ZB_BUF_ERROR) *dst_len = seg + cd;
    if (rc) return rc;
    if (classify(dst) == kDevice) { set_error("zb200_zip_build: the archive buffer must be host memory"); return ZB_STREAM_ERROR; }
    size_t dl = cd;
    if ((rc = zb200_zip_directory(names, members.data(), n, dos_datetime, seg, (uint8_t*)dst + seg, &dl)) != 0) return rc;
    *dst_len = seg + dl;
    return 0;
}

// ---- reading: the central directory (unzOpen2, unzip.c:380-491) ----
// The end record is searched back from the end through at most 65535 bytes of comment; byte_before_the_zipfile (bytes in
// front of the archive: a self-extractor stub, concatenated data) is where the directory really starts minus where the
// end record says it starts, and is added to every offset.  ZIP64 and multi-disk archives are refused as the writer
// refuses them.  A device archive has its tail and then its directory copied to the host.
ZB_API int zb200_zip_list(const void* archive, size_t arc_len, zb200_zip_entry* entries, size_t* n)
{
    if (archive == nullptr || n == nullptr || (entries == nullptr && *n != 0)) return ZB_STREAM_ERROR;
    const bool on_dev = classify(archive) == kDevice;
    auto fetch = [&](std::vector<uint8_t>& v, uint64_t off, uint64_t len) -> int {
        v.resize(len);
        if (!on_dev) { memcpy(v.data(), (const uint8_t*)archive + off, len); return 0; }
        ZB_CUDA(cudaMemcpy(v.data(), (const uint8_t*)archive + off, len, cudaMemcpyDeviceToHost));
        return 0;
    };
    if (arc_len < 22) { set_error("zb200_zip_list: %zu bytes hold no end record", arc_len); return ZB_STREAM_ERROR; }
    const uint64_t tail_len = std::min<uint64_t>(arc_len, 22 + 0xffff + 20);
    const uint64_t tail_at = arc_len - tail_len;
    std::vector<uint8_t> tail, cd;
    int rc = fetch(tail, tail_at, tail_len);
    if (rc) return rc;
    int64_t e = -1;
    for (int64_t p = (int64_t)tail_len - 22; p >= 0 && e < 0; p--)
        if (get32(&tail[p]) == 0x06054b50u && (uint64_t)p + 22 + get16(&tail[p + 20]) <= tail_len) e = p;
    if (e < 0) { set_error("zb200_zip_list: no end of central directory record"); return ZB_STREAM_ERROR; }
    const uint8_t* er = &tail[e];
    const uint64_t end_pos = tail_at + (uint64_t)e;
    const uint32_t disk = get16(er + 4), cd_disk = get16(er + 6), n_here = get16(er + 8), n_all = get16(er + 10);
    const uint64_t cd_size = get32(er + 12), cd_off = get32(er + 16);
    if (e >= 20 && get32(er - 20) == 0x07064b50u) { set_error("zb200_zip_list: ZIP64 archive"); return ZB_STREAM_ERROR; }
    if (disk != 0 || cd_disk != 0 || n_here != n_all) { set_error("zb200_zip_list: multi-disk archive"); return ZB_STREAM_ERROR; }
    if (n_all == 0xffffu || cd_size == 0xffffffffull || cd_off == 0xffffffffull) { set_error("zb200_zip_list: ZIP64 archive"); return ZB_STREAM_ERROR; }
    if (end_pos < cd_off + cd_size) { set_error("zb200_zip_list: central directory outside the archive"); return ZB_STREAM_ERROR; }
    const uint64_t before = end_pos - (cd_off + cd_size);      // byte_before_the_zipfile
    if (n_all > *n) { *n = n_all; set_error("zb200_zip_list: %u members, room for fewer", n_all); return ZB_BUF_ERROR; }
    if ((rc = fetch(cd, before + cd_off, cd_size)) != 0) return rc;
    uint64_t p = 0;
    for (uint32_t i = 0; i < n_all; i++) {
        if (p + 46 > cd_size || get32(&cd[p]) != 0x02014b50u) { set_error("zb200_zip_list: directory record %u is damaged", i); return ZB_STREAM_ERROR; }
        const uint8_t* h = &cd[p];
        const uint32_t nl = get16(h + 28), xl = get16(h + 30), cl = get16(h + 32);
        if (p + 46 + nl + xl + cl > cd_size) { set_error("zb200_zip_list: directory record %u is truncated", i); return ZB_STREAM_ERROR; }
        zb200_zip_entry& z = entries[i];
        z.crc32 = get32(h + 16);
        z.comp_len = get32(h + 20); z.raw_len = get32(h + 24); z.local_off = get32(h + 42);
        if (z.comp_len == 0xffffffffull || z.raw_len == 0xffffffffull || z.local_off == 0xffffffffull || get16(h + 34) == 0xffffu) {
            set_error("zb200_zip_list: member %u needs ZIP64", i);
            return ZB_STREAM_ERROR;
        }
        z.local_off += before;
        z.name_off = before + cd_off + p + 46;
        z.method = (uint16_t)get16(h + 10); z.flags = (uint16_t)get16(h + 8);
        z.name_len = (uint16_t)nl; z.reserved16 = 0; z.reserved32 = 0;
        p += 46 + nl + xl + cl;
    }
    *n = n_all;
    return 0;
}

// ---- reading: the members ----
ZB_API int zb200_zip_extract(const void* archive, size_t arc_len, const zb200_zip_entry* entries, size_t n, void* dst,
                             const uint64_t* dst_off, uint64_t* dst_len, int32_t* status, void* stream)
{
    int rc = ensure_init();
    if (rc) return rc;
    if (n == 0) return 0;
    if (archive == nullptr || entries == nullptr || dst == nullptr || dst_off == nullptr || dst_len == nullptr || status == nullptr ||
        n > 0xffffffffu) {
        set_error("zb200_zip_extract: bad argument");
        return ZB_STREAM_ERROR;
    }
    for (size_t i = 0; i < n; i++)
        if (dst_off[i + 1] < dst_off[i]) { set_error("zb200_zip_extract: dst_off must not decrease"); return ZB_STREAM_ERROR; }
    const uint32_t nn = (uint32_t)n;
    const uint64_t dst_base = dst_off[0], dst_span = dst_off[n] - dst_off[0];   // the slots: nothing outside them is touched
    Ctx* c = ctx_acquire((cudaStream_t)stream);
    if (!c) return ZB_MEM_ERROR;
    cudaStream_t s = pick_stream(c, stream);
    do {
        const uint8_t* d_arc = to_device(c, archive, arc_len, s, &rc);
        if (rc) break;
        const bool dst_on_host = classify(dst) != kDevice;
        uint8_t* d_dst = (uint8_t*)dst;
        if (dst_on_host) {                                      // staged: only the span of the slots, d_dst[dst_off[0]] is its first byte
            if ((rc = c->out.ensure(dst_span + 16)) != 0) break;
            d_dst = c->out.as<uint8_t>() - dst_base;
        }
        // the directory's view of every member, for k_zip_locate (ws[0]: decode_members keeps its tables elsewhere)
        const size_t tab = n * sizeof(zb200_zip_entry) + (n + 1) * 8 + n * sizeof(ZipLoc);
        if ((rc = c->ws[0].ensure(tab + 64)) != 0) break;
        uint8_t* w = c->ws[0].as<uint8_t>();
        zb200_zip_entry* d_ent = (zb200_zip_entry*)w;
        uint64_t* d_doff = (uint64_t*)(w + n * sizeof(zb200_zip_entry));
        ZipLoc* d_loc = (ZipLoc*)(d_doff + n + 1);
        cudaError_t e = cudaMemcpyAsync(d_ent, entries, n * sizeof(zb200_zip_entry), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_doff, dst_off, (n + 1) * 8, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) { set_error("zb200_zip_extract: table upload failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        ZB_LAUNCH(k_zip_locate, (nn + 255) / 256, 256, 0, s, d_arc, (uint64_t)arc_len, d_ent, d_doff, nn, d_loc);
        std::vector<ZipLoc> loc(n);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(loc.data(), d_loc, n * sizeof(ZipLoc), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { set_error("zb200_zip_extract: locate failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        std::vector<MemberSpan> ms(n);
        for (size_t i = 0; i < n; i++)
            ms[i] = MemberSpan{loc[i].data_off, loc[i].data_off + entries[i].comp_len, dst_off[i], entries[i].raw_len, entries[i].crc32,
                               loc[i].route, loc[i].status, 0};
        if ((rc = decode_members(c, d_arc, arc_len, d_dst, ms.data(), n, s)) != 0) break;
        uint64_t* p_len = (uint64_t*)c->pinned;
        int32_t* p_st = (int32_t*)(p_len + n);
        uint8_t* h_span = (uint8_t*)dst + dst_base;
        const bool drain_threads = dst_on_host && dst_span >= HostStager::kMinBytes && classify(dst) == kHostPageable;
        if (e == cudaSuccess && dst_on_host && !drain_threads && dst_span)
            e = cudaMemcpyAsync(h_span, d_dst + dst_base, dst_span, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { set_error("zb200_zip_extract: failed: %s", cudaGetErrorString(e)); rc = ZB_STREAM_ERROR; break; }
        if (drain_threads) {
            HostDrainer drainer;
            if ((rc = drainer.drain(h_span, d_dst + dst_base, dst_span)) != 0) break;
        }
        for (size_t i = 0; i < n; i++) { dst_len[i] = p_len[i]; status[i] = p_st[i]; }
    } while (0);
    if (rc) cudaStreamSynchronize(s);
    ctx_release(c, s);
    return rc;
}
