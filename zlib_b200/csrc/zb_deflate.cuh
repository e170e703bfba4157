// zb_deflate.cuh -- data layout of the deflate pipeline in HBM (shared by its kernels).
#pragma once
#include "zb_common.cuh"

namespace zb {

constexpr uint32_t kChunk = ZB200_CHUNK;         // input bytes linked by one CTA / packed by one CTA; ends byte-aligned
constexpr uint32_t kBlockBytes = 32768;          // input bytes per DEFLATE block = per CTA of the walk kernel (the reference
constexpr uint32_t kBlocksPerChunk = kChunk / kBlockBytes;   // closes a block every 16 Ki symbols, 45-60 KiB of text, deflate.c:291)
constexpr uint32_t kWindow = 32768;              // DEFLATE history (h/zconf.h MAX_WBITS = 15)
constexpr uint32_t kMinMatch = 3, kMaxMatch = 258;
constexpr uint32_t kHistSize = 320;              // 0..287 literal/length, 288..319 distance
constexpr uint32_t kHdrWords = 144;              // dynamic-block header, <= 4495 bits
constexpr uint32_t kTooFar = 4096;               // deflate.c:108-110
constexpr uint32_t kSlabChunks = 888;            // chunks per pipeline slab (2 waves of 3 link CTAs on 148 SMs)

// Job-mode framing beyond the public ZB200_WRAP_* values: a BGZF block (SAM/BAM specification 4.1), a gzip member whose
// 18-byte header carries the 'BC' extra subfield with BSIZE = member length - 1.  Only zb200_bgzf_compress asks for it.
constexpr int kWrapBgzf = 4;
constexpr uint32_t kBgzfHeader = 18;

// zb200_deflate_batch with any job-mode framing, kWrapBgzf included (zb200_deflate_batch itself takes the public ones).
int deflate_batch(const void* src, const uint64_t* src_off, size_t n, void* dst, const uint64_t* dst_off, uint64_t* dst_len,
                  uint32_t* crc, uint32_t* adler, int32_t* status, int level, int wrap, void* stream);

// configuration_table of the reference (deflate.c:137-149); kind 0 stored, 1 greedy, 2 lazy
struct LevelCfg { uint16_t good, lazy, nice, chain; int kind; };

// One DEFLATE block = kBlockUnits consecutive units; filled in by the code-construction kernel.
struct BlockMeta {
    uint32_t in_len;                             // input bytes the block covers
    uint32_t type;                               // 0 stored, 1 fixed, 2 dynamic
    uint32_t body_bits;                          // bits after the 3 header bits (types 1, 2)
    uint32_t hdr_bits;                           // dynamic header length in bits (type 2)
};

struct ChunkMeta {
    uint32_t nblocks;
    uint32_t stored;                             // 1 = whole chunk emitted as stored blocks
    uint64_t bytes;                              // compressed size of the chunk
    uint64_t offset;                             // byte offset in the output stream
};

// Job mode (zb200_deflate_batch): many independent inputs share one slab.  Chunks never cross a job boundary and the
// kernels take a chunk's position, its job's span (history and hashing stay inside it) and its role from this table
// instead of computing them from the chunk index.  Positions are relative to the slab buffer.
struct ChunkDesc {
    uint32_t beg, len;                           // first byte and length (1..kChunk) of the chunk
    uint32_t job_beg, job_end;                   // span of the job the chunk belongs to
    uint32_t job, first;                         // job index within the slab; index of the job's first chunk
    uint32_t last, pad;                          // 1 = last chunk of its job
};
struct JobDesc {
    uint64_t dst_off, dst_cap;                   // the job's output slot in the destination arena
    uint32_t first_chunk, nchunks;               // its chunks within the slab (nchunks == 0: empty input)
    uint32_t src_beg, src_len;
};
struct JobResult {                               // 32 bytes per job, copied to the host as they are
    uint64_t total;                              // length of the finished stream (header + blocks + trailer)
    uint32_t crc, adler;                         // checksums of the job's input
    uint32_t err, pad[3];                        // chunks packed to a size other than planned (must stay 0)
};

// Token: literal = byte value; match = (distance << 16) | (length - 3).
__device__ __forceinline__ uint32_t len_code(uint32_t l)       // l = length - 3; trees.c _length_code
{
    if (l < 8) return l;
    if (l == 255) return 28;
    const uint32_t e = 29 - __clz(l);                           // extra bits = msb - 2
    return 4 * e + 4 + ((l >> e) & 3);
}
__device__ __forceinline__ uint32_t len_extra_bits(uint32_t code) { return (code < 8 || code == 28) ? 0 : (code >> 2) - 1; }
__device__ __forceinline__ uint32_t dist_code(uint32_t d)      // d = distance - 1; trees.c d_code
{
    if (d < 4) return d;
    const uint32_t msb = 31 - __clz(d);
    return 2 * msb + ((d >> (msb - 1)) & 1);
}
__device__ __forceinline__ uint32_t dist_extra_bits(uint32_t code) { return code < 4 ? 0 : (code >> 1) - 1; }

}  // namespace zb
