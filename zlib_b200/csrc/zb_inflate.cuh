// zb_inflate.cuh -- state shared between the inflate kernels and the host shim.
#pragma once
#include "zb_common.cuh"

namespace zb {

// Where a stream stands (the reference's inflate_mode, h/inflate.h:20-51, collapsed to the
// points at which this decoder can pause).
enum InfMode { kModeHead = 0, kModeBlock, kModeStored, kModeCodes, kModeCopy, kModeTrailer, kModeDone, kModeBad, kModeDict };

// strm->msg texts of the reference (inflate.c, inffast.c), by index.
enum InfMsg { kMsgNone = 0, kMsgHeader, kMsgMethod, kMsgWindow, kMsgNeedDict, kMsgBlockType, kMsgStored,
              kMsgTooMany, kMsgCodeLens, kMsgRepeat, kMsgLitSet, kMsgDistSet, kMsgBadLit, kMsgBadDist,
              kMsgFar, kMsgCheck, kMsgLength, kMsgFlags, kMsgHcrc };

constexpr int kWrapAuto = 3;             // windowBits + 32: zlib or gzip, detected from the header (inflate.c:596)
constexpr uint32_t kFlagGzipTrailer = 1;   // InfState::flags: crc / isize hold a gzip trailer that is still to be checked

// Per-call outcome codes of the streaming kernel (beyond zlib's own codes).
enum { kNeedInput = 100, kNeedOutput = 101 };

struct InfState {
    int32_t  mode, last, msg, wrap;
    uint32_t bit_off;                  // bits of the first input byte that are already consumed
    uint32_t stored_left, copy_len, copy_dist;
    uint32_t s1, s2;                   // running Adler-32 of the output
    uint32_t crc, isize;               // running CRC-32 / length (gzip)
    int32_t  nlen, ndist;              // sizes of the code in force (for table rebuild on resume)
    uint64_t hist;                     // valid bytes of history in front of the output pointer
    uint64_t total_out;
    uint32_t dict_id, flags;
    uint8_t  lens[320];
};

struct InfCallResult {                 // written by the streaming kernel
    uint64_t out_len, in_used;
    int32_t  status, msg;
};

// ---- entry points for the ZIP reader (zb_zip.cu) ----
// k_inflate_batch over a subset of members: stream k of the launch is member ids[k], which occupies d_src[d_beg[i] ..
// d_end[i]) and decodes (raw deflate) into d_dst[d_dst_beg[i] .. d_dst_end[i]); d_dst_len / d_status are indexed by member.
int inflate_members_launch(const uint8_t* d_src, const uint64_t* d_beg, const uint64_t* d_end, uint8_t* d_dst, const uint64_t* d_dst_beg,
                           const uint64_t* d_dst_end, const uint32_t* d_ids, size_t nids, uint64_t* d_dst_len, int32_t* d_status,
                           cudaStream_t s, uint64_t* d_in_used = nullptr);
// The one-stream segment decoder (counting pass, then the block finder): 0 = decoded, 1 = declined, negative = CUDA error.
int inflate_single_parallel(Ctx* c, const uint8_t* d_src, uint64_t len, uint8_t* d_dst, uint64_t cap, int wrap,
                            uint64_t* out_len, int32_t* status, cudaStream_t s, uint64_t* in_used = nullptr, uint32_t* adler = nullptr,
                            int* wrap_found = nullptr, void* h_dst = nullptr, uint64_t* need = nullptr);
// (*need: set when the stream was declined because its output, *need bytes, does not fit cap)
// A raw stream at d_src[in_beg .. in_end) whose output is exactly out_len bytes at d_dst + out_off, with nmarks sync markers:
// marks[first_mark ..] are the byte positions right behind them, ascending.
struct PlannedStream { uint64_t in_beg, in_end, out_off, out_len; uint32_t first_mark, nmarks; };
// Segment decode of all of them together; ok[i] = 1 where stream i came out exactly as planned (and, with exact_end, its
// data ends in the last byte of in_end rather than anywhere before it).
int inflate_planned(Ctx* c, const uint8_t* d_src, uint64_t src_len, uint8_t* d_dst, const PlannedStream* ps, size_t np,
                    const uint64_t* marks, uint8_t* ok, cudaStream_t s, bool exact_end = false);
// k_find_markers: every 00 00 FF FF in d_src[first .. last) -> pos[] (the byte behind it), count in *d_count.
int find_markers_launch(const uint8_t* d_src, uint64_t first, uint64_t last, uint32_t* d_count, uint64_t* d_pos, uint32_t cap, cudaStream_t s);

// ---- members of a container whose data spans, output slots, lengths and CRC-32 are stated (zb_zip.cu) ----
// A piece of a byte-moving launch: one CTA copies src[0 .. len) to dst (device memory, no overlap).
struct Piece { const uint8_t* src; uint8_t* dst; uint64_t len; };
constexpr uint32_t kPieceBytes = 256u << 10;
int gather_launch(const Piece* d_pieces, size_t n, cudaStream_t s);
enum { kMemberSkip = 0, kMemberStored = 1, kMemberDeflated = 2 };
struct MemberSpan {
    uint64_t beg, end;               // raw deflate (or stored) data in the source
    uint64_t dst, raw_len;           // output slot and the length the container states
    uint32_t crc32;                  // the CRC-32 it states
    int32_t route, status;           // kMember*; status of a member that is skipped
    uint32_t exact_end;              // 1: the deflate data must end in the last byte of the span (gzip members)
};
// Decodes members[0 .. n) of d_src into d_dst, routed by length: stored -> k_zip_gather, up to one ZB200_CHUNK of output ->
// one k_inflate_batch launch, longer -> sync markers + inflate_planned, else inflate_single_parallel, else the batch.  CRC-32
// and length are checked on the device.  Enqueues everything up to the copy of the results into c->pinned: uint64 lengths
// [n], then int32 statuses [n] (Z_OK, Z_DATA_ERROR, ZB200_UNZ_CRCERROR or the skipped member's status); the caller
// synchronises s before reading them.
int decode_members(Ctx* c, const uint8_t* d_src, uint64_t src_len, uint8_t* d_dst, const MemberSpan* members, size_t n, cudaStream_t s);

}  // namespace zb
