/* zb200.h -- C-ABI extensions of the zb200 engine (additive to zlib.h).
 *
 * zlib.h's calls take one host buffer at a time and 32-bit lengths
 * (h/zlib.h:84,88,1285 in the reference).  The work a B200 is good at is the
 * same arithmetic over device-resident data and over many independent streams
 * at once.  These entry points expose exactly that, with plain pointers and
 * sizes only, so that a maintainer of the reference can bind them from C (or
 * cgo / JNI / ctypes) without any CUDA or torch type.  Each one names the
 * reference routine whose arithmetic it performs.
 *
 * Conventions
 *   - Every buffer argument may be host memory (pageable or pinned) or device
 *     memory of the current device; the library detects which.
 *   - `stream` is a cudaStream_t passed as void* (NULL = CUDA's default stream 0,
 *     as everywhere in CUDA).  Calls whose results land in host variables synchronise that
 *     stream before returning; the *_dev variants never synchronise.
 *   - Return value: Z_OK (0) or a negative zlib error code; text of the last
 *     failure on this thread is available from zb200_last_error().
 *   - There is no CPU implementation behind any of these.
 */
#ifndef ZB200_H
#define ZB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZB200_WRAP_RAW   0      /* windowBits < 0      (qcsrc/deflate.c:255-258) */
#define ZB200_WRAP_ZLIB  1      /* windowBits 8..15    RFC 1950 */
#define ZB200_WRAP_GZIP  2      /* windowBits + 16     RFC 1952 (qcsrc/deflate.c:259-264) */
#define ZB200_WRAP_AUTO  3      /* inflate only: windowBits + 32, zlib or gzip by the first two bytes (qcsrc/inflate.c:596) */

#define ZB200_CHUNK      131072u /* input bytes per independently parsed chunk */

/* ---- lifetime ---------------------------------------------------------- */
int         zb200_init(int device);          /* device < 0: keep the current device */
int         zb200_device_count(void);
const char *zb200_last_error(void);
const char *zb200_build_info(void);          /* "sm_100a, nvcc x.y, ..." */

/* Pinned host memory and device memory without CUDA headers. */
void *zb200_alloc_pinned(size_t bytes);
void  zb200_free_pinned(void *p);
void *zb200_alloc_device(size_t bytes);
void  zb200_free_device(void *p);
int   zb200_copy(void *dst, const void *src, size_t bytes, void *stream);   /* any direction, synchronous */
int   zb200_copy_async(void *dst, const void *src, size_t bytes, void *stream);   /* returns once enqueued */
int   zb200_sync(void *stream);
/* Page-locks host memory the caller already owns (e.g. a shared-memory mapping that several one-GPU processes
 * write their shards into), so that copies to and from it run at pinned speed and asynchronously. */
int   zb200_host_register(void *host_ptr, size_t bytes);
int   zb200_host_unregister(void *host_ptr);
/* Device memory of ANOTHER process on the same box (one process per GPU: torchrun, MPI): the owner exports a 64-byte
 * handle for a buffer it got from zb200_alloc_device, the others open it and may then name it as the destination of
 * zb200_copy_async -- the copy engines move the bytes over NVLink without occupying an SM on either side. */
int   zb200_ipc_export(void *dev_ptr, unsigned char handle[64]);
int   zb200_ipc_open(const unsigned char handle[64], void **peer_ptr);
int   zb200_ipc_close(void *peer_ptr);

/* ---- checksums: crc32() + adler32() in one pass (qcsrc/crc32.c:219, adler32.c:57) ----
 * Computes crc32(0, buf, len) and adler32(1, buf, len); either result pointer may
 * be NULL.  len is 64-bit (the reference's uInt len forces callers to slice). */
int zb200_checksum(const void *buf, size_t len, uint32_t *crc, uint32_t *adler, void *stream);

/* Device-resident form: out2[0] = crc32, out2[1] = adler32, written by the GPU. */
int zb200_checksum_dev(const void *d_buf, size_t len, uint32_t *d_out2, void *stream);

/* n independent buffers in one launch sequence (per-file CRCs of a ZIP archive,
 * per-slice checksums ahead of a _combine tree).  offsets has n+1 entries. */
int zb200_checksum_batch(const void *base, const uint64_t *offsets, size_t n,
                         uint32_t *crc, uint32_t *adler, void *stream);

/* ---- deflate: whole buffer -> one stream (qcsrc/compress.c:22 compress2) ----
 * Input is cut into ZB200_CHUNK-byte chunks, each parsed with the previous
 * 32 KiB as its dictionary, each ending byte-aligned; the result is one valid
 * raw / zlib / gzip stream.  level 0..9 or -1.  *dst_len: in = capacity,
 * out = bytes written.  Z_BUF_ERROR if the capacity is too small. */
int zb200_deflate(const void *src, size_t src_len, void *dst, size_t *dst_len,
                  int level, int wrap, void *stream);

/* As above, also returning what a multi-GPU assembler needs: the checksums of
 * the UNCOMPRESSED input (for crc32_combine / adler32_combine across ranks).
 * flags: bit0 = this shard is not the last one (do not set BFINAL, end on a
 *        byte boundary with an empty stored block instead);
 *        bit1 = omit the stream header; bit2 = omit the trailer.
 * dict/dict_len: up to 32 KiB that precedes src in the logical stream (the tail
 * of the previous rank's shard), or NULL. */
#define ZB200_DEFLATE_NOT_LAST   1
#define ZB200_DEFLATE_NO_HEADER  2
#define ZB200_DEFLATE_NO_TRAILER 4
int zb200_deflate_shard(const void *src, size_t src_len, const void *dict, size_t dict_len,
                        void *dst, size_t *dst_len, int level, int wrap, int flags,
                        uint32_t *crc, uint32_t *adler, void *stream);

/* The same call in two halves: _begin enqueues everything and returns (for pinned host or device buffers without
 * blocking), _end waits and reports.  A caller with several pieces begins piece j + 1 before it ends piece j, so the
 * GPU is never idle while the host reads a length (the multi-GPU rounds do this).  Every _begin needs its _end. */
int zb200_deflate_shard_begin(void **job, const void *src, size_t src_len, const void *dict, size_t dict_len,
                              void *dst, size_t dst_cap, int level, int wrap, int flags, void *stream);
int zb200_deflate_shard_end(void *job, size_t *dst_len, uint32_t *crc, uint32_t *adler);

/* n independent inputs -> n independent streams (minizip-style per-file streams).
 * src/dst are single arenas; src_off and dst_off have n+1 entries (dst_off gives
 * each stream's slot, which must hold compressBound of its input). */
int zb200_deflate_batch(const void *src, const uint64_t *src_off, size_t n,
                        void *dst, const uint64_t *dst_off, uint64_t *dst_len,
                        uint32_t *crc, uint32_t *adler, int32_t *status,
                        int level, int wrap, void *stream);

/* ---- ZIP32 archive of n files compressed in one batch (qcsrc/zip.c:902-1128 member by member) ----
 * names[i] is the member name, file i is src[src_off[i] .. src_off[i+1]) (host or device memory).  The archive is
 * written to dst (host memory); *dst_len: in = capacity, out = archive size (the size needed when Z_BUF_ERROR is
 * returned).  dos_datetime = MS-DOS time in the low and date in the high 16 bits, as in zip.c's dosDate.
 * Z_STREAM_ERROR beyond ZIP32 (65535 members, sizes and offsets below 4 GiB). */
size_t zb200_zip_bound(const char *const *names, const uint64_t *src_off, size_t n);
int zb200_zip_build(const char *const *names, const void *src, const uint64_t *src_off, size_t n,
                    int level, uint32_t dos_datetime, void *dst, size_t *dst_len);

/* The two halves of zb200_zip_build, for archives whose members are compressed on several GPUs (BASELINE
 * config 5): a *segment* is the run of [local header | name | raw deflate data] records of some members, laid out
 * on the device and delivered to dst (host or device memory) in one piece; segments concatenate.  members[i]
 * receives what the central directory needs; local_off is relative to the segment -- add the segment's position in
 * the archive before calling zb200_zip_directory, which writes the central directory and the end record for ALL
 * members of the archive at dst (host memory; the directory starts at byte cd_offset of the archive). */
typedef struct zb200_zip_member {
    uint64_t local_off;              /* position of the member's local header */
    uint64_t comp_len, raw_len;
    uint32_t crc32, reserved;
} zb200_zip_member;
int zb200_zip_segment(const char *const *names, const void *src, const uint64_t *src_off, size_t n,
                      int level, uint32_t dos_datetime, void *dst, size_t *dst_len, zb200_zip_member *members);
int zb200_zip_directory(const char *const *names, const zb200_zip_member *members, size_t n,
                        uint32_t dos_datetime, uint64_t cd_offset, void *dst, size_t *dst_len);

/* ---- ZIP32 archives: reading (qcsrc/unzip.c, member by member in the reference) ----
 * zb200_zip_list parses the central directory on the host, as unzOpen does: the end record is searched back through
 * the archive comment, leading bytes in front of the archive are allowed (every offset below is into the buffer as
 * given), multi-disk and ZIP64 archives are refused with Z_STREAM_ERROR.  The archive may be host or device memory (a
 * device archive has its end record and directory copied to the host).  *n: in = capacity, out = member count;
 * Z_BUF_ERROR (with *n = the count needed) when the capacity is too small.
 * zb200_zip_extract decodes entries[0 .. n) -- any subset of an archive, in any order -- into dst[dst_off[i] ..
 * dst_off[i+1]), all on the GPU; archive and dst may each be host or device memory.  dst_len[i] = bytes produced;
 * status[i] = Z_OK (length and CRC-32 as the directory states), ZB200_UNZ_BADZIPFILE (local header missing or not
 * coherent with the directory as unzip.c checks it, a method other than stored / deflated, a stored member whose sizes
 * differ, data outside the archive), Z_STREAM_ERROR (encrypted), Z_BUF_ERROR (slot smaller than raw_len), Z_DATA_ERROR
 * (invalid deflate data or a length other than raw_len), ZB200_UNZ_CRCERROR.  Returns Z_OK when the batch ran. */
typedef struct zb200_zip_entry {
    uint64_t local_off;          /* local header, as an offset into the archive buffer */
    uint64_t comp_len, raw_len;
    uint64_t name_off;           /* the member name inside the archive buffer (its central directory record) */
    uint32_t crc32;
    uint16_t method, flags;      /* compression method, general purpose bit flag */
    uint16_t name_len, reserved16;
    uint32_t reserved32;
} zb200_zip_entry;               /* 48 bytes */

#define ZB200_UNZ_BADZIPFILE (-103)   /* values of minizip's unzip.h */
#define ZB200_UNZ_CRCERROR   (-105)

int zb200_zip_list(const void *archive, size_t arc_len, zb200_zip_entry *entries, size_t *n);
int zb200_zip_extract(const void *archive, size_t arc_len, const zb200_zip_entry *entries, size_t n,
                      void *dst, const uint64_t *dst_off, uint64_t *dst_len, int32_t *status, void *stream);

/* ---- gzip files of several members (RFC 1952 2.2: cat a.gz b.gz, gzip append mode, BGZF) ----
 * zb200_gunzip: gzip FILE -> its content, all members decoded on the GPU (what gzip -d / Python's gzip.decompress return).
 * src, dst: host or device memory.  *dst_len: in = capacity, out = bytes written; on Z_BUF_ERROR, the sum of the
 * members' ISIZE fields (exact when every member is below 4 GiB).  *members: out = member count on Z_OK, index of the
 * first member that failed on Z_DATA_ERROR (zb200_last_error() names it and its byte offset).
 * Accepted and refused exactly as Python 3.12's gzip.decompress does (zero bytes after a member are skipped, empty input
 * is zero members; leading zeros, trailing non-zero bytes, truncation, a wrong CRC-32 or ISIZE, a method other than 8
 * are Z_DATA_ERROR), except that reserved FLG bits and a wrong FHCRC are Z_DATA_ERROR as in zlib's inflate.
 * inflate(), uncompress() and zb200_inflate_batch still stop at the end of the first member. */
int zb200_gunzip(const void *src, size_t src_len, void *dst, size_t *dst_len, size_t *members, void *stream);

/* BGZF (SAM/BAM specification 4.1): src cut into 65280-byte blocks (bgzip's BGZF_BLOCK_SIZE), each one independent gzip
 * member with the 'BC' extra subfield holding BSIZE = member length - 1, followed by the 28-byte BGZF EOF block.
 * level 0..9 or -1.  src, dst: host or device memory.  *dst_len: in = capacity, out = bytes written. */
size_t zb200_bgzf_bound(size_t src_len);     /* ceil(src_len / 65280) * 65536 + 28 */
int    zb200_bgzf_compress(const void *src, size_t src_len, void *dst, size_t *dst_len, int level, void *stream);

/* ---- inflate: n independent streams (qcsrc/uncompr.c:26 uncompress, batched) ----
 * Stream i occupies src[src_off[i] .. src_off[i+1]) and is decoded into
 * dst[dst_off[i] .. dst_off[i+1]).  Per stream: dst_len[i] = bytes produced,
 * status[i] = Z_OK / Z_DATA_ERROR / Z_BUF_ERROR with uncompress()'s mapping
 * (qcsrc/uncompr.c:53-55).  Returns Z_OK if the batch ran, whatever the per-stream
 * statuses are.  wrap: ZB200_WRAP_RAW / _ZLIB / _GZIP / _AUTO; gzip members have their
 * header fields skipped (FHCRC verified) and CRC-32 + ISIZE checked (qcsrc/inflate.c:634-759,1099-1112). */
int zb200_inflate_batch(const void *src, const uint64_t *src_off, size_t n,
                        void *dst, const uint64_t *dst_off, uint64_t *dst_len,
                        int32_t *status, int wrap, void *stream);

/* Fully device-resident form: every pointer is device memory, nothing is copied,
 * nothing synchronises -- and therefore every stream is decoded by one warp, however long
 * it is.  zb200_inflate_batch (which may synchronise) decodes the long streams of a call in
 * parallel: at their sync markers, or at block starts it finds (see DESIGN.md). */
int zb200_inflate_batch_dev(const void *d_src, const uint64_t *d_src_off, size_t n,
                            void *d_dst, const uint64_t *d_dst_off, uint64_t *d_dst_len,
                            int32_t *d_status, int wrap, void *stream);

/* ---- sizing: what zb200_inflate_batch would produce, without producing it ----
 * Stream i = src[src_off[i] .. src_off[i+1]), as in zb200_inflate_batch (same wrap values, RAW / ZLIB / GZIP / AUTO).
 * out_len[i]  = the bytes zb200_inflate_batch writes for that stream into a slot of unlimited size (or of `limit` bytes).
 * src_used[i] = input bytes the stream occupies, through its trailer (may be NULL): where the next thing in the buffer starts.
 * status[i]   = what zb200_inflate_batch would return for it, with one exception: the zlib Adler-32 and the gzip CRC-32
 *               are NOT verified (they need the output bytes); a stream whose only fault is a wrong check value is Z_OK.
 *               The gzip ISIZE is verified (against out_len mod 2^32), and so is FHCRC.
 * limit: 0 = none; otherwise counting stops at `limit` bytes and a stream with input left reports Z_BUF_ERROR and
 *        out_len = limit, exactly what zb200_inflate_batch reports for a slot of `limit` bytes (a bound on hostile input).
 * src: host (pageable or pinned) or device memory; the results land in host arrays (the call synchronises its stream).
 * Feeding out_len back as slot sizes makes zb200_inflate_batch reproduce the same lengths and statuses (but for the
 * check values).  Long streams are sized by the counting pass of the segment decoder (see DESIGN.md), all others by a
 * count-only form of the batch kernel: no output is stored, so a 5 MB stream may stand for 5 GiB. */
int zb200_inflate_batch_size(const void *src, const uint64_t *src_off, size_t n, uint64_t *out_len, uint64_t *src_used,
                             int32_t *status, int wrap, uint64_t limit, void *stream);

/* Device-resident form: every pointer is device memory, nothing is copied, nothing synchronises (so, like
 * zb200_inflate_batch_dev, every stream is counted by one warp however long it is).  d_dst_off (may be NULL; n + 1
 * entries) receives the exclusive prefix sum of d_out_len, i.e. a ready d_dst_off for zb200_inflate_batch_dev. */
int zb200_inflate_batch_size_dev(const void *d_src, const uint64_t *d_src_off, size_t n, uint64_t *d_out_len,
                                 uint64_t *d_src_used, int32_t *d_status, uint64_t *d_dst_off, int wrap, uint64_t limit,
                                 void *stream);

/* ---- all GPUs of the box behind one call (SURVEY.md 8(e)): one host thread per device inside the library ----
 * Host buffers, like zlib.h's own calls (pinned memory moves fastest).  ndev <= 0 means every visible device.
 * zb200_multi_deflate: the input is cut into chunk-aligned pieces dealt round robin over the devices; every piece is
 *   compressed with the 32 KiB in front of it as dictionary and ends on a byte boundary; one NCCL all-gather per round of
 *   {compressed bytes, input bytes, crc32, adler32} places every piece in the stream, the bytes go D2H straight there.
 *   Result: ONE valid raw / zlib / gzip stream in dst (what compress2 returns for the whole buffer, qcsrc/compress.c:22).
 * zb200_multi_checksum: a slice per device, all-gather of {crc32, adler32, len}, crc32_combine / adler32_combine fold
 *   (qcsrc/crc32.c:370, qcsrc/adler32.c:128) in slice order.
 * zb200_multi_inflate_batch: zb200_inflate_batch with the streams dealt to the devices in contiguous ranges of nearly
 *   equal compressed size; no exchange.
 * NCCL (libnccl.so.2) is loaded at run time by the first of these calls. */
int zb200_multi_devices(void);
int zb200_multi_deflate(const void *src, size_t src_len, void *dst, size_t *dst_len, int level, int wrap, int ndev,
                        uint32_t *crc, uint32_t *adler);
int zb200_multi_checksum(const void *buf, size_t len, int ndev, uint32_t *crc, uint32_t *adler);
int zb200_multi_inflate_batch(const void *src, const uint64_t *src_off, size_t n, void *dst, const uint64_t *dst_off,
                              uint64_t *dst_len, int32_t *status, int wrap, int ndev);

/* ---- instrumentation -------------------------------------------------- */
/* Number of kernels this library has launched since load (all threads). */
uint64_t zb200_kernel_launches(void);

/* Per-kernel device time: zb200_profile(1) starts bracketing every launch with CUDA events on its
 * stream, zb200_profile_report() synchronises and writes "kernel=total_ms:launches;..." . */
void zb200_profile(int enable);
int  zb200_profile_report(char *out, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* ZB200_H */
