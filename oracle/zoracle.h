/* zoracle.h -- CPU oracle for the zb200 hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C restatement of the reference's algorithms (zlib 1.2.3 as shipped in
 * ChrisHird/ZLIB, /root/reference).  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this library; the
 * product (libzb200.so) never links, loads or calls it.
 *
 * Pinning: tests/test_oracle_pin.py checks every function here against
 *   (1) the known-answer anchors listed in SURVEY.md section 8(c), committed
 *       under tests/golden/, and
 *   (2) oracle/_ref/libzref.so = the unmodified reference sources compiled by
 *       oracle/Makefile, whenever that build is present,
 * including BYTE-IDENTICAL compressed output for zo_deflate at levels 0..9.
 */
#ifndef ZORACLE_H
#define ZORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZO_OK            0
#define ZO_STREAM_END    1
#define ZO_NEED_DICT     2
#define ZO_STREAM_ERROR (-2)
#define ZO_DATA_ERROR   (-3)
#define ZO_MEM_ERROR    (-4)
#define ZO_BUF_ERROR    (-5)

/* wrap: 0 = raw deflate, 1 = zlib (RFC 1950), 2 = gzip (RFC 1952) */

uint32_t zo_crc32(uint32_t crc, const uint8_t *buf, size_t len);
uint32_t zo_adler32(uint32_t adler, const uint8_t *buf, size_t len);
uint32_t zo_crc32_combine(uint32_t crc1, uint32_t crc2, int64_t len2);
uint32_t zo_adler32_combine(uint32_t adler1, uint32_t adler2, int64_t len2);

size_t zo_compress_bound(size_t n);

/* One-shot compressor: byte-identical to the reference's
 * deflateInit2(level, 8, wbits(wrap), 8, Z_DEFAULT_STRATEGY) + deflate(Z_FINISH)
 * with all input available and ample output space. */
int zo_deflate(const uint8_t *in, size_t n, uint8_t *out, size_t cap,
               size_t *out_len, int level, int wrap);

/* One-shot decompressor with the error mapping of the reference's
 * uncompress() (uncompr.c:26-61).  *in_used receives the bytes consumed. */
int zo_inflate(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap,
               size_t *out_len, size_t *in_used, int wrap);

/* Last error text of zo_inflate on this thread (same strings as strm->msg). */
const char *zo_last_msg(void);

/* Largest match distance the last zo_inflate on this thread decoded (0 if none): what a
 * stream asks of the window its header declares. */
size_t zo_last_max_dist(void);

#ifdef __cplusplus
}
#endif
#endif
