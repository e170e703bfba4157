/* zapi_stream.c -- the streaming half of zlib.h over the zb200 engine (host C).
 *
 * deflate side (qcsrc/deflate.c:204-947): the reference compresses as bytes arrive through
 * a 64 KiB sliding window.  The engine wants whole chunks, so this shim only does the
 * stream bookkeeping the reference's deflate() driver does (deflate.c:552-856): header,
 * trailer, flush semantics, return codes, totals -- and accumulates input until there is
 * something worth a launch (a flush request, Z_FINISH, or ZS_BATCH bytes).  Every batch goes
 * to zb200_deflate_shard() with the previous 32 KiB as dictionary; a batch that is not the
 * last ends with the empty stored block of Z_SYNC_FLUSH, so batches concatenate.
 *
 * inflate side (qcsrc/inflate.c:103-1368): the device keeps the decoder state
 * (zb200i_inflater); each inflate() call is one resume of that state.
 *
 * No byte of deflate/inflate/checksum arithmetic is computed here.
 */
#include "../../include/zlib.h"
#include "../../include/zb200.h"
#include "zb200_internal.h"
#include <stdlib.h>
#include <string.h>

#define ZAPI __attribute__((visibility("default")))
#define BASE 65521UL
#define ZS_BATCH (32u << 20)          /* input bytes gathered before an unforced launch */
#define ZS_WINDOW 32768u

enum { KIND_DEFLATE = 0x5a44, KIND_INFLATE = 0x5a49 };
enum { ST_INIT = 1, ST_BUSY = 2, ST_FINISH = 3 };
enum { GZ_FIXED = 0, GZ_XLEN, GZ_EXTRA, GZ_NAME, GZ_COMMENT, GZ_HCRC, GZ_DONE };   /* gzip header capture, see gz_capture */

struct internal_state {
    int kind;
    z_streamp strm;
    /* ---- deflate ---- */
    int level, strategy, wrap, status, last_flush, wbits, mem_level;
    unsigned char *in; size_t in_len, in_cap;          /* gathered, not yet compressed */
    unsigned char hist[ZS_WINDOW]; size_t hist_len;    /* tail of what was already compressed */
    unsigned char *out; size_t out_pos, out_len, out_cap;   /* compressed, not yet delivered */
    uLong check;                                       /* running adler32 / crc32 of the input */
    int dict_set; uLong dict_id;
    unsigned bi_bits; unsigned long bi_val;            /* bits that precede the next block (deflatePrime, Z_PARTIAL_FLUSH): deflate.h bi_valid / bi_buf */
    gz_headerp gzhead;
    int trailer_done;
    /* ---- inflate ---- */
    zb200i_inflater *inf;
    int inf_wrap, inf_done, inf_bad, inf_started;
    int sync_on; unsigned sync_have;                   /* inflateSync under way (mode SYNC) and the marker bytes matched so far: state->have */
    uLong inf_dict_id;
    /* gzip header capture for inflateGetHeader (inflate.c:634-759): a host-side shadow of the bytes the device skips */
    gz_headerp gz_head;
    int gz_st; unsigned gz_have, gz_flags, gz_xlen;
    unsigned char gz_fix[10];
};
typedef struct internal_state zs;

static const char *const z_msgs[] = {"need dictionary", "stream end", "", "file error", "stream error",
                                     "data error", "insufficient memory", "buffer error", "incompatible version", ""};
#define ERR_MSG(e) ((char *)z_msgs[2 - (e)])
#define ERR_RETURN(strm, e) return ((strm)->msg = ERR_MSG(e), (e))

static voidpf def_alloc(voidpf opaque, uInt items, uInt size) { (void)opaque; return malloc((size_t)items * size); }
static void def_free(voidpf opaque, voidpf p) { (void)opaque; free(p); }

/* exact Adler-32 concatenation (the public adler32_combine keeps the reference's '>' folds) */
static uLong adler_join(uLong a1, uLong a2, size_t len2)
{
    unsigned long rem = (unsigned long)(len2 % BASE);
    unsigned long s1 = a1 & 0xffff, s2 = (a1 >> 16) & 0xffff;
    unsigned long t1 = a2 & 0xffff, t2 = (a2 >> 16) & 0xffff;
    unsigned long r1 = (s1 + t1 + BASE - 1) % BASE;
    unsigned long r2 = (s2 + t2 + rem * s1 + BASE - rem) % BASE;
    return r1 | (r2 << 16);
}

/* ======================================================================== deflate */

/* Every byte a stream owns comes from the caller's allocator (deflate.c:243-247 promises that for the reference's
 * window, hash tables and pending buffer; here it is the gather buffer and the pending output).  zalloc takes 32-bit
 * item counts and sizes, so buffers are requested in 4 KiB items.  `keep` bytes of the old buffer survive. */
static int zs_reserve(z_streamp strm, unsigned char **buf, size_t *cap, size_t want, size_t keep)
{
    unsigned char *p;
    size_t n;
    if (want <= *cap) return 0;
    n = *cap ? *cap : 4096;
    while (n < want) n *= 2;
    if ((n >> 12) > 0xffffffffUL) return -1;
    p = (unsigned char *)strm->zalloc(strm->opaque, (uInt)(n >> 12), 4096u);
    if (!p) return -1;
    if (*buf) {
        if (keep) memcpy(p, *buf, keep);
        strm->zfree(strm->opaque, *buf);
    }
    *buf = p; *cap = n;
    return 0;
}

static int out_append(zs *s, const unsigned char *p, size_t n)
{
    if (s->out_pos == s->out_len) s->out_pos = s->out_len = 0;
    if (zs_reserve(s->strm, &s->out, &s->out_cap, s->out_len + n, s->out_len)) return -1;
    memcpy(s->out + s->out_len, p, n);
    s->out_len += n;
    return 0;
}

static void out_deliver(z_streamp strm)                     /* flush_pending, deflate.c:532 */
{
    zs *s = strm->state;
    size_t n = s->out_len - s->out_pos;
    if (n > strm->avail_out) n = strm->avail_out;
    if (n == 0) return;
    memcpy(strm->next_out, s->out + s->out_pos, n);
    strm->next_out += n; strm->avail_out -= (uInt)n; strm->total_out += n;
    s->out_pos += n;
}

ZAPI int deflateInit2_(z_streamp strm, int level, int method, int windowBits, int memLevel, int strategy,
                       const char *version, int stream_size)
{
    zs *s;
    int wrap = 1;
    if (version == Z_NULL || version[0] != ZLIB_VERSION[0] || stream_size != (int)sizeof(z_stream))
        return Z_VERSION_ERROR;                                 /* deflate.c:236-239 */
    if (strm == Z_NULL) return Z_STREAM_ERROR;
    strm->msg = Z_NULL;
    if (strm->zalloc == (alloc_func)0) { strm->zalloc = def_alloc; strm->opaque = (voidpf)0; }
    if (strm->zfree == (free_func)0) strm->zfree = def_free;
    if (level == Z_DEFAULT_COMPRESSION) level = 6;
    if (windowBits < 0) { wrap = 0; windowBits = -windowBits; }
    else if (windowBits > 15) { wrap = 2; windowBits -= 16; }
    if (memLevel < 1 || memLevel > MAX_MEM_LEVEL || method != Z_DEFLATED || windowBits < 8 || windowBits > 15 ||
        level < 0 || level > 9 || strategy < 0 || strategy > Z_FIXED)
        return Z_STREAM_ERROR;                                  /* deflate.c:265-269 */
    if (windowBits == 8) windowBits = 9;                        /* deflate.c:270: the reference never runs a 256-byte window */
    if (zb200_init(-1) != Z_OK) return Z_STREAM_ERROR;          /* no device, no stream: there is no CPU path */
    s = (zs *)strm->zalloc(strm->opaque, 1, (uInt)sizeof(zs));
    if (s == Z_NULL) return Z_MEM_ERROR;
    memset(s, 0, sizeof(zs));
    strm->state = s;
    s->kind = KIND_DEFLATE; s->strm = strm;
    s->level = level; s->strategy = strategy; s->wrap = wrap; s->wbits = windowBits; s->mem_level = memLevel;
    return deflateReset(strm);
}

ZAPI int deflateInit_(z_streamp strm, int level, const char *version, int stream_size)
{
    return deflateInit2_(strm, level, Z_DEFLATED, MAX_WBITS, 8, Z_DEFAULT_STRATEGY, version, stream_size);
}

ZAPI int deflateReset(z_streamp strm)                           /* deflate.c:357-390 */
{
    zs *s;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    strm->total_in = strm->total_out = 0;
    strm->msg = Z_NULL;
    strm->data_type = Z_UNKNOWN;
    s->in_len = 0; s->hist_len = 0; s->out_pos = s->out_len = 0;
    if (s->wrap < 0) s->wrap = -s->wrap;
    s->status = s->wrap ? ST_INIT : ST_BUSY;
    strm->adler = s->wrap == 2 ? 0UL : 1UL;
    s->check = strm->adler;
    s->last_flush = Z_NO_FLUSH;
    s->dict_set = 0; s->trailer_done = 0;
    s->bi_bits = 0; s->bi_val = 0;
    return Z_OK;
}

ZAPI int deflateEnd(z_streamp strm)                             /* deflate.c:859-887 */
{
    zs *s;
    int busy;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    busy = s->status == ST_BUSY;            /* deflate.c:886: ending before Z_FINISH completed is a data error */
    if (s->in) strm->zfree(strm->opaque, s->in);
    if (s->out) strm->zfree(strm->opaque, s->out);
    strm->zfree(strm->opaque, s);
    strm->state = Z_NULL;
    return busy ? Z_DATA_ERROR : Z_OK;
}

ZAPI int deflateSetDictionary(z_streamp strm, const Bytef *dictionary, uInt dictLength)   /* deflate.c:315-354 */
{
    zs *s;
    size_t n = dictLength;
    if (strm == Z_NULL || strm->state == Z_NULL || dictionary == Z_NULL || strm->state->kind != KIND_DEFLATE)
        return Z_STREAM_ERROR;
    s = strm->state;
    if (s->wrap == 2 || (s->wrap == 1 && s->status != ST_INIT)) return Z_STREAM_ERROR;
    if (s->wrap) {
        strm->adler = adler32(strm->adler, dictionary, dictLength);
        s->dict_set = 1; s->dict_id = strm->adler;
    }
    if (n < 3) return Z_OK;
    if (n > ZS_WINDOW) { dictionary += n - ZS_WINDOW; n = ZS_WINDOW; }
    memcpy(s->hist, dictionary, n);
    s->hist_len = n;
    return Z_OK;
}

ZAPI uLong deflateBound(z_streamp strm, uLong sourceLen)        /* deflate.c:489-517 */
{
    zs *s;
    uLong destLen = sourceLen + ((sourceLen + 7) >> 3) + ((sourceLen + 63) >> 6) + 11, more = 0;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return destLen;
    s = strm->state;
    /* both formulas count the 6 bytes of the zlib wrapper; what a stream writes beyond them is added, as zlib 1.2.5.1
     * and later do: the dictionary id, or the gzip wrapper (18 bytes) and the deflateSetHeader fields */
    if ((s->wrap == 1 || s->wrap == -1) && s->dict_set) more = 4;      /* the wrap turns negative once the trailer is out */
    else if (s->wrap == 2 || s->wrap == -2) {
        gz_headerp g = s->gzhead;
        more = 18 - 6;
        if (g != Z_NULL) {
            if (g->extra != Z_NULL) more += 2 + (g->extra_len & 0xffff);
            if (g->name != Z_NULL) more += (uLong)strlen((const char *)g->name) + 1;
            if (g->comment != Z_NULL) more += (uLong)strlen((const char *)g->comment) + 1;
            if (g->hcrc) more += 2;
        }
    }
    if (s->wbits != 15 || s->mem_level != 8) return destLen + more;
    return compressBound(sourceLen) + more;
}

ZAPI int deflateTune(z_streamp strm, int good_length, int max_lazy, int nice_length, int max_chain)
{
    (void)good_length; (void)max_lazy; (void)nice_length; (void)max_chain;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return Z_STREAM_ERROR;
    return Z_OK;            /* search budgets are fixed per level in the kernels (deflate.c:454-470 only stores them) */
}

ZAPI int deflatePrime(z_streamp strm, int bits, int value)     /* deflate.c:404-414 */
{
    zs *s;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return Z_STREAM_ERROR;
    if (bits < 0 || bits > 16) return Z_STREAM_ERROR;
    s = strm->state;
    s->bi_bits = (unsigned)bits;                                /* the reference overwrites bi_valid / bi_buf the same way */
    s->bi_val = (unsigned long)value & ((1UL << bits) - 1UL);
    return Z_OK;
}

ZAPI int deflateSetHeader(z_streamp strm, gz_headerp head)      /* deflate.c:393-401 */
{
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return Z_STREAM_ERROR;
    if (strm->state->wrap != 2) return Z_STREAM_ERROR;
    strm->state->gzhead = head;
    return Z_OK;
}

/* Framing bits written by the host: appends `n` bits to the pending ones and moves whole bytes to the output.  Only
 * block headers of EMPTY blocks and alignment go through here (send_bits, trees.c:217); data never does. */
static int bits_put(zs *s, unsigned long value, unsigned n)
{
    s->bi_val |= value << s->bi_bits;
    s->bi_bits += n;
    while (s->bi_bits >= 8) {
        unsigned char b = (unsigned char)(s->bi_val & 0xff);
        if (out_append(s, &b, 1)) return -1;
        s->bi_val >>= 8; s->bi_bits -= 8;
    }
    return 0;
}

static int bits_align(zs *s)                                    /* bi_windup, trees.c:1178 */
{
    return s->bi_bits ? bits_put(s, 0, 8 - s->bi_bits) : 0;
}

static int bits_marker(zs *s)                                   /* _tr_stored_block(0 bytes), trees.c:867: 000, pad, 00 00 FF FF */
{
    static const unsigned char m[4] = {0, 0, 0xff, 0xff};
    if (bits_put(s, 0, 3) || bits_align(s)) return -1;
    return out_append(s, m, 4);
}

enum { END_NONE = 0, END_MARK = 1, END_PARTIAL = 2 };

/* compress everything gathered so far into the pending buffer; `end` says how a batch that is not the last one ends:
 * as the blocks fall (END_NONE: a byte-aligning marker all the same, batches concatenate on byte boundaries), with the
 * empty stored block of Z_SYNC_FLUSH / Z_FULL_FLUSH (END_MARK), or with the empty static block of Z_PARTIAL_FLUSH
 * (END_PARTIAL, _tr_align, trees.c:892) after which the stream stays where its bits fall. */
static int zs_compress(z_streamp strm, int level, int final, int end)
{
    zs *s = strm->state;
    size_t cap, got;
    uint32_t crc = 0, adler = 1, tail = 0;
    int rc, flags = 0;
    /* whole bytes of a deflatePrime (up to 16 bits) leave first */
    if (s->bi_bits >= 8 && bits_put(s, 0, 0)) return Z_MEM_ERROR;
    if (s->in_len == 0) {                                       /* nothing gathered: the empty blocks are host framing */
        if (final) { if (bits_put(s, 3, 10) || bits_align(s)) return Z_MEM_ERROR; }      /* final empty static block: 03 00 when aligned */
        else if (end == END_PARTIAL) { if (bits_put(s, 2, 10)) return Z_MEM_ERROR; }
        else if (end == END_MARK || s->bi_bits) { if (bits_marker(s)) return Z_MEM_ERROR; }
        return Z_OK;
    }
    if (level == 0) {                                           /* stored blocks are whole bytes: pending bits are closed first */
        if (s->bi_bits && bits_marker(s)) return Z_MEM_ERROR;
        if (end == END_PARTIAL) end = END_MARK;
    }
    if (!final) flags |= ZB200_DEFLATE_NOT_LAST;
    if (end == END_MARK) flags |= ZB200I_DEFLATE_FORCE_MARK;
    if (s->strategy != Z_DEFAULT_STRATEGY) flags |= (s->strategy << 8);       /* Z_FILTERED, Z_HUFFMAN_ONLY, Z_RLE, Z_FIXED */
    if (s->wbits != 15) flags |= ZB200I_DEFLATE_WBITS(s->wbits);              /* match distances stay inside the declared window */
    cap = (size_t)compressBound((uLong)s->in_len) + 64;
    if (s->out_pos == s->out_len) s->out_pos = s->out_len = 0;
    if (zs_reserve(strm, &s->out, &s->out_cap, s->out_len + cap, s->out_len)) return Z_MEM_ERROR;
    got = cap;
    if (s->bi_bits || (end == END_PARTIAL && !final))
        rc = zb200i_deflate_shard_bits(s->in, s->in_len, s->hist_len ? s->hist : NULL, s->hist_len, s->out + s->out_len, &got,
                                       level, flags, s->bi_bits, (uint32_t)s->bi_val, end == END_PARTIAL && !final, &tail, &crc, &adler);
    else
        rc = zb200_deflate_shard(s->in, s->in_len, s->hist_len ? s->hist : NULL, s->hist_len, s->out + s->out_len, &got,
                                 level, ZB200_WRAP_RAW, flags | ZB200_DEFLATE_NO_HEADER | ZB200_DEFLATE_NO_TRAILER, &crc, &adler, NULL);
    if (rc != Z_OK) return rc;
    s->out_len += got;
    s->bi_bits = tail & 0xff; s->bi_val = tail >> 8;
    if (s->wrap == 1) s->check = adler_join(s->check, adler, s->in_len);
    else if (s->wrap == 2) s->check = crc32_combine(s->check, crc, (z_off_t)s->in_len);
    strm->adler = s->check;
    /* keep the last 32 KiB as the next batch's dictionary */
    if (s->in_len >= ZS_WINDOW) { memcpy(s->hist, s->in + s->in_len - ZS_WINDOW, ZS_WINDOW); s->hist_len = ZS_WINDOW; }
    else {
        size_t keep = ZS_WINDOW - s->in_len;
        if (keep > s->hist_len) keep = s->hist_len;
        memmove(s->hist, s->hist + s->hist_len - keep, keep);
        memcpy(s->hist + keep, s->in, s->in_len);
        s->hist_len = keep + s->in_len;
    }
    s->in_len = 0;
    return Z_OK;
}

static int put_header(z_streamp strm)                           /* deflate.c:577-753 */
{
    zs *s = strm->state;
    unsigned char h[16];
    if (s->wrap == 2) {
        gz_headerp g = s->gzhead;
        unsigned xfl = s->level == 9 ? 2 : (s->strategy >= Z_HUFFMAN_ONLY || s->level < 2 ? 4 : 0);
        size_t start = s->out_len;
        h[0] = 31; h[1] = 139; h[2] = 8;
        if (g == Z_NULL) {
            h[3] = 0; h[4] = h[5] = h[6] = h[7] = 0; h[8] = (unsigned char)xfl; h[9] = 3;
            if (out_append(s, h, 10)) return Z_MEM_ERROR;
        } else {
            h[3] = (unsigned char)((g->text ? 1 : 0) + (g->hcrc ? 2 : 0) + (g->extra == Z_NULL ? 0 : 4) +
                                   (g->name == Z_NULL ? 0 : 8) + (g->comment == Z_NULL ? 0 : 16));
            h[4] = (unsigned char)(g->time & 0xff); h[5] = (unsigned char)((g->time >> 8) & 0xff);
            h[6] = (unsigned char)((g->time >> 16) & 0xff); h[7] = (unsigned char)((g->time >> 24) & 0xff);
            h[8] = (unsigned char)xfl; h[9] = (unsigned char)(g->os & 0xff);
            if (out_append(s, h, 10)) return Z_MEM_ERROR;
            if (g->extra != Z_NULL) {
                h[0] = (unsigned char)(g->extra_len & 0xff); h[1] = (unsigned char)((g->extra_len >> 8) & 0xff);
                if (out_append(s, h, 2) || out_append(s, g->extra, g->extra_len & 0xffff)) return Z_MEM_ERROR;
            }
            if (g->name != Z_NULL && out_append(s, g->name, strlen((const char *)g->name) + 1)) return Z_MEM_ERROR;
            if (g->comment != Z_NULL && out_append(s, g->comment, strlen((const char *)g->comment) + 1)) return Z_MEM_ERROR;
            if (g->hcrc) {
                uLong c = crc32(0UL, s->out + start, (uInt)(s->out_len - start));
                h[0] = (unsigned char)(c & 0xff); h[1] = (unsigned char)((c >> 8) & 0xff);
                if (out_append(s, h, 2)) return Z_MEM_ERROR;
            }
        }
        strm->adler = s->check = 0UL;
    } else {
        uInt header = (Z_DEFLATED + ((uInt)(s->wbits - 8) << 4)) << 8;
        uInt lf = (s->strategy >= Z_HUFFMAN_ONLY || s->level < 2) ? 0 : s->level < 6 ? 1 : s->level == 6 ? 2 : 3;
        size_t n = 2;
        header |= lf << 6;
        if (s->dict_set) header |= 0x20;
        header += 31 - (header % 31);
        h[0] = (unsigned char)(header >> 8); h[1] = (unsigned char)(header & 0xff);
        if (s->dict_set) {
            h[2] = (unsigned char)(s->dict_id >> 24); h[3] = (unsigned char)(s->dict_id >> 16);
            h[4] = (unsigned char)(s->dict_id >> 8); h[5] = (unsigned char)s->dict_id;
            n = 6;
        }
        if (out_append(s, h, n)) return Z_MEM_ERROR;
        strm->adler = s->check = 1UL;
    }
    s->status = ST_BUSY;
    return Z_OK;
}

ZAPI int deflate(z_streamp strm, int flush)                     /* deflate.c:552-856 */
{
    zs *s;
    int old_flush, rc;
    if (strm == Z_NULL || strm->state == Z_NULL || flush > Z_FINISH || flush < 0 || strm->state->kind != KIND_DEFLATE)
        return Z_STREAM_ERROR;
    s = strm->state;
    if (strm->next_out == Z_NULL || (strm->next_in == Z_NULL && strm->avail_in != 0) ||
        (s->status == ST_FINISH && flush != Z_FINISH))
        ERR_RETURN(strm, Z_STREAM_ERROR);
    if (strm->avail_out == 0) ERR_RETURN(strm, Z_BUF_ERROR);
    s->strm = strm;
    old_flush = s->last_flush;
    s->last_flush = flush;

    if (s->status == ST_INIT && (rc = put_header(strm)) != Z_OK) ERR_RETURN(strm, rc);

    if (s->out_len != s->out_pos) {                             /* deflate.c:755-769 */
        out_deliver(strm);
        if (strm->avail_out == 0) { s->last_flush = -1; return Z_OK; }
    } else if (strm->avail_in == 0 && flush <= old_flush && flush != Z_FINISH) {
        ERR_RETURN(strm, Z_BUF_ERROR);
    }
    if (s->status == ST_FINISH && strm->avail_in != 0) ERR_RETURN(strm, Z_BUF_ERROR);

    if (strm->avail_in != 0 || s->in_len != 0 || (flush != Z_NO_FLUSH && s->status != ST_FINISH)) {
        /* gather (read_buf, deflate.c:956): the engine is greedy, like the reference at any level */
        while (strm->avail_in != 0) {
            size_t room = ZS_BATCH - s->in_len, n = strm->avail_in < room ? strm->avail_in : room;
            if (zs_reserve(strm, &s->in, &s->in_cap, s->in_len + n, s->in_len)) ERR_RETURN(strm, Z_MEM_ERROR);
            memcpy(s->in + s->in_len, strm->next_in, n);
            s->in_len += n; strm->next_in += n; strm->avail_in -= (uInt)n; strm->total_in += n;
            if (s->in_len == ZS_BATCH && (strm->avail_in != 0 || flush == Z_NO_FLUSH)) {
                if ((rc = zs_compress(strm, s->level, 0, END_NONE)) != Z_OK) ERR_RETURN(strm, rc);
            }
        }
        if (flush != Z_NO_FLUSH && s->status != ST_FINISH) {
            if (flush == Z_FINISH) {
                if ((rc = zs_compress(strm, s->level, 1, END_NONE)) != Z_OK) ERR_RETURN(strm, rc);
                s->status = ST_FINISH;
            } else {
                /* deflate.c:808-825: PARTIAL ends on the ten bits of an empty static block and stays unaligned,
                 * SYNC and FULL end on the empty stored block */
                if ((rc = zs_compress(strm, s->level, 0, flush == Z_PARTIAL_FLUSH ? END_PARTIAL : END_MARK)) != Z_OK) ERR_RETURN(strm, rc);
                if (flush == Z_FULL_FLUSH) s->hist_len = 0;     /* forget history */
            }
        }
        out_deliver(strm);
        if (s->out_len != s->out_pos) { s->last_flush = -1; return Z_OK; }
        if (strm->avail_out == 0 && flush != Z_FINISH) { s->last_flush = -1; return Z_OK; }
    }
    if (flush != Z_FINISH) return Z_OK;
    if (s->out_len != s->out_pos) { s->last_flush = -1; return Z_OK; }
    if (s->wrap <= 0) return Z_STREAM_END;

    {   /* trailer, deflate.c:832-855 */
        unsigned char t[8];
        size_t n;
        if (s->wrap == 2) {
            uLong c = s->check, l = strm->total_in;
            t[0] = (unsigned char)(c & 0xff); t[1] = (unsigned char)((c >> 8) & 0xff);
            t[2] = (unsigned char)((c >> 16) & 0xff); t[3] = (unsigned char)((c >> 24) & 0xff);
            t[4] = (unsigned char)(l & 0xff); t[5] = (unsigned char)((l >> 8) & 0xff);
            t[6] = (unsigned char)((l >> 16) & 0xff); t[7] = (unsigned char)((l >> 24) & 0xff);
            n = 8;
        } else {
            uLong a = s->check;
            t[0] = (unsigned char)(a >> 24); t[1] = (unsigned char)(a >> 16); t[2] = (unsigned char)(a >> 8); t[3] = (unsigned char)a;
            n = 4;
        }
        if (out_append(s, t, n)) ERR_RETURN(strm, Z_MEM_ERROR);
        s->wrap = -s->wrap;                                     /* write the trailer only once */
        s->trailer_done = 1;
        out_deliver(strm);
    }
    return s->out_len != s->out_pos ? Z_OK : Z_STREAM_END;
}

ZAPI int deflateParams(z_streamp strm, int level, int strategy)  /* deflate.c:416-451 */
{
    zs *s;
    int err = Z_OK;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_DEFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    if (level == Z_DEFAULT_COMPRESSION) level = 6;
    if (level < 0 || level > 9 || strategy < 0 || strategy > Z_FIXED) return Z_STREAM_ERROR;
    if ((level != s->level || strategy != s->strategy) && strm->total_in != 0) {
        /* what was gathered goes out under the old parameters: deflate(strm, Z_PARTIAL_FLUSH), deflate.c:438-441, with its
         * return codes (Z_BUF_ERROR when avail_out is 0, Z_STREAM_ERROR without an output buffer) */
        err = deflate(strm, Z_PARTIAL_FLUSH);
    }
    s->level = level; s->strategy = strategy;
    return err;
}

ZAPI int deflateCopy(z_streamp dest, z_streamp source)          /* deflate.c:894-947 */
{
    zs *s, *d;
    if (source == Z_NULL || dest == Z_NULL || source->state == Z_NULL || source->state->kind != KIND_DEFLATE)
        return Z_STREAM_ERROR;
    s = source->state;
    memcpy(dest, source, sizeof(z_stream));
    d = (zs *)dest->zalloc(dest->opaque, 1, (uInt)sizeof(zs));
    if (d == Z_NULL) return Z_MEM_ERROR;
    memcpy(d, s, sizeof(zs));
    dest->state = d; d->strm = dest;
    d->in = d->out = NULL; d->in_cap = d->out_cap = 0;
    if (zs_reserve(dest, &d->in, &d->in_cap, s->in_len + 1, 0) || zs_reserve(dest, &d->out, &d->out_cap, s->out_len + 1, 0)) {
        deflateEnd(dest);
        return Z_MEM_ERROR;
    }
    memcpy(d->in, s->in, s->in_len);
    memcpy(d->out, s->out, s->out_len);
    return Z_OK;
}

/* ======================================================================== inflate */

ZAPI int inflateInit2_(z_streamp strm, int windowBits, const char *version, int stream_size)   /* inflate.c:144-185 */
{
    zs *s;
    int wrap, rc;
    if (version == Z_NULL || version[0] != ZLIB_VERSION[0] || stream_size != (int)sizeof(z_stream)) return Z_VERSION_ERROR;
    if (strm == Z_NULL) return Z_STREAM_ERROR;
    strm->msg = Z_NULL;
    if (strm->zalloc == (alloc_func)0) { strm->zalloc = def_alloc; strm->opaque = (voidpf)0; }
    if (strm->zfree == (free_func)0) strm->zfree = def_free;
    if (windowBits < 0) { wrap = 0; windowBits = -windowBits; }
    else { wrap = (windowBits >> 4) + 1; if (windowBits < 48) windowBits &= 15; }
    if (windowBits < 8 || windowBits > 15) return Z_STREAM_ERROR;
    if (wrap > 3) return Z_STREAM_ERROR;      /* 2 = gzip (windowBits + 16), 3 = zlib or gzip (+ 32), inflate.c:159-167 */
    if (zb200_init(-1) != Z_OK) return Z_STREAM_ERROR;
    s = (zs *)strm->zalloc(strm->opaque, 1, (uInt)sizeof(zs));
    if (s == Z_NULL) return Z_MEM_ERROR;
    memset(s, 0, sizeof(zs));
    s->kind = KIND_INFLATE; s->strm = strm; s->inf_wrap = wrap; s->wbits = windowBits;
    rc = zb200i_inflate_open(&s->inf, wrap | (windowBits << 8));   /* the window size rides along (inflate.c:622) */
    if (rc != Z_OK) { strm->zfree(strm->opaque, s); return rc == Z_MEM_ERROR ? Z_MEM_ERROR : Z_STREAM_ERROR; }
    strm->state = s;
    strm->total_in = strm->total_out = 0;
    strm->adler = 1;
    return Z_OK;
}

ZAPI int inflateInit_(z_streamp strm, const char *version, int stream_size)
{
    return inflateInit2_(strm, MAX_WBITS, version, stream_size);
}

ZAPI int inflateReset(z_streamp strm)                           /* inflate.c:103-126 */
{
    zs *s;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    strm->total_in = strm->total_out = 0;
    strm->msg = Z_NULL;
    strm->adler = 1;
    s->inf_done = s->inf_bad = s->inf_started = 0;
    s->sync_on = 0; s->sync_have = 0;
    s->gz_head = Z_NULL; s->gz_st = GZ_FIXED; s->gz_have = 0;
    return zb200i_inflate_reset(s->inf, s->inf_wrap | (s->wbits << 8)) == 0 ? Z_OK : Z_STREAM_ERROR;
}

ZAPI int inflateEnd(z_streamp strm)                             /* inflate.c:1155-1167 */
{
    if (strm == Z_NULL || strm->state == Z_NULL || strm->zfree == (free_func)0 || strm->state->kind != KIND_INFLATE)
        return Z_STREAM_ERROR;
    zb200i_inflate_close(strm->state->inf);
    strm->zfree(strm->opaque, strm->state);
    strm->state = Z_NULL;
    return Z_OK;
}

/* Walks the gzip header as its bytes are consumed and fills the caller's gz_header the way inflate.c:634-759 does:
 * fixed fields, then FEXTRA / FNAME / FCOMMENT clipped to the caller's buffers, then FHCRC; done = 1 at the end of the
 * header, -1 if the stream turns out not to be gzip (windowBits + 32).  The device decoder validates the same bytes.
 * Returns how many of the n bytes it took to see that the magic is not gzip's, 0 if it did not see that. */
static size_t gz_capture(zs *s, const unsigned char *p, size_t n)
{
    gz_headerp h = s->gz_head;
    const size_t n0 = n;
    while (n && s->gz_st != GZ_DONE) {
        const unsigned c = *p++;
        n--;
        switch (s->gz_st) {
        case GZ_FIXED:
            s->gz_fix[s->gz_have++] = (unsigned char)c;
            if (s->gz_have == 2 && (s->gz_fix[0] != 0x1f || s->gz_fix[1] != 0x8b)) {      /* a zlib stream */
                if (h != Z_NULL) h->done = -1;
                s->gz_st = GZ_DONE;
                return n0 - n;
            }
            if (s->gz_have < 10) break;
            s->gz_flags = s->gz_fix[3];
            if (h != Z_NULL) {
                h->text = (int)(s->gz_flags & 1);
                h->time = (uLong)s->gz_fix[4] | ((uLong)s->gz_fix[5] << 8) | ((uLong)s->gz_fix[6] << 16) | ((uLong)s->gz_fix[7] << 24);
                h->xflags = s->gz_fix[8]; h->os = s->gz_fix[9];
                if (!(s->gz_flags & 4)) h->extra = Z_NULL;
                if (!(s->gz_flags & 8)) h->name = Z_NULL;
                if (!(s->gz_flags & 16)) h->comment = Z_NULL;
            }
            s->gz_have = 0;
            s->gz_st = (s->gz_flags & 4) ? GZ_XLEN : (s->gz_flags & 8) ? GZ_NAME : (s->gz_flags & 16) ? GZ_COMMENT : (s->gz_flags & 2) ? GZ_HCRC : GZ_DONE;
            break;
        case GZ_XLEN:
            s->gz_xlen = s->gz_have ? (s->gz_xlen | (c << 8)) : c;
            if (++s->gz_have < 2) break;
            if (h != Z_NULL) h->extra_len = s->gz_xlen;
            s->gz_have = 0;
            s->gz_st = s->gz_xlen ? GZ_EXTRA : (s->gz_flags & 8) ? GZ_NAME : (s->gz_flags & 16) ? GZ_COMMENT : (s->gz_flags & 2) ? GZ_HCRC : GZ_DONE;
            break;
        case GZ_EXTRA:
            if (h != Z_NULL && h->extra != Z_NULL && s->gz_have < h->extra_max) h->extra[s->gz_have] = (Bytef)c;
            if (++s->gz_have < s->gz_xlen) break;
            s->gz_have = 0;
            s->gz_st = (s->gz_flags & 8) ? GZ_NAME : (s->gz_flags & 16) ? GZ_COMMENT : (s->gz_flags & 2) ? GZ_HCRC : GZ_DONE;
            break;
        case GZ_NAME:
            if (h != Z_NULL && h->name != Z_NULL && s->gz_have < h->name_max) h->name[s->gz_have] = (Bytef)c;
            s->gz_have++;
            if (c != 0) break;
            s->gz_have = 0;
            s->gz_st = (s->gz_flags & 16) ? GZ_COMMENT : (s->gz_flags & 2) ? GZ_HCRC : GZ_DONE;
            break;
        case GZ_COMMENT:
            if (h != Z_NULL && h->comment != Z_NULL && s->gz_have < h->comm_max) h->comment[s->gz_have] = (Bytef)c;
            s->gz_have++;
            if (c != 0) break;
            s->gz_have = 0;
            s->gz_st = (s->gz_flags & 2) ? GZ_HCRC : GZ_DONE;
            break;
        case GZ_HCRC:
            if (++s->gz_have == 2) s->gz_st = GZ_DONE;
            break;
        default:
            break;
        }
        if (s->gz_st == GZ_DONE && h != Z_NULL && h->done == 0) {
            h->hcrc = (int)((s->gz_flags >> 1) & 1);
            h->done = 1;
        }
    }
    return 0;
}

ZAPI int inflate(z_streamp strm, int flush)                     /* inflate.c:554-1153 */
{
    zs *s;
    size_t in_used = 0, out_len = 0;
    int status = 0, msg = 0, rc;
    uint32_t check = 1;
    uInt in0, out0;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE || strm->next_out == Z_NULL ||
        (strm->next_in == Z_NULL && strm->avail_in != 0))
        return Z_STREAM_ERROR;
    s = strm->state;
    if (s->inf_bad) return Z_DATA_ERROR;
    if (s->inf_done) return Z_STREAM_END;
    in0 = strm->avail_in; out0 = strm->avail_out;
    if (zb200i_inflate_mode(s->inf) == 8 /* awaiting dictionary */) { strm->adler = s->inf_dict_id; return Z_NEED_DICT; }
    if (out0 == 0 && in0 == 0) return Z_BUF_ERROR;
    if (!s->inf_started && flush == Z_FINISH && s->gz_head == Z_NULL && in0 >= 65536u && s->wbits == 15) {
        /* uncompress() spelled out: the whole stream and the whole buffer in the first call */
        if (zb200i_inflate_try_parallel(strm->next_in, in0, strm->next_out, out0, s->inf_wrap, &in_used, &out_len, &check) == 0) {
            strm->next_in += in_used; strm->avail_in -= (uInt)in_used; strm->total_in += in_used;
            strm->next_out += out_len; strm->avail_out -= (uInt)out_len; strm->total_out += out_len;
            if (s->inf_wrap) strm->adler = check;
            s->inf_started = s->inf_done = 1;
            return Z_STREAM_END;
        }
        in_used = out_len = 0; check = 1;
    }
    s->inf_started = 1;

    rc = zb200i_inflate_run(s->inf, strm->next_in, in0, strm->next_out, out0, &in_used, &out_len, &status, &msg, &check);
    if (rc != Z_OK) { strm->msg = ERR_MSG(rc == Z_MEM_ERROR ? Z_MEM_ERROR : Z_STREAM_ERROR); return rc == Z_MEM_ERROR ? Z_MEM_ERROR : Z_STREAM_ERROR; }
    if (s->inf_wrap >= 2 && s->gz_st != GZ_DONE) {
        size_t at = gz_capture(s, strm->next_in, in_used);
        if (at && s->inf_wrap == 2) {
            /* inflate.c:597-602: gzip only, and the first two bytes are not its magic.  The reference refuses the stream
             * right there; the device parser would wait for the whole fixed header.  What followed goes back to the caller. */
            if (zb200i_inflate_resync(s->inf) != 0) return Z_STREAM_ERROR;       /* drops the bytes the device holds */
            in_used = at; out_len = 0;
            status = Z_DATA_ERROR; msg = 1;                                         /* "incorrect header check" */
        }
    }
    if (in_used || out_len) s->sync_on = 0;                     /* decoding went on: an earlier inflateSync is over */
    strm->next_in += in_used; strm->avail_in -= (uInt)in_used; strm->total_in += in_used;
    strm->next_out += out_len; strm->avail_out -= (uInt)out_len; strm->total_out += out_len;
    if (s->inf_wrap) strm->adler = check;
    if (status == Z_STREAM_END) { s->inf_done = 1; return Z_STREAM_END; }
    if (status == Z_NEED_DICT) { s->inf_dict_id = check; strm->adler = check; return Z_NEED_DICT; }
    if (status == Z_DATA_ERROR) { s->inf_bad = 1; strm->msg = (char *)zb200i_inflate_msg(msg); return Z_DATA_ERROR; }
    /* inflate.c:1150-1152: no progress, or Z_FINISH without reaching the end, is a buffer error */
    if ((in_used == 0 && out_len == 0) || flush == Z_FINISH) return Z_BUF_ERROR;
    return Z_OK;
}

ZAPI int inflateSetDictionary(z_streamp strm, const Bytef *dictionary, uInt dictLength)   /* inflate.c:1169-1209 */
{
    zs *s;
    int mode;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    mode = zb200i_inflate_mode(s->inf);
    if (s->inf_wrap != 0 && mode != 8) return Z_STREAM_ERROR;
    if (mode == 8) {
        uLong id = adler32(adler32(0L, Z_NULL, 0), dictionary, dictLength);
        if (id != s->inf_dict_id) return Z_DATA_ERROR;
    }
    s->inf_started = 1;                                         /* so does the dictionary */
    return zb200i_inflate_set_dict(s->inf, dictionary, dictLength) == 0 ? Z_OK : Z_MEM_ERROR;
}

/* inflate.c:1239-1260: scan for the 00 00 FF FF of an empty stored block */
static unsigned syncsearch(unsigned *have, const unsigned char *buf, unsigned len)
{
    unsigned got = *have, next = 0;
    while (next < len && got < 4) {
        if ((int)(buf[next]) == (got < 2 ? 0 : 0xff)) got++;
        else if (buf[next]) got = 0;
        else got = 4 - got;
        next++;
    }
    *have = got;
    return next;
}

ZAPI int inflateSync(z_streamp strm)                            /* inflate.c:1262-1303 */
{
    zs *s;
    unsigned used;
    uLong in, out;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    if (strm->avail_in == 0 && (s->sync_on || zb200i_inflate_pending_input(s->inf) == 0)) return Z_BUF_ERROR;
    if (!s->sync_on) {
        /* the first call searches the bytes the stream already holds (the reference: its bit buffer), then the caller's;
         * later calls go on with the caller's bytes and the part of a marker matched so far */
        size_t pn = zb200i_inflate_pending_input(s->inf);
        s->sync_on = 1; s->sync_have = 0;
        if (pn) {
            unsigned at = syncsearch(&s->sync_have, zb200i_inflate_pending_bytes(s->inf), (unsigned)pn);
            if (s->sync_have == 4) {                            /* the marker lies inside held bytes: decoding resumes right behind it */
                in = strm->total_in; out = strm->total_out;
                if (zb200i_inflate_resync_keep(s->inf, at) != 0) return Z_STREAM_ERROR;
                strm->total_in = in; strm->total_out = out;
                s->inf_bad = 0; s->inf_done = 0; s->sync_on = 0; s->sync_have = 0;
                return Z_OK;
            }
        }
    }
    used = syncsearch(&s->sync_have, strm->next_in, strm->avail_in);
    strm->avail_in -= used; strm->next_in += used; strm->total_in += used;
    if (s->sync_have != 4) return Z_DATA_ERROR;
    in = strm->total_in; out = strm->total_out;
    if (zb200i_inflate_resync(s->inf) != 0) return Z_STREAM_ERROR;
    strm->total_in = in; strm->total_out = out;
    s->inf_bad = 0; s->inf_done = 0; s->sync_on = 0; s->sync_have = 0;
    return Z_OK;
}

ZAPI int inflateSyncPoint(z_streamp strm)                       /* inflate.c:1313-1321 */
{
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE) return Z_STREAM_ERROR;
    return 0;
}

ZAPI int inflateCopy(z_streamp dest, z_streamp source)          /* inflate.c:1323-1368 */
{
    zs *s, *d;
    if (dest == Z_NULL || source == Z_NULL || source->state == Z_NULL || source->state->kind != KIND_INFLATE)
        return Z_STREAM_ERROR;
    s = source->state;
    d = (zs *)source->zalloc(source->opaque, 1, (uInt)sizeof(zs));
    if (d == Z_NULL) return Z_MEM_ERROR;
    memcpy(dest, source, sizeof(z_stream));
    memcpy(d, s, sizeof(zs));
    d->inf = NULL; d->strm = dest;
    if (zb200i_inflate_clone(&d->inf, s->inf) != 0) { source->zfree(source->opaque, d); return Z_MEM_ERROR; }
    dest->state = d;
    return Z_OK;
}

ZAPI int inflatePrime(z_streamp strm, int bits, int value)     /* inflate.c:128-142 */
{
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE) return Z_STREAM_ERROR;
    if (bits > 16 || bits < 0) return Z_STREAM_ERROR;
    strm->state->inf_started = 1;                               /* primed bits live in the streaming decoder */
    return zb200i_inflate_prime(strm->state->inf, bits, value) == 0 ? Z_OK : Z_STREAM_ERROR;
}

ZAPI int inflateGetHeader(z_streamp strm, gz_headerp head)      /* inflate.c:1211-1227 */
{
    zs *s;
    if (strm == Z_NULL || strm->state == Z_NULL || strm->state->kind != KIND_INFLATE) return Z_STREAM_ERROR;
    s = strm->state;
    if ((s->inf_wrap & 2) == 0) return Z_STREAM_ERROR;          /* only for gzip decoding (windowBits + 16 or + 32) */
    s->gz_head = head;
    head->done = 0;
    return Z_OK;
}
