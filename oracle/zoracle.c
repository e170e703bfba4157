/* zoracle.c -- CPU oracle for the zb200 hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of the algorithms of the reference (zlib 1.2.3 inside
 * ChrisHird/ZLIB).  Nothing here is shipped or called by the product library;
 * see zoracle.h for who may load it and how it is pinned (known-answer vectors
 * + differential tests against oracle/_ref/libzref.so, byte-identical for
 * deflate levels 0..9).
 *
 * Reference anchors (paths under /root/reference):
 *   checksums  qcsrc/crc32.c:219-423, qcsrc/adler32.c:57-149
 *   deflate    qcsrc/deflate.c:137-149 (levels), :189 (hash insert), :1027
 *              (longest_match), :1266 (fill_window), :1390/:1448/:1554 (level
 *              drivers); qcsrc/trees.c:490-1120 (code construction, block
 *              choice, bit packing)
 *   inflate    qcsrc/inflate.c:554-1153, qcsrc/inftrees.c:32-329,
 *              qcsrc/inffast.c:67-302, qcsrc/uncompr.c:26-61
 */
#include "zoracle.h"
#include <stdlib.h>
#include <string.h>

#define API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------ */
/* Checksums                                                                 */
/* ------------------------------------------------------------------------ */

#define CRC_POLY 0xEDB88320u        /* reflected CRC-32 polynomial, crc32.c:66-96 */
static uint32_t crc_tab[4][256];
static int crc_ready;

static void crc_setup(void)
{
    if (crc_ready) return;
    for (unsigned n = 0; n < 256; n++) {
        uint32_t c = n;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
        crc_tab[0][n] = c;
    }
    /* slice tables: advance table k-1 by one more zero byte (crc32.c:107-118) */
    for (unsigned n = 0; n < 256; n++)
        for (int k = 1; k < 4; k++) {
            uint32_t c = crc_tab[k - 1][n];
            crc_tab[k][n] = crc_tab[0][c & 0xff] ^ (c >> 8);
        }
    crc_ready = 1;
}

/* crc32.c:219-296: init/final xor 0xffffffff, NULL -> 0, four bytes a step. */
API uint32_t zo_crc32(uint32_t crc, const uint8_t *buf, size_t len)
{
    if (buf == NULL) return 0;
    crc_setup();
    uint32_t c = ~crc;
    while (len && ((uintptr_t)buf & 3)) { c = crc_tab[0][(c ^ *buf++) & 0xff] ^ (c >> 8); len--; }
    while (len >= 4) {
        uint32_t w;
        memcpy(&w, buf, 4);
        c ^= w;                                    /* little-endian host */
        c = crc_tab[3][c & 0xff] ^ crc_tab[2][(c >> 8) & 0xff] ^
            crc_tab[1][(c >> 16) & 0xff] ^ crc_tab[0][c >> 24];
        buf += 4; len -= 4;
    }
    while (len--) c = crc_tab[0][(c ^ *buf++) & 0xff] ^ (c >> 8);
    return ~c;
}

/* a(x)*b(x) mod P in the reflected representation (bit 31 = x^0). */
static uint32_t gf2_mulmod(uint32_t a, uint32_t b)
{
    uint32_t r = 0;
    for (int i = 31; i >= 0; i--) {       /* walk b from x^0 upwards */
        if ((b >> i) & 1) r ^= a;
        a = (a & 1) ? (a >> 1) ^ CRC_POLY : a >> 1;   /* a *= x */
    }
    return r;
}

/* crc32.c:370-423 computes crc1 * x^(8*len2) mod P by squaring a 32x32 GF(2)
 * operator; the same function written as square-and-multiply on polynomials. */
API uint32_t zo_crc32_combine(uint32_t crc1, uint32_t crc2, int64_t len2)
{
    if (len2 <= 0) return crc1;           /* crc32.c:383-385 degenerate case */
    uint32_t p = 0x00800000u;             /* x^8 */
    uint32_t acc = 0x80000000u;           /* x^0 */
    uint64_t n = (uint64_t)len2;
    while (n) {
        if (n & 1) acc = gf2_mulmod(acc, p);
        p = gf2_mulmod(p, p);
        n >>= 1;
    }
    return gf2_mulmod(crc1, acc) ^ crc2;
}

#define ADLER_BASE 65521u
#define ADLER_NMAX 5552u

/* adler32.c:57-125: s1 = 1 + sum b, s2 = sum of s1; NULL -> 1. */
API uint32_t zo_adler32(uint32_t adler, const uint8_t *buf, size_t len)
{
    uint32_t s1 = adler & 0xffff, s2 = (adler >> 16) & 0xffff;
    if (len == 1 && buf != NULL) {        /* reference handles len 1 before the NULL test */
        s1 += buf[0]; if (s1 >= ADLER_BASE) s1 -= ADLER_BASE;
        s2 += s1;     if (s2 >= ADLER_BASE) s2 -= ADLER_BASE;
        return s1 | (s2 << 16);
    }
    if (buf == NULL) return 1;
    do {                                  /* runs once for len 0: non-canonical seeds get reduced */
        size_t n = len < ADLER_NMAX ? len : ADLER_NMAX;   /* deferred modulo window */
        len -= n;
        while (n--) { s1 += *buf++; s2 += s1; }
        s1 %= ADLER_BASE; s2 %= ADLER_BASE;
    } while (len);
    return s1 | (s2 << 16);
}

/* adler32.c:128-149, including its use of '>' (not '>=') in the final folds,
 * which the product must reproduce bit for bit. */
API uint32_t zo_adler32_combine(uint32_t adler1, uint32_t adler2, int64_t len2)
{
    unsigned rem = (unsigned)(len2 % (int64_t)ADLER_BASE);
    unsigned long sum1 = adler1 & 0xffff;
    unsigned long sum2 = ((unsigned long)rem * sum1) % ADLER_BASE;
    sum1 += (adler2 & 0xffff) + ADLER_BASE - 1;
    sum2 += ((adler1 >> 16) & 0xffff) + ((adler2 >> 16) & 0xffff) + ADLER_BASE - rem;
    if (sum1 > ADLER_BASE) sum1 -= ADLER_BASE;
    if (sum1 > ADLER_BASE) sum1 -= ADLER_BASE;
    if (sum2 > (ADLER_BASE << 1)) sum2 -= (ADLER_BASE << 1);
    if (sum2 > ADLER_BASE) sum2 -= ADLER_BASE;
    return (uint32_t)(sum1 | (sum2 << 16));
}

/* compress.c:75-79 */
API size_t zo_compress_bound(size_t n) { return n + (n >> 12) + (n >> 14) + 11; }

/* ------------------------------------------------------------------------ */
/* Shared DEFLATE alphabets (RFC 1951; trees.c:61-71, inftrees.c:60-73)      */
/* ------------------------------------------------------------------------ */

enum { NLIT = 286, NDIST = 30, NBL = 19, EOB = 256, MAXBITS = 15 };
enum { WSIZE = 32768, WMASK = WSIZE - 1, MINM = 3, MAXM = 258,
       MIN_LOOK = MAXM + MINM + 1, MAX_DIST = WSIZE - MIN_LOOK };

static const uint8_t len_extra[29] = {0,0,0,0,0,0,0,0,1,1,1,1,2,2,2,2,3,3,3,3,4,4,4,4,5,5,5,5,0};
static const uint8_t dist_extra[30] = {0,0,0,0,1,1,2,2,3,3,4,4,5,5,6,6,7,7,8,8,9,9,10,10,11,11,12,12,13,13};
static const uint8_t bl_extra[19] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,2,3,7};
static const uint8_t bl_perm[19] = {16,17,18,0,8,7,9,6,10,5,11,4,12,3,13,2,14,1,15};

static uint16_t len_base[29];      /* match length - 3 at which each length code starts */
static uint16_t dist_base[30];     /* distance - 1 at which each distance code starts */
static uint8_t  len_code_of[256];  /* (length-3) -> length code 0..28 */
static uint8_t  dist_code_of[32768];/* (distance-1) -> distance code 0..29 */
static uint16_t fix_lcode[288]; static uint8_t fix_llen[288];
static uint16_t fix_dcode[30];
static int alpha_ready;

static unsigned bitrev(unsigned v, int n)
{
    unsigned r = 0;
    while (n--) { r = (r << 1) | (v & 1); v >>= 1; }
    return r;
}

static void crc_setup(void);
__attribute__((constructor)) static void alpha_setup(void)
{
    crc_setup();
    if (alpha_ready) return;
    unsigned v = 0;
    for (int c = 0; c < 28; c++) {
        len_base[c] = (uint16_t)v;
        for (unsigned k = 0; k < (1u << len_extra[c]); k++) len_code_of[v++] = (uint8_t)c;
    }
    /* length 258 has its own code with no extra bits (trees.c:267-272) */
    len_base[28] = 255; len_code_of[255] = 28;
    v = 0;
    for (int c = 0; c < 30; c++) {
        dist_base[c] = (uint16_t)v;
        for (unsigned k = 0; k < (1u << dist_extra[c]); k++) dist_code_of[v++] = (uint8_t)c;
    }
    /* fixed code, RFC 1951 3.2.6 (trees.c:291-305) */
    for (int s = 0; s < 288; s++) fix_llen[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    unsigned next[10] = {0}, cnt[10] = {0}, code = 0;
    for (int s = 0; s < 288; s++) cnt[fix_llen[s]]++;
    for (int b = 1; b <= 9; b++) { code = (code + cnt[b - 1]) << 1; next[b] = code; }
    for (int s = 0; s < 288; s++) fix_lcode[s] = (uint16_t)bitrev(next[fix_llen[s]]++, fix_llen[s]);
    for (int s = 0; s < 30; s++) fix_dcode[s] = (uint16_t)bitrev((unsigned)s, 5);
    alpha_ready = 1;
}

/* ------------------------------------------------------------------------ */
/* Compressor                                                                */
/* ------------------------------------------------------------------------ */

typedef struct { uint16_t good, lazy, nice, chain; int kind; } level_cfg;   /* deflate.c:137-149 */
static const level_cfg level_tab[10] = {
    {0, 0, 0, 0, 0},      {4, 4, 8, 4, 1},       {4, 5, 16, 8, 1},     {4, 6, 32, 32, 1},
    {4, 4, 16, 16, 2},    {8, 16, 32, 32, 2},    {8, 16, 128, 128, 2}, {8, 32, 128, 256, 2},
    {32, 128, 258, 1024, 2}, {32, 258, 258, 4096, 2}};

enum { SYM_CAP = 16384 };           /* lit_bufsize at memLevel 8 (deflate.c:291) */
enum { TREE_MAX = 2 * NLIT + 1 };   /* heap size, trees.c HEAP_SIZE = 2*L_CODES+1 */

typedef struct {
    uint16_t freq[TREE_MAX];        /* leaf and internal node weights */
    uint16_t up[TREE_MAX];          /* parent link, later reused as nothing */
    uint16_t len[TREE_MAX];
    uint16_t code[NLIT + 2];
    int nsym, max_code, max_len;
    const uint8_t *extra; int extra_base;
    const uint8_t *fixed_len;       /* NULL for the code-length alphabet */
} huff;

typedef struct {
    const level_cfg *cfg; int level, wrap;
    /* sliding window and chains (deflate.c:282-289) */
    uint8_t *win; uint16_t *prev, *head;
    unsigned strstart, look, match_start, match_len, prev_len, prev_match, ins_h;
    int match_avail; long block_start;
    const uint8_t *src; size_t src_left; uint32_t check;
    /* pending symbols of the open block */
    uint8_t *sym_lc; uint16_t *sym_dist; unsigned nsym;
    huff lt, dt, bt;
    unsigned long opt_bits, fix_bits;
    int heap[TREE_MAX], heap_len, heap_max; uint8_t depth[TREE_MAX]; uint16_t bl_count[MAXBITS + 1];
    /* output */
    uint8_t *out; size_t out_pos, out_cap; int overflow;
    uint64_t acc; int acc_n;
} enc;

static void put_byte(enc *e, unsigned b)
{
    if (e->out_pos < e->out_cap) e->out[e->out_pos] = (uint8_t)b; else e->overflow = 1;
    e->out_pos++;
}
static void put_bits(enc *e, unsigned v, int n)   /* LSB first, trees.c:217-229 */
{
    e->acc |= (uint64_t)v << e->acc_n; e->acc_n += n;
    while (e->acc_n >= 8) { put_byte(e, (unsigned)(e->acc & 0xff)); e->acc >>= 8; e->acc_n -= 8; }
}
static void byte_align(enc *e)                    /* trees.c:1178 bi_windup */
{
    if (e->acc_n > 0) put_byte(e, (unsigned)(e->acc & 0xff));
    e->acc = 0; e->acc_n = 0;
}

static void block_reset(enc *e)                   /* trees.c:408-421 */
{
    memset(e->lt.freq, 0, sizeof(uint16_t) * NLIT);
    memset(e->dt.freq, 0, sizeof(uint16_t) * NDIST);
    memset(e->bt.freq, 0, sizeof(uint16_t) * NBL);
    e->lt.freq[EOB] = 1;
    e->opt_bits = e->fix_bits = 0; e->nsym = 0;
}

/* node a sorts before node b: lighter first, ties by shallower subtree (trees.c:445-447) */
static int lighter(const enc *e, const huff *t, int a, int b)
{
    return t->freq[a] < t->freq[b] || (t->freq[a] == t->freq[b] && e->depth[a] <= e->depth[b]);
}
static void sift_down(enc *e, const huff *t, int k)   /* trees.c:455-480 */
{
    int v = e->heap[k];
    for (int j = k << 1; j <= e->heap_len; j <<= 1) {
        if (j < e->heap_len && lighter(e, t, e->heap[j + 1], e->heap[j])) j++;
        if (lighter(e, t, v, e->heap[j])) break;
        e->heap[k] = e->heap[j]; k = j;
    }
    e->heap[k] = v;
}

/* Bit lengths from the parent links, limited to t->max_len with the reference's
 * repair procedure (trees.c:490-567). */
static void assign_lengths(enc *e, huff *t)
{
    int over = 0;
    memset(e->bl_count, 0, sizeof(e->bl_count));
    t->len[e->heap[e->heap_max]] = 0;
    int h;
    for (h = e->heap_max + 1; h < TREE_MAX; h++) {
        int n = e->heap[h];
        int bits = t->len[t->up[n]] + 1;
        if (bits > t->max_len) { bits = t->max_len; over++; }
        t->len[n] = (uint16_t)bits;
        if (n > t->max_code) continue;            /* internal node */
        e->bl_count[bits]++;
        int xb = n >= t->extra_base ? t->extra[n - t->extra_base] : 0;
        e->opt_bits += (unsigned long)t->freq[n] * (unsigned)(bits + xb);
        if (t->fixed_len) e->fix_bits += (unsigned long)t->freq[n] * (unsigned)(t->fixed_len[n] + xb);
    }
    if (!over) return;
    do {
        int bits = t->max_len - 1;
        while (e->bl_count[bits] == 0) bits--;
        e->bl_count[bits]--; e->bl_count[bits + 1] += 2; e->bl_count[t->max_len]--;
        over -= 2;
    } while (over > 0);
    for (int bits = t->max_len; bits != 0; bits--) {
        int n = e->bl_count[bits];
        while (n != 0) {
            int m = e->heap[--h];
            if (m > t->max_code) continue;
            if (t->len[m] != (unsigned)bits) {
                e->opt_bits += (unsigned long)(((long)bits - (long)t->len[m]) * (long)t->freq[m]);
                t->len[m] = (uint16_t)bits;
            }
            n--;
        }
    }
}

static void assign_codes(enc *e, huff *t)          /* trees.c:577-609 */
{
    unsigned next[MAXBITS + 1], code = 0;
    for (int b = 1; b <= MAXBITS; b++) { code = (code + e->bl_count[b - 1]) << 1; next[b] = code; }
    for (int n = 0; n <= t->max_code; n++)
        if (t->len[n]) t->code[n] = (uint16_t)bitrev(next[t->len[n]]++, t->len[n]);
}

static void make_code(enc *e, huff *t)             /* trees.c:619-700 build_tree */
{
    int max_code = -1;
    e->heap_len = 0; e->heap_max = TREE_MAX;
    for (int n = 0; n < t->nsym; n++) {
        if (t->freq[n]) { e->heap[++e->heap_len] = max_code = n; e->depth[n] = 0; }
        else t->len[n] = 0;
    }
    while (e->heap_len < 2) {                      /* force two codes, trees.c:650-656 */
        int n = e->heap[++e->heap_len] = (max_code < 2 ? ++max_code : 0);
        t->freq[n] = 1; e->depth[n] = 0;
        e->opt_bits--; if (t->fixed_len) e->fix_bits -= t->fixed_len[n];
    }
    t->max_code = max_code;
    for (int n = e->heap_len / 2; n >= 1; n--) sift_down(e, t, n);
    int node = t->nsym;
    do {
        int n = e->heap[1];
        e->heap[1] = e->heap[e->heap_len--]; sift_down(e, t, 1);
        int m = e->heap[1];
        e->heap[--e->heap_max] = n; e->heap[--e->heap_max] = m;
        t->freq[node] = (uint16_t)(t->freq[n] + t->freq[m]);
        e->depth[node] = (uint8_t)((e->depth[n] >= e->depth[m] ? e->depth[n] : e->depth[m]) + 1);
        t->up[n] = t->up[m] = (uint16_t)node;
        e->heap[1] = node++; sift_down(e, t, 1);
    } while (e->heap_len >= 2);
    e->heap[--e->heap_max] = e->heap[1];
    assign_lengths(e, t);
    assign_codes(e, t);
}

/* Run-length walk over a code-length array (trees.c:707-797).  emit==0 tallies the
 * code-length alphabet, emit==1 writes it. */
static void walk_lengths(enc *e, huff *t, int max_code, int emit)
{
    int prevlen = -1, nextlen = t->len[0], count = 0, maxc = 7, minc = 4;
    if (nextlen == 0) { maxc = 138; minc = 3; }
    if (!emit) t->len[max_code + 1] = 0xffff;      /* sentinel */
    for (int n = 0; n <= max_code; n++) {
        int cur = nextlen; nextlen = t->len[n + 1];
        if (++count < maxc && cur == nextlen) continue;
        if (count < minc) {
            if (emit) { do put_bits(e, e->bt.code[cur], e->bt.len[cur]); while (--count); }
            else e->bt.freq[cur] = (uint16_t)(e->bt.freq[cur] + count);
        } else if (cur != 0) {
            if (cur != prevlen) {
                if (emit) { put_bits(e, e->bt.code[cur], e->bt.len[cur]); count--; }
                else e->bt.freq[cur]++;
            }
            if (emit) { put_bits(e, e->bt.code[16], e->bt.len[16]); put_bits(e, (unsigned)count - 3, 2); }
            else e->bt.freq[16]++;
        } else if (count <= 10) {
            if (emit) { put_bits(e, e->bt.code[17], e->bt.len[17]); put_bits(e, (unsigned)count - 3, 3); }
            else e->bt.freq[17]++;
        } else {
            if (emit) { put_bits(e, e->bt.code[18], e->bt.len[18]); put_bits(e, (unsigned)count - 11, 7); }
            else e->bt.freq[18]++;
        }
        count = 0; prevlen = cur;
        if (nextlen == 0) { maxc = 138; minc = 3; }
        else if (cur == nextlen) { maxc = 6; minc = 3; }
        else { maxc = 7; minc = 4; }
    }
}

static void write_symbols(enc *e, const uint16_t *lc, const uint16_t *ll_len_u16, const uint8_t *ll_len_u8,
                          const uint16_t *dc, const uint16_t *dl_u16, int dl_fixed)
{   /* trees.c:1072-1120 compress_block */
    for (unsigned i = 0; i < e->nsym; i++) {
        unsigned d = e->sym_dist[i], v = e->sym_lc[i];
        if (d == 0) {
            put_bits(e, lc[v], ll_len_u16 ? ll_len_u16[v] : ll_len_u8[v]);
        } else {
            unsigned c = len_code_of[v], s = c + 257;
            put_bits(e, lc[s], ll_len_u16 ? ll_len_u16[s] : ll_len_u8[s]);
            if (len_extra[c]) put_bits(e, v - len_base[c], len_extra[c]);
            d--; c = dist_code_of[d];
            put_bits(e, dc[c], dl_fixed ? 5 : dl_u16[c]);
            if (dist_extra[c]) put_bits(e, d - dist_base[c], dist_extra[c]);
        }
    }
    put_bits(e, lc[EOB], ll_len_u16 ? ll_len_u16[EOB] : ll_len_u8[EOB]);
}

static void stored_block(enc *e, const uint8_t *buf, unsigned long n, int last)  /* trees.c:867-879 */
{
    put_bits(e, (unsigned)last, 3);
    byte_align(e);
    put_byte(e, n & 0xff); put_byte(e, (n >> 8) & 0xff);
    put_byte(e, ~n & 0xff); put_byte(e, (~n >> 8) & 0xff);
    for (unsigned long i = 0; i < n; i++) put_byte(e, buf[i]);
}

/* Close the open block: choose stored / fixed / dynamic (trees.c:921-1016). */
static void close_block(enc *e, int last)
{
    const uint8_t *buf = e->block_start >= 0 ? e->win + e->block_start : NULL;
    unsigned long raw = (unsigned long)((long)e->strstart - e->block_start);
    unsigned long optb, fixb; int max_bl = 0;
    if (e->level > 0) {
        make_code(e, &e->lt);
        make_code(e, &e->dt);
        walk_lengths(e, &e->lt, e->lt.max_code, 0);
        walk_lengths(e, &e->dt, e->dt.max_code, 0);
        make_code(e, &e->bt);
        for (max_bl = NBL - 1; max_bl >= 3; max_bl--) if (e->bt.len[bl_perm[max_bl]]) break;
        e->opt_bits += 3 * ((unsigned long)max_bl + 1) + 5 + 5 + 4;
        optb = (e->opt_bits + 3 + 7) >> 3; fixb = (e->fix_bits + 3 + 7) >> 3;
        if (fixb <= optb) optb = fixb;
    } else {
        optb = fixb = raw + 5;
    }
    if (raw + 4 <= optb && buf != NULL) {
        stored_block(e, buf, raw, last);
    } else if (fixb == optb) {
        put_bits(e, 2u + (unsigned)last, 3);
        write_symbols(e, fix_lcode, NULL, fix_llen, fix_dcode, NULL, 1);
    } else {
        put_bits(e, 4u + (unsigned)last, 3);
        put_bits(e, (unsigned)e->lt.max_code + 1 - 257, 5);
        put_bits(e, (unsigned)e->dt.max_code + 1 - 1, 5);
        put_bits(e, (unsigned)max_bl + 1 - 4, 4);
        for (int r = 0; r <= max_bl; r++) put_bits(e, e->bt.len[bl_perm[r]], 3);
        walk_lengths(e, &e->lt, e->lt.max_code, 1);
        walk_lengths(e, &e->dt, e->dt.max_code, 1);
        write_symbols(e, e->lt.code, e->lt.len, NULL, e->dt.code, e->dt.len, 0);
    }
    block_reset(e);
    if (last) byte_align(e);
    e->block_start = (long)e->strstart;
}

static int tally(enc *e, unsigned dist, unsigned lc)   /* deflate.h:308-324, trees.c:1022 */
{
    e->sym_dist[e->nsym] = (uint16_t)dist; e->sym_lc[e->nsym++] = (uint8_t)lc;
    if (dist == 0) e->lt.freq[lc]++;
    else { e->lt.freq[len_code_of[lc] + 257]++; e->dt.freq[dist_code_of[dist - 1]]++; }
    return e->nsym == SYM_CAP - 1;
}

#define HASH_STEP(h, c) ((((h) << 5) ^ (c)) & 0x7fff)     /* deflate.c:170, 15-bit hash, shift 5 */

static unsigned chain_in(enc *e, unsigned pos)          /* deflate.c:189-192 INSERT_STRING */
{
    e->ins_h = HASH_STEP(e->ins_h, e->win[pos + 2]);
    unsigned old = e->prev[pos & WMASK] = e->head[e->ins_h];
    e->head[e->ins_h] = (uint16_t)pos;
    return old;
}

static void refill(enc *e)                               /* deflate.c:1266-1358 fill_window */
{
    do {
        unsigned more = 2u * WSIZE - e->look - e->strstart;
        if (e->strstart >= (unsigned)WSIZE + MAX_DIST) {
            memcpy(e->win, e->win + WSIZE, WSIZE);
            e->match_start -= WSIZE; e->strstart -= WSIZE; e->block_start -= WSIZE;
            for (unsigned i = 0; i < 32768; i++) e->head[i] = (uint16_t)(e->head[i] >= WSIZE ? e->head[i] - WSIZE : 0);
            for (unsigned i = 0; i < WSIZE; i++) e->prev[i] = (uint16_t)(e->prev[i] >= WSIZE ? e->prev[i] - WSIZE : 0);
            more += WSIZE;
        }
        if (e->src_left == 0) return;
        size_t n = e->src_left < more ? e->src_left : more;   /* deflate.c:956 read_buf */
        if (e->wrap == 1) e->check = zo_adler32(e->check, e->src, n);
        else if (e->wrap == 2) e->check = zo_crc32(e->check, e->src, n);
        memcpy(e->win + e->strstart + e->look, e->src, n);
        e->src += n; e->src_left -= n; e->look += (unsigned)n;
        if (e->look >= MINM) {
            e->ins_h = e->win[e->strstart];
            e->ins_h = HASH_STEP(e->ins_h, e->win[e->strstart + 1]);
        }
    } while (e->look < MIN_LOOK && e->src_left != 0);
}

/* deflate.c:1027-1168: walk the chain from `cand`, return the best length (> prev_len
 * or prev_len itself), never beyond the lookahead. */
static unsigned best_match(enc *e, unsigned cand)
{
    unsigned chain = e->cfg->chain, nice = e->cfg->nice;
    const uint8_t *scan = e->win + e->strstart;
    int best = (int)e->prev_len;
    unsigned limit = e->strstart > (unsigned)MAX_DIST ? e->strstart - MAX_DIST : 0;
    unsigned room = e->look < MAXM ? e->look : MAXM;   /* comparable bytes */
    if (e->prev_len >= e->cfg->good) chain >>= 2;
    if (nice > e->look) nice = e->look;
    do {
        const uint8_t *m = e->win + cand;
        /* quick rejects, deflate.c:1121-1124; bytes past the input never decide the result */
        if (m[best] != scan[best] || m[best - 1] != scan[best - 1] || m[0] != scan[0] || m[1] != scan[1])
            continue;
        unsigned len = 3;                         /* byte 2 is implied equal by the hash (deflate.c:1126-1131) */
        while (len < room && m[len] == scan[len]) len++;
        if ((int)len > best) {
            e->match_start = cand; best = (int)len;
            if (len >= nice) break;
        }
    } while ((cand = e->prev[cand & WMASK]) > limit && --chain != 0);
    return (unsigned)best <= e->look ? (unsigned)best : e->look;
}

static void run_stored(enc *e)                           /* deflate.c:1390-1439, flush = Z_FINISH */
{
    unsigned long max_block = 0xffff;
    if (max_block > 4ul * SYM_CAP - 5) max_block = 4ul * SYM_CAP - 5;
    for (;;) {
        if (e->look <= 1) { refill(e); if (e->look == 0) break; }
        e->strstart += e->look; e->look = 0;
        unsigned long max_start = (unsigned long)e->block_start + max_block;
        if (e->strstart == 0 || e->strstart >= max_start) {
            e->look = (unsigned)(e->strstart - max_start); e->strstart = (unsigned)max_start;
            close_block(e, 0);
        }
        if (e->strstart - (unsigned)e->block_start >= (unsigned)MAX_DIST) close_block(e, 0);
    }
    close_block(e, 1);
}

static void run_greedy(enc *e)                           /* deflate.c:1448-1546 deflate_fast */
{
    for (;;) {
        /* The reference keeps a stale chain head when fewer than 3 bytes remain; the
         * search it then runs cannot return >= 3, so starting from "none" is the same. */
        unsigned head = 0;
        if (e->look < MIN_LOOK) { refill(e); if (e->look == 0) break; }
        if (e->look >= MINM) head = chain_in(e, e->strstart);
        if (head != 0 && e->strstart - head <= (unsigned)MAX_DIST) e->match_len = best_match(e, head);
        int full;
        if (e->match_len >= MINM) {
            full = tally(e, e->strstart - e->match_start, e->match_len - MINM);
            e->look -= e->match_len;
            if (e->match_len <= e->cfg->lazy && e->look >= MINM) {   /* max_insert_length */
                e->match_len--;
                do { e->strstart++; chain_in(e, e->strstart); } while (--e->match_len != 0);
                e->strstart++;
            } else {
                e->strstart += e->match_len; e->match_len = 0;
                e->ins_h = e->win[e->strstart];
                e->ins_h = HASH_STEP(e->ins_h, e->win[e->strstart + 1]);
            }
        } else {
            full = tally(e, 0, e->win[e->strstart]);
            e->look--; e->strstart++;
        }
        if (full) close_block(e, 0);
    }
    close_block(e, 1);
}

static void run_lazy(enc *e)                             /* deflate.c:1554-1674 deflate_slow */
{
    for (;;) {
        unsigned head = 0;
        if (e->look < MIN_LOOK) { refill(e); if (e->look == 0) break; }
        if (e->look >= MINM) head = chain_in(e, e->strstart);
        e->prev_len = e->match_len; e->prev_match = e->match_start;
        e->match_len = MINM - 1;
        if (head != 0 && e->prev_len < e->cfg->lazy && e->strstart - head <= (unsigned)MAX_DIST) {
            e->match_len = best_match(e, head);
            if (e->match_len == MINM && e->strstart - e->match_start > 4096)   /* TOO_FAR */
                e->match_len = MINM - 1;
        }
        if (e->prev_len >= MINM && e->match_len <= e->prev_len) {
            unsigned max_insert = e->strstart + e->look - MINM;
            int full = tally(e, e->strstart - 1 - e->prev_match, e->prev_len - MINM);
            e->look -= e->prev_len - 1; e->prev_len -= 2;
            do { if (++e->strstart <= max_insert) chain_in(e, e->strstart); } while (--e->prev_len != 0);
            e->match_avail = 0; e->match_len = MINM - 1; e->strstart++;
            if (full) close_block(e, 0);
        } else if (e->match_avail) {
            if (tally(e, 0, e->win[e->strstart - 1])) close_block(e, 0);
            e->strstart++; e->look--;
        } else {
            e->match_avail = 1; e->strstart++; e->look--;
        }
    }
    if (e->match_avail) { tally(e, 0, e->win[e->strstart - 1]); e->match_avail = 0; }
    close_block(e, 1);
}

API int zo_deflate(const uint8_t *in, size_t n, uint8_t *out, size_t cap,
                   size_t *out_len, int level, int wrap)
{
    if (level == -1) level = 6;
    if (level < 0 || level > 9 || wrap < 0 || wrap > 2 || (n && !in) || !out || !out_len)
        return ZO_STREAM_ERROR;
    alpha_setup();
    enc *e = (enc *)calloc(1, sizeof(enc));
    if (!e) return ZO_MEM_ERROR;
    e->win = (uint8_t *)calloc(2 * WSIZE + MIN_LOOK, 1);   /* guard bytes read as zero */
    e->prev = (uint16_t *)calloc(WSIZE, 2);
    e->head = (uint16_t *)calloc(32768, 2);
    e->sym_lc = (uint8_t *)malloc(SYM_CAP); e->sym_dist = (uint16_t *)malloc(SYM_CAP * 2);
    if (!e->win || !e->prev || !e->head || !e->sym_lc || !e->sym_dist) {
        free(e->win); free(e->prev); free(e->head); free(e->sym_lc); free(e->sym_dist); free(e);
        return ZO_MEM_ERROR;
    }
    e->cfg = &level_tab[level]; e->level = level; e->wrap = wrap;
    e->src = in; e->src_left = n; e->out = out; e->out_cap = cap;
    e->match_len = e->prev_len = MINM - 1;
    e->lt.nsym = NLIT; e->lt.max_len = 15; e->lt.extra = len_extra; e->lt.extra_base = 257; e->lt.fixed_len = fix_llen;
    static const uint8_t five[30] = {5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5,5};
    e->dt.nsym = NDIST; e->dt.max_len = 15; e->dt.extra = dist_extra; e->dt.extra_base = 0; e->dt.fixed_len = five;
    e->bt.nsym = NBL; e->bt.max_len = 7; e->bt.extra = bl_extra; e->bt.extra_base = 0; e->bt.fixed_len = NULL;
    block_reset(e);

    if (wrap == 1) {                                  /* deflate.c:625-649 */
        unsigned flevel = level < 2 ? 0 : level < 6 ? 1 : level == 6 ? 2 : 3;
        unsigned hdr = (0x78u << 8) | (flevel << 6);
        hdr += 31 - hdr % 31;
        put_byte(e, hdr >> 8); put_byte(e, hdr & 0xff);
        e->check = 1;
    } else if (wrap == 2) {                           /* deflate.c:579-597 */
        static const uint8_t fixed_head[8] = {31, 139, 8, 0, 0, 0, 0, 0};
        for (int i = 0; i < 8; i++) put_byte(e, fixed_head[i]);
        put_byte(e, level == 9 ? 2 : level < 2 ? 4 : 0);
        put_byte(e, 3);                               /* OS_CODE 3 = unix (zutil.h) */
        e->check = 0;
    }
    if (e->cfg->kind == 0) run_stored(e); else if (e->cfg->kind == 1) run_greedy(e); else run_lazy(e);
    if (wrap == 1) {
        put_byte(e, e->check >> 24); put_byte(e, (e->check >> 16) & 0xff);
        put_byte(e, (e->check >> 8) & 0xff); put_byte(e, e->check & 0xff);
    } else if (wrap == 2) {
        for (int i = 0; i < 4; i++) put_byte(e, (e->check >> (8 * i)) & 0xff);
        for (int i = 0; i < 4; i++) put_byte(e, (unsigned)((n >> (8 * i)) & 0xff));
    }
    *out_len = e->out_pos;
    int rc = e->overflow ? ZO_BUF_ERROR : ZO_OK;
    free(e->win); free(e->prev); free(e->head); free(e->sym_lc); free(e->sym_dist); free(e);
    return rc;
}

/* ------------------------------------------------------------------------ */
/* Decompressor                                                              */
/* ------------------------------------------------------------------------ */

static __thread const char *last_msg;
static __thread size_t last_max_dist;
API const char *zo_last_msg(void) { return last_msg; }
API size_t zo_last_max_dist(void) { return last_max_dist; }

typedef struct {
    const uint8_t *in; size_t in_len; uint64_t bitpos;   /* next unread bit */
    uint8_t *out; size_t out_cap, out_pos;
    int short_in, short_out;
} dec;

/* canonical decoder tables: count per length + symbols sorted by (length, symbol) */
typedef struct { uint16_t count[MAXBITS + 1]; uint16_t sym[288]; int nsyms_coded; int maxlen; } dcode;

static int need(dec *d, unsigned n)      /* are n more bits present? */
{
    if (d->bitpos + n > (uint64_t)d->in_len * 8) { d->short_in = 1; return 0; }
    return 1;
}
static unsigned peek1(const dec *d, uint64_t pos) { return (d->in[pos >> 3] >> (pos & 7)) & 1u; }
static unsigned take(dec *d, unsigned n)
{
    unsigned v = 0;
    for (unsigned i = 0; i < n; i++) v |= peek1(d, d->bitpos + i) << i;
    d->bitpos += n;
    return v;
}

/* inftrees.c:107-138: validity rules.  kind 0 = code lengths, 1 = lit/len, 2 = dist. */
static int dcode_build(dcode *c, const uint16_t *lens, int n, int kind)
{
    memset(c->count, 0, sizeof(c->count));
    for (int i = 0; i < n; i++) c->count[lens[i]]++;
    int maxlen = MAXBITS;
    while (maxlen >= 1 && c->count[maxlen] == 0) maxlen--;
    c->maxlen = maxlen; c->nsyms_coded = n - c->count[0];
    if (maxlen == 0) return 0;                      /* no codes: error only when used */
    int left = 1;
    for (int len = 1; len <= MAXBITS; len++) {
        left = (left << 1) - c->count[len];
        if (left < 0) return -1;                    /* over-subscribed */
    }
    if (left > 0 && (kind == 0 || maxlen != 1)) return -1;   /* incomplete */
    uint16_t offs[MAXBITS + 2]; offs[1] = 0;
    for (int len = 1; len <= MAXBITS; len++) offs[len + 1] = (uint16_t)(offs[len] + c->count[len]);
    for (int i = 0; i < n; i++) if (lens[i]) c->sym[offs[lens[i]]++] = (uint16_t)i;
    return 0;
}

/* Decode one symbol.  Returns -1 when input runs out, -2 for a bit pattern that is
 * not a code (possible only in an incomplete/empty code).  An empty code-length
 * code yields symbol 0 and uses one bit, as the reference's marker table does
 * (inftrees.c:116-124 feeding inflate.c:880-886). */
static int dcode_next(dec *d, const dcode *c, int kind)
{
    if (c->maxlen == 0) {
        if (kind == 0) { if (!need(d, 1)) return -1; d->bitpos++; return 0; }
        if (!need(d, 1)) return -1;
        return -2;
    }
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= c->maxlen; len++) {
        if (!need(d, (unsigned)len)) return -1;
        code |= (int)peek1(d, d->bitpos + (unsigned)len - 1);
        int cnt = c->count[len];
        if (code - cnt < first) { d->bitpos += (unsigned)len; return c->sym[index + (code - first)]; }
        index += cnt; first += cnt; first <<= 1; code <<= 1;
    }
    return -2;
}

static const uint16_t d_len_base[31] = {3,4,5,6,7,8,9,10,11,13,15,17,19,23,27,31,35,43,51,59,67,83,99,115,131,163,195,227,258,0,0};
static const uint16_t d_dist_base[30] = {1,2,3,4,5,7,9,13,17,25,33,49,65,97,129,193,257,385,513,769,1025,1537,2049,3073,4097,6145,8193,12289,16385,24577};

#define FAIL(m) do { last_msg = (m); return ZO_DATA_ERROR; } while (0)

static int inflate_codes(dec *d, const dcode *lc, const dcode *dc)    /* inflate.c:951-1076 / inffast.c */
{
    for (;;) {
        int s = dcode_next(d, lc, 1);
        if (s == -1) return 1;
        if (s == -2 || s > 285) FAIL("invalid literal/length code");
        if (s < 256) {
            if (d->out_pos >= d->out_cap) { d->short_out = 1; return 1; }
            d->out[d->out_pos++] = (uint8_t)s;
            continue;
        }
        if (s == EOB) return 0;
        s -= 257;
        if (!need(d, len_extra[s])) return 1;
        unsigned len = d_len_base[s] + take(d, len_extra[s]);
        int t = dcode_next(d, dc, 2);
        if (t == -1) return 1;
        if (t == -2 || t > 29) FAIL("invalid distance code");
        if (!need(d, dist_extra[t])) return 1;
        unsigned dist = d_dist_base[t] + take(d, dist_extra[t]);
        if (dist > d->out_pos) FAIL("invalid distance too far back");
        if (dist > last_max_dist) last_max_dist = dist;
        for (unsigned i = 0; i < len; i++) {
            if (d->out_pos >= d->out_cap) { d->short_out = 1; return 1; }
            d->out[d->out_pos] = d->out[d->out_pos - dist]; d->out_pos++;
        }
    }
}

static int inflate_raw(dec *d)
{
    static dcode fix_l, fix_d; static int fix_ready;
    alpha_setup();
    if (!fix_ready) {
        uint16_t l[288]; for (int i = 0; i < 288; i++) l[i] = fix_llen[i];
        dcode_build(&fix_l, l, 288, 1);
        for (int i = 0; i < 30; i++) l[i] = 5;
        /* the fixed distance code has 32 five-bit entries; 30 and 31 are invalid (inffixed.h) */
        l[30] = l[31] = 5; dcode_build(&fix_d, l, 32, 2);
        fix_ready = 1;
    }
    int last;
    do {
        if (!need(d, 3)) return 1;
        last = (int)take(d, 1);
        unsigned type = take(d, 2);
        if (type == 0) {                              /* inflate.c:807-836 */
            d->bitpos = (d->bitpos + 7) & ~7ull;
            if (!need(d, 32)) return 1;
            unsigned len = take(d, 16), nlen = take(d, 16);
            if (len != (nlen ^ 0xffff)) FAIL("invalid stored block lengths");
            for (unsigned i = 0; i < len; i++) {
                if (!need(d, 8)) return 1;
                if (d->out_pos >= d->out_cap) { d->short_out = 1; return 1; }
                d->out[d->out_pos++] = d->in[d->bitpos >> 3]; d->bitpos += 8;
            }
        } else if (type == 1) {
            int r = inflate_codes(d, &fix_l, &fix_d);
            if (r) return r;
        } else if (type == 2) {                       /* inflate.c:837-949 */
            if (!need(d, 14)) return 1;
            unsigned nlen = take(d, 5) + 257, ndist = take(d, 5) + 1, ncode = take(d, 4) + 4;
            if (nlen > 286 || ndist > 30) FAIL("too many length or distance symbols");
            uint16_t lens[320]; memset(lens, 0, sizeof(lens));
            uint16_t cl[19]; memset(cl, 0, sizeof(cl));
            for (unsigned i = 0; i < ncode; i++) { if (!need(d, 3)) return 1; cl[bl_perm[i]] = (uint16_t)take(d, 3); }
            dcode clc, lc, dc;
            if (dcode_build(&clc, cl, 19, 0)) FAIL("invalid code lengths set");
            unsigned have = 0;
            while (have < nlen + ndist) {
                int s = dcode_next(d, &clc, 0);
                if (s == -1) return 1;
                if (s < 16) { lens[have++] = (uint16_t)s; continue; }
                unsigned rep, val = 0;
                if (s == 16) {
                    if (!need(d, 2)) return 1;
                    if (have == 0) FAIL("invalid bit length repeat");
                    val = lens[have - 1]; rep = 3 + take(d, 2);
                } else if (s == 17) { if (!need(d, 3)) return 1; rep = 3 + take(d, 3); }
                else { if (!need(d, 7)) return 1; rep = 11 + take(d, 7); }
                if (have + rep > nlen + ndist) FAIL("invalid bit length repeat");
                while (rep--) lens[have++] = (uint16_t)val;
            }
            if (dcode_build(&lc, lens, (int)nlen, 1)) FAIL("invalid literal/lengths set");
            if (dcode_build(&dc, lens + nlen, (int)ndist, 2)) FAIL("invalid distances set");
            int r = inflate_codes(d, &lc, &dc);
            if (r) return r;
        } else FAIL("invalid block type");
    } while (!last);
    d->bitpos = (d->bitpos + 7) & ~7ull;
    return 0;
}

API int zo_inflate(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap,
                   size_t *out_len, size_t *in_used, int wrap)
{
    dec d; memset(&d, 0, sizeof(d));
    d.in = in; d.in_len = in_len; d.out = out; d.out_cap = out_cap;
    last_msg = NULL;
    last_max_dist = 0;
    int rc = 1;
    crc_setup();
    if (out_len) *out_len = 0;
    if (in_used) *in_used = 0;
    if (wrap == 1) {                                  /* inflate.c:589-632 */
        if (!need(&d, 16)) goto shortfall;
        unsigned cmf = take(&d, 8), flg = take(&d, 8);
        if (((cmf << 8) + flg) % 31) { last_msg = "incorrect header check"; return ZO_DATA_ERROR; }
        if ((cmf & 15) != 8) { last_msg = "unknown compression method"; return ZO_DATA_ERROR; }
        if ((cmf >> 4) + 8 > 15) { last_msg = "invalid window size"; return ZO_DATA_ERROR; }
        if (flg & 0x20) return ZO_DATA_ERROR;         /* Z_NEED_DICT -> uncompr.c:53 */
    } else if (wrap == 2) {                           /* inflate.c:596-602, 634-759 */
        if (!need(&d, 80)) goto shortfall;
        unsigned id = take(&d, 16);
        if (id != 0x8b1f) { last_msg = "incorrect header check"; return ZO_DATA_ERROR; }
        if (take(&d, 8) != 8) { last_msg = "unknown compression method"; return ZO_DATA_ERROR; }
        unsigned flags = take(&d, 8);
        if (flags & 0xe0) { last_msg = "unknown header flags set"; return ZO_DATA_ERROR; }
        take(&d, 32); take(&d, 16);                   /* mtime, xfl, os */
        if (flags & 4) {
            if (!need(&d, 16)) goto shortfall;
            unsigned xl = take(&d, 16);
            if (!need(&d, 8 * xl)) goto shortfall;
            d.bitpos += 8ull * xl;
        }
        for (unsigned f = 8; f <= 16; f <<= 1)
            if (flags & f) for (;;) { if (!need(&d, 8)) goto shortfall; if (take(&d, 8) == 0) break; }
        if (flags & 2) {
            if (!need(&d, 16)) goto shortfall;
            unsigned hc = zo_crc32(0, in, (size_t)(d.bitpos >> 3)) & 0xffff;
            if (take(&d, 16) != hc) { last_msg = "header crc mismatch"; return ZO_DATA_ERROR; }
        }
    }
    rc = inflate_raw(&d);
    if (out_len) *out_len = d.out_pos;
    if (rc < 0) return rc;
    if (rc == 0 && wrap == 1) {                       /* inflate.c:1077-1098 */
        if (!need(&d, 32)) goto shortfall;
        uint32_t want = 0; for (int i = 0; i < 4; i++) want = (want << 8) | take(&d, 8);
        if (want != zo_adler32(1, out, d.out_pos)) { last_msg = "incorrect data check"; return ZO_DATA_ERROR; }
    } else if (rc == 0 && wrap == 2) {                /* inflate.c:1077-1112 */
        if (!need(&d, 32)) goto shortfall;
        uint32_t want = take(&d, 16); want |= take(&d, 16) << 16;
        if (want != zo_crc32(0, out, d.out_pos)) { last_msg = "incorrect data check"; return ZO_DATA_ERROR; }
        if (!need(&d, 32)) goto shortfall;
        uint32_t isz = take(&d, 16); isz |= take(&d, 16) << 16;
        if (isz != (uint32_t)d.out_pos) { last_msg = "incorrect length check"; return ZO_DATA_ERROR; }
    }
    if (rc == 0) { if (in_used) *in_used = (size_t)(d.bitpos >> 3); return ZO_OK; }
shortfall:
    if (out_len) *out_len = d.out_pos;
    /* uncompr.c:53-55: running out of input is a data error, running out of room
     * with input left over is a buffer error. */
    if (d.short_out && ((d.bitpos + 7) >> 3) < d.in_len) return ZO_BUF_ERROR;
    return ZO_DATA_ERROR;
}
