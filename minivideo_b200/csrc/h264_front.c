/*
 * h264_front.c -- host front end: Annex-B / SPS / PPS / slice header / CAVLC -> mvgpu.h SoA.
 * See include/mvfront.h for the interface and the reference functions it stands in for.
 * Written from ITU-T H.264 (clauses 7.3, 7.4, 8.3.1.1, 8.3.2.1, 9.1, 9.2); comments name the
 * reference lines whose observable behaviour matters for drop-in parity.
 */
#define _GNU_SOURCE
#include "mvfront.h"

#include <limits.h>
#include <math.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include "h264_cavlc_tables.h"

/* ------------------------------------------------------------------------ */
/* CAVLC decode look-up tables, built once from the (length, code) tables     */

static uint16_t lut_ct[3][1 << 16];      /* len<<7 | TotalCoeff<<2 | TrailingOnes, indexed by next 16 bits */
static uint16_t lut_ct10[3][1 << 10];    /* the codes of up to 10 bits (almost all that occur) in 2 KB: stays in L1;
                                            0 = longer code, use lut_ct                                     */
static uint16_t lut_ctc[1 << 8];         /* chroma DC coeff_token, next 8 bits                             */
static uint8_t  lut_tz4[15][1 << 9];     /* len<<4 | total_zeros, next 9 bits                              */
static uint8_t  lut_tz2[3][1 << 3];
static uint8_t  lut_run3[7][8];          /* run_before for zerosLeft 0..6 (Table 9-10): codes of at most 3 bits,
                                            len<<4 | run, next 3 bits; row 0 = nothing left to place (no bits, run 0);
                                            entries no code leads to say run 15, which no zerosLeft allows;
                                            zerosLeft > 6 is decoded arithmetically                             */
static uint8_t  cbp_from_codenum[48];
static uint8_t  zz4[16], zz8[64];
static pthread_once_t lut_once = PTHREAD_ONCE_INIT;

static void fill16(uint16_t *lut, int bits, int len, unsigned code, uint16_t val)
{
    if (!len) return;
    unsigned lo = code << (bits - len), n = 1u << (bits - len);
    for (unsigned i = 0; i < n; i++) lut[lo + i] = val;
}
static void fill8s(uint8_t *lut, int bits, const char *str, int sym)
{
    int len = (int)strlen(str);
    unsigned code = 0;
    for (int i = 0; i < len; i++) code = (code << 1) | (unsigned)(str[i] == '1');
    unsigned lo = code << (bits - len), n = 1u << (bits - len);
    for (unsigned i = 0; i < n; i++) lut[lo + i] = (uint8_t)(len << 4 | sym);
}
static void pack_choose(void);
static void zigzag_build(int n, uint8_t *zz)
{
    int r = 0, c = 0, up = 1;
    for (int k = 0; k < n * n; k++) {
        zz[k] = (uint8_t)(r * n + c);
        if (up) { if (c == n - 1) { r++; up = 0; } else if (r == 0) { c++; up = 0; } else { r--; c++; } }
        else    { if (r == n - 1) { c++; up = 1; } else if (c == 0) { r++; up = 1; } else { r++; c--; } }
    }
}
static void build_luts(void)
{
    for (int t = 0; t < 3; t++)
        for (int t1 = 0; t1 < 4; t1++)
            for (int tc = t1; tc <= 16; tc++)
            {
                fill16(lut_ct[t], 16, ct_len[t][t1][tc], ct_code[t][t1][tc], (uint16_t)(ct_len[t][t1][tc] << 7 | tc << 2 | t1));
                if (ct_len[t][t1][tc] <= 10)
                    fill16(lut_ct10[t], 10, ct_len[t][t1][tc], ct_code[t][t1][tc], (uint16_t)(ct_len[t][t1][tc] << 7 | tc << 2 | t1));
            }
    for (int t1 = 0; t1 < 4; t1++)
        for (int tc = t1; tc <= 4; tc++)
            fill16(lut_ctc, 8, ctc_len[t1][tc], ctc_code[t1][tc], (uint16_t)(ctc_len[t1][tc] << 7 | tc << 2 | t1));
    for (int tc = 1; tc <= 15; tc++)
        for (int tz = 0; tz <= 16 - tc; tz++) fill8s(lut_tz4[tc - 1], 9, tz4x4[tc - 1][tz], tz);
    for (int tc = 1; tc <= 3; tc++)
        for (int tz = 0; tz <= 4 - tc; tz++) fill8s(lut_tz2[tc - 1], 3, tz2x2[tc - 1][tz], tz);
    for (int zl = 1; zl <= 6; zl++) {
        memset(lut_run3[zl], 0x1f, 8);
        for (int run = 0; run <= zl; run++) fill8s(lut_run3[zl], 3, runb[zl - 1][run], run);
    }
    for (int k = 0; k < 48; k++) cbp_from_codenum[k] = cbp_intra_by_codenum[k];
    zigzag_build(4, zz4); zigzag_build(8, zz8);
    pack_choose();
}

/* ------------------------------------------------------------------------ */
/* bit reader over an unescaped RBSP (8 zero bytes of padding behind it)      */

typedef struct { const uint8_t *p; size_t pos, nbits; uint64_t win; size_t wbit; } br_t;
#define BR_INIT(ptr, nbits) { (ptr), 0, (nbits), 0, (size_t)-4096 }

/* at least 32 valid bits starting at the read position, left-aligned in 64.  The 8 bytes last loaded are kept:
 * a reload (one unaligned load and a byte swap) is needed only every four bytes or so */
static inline uint64_t br_window(const br_t *bc)
{
    br_t *b = (br_t *)bc;
    size_t off = b->pos - b->wbit;
    if (off > 32) {
        uint64_t w;
        memcpy(&w, b->p + (b->pos >> 3), 8);
        b->win = __builtin_bswap64(w);
        b->wbit = b->pos & ~(size_t)7;
        off = b->pos & 7;
    }
    return b->win << off;
}
static inline uint32_t br_peek(const br_t *b, int n)      /* 1 <= n <= 32 */
{
    return (uint32_t)(br_window(b) >> (64 - n));
}
static inline void br_skip(br_t *b, int n) { b->pos += (size_t)n; }
static inline uint32_t br_get(br_t *b, int n)
{
    if (n == 0) return 0;
    const uint32_t v = br_peek(b, n);
    b->pos += (size_t)n;
    return v;
}
static inline int br_bit(br_t *b) { return (int)br_get(b, 1); }
/* number of leading zero bits at the read position, capped at 32 */
static inline int br_zeros(const br_t *b)
{
    const uint32_t w = (uint32_t)(br_window(b) >> 32);
    return w ? __builtin_clz(w) : 32;
}
static uint32_t br_ue(br_t *b)
{
    const int z = br_zeros(b);
    if (z >= 32) { b->pos += 33; return 0xffffffffu; }
    b->pos += (size_t)z + 1;
    if (z == 0) return 0;
    return (1u << z) - 1 + br_get(b, z);
}
static int br_se(br_t *b)
{
    uint32_t k = br_ue(b);
    return (k & 1) ? (int)((k + 1) >> 1) : -(int)(k >> 1);
}
static inline int br_overrun(const br_t *b) { return b->pos > b->nbits; }

/* ------------------------------------------------------------------------ */

/* off: NAL header byte.  sample: the size mvf_select_idr() gives the picture of an IDR NAL -- the distance to the
 * next NAL header in an Annex-B stream (esparser.c:91,:130), the stsz size of the sample that holds it in an MP4 */
typedef struct { size_t off, size, sample; int type; } nal_t;

typedef struct {
    int valid, id, err_code, profile_idc, level_idc, chroma_format_idc;
    int log2_max_frame_num, poc_type, log2_max_poc_lsb, delta_pic_order_always_zero;
    int width_mbs, height_mbs, frame_mbs_only;
    int crop[4];
    uint8_t list4[6][16], list8[2][64];                     /* zig-zag order */
} sps_t;

typedef struct {
    int valid, id, sps_id, err_code, entropy_cabac, bottom_field_poc_present, init_qp, cb_off, cr_off;
    int deblocking_control, constrained_intra, redundant_pic_cnt, transform8x8, has_extension;
} pps_t;

/* A "parameter generation": the SPS + PPS pair in force for a run of IDR pictures.  The reference decodes every
 * SPS / PPS NAL where it meets it (h264.c:128-150) and each slice looks its PPS up by pic_parameter_set_id and
 * the SPS through it (h264_slice.c:168-169), so later pictures use later tables, offsets, QPs and even geometry.
 * mvf_open_annexb() replays that in stream order and gives every IDR picture the index of its generation. */
typedef struct { sps_t sps; pps_t pps; } paramgen_t;

#define MVF_MAX_SPS 32
#define MVF_MAX_PPS 256

struct mvf_stream {
    const uint8_t *data; size_t len;
    uint8_t *own;                                           /* data when the stream holds a copy (transport streams) */
    nal_t *nals; int n_nals;
    int *idr; int n_idr;                                    /* indices into nals[] */
    int *idr_gen;                                           /* per IDR picture: its generation, or -1 (no usable SPS/PPS) */
    paramgen_t *gens; int n_gens, cap_gens;
    int max_mbs;                                            /* largest picture of any generation, in macroblocks */
    char err[256];
    pthread_mutex_t err_mu;                                 /* several parsers may report into err */
};

static char g_open_error[256];

static int sfail(mvf_stream *s, int code, const char *fmt, ...)
{
    char *dst = s ? s->err : g_open_error;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 256, fmt, ap);
    va_end(ap);
    return code;
}

/* Zero bytes kept behind every unescaped RBSP.  The bit reader never checks bounds inside a macroblock (a corrupt
 * slice is caught by br_overrun() after the macroblock it happens in); one macroblock reads at most 27 residual
 * blocks of at most 16 x 28 + 60 bits plus a few hundred bits of header: well under 2 KB. */
#define RBSP_SLACK 4096

/* NAL payload (after the header byte) -> RBSP (`dst` holds n + RBSP_SLACK bytes); returns the RBSP length (7.4.1.1) */
static size_t unescape(const uint8_t *src, size_t n, uint8_t *dst)
{
    /* emulation_prevention_three_byte (7.4.1): the 03 of every 00 00 03 goes.  An escape can only follow a zero byte,
     * so the stretches between zero bytes (hundreds of bytes in entropy-coded data) are copied wholesale. */
    size_t o = 0, i = 0;
    int zeros = 0;
    while (i < n) {
        if (zeros == 0) {
            const uint8_t *z = memchr(src + i, 0, n - i);
            const size_t run = z ? (size_t)(z - (src + i)) : n - i;
            memcpy(dst + o, src + i, run);
            o += run; i += run;
            if (i >= n) break;
        }
        if (zeros >= 2 && src[i] == 3) { zeros = 0; i++; continue; }
        dst[o++] = src[i];
        zeros = src[i] == 0 ? zeros + 1 : 0;
        i++;
    }
    memset(dst + o, 0, RBSP_SLACK);
    return o;
}

/* bits before the rbsp_stop_one_bit (7.3.2.11) */
static size_t rbsp_payload_bits(const uint8_t *rbsp, size_t n)
{
    while (n > 0 && rbsp[n - 1] == 0) n--;                  /* trailing zero bytes (cabac_zero_words, padding) */
    if (n == 0) return 0;
    int b = 0;
    while (!((rbsp[n - 1] >> b) & 1)) b++;
    return (n - 1) * 8 + (size_t)(7 - b);
}

static const uint8_t default4_intra[16] = {6,13,13,20,20,20,28,28,28,28,32,32,32,37,37,42};
static const uint8_t default4_inter[16] = {10,14,14,20,20,20,24,24,24,24,27,27,27,30,30,34};
static const uint8_t default8_intra[64] = {6,10,10,13,11,13,16,16,16,16,18,18,18,18,18,23,23,23,23,23,23,25,25,25,25,25,25,25,
    27,27,27,27,27,27,27,27,29,29,29,29,29,29,29,31,31,31,31,31,31,33,33,33,33,33,36,36,36,36,38,38,38,40,40,42};
static const uint8_t default8_inter[64] = {9,13,13,15,13,15,17,17,17,17,19,19,19,19,19,21,21,21,21,21,21,22,22,22,22,22,22,22,
    24,24,24,24,24,24,24,24,25,25,25,25,25,25,25,27,27,27,27,27,27,28,28,28,28,28,30,30,30,30,32,32,32,33,33,35};

/* 7.3.2.1.1.1; returns 1 when the list says "use default" */
static int parse_scaling_list(br_t *b, uint8_t *list, int n)
{
    int last = 8, next = 8, use_default = 0;
    for (int j = 0; j < n; j++) {
        if (next != 0) {
            int delta = br_se(b);
            next = (last + delta + 256) % 256;
            use_default = (j == 0 && next == 0);
        }
        list[j] = (uint8_t)(next == 0 ? last : next);
        last = list[j];
    }
    return use_default;
}

/* seq_parameter_set_rbsp (7.3.2.1.1; decodeSPS, h264_parameterset.c:123-397).  *out is written only on success;
 * *id receives seq_parameter_set_id (or -1) whenever it could be read, so that a failed SPS can retire the one
 * it would have replaced. */
static int parse_sps(mvf_stream *s, const uint8_t *rbsp, size_t n, sps_t *out, int *id)
{
    br_t b = BR_INIT(rbsp, n * 8);
    sps_t v;
    memset(&v, 0, sizeof v);
    *id = -1;
    v.profile_idc = (int)br_get(&b, 8);
    br_get(&b, 8);                                          /* constraint_set flags + reserved */
    v.level_idc = (int)br_get(&b, 8);
    {
        const uint32_t sid = br_ue(&b);                     /* seq_parameter_set_id, 0..31 (7.4.2.1.1) */
        if (sid >= MVF_MAX_SPS) return sfail(s, MVG_FAILURE, "bad SPS (seq_parameter_set_id %u)", sid);
        v.id = *id = (int)sid;
    }
    v.chroma_format_idc = 1;
    for (int i = 0; i < 6; i++) memset(v.list4[i], 16, 16);
    for (int i = 0; i < 2; i++) memset(v.list8[i], 16, 64);
    int p = v.profile_idc;
    if (p == 100 || p == 110 || p == 122 || p == 244 || p == 44 || p == 83 || p == 86 || p == 118 || p == 128) {
        v.chroma_format_idc = (int)br_ue(&b);
        if (v.chroma_format_idc != 1)                       /* h264_parameterset.c:175-199 */
            return sfail(s, MVG_UNSUPPORTED, "chroma_format_idc %d (only 4:2:0 is supported)", v.chroma_format_idc);
        if (br_ue(&b) != 0 || br_ue(&b) != 0) return sfail(s, MVG_UNSUPPORTED, "bit depth > 8");
        if (br_bit(&b)) return sfail(s, MVG_UNSUPPORTED, "qpprime_y_zero_transform_bypass_flag");
        if (br_bit(&b)) {                                   /* seq_scaling_matrix_present_flag */
            for (int i = 0; i < 8; i++) {
                uint8_t *dst = i < 6 ? v.list4[i] : v.list8[i - 6];
                int len = i < 6 ? 16 : 64;
                int present = br_bit(&b), use_default = 0;
                if (present) use_default = parse_scaling_list(&b, dst, len);
                if (!present || use_default) {              /* fall-back rule A / default (Table 7-2) */
                    if (!present && (i == 1 || i == 2 || i == 4 || i == 5)) memcpy(dst, v.list4[i - 1], 16);
                    else if (i == 0 || i == 1 || i == 2) memcpy(dst, default4_intra, 16);
                    else if (i < 6) memcpy(dst, default4_inter, 16);
                    else memcpy(dst, i == 6 ? default8_intra : default8_inter, 64);
                }
            }
        }
    }
    {   /* log2_max_frame_num_minus4 and log2_max_pic_order_cnt_lsb_minus4 are 0..12 (7.4.2.1.1); they become bit counts */
        const uint32_t fn = br_ue(&b), pt = br_ue(&b);
        if (fn > 12 || pt > 2) return sfail(s, MVG_FAILURE, "bad SPS (log2_max_frame_num_minus4 %u, pic_order_cnt_type %u)", fn, pt);
        v.log2_max_frame_num = (int)fn + 4;
        v.poc_type = (int)pt;
    }
    if (v.poc_type == 0) {
        const uint32_t pl = br_ue(&b);
        if (pl > 12) return sfail(s, MVG_FAILURE, "bad SPS (log2_max_pic_order_cnt_lsb_minus4 %u)", pl);
        v.log2_max_poc_lsb = (int)pl + 4;
    }
    else if (v.poc_type == 1) {
        v.delta_pic_order_always_zero = br_bit(&b);
        br_se(&b); br_se(&b);
        uint32_t cyc = br_ue(&b);
        if (cyc > 255) return sfail(s, MVG_FAILURE, "bad SPS");
        for (uint32_t i = 0; i < cyc; i++) br_se(&b);
    }
    br_ue(&b);                                              /* max_num_ref_frames */
    br_bit(&b);                                             /* gaps_in_frame_num_value_allowed_flag */
    {
        const uint32_t wm = br_ue(&b), hm = br_ue(&b);      /* pic_width_in_mbs_minus1, pic_height_in_map_units_minus1 */
        if (wm > 1023 || hm > 1023) return sfail(s, MVG_FAILURE, "bad SPS (%u x %u macroblocks)", wm + 1, hm + 1);
        v.width_mbs = (int)wm + 1; v.height_mbs = (int)hm + 1;
    }
    v.frame_mbs_only = br_bit(&b);
    if (!v.frame_mbs_only) return sfail(s, MVG_UNSUPPORTED, "interlaced (frame_mbs_only_flag = 0)");
    br_bit(&b);                                             /* direct_8x8_inference_flag */
    if (br_bit(&b)) for (int i = 0; i < 4; i++) { const uint32_t cr = br_ue(&b); v.crop[i] = cr > 16384 ? 16384 : (int)cr; }
    if (br_overrun(&b) || v.width_mbs > 1024 || v.height_mbs > 1024) return sfail(s, MVG_FAILURE, "truncated or bad SPS");
    v.valid = 1;
    *out = v;
    return MVG_SUCCESS;
}

/* pic_parameter_set_rbsp (7.3.2.2; decodePPS, h264_parameterset.c:812-926) */
static int parse_pps(mvf_stream *s, const uint8_t *rbsp, size_t n, pps_t *out, int *id)
{
    br_t b = BR_INIT(rbsp, rbsp_payload_bits(rbsp, n));
    pps_t v;
    memset(&v, 0, sizeof v);
    *id = -1;
    {
        const uint32_t pid = br_ue(&b), sid = br_ue(&b);    /* 0..255, 0..31 (7.4.2.2) */
        if (pid >= MVF_MAX_PPS || sid >= MVF_MAX_SPS)
            return sfail(s, MVG_FAILURE, "bad PPS (pic_parameter_set_id %u, seq_parameter_set_id %u)", pid, sid);
        v.id = *id = (int)pid; v.sps_id = (int)sid;
    }
    v.entropy_cabac = br_bit(&b);
    v.bottom_field_poc_present = br_bit(&b);
    if (br_ue(&b) != 0) return sfail(s, MVG_UNSUPPORTED, "FMO (num_slice_groups_minus1 > 0)");
    br_ue(&b); br_ue(&b);                                   /* num_ref_idx defaults */
    br_bit(&b); br_get(&b, 2);                              /* weighted prediction */
    {   /* pic_init_qp_minus26 is -26..25, the chroma offsets -12..12 (7.4.2.2) */
        const int iq = br_se(&b);
        br_se(&b);                                          /* pic_init_qs */
        const int co = br_se(&b);
        if (iq < -26 || iq > 25 || co < -12 || co > 12) return sfail(s, MVG_FAILURE, "bad PPS (pic_init_qp_minus26 %d, chroma_qp_index_offset %d)", iq, co);
        v.init_qp = 26 + iq; v.cb_off = co;
    }
    v.deblocking_control = br_bit(&b);
    v.constrained_intra = br_bit(&b);
    v.redundant_pic_cnt = br_bit(&b);
    v.cr_off = v.cb_off;
    if (b.pos < b.nbits) {                                  /* more_rbsp_data() */
        v.has_extension = 1;
        v.transform8x8 = br_bit(&b);
        if (br_bit(&b)) return sfail(s, MVG_UNSUPPORTED, "PPS scaling lists (h264_parameterset.c:904-921)");
        v.cr_off = br_se(&b);
        if (v.cr_off < -12 || v.cr_off > 12) return sfail(s, MVG_FAILURE, "bad PPS (second_chroma_qp_index_offset %d)", v.cr_off);
    }
    if (v.entropy_cabac) return sfail(s, MVG_UNSUPPORTED, "CABAC (entropy_coding_mode_flag = 1)");
    if (b.pos > b.nbits + 1) return sfail(s, MVG_FAILURE, "truncated PPS");
    v.valid = 1;
    *out = v;
    return MVG_SUCCESS;
}

/* The generation of an IDR slice: read pic_parameter_set_id from the first bytes of its header (7.3.3), follow it
 * to the PPS and SPS stored under those ids at this point of the stream, and find or append the pair.
 * Returns the generation index, or -1 with a message in s->err when the picture names a parameter set the stream
 * has not delivered (or delivered broken). */
static int generation_of(mvf_stream *s, const nal_t *nl, const sps_t *sps_tab, const pps_t *pps_tab)
{
    uint8_t head[48 + 8];
    size_t n = nl->size > 1 ? nl->size - 1 : 0, o = 0;
    int zeros = 0;
    for (size_t i = 0; i < n && o < 48; i++) {              /* unescape the first bytes (7.4.1) */
        const uint8_t c = s->data[nl->off + 1 + i];
        if (zeros >= 2 && c == 3) { zeros = 0; continue; }
        head[o++] = c;
        zeros = c == 0 ? zeros + 1 : 0;
    }
    memset(head + o, 0, 8);
    br_t b = BR_INIT(head, o * 8);
    br_ue(&b); br_ue(&b);                                   /* first_mb_in_slice, slice_type */
    const uint32_t pid = br_ue(&b);
    if (br_overrun(&b) || pid >= MVF_MAX_PPS) { sfail(s, MVG_FAILURE, "slice header: pic_parameter_set_id out of range"); return -1; }
    /* a generation index of -1 / -2 = the picture cannot be decoded (MVG_FAILURE / MVG_UNSUPPORTED) */
    const pps_t *pps = &pps_tab[pid];
    if (!pps->valid) {
        if (pps->err_code == 0) sfail(s, MVG_FAILURE, "slice refers to PPS %u, which the stream has not delivered", pid);
        else sfail(s, pps->err_code, "slice refers to PPS %u, which is %s", pid, pps->err_code == MVG_UNSUPPORTED ? "unsupported" : "damaged");
        return pps->err_code == MVG_UNSUPPORTED ? -2 : -1;
    }
    const sps_t *sps = &sps_tab[pps->sps_id];
    if (!sps->valid) {
        if (sps->err_code == 0) sfail(s, MVG_FAILURE, "PPS %u refers to SPS %d, which the stream has not delivered", pid, pps->sps_id);
        else sfail(s, sps->err_code, "PPS %u refers to SPS %d, which is %s", pid, pps->sps_id, sps->err_code == MVG_UNSUPPORTED ? "unsupported" : "damaged");
        return sps->err_code == MVG_UNSUPPORTED ? -2 : -1;
    }
    paramgen_t g;
    memset(&g, 0, sizeof g);
    g.sps = *sps; g.pps = *pps;
    /* the PPS extension (transform_8x8_mode_flag, second_chroma_qp_index_offset) only exists for the reference when
     * the SPS says High or above (h264_parameterset.c:898-926) */
    if (g.sps.profile_idc < 100) { g.pps.transform8x8 = 0; g.pps.cr_off = g.pps.cb_off; }
    for (int k = s->n_gens - 1; k >= 0; k--)
        if (memcmp(&s->gens[k], &g, sizeof g) == 0) return k;
    if (s->n_gens == s->cap_gens) {
        const int cap = s->cap_gens ? 2 * s->cap_gens : 4;
        paramgen_t *ng = realloc(s->gens, sizeof(paramgen_t) * (size_t)cap);
        if (!ng) { sfail(s, MVG_FAILURE, "out of memory"); return -1; }
        s->gens = ng; s->cap_gens = cap;
    }
    s->gens[s->n_gens] = g;
    if (g.sps.width_mbs * g.sps.height_mbs > s->max_mbs) s->max_mbs = g.sps.width_mbs * g.sps.height_mbs;
    return s->n_gens++;
}

static mvf_stream *stream_new(const uint8_t *data, size_t len)
{
    pthread_once(&lut_once, build_luts);
    mvf_stream *s = calloc(1, sizeof *s);
    if (!s) return NULL;
    s->data = data; s->len = len;
    pthread_mutex_init(&s->err_mu, NULL);
    return s;
}

/* room for one more entry in s->nals (*cap entries allocated); 0 when out of memory */
static int nals_reserve(mvf_stream *s, int *cap)
{
    if (s->n_nals < *cap) return 1;
    if (*cap > INT_MAX / 4) return 0;
    const int nc = *cap ? 2 * *cap : 1024;
    nal_t *nn = realloc(s->nals, sizeof(nal_t) * (size_t)nc);
    if (!nn) return 0;
    s->nals = nn; *cap = nc;
    return 1;
}

static int index_stream(mvf_stream *s);

int mvf_open_annexb(const uint8_t *data, size_t len, mvf_stream **out)
{
    if (!out) return MVG_FAILURE;
    *out = NULL;
    if (!data || len < 5) return sfail(NULL, MVG_FAILURE, "mvf_open_annexb: empty stream");
    mvf_stream *s = stream_new(data, len);
    if (!s) return sfail(NULL, MVG_FAILURE, "out of memory");

    /* start codes 00 00 01 (a 4-byte start code is the same with one more leading zero) */
    int cap = 0;
    /* look for the 01 (one byte in 256 of entropy-coded data) and check the two bytes before it */
    for (const uint8_t *q = data + 2, *const end = data + len - 1; q < end; q++) {
        q = memchr(q, 1, (size_t)(end - q));
        if (!q) break;
        if (q[-1] != 0 || q[-2] != 0) continue;
        if (!nals_reserve(s, &cap)) { mvf_close(s); return sfail(NULL, MVG_FAILURE, "out of memory"); }
        s->nals[s->n_nals].off = (size_t)(q - data) + 1;
        s->nals[s->n_nals].type = q[1] & 31;
        s->n_nals++;
    }
    for (int k = 0; k < s->n_nals; k++) {
        size_t end = k + 1 < s->n_nals ? s->nals[k + 1].off - 3 : len;
        while (end > s->nals[k].off && data[end - 1] == 0) end--;          /* trailing_zero_8bits */
        s->nals[k].size = end - s->nals[k].off;
        s->nals[k].sample = (k + 1 < s->n_nals ? s->nals[k + 1].off : len) - s->nals[k].off;
    }
    const int rc = index_stream(s);
    if (rc == MVG_SUCCESS) *out = s;
    return rc;
}

/* The part of opening that does not depend on the container: s->nals[] holds the NAL units in stream order.
 * Replays the parameter sets, indexes the IDR pictures and their generations.  Closes s on failure. */
static int index_stream(mvf_stream *s)
{
    s->idr = malloc(sizeof(int) * (size_t)(s->n_nals + 1));
    s->idr_gen = malloc(sizeof(int) * (size_t)(s->n_nals + 1));
    sps_t *sps_tab = calloc(MVF_MAX_SPS, sizeof *sps_tab);
    pps_t *pps_tab = calloc(MVF_MAX_PPS, sizeof *pps_tab);
    if (!s->idr || !s->idr_gen || !sps_tab || !pps_tab) {
        free(sps_tab); free(pps_tab); mvf_close(s);
        return sfail(NULL, MVG_FAILURE, "out of memory");
    }
    /* Parameter sets in stream order, as the reference's NAL loop meets them (h264.c:128-150): a new SPS / PPS
     * replaces the one stored under its id (h264_parameterset.c:162-164, :835-837 -- the reference files a PPS under
     * its seq_parameter_set_id and looks it up by pic_parameter_set_id, which is the same slot whenever the two
     * ids are equal, the only case it decodes; this front end files it under pic_parameter_set_id as 7.4.1.2.1 says).
     * One that cannot be used retires the slot: pictures that name it fail one by one, with its message. */
    int rc_first = MVG_SUCCESS, usable = 0;
    char err_first[256] = "";
    uint8_t *tmp = NULL;
    for (int k = 0; k < s->n_nals; k++) {
        const nal_t *nl = &s->nals[k];
        if (nl->type == 5) {
            s->idr_gen[s->n_idr] = generation_of(s, nl, sps_tab, pps_tab);
            if (s->idr_gen[s->n_idr] >= 0) usable++;
            else if (rc_first == MVG_SUCCESS) { rc_first = MVG_FAILURE; memcpy(err_first, s->err, sizeof err_first); }
            s->idr[s->n_idr++] = k;
            continue;
        }
        if (nl->type != 7 && nl->type != 8) continue;
        {
            uint8_t *nt = realloc(tmp, nl->size + RBSP_SLACK);
            if (!nt) { free(tmp); free(sps_tab); free(pps_tab); mvf_close(s); return sfail(NULL, MVG_FAILURE, "out of memory"); }
            tmp = nt;
        }
        size_t n = unescape(s->data + nl->off + 1, nl->size ? nl->size - 1 : 0, tmp);
        int id = -1, rc;
        if (nl->type == 7) {
            sps_t v;
            rc = parse_sps(s, tmp, n, &v, &id);
            if (rc == MVG_SUCCESS) sps_tab[id] = v;
            else if (id >= 0) { memset(&sps_tab[id], 0, sizeof sps_tab[id]); sps_tab[id].err_code = rc; }
        } else {
            pps_t v;
            rc = parse_pps(s, tmp, n, &v, &id);
            if (rc == MVG_SUCCESS) pps_tab[id] = v;
            else if (id >= 0) { memset(&pps_tab[id], 0, sizeof pps_tab[id]); pps_tab[id].err_code = rc; }
        }
        if (rc != MVG_SUCCESS && rc_first == MVG_SUCCESS) { rc_first = rc; memcpy(err_first, s->err, sizeof err_first); }
    }
    free(tmp); free(sps_tab); free(pps_tab);
    if (!usable) {          /* nothing to decode: answer with the first thing that went wrong */
        if (rc_first == MVG_SUCCESS) { rc_first = MVG_FAILURE; snprintf(err_first, sizeof err_first, "no SPS/PPS in the stream"); }
        memcpy(g_open_error, err_first, sizeof g_open_error);
        mvf_close(s);
        return rc_first;
    }
    s->err[0] = 0;
    return MVG_SUCCESS;
}

/* ------------------------------------------------------------------------ */
/* MP4 / QuickTime (ISO/IEC 14496-12, the AVC file format of 14496-15): the NAL units of the first H.264 video
 * track, in decode order, indexed in place                                   */

static uint32_t rd32(const uint8_t *p) { return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3]; }
static uint64_t rd64(const uint8_t *p) { return (uint64_t)rd32(p) << 32 | rd32(p + 4); }
#define FOURCC(a, b, c, d) ((uint32_t)(a) << 24 | (uint32_t)(b) << 16 | (uint32_t)(c) << 8 | (uint32_t)(d))

typedef struct { size_t body, end; } box_t;         /* payload [body, end) in the file */

/* the box whose header starts at d[pos], inside a parent that ends at `end`.  0 when its header is cut short or
 * its size is below the header or runs past the parent.  size 0 means "to the end of the parent" (of the file at
 * the top level), size 1 a 64-bit largesize. */
static int box_read(const uint8_t *d, size_t pos, size_t end, uint32_t *type, box_t *b)
{
    if (end - pos < 8) return 0;
    uint64_t size = rd32(d + pos);
    size_t hdr = 8;
    *type = rd32(d + pos + 4);
    if (size == 1) {
        if (end - pos < 16) return 0;
        size = rd64(d + pos + 8);
        hdr = 16;
    } else if (size == 0) size = end - pos;
    if (size < hdr || size > end - pos) return 0;
    b->body = pos + hdr; b->end = pos + (size_t)size;
    return 1;
}

/* first child of type `want`: 1 found, 0 absent, -1 a malformed child before it */
static int box_find(const uint8_t *d, box_t parent, uint32_t want, box_t *out)
{
    for (size_t pos = parent.body; pos < parent.end; pos = out->end) {
        uint32_t t;
        if (!box_read(d, pos, parent.end, &t, out)) return -1;
        if (t == want) return 1;
    }
    return 0;
}

/* the four-character code as text, for messages */
static const char *fourcc_str(uint32_t t, char buf[5])
{
    for (int i = 0; i < 4; i++) { const char c = (char)(t >> (24 - 8 * i)); buf[i] = c >= 32 && c < 127 ? c : '?'; }
    buf[4] = 0;
    return buf;
}

static int nal_append(mvf_stream *s, int *cap, size_t off, size_t size, size_t sample)
{
    if (!nals_reserve(s, cap)) return 0;
    nal_t *nl = &s->nals[s->n_nals++];
    nl->off = off; nl->size = size; nl->sample = sample; nl->type = s->data[off] & 31;
    return 1;
}

/* AVCDecoderConfigurationRecord (14496-15 5.3.3.1) at [c.body, c.end) -- an MP4 avcC box or a Matroska CodecPrivate;
 * `who` and `where` name them in messages.  Checks it and reads lengthSizeMinusOne; with `cap` it also appends its SPS
 * and PPS NAL units to s->nals.  Whatever follows the PPS list (the High-profile fields) is not read.  1 = ok,
 * 0 = malformed (message in g_open_error), -1 = out of memory. */
static int avcc_walk(mvf_stream *s, const char *who, const char *where, box_t c, int *len_size, int *cap)
{
    const uint8_t *d = s->data;
    if (c.end - c.body < 7) { sfail(NULL, MVG_FAILURE, "%s: avcC %s too short", who, where); return 0; }
    const int lsm1 = d[c.body + 4] & 3;
    if (lsm1 == 2) { sfail(NULL, MVG_FAILURE, "%s: avcC lengthSizeMinusOne 2 is invalid (1, 2 or 4 byte lengths)", who); return 0; }
    *len_size = lsm1 + 1;
    size_t p = c.body + 5;
    for (int list = 0; list < 2; list++) {
        if (p >= c.end) { sfail(NULL, MVG_FAILURE, "%s: avcC %s truncated", who, where); return 0; }
        const int n = list == 0 ? d[p] & 31 : d[p];
        p++;
        for (int i = 0; i < n; i++) {
            if (c.end - p < 2) { sfail(NULL, MVG_FAILURE, "%s: avcC %s truncated", who, where); return 0; }
            const size_t sz = (size_t)d[p] << 8 | d[p + 1];
            p += 2;
            if (sz > c.end - p) { sfail(NULL, MVG_FAILURE, "%s: avcC parameter set runs past its %s", who, where); return 0; }
            if (sz && cap && !nal_append(s, cap, p, sz, 0)) return -1;
            p += sz;
        }
    }
    return 1;
}

/* the length-prefixed NAL units (`L`-byte lengths) of one sample / frame [off, off + size), each sized for
 * mvf_select_idr() by the whole sample.  A length field that runs past the sample drops every NAL unit of the sample,
 * like a damaged picture.  0 when out of memory. */
static int sample_nals(mvf_stream *s, int *cap, size_t off, size_t size, int L)
{
    const uint8_t *data = s->data;
    const int before = s->n_nals;
    for (size_t p = off, e = off + size; p < e; ) {
        if (e - p < (size_t)L) { s->n_nals = before; break; }
        size_t n = 0;
        for (int j = 0; j < L; j++) n = n << 8 | data[p + j];
        p += (size_t)L;
        if (n > e - p) { s->n_nals = before; break; }
        if (n && !nal_append(s, cap, p, n, size)) return 0;
        p += n;
    }
    return 1;
}

typedef struct { box_t avcc; int len_size; } sdesc_t;

int mvf_open_mp4(const uint8_t *data, size_t len, mvf_stream **out)
{
    if (!out) return MVG_FAILURE;
    *out = NULL;
    if (!data || len < 8) return sfail(NULL, MVG_FAILURE, "mvf_open_mp4: empty file");
    mvf_stream *s = stream_new(data, len);
    if (!s) return sfail(NULL, MVG_FAILURE, "out of memory");
    sdesc_t *desc = NULL;
    int rc = MVG_FAILURE, cap = 0;
    char cc[5];
#define MP4_FAIL(code, ...) do { rc = sfail(NULL, code, __VA_ARGS__); goto fail; } while (0)

    /* top level: ftyp, moov, mdat, ... in any order; the sample table addresses mdat by absolute file offsets */
    box_t moov = {0, 0}, b;
    int have_moov = 0;
    for (size_t pos = 0; pos < len; pos = b.end) {
        uint32_t t;
        if (!box_read(data, pos, len, &t, &b)) MP4_FAIL(MVG_FAILURE, "mp4: truncated or overlapping box at offset %zu", pos);
        if (t == FOURCC('m', 'o', 'o', 'f')) MP4_FAIL(MVG_UNSUPPORTED, "mp4: fragmented file (moof); only files with a complete moov index are supported");
        if (t == FOURCC('m', 'o', 'o', 'v') && !have_moov) { moov = b; have_moov = 1; }
    }
    if (!have_moov) MP4_FAIL(MVG_FAILURE, "mp4: no moov box");

    /* the first track whose handler is 'vide' and whose first sample description is avc1 / avc3 */
    box_t stbl = {0, 0}, stsd = {0, 0};
    int found = 0;
    uint32_t other_codec = 0;
    for (size_t pos = moov.body; pos < moov.end; pos = b.end) {
        uint32_t t;
        if (!box_read(data, pos, moov.end, &t, &b)) MP4_FAIL(MVG_FAILURE, "mp4: truncated or overlapping box at offset %zu", pos);
        if (t == FOURCC('m', 'v', 'e', 'x')) MP4_FAIL(MVG_UNSUPPORTED, "mp4: fragmented file (mvex); only files with a complete moov index are supported");
        if (t != FOURCC('t', 'r', 'a', 'k') || found) continue;
        box_t mdia, hdlr, minf, st, sd, e;
        int r = box_find(data, b, FOURCC('m', 'd', 'i', 'a'), &mdia);
        if (r == 1) r = box_find(data, mdia, FOURCC('h', 'd', 'l', 'r'), &hdlr);
        if (r < 0) MP4_FAIL(MVG_FAILURE, "mp4: truncated or overlapping box in a track");
        if (r == 0 || hdlr.end - hdlr.body < 12 || rd32(data + hdlr.body + 8) != FOURCC('v', 'i', 'd', 'e')) continue;
        r = box_find(data, mdia, FOURCC('m', 'i', 'n', 'f'), &minf);
        if (r == 1) r = box_find(data, minf, FOURCC('s', 't', 'b', 'l'), &st);
        if (r == 1) r = box_find(data, st, FOURCC('s', 't', 's', 'd'), &sd);
        if (r < 0) MP4_FAIL(MVG_FAILURE, "mp4: truncated or overlapping box in the video track");
        if (r == 0) MP4_FAIL(MVG_FAILURE, "mp4: video track without a sample description (stsd)");
        uint32_t et;
        if (sd.end - sd.body < 8 || rd32(data + sd.body + 4) == 0 || !box_read(data, sd.body + 8, sd.end, &et, &e))
            MP4_FAIL(MVG_FAILURE, "mp4: empty or truncated sample description (stsd)");
        if (et == FOURCC('a', 'v', 'c', '1') || et == FOURCC('a', 'v', 'c', '3')) { stbl = st; stsd = sd; found = 1; }
        else if (!other_codec) other_codec = et;
    }
    if (!found && other_codec) MP4_FAIL(MVG_UNSUPPORTED, "mp4: the video track holds '%s', not H.264 (avc1 / avc3)", fourcc_str(other_codec, cc));
    if (!found) MP4_FAIL(MVG_UNSUPPORTED, "mp4: no video track");

    /* sample descriptions: every one must be H.264 with a usable avcC */
    const uint32_t n_desc = rd32(data + stsd.body + 4);
    if (n_desc > (stsd.end - stsd.body - 8) / 8) MP4_FAIL(MVG_FAILURE, "mp4: stsd entry count %u exceeds its box", n_desc);
    desc = calloc(n_desc, sizeof *desc);
    if (!desc) MP4_FAIL(MVG_FAILURE, "out of memory");
    for (size_t pos = stsd.body + 8, i = 0; i < n_desc; i++, pos = b.end) {
        uint32_t t;
        box_t avcc;
        if (!box_read(data, pos, stsd.end, &t, &b)) MP4_FAIL(MVG_FAILURE, "mp4: truncated or overlapping sample description %zu", i + 1);
        if (t != FOURCC('a', 'v', 'c', '1') && t != FOURCC('a', 'v', 'c', '3'))
            MP4_FAIL(MVG_UNSUPPORTED, "mp4: sample description %zu is '%s', not H.264 (avc1 / avc3)", i + 1, fourcc_str(t, cc));
        /* VisualSampleEntry: 8 bytes of SampleEntry + 70 of visual fields, then its boxes */
        const box_t inner = { b.body + 78, b.end };
        if (b.end - b.body < 78 || box_find(data, inner, FOURCC('a', 'v', 'c', 'C'), &avcc) != 1)
            MP4_FAIL(MVG_FAILURE, "mp4: sample description %zu has no readable avcC box", i + 1);
        desc[i].avcc = avcc;
        if (avcc_walk(s, "mp4", "box", avcc, &desc[i].len_size, NULL) != 1) goto fail;
    }

    /* sample table: sizes (stsz), samples per chunk and their description (stsc), chunk offsets (stco / co64).  Sync
     * marks (stss) are not needed: as in an Annex-B stream, the pictures are the IDR NAL units, wherever they are. */
    box_t stsz, stsc, stco;
    int r = box_find(data, stbl, FOURCC('s', 't', 's', 'z'), &stsz), co64 = 0;
    if (r == 1) r = box_find(data, stbl, FOURCC('s', 't', 's', 'c'), &stsc);
    if (r == 1) {
        r = box_find(data, stbl, FOURCC('s', 't', 'c', 'o'), &stco);
        if (r == 0) { r = box_find(data, stbl, FOURCC('c', 'o', '6', '4'), &stco); co64 = 1; }
    }
    if (r < 0) MP4_FAIL(MVG_FAILURE, "mp4: truncated or overlapping box in the sample table");
    if (r == 0) MP4_FAIL(MVG_FAILURE, "mp4: the sample table lacks stsz, stsc or stco / co64");
    if (stsz.end - stsz.body < 12 || stsc.end - stsc.body < 8 || stco.end - stco.body < 8)
        MP4_FAIL(MVG_FAILURE, "mp4: truncated stsz, stsc or chunk offset box");
    const uint32_t const_size = rd32(data + stsz.body + 4), n_samples = rd32(data + stsz.body + 8);
    const uint32_t n_runs = rd32(data + stsc.body + 4), n_chunks = rd32(data + stco.body + 4);
    const size_t co_size = co64 ? 8 : 4;
    if (const_size == 0 && n_samples > (stsz.end - stsz.body - 12) / 4) MP4_FAIL(MVG_FAILURE, "mp4: stsz sample count %u exceeds its box", n_samples);
    if (n_samples > len) MP4_FAIL(MVG_FAILURE, "mp4: stsz sample count %u exceeds the file size", n_samples);
    if (n_runs > (stsc.end - stsc.body - 8) / 12) MP4_FAIL(MVG_FAILURE, "mp4: stsc entry count %u exceeds its box", n_runs);
    if (n_chunks > (stco.end - stco.body - 8) / co_size) MP4_FAIL(MVG_FAILURE, "mp4: chunk offset count %u exceeds its box", n_chunks);
    const uint8_t *run = data + stsc.body + 8;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n_runs; i++) {
        const uint32_t first = rd32(run + 12 * i), per = rd32(run + 12 * i + 4), di = rd32(run + 12 * i + 8);
        const uint64_t next = i + 1 < n_runs ? rd32(run + 12 * (i + 1)) : (uint64_t)n_chunks + 1;
        if ((i == 0 && first != 1) || first > n_chunks || next <= first)
            MP4_FAIL(MVG_FAILURE, "mp4: stsc entry %u: first_chunk %u (chunks must start at 1 and increase, %u chunks)", i + 1, first, n_chunks);
        if (di < 1 || di > n_desc) MP4_FAIL(MVG_FAILURE, "mp4: stsc entry %u names sample description %u of %u", i + 1, di, n_desc);
        total += (next - first) * per;
        if (total > n_samples) break;
    }
    if (total != n_samples) MP4_FAIL(MVG_FAILURE, "mp4: stsc describes %s samples, stsz %u", total > n_samples ? "more" : "fewer", n_samples);

    /* every sample in decode order: the parameter sets of its description first whenever the description changes,
     * then its length-prefixed NAL units */
    uint32_t sample = 0;
    int cur_desc = -1;
    for (uint32_t i = 0; i < n_runs; i++) {
        const uint32_t first = rd32(run + 12 * i), per = rd32(run + 12 * i + 4), di = rd32(run + 12 * i + 8) - 1;
        const uint64_t next = i + 1 < n_runs ? rd32(run + 12 * (i + 1)) : (uint64_t)n_chunks + 1;
        for (uint64_t c = first; c < next && per; c++) {
            const uint8_t *co = data + stco.body + 8 + co_size * (c - 1);
            const uint64_t chunk = co64 ? rd64(co) : rd32(co);
            if (chunk > len) MP4_FAIL(MVG_FAILURE, "mp4: chunk %u lies outside the file", (uint32_t)c);
            size_t off = (size_t)chunk;
            for (uint32_t k = 0; k < per; k++, sample++) {
                const size_t size = const_size ? const_size : rd32(data + stsz.body + 12 + 4 * (size_t)sample);
                if (size > len - off) MP4_FAIL(MVG_FAILURE, "mp4: sample %u lies outside the file", sample + 1);
                if ((int)di != cur_desc) {
                    int dummy;
                    const int w = avcc_walk(s, "mp4", "box", desc[di].avcc, &dummy, &cap);
                    if (w < 0) MP4_FAIL(MVG_FAILURE, "out of memory");
                    cur_desc = (int)di;
                }
                if (!sample_nals(s, &cap, off, size, desc[di].len_size)) MP4_FAIL(MVG_FAILURE, "out of memory");
                off += size;
            }
        }
    }
    free(desc);
#undef MP4_FAIL
    rc = index_stream(s);
    if (rc == MVG_SUCCESS) *out = s;
    return rc;
fail:
    free(desc);
    mvf_close(s);
    return rc;
}

/* ------------------------------------------------------------------------ */
/* MPEG-2 transport stream (ISO/IEC 13818-1): the PES payloads of the first H.264 stream, scanned for start codes as
 * they arrive, exactly as mvf_open_annexb() scans a stream held in one piece.  The NAL units are not contiguous in the
 * file, so the stream keeps a copy of the ones read later -- SPS, PPS and IDR slices -- and of nothing else.      */

static uint32_t crc32_mpeg(const uint8_t *p, size_t n)          /* 13818-1 Annex A: polynomial 04C11DB7, no reflection */
{
    uint32_t c = 0xFFFFFFFFu;
    for (size_t i = 0; i < n; i++) {
        c ^= (uint32_t)p[i] << 24;
        for (int k = 0; k < 8; k++) c = c & 0x80000000u ? c << 1 ^ 0x04C11DB7u : c << 1;
    }
    return c;
}

/* Annex-B scan over a byte stream that arrives in pieces.  ES offsets count the bytes fed; a kept NAL unit's bytes
 * go to buf, every other byte is only looked at. */
typedef struct {
    uint8_t *buf; size_t len, cap;
    size_t pos;             /* bytes fed so far */
    int zeros;              /* zero bytes (up to 2) at the end of what was fed since the last damage */
    int pend;               /* the last byte fed completed 00 00 01: a start code if any byte follows */
    int in_nal, keep, type;
    size_t nal_es, nal_buf; /* the current NAL header byte: its ES offset and, when kept, its offset in buf */
} es_scan;

static int es_put(es_scan *e, const uint8_t *p, size_t n)
{
    if (!n) return 1;
    if (e->cap - e->len < n) {
        size_t nc = e->cap ? e->cap : 1 << 20;
        while (nc - e->len < n) { if (nc > SIZE_MAX / 2) return 0; nc *= 2; }
        uint8_t *nb = realloc(e->buf, nc);
        if (!nb) return 0;
        e->buf = nb; e->cap = nc;
    }
    memcpy(e->buf + e->len, p, n);
    e->len += n;
    return 1;
}

/* the current NAL unit ends at ES offset `end` (the start code's first zero, or the end of the stream) and the next
 * NAL header, if any, is at `next`: the size and sample rules of mvf_open_annexb() */
static int es_finish(mvf_stream *s, es_scan *e, int *cap, size_t end, size_t next)
{
    if (!e->in_nal || !e->keep) return 1;
    size_t n = e->nal_buf + (end - e->nal_es);
    while (n > e->nal_buf && e->buf[n - 1] == 0) n--;                  /* trailing_zero_8bits */
    e->len = n;
    if (!nals_reserve(s, cap)) return 0;
    nal_t *nl = &s->nals[s->n_nals++];
    nl->off = e->nal_buf; nl->size = n - e->nal_buf; nl->sample = next - e->nal_es; nl->type = e->type;
    return 1;
}

static void es_start(es_scan *e, size_t off, uint8_t header)
{
    e->in_nal = 1;
    e->type = header & 31;
    e->keep = e->type == 5 || e->type == 7 || e->type == 8;
    e->nal_es = off;
    e->nal_buf = e->len;
}

/* lost bytes: the NAL unit they fall into is dropped, and no start code spans them; the scan resumes at the next one */
static void es_damage(es_scan *e)
{
    if (e->in_nal && e->keep) e->len = e->nal_buf;
    e->in_nal = 0; e->zeros = 0; e->pend = 0;
}

static int es_feed(mvf_stream *s, es_scan *e, int *cap, const uint8_t *c, size_t n)
{
    if (!n) return 1;
    size_t from = 0;            /* c[from..) not yet copied for a kept NAL unit */
    if (e->pend) {              /* the 01 was the last byte fed, at ES offset pos - 1 */
        e->pend = 0;
        if (!es_finish(s, e, cap, e->pos - 3, e->pos)) return 0;
        es_start(e, e->pos, c[0]);
    }
    for (size_t i = 0; i < n; i++) {
        const uint8_t *q = memchr(c + i, 1, n - i);
        if (!q) break;
        const size_t k = (size_t)(q - c);
        i = k;
        const int z = k >= 2 ? (c[k - 1] == 0 && c[k - 2] == 0) : k == 1 ? (c[0] == 0 && e->zeros >= 1) : e->zeros >= 2;
        if (!z) continue;
        if (e->in_nal && e->keep && !es_put(e, c + from, k + 1 - from)) return 0;
        from = k + 1;
        if (k + 1 == n) { e->pend = 1; break; }
        if (!es_finish(s, e, cap, e->pos + k - 2, e->pos + k + 1)) return 0;
        es_start(e, e->pos + k + 1, c[k + 1]);
    }
    if (e->in_nal && e->keep && !es_put(e, c + from, n - from)) return 0;
    if (n >= 2) e->zeros = c[n - 1] ? 0 : c[n - 2] ? 1 : 2;
    else e->zeros = c[0] ? 0 : e->zeros ? 2 : 1;
    e->pos += n;
    return 1;
}

/* 188-byte packets, with a 4-byte TP_extra_header before each (M2TS, 192) or 16 parity bytes after each (204): the
 * first offset below 204 from which sync bytes repeat at one of these periods over five packets (over every whole
 * packet of a shorter file).  0 when there is none. */
static int ts_sync(const uint8_t *d, size_t len, size_t *first, size_t *period)
{
    static const size_t per[3] = {188, 192, 204};
    for (size_t o = 0; o < 204 && o + 188 <= len; o++) {
        if (d[o] != 0x47) continue;
        for (int k = 0; k < 3; k++) {
            const size_t whole = (len - o - 188) / per[k] + 1, need = whole < 5 ? whole : 5;
            size_t i = 1;
            while (i < need && d[o + i * per[k]] == 0x47) i++;
            if (i == need) { *first = o; *period = per[k]; return 1; }
        }
    }
    return 0;
}

/* the next packet at or after `pos`; after lost sync, the next offset at which the period holds again (for the
 * packets that follow, as far as the file goes).  NULL at the end. */
static const uint8_t *ts_packet(const uint8_t *d, size_t len, size_t per, size_t *pos, int *lost)
{
    size_t q = *pos;
    *lost = 0;
    if (q + 188 > len) return NULL;
    if (d[q] != 0x47) {
        *lost = 1;
        for (q++; q + 188 <= len; q++)
            if (d[q] == 0x47 && (q + per + 188 > len || d[q + per] == 0x47) && (q + 2 * per + 188 > len || d[q + 2 * per] == 0x47))
                break;
        if (q + 188 > len) return NULL;
    }
    *pos = q + per;
    return d + q;
}

/* PSI section assembly on one PID (2.4.4): sections may span packets; 3 + section_length is at most 1024 bytes */
typedef struct { uint8_t b[1024]; size_t have, need; int on; } psi_t;

#define TS_MAX_PROGRAMS 64

typedef struct {
    int n_prog, have_pat;
    int prog_num[TS_MAX_PROGRAMS], pmt_pid[TS_MAX_PROGRAMS];
    int pmt_seen[TS_MAX_PROGRAMS], h264_pid[TS_MAX_PROGRAMS], other_video[TS_MAX_PROGRAMS];
    psi_t pat, pmt[TS_MAX_PROGRAMS];
} ts_psi;

static int ts_video_type(int st)    /* stream_type values of video other than H.264 (13818-1 Table 2-34 and its amendments) */
{
    return st == 0x01 || st == 0x02 || st == 0x10 || st == 0x1E || st == 0x1F || st == 0x20 || st == 0x24 ||
           st == 0x27 || st == 0x33 || st == 0x42 || st == 0xD1 || st == 0xEA;
}

/* a complete section: CRC_32 over the whole of it gives 0 (Annex A); PAT and PMT sections with current_next_indicator
 * set are taken, the first good copy of each */
static void ts_section(ts_psi *t, int prog, const uint8_t *b, size_t n)
{
    if (n < 12 || !(b[1] & 0x80) || !(b[5] & 1) || crc32_mpeg(b, n) != 0) return;
    const size_t end = n - 4;
    if (prog < 0) {
        if (b[0] != 0x00 || t->have_pat) return;
        for (size_t p = 8; p + 4 <= end && t->n_prog < TS_MAX_PROGRAMS; p += 4) {
            const int num = b[p] << 8 | b[p + 1], pid = (b[p + 2] & 0x1F) << 8 | b[p + 3];
            if (num == 0) continue;                         /* the network PID */
            const int i = t->n_prog++;
            t->prog_num[i] = num; t->pmt_pid[i] = pid;
            t->pmt_seen[i] = 0; t->h264_pid[i] = -1; t->other_video[i] = 0;
        }
        t->have_pat = 1;
        return;
    }
    if (b[0] != 0x02 || t->pmt_seen[prog] || (b[3] << 8 | b[4]) != t->prog_num[prog]) return;
    size_t p = 12 + (size_t)((b[10] & 0x0F) << 8 | b[11]);           /* past program_info */
    while (p + 5 <= end) {
        const int st = b[p], pid = (b[p + 1] & 0x1F) << 8 | b[p + 2];
        if (st == 0x1B && t->h264_pid[prog] < 0) t->h264_pid[prog] = pid;
        else if (ts_video_type(st) && !t->other_video[prog]) t->other_video[prog] = st;
        p += 5 + (size_t)((b[p + 3] & 0x0F) << 8 | b[p + 4]);
    }
    t->pmt_seen[prog] = 1;
}

/* one packet payload of a PSI PID */
static void ts_psi_feed(ts_psi *t, int prog, psi_t *a, int pusi, const uint8_t *p, size_t n)
{
    size_t i = 0;
    if (pusi) {
        if (!n) return;
        const size_t ptr = p[0];
        i = 1;
        if (a->on) {                                        /* the tail of the section in progress */
            const size_t take = ptr < n - 1 ? ptr : n - 1;
            if (a->have + take <= a->need) { memcpy(a->b + a->have, p + 1, take); a->have += take; }
            if (a->have == a->need) ts_section(t, prog, a->b, a->need);
        }
        a->on = 0;
        i += ptr;
        while (i < n && p[i] != 0xFF) {                     /* sections that start here; 0xFF is stuffing */
            if (n - i < 3) { memcpy(a->b, p + i, n - i); a->have = n - i; a->need = 0; a->on = 1; return; }
            const size_t need = 3 + (size_t)((p[i + 1] & 0x0F) << 8 | p[i + 2]);
            if (need > sizeof a->b) return;
            if (n - i >= need) { ts_section(t, prog, p + i, need); i += need; continue; }
            memcpy(a->b, p + i, n - i); a->have = n - i; a->need = need; a->on = 1;
            return;
        }
        return;
    }
    if (!a->on) return;
    if (a->need == 0) {                                     /* the section header itself was split */
        const size_t take = 3 - a->have < n ? 3 - a->have : n;
        memcpy(a->b + a->have, p, take); a->have += take; p += take; n -= take;
        if (a->have < 3) return;
        a->need = 3 + (size_t)((a->b[1] & 0x0F) << 8 | a->b[2]);
        if (a->need > sizeof a->b) { a->on = 0; return; }
    }
    const size_t take = a->need - a->have < n ? a->need - a->have : n;
    memcpy(a->b + a->have, p, take);
    a->have += take;
    if (a->have == a->need) { ts_section(t, prog, a->b, a->need); a->on = 0; }
}

/* the chosen program once it is certain: the first program of the PAT whose PMT lists H.264, all earlier ones seen */
static int ts_choice(const ts_psi *t, int at_end)
{
    for (int i = 0; i < t->n_prog; i++) {
        if (t->pmt_seen[i] && t->h264_pid[i] >= 0) return i;
        if (!t->pmt_seen[i] && !at_end) return -1;
    }
    return -1;
}

int mvf_open_ts(const uint8_t *data, size_t len, mvf_stream **out)
{
    if (!out) return MVG_FAILURE;
    *out = NULL;
    size_t first, per;
    if (!data || !ts_sync(data, len, &first, &per)) return sfail(NULL, MVG_FAILURE, "ts: no sync bytes at a 188, 192 or 204 byte period");
    ts_psi *t = calloc(1, sizeof *t);
    mvf_stream *s = stream_new(data, len);
    es_scan e;
    memset(&e, 0, sizeof e);
    int rc = MVG_FAILURE, cap = 0;
#define TS_FAIL(code, ...) do { rc = sfail(NULL, code, __VA_ARGS__); goto fail; } while (0)
    if (!s || !t) TS_FAIL(MVG_FAILURE, "out of memory");

    /* pass 1: PAT and PMTs, until the choice is certain or the file ends */
    int lost, prog = -1;
    const uint8_t *pk;
    for (size_t pos = first; prog < 0 && (pk = ts_packet(data, len, per, &pos, &lost)); ) {
        const int pid = (pk[1] & 0x1F) << 8 | pk[2], afc = pk[3] >> 4 & 3;
        if (pk[1] & 0x80 || !(afc & 1)) continue;
        const size_t o = afc & 2 ? 5 + (size_t)pk[4] : 4;
        if (o >= 188) continue;
        if (pid == 0) ts_psi_feed(t, -1, &t->pat, pk[1] & 0x40, pk + o, 188 - o);
        else
            for (int i = 0; i < t->n_prog; i++)
                if (t->pmt_pid[i] == pid) ts_psi_feed(t, i, &t->pmt[i], pk[1] & 0x40, pk + o, 188 - o);
        if (t->have_pat) prog = ts_choice(t, 0);
    }
    if (!t->have_pat) TS_FAIL(MVG_FAILURE, "ts: no program association table (PAT)");
    if (prog < 0) prog = ts_choice(t, 1);
    if (prog < 0) {
        for (int i = 0; i < t->n_prog; i++)
            if (t->other_video[i])
                TS_FAIL(MVG_UNSUPPORTED, "ts: program %d carries video of stream_type 0x%02X, not H.264 (0x1B)", t->prog_num[i], t->other_video[i]);
        for (int i = 0; i < t->n_prog; i++)
            if (!t->pmt_seen[i]) TS_FAIL(MVG_FAILURE, "ts: no program map table (PMT) for program %d on PID 0x%X", t->prog_num[i], t->pmt_pid[i]);
        TS_FAIL(MVG_UNSUPPORTED, "ts: no video stream in %s", t->n_prog ? "any program" : "the PAT (it lists no program)");
    }
    const int vpid = t->h264_pid[prog];

    /* pass 2: the PES packets of that PID from the start of the file */
    int last_cc = -1, dup = 0, in_hdr = 0, in_pes = 0, bounded = 0;
    size_t hlen = 0, left = 0, n_pes = 0;
    uint8_t hdr[9 + 255];
    /* Lost bytes (lost sync, a continuity gap, an errored packet) drop the NAL unit they fall into.  What follows on
     * the PID up to the next payload_unit_start_indicator is still payload of one PES packet, so it is scanned on, but
     * that packet's length no longer says anything; only a PES header cut in two loses the rest of its packet. */
#define TS_DAMAGE() do { es_damage(&e); if (in_hdr) in_hdr = in_pes = 0; else { in_pes = n_pes > 0; bounded = 0; } } while (0)
    for (size_t pos = first; (pk = ts_packet(data, len, per, &pos, &lost)); ) {
        if (lost) TS_DAMAGE();
        const int pid = (pk[1] & 0x1F) << 8 | pk[2];
        if (pk[1] & 0x80) {                                 /* transport_error_indicator: the packet cannot be trusted */
            if (pid == vpid) TS_DAMAGE();
            continue;
        }
        if (pid != vpid) continue;
        if (pk[3] >> 6) TS_FAIL(MVG_UNSUPPORTED, "ts: the video packets are scrambled (transport_scrambling_control %d)", pk[3] >> 6);
        const int afc = pk[3] >> 4 & 3, cc = pk[3] & 15;
        size_t o = 4;
        int disc = 0;
        if (afc & 2) {
            o = 5 + (size_t)pk[4];
            disc = pk[4] && (pk[5] & 0x80);                 /* discontinuity_indicator */
        }
        if (!(afc & 1)) continue;                           /* no payload: the counter does not advance */
        if (last_cc >= 0 && cc == last_cc && !dup && !disc) { dup = 1; continue; }     /* a duplicate packet */
        const int gap = last_cc >= 0 && cc != ((last_cc + 1) & 15) && !disc;
        last_cc = cc; dup = 0;
        if (gap || o > 188) {
            TS_DAMAGE();
            if (o > 188) continue;
        }
        const uint8_t *p = pk + o;
        size_t n = 188 - o;
        if (pk[1] & 0x40) {                                 /* payload_unit_start_indicator: a new PES packet */
            if ((in_pes && bounded && left) || in_hdr) es_damage(&e);          /* the previous one was cut short */
            in_pes = 0; in_hdr = 1; hlen = 0;
        }
        if (in_hdr) {
            const size_t want = hlen < 9 ? 9 : 9 + (size_t)hdr[8];
            size_t take = want - hlen < n ? want - hlen : n;
            memcpy(hdr + hlen, p, take); hlen += take; p += take; n -= take;
            if (hlen == 9 && hdr[8] && n) {
                take = hdr[8] < n ? hdr[8] : n;
                memcpy(hdr + hlen, p, take); hlen += take; p += take; n -= take;
            }
            if (hlen < 9 || hlen < 9 + (size_t)hdr[8]) continue;
            in_hdr = 0;
            if (hdr[0] || hdr[1] || hdr[2] != 1 || hdr[3] < 0xE0 || hdr[3] > 0xEF || (hdr[6] & 0xC0) != 0x80) {
                es_damage(&e);                              /* not a video PES header */
                continue;
            }
            if (hdr[6] >> 4 & 3) TS_FAIL(MVG_UNSUPPORTED, "ts: the video PES packets are scrambled (PES_scrambling_control %d)", hdr[6] >> 4 & 3);
            const size_t plen = (size_t)hdr[4] << 8 | hdr[5];
            bounded = plen != 0;
            if (bounded && plen < 3 + (size_t)hdr[8]) { es_damage(&e); continue; }
            left = bounded ? plen - 3 - hdr[8] : 0;
            in_pes = 1; n_pes++;
        }
        if (!in_pes) continue;
        if (bounded) {
            if (n > left) n = left;
            left -= n;
        }
        if (!es_feed(s, &e, &cap, p, n)) TS_FAIL(MVG_FAILURE, "out of memory");
        if (bounded && !left) in_pes = 0;
    }
    if ((in_pes && bounded && left) || in_hdr) es_damage(&e);
#undef TS_DAMAGE
    if (!n_pes) TS_FAIL(MVG_FAILURE, "ts: the H.264 stream of program %d (PID 0x%X) carries no PES packet", t->prog_num[prog], vpid);
    if (!es_finish(s, &e, &cap, e.pos, e.pos)) TS_FAIL(MVG_FAILURE, "out of memory");
#undef TS_FAIL
    free(t);
    {   /* the copy is final: give back the unused capacity, and point the stream at it */
        uint8_t *b = e.len ? realloc(e.buf, e.len) : e.buf;
        if (b) e.buf = b;
    }
    s->data = s->own = e.buf; s->len = e.len;
    rc = index_stream(s);
    if (rc == MVG_SUCCESS) *out = s;
    return rc;
fail:
    free(t); free(e.buf);
    if (s) mvf_close(s);
    return rc;
}

/* ------------------------------------------------------------------------ */
/* Matroska / WebM (EBML, RFC 8794; Matroska, RFC 9559): the frames of the first H.264 video track, in file order, their
 * length-prefixed NAL units indexed in place                                  */

#define MKV_SEGMENT      0x18538067u
#define MKV_CLUSTER      0x1F43B675u
#define MKV_TRACKS       0x1654AE6Bu

/* an EBML variable-length integer at d[*pos]: an element ID keeps its length marker (1..4 bytes), a size loses it
 * (1..8 bytes; all value bits set = unknown, returned as UINT64_MAX).  0 when it is cut short or too wide. */
static int ebml_vint(const uint8_t *d, size_t *pos, size_t end, int is_id, uint64_t *v)
{
    if (*pos >= end || !d[*pos]) return 0;
    const int w = __builtin_clz(d[*pos]) - 23;
    if (w > (is_id ? 4 : 8) || end - *pos < (size_t)w) return 0;
    uint64_t x = is_id ? d[*pos] : d[*pos] & (0xFFu >> w);
    for (int i = 1; i < w; i++) x = x << 8 | d[*pos + i];
    *pos += (size_t)w;
    *v = !is_id && x == (1ull << (7 * w)) - 1 ? UINT64_MAX : x;
    return 1;
}

typedef struct { uint32_t id; size_t body, end; int unknown; } ebml_t;

/* the element at d[pos] inside a parent that ends at `end`; an unknown size reaches to `end` for now.  0 when its
 * header is cut short or its size runs past the parent. */
static int ebml_read(const uint8_t *d, size_t pos, size_t end, ebml_t *e)
{
    uint64_t id, size;
    if (!ebml_vint(d, &pos, end, 1, &id) || !ebml_vint(d, &pos, end, 0, &size)) return 0;
    e->id = (uint32_t)id; e->body = pos;
    e->unknown = size == UINT64_MAX;
    if (!e->unknown && size > end - pos) return 0;
    e->end = e->unknown ? end : pos + (size_t)size;
    return 1;
}

static uint64_t ebml_uint(const uint8_t *d, ebml_t e)
{
    uint64_t v = 0;
    for (size_t p = e.body; p < e.end && p < e.body + 8; p++) v = v << 8 | d[p];
    return v;
}

static int ebml_is(const uint8_t *d, ebml_t e, const char *str)
{
    const size_t n = strlen(str);
    size_t m = e.end - e.body;
    while (m > 0 && d[e.body + m - 1] == 0) m--;            /* strings may be zero-padded */
    return m == n && !memcmp(d + e.body, str, n);
}

static int mkv_segment_child(uint32_t id)
{
    return id == 0x114D9B74u || id == 0x1549A966u || id == MKV_TRACKS || id == MKV_CLUSTER || id == 0x1C53BB6Bu ||
           id == 0x1941A469u || id == 0x1043A770u || id == 0x1254C367u || id == 0xECu || id == 0xBFu;
}

static int mkv_cluster_child(uint32_t id)
{
    return id == 0xE7u || id == 0x5854u || id == 0xA7u || id == 0xABu || id == 0xA3u || id == 0xA0u || id == 0xAFu ||
           id == 0xECu || id == 0xBFu;
}

typedef struct { uint64_t number; int len_size, replayed; box_t priv; } mkv_track;

/* the frames of a SimpleBlock or Block [b, end) of the track: header, lacing (Xiph, EBML, fixed), then each frame's NAL
 * units.  Returns 1, or a return code with a message for a damaged block or when out of memory. */
static int mkv_block(mvf_stream *s, mkv_track *tr, size_t b, size_t end, int *cap)
{
    const uint8_t *d = s->data;
    uint64_t tn;
    size_t p = b;
    if (!ebml_vint(d, &p, end, 0, &tn) || end - p < 3) return sfail(NULL, MVG_FAILURE, "mkv: truncated block header at offset %zu", b);
    if (tn != tr->number) return 1;
    const int lacing = d[p + 2] >> 1 & 3;
    p += 3;
    size_t sizes[256];
    int count = 1;
    if (lacing) {
        if (p >= end) return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
        count = d[p++] + 1;
        if (lacing == 2) {                                  /* fixed */
            if ((end - p) % (size_t)count) return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
            for (int i = 0; i < count; i++) sizes[i] = (end - p) / (size_t)count;
        } else {
            size_t sum = 0;
            for (int i = 0; i < count - 1; i++) {
                uint64_t v = 0;
                if (lacing == 1) {                          /* Xiph: 255s and a final byte */
                    uint8_t c;
                    do {
                        if (p >= end) return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
                        c = d[p++]; v += c;
                    } while (c == 255);
                } else {                                    /* EBML: a size, then signed differences */
                    const size_t at = p;
                    if (!ebml_vint(d, &p, end, 0, &v) || v == UINT64_MAX)
                        return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
                    if (i > 0) {
                        const int w = (int)(p - at);
                        const int64_t delta = (int64_t)v - (int64_t)((1ull << (7 * w - 1)) - 1);
                        if ((int64_t)sizes[i - 1] + delta < 0) return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
                        v = (uint64_t)((int64_t)sizes[i - 1] + delta);
                    }
                }
                if (v > end - p || sum + v > end - p) return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
                sizes[i] = (size_t)v; sum += (size_t)v;
            }
            if (sum > end - p) return sfail(NULL, MVG_FAILURE, "mkv: lace sizes overrun their block at offset %zu", b);
            sizes[count - 1] = end - p - sum;
        }
    } else sizes[0] = end - p;
    for (int i = 0; i < count; i++) {
        if (!tr->replayed) {                                /* the CodecPrivate parameter sets before the first frame */
            int dummy;
            if (avcc_walk(s, "mkv", "CodecPrivate", tr->priv, &dummy, cap) < 0) return sfail(NULL, MVG_FAILURE, "out of memory");
            tr->replayed = 1;
        }
        if (!sample_nals(s, cap, p, sizes[i], tr->len_size)) return sfail(NULL, MVG_FAILURE, "out of memory");
        p += sizes[i];
    }
    return 1;
}

/* the next child of a Segment from `pos` (which ends at `end`): 1 with *e, 0 at its end, -1 damaged.  An unknown-size
 * Segment ends at the first element that cannot be its child; an unknown-size Cluster at the first one that cannot be
 * the Cluster's, and its end is found by walking it. */
static int mkv_next(const uint8_t *d, size_t pos, size_t end, int seg_unknown, ebml_t *e)
{
    if (pos >= end) return 0;
    if (!ebml_read(d, pos, end, e)) return -1;
    if (seg_unknown && !mkv_segment_child(e->id)) return 0;
    if (e->unknown) {
        if (e->id != MKV_CLUSTER) return -1;
        ebml_t c;
        size_t p = e->body;
        while (p < end) {
            if (!ebml_read(d, p, end, &c)) return -1;
            if (!mkv_cluster_child(c.id)) break;
            if (c.unknown) return -1;
            p = c.end;
        }
        e->end = p;
    }
    return 1;
}

int mvf_open_mkv(const uint8_t *data, size_t len, mvf_stream **out)
{
    if (!out) return MVG_FAILURE;
    *out = NULL;
    if (!data || len < 4 || rd32(data) != 0x1A45DFA3u) return sfail(NULL, MVG_FAILURE, "mkv: no EBML header");
    mvf_stream *s = stream_new(data, len);
    if (!s) return sfail(NULL, MVG_FAILURE, "out of memory");
    int rc = MVG_FAILURE, cap = 0;
#define MKV_FAIL(code, ...) do { rc = sfail(NULL, code, __VA_ARGS__); goto fail; } while (0)

    /* EBML header (its DocType), then the first Segment */
    ebml_t e, seg = {0, 0, 0, 0};
    int webm = 0, have_seg = 0;
    if (!ebml_read(data, 0, len, &e) || e.unknown) MKV_FAIL(MVG_FAILURE, "mkv: damaged EBML header");
    for (size_t p = e.body; p < e.end; ) {
        ebml_t c;
        if (!ebml_read(data, p, e.end, &c) || c.unknown) MKV_FAIL(MVG_FAILURE, "mkv: damaged EBML header");
        if (c.id == 0x4282u) webm = ebml_is(data, c, "webm");               /* DocType */
        p = c.end;
    }
    for (size_t p = e.end; p < len && !have_seg; ) {
        if (!ebml_read(data, p, len, &seg)) MKV_FAIL(MVG_FAILURE, "mkv: damaged element at offset %zu", p);
        if (seg.id == MKV_SEGMENT) have_seg = 1;
        else if (seg.unknown) MKV_FAIL(MVG_FAILURE, "mkv: element of unknown size at offset %zu", p);
        else p = seg.end;
    }
    if (!have_seg) MKV_FAIL(MVG_FAILURE, "mkv: no Segment");

    /* the first Tracks element: the first TrackEntry of type video (1) whose CodecID is V_MPEG4/ISO/AVC */
    mkv_track tr;
    memset(&tr, 0, sizeof tr);
    int found = 0, r;
    char other[64] = "";
    for (size_t p = seg.body; (r = mkv_next(data, p, seg.end, seg.unknown, &e)) == 1 && !found; p = e.end) {
        if (e.id != MKV_TRACKS) continue;
        for (size_t q = e.body; q < e.end && !found; ) {
            ebml_t te;
            if (!ebml_read(data, q, e.end, &te) || te.unknown) MKV_FAIL(MVG_FAILURE, "mkv: damaged Tracks element at offset %zu", q);
            q = te.end;
            if (te.id != 0xAEu) continue;                   /* TrackEntry */
            uint64_t number = 0, type = 0;
            int avc = 0, encoded = 0, have_priv = 0;
            ebml_t codec = {0, 0, 0, 0}, priv = {0, 0, 0, 0};
            for (size_t k = te.body; k < te.end; ) {
                ebml_t c;
                if (!ebml_read(data, k, te.end, &c) || c.unknown) MKV_FAIL(MVG_FAILURE, "mkv: damaged TrackEntry at offset %zu", k);
                if (c.id == 0xD7u) number = ebml_uint(data, c);
                else if (c.id == 0x83u) type = ebml_uint(data, c);
                else if (c.id == 0x86u) { codec = c; avc = ebml_is(data, c, "V_MPEG4/ISO/AVC"); }
                else if (c.id == 0x63A2u) { priv = c; have_priv = 1; }
                else if (c.id == 0x6D80u) encoded = 1;      /* ContentEncodings */
                k = c.end;
            }
            if (type != 1) continue;
            if (!avc) {
                if (!other[0]) {
                    size_t n = codec.end - codec.body < sizeof other - 1 ? codec.end - codec.body : sizeof other - 1;
                    for (size_t i = 0; i < n; i++) { const char ch = (char)data[codec.body + i]; other[i] = ch >= 32 && ch < 127 ? ch : '?'; }
                    other[n] = 0;
                    if (!n) snprintf(other, sizeof other, "no CodecID");
                }
                continue;
            }
            if (encoded) MKV_FAIL(MVG_UNSUPPORTED, "mkv: the H.264 track has ContentEncodings (compressed or encrypted frames)");
            if (!number) MKV_FAIL(MVG_FAILURE, "mkv: the H.264 track has no TrackNumber");
            if (!have_priv) MKV_FAIL(MVG_FAILURE, "mkv: the H.264 track has no CodecPrivate (avcC)");
            tr.number = number;
            tr.priv = (box_t){priv.body, priv.end};
            const int w = avcc_walk(s, "mkv", "CodecPrivate", tr.priv, &tr.len_size, NULL);
            if (w != 1) { rc = MVG_FAILURE; goto fail; }
            found = 1;
        }
    }
    if (r < 0) MKV_FAIL(MVG_FAILURE, "mkv: damaged EBML structure in the Segment");
    if (!found && !strcmp(other, "V_MS/VFW/FOURCC"))
        MKV_FAIL(MVG_UNSUPPORTED, "mkv: the video track is V_MS/VFW/FOURCC (Video for Windows); only V_MPEG4/ISO/AVC is supported");
    if (!found && other[0]) MKV_FAIL(MVG_UNSUPPORTED, "mkv: the video track holds %s, not H.264 (V_MPEG4/ISO/AVC)", other);
    if (!found && webm) MKV_FAIL(MVG_UNSUPPORTED, "mkv: WebM file without an H.264 video track");
    if (!found) MKV_FAIL(MVG_UNSUPPORTED, "mkv: no video track");

    /* every Cluster in file order: SimpleBlocks, and Blocks inside BlockGroups, of that track */
    for (size_t p = seg.body; (r = mkv_next(data, p, seg.end, seg.unknown, &e)) == 1; p = e.end) {
        if (e.id != MKV_CLUSTER) continue;
        for (size_t q = e.body; q < e.end; ) {
            ebml_t c;
            if (!ebml_read(data, q, e.end, &c) || c.unknown) MKV_FAIL(MVG_FAILURE, "mkv: damaged Cluster at offset %zu", q);
            q = c.end;
            int br = 1;
            if (c.id == 0xA3u) br = mkv_block(s, &tr, c.body, c.end, &cap);             /* SimpleBlock */
            else if (c.id == 0xA0u)                                                     /* BlockGroup */
                for (size_t k = c.body; k < c.end && br == 1; ) {
                    ebml_t bl;
                    if (!ebml_read(data, k, c.end, &bl) || bl.unknown) MKV_FAIL(MVG_FAILURE, "mkv: damaged BlockGroup at offset %zu", k);
                    if (bl.id == 0xA1u) br = mkv_block(s, &tr, bl.body, bl.end, &cap);  /* Block */
                    k = bl.end;
                }
            if (br != 1) { rc = br; goto fail; }
        }
    }
    if (r < 0) MKV_FAIL(MVG_FAILURE, "mkv: damaged EBML structure in the Segment");
#undef MKV_FAIL
    rc = index_stream(s);
    if (rc == MVG_SUCCESS) *out = s;
    return rc;
fail:
    mvf_close(s);
    return rc;
}

int mvf_close(mvf_stream *s)
{
    if (!s) return MVG_FAILURE;
    pthread_mutex_destroy(&s->err_mu);
    free(s->nals); free(s->idr); free(s->idr_gen); free(s->gens); free(s->own); free(s);
    return MVG_SUCCESS;
}

const char *mvf_last_error(const mvf_stream *s) { return s ? s->err : g_open_error; }

/* normAdjust x scaling matrix (spec 8.5.9; h264.c:419-493, h264_transform.c:645-741); the same
 * tables mvg_build_level_scale() produces, rebuilt here so that libmvfront.so has no CUDA dependency */
static void build_level_scale(const uint8_t l4[3][16], const uint8_t l8[64], int32_t *ls4, int32_t *ls8)
{
    static const int v4[6][3] = {{10,16,13},{11,18,14},{13,20,16},{14,23,18},{16,25,20},{18,29,23}};
    static const int v8[6][6] = {{20,18,32,19,25,24},{22,19,35,21,28,26},{26,23,42,24,33,31},
                                 {28,25,45,26,35,33},{32,28,51,30,40,38},{36,32,58,34,46,43}};
    for (int c = 0; c < 3; c++) {
        int m[16];
        for (int k = 0; k < 16; k++) m[zz4[k]] = l4[c][k];
        for (int q = 0; q < 6; q++)
            for (int i = 0; i < 4; i++)
                for (int j = 0; j < 4; j++) {
                    int cls = (!(i & 1) && !(j & 1)) ? 0 : ((i & 1) && (j & 1)) ? 1 : 2;
                    ls4[(c * 6 + q) * 16 + i * 4 + j] = m[i * 4 + j] * v4[q][cls];
                }
    }
    int m8[64];
    for (int k = 0; k < 64; k++) m8[zz8[k]] = l8[k];
    for (int q = 0; q < 6; q++)
        for (int i = 0; i < 8; i++)
            for (int j = 0; j < 8; j++) {
                int cls;
                if (i % 4 == 0 && j % 4 == 0) cls = 0;
                else if (i % 2 == 1 && j % 2 == 1) cls = 1;
                else if (i % 4 == 2 && j % 4 == 2) cls = 2;
                else if ((i % 4 == 0 && j % 2 == 1) || (i % 2 == 1 && j % 4 == 0)) cls = 3;
                else if ((i % 4 == 0 && j % 4 == 2) || (i % 4 == 2 && j % 4 == 0)) cls = 4;
                else cls = 5;
                ls8[q * 64 + i * 8 + j] = m8[i * 8 + j] * v8[q][cls];
            }
}

int mvf_get_generation_info(const mvf_stream *s, int gen, mvf_info *o)
{
    if (!s || !o || gen < 0 || gen >= s->n_gens) return MVG_FAILURE;
    const sps_t *sps = &s->gens[gen].sps; const pps_t *pps = &s->gens[gen].pps;
    memset(o, 0, sizeof *o);
    o->width_mbs = sps->width_mbs; o->height_mbs = sps->height_mbs;
    o->profile_idc = sps->profile_idc; o->level_idc = sps->level_idc;
    o->n_idr = s->n_idr; o->transform_8x8_mode = pps->transform8x8;
    o->cb_qp_offset = pps->cb_off; o->cr_qp_offset = pps->cr_off; o->pic_init_qp = pps->init_qp;
    o->crop_left = sps->crop[0]; o->crop_right = sps->crop[1]; o->crop_top = sps->crop[2]; o->crop_bottom = sps->crop[3];
    o->n_generations = s->n_gens; o->generation = gen;
    uint8_t l4[3][16];
    for (int c = 0; c < 3; c++) memcpy(l4[c], sps->list4[c], 16);           /* intra Y, Cb, Cr */
    build_level_scale(l4, sps->list8[0], o->level_scale4x4, o->level_scale8x8);
    return MVG_SUCCESS;
}

/* the parameters of the first decodable IDR picture (all there is for a stream that never changes them) */
int mvf_get_info(const mvf_stream *s, mvf_info *o) { return mvf_get_generation_info(s, 0, o); }

int mvf_generation_count(const mvf_stream *s) { return s ? s->n_gens : 0; }

int mvf_picture_generation(const mvf_stream *s, int idr_index)
{
    if (!s || idr_index < 0 || idr_index >= s->n_idr) return -1;
    return s->idr_gen[idr_index] < 0 ? -1 : s->idr_gen[idr_index];
}

/* demuxer/filter.c:52-215, on IDR indices instead of bitstream-map samples */
int mvf_select_idr(const mvf_stream *s, int n_wanted, int mode, int32_t *indices)
{
    if (!s || !indices || n_wanted < 0) return 0;
    int n_idr = s->n_idr;
    if (n_wanted > n_idr) n_wanted = n_idr;                 /* filter.c:79-87 */
    if (mode == 0) {                                        /* PICTURE_UNFILTERED, filter.c:88-92 */
        for (int i = 0; i < n_wanted; i++) indices[i] = i;
        return n_wanted;
    }
    if (n_idr < 1) return 0;
    long long payload = 0;
    long long *size = malloc(sizeof(long long) * (size_t)n_idr);
    int *cand = malloc(sizeof(int) * (size_t)n_idr), n_cand = 0;
    if (!size || !cand) { free(size); free(cand); return 0; }
    for (int i = 0; i < n_idr; i++) {
        size[i] = (long long)s->nals[s->idr[i]].sample;
        payload += size[i];
    }
    int threshold = (int)(((double)payload / (double)n_idr) / 1.66);          /* filter.c:109 */
    int borders = n_idr > 48 ? (int)ceil(n_idr * 0.03) : 0;                   /* filter.c:114-118 */
    for (int i = borders; i < n_idr - borders; i++)
        if (size[i] > threshold) cand[n_cand++] = i;                          /* filter.c:120-131 */
    if (n_wanted > n_cand) n_wanted = n_cand;
    int n_out = 0;
    if (mode == 1) {                                        /* PICTURE_ORDERED */
        for (int i = 0; i < n_wanted; i++) indices[n_out++] = cand[i];
    } else if (n_wanted == 1) {
        indices[n_out++] = cand[0];                         /* the reference divides by zero here (filter.c:140) */
    } else if (n_wanted > 1) {
        int jump = n_cand / (n_wanted - 1);                 /* filter.c:140: ceil() of an integer quotient */
        for (int i = 0; i < n_wanted; i++) {
            int j = i * jump;
            if (j >= n_cand) break;                         /* the reference reads one past the end there */
            indices[n_out++] = cand[j];
        }
    }
    free(size); free(cand);
    return n_out;
}

/* ------------------------------------------------------------------------ */
/* slice + macroblock parsing                                                 */

typedef struct {
    const mvf_stream *s;
    uint8_t *rbsp; size_t rbsp_cap;
    uint8_t *tot_luma, *tot_chroma[2];
    int8_t *mode_grid;
    char err[200];
    /* packed output: levels of the macroblock being parsed, and the words of the picture so far */
    int packed;
    int16_t mb_levels[384];
    uint32_t *pk_nzb, *pk_off;          /* [N] of the output slot */
    uint16_t *pk_words; size_t pk_n, pk_cap;
} worker_t;

static inline int16_t clamp16(int v) { return (int16_t)(v < -32768 ? -32768 : (v > 32767 ? 32767 : v)); }

/* 9.2: one residual block of max_num 16 / 15 / 4 levels.  The non-zero levels go straight to their place,
 * dst[scan index * stride] (the destination must hold zeros), clamped to int16.  Returns TotalCoeff or -1.
 *
 * The bits live in a register window: `win` holds the stream left-aligned at the read position, `have` says how many
 * of its bits are real.  A refill is one unaligned 8-byte load + byte swap + shift (the RBSP has RBSP_SLACK zero bytes
 * behind it, so it never needs a bounds check) and happens at fixed points of the code -- block entry, every second
 * level, every fourth run -- so that its branches are periodic; the data-dependent "window nearly empty" test beside
 * them is almost never true.  Between refills a symbol costs shift + table look-up + shift instead of address +
 * load + swap + shift + look-up: the chain from one symbol's length to the next symbol's bits is what bounds CAVLC. */
static int read_residual_block(br_t *b, int16_t *dst, const int stride, const int max_num, int nC)
{
    const uint8_t *const base = b->p;
    size_t pos = b->pos;
    uint64_t win;
    int have;
#define RRB_REFILL()   do { uint64_t t_; memcpy(&t_, base + (pos >> 3), 8); win = __builtin_bswap64(t_) << (pos & 7); have = 64 - (int)(pos & 7); } while (0)
#define RRB_SKIP(n)    do { const int n_ = (int)(n); win <<= n_; pos += (size_t)n_; have -= n_; } while (0)
#define RRB_PEEK(n)    ((uint32_t)(win >> (64 - (n))))
#define RRB_FAIL()     do { b->pos = pos; return -1; } while (0)
    RRB_REFILL();                                   /* >= 57 bits */
    int tc, t1;
    if (nC == -1) {
        uint16_t e = lut_ctc[RRB_PEEK(8)];
        if (!e) RRB_FAIL();
        RRB_SKIP(e >> 7); tc = (e >> 2) & 31; t1 = e & 3;
    } else if (nC >= 8) {
        uint32_t v = RRB_PEEK(6);
        RRB_SKIP(6);
        if (v == 3) { tc = 0; t1 = 0; } else { tc = (int)(v >> 2) + 1; t1 = (int)(v & 3); if (t1 > tc) RRB_FAIL(); }
    } else {
        const int t = nC < 2 ? 0 : (nC < 4 ? 1 : 2);
        const uint32_t bits = RRB_PEEK(16);
        uint16_t e = lut_ct10[t][bits >> 6];
        if (!e) e = lut_ct[t][bits];
        if (!e) RRB_FAIL();
        RRB_SKIP(e >> 7); tc = (e >> 2) & 31; t1 = e & 3;
    }
    if (tc == 0) { b->pos = pos; return 0; }
    if (tc > max_num) RRB_FAIL();

    int level[16];
    int suffix_len = (tc > 10 && t1 < 3) ? 1 : 0;
    {   /* trailing ones: up to three sign bits, taken without a branch (the ones beyond t1 are overwritten by the
         * level loop; coeff_token took at most 16 bits, so at least 41 are left in the window) */
        const uint32_t signs = RRB_PEEK(3);
        level[0] = 1 - (int)((signs >> 1) & 2); level[1] = 1 - (int)(signs & 2); level[2] = 1 - (int)((signs << 1) & 2);
        RRB_SKIP(t1);
    }
    int first_adj = t1 < 3 ? 2 : 0;                 /* the first level after fewer than three trailing ones (9.2.2.1) */
    for (int i = t1, k = 0; i < tc; i++, k++) {
        if (!(k & 1) || have < 32) RRB_REFILL();    /* a level is 28 bits at most unless it is an escape */
        const uint32_t w32 = (uint32_t)(win >> 32);
        if (!w32) RRB_FAIL();                       /* 32 or more zero bits */
        const int prefix = __builtin_clz(w32);
        int code;
        if (prefix < 14) {              /* the common case: prefix, stop bit and suffix (<= 20 bits) from the window */
            code = (prefix << suffix_len) + (int)((uint64_t)(uint32_t)(w32 << (prefix + 1)) >> (32 - suffix_len));
            RRB_SKIP(prefix + 1 + suffix_len);
        } else {
            RRB_SKIP(prefix + 1);
            RRB_REFILL();
            code = (prefix < 15 ? prefix : 15) << suffix_len;           /* 9.2.2.1 */
            int ssize = suffix_len;
            if (prefix == 14 && suffix_len == 0) ssize = 4;
            else if (prefix >= 15) ssize = prefix - 3;
            if (ssize > 0) { code += (int)RRB_PEEK(ssize); RRB_SKIP(ssize); }
            if (prefix >= 15 && suffix_len == 0) code += 15;
            if (prefix >= 16) code += (1 << (prefix - 3)) - 4096;
            RRB_REFILL();
        }
        code += first_adj; first_adj = 0;
        const int sign = -(code & 1), mag = (code + 2) >> 1;            /* odd: -(code + 1) / 2, even: (code + 2) / 2 */
        level[i] = (mag ^ sign) - sign;
        suffix_len += suffix_len == 0;
        suffix_len += (mag > (3 << (suffix_len - 1))) & (suffix_len < 6);
    }
    int zeros_left = 0;
    RRB_REFILL();
    if (tc < max_num) {
        uint8_t e = max_num == 4 ? lut_tz2[tc - 1][RRB_PEEK(3)] : lut_tz4[tc - 1][RRB_PEEK(9)];
        if (!e) RRB_FAIL();
        RRB_SKIP(e >> 4); zeros_left = e & 15;
    }
    int at = zeros_left + tc - 1;                                       /* scan index of the first (highest) level */
    if (at >= max_num) RRB_FAIL();
    /* run_before for every level but the last, while there are zeros left to place (the branch on zerosLeft is worth
     * keeping: predicted, it takes the table look-ups off the dependency chain; a branch-free loop was 20 % slower) */
    for (int i = 0; i < tc - 1; i++) {
        dst[at * stride] = clamp16(level[i]);
        int run = 0;
        if (zeros_left > 0) {
            if ((i & 3) == 3 || have < 11) RRB_REFILL();                /* total_zeros took <= 9 bits, a run takes <= 11 */
            if (zeros_left < 7) {
                const uint8_t e = lut_run3[zeros_left][RRB_PEEK(3)];
                RRB_SKIP(e >> 4); run = e & 15;
            } else {                                /* Table 9-10, zerosLeft > 6: 3 bits for runs 0..6, then unary */
                const uint32_t t3 = RRB_PEEK(3);
                if (t3) { run = 7 - (int)t3; RRB_SKIP(3); }
                else {
                    const uint32_t w32 = (uint32_t)(win >> 32);
                    const int z = w32 ? __builtin_clz(w32) : 32;
                    if (z > 10) RRB_FAIL();
                    run = z + 4; RRB_SKIP(z + 1);
                }
            }
            if (run > zeros_left) RRB_FAIL();       /* also catches the invalid codes of lut_run3 (run 15) */
            zeros_left -= run;
        }
        at -= 1 + run;
        if (at < 0) RRB_FAIL();
    }
    dst[at * stride] = clamp16(level[tc - 1]);
    b->pos = pos;
    return tc;
#undef RRB_REFILL
#undef RRB_SKIP
#undef RRB_PEEK
#undef RRB_FAIL
}

static int pack_mb(worker_t *w, size_t m, uint32_t touched);

static int wfail(worker_t *w, int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(w->err, sizeof w->err, fmt, ap);
    va_end(ap);
    return code;
}

static int parse_picture(worker_t *w, int idr_index, const mvf_batch *out, size_t pic_slot, int want_w, int want_h)
{
    const mvf_stream *s = w->s;
    const int gen = s->idr_gen[idr_index];
    if (gen < 0)
        return wfail(w, gen == -2 ? MVG_UNSUPPORTED : MVG_FAILURE, "picture %d: no usable SPS/PPS (missing, damaged or unsupported parameter set)", idr_index);
    const sps_t *sps = &s->gens[gen].sps; const pps_t *pps = &s->gens[gen].pps;
    if (sps->width_mbs != want_w || sps->height_mbs != want_h)
        return wfail(w, MVG_FAILURE, "picture %d is %dx%d macroblocks, the batch %dx%d: parse each parameter generation in a call of its own",
                     idr_index, sps->width_mbs, sps->height_mbs, want_w, want_h);
    const nal_t *nl = &s->nals[s->idr[idr_index]];
    if (nl->size + RBSP_SLACK > w->rbsp_cap) {
        w->rbsp_cap = nl->size * 2 + RBSP_SLACK;
        uint8_t *nb = realloc(w->rbsp, w->rbsp_cap);
        if (!nb) return wfail(w, MVG_FAILURE, "picture %d: out of memory", idr_index);
        w->rbsp = nb;
    }
    size_t n = unescape(s->data + nl->off + 1, nl->size - 1, w->rbsp);
    br_t b = BR_INIT(w->rbsp, rbsp_payload_bits(w->rbsp, n));
    int nal_ref_idc = (s->data[nl->off] >> 5) & 3;

    /* ---- slice header, 7.3.3 (h264_slice.c:156-334) ---- */
    if (br_ue(&b) != 0) return wfail(w, MVG_UNSUPPORTED, "picture %d: first_mb_in_slice != 0 (one slice per picture only)", idr_index);
    uint32_t slice_type = br_ue(&b);
    if (slice_type != 2 && slice_type != 7) return wfail(w, MVG_UNSUPPORTED, "picture %d: slice_type %u is not I", idr_index, slice_type);
    br_ue(&b);                                              /* pic_parameter_set_id */
    br_get(&b, sps->log2_max_frame_num);                    /* frame_num */
    br_ue(&b);                                              /* idr_pic_id */
    if (sps->poc_type == 0) {
        br_get(&b, sps->log2_max_poc_lsb);
        if (pps->bottom_field_poc_present) br_se(&b);
    } else if (sps->poc_type == 1 && !sps->delta_pic_order_always_zero) {
        br_se(&b);
        if (pps->bottom_field_poc_present) br_se(&b);
    }
    if (pps->redundant_pic_cnt) br_ue(&b);
    if (nal_ref_idc) { br_bit(&b); br_bit(&b); }            /* dec_ref_pic_marking of an IDR picture */
    const int sqd = br_se(&b);                              /* slice_qp_delta */
    if (sqd < -51 || sqd > 51) return wfail(w, MVG_FAILURE, "picture %d: slice_qp_delta %d out of range", idr_index, sqd);
    int qp = pps->init_qp + sqd;                            /* SliceQPY */
    if (pps->deblocking_control) {
        if (br_ue(&b) != 1) { br_se(&b); br_se(&b); }
    }
    if (qp < 0 || qp > 51) return wfail(w, MVG_FAILURE, "picture %d: SliceQPY %d out of range", idr_index, qp);

    /* ---- slice data, 7.3.4 / 7.3.5 ----
     * Neighbour context (TotalCoeff for nC, 9.2.1; prediction modes for 8.3.1.1 / 8.3.2.1) is kept as one line of the
     * macroblock row above plus the column to the left, and per macroblock in small local grids with a border:
     * grid[y + 1][x + 1] is block (x, y), row 0 the blocks above, column 0 the blocks to the left.  An unavailable
     * TotalCoeff neighbour holds NA (more than any two real counts add up to), an unavailable mode -1. */
    enum { NA = 64 };
    static const uint8_t BX[16] = {0, 1, 0, 1, 2, 3, 2, 3, 0, 1, 0, 1, 2, 3, 2, 3}, BY[16] = {0, 0, 1, 1, 0, 0, 1, 1, 2, 2, 3, 3, 2, 2, 3, 3};
    const int W = sps->width_mbs, H = sps->height_mbs;
    const size_t N = (size_t)W * H;
    uint8_t *const top_l = w->tot_luma, *const top_c[2] = {w->tot_chroma[0], w->tot_chroma[1]};
    int8_t *const top_m = w->mode_grid;
    if (w->packed) memset(w->mb_levels, 0, sizeof w->mb_levels);      /* a failed picture may have left levels behind */
#define NC_OF(a, b) ((a) + (b) < NA ? ((a) + (b) + 1) >> 1 : ((a) + (b) < 2 * NA ? (a) + (b) - NA : 0))

    for (int my = 0; my < H; my++) {
        uint8_t left_l[4] = {NA, NA, NA, NA}, left_c[2][2] = {{NA, NA}, {NA, NA}};
        int8_t left_m[4] = {-1, -1, -1, -1};
        for (int mx = 0; mx < W; mx++) {
            const size_t mbi = pic_slot * N + (size_t)my * W + mx;
            int16_t *cf = w->packed ? w->mb_levels : out->coeff + mbi * 384;
            uint8_t *modes = out->luma_modes + mbi * 16;
            if (!w->packed) memset(cf, 0, 768);         /* packed mode: pack_mb() hands the buffer back zeroed */
            memset(modes, 0, 16);
            uint8_t gl[5][8], gc[2][3][4];
            int8_t gm[5][8];
            for (int i = 0; i < 4; i++) {
                gl[0][i + 1] = my ? top_l[mx * 4 + i] : NA; gl[i + 1][0] = left_l[i];
                gm[0][i + 1] = my ? top_m[mx * 4 + i] : -1; gm[i + 1][0] = left_m[i];
            }
            for (int c = 0; c < 2; c++)
                for (int i = 0; i < 2; i++) { gc[c][0][i + 1] = my ? top_c[c][mx * 2 + i] : NA; gc[c][i + 1][0] = left_c[c][i]; }

            uint32_t mb_type = br_ue(&b);
            if (mb_type == 25) return wfail(w, MVG_UNSUPPORTED, "picture %d: I_PCM macroblock (h264_macroblock.c:151-154)", idr_index);
            if (mb_type > 25) return wfail(w, MVG_FAILURE, "picture %d mb %d: bad mb_type %u", idr_index, my * W + mx, mb_type);
            int kind, i16_mode = 0, cbp_l, cbp_c;
            if (mb_type == 0) {
                kind = (pps->transform8x8 && br_bit(&b)) ? MVG_MB_I8x8 : MVG_MB_I4x4;
                if (kind == MVG_MB_I4x4) {
                    for (int i = 0; i < 16; i++) {
                        const int x = BX[i], y = BY[i], a = gm[y + 1][x], bb = gm[y][x + 1];
                        const int pred = (a | bb) < 0 ? 2 : (a < bb ? a : bb);      /* 8.3.1.1 */
                        const uint32_t f = br_peek(&b, 4);                           /* prev_intra4x4_pred_mode_flag, rem_intra4x4_pred_mode */
                        const int rem = (int)(f & 7);
                        const int mode = (f & 8) ? pred : (rem < pred ? rem : rem + 1);
                        br_skip(&b, (f & 8) ? 1 : 4);
                        modes[i] = (uint8_t)mode;
                        gm[y + 1][x + 1] = (int8_t)mode;
                    }
                } else {
                    for (int i = 0; i < 4; i++) {
                        const int x = (i & 1) * 2, y = (i >> 1) * 2, a = gm[y + 1][x], bb = gm[y][x + 1];
                        const int pred = (a | bb) < 0 ? 2 : (a < bb ? a : bb);      /* 8.3.2.1 */
                        const uint32_t f = br_peek(&b, 4);
                        const int rem = (int)(f & 7);
                        const int mode = (f & 8) ? pred : (rem < pred ? rem : rem + 1);
                        br_skip(&b, (f & 8) ? 1 : 4);
                        modes[i] = (uint8_t)mode;
                        gm[y + 1][x + 1] = gm[y + 1][x + 2] = gm[y + 2][x + 1] = gm[y + 2][x + 2] = (int8_t)mode;
                    }
                }
            } else {
                kind = MVG_MB_I16x16;
                int t = (int)mb_type - 1;
                i16_mode = t & 3; cbp_c = (t >> 2) % 3; cbp_l = t >= 12 ? 15 : 0;
                for (int y = 1; y < 5; y++) gm[y][1] = gm[y][2] = gm[y][3] = gm[y][4] = 2;
            }
            for (int i = 0; i < 4; i++) { top_m[mx * 4 + i] = gm[4][i + 1]; left_m[i] = gm[i + 1][4]; }
            uint32_t chroma_mode = br_ue(&b);
            if (chroma_mode > 3) return wfail(w, MVG_FAILURE, "picture %d mb %d: intra_chroma_pred_mode %u", idr_index, my * W + mx, chroma_mode);
            if (kind != MVG_MB_I16x16) {
                uint32_t cn = br_ue(&b);
                if (cn > 47) return wfail(w, MVG_FAILURE, "picture %d mb %d: coded_block_pattern codeNum %u", idr_index, my * W + mx, cn);
                int cbp = cbp_from_codenum[cn];
                cbp_l = cbp & 15; cbp_c = cbp >> 4;
            }
            uint32_t touched = 0;                           /* blocks of cf[] that received levels (for pack_mb) */
            for (int y = 1; y < 5; y++) gl[y][1] = gl[y][2] = gl[y][3] = gl[y][4] = 0;
            for (int c = 0; c < 2; c++) gc[c][1][1] = gc[c][1][2] = gc[c][2][1] = gc[c][2][2] = 0;
            if (cbp_l || cbp_c || kind == MVG_MB_I16x16) {
                int delta = br_se(&b);
                if (delta < -26 || delta > 25) return wfail(w, MVG_FAILURE, "picture %d mb %d: mb_qp_delta %d out of range", idr_index, my * W + mx, delta);
                if (delta) qp = (qp + delta + 52) % 52;     /* h264_macroblock.c:263-266 */
                /* residual_luma, 7.3.5.3.1 */
                if (kind == MVG_MB_I16x16) {
                    int16_t dc[16] = {0};
                    const int tcdc = read_residual_block(&b, dc, 1, 16, NC_OF(gl[1][0], gl[0][1]));
                    if (tcdc < 0) goto bad_block;
                    if (tcdc > 0) {                          /* the DC levels go to slot 0 of all sixteen blocks */
                        touched |= 0xffffu;
                        for (int k = 0; k < 16; k++) {
                            int r = zz4[k] >> 2, c = zz4[k] & 3;
                            cf[((r & 1) * 2 + (r >> 1) * 8 + (c & 1) + (c >> 1) * 4) * 16] = dc[k];
                        }
                    }
                }
                for (int b8 = 0; b8 < 4; b8++) {
                    if (!((cbp_l >> b8) & 1)) continue;
                    for (int i4 = 0; i4 < 4; i4++) {
                        const int blk = b8 * 4 + i4, x = BX[blk], y = BY[blk];
                        const int nC = NC_OF(gl[y + 1][x], gl[y][x + 1]);
                        int tc;
                        if (kind == MVG_MB_I4x4) tc = read_residual_block(&b, cf + blk * 16, 1, 16, nC);
                        else if (kind == MVG_MB_I8x8) tc = read_residual_block(&b, cf + b8 * 64 + i4, 4, 16, nC);   /* h264_macroblock.c:1182 */
                        else tc = read_residual_block(&b, cf + blk * 16 + 1, 1, 15, nC);
                        if (tc < 0) goto bad_block;
                        if (tc > 0) touched |= kind == MVG_MB_I8x8 ? 0xfu << (4 * b8) : 1u << blk;   /* 8x8: interleaved over its four blocks */
                        gl[y + 1][x + 1] = (uint8_t)tc;
                    }
                }
                /* residual chroma: DC of both planes, then AC of both planes (h264_macroblock.c:1222-1292) */
                if (cbp_c & 3)
                    for (int c = 0; c < 2; c++) {
                        const int tcc = read_residual_block(&b, cf + 256 + c * 64, 16, 4, -1);
                        if (tcc < 0) goto bad_block;
                        if (tcc > 0) touched |= 0xfu << (16 + 4 * c);
                    }
                if (cbp_c & 2)
                    for (int c = 0; c < 2; c++)
                        for (int blk = 0; blk < 4; blk++) {
                            const int x = blk & 1, y = blk >> 1;
                            const int tc = read_residual_block(&b, cf + 256 + c * 64 + blk * 16 + 1, 1, 15, NC_OF(gc[c][y + 1][x], gc[c][y][x + 1]));
                            if (tc < 0) goto bad_block;
                            if (tc > 0) touched |= 1u << (16 + 4 * c + blk);
                            gc[c][y + 1][x + 1] = (uint8_t)tc;
                        }
            }
            for (int i = 0; i < 4; i++) { top_l[mx * 4 + i] = gl[4][i + 1]; left_l[i] = gl[i + 1][4]; }
            for (int c = 0; c < 2; c++)
                for (int i = 0; i < 2; i++) { top_c[c][mx * 2 + i] = gc[c][2][i + 1]; left_c[c][i] = gc[c][i + 1][2]; }
            out->mb_kind[mbi] = (uint8_t)kind;
            out->i16_mode[mbi] = (uint8_t)i16_mode;
            out->chroma_mode[mbi] = (uint8_t)chroma_mode;
            out->qp_y[mbi] = (int8_t)qp;
            if (out->cbp) out->cbp[mbi] = (uint8_t)(cbp_c << 4 | cbp_l);
            if (w->packed && !pack_mb(w, (size_t)my * W + mx, touched)) return wfail(w, MVG_FAILURE, "picture %d: out of memory while packing", idr_index);
            if (br_overrun(&b)) return wfail(w, MVG_FAILURE, "picture %d: slice data ends at macroblock %d of %zu", idr_index, my * W + mx, N);
            continue;
        bad_block:
            return wfail(w, MVG_FAILURE, "picture %d mb %d: invalid CAVLC code", idr_index, my * W + mx);
        }
    }
#undef NC_OF
    return MVG_SUCCESS;
}

/* the 384 levels of one macroblock -> chunk bitmap, masks and non-zero levels appended to the worker's words.
 * `touched`: the blocks the parser wrote levels into (a superset of the non-zero ones); the others hold zeros.  Every
 * non-zero block is zeroed again for the next macroblock (so that the parser needs no 768-byte memset per macroblock). */
static int pack_reserve(worker_t *w)
{
    if (w->pk_n + MVG_PACKED_WORDS_PER_MB > w->pk_cap) {
        size_t cap = w->pk_cap * 2 + 64 * MVG_PACKED_WORDS_PER_MB;
        uint16_t *w2 = realloc(w->pk_words, cap * sizeof *w2);
        if (!w2) return 0;
        w->pk_words = w2; w->pk_cap = cap;
    }
    return 1;
}

static int pack_mb_generic(worker_t *w, size_t m, uint32_t touched)
{
    if (!pack_reserve(w)) return 0;
    int16_t *c = w->mb_levels;
    uint16_t *dst = w->pk_words + w->pk_n;
    uint32_t nzb = 0;
    uint16_t masks[24], lv[384];
    int n_coded = 0, n_lv = 0;
    for (uint32_t todo = touched; todo; todo &= todo - 1) {
        const int b = __builtin_ctz(todo);
        int16_t *cb = c + b * 16;
#if defined(__SSE2__)
        const __m128i z = _mm_setzero_si128();
        const __m128i v0 = _mm_loadu_si128((const __m128i *)cb), v1 = _mm_loadu_si128((const __m128i *)(cb + 8));
        unsigned mask = ~(unsigned)_mm_movemask_epi8(_mm_packs_epi16(_mm_cmpeq_epi16(v0, z), _mm_cmpeq_epi16(v1, z))) & 0xffffu;
        if (!mask) continue;
        _mm_storeu_si128((__m128i *)cb, z); _mm_storeu_si128((__m128i *)(cb + 8), z);
        const uint16_t keep = (uint16_t)mask;
        int16_t tmp[16];
        _mm_storeu_si128((__m128i *)tmp, v0); _mm_storeu_si128((__m128i *)(tmp + 8), v1);
        while (mask) { int k = __builtin_ctz(mask); mask &= mask - 1; lv[n_lv++] = (uint16_t)tmp[k]; }
#else
        uint64_t q[4];
        memcpy(q, cb, 32);
        if (!(q[0] | q[1] | q[2] | q[3])) continue;
        unsigned mask = 0;
        for (int k = 0; k < 16; k++) if (cb[k]) { mask |= 1u << k; lv[n_lv++] = (uint16_t)cb[k]; }
        memset(cb, 0, 32);
        const uint16_t keep = (uint16_t)mask;
#endif
        nzb |= 1u << b;
        masks[n_coded++] = keep;
    }
    w->pk_nzb[m] = nzb;
    w->pk_off[m] = (uint32_t)w->pk_n;
    memcpy(dst, masks, (size_t)n_coded * sizeof *dst);
    memcpy(dst + n_coded, lv, (size_t)n_lv * sizeof *dst);
    w->pk_n += (size_t)(n_coded + n_lv);
    return 1;
}

#if defined(__x86_64__) && defined(__GNUC__)
#include <immintrin.h>
/* the same with AVX-512 (VBMI2): the non-zero levels of a block leave with one compress-store.  Chosen at run time. */
__attribute__((target("avx512f,avx512bw,avx512vl,avx512vbmi2,popcnt")))
static int pack_mb_avx512(worker_t *w, size_t m, uint32_t touched)
{
    if (!pack_reserve(w)) return 0;
    int16_t *c = w->mb_levels;
    uint16_t *dst = w->pk_words + w->pk_n;
    uint32_t nzb = 0;
    uint16_t masks[24];
    int n_coded = 0;
    /* the masks come first in the output and their number decides where the levels start: masks in a first pass */
    for (uint32_t todo = touched; todo; todo &= todo - 1) {
        const int b = __builtin_ctz(todo);
        const __m256i v = _mm256_loadu_si256((const __m256i *)(c + b * 16));
        const __mmask16 k = _mm256_test_epi16_mask(v, v);
        if (k) { nzb |= 1u << b; masks[n_coded++] = (uint16_t)k; }
    }
    uint16_t *lv = dst + n_coded;
    const __m256i z = _mm256_setzero_si256();
    int i = 0;
    for (uint32_t todo = nzb; todo; todo &= todo - 1, i++) {
        int16_t *cb = c + __builtin_ctz(todo) * 16;
        const __m256i v = _mm256_loadu_si256((const __m256i *)cb);
        _mm256_mask_compressstoreu_epi16(lv, (__mmask16)masks[i], v);
        _mm256_storeu_si256((__m256i *)cb, z);
        lv += __builtin_popcount(masks[i]);
        dst[i] = masks[i];
    }
    w->pk_nzb[m] = nzb;
    w->pk_off[m] = (uint32_t)w->pk_n;
    w->pk_n += (size_t)(lv - dst);
    return 1;
}
#endif

static int (*pack_mb_impl)(worker_t *, size_t, uint32_t) = pack_mb_generic;
static int pack_mb(worker_t *w, size_t m, uint32_t touched) { return pack_mb_impl(w, m, touched); }

static void pack_choose(void)       /* called once from build_luts() */
{
#if defined(__x86_64__) && defined(__GNUC__)
    __builtin_cpu_init();
    if (__builtin_cpu_supports("avx512vbmi2") && __builtin_cpu_supports("avx512bw") && __builtin_cpu_supports("avx512vl") &&
        !getenv("MVF_NO_AVX512"))
        pack_mb_impl = pack_mb_avx512;
#endif
}

/* ------------------------------------------------------------------------ */
/* the parser: persistent worker threads, one IDR slice per thread at a time  */

typedef struct { uint16_t *w; size_t n, cap; } picbuf_t;

struct mvf_parser {
    mvf_stream *s;
    int n_workers;                      /* threads started (0: everything runs in the caller) */
    int scratch_count;                  /* entries of workers[] */
    pthread_t *th;
    worker_t *workers;                  /* n_workers, or 1 for the inline case */
    pthread_mutex_t mu;
    pthread_cond_t cv_work, cv_done;
    unsigned job_seq; int quit, active;
    /* the job in flight */
    const int32_t *indices; int first, count, W, H, strict;
    const mvf_batch *out; const mvf_packed_batch *pk; int32_t *status;
    int next;                           /* next picture to claim (atomic) */
    uint8_t *done; int done_cap;        /* per picture: finished (release/acquire) */
    picbuf_t *pic; int pic_cap;         /* packed output: the words of each picture, kept between calls */
    int rc; char err[200];              /* first failure */
};

static int worker_scratch(worker_t *w, const mvf_stream *s)
{
    const size_t N = (size_t)s->max_mbs;
    memset(w, 0, sizeof *w);
    w->s = s;
    /* one line of neighbour context per macroblock row (TotalCoeff of luma / Cb / Cr blocks, prediction modes): N bounds
     * the picture width of every generation */
    w->tot_luma = malloc(N * 4 + 16); w->tot_chroma[0] = malloc(N * 2 + 16); w->tot_chroma[1] = malloc(N * 2 + 16);
    w->mode_grid = malloc(N * 4 + 16);
    return w->tot_luma && w->tot_chroma[0] && w->tot_chroma[1] && w->mode_grid;
}
static void worker_release(worker_t *w)
{
    free(w->rbsp); free(w->tot_luma); free(w->tot_chroma[0]); free(w->tot_chroma[1]); free(w->mode_grid);
    memset(w, 0, sizeof *w);
}

/* a picture that could not be parsed leaves a slot the kernels can still run over: no levels, all-zero side information */
static void blank_picture(const mvf_parser *p, int i)
{
    const size_t N = (size_t)p->W * p->H, o = (size_t)i * N;
    if (p->pk) {
        memset(p->pk->mb_kind + o, 0, N); memset(p->pk->i16_mode + o, 0, N); memset(p->pk->chroma_mode + o, 0, N);
        memset(p->pk->qp_y + o, 0, N); memset(p->pk->luma_modes + o * 16, 0, N * 16);
        memset(p->pk->nz_blocks + o, 0, N * 4); memset(p->pk->word_off + o, 0, N * 4);
    } else {
        memset(p->out->mb_kind + o, 0, N); memset(p->out->i16_mode + o, 0, N); memset(p->out->chroma_mode + o, 0, N);
        memset(p->out->qp_y + o, 0, N); memset(p->out->cbp + o, 0, N); memset(p->out->luma_modes + o * 16, 0, N * 16);
        memset(p->out->coeff + o * 384, 0, N * 768);
    }
}

/* claim pictures of the current job until none is left */
static void work_on_job(mvf_parser *p, worker_t *w)
{
    const mvf_stream *s = p->s;
    const size_t N = (size_t)p->W * p->H;
    mvf_batch view;                                         /* packed output: the small arrays of the output batch */
    memset(&view, 0, sizeof view);
    w->packed = p->pk != NULL;
    if (p->pk) {
        view.mb_kind = p->pk->mb_kind; view.i16_mode = p->pk->i16_mode; view.chroma_mode = p->pk->chroma_mode;
        view.qp_y = p->pk->qp_y; view.luma_modes = p->pk->luma_modes;
    }
    for (;;) {
        const int i = __atomic_fetch_add(&p->next, 1, __ATOMIC_RELAXED);
        if (i >= p->count) break;
        const int idx = p->indices ? p->indices[i] : p->first + i;
        int rc = (idx < 0 || idx >= s->n_idr) ? wfail(w, MVG_FAILURE, "IDR index %d out of range (0..%d)", idx, s->n_idr - 1)
                                              : MVG_SUCCESS;
        if (rc == MVG_SUCCESS) {
            if (p->pk) {
                w->pk_nzb = p->pk->nz_blocks + (size_t)i * N; w->pk_off = p->pk->word_off + (size_t)i * N;
                w->pk_words = p->pic[i].w; w->pk_n = 0; w->pk_cap = p->pic[i].cap;
            }
            rc = parse_picture(w, idx, p->pk ? &view : p->out, (size_t)i, p->W, p->H);
            if (p->pk) { p->pic[i].w = w->pk_words; p->pic[i].cap = w->pk_cap; p->pic[i].n = rc == MVG_SUCCESS ? w->pk_n : 0; }
        } else if (p->pk) p->pic[i].n = 0;
        if (p->status) p->status[i] = rc;
        if (rc != MVG_SUCCESS) {
            if (!p->strict) blank_picture(p, i);
            pthread_mutex_lock(&p->mu);
            if (p->rc == MVG_SUCCESS) { p->rc = rc; memcpy(p->err, w->err, sizeof p->err); }
            pthread_mutex_unlock(&p->mu);
            if (p->strict) __atomic_store_n(&p->next, p->count, __ATOMIC_RELAXED);      /* all or nothing: stop handing out work */
        }
        __atomic_store_n(&p->done[i], 1, __ATOMIC_RELEASE);
        if (p->n_workers) { pthread_mutex_lock(&p->mu); pthread_cond_broadcast(&p->cv_done); pthread_mutex_unlock(&p->mu); }
    }
}

typedef struct { mvf_parser *p; int k; } worker_arg_t;

static void *worker_main(void *arg)
{
    worker_arg_t *a = arg;
    mvf_parser *p = a->p;
    worker_t *w = &p->workers[a->k];
    free(a);
    unsigned seen = 0;
    for (;;) {
        pthread_mutex_lock(&p->mu);
        while (!p->quit && p->job_seq == seen) pthread_cond_wait(&p->cv_work, &p->mu);
        if (p->quit) { pthread_mutex_unlock(&p->mu); return NULL; }
        seen = p->job_seq;
        pthread_mutex_unlock(&p->mu);
        work_on_job(p, w);
        pthread_mutex_lock(&p->mu);
        if (--p->active == 0) pthread_cond_broadcast(&p->cv_done);
        pthread_mutex_unlock(&p->mu);
    }
}

int mvf_parser_create(mvf_stream *s, int n_threads, mvf_parser **out)
{
    if (!out) return MVG_FAILURE;
    *out = NULL;
    if (!s) return MVG_FAILURE;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 256) n_threads = 256;
    mvf_parser *p = calloc(1, sizeof *p);
    if (!p) return sfail(s, MVG_FAILURE, "mvf_parser_create: out of memory");
    p->s = s;
    pthread_mutex_init(&p->mu, NULL); pthread_cond_init(&p->cv_work, NULL); pthread_cond_init(&p->cv_done, NULL);
    const int n_scratch = n_threads;
    p->workers = calloc((size_t)n_scratch, sizeof *p->workers);
    p->th = calloc((size_t)n_threads, sizeof *p->th);
    int ok = p->workers && p->th;
    if (p->workers) p->scratch_count = n_scratch;
    for (int k = 0; ok && k < n_scratch; k++) ok = worker_scratch(&p->workers[k], s);
    if (!ok) { mvf_parser_destroy(p); return sfail(s, MVG_FAILURE, "mvf_parser_create: out of memory (%d workers, %d macroblocks per picture)", n_threads, s->max_mbs); }
    if (n_threads > 1)
        for (int k = 0; k < n_threads; k++) {
            worker_arg_t *a = malloc(sizeof *a);
            if (!a) break;
            a->p = p; a->k = k;
            if (pthread_create(&p->th[p->n_workers], NULL, worker_main, a) != 0) { free(a); break; }
            p->n_workers++;
        }
    /* no thread could be started (or one was asked for): the caller's thread parses, with workers[0]'s scratch */
    *out = p;
    return MVG_SUCCESS;
}

int mvf_parser_destroy(mvf_parser *p)
{
    if (!p) return MVG_FAILURE;
    pthread_mutex_lock(&p->mu); p->quit = 1; pthread_cond_broadcast(&p->cv_work); pthread_mutex_unlock(&p->mu);
    for (int k = 0; k < p->n_workers; k++) pthread_join(p->th[k], NULL);
    free(p->th);
    if (p->workers) { for (int k = 0; k < p->scratch_count; k++) worker_release(&p->workers[k]); free(p->workers); }
    for (int i = 0; i < p->pic_cap; i++) free(p->pic[i].w);
    free(p->pic); free(p->done);
    pthread_mutex_destroy(&p->mu); pthread_cond_destroy(&p->cv_work); pthread_cond_destroy(&p->cv_done);
    free(p);
    return MVG_SUCCESS;
}

const char *mvf_parser_last_error(const mvf_parser *p) { return p ? p->err : ""; }

/* run one job: `out` xor `pk` is set */
static int parser_run(mvf_parser *p, const int32_t *indices, int first, int count, const mvf_batch *out, mvf_packed_batch *pk,
                      int32_t *status)
{
    mvf_stream *s = p->s;
    p->rc = MVG_SUCCESS; p->err[0] = 0;
    if (count == 0) return MVG_SUCCESS;
    /* geometry of the call: that of the first requested picture that has any */
    p->W = p->H = 0;
    for (int i = 0; i < count && !p->W; i++) {
        const int idx = indices ? indices[i] : first + i;
        if (idx >= 0 && idx < s->n_idr && s->idr_gen[idx] >= 0) { p->W = s->gens[s->idr_gen[idx]].sps.width_mbs; p->H = s->gens[s->idr_gen[idx]].sps.height_mbs; }
    }
    if (!p->W) { p->W = s->gens[0].sps.width_mbs; p->H = s->gens[0].sps.height_mbs; }
    if (count > p->done_cap) {
        uint8_t *d = realloc(p->done, (size_t)count);
        if (!d) { snprintf(p->err, sizeof p->err, "out of memory"); return MVG_FAILURE; }
        p->done = d; p->done_cap = count;
    }
    memset(p->done, 0, (size_t)count);
    if (pk && count > p->pic_cap) {
        picbuf_t *np = realloc(p->pic, sizeof(picbuf_t) * (size_t)count);
        if (!np) { snprintf(p->err, sizeof p->err, "out of memory"); return MVG_FAILURE; }
        memset(np + p->pic_cap, 0, sizeof(picbuf_t) * (size_t)(count - p->pic_cap));
        p->pic = np; p->pic_cap = count;
    }
    p->indices = indices; p->first = first; p->count = count; p->out = out; p->pk = pk; p->status = status;
    p->strict = status == NULL;
    __atomic_store_n(&p->next, 0, __ATOMIC_RELAXED);

    const int threaded = p->n_workers > 0 && count > 1;
    if (threaded) {
        pthread_mutex_lock(&p->mu);
        p->active = p->n_workers; p->job_seq++;
        pthread_cond_broadcast(&p->cv_work);
        pthread_mutex_unlock(&p->mu);
    } else {
        const int keep = p->n_workers;
        p->n_workers = 0;                   /* no signalling inside work_on_job */
        work_on_job(p, &p->workers[0]);
        p->n_workers = keep;
    }
    int rc = MVG_SUCCESS;
    if (pk) {
        /* the words of the pictures, in picture order, while the workers are still parsing the later ones */
        pk->pic_off[0] = 0;
        for (int i = 0; i < count; i++) {
            int abandoned = 0;      /* all-or-nothing mode: after a failure the pictures not yet claimed never get done */
            if (threaded && !__atomic_load_n(&p->done[i], __ATOMIC_ACQUIRE)) {
                pthread_mutex_lock(&p->mu);
                while (!__atomic_load_n(&p->done[i], __ATOMIC_ACQUIRE) && !(p->strict && p->rc != MVG_SUCCESS))
                    pthread_cond_wait(&p->cv_done, &p->mu);
                abandoned = !__atomic_load_n(&p->done[i], __ATOMIC_ACQUIRE);
                pthread_mutex_unlock(&p->mu);
            } else if (!threaded && !p->done[i]) abandoned = 1;
            if (abandoned) {
                for (int k = i; k < count; k++) pk->pic_off[k + 1] = pk->pic_off[i];
                break;
            }
            const uint64_t at = pk->pic_off[i], n = p->pic[i].n;
            pk->pic_off[i + 1] = at + n;
            if (n && at + n <= pk->words_capacity) memcpy(pk->words + at, p->pic[i].w, (size_t)n * sizeof(uint16_t));
        }
        pk->words_needed = (size_t)pk->pic_off[count];
        if (pk->pic_off[count] > pk->words_capacity) {
            rc = MVG_FAILURE;
            snprintf(p->err, sizeof p->err, "mvf_parse_pictures_packed: %llu words needed, capacity %zu",
                     (unsigned long long)pk->pic_off[count], pk->words_capacity);
        }
    }
    if (threaded) {
        pthread_mutex_lock(&p->mu);
        while (p->active) pthread_cond_wait(&p->cv_done, &p->mu);
        pthread_mutex_unlock(&p->mu);
    }
    if (rc == MVG_SUCCESS && p->strict) rc = p->rc;         /* tolerant mode: per-picture codes are in status[] */
    return rc;
}

static void publish_error(mvf_parser *p)
{
    pthread_mutex_lock(&p->s->err_mu);
    memcpy(p->s->err, p->err, sizeof p->err);
    pthread_mutex_unlock(&p->s->err_mu);
}

int mvf_parser_parse(mvf_parser *p, const int32_t *indices, int first, int count, mvf_batch *out)
{
    if (!p || !out || count < 0) return MVG_FAILURE;
    if (!out->mb_kind || !out->i16_mode || !out->chroma_mode || !out->qp_y || !out->cbp || !out->luma_modes || !out->coeff) {
        snprintf(p->err, sizeof p->err, "mvf_parse_pictures: a batch pointer is NULL");
        publish_error(p);
        return MVG_FAILURE;
    }
    out->n_pics = count;
    const int rc = parser_run(p, indices, first, count, out, NULL, out->status);
    if (p->err[0]) publish_error(p);
    return rc;
}

int mvf_parser_parse_packed(mvf_parser *p, const int32_t *indices, int first, int count, mvf_packed_batch *out)
{
    if (!p || !out || count < 0) return MVG_FAILURE;
    if (!out->mb_kind || !out->i16_mode || !out->chroma_mode || !out->qp_y || !out->luma_modes || !out->nz_blocks ||
        !out->word_off || !out->pic_off || !out->words) {
        snprintf(p->err, sizeof p->err, "mvf_parse_pictures_packed: a batch pointer is NULL");
        publish_error(p);
        return MVG_FAILURE;
    }
    out->n_pics = count;
    out->pic_off[0] = 0;
    out->words_needed = 0;
    const int rc = parser_run(p, indices, first, count, NULL, out, out->status);
    if (p->err[0]) publish_error(p);
    return rc;
}

/* one-shot forms: a parser for the duration of the call */
int mvf_parse_pictures(mvf_stream *s, const int32_t *indices, int first, int count, mvf_batch *out, int n_threads)
{
    if (!s || !out || count < 0) return MVG_FAILURE;
    mvf_parser *p = NULL;
    if (mvf_parser_create(s, n_threads < count ? n_threads : count, &p) != MVG_SUCCESS) return MVG_FAILURE;
    const int rc = mvf_parser_parse(p, indices, first, count, out);
    mvf_parser_destroy(p);
    return rc;
}

int mvf_parse_pictures_packed(mvf_stream *s, const int32_t *indices, int first, int count, mvf_packed_batch *out, int n_threads)
{
    if (!s || !out || count < 0) return MVG_FAILURE;
    mvf_parser *p = NULL;
    if (mvf_parser_create(s, n_threads < count ? n_threads : count, &p) != MVG_SUCCESS) return MVG_FAILURE;
    const int rc = mvf_parser_parse_packed(p, indices, first, count, out);
    mvf_parser_destroy(p);
    return rc;
}
