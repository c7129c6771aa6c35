/* Test helper (built by tests/test_mp4_fuzz.py with -fsanitize=address,undefined): open many damaged copies of a
 * valid MP4 file with mvf_open_mp4(); it must answer SUCCESS / FAILURE / UNSUPPORTED and never touch memory it does
 * not own.  Files that still open are also run through frame selection and a parse of every picture.
 *
 *   fuzz_mp4 <file.mp4> <rounds> <NAL length size>
 *
 * The damage follows the box structure: box sizes set to 0, 1, 7 or to what is left of the parent +- 1, entry counts
 * set to 0, 1 or 2^32 - 1, chunk offsets past the end of the file, bit flips in NAL length fields, truncation at every
 * box boundary, and random bytes in moov.  NAL length fields are found by walking mdat as one run of length-prefixed
 * NAL units, which is how tests/mp4_mux.py lays out a file without audio or chunk gaps. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "mvfront.h"

static unsigned long long rng = 0x9E3779B97F4A7C15ull;
static unsigned rnd(void) { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (unsigned)(rng >> 32); }

static uint32_t rd32(const uint8_t *p) { return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | p[3]; }
static void wr32(uint8_t *p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; }

typedef struct { size_t off, end, parent_end; uint32_t type; } box_t;
static box_t boxes[4096];
static int n_boxes;
static size_t lenfields[1 << 16];
static int n_lenfields;
static size_t moov_off, moov_end;

static int is_container(uint32_t t)
{
    static const char *const c[] = {"moov", "trak", "mdia", "minf", "stbl", "dinf"};
    for (int i = 0; i < 6; i++) if (t == rd32((const uint8_t *)c[i])) return 1;
    return 0;
}

/* the boxes of the valid file (32-bit sizes inside moov, as the muxer writes them) */
static void walk(const uint8_t *d, size_t pos, size_t end, int len_size)
{
    while (pos + 8 <= end && n_boxes < 4096) {
        size_t size = rd32(d + pos), hdr = 8;
        const uint32_t t = rd32(d + pos + 4);
        if (size == 1) { size = (size_t)rd32(d + pos + 8) << 32 | rd32(d + pos + 12); hdr = 16; }
        if (size < hdr || size > end - pos) return;
        boxes[n_boxes++] = (box_t){pos, pos + size, end, t};
        if (is_container(t)) walk(d, pos + hdr, pos + size, len_size);
        if (t == rd32((const uint8_t *)"stsd") && size > 16) walk(d, pos + 16, pos + size, len_size);
        if ((t == rd32((const uint8_t *)"avc1") || t == rd32((const uint8_t *)"avc3")) && size > hdr + 78)
            walk(d, pos + hdr + 78, pos + size, len_size);
        if (t == rd32((const uint8_t *)"moov")) { moov_off = pos; moov_end = pos + size; }
        if (t == rd32((const uint8_t *)"mdat"))
            for (size_t p = pos + hdr; p + (size_t)len_size <= pos + size && n_lenfields < (1 << 16); ) {
                size_t n = 0;
                for (int j = 0; j < len_size; j++) n = n << 8 | d[p + j];
                lenfields[n_lenfields++] = p;
                p += (size_t)len_size + n;
            }
        pos += size;
    }
}

/* offset of the entry count of a full box with one, or 0 */
static size_t count_field(const box_t *b)
{
    static const char *const c[] = {"stsd", "stsc", "stco", "co64", "stss", "stts"};
    if (b->type == rd32((const uint8_t *)"stsz")) return b->off + 16;
    for (int i = 0; i < 6; i++) if (b->type == rd32((const uint8_t *)c[i])) return b->off + 12;
    return 0;
}

int main(int argc, char **argv)
{
    if (argc < 4) return 2;
    FILE *f = fopen(argv[1], "rb");
    if (!f) return 2;
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    uint8_t *orig = malloc((size_t)n), *buf = malloc((size_t)n);
    if (fread(orig, 1, (size_t)n, f) != (size_t)n) return 2;
    fclose(f);
    const int rounds = atoi(argv[2]), len_size = atoi(argv[3]);
    walk(orig, 0, (size_t)n, len_size);
    int n_count = 0, n_chunk = 0;
    for (int i = 0; i < n_boxes; i++) {
        n_count += count_field(&boxes[i]) != 0;
        n_chunk += boxes[i].type == rd32((const uint8_t *)"stco") || boxes[i].type == rd32((const uint8_t *)"co64");
    }
    if (n_boxes < 10 || !n_count || !n_chunk || !n_lenfields || !moov_end) { fprintf(stderr, "not a muxer file\n"); return 2; }
    int opened = 0, parsed = 0, by_rc[3] = {0, 0, 0};
    for (int r = 0; r < rounds; r++) {
        memcpy(buf, orig, (size_t)n);
        size_t len = (size_t)n;
        const int kind = r % 6;
        for (int rep = 0; rep < 1 + (r / 6) % 2; rep++) {
            if (kind == 0) {                                    /* box sizes */
                const box_t *b = &boxes[rnd() % n_boxes];
                static const uint32_t fixed[3] = {0, 1, 7};
                const unsigned k = rnd() % 5;
                const uint32_t v = k < 3 ? fixed[k] : (uint32_t)(b->parent_end - b->off) + (k == 3 ? 1u : (uint32_t)-1);
                wr32(buf + b->off, v);
            } else if (kind == 1) {                             /* entry counts */
                const box_t *b;
                do b = &boxes[rnd() % n_boxes]; while (!count_field(b));
                static const uint32_t vals[3] = {0, 1, 0xFFFFFFFFu};
                wr32(buf + count_field(b), vals[rnd() % 3]);
            } else if (kind == 2) {                             /* chunk offsets past the end of the file */
                const box_t *b;
                do b = &boxes[rnd() % n_boxes]; while (b->type != rd32((const uint8_t *)"stco") && b->type != rd32((const uint8_t *)"co64"));
                const size_t w = b->type == rd32((const uint8_t *)"co64") ? 8 : 4, cnt = (b->end - b->off - 16) / w;
                if (cnt) {
                    uint8_t *e = buf + b->off + 16 + w * (rnd() % cnt);
                    const uint32_t v = rnd() & 1 ? (uint32_t)len + rnd() % 4096 : 0xFFFFFFFFu - rnd() % 16;
                    if (w == 8) { wr32(e, rnd() & 1 ? 0 : 1); wr32(e + 4, v); } else wr32(e, v);
                }
            } else if (kind == 3) {                             /* NAL length fields */
                const size_t p = lenfields[rnd() % n_lenfields];
                buf[p + rnd() % (unsigned)len_size] ^= (uint8_t)(1u << (rnd() % 8));
            } else if (kind == 4) {                             /* truncation at box boundaries, each in turn */
                const box_t *b = &boxes[(r / 6) % n_boxes];
                len = (r / 6 / n_boxes) % 2 ? b->end : b->off;
                if (len == 0) len = 1;
            } else {                                            /* random bytes in moov */
                for (int k = 0; k < 1 + (int)(rnd() % 4); k++) buf[moov_off + rnd() % (moov_end - moov_off)] = (uint8_t)rnd();
            }
        }
        uint8_t *exact = malloc(len);                       /* exact-size copy: the sanitizer sees any read past the file */
        memcpy(exact, buf, len);
        mvf_stream *s = NULL;
        const int rc = mvf_open_mp4(exact, len, &s);
        if (rc != MVG_SUCCESS && rc != MVG_FAILURE && rc != MVG_UNSUPPORTED) { fprintf(stderr, "round %d: return code %d\n", r, rc); return 1; }
        by_rc[rc + 1]++;
        if (rc == MVG_SUCCESS) {
            opened++;
            mvf_info in;
            mvf_get_info(s, &in);
            const int P = in.n_idr;
            int32_t *sel = malloc(sizeof(int32_t) * (size_t)(P + 8)), *idx = malloc(sizeof(int32_t) * (size_t)(P + 1));
            int32_t *status = malloc(sizeof(int32_t) * (size_t)(P + 1));
            for (int mode = 0; mode < 3; mode++) mvf_select_idr(s, P + 3, mode, sel);
            for (int g = 0; g < mvf_generation_count(s); g++) {         /* every picture, one call per generation */
                mvf_info gi;
                mvf_get_generation_info(s, g, &gi);
                int cnt = 0;
                for (int i = 0; i < P; i++) if (mvf_picture_generation(s, i) == g) idx[cnt++] = i;
                if (!cnt || gi.width_mbs * gi.height_mbs > 64 * 64) continue;
                const size_t N = (size_t)gi.width_mbs * gi.height_mbs * (size_t)cnt;
                mvf_batch b;
                memset(&b, 0, sizeof b);
                b.mb_kind = malloc(N); b.i16_mode = malloc(N); b.chroma_mode = malloc(N); b.qp_y = malloc(N);
                b.cbp = malloc(N); b.luma_modes = malloc(N * 16); b.coeff = malloc(N * 768); b.status = status;
                mvf_parse_pictures(s, idx, 0, cnt, &b, 1 + r % 3);
                for (int i = 0; i < cnt; i++) parsed += status[i] == MVG_SUCCESS;
                free(b.mb_kind); free(b.i16_mode); free(b.chroma_mode); free(b.qp_y); free(b.cbp); free(b.luma_modes); free(b.coeff);
            }
            free(sel); free(idx); free(status);
            mvf_close(s);
        } else if (!mvf_last_error(NULL)[0]) { fprintf(stderr, "round %d: refused without a message\n", r); return 1; }
        free(exact);
    }
    free(orig); free(buf);
    printf("rounds=%d opened=%d parsed=%d failure=%d unsupported=%d boxes=%d length_fields=%d\n",
           rounds, opened, parsed, by_rc[1], by_rc[0], n_boxes, n_lenfields);
    return 0;
}
