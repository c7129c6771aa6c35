/* Test helper (built by tests/test_mkv_fuzz.py with -fsanitize=address,undefined): open many damaged copies of a valid
 * Matroska file with mvf_open_mkv(); it must answer SUCCESS / FAILURE / UNSUPPORTED and never touch memory it does not
 * own.  Files that still open are also run through frame selection and a parse of every picture.
 *
 *   fuzz_mkv <file.mkv> <rounds>
 *
 * The damage follows the EBML structure: the width marker and the value of element sizes (unknown sizes included),
 * element IDs, lace counts and lace sizes of blocks, the bytes of CodecPrivate, NAL length fields, truncation at
 * every element boundary, and random bytes. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "mvfront.h"

static unsigned long long rng = 0x9E3779B97F4A7C15ull;
static unsigned rnd(void) { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (unsigned)(rng >> 32); }

typedef struct { size_t id_at, size_at, body, end; uint32_t id; } el_t;
static el_t els[1 << 14];
static int n_els;
static size_t blocks[1 << 12];
static int n_blocks;
static size_t priv_at, priv_end;

static int is_master(uint32_t id)
{
    return id == 0x1A45DFA3u || id == 0x18538067u || id == 0x114D9B74u || id == 0x4DBBu || id == 0x1549A966u ||
           id == 0x1654AE6Bu || id == 0xAEu || id == 0x1F43B675u || id == 0xA0u || id == 0x1C53BB6Bu || id == 0xBBu ||
           id == 0xB7u || id == 0xE0u || id == 0xE1u || id == 0x6D80u || id == 0x6240u || id == 0x5034u;
}

static void walk(const uint8_t *d, size_t pos, size_t end)
{
    while (pos < end && n_els < (1 << 14)) {
        const size_t id_at = pos;
        int w = 1;
        while (w <= 4 && !(d[pos] & (0x80 >> (w - 1)))) w++;
        uint32_t id = 0;
        for (int i = 0; i < w; i++) id = id << 8 | d[pos + i];
        pos += (size_t)w;
        const size_t size_at = pos;
        int sw = 1;
        while (sw <= 8 && !(d[pos] & (0x80 >> (sw - 1)))) sw++;
        unsigned long long size = d[pos] & (0xFFu >> sw);
        int ones = size == (0xFFu >> sw);
        for (int i = 1; i < sw; i++) { size = size << 8 | d[pos + i]; ones &= d[pos + i] == 0xFF; }
        pos += (size_t)sw;
        const size_t e = ones ? end : pos + size;
        els[n_els++] = (el_t){id_at, size_at, pos, e, id};
        if (id == 0xA3u || id == 0xA1u) { if (n_blocks < (1 << 12)) blocks[n_blocks++] = pos; }
        if (id == 0x63A2u) { priv_at = pos; priv_end = e; }
        if (is_master(id)) walk(d, pos, e);
        if (ones && id == 0x1F43B675u) return;      /* an unknown-size Cluster: its children were walked as its siblings */
        pos = e;
    }
}

static void exercise(mvf_stream *s, int r, int *parsed)
{
    mvf_info in;
    mvf_get_info(s, &in);
    const int P = in.n_idr;
    int32_t *sel = malloc(sizeof(int32_t) * (size_t)(P + 8)), *idx = malloc(sizeof(int32_t) * (size_t)(P + 1));
    int32_t *status = malloc(sizeof(int32_t) * (size_t)(P + 1));
    for (int mode = 0; mode < 3; mode++) mvf_select_idr(s, P + 3, mode, sel);
    for (int g = 0; g < mvf_generation_count(s); g++) {
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
        for (int i = 0; i < cnt; i++) *parsed += status[i] == MVG_SUCCESS;
        free(b.mb_kind); free(b.i16_mode); free(b.chroma_mode); free(b.qp_y); free(b.cbp); free(b.luma_modes); free(b.coeff);
    }
    free(sel); free(idx); free(status);
}

int main(int argc, char **argv)
{
    if (argc < 3) return 2;
    FILE *f = fopen(argv[1], "rb");
    if (!f) return 2;
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    uint8_t *orig = malloc((size_t)n), *buf = malloc((size_t)n);
    if (fread(orig, 1, (size_t)n, f) != (size_t)n) return 2;
    fclose(f);
    const int rounds = atoi(argv[2]);
    walk(orig, 0, (size_t)n);
    if (n_els < 20 || !n_blocks || !priv_end) { fprintf(stderr, "not a muxer file\n"); return 2; }
    int opened = 0, parsed = 0, by_rc[3] = {0, 0, 0};
    for (int r = 0; r < rounds; r++) {
        memcpy(buf, orig, (size_t)n);
        size_t len = (size_t)n;
        const int kind = r % 7;
        for (int rep = 0; rep < 1 + (r / 7) % 2; rep++) {
            const el_t *e = &els[rnd() % n_els];
            if (kind == 0) {                                    /* vint width markers */
                buf[e->size_at] = (uint8_t)(rnd() % 4 == 0 ? 0 : buf[e->size_at] >> (1 + rnd() % 3) | (rnd() & 1 ? 0x80 : 0));
            } else if (kind == 1) {                             /* size values, unknown sizes */
                const unsigned k = rnd() % 4;
                buf[e->size_at] = k == 0 ? 0xFF : k == 1 ? 0x80 : (uint8_t)(buf[e->size_at] ^ (1u << (rnd() % 7)));
                if (k == 3 && e->body - e->size_at > 1) buf[e->size_at + 1 + rnd() % (e->body - e->size_at - 1)] ^= (uint8_t)(1u << (rnd() % 8));
            } else if (kind == 2) {                             /* IDs */
                buf[e->id_at + rnd() % (e->size_at - e->id_at)] ^= (uint8_t)(1u << (rnd() % 8));
            } else if (kind == 3) {                             /* lace flags, counts and sizes */
                uint8_t *b = buf + blocks[rnd() % n_blocks];
                const unsigned k = rnd() % 3;
                if (k == 0) b[3] = (uint8_t)((b[3] & ~6u) | (rnd() & 6));
                else if (k == 1) b[4] = (uint8_t)rnd();
                else b[5 + rnd() % 3] = (uint8_t)rnd();
            } else if (kind == 4) {                             /* CodecPrivate */
                buf[priv_at + rnd() % (priv_end - priv_at)] = (uint8_t)(rnd() % 3 ? rnd() : 0xFF);
            } else if (kind == 5) {                             /* truncation at element boundaries, each in turn */
                const el_t *t = &els[(r / 7) % n_els];
                len = (r / 7 / n_els) % 2 ? t->end : t->id_at;
                if (len == 0 || len > (size_t)n) len = 1;
            } else {                                            /* random bytes */
                for (int k = 0; k < 1 + (int)(rnd() % 6); k++) buf[rnd() % len] = (uint8_t)rnd();
            }
        }
        uint8_t *exact = malloc(len);                       /* exact-size copy: the sanitizer sees any read past the file */
        memcpy(exact, buf, len);
        mvf_stream *s = NULL;
        const int rc = mvf_open_mkv(exact, len, &s);
        if (rc != MVG_SUCCESS && rc != MVG_FAILURE && rc != MVG_UNSUPPORTED) { fprintf(stderr, "round %d: return code %d\n", r, rc); return 1; }
        by_rc[rc + 1]++;
        if (rc == MVG_SUCCESS) { opened++; exercise(s, r, &parsed); mvf_close(s); }
        else if (!mvf_last_error(NULL)[0]) { fprintf(stderr, "round %d: refused without a message\n", r); return 1; }
        free(exact);
    }
    free(orig); free(buf);
    printf("rounds=%d opened=%d parsed=%d failure=%d unsupported=%d elements=%d blocks=%d\n",
           rounds, opened, parsed, by_rc[1], by_rc[0], n_els, n_blocks);
    return 0;
}
