/* Test helper (built by tests/test_ts_fuzz.py with -fsanitize=address,undefined): open many damaged copies of a valid
 * transport stream with mvf_open_ts(); it must answer SUCCESS / FAILURE / UNSUPPORTED and never touch memory it does
 * not own.  Streams that still open are also run through frame selection and a parse of every picture.
 *
 *   fuzz_ts <file.ts> <rounds> <packet size 188 | 192 | 204>
 *
 * The damage follows the packet structure: continuity counters, transport_error_indicator, pointer_field and
 * section_length of PSI packets, PES_packet_length and PES_header_data_length of PES headers, adaptation_field_length,
 * truncation at and inside packets, and random bytes anywhere. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "mvfront.h"

static unsigned long long rng = 0x9E3779B97F4A7C15ull;
static unsigned rnd(void) { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (unsigned)(rng >> 32); }

static size_t psi[1 << 12], pes[1 << 16], afs[1 << 16], all[1 << 18];
static int n_psi, n_pes, n_afs, n_all;

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
    if (argc < 4) return 2;
    FILE *f = fopen(argv[1], "rb");
    if (!f) return 2;
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    uint8_t *orig = malloc((size_t)n), *buf = malloc((size_t)n);
    if (fread(orig, 1, (size_t)n, f) != (size_t)n) return 2;
    fclose(f);
    const int rounds = atoi(argv[2]);
    const size_t per = (size_t)atoi(argv[3]), lead = per == 192 ? 4 : 0;
    for (size_t p = lead; p + 188 <= (size_t)n && n_all < (1 << 18); p += per) {      /* the packets of the valid file */
        const uint8_t *k = orig + p;
        if (k[0] != 0x47) { fprintf(stderr, "not a muxer file\n"); return 2; }
        all[n_all++] = p;
        const int pid = (k[1] & 0x1F) << 8 | k[2], pusi = k[1] & 0x40, afc = k[3] >> 4 & 3;
        if (afc & 2 && n_afs < (1 << 16)) afs[n_afs++] = p;
        const size_t o = afc & 2 ? 5 + (size_t)k[4] : 4;
        if (!pusi || o + 9 > 188) continue;
        if (pid < 0x100 || pid == 0x1000 || pid == 0x1001) { if (n_psi < (1 << 12)) psi[n_psi++] = p + o; }
        else if (!k[o] && !k[o + 1] && k[o + 2] == 1 && n_pes < (1 << 16)) pes[n_pes++] = p + o;
    }
    if (n_all < 10 || !n_psi || !n_pes || !n_afs) { fprintf(stderr, "not a muxer file\n"); return 2; }
    int opened = 0, parsed = 0, by_rc[3] = {0, 0, 0};
    for (int r = 0; r < rounds; r++) {
        memcpy(buf, orig, (size_t)n);
        size_t len = (size_t)n;
        const int kind = r % 8;
        for (int rep = 0; rep < 1 + (r / 8) % 3; rep++) {
            if (kind == 0) {                                    /* continuity counters */
                uint8_t *k = buf + all[rnd() % n_all];
                k[3] = (uint8_t)((k[3] & 0xF0) | (rnd() & 15));
            } else if (kind == 1) {                             /* transport_error_indicator */
                buf[all[rnd() % n_all] + 1] |= 0x80;
            } else if (kind == 2) {                             /* pointer_field */
                buf[psi[rnd() % n_psi]] = (uint8_t)(rnd() % 3 == 0 ? 0xFF : rnd() % 190);
            } else if (kind == 3) {                             /* section_length */
                uint8_t *q = buf + psi[rnd() % n_psi];
                q += 1 + q[0];
                if (q + 3 <= buf + len) { q[1] = (uint8_t)((q[1] & 0xF0) | (rnd() & 15)); q[2] = (uint8_t)rnd(); }
            } else if (kind == 4) {                             /* PES_packet_length, PES_header_data_length */
                uint8_t *q = buf + pes[rnd() % n_pes];
                if (rnd() & 1) { const unsigned v = rnd() % 4 ? rnd() % 400 : 0xFFFF; q[4] = (uint8_t)(v >> 8); q[5] = (uint8_t)v; }
                else q[8] = (uint8_t)(rnd() % 4 ? rnd() % 200 : 255);
            } else if (kind == 5) {                             /* adaptation_field_length */
                buf[afs[rnd() % n_afs] + 4] = (uint8_t)(rnd() % 3 ? rnd() % 190 : 183 + rnd() % 73);
            } else if (kind == 6) {                             /* truncation at and inside packets */
                len = all[(r / 8) % n_all] + (rnd() & 1 ? 0 : rnd() % 188);
                if (len == 0) len = 1;
            } else {                                            /* random bytes */
                for (int k = 0; k < 1 + (int)(rnd() % 8); k++) buf[rnd() % len] = (uint8_t)rnd();
            }
        }
        uint8_t *exact = malloc(len);                       /* exact-size copy: the sanitizer sees any read past the file */
        memcpy(exact, buf, len);
        mvf_stream *s = NULL;
        const int rc = mvf_open_ts(exact, len, &s);
        free(exact);                                        /* the stream keeps its own copy */
        if (rc != MVG_SUCCESS && rc != MVG_FAILURE && rc != MVG_UNSUPPORTED) { fprintf(stderr, "round %d: return code %d\n", r, rc); return 1; }
        by_rc[rc + 1]++;
        if (rc == MVG_SUCCESS) { opened++; exercise(s, r, &parsed); mvf_close(s); }
        else if (!mvf_last_error(NULL)[0]) { fprintf(stderr, "round %d: refused without a message\n", r); return 1; }
    }
    free(orig); free(buf);
    printf("rounds=%d opened=%d parsed=%d failure=%d unsupported=%d packets=%d\n", rounds, opened, parsed, by_rc[1], by_rc[0], n_all);
    return 0;
}
