/*
 * mv_thumbcore.c -- thumbnail extraction over the GPU path, shared by the mv_thumbnailer CLI and by the
 * drop-in public API (minivideo_shim.c):
 *
 * Annex-B bytes -> mvf_open_annexb() (MP4 / QuickTime, transport streams, Matroska: mvf_open_mp4() / _ts() / _mkv(),
 * picked by mvt_container()) -> mvf_select_idr() (demuxer/filter.c semantics) ->
 * mvf_parse_pictures_packed() (threaded CAVLC, packed levels) -> mvg_decode_host_packed() (pinned copies +
 * kernels 0-4) -> picture
 * files named like export_idr() names them (export.c:627-642,:704-705): <input base name>[_<k>].<ext>
 * with k counting exported pictures when more than one was requested.  File contents are byte-identical
 * to the reference's: planar I420 (export.c:100-151), its "super sampled" planar 4:4:4 (export.c:197-330),
 * 24-bit bottom-up BMP, run-length TGA and PNG as stb_image_write v1.01 produces them (export.c:535-539,
 * :566-570,:597-601; PNG in mv_png.c).  Parsing, GPU work and file encoding of successive batches overlap.
 * No CPU fallback: without a CUDA device mvt_extract() fails.
 */
#include <limits.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include "mvfront.h"
#include "mvgpu.h"
#include "mv_thumbcore.h"
#include "mv_png.h"

#include <time.h>
/* MVT_TIMING=1 in the environment: stage times of every feeder on stderr */
static double now_s(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }


/* ---- picture files, built in memory and written with one fwrite() ------------------------------------ */

static int write_raw(const char *path, const uint8_t *data, size_t n)
{
    FILE *f = fopen(path, "wb");
    if (!f) return 0;
    size_t w = fwrite(data, 1, n, f);
    return fclose(f) == 0 && w == n;
}

static uint8_t *le16(uint8_t *o, unsigned v) { o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); return o + 2; }
static uint8_t *le32(uint8_t *o, unsigned v) { o = le16(o, v & 0xffff); return le16(o, v >> 16); }

/* 24-bit uncompressed BMP: 14-byte file header, 40-byte BITMAPINFOHEADER, rows bottom-up, BGR,
 * padded to 4 bytes -- the layout stbi_write_bmp() produces for 3 components */
static int write_bmp(const char *path, const uint8_t *rgb, int w, int h)
{
    const int pad = (4 - (w * 3) % 4) % 4;
    const size_t line = (size_t)w * 3 + (size_t)pad, total = 54 + line * (size_t)h;
    uint8_t *buf = malloc(total), *o = buf;
    if (!buf) return 0;
    *o++ = 'B'; *o++ = 'M';
    o = le32(o, (unsigned)total); o = le16(o, 0); o = le16(o, 0); o = le32(o, 54);
    o = le32(o, 40); o = le32(o, (unsigned)w); o = le32(o, (unsigned)h); o = le16(o, 1); o = le16(o, 24);
    for (int i = 0; i < 6; i++) o = le32(o, 0);
    for (int y = h - 1; y >= 0; y--) {
        const uint8_t *src = rgb + (size_t)y * w * 3;
        for (int x = 0; x < w; x++) { o[3 * x] = src[3 * x + 2]; o[3 * x + 1] = src[3 * x + 1]; o[3 * x + 2] = src[3 * x]; }
        memset(o + w * 3, 0, (size_t)pad);
        o += line;
    }
    int ok = write_raw(path, buf, total);
    free(buf);
    return ok;
}

static int same_px(const uint8_t *a, const uint8_t *b) { return a[0] == b[0] && a[1] == b[1] && a[2] == b[2]; }
static uint8_t *put_bgr(uint8_t *o, const uint8_t *p) { o[0] = p[2]; o[1] = p[1]; o[2] = p[0]; return o + 3; }

/* run-length true-colour TGA (image type 10), origin bottom-left, BGR.  Packets are formed the way
 * stbi_write_tga() forms them so the files compare equal: a raw packet keeps growing while pixel k
 * differs from pixel k-2 and gives its last pixel back when they match; a run packet grows while
 * pixels equal its first one; both stop at 128 pixels. */
static int write_tga(const char *path, const uint8_t *rgb, int w, int h)
{
    /* worst case: every packet is a raw one of a single pixel (1 + 3 bytes) */
    uint8_t *buf = malloc(18 + (size_t)w * h * 4), *o = buf;
    if (!buf) return 0;
    *o++ = 0; *o++ = 0; *o++ = 10;
    o = le16(o, 0); o = le16(o, 0); *o++ = 0;
    o = le16(o, 0); o = le16(o, 0); o = le16(o, (unsigned)w); o = le16(o, (unsigned)h);
    *o++ = 24; *o++ = 0;
    for (int y = h - 1; y >= 0; y--) {
        const uint8_t *row = rgb + (size_t)y * w * 3;
        int len;
        for (int i = 0; i < w; i += len) {
            const uint8_t *first = row + 3 * i;
            int is_run = 0;
            len = 1;
            if (i < w - 1) {
                len = 2;
                is_run = same_px(first, first + 3);
                if (is_run) {
                    for (int k = i + 2; k < w && len < 128 && same_px(first, row + 3 * k); k++) len++;
                } else {
                    for (int k = i + 2; k < w && len < 128; k++) {
                        if (same_px(row + 3 * (k - 2), row + 3 * k)) { len--; break; }
                        len++;
                    }
                }
            }
            if (is_run) { *o++ = (uint8_t)(len + 127); o = put_bgr(o, first); }
            else { *o++ = (uint8_t)(len - 1); for (int k = 0; k < len; k++) o = put_bgr(o, first + 3 * k); }
        }
    }
    int ok = write_raw(path, buf, (size_t)(o - buf));
    free(buf);
    return ok;
}

static int write_png(const char *path, const uint8_t *rgb, int w, int h)
{
    size_t n = 0;
    uint8_t *png = mvt_png_encode(rgb, w, h, &n);
    if (!png) return 0;
    int ok = write_raw(path, png, n);
    free(png);
    return ok;
}

/* planar 4:4:4 as export_idr_yuv444() writes it (export.c:197-330): the luma plane, then Cb and Cr "super
 * sampled" -- each chroma sample goes to the left, right and lower-left positions of its 2x2 cell and the
 * lower-right one keeps the 0 of the calloc()ed plane (export.c:268-269 never writes [i + img_width + 1]) */
static int write_yuv444(const char *path, const uint8_t *i420, int w, int h)
{
    const size_t plane = (size_t)w * h;
    uint8_t *buf = calloc(3, plane);
    if (!buf) return 0;
    memcpy(buf, i420, plane);
    for (int c = 0; c < 2; c++) {
        const uint8_t *src = i420 + plane + (size_t)c * (plane / 4);
        uint8_t *dst = buf + plane * (size_t)(1 + c);
        for (int y = 0; y < h / 2; y++) {
            uint8_t *r0 = dst + (size_t)(2 * y) * w, *r1 = r0 + w;
            for (int x = 0; x < w / 2; x++) { uint8_t v = src[(size_t)y * (w / 2) + x]; r0[2 * x] = v; r0[2 * x + 1] = v; r1[2 * x] = v; }
        }
    }
    int ok = write_raw(path, buf, 3 * plane);
    free(buf);
    return ok;
}

/* one picture file from host pixels (RGB24 top-down; MVT_YUV420 / MVT_YUV444: planar I420): the writers above behind
 * one entry point, so that tests can pin them against the reference's writers without a GPU */
int mvt_write_image(const char *path, int fmt, const uint8_t *pixels, int w, int h)
{
    if (!path || !pixels || w < 1 || h < 1) return 0;
    switch (fmt) {
    case MVT_YUV420: return write_raw(path, pixels, (size_t)w * h * 3 / 2);
    case MVT_YUV444: return write_yuv444(path, pixels, w, h);
    case MVT_BMP:    return write_bmp(path, pixels, w, h);
    case MVT_TGA:    return write_tga(path, pixels, w, h);
    case MVT_PNG:    return write_png(path, pixels, w, h);
    default:         return 0;
    }
}

static const char *const file_ext[] = {"yuv", "bmp", "tga", "png", "yuv"};
static int fmt_is_yuv(int fmt) { return fmt == MVT_YUV420 || fmt == MVT_YUV444; }

/* ---- the job: which pictures, in which order, under which number ---------------------------------------
 * Candidates are the selected IDR pictures in export order.  The reference decodes sample after sample, counts a
 * picture that fails (h264.c:103-109) and goes on; the export number of a picture is the count of pictures decoded
 * before it (export.c:630 uses idrCounter).  Every mode hands the decoder exactly the selected samples
 * (filter.c:88-92, :140-186): a picture that fails is not replaced by a later one (checked against the reference CLI
 * in tests/test_thumbnailer.py).  More than 64 errors in a row end the run (h264.c:181).
 * Batches are dealt to the feeders in candidate order and never cross
 * a parameter generation (mvfront.h); the number of a picture is known once every earlier batch has been parsed. */
typedef struct { int first, cnt, gen, parsed, n_ok; } batchrec_t;

typedef struct {
    mvf_stream *st; const int32_t *cand; int n_cand, batch;
    pthread_mutex_t mu; pthread_cond_t cv;
    int next_cand, n_fail_known, n_unparsed, failed;
    batchrec_t *rec; int n_rec, cap_rec;
    int8_t *ok;                     /* per candidate: 1 decoded, 0 failed (valid once its batch is parsed) */
    int seq_done, run_errors;       /* batches [0, seq_done) are parsed; failures in a row at that point */
} job_t;

/* next batch for a feeder; 0 when there is nothing left (or the job failed) */
static int job_take(job_t *j, int *seq)
{
    pthread_mutex_lock(&j->mu);
    for (;;) {
        if (j->failed) break;
        const int limit = j->n_cand;
        if (j->next_cand < limit) {
            if (j->n_rec == j->cap_rec) {
                const int cap = j->cap_rec ? 2 * j->cap_rec : 64;
                batchrec_t *nr = realloc(j->rec, sizeof *nr * (size_t)cap);
                if (!nr) { j->failed = 1; break; }
                j->rec = nr; j->cap_rec = cap;
            }
            batchrec_t *r = &j->rec[j->n_rec];
            r->first = j->next_cand; r->parsed = 0; r->n_ok = 0;
            r->gen = mvf_picture_generation(j->st, j->cand[r->first]);
            int cnt = 1;
            while (cnt < j->batch && r->first + cnt < limit) {
                const int g = mvf_picture_generation(j->st, j->cand[r->first + cnt]);
                if (g >= 0 && r->gen >= 0 && g != r->gen) break;      /* a new SPS/PPS pair: next batch */
                if (r->gen < 0) r->gen = g;
                cnt++;
            }
            r->cnt = cnt;
            j->next_cand += cnt; j->n_unparsed++;
            *seq = j->n_rec++;
            pthread_mutex_unlock(&j->mu);
            return 1;
        }
        break;
    }
    pthread_mutex_unlock(&j->mu);
    return 0;
}

static void job_parsed(job_t *j, int seq, const int32_t *status)
{
    pthread_mutex_lock(&j->mu);
    batchrec_t *r = &j->rec[seq];
    for (int k = 0; k < r->cnt; k++) {
        j->ok[r->first + k] = status[k] == MVG_SUCCESS;
        if (status[k] == MVG_SUCCESS) r->n_ok++; else j->n_fail_known++;
    }
    r->parsed = 1; j->n_unparsed--;
    while (j->seq_done < j->n_rec && j->rec[j->seq_done].parsed) {      /* errors in a row, in candidate order */
        const batchrec_t *q = &j->rec[j->seq_done++];
        for (int k = 0; k < q->cnt; k++) {
            j->run_errors = j->ok[q->first + k] ? 0 : j->run_errors + 1;
            if (j->run_errors > 64 && !j->failed) { fprintf(stderr, "mvt_extract: more than 64 pictures in a row failed, giving up (h264.c:181)\n"); j->failed = 1; }
        }
    }
    pthread_cond_broadcast(&j->cv);
    pthread_mutex_unlock(&j->mu);
}

/* export number of the first picture of batch `seq`: pictures decoded in all earlier batches; -1 when the job failed */
static int job_number(job_t *j, int seq)
{
    pthread_mutex_lock(&j->mu);
    while (j->seq_done < seq && !j->failed) pthread_cond_wait(&j->cv, &j->mu);
    int n = 0;
    for (int q = 0; q < seq && q < j->n_rec; q++) n += j->rec[q].n_ok;
    const int bad = j->failed && j->seq_done < seq;
    pthread_mutex_unlock(&j->mu);
    return bad ? -1 : n;
}

static void job_fail(job_t *j) { pthread_mutex_lock(&j->mu); j->failed = 1; pthread_cond_broadcast(&j->cv); pthread_mutex_unlock(&j->mu); }

/* ---- one feeder per GPU -------------------------------------------------------------------------------
 * (SURVEY.md section 8e) its own context, pinned buffers, parser and helper threads; it takes batches from the job,
 * no data crosses GPUs.  Inside a feeder three stages run concurrently over two buffer sets: CAVLC parsing of batch
 * k+1 (parser thread, a persistent mvf_parser with `threads` workers), GPU reconstruction of batch k (this thread),
 * file encoding + writing of batch k-1 (writer thread, `threads` workers). */
typedef struct {
    job_t *job; mvf_stream *st; const mvf_info *gens; int n_gens, max_w, max_h;
    const char *base, *outdir; int fmt, scale, device, threads, batch, numbered;
    int exported, rc;
} feeder_t;

enum { SLOT_FREE, SLOT_PARSED, SLOT_DECODED };

typedef struct {
    mvf_packed_batch pb; uint8_t *out; int32_t *status;
    int state, seq, first, cnt, gen, n_ok;
    size_t pic_bytes; int ow, oh;       /* of this batch's generation */
} slot_t;

typedef struct {
    feeder_t *f;
    slot_t slot[2];
    pthread_mutex_t mu; pthread_cond_t cv;
    int failed;                         /* any stage: stop everything */
    int final;                          /* batches this feeder got in all, -1 while the parser is still taking them */
    /* writer workers */
    const slot_t *wslot; int wnext, wexported;
    int wnumber[256];                   /* per picture of the slot: export number, -1 = not decoded (batch <= 256) */
} pipe_t;

static void pipe_fail(pipe_t *p)
{
    pthread_mutex_lock(&p->mu); p->failed = 1; pthread_cond_broadcast(&p->cv); pthread_mutex_unlock(&p->mu);
    job_fail(p->f->job);
}

/* wait until the slot of this feeder's k-th batch reaches `state`: 1 = it has, 0 = the pipeline failed or there is no
 * k-th batch (stages work through the batches in order over two slots, so the slot can only belong to batch k) */
static int pipe_wait(pipe_t *p, int k, int state)
{
    slot_t *s = &p->slot[k & 1];
    pthread_mutex_lock(&p->mu);
    while (s->state != state && !p->failed && !(p->final >= 0 && k >= p->final)) pthread_cond_wait(&p->cv, &p->mu);
    const int ok = !p->failed && s->state == state && !(p->final >= 0 && k >= p->final);
    pthread_mutex_unlock(&p->mu);
    return ok;
}

static void pipe_set(pipe_t *p, slot_t *s, int state)
{
    pthread_mutex_lock(&p->mu); s->state = state; pthread_cond_broadcast(&p->cv); pthread_mutex_unlock(&p->mu);
}

/* pinned words buffer of a slot: grown when a batch needs more than was guessed (a parsed picture needs about a
 * fifth of the worst case, so the worst case is not what gets pinned: pinning costs about a second per GB) */
static int slot_words(mvf_packed_batch *pb, size_t words)
{
    if (words <= pb->words_capacity) return 1;
    uint16_t *nw = mvg_host_alloc(words * sizeof(uint16_t));
    if (!nw) return 0;
    mvg_host_free(pb->words);
    pb->words = nw; pb->words_capacity = words;
    return 1;
}

static void *parser_main(void *arg)
{
    pipe_t *p = arg; feeder_t *f = p->f;
    mvf_parser *ps = NULL;
    if (mvf_parser_create(f->st, f->threads, &ps) != MVG_SUCCESS) {
        fprintf(stderr, "mvt_extract: %s\n", mvf_last_error(f->st));
        pipe_fail(p);
        return NULL;
    }
    int k = 0, seq;
    for (; job_take(f->job, &seq); k++) {
        slot_t *s = &p->slot[k & 1];
        if (!pipe_wait(p, k, SLOT_FREE)) break;
        pthread_mutex_lock(&f->job->mu);                /* rec[] may move (realloc) under the job mutex */
        const batchrec_t rr = f->job->rec[seq];
        pthread_mutex_unlock(&f->job->mu);
        s->seq = seq; s->first = rr.first; s->cnt = rr.cnt; s->gen = rr.gen < 0 ? 0 : rr.gen;
        const mvf_info *gi = &f->gens[s->gen];
        const int W = 16 * gi->width_mbs, H = 16 * gi->height_mbs;
        s->ow = fmt_is_yuv(f->fmt) ? W : W / f->scale; s->oh = fmt_is_yuv(f->fmt) ? H : H / f->scale;
        s->pic_bytes = fmt_is_yuv(f->fmt) ? (size_t)W * H * 3 / 2 : (size_t)s->ow * s->oh * 3;
        s->pb.status = s->status;
        int rc = mvf_parser_parse_packed(ps, f->job->cand + s->first, 0, s->cnt, &s->pb);
        if (rc != MVG_SUCCESS && s->pb.words_needed > s->pb.words_capacity) {       /* guessed too small: once more with room */
            if (slot_words(&s->pb, s->pb.words_needed + s->pb.words_needed / 8))
                rc = mvf_parser_parse_packed(ps, f->job->cand + s->first, 0, s->cnt, &s->pb);
        }
        if (rc != MVG_SUCCESS) {
            fprintf(stderr, "mvt_extract: %s\n", mvf_parser_last_error(ps));
            pipe_fail(p);
            break;
        }
        s->n_ok = 0;
        for (int i = 0; i < s->cnt; i++) {
            if (s->status[i] == MVG_SUCCESS) s->n_ok++;
            else fprintf(stderr, "mvt_extract: picture %d skipped (%s)\n", f->job->cand[s->first + i],
                         s->n_ok == i ? mvf_parser_last_error(ps) : "see above");
        }
        job_parsed(f->job, seq, s->status);
        pipe_set(p, s, SLOT_PARSED);
    }
    /* tell the stages behind how many batches there were */
    pthread_mutex_lock(&p->mu); p->final = k; pthread_cond_broadcast(&p->cv); pthread_mutex_unlock(&p->mu);
    mvf_parser_destroy(ps);
    return NULL;
}

static void *write_worker(void *arg)
{
    pipe_t *p = arg; feeder_t *f = p->f; const slot_t *s = p->wslot;
    for (;;) {
        int k = __atomic_fetch_add(&p->wnext, 1, __ATOMIC_RELAXED);
        if (k >= s->cnt || __atomic_load_n(&p->failed, __ATOMIC_RELAXED)) return NULL;
        if (p->wnumber[k] < 0) continue;                /* a picture that failed to parse: no file, no number */
        char path[PATH_MAX];
        /* export_idr() numbers pictures in export order (export.c:630) */
        if (f->numbered) snprintf(path, sizeof path, "%s/%s_%d.%s", f->outdir, f->base, p->wnumber[k], file_ext[f->fmt]);
        else snprintf(path, sizeof path, "%s/%s.%s", f->outdir, f->base, file_ext[f->fmt]);
        const uint8_t *px = s->out + (size_t)k * s->pic_bytes;
        int ok = f->fmt == MVT_YUV420 ? write_raw(path, px, s->pic_bytes)
               : f->fmt == MVT_YUV444 ? write_yuv444(path, px, s->ow, s->oh)
               : f->fmt == MVT_BMP    ? write_bmp(path, px, s->ow, s->oh)
               : f->fmt == MVT_TGA    ? write_tga(path, px, s->ow, s->oh)
                                      : write_png(path, px, s->ow, s->oh);
        if (!ok) { fprintf(stderr, "mvt_extract: cannot write '%s'\n", path); pipe_fail(p); return NULL; }
        __atomic_fetch_add(&p->wexported, 1, __ATOMIC_RELAXED);
    }
}

static void *writer_main(void *arg)
{
    pipe_t *p = arg; feeder_t *f = p->f;
    for (int k = 0; pipe_wait(p, k, SLOT_DECODED); k++) {
        slot_t *s = &p->slot[k & 1];
        int number = job_number(f->job, s->seq);        /* pictures decoded before this batch, over all feeders */
        if (number < 0) { pipe_fail(p); return NULL; }
        for (int i = 0; i < s->cnt; i++) p->wnumber[i] = s->status[i] == MVG_SUCCESS ? number++ : -1;
        p->wslot = s; p->wnext = 0;
        int nw = f->threads < s->cnt ? f->threads : s->cnt;
        if (nw > 256) nw = 256;
        pthread_t th[256]; int started = 0;
        for (int t = 1; t < nw; t++) { if (pthread_create(&th[started], NULL, write_worker, p) == 0) started++; }
        write_worker(p);
        for (int t = 0; t < started; t++) pthread_join(th[t], NULL);
        if (p->failed) return NULL;
        pipe_set(p, s, SLOT_FREE);
    }
    return NULL;
}

static void *feeder_main(void *arg)
{
    feeder_t *f = arg;
    const int batch = f->batch, fmt = f->fmt, scale = f->scale;
    f->rc = 1;
    const int timing = getenv("MVT_TIMING") != NULL;
    const double t0 = now_s();
    mvg_ctx *ctx = NULL;
    if (mvg_create(&ctx, f->device, f->max_w, f->max_h, batch) != MVG_SUCCESS) {
        fprintf(stderr, "mvt_extract: %s\n", mvg_last_error(NULL));
        job_fail(f->job);
        return NULL;
    }
    const double t1 = now_s();
    /* buffers for the largest picture of the stream; the words start at a fraction of the worst case and grow on demand */
    const size_t N = (size_t)f->max_w * f->max_h, nb = N * (size_t)batch;
    const size_t max_pic = fmt_is_yuv(fmt) ? N * 384 : (N * 768) / ((size_t)scale * scale);
    pipe_t p;
    memset(&p, 0, sizeof p);
    p.f = f; p.final = -1;
    pthread_mutex_init(&p.mu, NULL); pthread_cond_init(&p.cv, NULL);
    int rc = 0;
    const int n_slots = (f->job->n_cand > batch || f->n_gens > 1) ? 2 : 1;     /* batches end at parameter generations too */
    for (int k = 0; k < n_slots; k++) {
        /* parsed pictures travel in the packed transfer format (mvgpu.h): a fifth of the dense levels on the bus */
        mvf_packed_batch *pb = &p.slot[k].pb;
        pb->n_pics = 0;
        pb->mb_kind = mvg_host_alloc(nb); pb->i16_mode = mvg_host_alloc(nb); pb->chroma_mode = mvg_host_alloc(nb);
        pb->qp_y = mvg_host_alloc(nb); pb->luma_modes = mvg_host_alloc(nb * 16);
        pb->nz_blocks = mvg_host_alloc(nb * sizeof(uint32_t)); pb->word_off = mvg_host_alloc(nb * sizeof(uint32_t));
        pb->pic_off = mvg_host_alloc(((size_t)batch + 1) * sizeof(uint64_t));
        pb->words_capacity = nb * (MVG_PACKED_WORDS_PER_MB / 4);
        pb->words = mvg_host_alloc(pb->words_capacity * sizeof(uint16_t));
        p.slot[k].out = mvg_host_alloc(max_pic * (size_t)batch);
        p.slot[k].status = malloc(sizeof(int32_t) * (size_t)batch);
        if (!pb->mb_kind || !pb->i16_mode || !pb->chroma_mode || !pb->qp_y || !pb->luma_modes || !pb->nz_blocks ||
            !pb->word_off || !pb->pic_off || !pb->words || !p.slot[k].out || !p.slot[k].status) {
            fprintf(stderr, "mvt_extract: pinned host allocation failed\n");
            rc = 1;
        }
    }
    if (n_slots == 1) p.slot[1].state = SLOT_FREE;      /* never used: a second batch cannot exist */
    const double t2 = now_s();
    double t_gpu = 0;
    pthread_t parser, writer;
    int have_parser = 0, have_writer = 0;
    if (!rc) {
        have_parser = pthread_create(&parser, NULL, parser_main, &p) == 0;
        have_writer = have_parser && pthread_create(&writer, NULL, writer_main, &p) == 0;
        if (!have_parser || !have_writer) { fprintf(stderr, "mvt_extract: cannot start helper threads\n"); pipe_fail(&p); rc = 1; }
    } else job_fail(f->job);
    int cur_gen = -1;
    for (int k = 0; !rc && pipe_wait(&p, k, SLOT_PARSED); k++) {
        slot_t *s = &p.slot[k & 1];
        if (s->n_ok > 0) {
            if (s->gen != cur_gen) {        /* this batch's SPS/PPS pair: geometry, LevelScale tables, chroma QP offsets */
                const mvf_info *gi = &f->gens[s->gen];
                if (mvg_set_sps(ctx, gi->width_mbs, gi->height_mbs, gi->level_scale4x4, gi->level_scale8x8,
                                gi->cb_qp_offset, gi->cr_qp_offset) != MVG_SUCCESS) {
                    fprintf(stderr, "mvt_extract: %s\n", mvg_last_error(ctx));
                    pipe_fail(&p); rc = 1; break;
                }
                cur_gen = s->gen;
            }
            const mvf_packed_batch *pb = &s->pb;
            mvg_packed_batch gb = { s->cnt, pb->mb_kind, pb->i16_mode, pb->chroma_mode, pb->qp_y, pb->luma_modes,
                                    pb->nz_blocks, pb->word_off, pb->pic_off, pb->words };
            const double tg = now_s();
            int ok = fmt_is_yuv(fmt) ? mvg_decode_host_packed(ctx, &gb, s->out, NULL, 0) : mvg_decode_host_packed(ctx, &gb, NULL, s->out, scale);
            t_gpu += now_s() - tg;
            if (ok != MVG_SUCCESS) { fprintf(stderr, "mvt_extract: %s\n", mvg_last_error(ctx)); pipe_fail(&p); rc = 1; break; }
        }
        pipe_set(&p, s, SLOT_DECODED);
    }
    if (have_parser) pthread_join(parser, NULL);
    if (have_writer) pthread_join(writer, NULL);
    if (p.failed) rc = 1;
    f->exported = p.wexported;
    const double t3 = now_s();
    for (int q = 0; q < n_slots; q++) {
        mvf_packed_batch *pb = &p.slot[q].pb;
        mvg_host_free(pb->mb_kind); mvg_host_free(pb->i16_mode); mvg_host_free(pb->chroma_mode); mvg_host_free(pb->qp_y);
        mvg_host_free(pb->luma_modes); mvg_host_free(pb->nz_blocks); mvg_host_free(pb->word_off); mvg_host_free(pb->pic_off);
        mvg_host_free(pb->words); mvg_host_free(p.slot[q].out); free(p.slot[q].status);
    }
    pthread_mutex_destroy(&p.mu); pthread_cond_destroy(&p.cv);
    mvg_destroy(ctx);
    if (timing)
        fprintf(stderr, "mvt_extract[gpu %d]: context %.3f s, pinned buffers %.3f s, pipeline %.3f s (GPU calls %.3f s) for %d pictures, teardown %.3f s\n",
                f->device, t1 - t0, t2 - t1, t3 - t2, t_gpu, f->exported, now_s() - t3);
    f->rc = rc;
    return NULL;
}

/* GPUs this process may use, found without waking the CUDA runtime (which costs about a second per visible GPU):
 * the entries of CUDA_VISIBLE_DEVICES, else the devices the driver lists under /proc */
static int visible_gpus(void)
{
    const char *vis = getenv("CUDA_VISIBLE_DEVICES");
    if (vis) {
        if (!*vis) return 0;
        int n = 1;
        for (const char *c = vis; *c; c++) n += *c == ',';
        return n;
    }
    int n = 0;
    FILE *pf = popen("ls /proc/driver/nvidia/gpus 2>/dev/null | wc -l", "r");
    if (pf) { if (fscanf(pf, "%d", &n) != 1) n = 0; pclose(pf); }
    return n;
}

int mvt_is_mp4(const uint8_t *data, size_t len)
{
    if (!data || len < 8) return 0;
    if (!memcmp(data + 4, "ftyp", 4)) return 1;
    const uint64_t size = (uint64_t)data[0] << 24 | (uint64_t)data[1] << 16 | (uint64_t)data[2] << 8 | data[3];
    return size >= 8 && size <= len &&
           (!memcmp(data + 4, "moov", 4) || !memcmp(data + 4, "mdat", 4) || !memcmp(data + 4, "free", 4) || !memcmp(data + 4, "wide", 4));
}

int mvt_container(const uint8_t *data, size_t len)
{
    if (mvt_is_mp4(data, len)) return MVT_CONTAINER_MP4;       /* first, as before there were other containers */
    if (!data || len < 4) return MVT_ANNEXB;
    if ((data[0] == 0 && data[1] == 0 && data[2] == 1) || (data[0] == 0 && data[1] == 0 && data[2] == 0 && data[3] == 1))
        return MVT_ANNEXB;
    if (data[0] == 0x1A && data[1] == 0x45 && data[2] == 0xDF && data[3] == 0xA3) return MVT_CONTAINER_MKV;
    static const size_t per[3] = {188, 192, 204};
    for (size_t o = 0; o < 204 && o + 4 * 204 < len; o++) {
        if (data[o] != 0x47) continue;
        for (int k = 0; k < 3; k++) {
            int i = 1;
            while (i < 5 && data[o + (size_t)i * per[k]] == 0x47) i++;
            if (i == 5) return MVT_CONTAINER_TS;
        }
    }
    return MVT_ANNEXB;
}

int mvt_extract(const uint8_t *data, size_t len, const char *base, const char *outdir, int fmt, int n_want, int mode,
                int scale, int device, int threads, int batch, int *n_exported)
{
    if (n_exported) *n_exported = 0;
    if (!data || !base || n_want < 1 || scale < 1 || batch < 0 || fmt < MVT_YUV420 || fmt > MVT_YUV444) return MVG_FAILURE;
    if (!outdir || !*outdir) outdir = ".";
    if (threads < 1) { long c = sysconf(_SC_NPROCESSORS_ONLN); threads = c > 0 ? (int)c : 1; }
    mvf_stream *st = NULL;
    int (*const open[4])(const uint8_t *, size_t, mvf_stream **) = {
        [MVT_ANNEXB] = mvf_open_annexb, [MVT_CONTAINER_MP4] = mvf_open_mp4, [MVT_CONTAINER_TS] = mvf_open_ts, [MVT_CONTAINER_MKV] = mvf_open_mkv };
    static const char *const kind[4] = {"an H.264 elementary stream", "an MP4 / QuickTime file", "an MPEG-2 transport stream", "a Matroska / WebM file"};
    const int container = mvt_container(data, len);
    if (open[container](data, len, &st) != MVG_SUCCESS) {
        fprintf(stderr, "mvt_extract: cannot read the input as %s: %s\n", kind[container], mvf_last_error(NULL));
        return MVG_FAILURE;
    }
    mvf_info info;
    mvf_get_info(st, &info);
    const int n_gens = info.n_generations;
    mvf_info *gens = malloc(sizeof *gens * (size_t)n_gens);
    int32_t *sel = malloc(sizeof(int32_t) * (size_t)(n_want > info.n_idr ? n_want : info.n_idr + 1));
    int8_t *okflags = calloc((size_t)info.n_idr + 1, 1);
    if (!sel || !gens || !okflags) { fprintf(stderr, "mvt_extract: out of memory\n"); free(sel); free(gens); free(okflags); mvf_close(st); return MVG_FAILURE; }
    int max_w = 0, max_h = 0, rc = 0;
    for (int g = 0; g < n_gens; g++) {
        mvf_get_generation_info(st, g, &gens[g]);
        if (gens[g].width_mbs > max_w) max_w = gens[g].width_mbs;
        if (gens[g].height_mbs > max_h) max_h = gens[g].height_mbs;
        if (!fmt_is_yuv(fmt) && ((16 * gens[g].width_mbs) % scale || (16 * gens[g].height_mbs) % scale)) {
            fprintf(stderr, "mvt_extract: scale %d does not divide %dx%d\n", scale, 16 * gens[g].width_mbs, 16 * gens[g].height_mbs);
            rc = 1;
        }
    }
    /* candidates in export order: the selection (filter.c:52-215), all of it attempted */
    const int n_cand = mvf_select_idr(st, n_want, mode, sel), need = n_cand;
    if (n_cand < 1 && !rc) { fprintf(stderr, "mvt_extract: no picture to decode after filtering\n"); rc = 1; }
    if (rc) { free(sel); free(gens); free(okflags); mvf_close(st); return MVG_FAILURE; }
    /* the reference appends _<k> when more than one picture was requested after filtering (export.c:630) */
    int numbered;
    if (mode == 0) numbered = need > 1;
    else {      /* picture_number after filtering = min(requested, candidates) = what 'ordered' would return */
        int32_t *tmp = malloc(sizeof(int32_t) * (size_t)(n_want > info.n_idr ? n_want : info.n_idr + 1));
        numbered = tmp ? mvf_select_idr(st, n_want, 1, tmp) > 1 : n_cand > 1;
        free(tmp);
    }
    if (batch == 0) {
        /* pictures per GPU call: about 256 MB of output per buffer set (pinned memory costs ~1 s per GB to set
         * up), but never fewer than the PNG encoder threads that share a batch */
        const size_t W = 16 * (size_t)max_w, H = 16 * (size_t)max_h;
        const size_t pic = fmt_is_yuv(fmt) ? W * H * 3 / 2 : (W / (size_t)scale) * (H / (size_t)scale) * 3;
        batch = (int)(((size_t)256 << 20) / pic);
        if (fmt == MVT_PNG && batch < threads) batch = threads;
        batch = batch < 4 ? 4 : batch > 64 ? 64 : batch;
    }
    if (batch > 256) batch = 256;
    if (batch > need) batch = need;

    /* device >= 0: that GPU; device < 0: as many of the visible GPUs as the job can keep busy (about a million
     * macroblocks each; a small job on one GPU does not pay for waking eight), batches dealt in order */
    int n_gpus = 1;
    if (device < 0) {
        n_gpus = visible_gpus();
        if (n_gpus < 1) { fprintf(stderr, "mvt_extract: no CUDA device; this path has no CPU fallback\n"); free(sel); free(gens); free(okflags); mvf_close(st); return MVG_FAILURE; }
        const long long work = (long long)need * max_w * max_h;
        const int by_work = (int)((work + 999999) / 1000000), n_batches = (need + batch - 1) / batch;
        if (n_gpus > by_work) n_gpus = by_work;
        if (n_gpus > n_batches) n_gpus = n_batches;
        if (n_gpus > 64) n_gpus = 64;
        if (n_gpus < 1) n_gpus = 1;
        /* the runtime only wakes the GPUs it can see: narrow the list (the first n_gpus of the one in force, else
         * 0 .. n_gpus-1) before the first CUDA call of the process */
        {
            char list[512]; int o = 0;
            const char *vis = getenv("CUDA_VISIBLE_DEVICES");
            if (vis) {
                int seen = 0;
                for (const char *c = vis; *c && o < 500; c++) {
                    if (*c == ',' && ++seen == n_gpus) break;
                    list[o++] = *c;
                }
                list[o] = 0;
            } else
                for (int g = 0; g < n_gpus && o < 500; g++) o += snprintf(list + o, sizeof list - (size_t)o, g ? ",%d" : "%d", g);
            setenv("CUDA_VISIBLE_DEVICES", list, 1);
        }
    }
    job_t job;
    memset(&job, 0, sizeof job);
    job.st = st; job.cand = sel; job.n_cand = n_cand; job.batch = batch; job.ok = okflags;
    pthread_mutex_init(&job.mu, NULL); pthread_cond_init(&job.cv, NULL);
    feeder_t feeders[64];
    pthread_t th[64];
    for (int g = 0; g < n_gpus; g++) {
        feeder_t f = { &job, st, gens, n_gens, max_w, max_h, base, outdir, fmt, scale, device < 0 ? g : device,
                       threads / n_gpus > 0 ? threads / n_gpus : 1, batch, numbered, 0, 1 };
        feeders[g] = f;
    }
    int threaded[64] = {0};
    for (int g = 1; g < n_gpus; g++) threaded[g] = pthread_create(&th[g], NULL, feeder_main, &feeders[g]) == 0;
    feeder_main(&feeders[0]);
    int exported = 0;
    for (int g = 0; g < n_gpus; g++) {
        if (g > 0) {
            if (threaded[g]) pthread_join(th[g], NULL);
            else feeder_main(&feeders[g]);              /* no thread: take its share here */
        }
        exported += feeders[g].exported;
        if (feeders[g].rc) rc = 1;
    }
    if (n_exported) *n_exported = exported;
    if (!rc && exported < need) {
        fprintf(stderr, "mvt_extract: %d of %d pictures exported (%d could not be decoded)\n", exported, need, job.n_fail_known);
        rc = 1;             /* like the reference, which reports FAILURE when it runs out of samples first (h264.c:181) */
    }
    pthread_mutex_destroy(&job.mu); pthread_cond_destroy(&job.cv);
    free(job.rec);
    mvf_close(st);
    free(sel); free(gens); free(okflags);
    return rc ? MVG_FAILURE : MVG_SUCCESS;
}
