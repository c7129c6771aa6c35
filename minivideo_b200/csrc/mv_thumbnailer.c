/*
 * mv_thumbnailer.c -- command-line front of the GPU path, argument-compatible with the reference's
 * mini_thumbnailer (mini_thumbnailer/src/main.cpp:77-240):
 *
 *   mv_thumbnailer -i <file.264|.mp4|.ts|.m2ts|.mkv> [-o <dir>] [-f jpg|png|bmp|tga|yuv420|yuv444] [-n N] [-e unfiltered|ordered|distributed]
 *                  [-s scale] [-d device] [-t threads] [-b batch]
 *
 * The input is an H.264 elementary stream, an MP4 / QuickTime file, an MPEG-2 transport stream (188, 192 or 204-byte
 * packets) or a Matroska / WebM file, told apart by content (mvt_container), not by name.
 * The work is mvt_extract() (mv_thumbcore.c).  As in the reference's default build (no libjpeg, export.c:652-657)
 * 'jpg' -- also the default format, main.cpp:56 -- is written as PNG.  Extensions over the reference: -o is honoured (the reference
 * ignores it, h264.c:65), -s writes a box-downscaled RGB thumbnail, -d/-t/-b pick the GPU, parser threads and
 * batch size; -d all (or -d -1) spreads the pictures over every GPU of the box.  No CPU fallback: without a CUDA
 * device the program fails.
 */
#define _POSIX_C_SOURCE 200809L
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "mv_thumbcore.h"

static void usage(void)
{
    fprintf(stderr, "usage: mv_thumbnailer -i <file.264|.mp4|.mov|.ts|.m2ts|.mkv|.webm> [-o <dir>] [-f jpg|png|bmp|tga|yuv420|yuv444]\n"
                    "                      [-n picture_number] [-e unfiltered|ordered|distributed] [-s scale] [-d device] [-t threads] [-b batch]\n"
                    "  input: H.264 elementary stream, MP4 / QuickTime, MPEG-2 transport stream or Matroska / WebM (found from the content)\n");
}

int main(int argc, char **argv)
{
    const char *in = NULL, *outdir = ".";
    int fmt = MVT_PNG, n_want = 1, mode = 0, scale = 1, device = 0, threads = 0, batch = 0;
    for (int i = 1; i < argc; i++) {
        const char *a = argv[i], *v = i + 1 < argc ? argv[i + 1] : NULL;
        if (!strcmp(a, "-h") || !strcmp(a, "--help")) { usage(); return 0; }
        if (!v) { usage(); return 2; }
        if (!strcmp(a, "-i")) in = v;
        else if (!strcmp(a, "-o")) outdir = v;
        else if (!strcmp(a, "-f")) {
            if (!strcmp(v, "yuv420")) fmt = MVT_YUV420;
            else if (!strcmp(v, "bmp")) fmt = MVT_BMP;
            else if (!strcmp(v, "tga")) fmt = MVT_TGA;
            else if (!strcmp(v, "png")) fmt = MVT_PNG;
            else if (!strcmp(v, "jpg")) fmt = MVT_PNG;          /* "No jpg export library available, trying png" */
            else if (!strcmp(v, "yuv444")) fmt = MVT_YUV444;
            else { fprintf(stderr, "mv_thumbnailer: picture format '%s' is not supported (jpg, png, bmp, tga, yuv420, yuv444)\n", v); return 2; }
        }
        else if (!strcmp(a, "-n")) n_want = atoi(v);
        else if (!strcmp(a, "-e")) {
            if (!strcmp(v, "unfiltered")) mode = 0;
            else if (!strcmp(v, "ordered")) mode = 1;
            else if (!strcmp(v, "distributed")) mode = 2;
            else { fprintf(stderr, "mv_thumbnailer: unknown extraction mode '%s'\n", v); return 2; }
        }
        else if (!strcmp(a, "-s")) scale = atoi(v);
        else if (!strcmp(a, "-d")) device = !strcmp(v, "all") ? -1 : atoi(v);
        else if (!strcmp(a, "-t")) threads = atoi(v);
        else if (!strcmp(a, "-b")) batch = atoi(v);
        else if (!strcmp(a, "-q")) { /* JPEG quality: accepted, unused */ }
        else { fprintf(stderr, "mv_thumbnailer: unknown argument '%s'\n", a); usage(); return 2; }
        i++;
    }
    if (!in || n_want < 1 || scale < 1 || batch < 0) { usage(); return 2; }

    /* the whole stream in memory; read in growing chunks so that pipes and FIFOs (no size, no seeking) work too */
    FILE *f = fopen(in, "rb");
    if (!f) { fprintf(stderr, "mv_thumbnailer: cannot open '%s'\n", in); return 1; }
    size_t cap = 1u << 20, flen = 0;
    if (fseek(f, 0, SEEK_END) == 0) {
        const long sz = ftell(f);
        if (sz > 0) cap = (size_t)sz + 1;               /* + 1: the read that finds end-of-file */
        if (fseek(f, 0, SEEK_SET) != 0) { fprintf(stderr, "mv_thumbnailer: cannot rewind '%s'\n", in); fclose(f); return 1; }
    } else clearerr(f);
    uint8_t *data = malloc(cap + 8);
    while (data) {
        const size_t got = fread(data + flen, 1, cap - flen, f);
        flen += got;
        if (got == 0) break;
        if (flen == cap) {
            uint8_t *nd = realloc(data, cap * 2 + 8);
            if (!nd) { free(data); data = NULL; break; }
            data = nd; cap *= 2;
        }
    }
    if (!data || ferror(f)) { fprintf(stderr, "mv_thumbnailer: cannot read '%s'\n", in); free(data); fclose(f); return 1; }
    fclose(f);

    /* input base name without directory and extension (import.c: file_name) */
    char base[256];
    const char *slash = strrchr(in, '/');
    snprintf(base, sizeof base, "%s", slash ? slash + 1 : in);
    char *dot = strrchr(base, '.');
    if (dot) *dot = 0;

    /* One GPU asked for: make it the only one the CUDA runtime sees.  Initialising the runtime costs about a second
     * per visible GPU (6-7 s on an 8-GPU box), which is most of the run time of a small job. */
    if (device >= 0) {
        const char *vis = getenv("CUDA_VISIBLE_DEVICES");
        char id[64];
        if (!vis) snprintf(id, sizeof id, "%d", device);
        else {                                      /* the device-th entry of the list already in force */
            const char *p = vis;
            for (int k = 0; k < device && p; k++) { p = strchr(p, ','); if (p) p++; }
            if (p && *p && *p != ',') snprintf(id, sizeof id, "%.*s", (int)strcspn(p, ","), p);
            else id[0] = 0;                         /* no such entry: leave things alone, mvg_create() reports it */
        }
        if (id[0]) { setenv("CUDA_VISIBLE_DEVICES", id, 1); device = 0; }
    }

    int exported = 0;
    const int ok = mvt_extract(data, flen, base, outdir, fmt, n_want, mode, scale, device, threads, batch, &exported);
    printf("mv_thumbnailer: %d picture(s) exported\n", exported);
    free(data);
    return ok == 1 ? 0 : 1;
}
