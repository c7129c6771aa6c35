/*
 * minivideo_shim.c -- libminivideo_b200.so: the reference's public entry points (minivideo/src/minivideo.h:89-149),
 * same names, arguments and return codes, backed by the GPU path, so that the reference's own mini_thumbnailer
 * (mini_thumbnailer/src/main.cpp:255-285) links against it unchanged:
 *
 *   minivideo_print_infos / minivideo_get_infos / minivideo_endianness      informational
 *   minivideo_open(path, &media)      load the file                         (import.c: import_fileOpen)
 *   minivideo_parse(media, a, v, s)   picks the input path from the file: Annex-B ES (demuxer/esparser/esparser.c:40)
 *                                     or MP4 / QuickTime (the reference's MP4 demuxer)
 *   minivideo_decode(media, dir, format, quality, n, mode)
 *                                     IDR selection (demuxer/filter.c:52), CAVLC on the host threads, kernels,
 *                                     picture files as export_idr() names and lays them out (export.c:618-705)
 *   minivideo_close(&media)
 *
 * MediaFile_t is opaque to the caller (main.cpp only passes the pointer on), so this library defines its own.
 * Scope: what this repository accelerates -- H.264 elementary streams (.264/.h264/.avc, the reference's
 * es_fileParse path) and the H.264 video track of MP4 / QuickTime files (.mp4/.m4v/.mov/.3gp/.3g2), intra pictures,
 * CAVLC, output png (also for 'jpg', as in the reference's default build) / bmp / tga / yuv420 / yuv444.  Other
 * containers (AVI, MKV, ...), webp and minivideo_extract() answer FAILURE with a message.  Like the reference (h264.c:65) pictures are written
 * to the current directory unless an output directory is given.  No CPU fallback.
 */
#include <stdbool.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>

#include "mv_thumbcore.h"

#define SUCCESS 1           /* minivideo/src/typedef.h:40-42 */
#define FAILURE 0

typedef struct MediaFile_t {
    char     path[4096];
    char     base[256];     /* file name without directory and extension */
    uint8_t *data;
    size_t   len;
    int      parsed;
} MediaFile_t;

/* PictureFormat_e, minivideo/src/avcodecs.h:180-191 */
enum { PICTURE_BMP = 1, PICTURE_JPG = 2, PICTURE_PNG = 3, PICTURE_WEBP = 4, PICTURE_TGA = 5, PICTURE_YUV444 = 16, PICTURE_YUV420 = 17 };

void minivideo_print_infos(void)
{
    printf("\nminivideo_print_infos()\n* B200 intra-reconstruction path behind the MiniVideo API (libminivideo_b200)\n"
           "* H.264 elementary streams and MP4 / QuickTime files, CAVLC intra pictures; pictures: png, bmp, tga, yuv420, yuv444\n\n");
}

void minivideo_get_infos(int *major, int *minor, int *patch, const char **builddate, const char **buildtime)
{
    if (major) *major = 6;
    if (minor) *minor = 2;
    if (patch) *patch = 0;
    if (builddate) *builddate = __DATE__;
    if (buildtime) *buildtime = __TIME__;
}

int minivideo_endianness(void)
{
    const int i = 1;
    return *(const char *)&i == 1 ? 1234 : 4321;
}

int minivideo_open(const char *input_filepath, MediaFile_t **input_media)
{
    if (!input_filepath || !input_media) return FAILURE;
    *input_media = NULL;
    FILE *f = fopen(input_filepath, "rb");
    if (!f) { fprintf(stderr, "minivideo_open: cannot open '%s'\n", input_filepath); return FAILURE; }
    MediaFile_t *m = calloc(1, sizeof *m);
    if (!m) { fclose(f); return FAILURE; }
    fseek(f, 0, SEEK_END);
    long flen = ftell(f);
    fseek(f, 0, SEEK_SET);
    m->data = flen >= 0 ? malloc((size_t)flen + 8) : NULL;
    if (!m->data || fread(m->data, 1, (size_t)flen, f) != (size_t)flen) {
        fprintf(stderr, "minivideo_open: cannot read '%s'\n", input_filepath);
        fclose(f); free(m->data); free(m);
        return FAILURE;
    }
    fclose(f);
    m->len = (size_t)flen;
    snprintf(m->path, sizeof m->path, "%s", input_filepath);
    const char *slash = strrchr(input_filepath, '/');
    snprintf(m->base, sizeof m->base, "%s", slash ? slash + 1 : input_filepath);
    char *dot = strrchr(m->base, '.');
    if (dot) *dot = 0;
    *input_media = m;
    return SUCCESS;
}

int minivideo_parse(MediaFile_t *m, const bool extract_audio, const bool extract_video, const bool extract_subtitles)
{
    (void)extract_audio; (void)extract_subtitles;
    if (!m || !extract_video) return FAILURE;
    /* the reference picks its parser from the file (import.c); the ES and MP4 paths are in scope */
    const char *dot = strrchr(m->path, '.');
    const bool es = dot && (!strcmp(dot, ".264") || !strcmp(dot, ".h264") || !strcmp(dot, ".avc") || !strcmp(dot, ".H264") || !strcmp(dot, ".AVC"));
    const bool mp4 = dot && (!strcasecmp(dot, ".mp4") || !strcasecmp(dot, ".m4v") || !strcasecmp(dot, ".mov") ||
                             !strcasecmp(dot, ".3gp") || !strcasecmp(dot, ".3g2"));
    if (mp4 && !mvt_is_mp4(m->data, m->len)) {
        fprintf(stderr, "minivideo_parse: '%s' is not an MP4 / QuickTime file\n", m->path);
        return FAILURE;
    }
    if (!es && !mp4) {
        fprintf(stderr, "minivideo_parse: '%s' is neither an H.264 elementary stream nor an MP4 / QuickTime file; other containers are outside this library's scope\n", m->path);
        return FAILURE;
    }
    m->parsed = 1;
    return SUCCESS;
}

int minivideo_decode(MediaFile_t *m, const char *output_directory, const int picture_format, const int picture_quality,
                     const int picture_number, const int picture_extractionmode)
{
    (void)picture_quality;
    if (!m || !m->parsed) return FAILURE;
    int fmt;
    switch (picture_format) {
    case PICTURE_YUV420: fmt = MVT_YUV420; break;
    case PICTURE_BMP:    fmt = MVT_BMP; break;
    case PICTURE_TGA:    fmt = MVT_TGA; break;
    case PICTURE_YUV444: fmt = MVT_YUV444; break;
    case PICTURE_JPG:                                   /* default build: "No jpg export library available, trying png" (export.c:652-657) */
    case PICTURE_PNG:    fmt = MVT_PNG; break;
    default:
        fprintf(stderr, "minivideo_decode: picture format %d is not supported by the GPU path (jpg/png, bmp, tga, yuv420, yuv444)\n", picture_format);
        return FAILURE;
    }
    if (picture_extractionmode < 0 || picture_extractionmode > 2) return FAILURE;
    int n = picture_number < 1 ? 1 : picture_number > 999 ? 999 : picture_number;     /* minivideo.c clamps to 0..999 */
    int exported = 0;
    return mvt_extract(m->data, m->len, m->base, output_directory, fmt, n, picture_extractionmode, 1, 0, 0, 0, &exported);
}

int minivideo_extract(MediaFile_t *m, const char *output_directory, const bool extract_audio, const bool extract_video,
                      const bool extract_subtitles, const int output_format)
{
    (void)m; (void)output_directory; (void)extract_audio; (void)extract_video; (void)extract_subtitles; (void)output_format;
    fprintf(stderr, "minivideo_extract: track extraction is outside this library's scope\n");
    return FAILURE;
}

int minivideo_close(MediaFile_t **input_media)
{
    if (!input_media || !*input_media) return FAILURE;
    free((*input_media)->data);
    free(*input_media);
    *input_media = NULL;
    return SUCCESS;
}
