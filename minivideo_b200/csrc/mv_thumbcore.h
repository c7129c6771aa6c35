/*
 * mv_thumbcore.h -- thumbnail extraction over the GPU path (mv_thumbcore.c).
 */
#ifndef MV_THUMBCORE_H
#define MV_THUMBCORE_H

#include <stddef.h>
#include <stdint.h>

enum { MVT_YUV420, MVT_BMP, MVT_TGA, MVT_PNG, MVT_YUV444 };

/* Whether `data` is an MP4 / QuickTime file: bytes 4..7 are 'ftyp', or the file starts with a whole moov, mdat, free
 * or wide box.  An Annex-B stream (00 00 00 01 ...) never is. */
int mvt_is_mp4(const uint8_t *data, size_t len);

/* Decode up to `n_want` IDR pictures of `data` -- an Annex-B stream, or an MP4 / QuickTime file (mvt_is_mp4) -- (selection `mode`: 0 unfiltered, 1 ordered,
 * 2 distributed, demuxer/filter.c:52-215) on CUDA device `device` and write them as
 * <outdir>/<base>[_<k>].{yuv,bmp,tga,png}, named and laid out like export_idr() does (export.c:627-642, :100-151,
 * :197-330, :535-601).  scale > 1 writes box-downscaled RGB thumbnails (no reference counterpart).  threads < 1: one CAVLC
 * parser thread per core.  device < 0: every visible GPU, one feeder thread each, batches of `batch` pictures dealt
 * round-robin (disjoint pictures per GPU, nothing crosses GPUs); batch 0 picks a size from the picture size.  Returns MVG_SUCCESS (1) / MVG_FAILURE (0); messages go to stderr. */
int mvt_extract(const uint8_t *data, size_t len, const char *base, const char *outdir, int fmt, int n_want, int mode,
                int scale, int device, int threads, int batch, int *n_exported);

/* Write one picture file in format `fmt` from host pixels (RGB24 rows top-down, or planar I420 for the two YUV formats).
 * Returns 1 / 0. */
int mvt_write_image(const char *path, int fmt, const uint8_t *pixels, int w, int h);

#endif
