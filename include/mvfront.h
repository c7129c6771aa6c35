/*
 * mvfront.h -- host front end of the intra reconstruction path (libmvfront.so).
 *
 * Written from scratch in C: Annex-B elementary-stream scan or MP4 sample table walk, NAL unescape, SPS / PPS /
 * slice header, CAVLC macroblock parsing -> the structure-of-arrays of mvgpu.h, one IDR
 * slice per thread.  It replaces, for this path only, what the reference does on the way
 * to its per-macroblock hot-path call (citations relative to minivideo/src/):
 *
 *   es_fileParse()            demuxer/esparser/esparser.c:40     -> mvf_open_annexb()
 *   idr_filtering()           demuxer/filter.c:52                -> mvf_select_idr()
 *   nalu_clean_sample()       decoder/h264/h264_nalu.c:195       -> (inside) NAL unescape
 *   decodeSPS()/decodePPS()   decoder/h264/h264_parameterset.c:123,:812
 *   decodeSliceHeader()       decoder/h264/h264_slice.c:156
 *   macroblock_layer() parse half, mb_pred(), residual_luma/chroma()
 *                             decoder/h264/h264_macroblock.c:75-313,:393,:1102,:1222
 *   residual_block_cavlc()    decoder/h264/h264_cavlc.c:79
 *   Intra_4x4/8x8_deriv_PredMode()  decoder/h264/h264_intra_prediction.c:196,:977
 *
 * Return codes as in mvgpu.h (MVG_SUCCESS 1 / MVG_FAILURE 0 / MVG_UNSUPPORTED -1); never
 * exits.  Supported: what the reference supports for this path -- Baseline/Main/High 4:2:0
 * 8-bit, frame_mbs_only, CAVLC, one I slice per IDR picture, SPS scaling lists.
 * Unsupported (MVG_UNSUPPORTED): CABAC, I_PCM, FMO/ASO, interlace, PPS scaling lists.
 */
#ifndef MVFRONT_H
#define MVFRONT_H

#include <stddef.h>
#include <stdint.h>

#include "mvgpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mvf_stream mvf_stream;

typedef struct mvf_info {
    int32_t width_mbs, height_mbs;      /* PicWidthInMbs, PicHeightInMapUnits (frame_mbs_only) */
    int32_t profile_idc, level_idc;
    int32_t n_idr;                      /* IDR slice NAL units found                            */
    int32_t transform_8x8_mode;
    int32_t cb_qp_offset, cr_qp_offset; /* chroma_qp_index_offset, second_chroma_qp_index_offset */
    int32_t pic_init_qp;
    int32_t crop_left, crop_right, crop_top, crop_bottom;   /* parsed, never applied (export.c:80-81) */
    int32_t level_scale4x4[3 * 6 * 16]; /* ready for mvg_set_sps()                              */
    int32_t level_scale8x8[6 * 64];
    int32_t n_generations;              /* parameter generations in the stream (see below)      */
    int32_t generation;                 /* the one this structure describes                     */
} mvf_info;

/* Writable twin of mvg_batch: the caller allocates the arrays (pinned memory from
 * mvg_host_alloc() for full PCIe speed) for `n_pics` pictures. */
typedef struct mvf_batch {
    int32_t  n_pics;
    uint8_t *mb_kind, *i16_mode, *chroma_mode;
    int8_t  *qp_y;
    uint8_t *cbp, *luma_modes;
    int16_t *coeff;
    int32_t *status;    /* NULL, or [n_pics]: see "errors" below */
} mvf_batch;

/* Scan an Annex-B byte stream held in memory (it must stay valid until mvf_close), index the IDR slices and
 * replay the parameter sets in stream order the way the reference's NAL loop does (h264.c:128-150): every SPS /
 * PPS replaces the one stored under its id, every IDR slice resolves its PPS by pic_parameter_set_id and its SPS
 * through it (h264_slice.c:168-169).  Each distinct (SPS, PPS) pair in force for some IDR picture is a
 * "parameter generation"; most streams have exactly one.  A generation fixes picture geometry, the LevelScale
 * tables, the chroma QP offsets, pic_init_qp and transform_8x8_mode -- what mvg_set_sps() installs -- so a
 * caller reconstructs each generation's pictures with that generation's mvf_info.  FAILURE / UNSUPPORTED only
 * when no IDR picture at all has usable parameter sets. */
int mvf_open_annexb(const uint8_t *data, size_t len, mvf_stream **out);
/* The same stream from an MP4 / QuickTime file (ISO/IEC 14496-12) held in memory: the first video track whose
 * sample description is avc1 / avc3.  Its NAL units are indexed in place, in the order an Annex-B stream of the same
 * content would hold them: the avcC parameter sets of a sample description before the first sample that uses it,
 * then every sample's length-prefixed NAL units.  Everything above then applies unchanged; mvf_select_idr() sizes a
 * picture by its stsz sample size.  A sample whose NAL lengths run past it is skipped.  UNSUPPORTED: fragmented
 * files, video other than H.264, no video track; FAILURE: a damaged box structure or sample table. */
int mvf_open_mp4(const uint8_t *data, size_t len, mvf_stream **out);
int mvf_close(mvf_stream *s);
const char *mvf_last_error(const mvf_stream *s);      /* s may be NULL after a failed open */
int mvf_get_info(const mvf_stream *s, mvf_info *out);                       /* generation 0 */
int mvf_generation_count(const mvf_stream *s);
int mvf_get_generation_info(const mvf_stream *s, int generation, mvf_info *out);
int mvf_picture_generation(const mvf_stream *s, int idr_index);             /* -1: the picture has no usable SPS/PPS */

/* Frame selection, the work-list builder for the GPUs: mirrors idr_filtering()
 * (demuxer/filter.c:52-215).  mode 0 = unfiltered (first n), 1 = ordered, 2 = distributed.
 * Writes at most `n_wanted` IDR indices (0-based among the IDR slices) and returns how many. */
int mvf_select_idr(const mvf_stream *s, int n_wanted, int mode, int32_t *indices);

/* CAVLC-parse `count` IDR pictures given by `indices` (NULL = first, first+1, ...) into `out`
 * using up to `n_threads` host threads (one slice per thread).  All pictures of a call must have the geometry
 * of the first one (one parameter generation per call, or generations of equal picture size).
 * Errors: with out->status == NULL the call is all-or-nothing -- the first picture that fails fails the call
 * with its code.  With out->status pointing to `count` ints every picture reports its own code there
 * (MVG_SUCCESS / MVG_FAILURE / MVG_UNSUPPORTED), a failed picture leaves an all-zero slot, and the call itself
 * succeeds: the reference, too, counts a bad picture and goes on (h264.c:103-109, :181). */
int mvf_parse_pictures(mvf_stream *s, const int32_t *indices, int first, int count,
                       mvf_batch *out, int n_threads);

/* Writable twin of mvg_packed_batch (mvgpu.h): the caller allocates mb_kind .. word_off for `n_pics`
 * pictures, pic_off[n_pics + 1] and `words_capacity` uint16 words (n_pics * N * MVG_PACKED_WORDS_PER_MB
 * always suffices; a parsed picture typically needs a fifth of the dense levels). */
typedef struct mvf_packed_batch {
    int32_t   n_pics;
    uint8_t  *mb_kind, *i16_mode, *chroma_mode;
    int8_t   *qp_y;
    uint8_t  *luma_modes;
    uint32_t *nz_blocks, *word_off;
    uint64_t *pic_off;
    uint16_t *words;
    size_t    words_capacity;
    int32_t  *status;           /* NULL, or [n_pics]: per-picture codes (see mvf_parse_pictures) */
    size_t    words_needed;     /* out: words the pictures of the call need (also when the capacity was too small) */
} mvf_packed_batch;

/* mvf_parse_pictures() emitting the packed transfer format directly: the levels of a picture never exist
 * densely outside a per-thread scratch picture.  FAILURE (with a message) when `words` is too small. */
int mvf_parse_pictures_packed(mvf_stream *s, const int32_t *indices, int first, int count,
                              mvf_packed_batch *out, int n_threads);

/* A parser keeps its worker threads and their scratch memory between calls (the two functions above create and
 * destroy one per call).  One call at a time per parser; several parsers may share a stream.  While the workers
 * parse, the calling thread gathers finished pictures' words in order, so the packed output is complete when the
 * last picture is. */
typedef struct mvf_parser mvf_parser;
int mvf_parser_create(mvf_stream *s, int n_threads, mvf_parser **out);
int mvf_parser_destroy(mvf_parser *p);
int mvf_parser_parse(mvf_parser *p, const int32_t *indices, int first, int count, mvf_batch *out);
int mvf_parser_parse_packed(mvf_parser *p, const int32_t *indices, int first, int count, mvf_packed_batch *out);
const char *mvf_parser_last_error(const mvf_parser *p);     /* of this parser's last call (never NULL) */

#ifdef __cplusplus
}
#endif
#endif
