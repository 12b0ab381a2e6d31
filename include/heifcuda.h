/*
 * heifcuda.h — C ABI of the B200 HEVC-intra reconstruction + colour-conversion engine.
 *
 * Plain C, no torch / CUDA types in any signature.  Two layers:
 *
 *  (1) host front-end (CPU, serial CABAC parse): hc_parser_*  -> hc_records
 *      replaces the parse half of  third-party/libde265/libde265/slice.cc:5179-5346
 *      (decode_substream / read_coding_tree_unit) that libde265_v1_push_data / de265_decode
 *      (libheif/plugins/decoder_libde265.cc:269-369) drive in the reference.
 *
 *  (2) device engine (sm_100a kernels): hc_engine_*  reconstructs batches of parsed pictures and
 *      converts them to interleaved RGB.  Replaces the reconstruct half of the same loop
 *      (decode_TU slice.cc:3741, scale_coefficients transform.cc:692, decode_intra_prediction
 *      intrapred.cc:337, apply_deblocking_filter deblock.cc:1921,
 *      apply_sample_adaptive_offset_sequential sao.cc:552) and libheif's colour conversion
 *      (convert_colorspace colorconversion.cc:487, Op_YCbCr420_to_RGB24 yuv2rgb.cc:260 ...).
 *
 * The libheif decoder-plugin (struct heif_decoder_plugin, libheif/api/libheif/heif_plugin.h:53-112)
 * built on top of this ABI lives in libheif-cuda.so and is declared in heifcuda_plugin.h.
 *
 * All functions returning int return 0 on success and a negative HC_ERR_* code otherwise;
 * hc_last_error() gives the text for the calling thread.
 */
#ifndef HEIFCUDA_H
#define HEIFCUDA_H

#include <stddef.h>
#include <stdint.h>
#include "heifcuda_records.h"

#ifdef __cplusplus
extern "C" {
#endif
/* the libraries are built with -fvisibility=hidden -fno-gnu-unique: only this C ABI is exported, so that
 * no C++ symbol of the engine can bind to (or be bound by) another library of the host process */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define HC_OK 0
#define HC_ERR_BITSTREAM (-1)   /* malformed / unsupported bitstream                           */
#define HC_ERR_ARGUMENT (-2)
#define HC_ERR_NO_DEVICE (-3)   /* no CUDA device / engine not built: there is NO CPU fallback */
#define HC_ERR_CUDA (-4)
#define HC_ERR_MEMORY (-5)
#define HC_ERR_UNSUPPORTED (-6)

const char* hc_last_error(void);
/* 1 if this build of the library contains the CUDA engine (hc_engine_*), else 0. */
int hc_has_cuda_engine(void);

/* ------------------------------------------------------------------ host front-end -------- */
typedef struct hc_parser hc_parser;
typedef struct hc_records hc_records;

#define HC_STREAM_LENGTH_PREFIXED 0 /* 4-byte big-endian NAL lengths: what libheif's push_data gets */
#define HC_STREAM_ANNEXB 1          /* 00 00 01 start codes (.265 / .bit files)                     */
#define HC_STREAM_SINGLE_NAL 2      /* exactly one NAL unit                                         */

hc_parser* hc_parser_new(void);
void hc_parser_free(hc_parser* p);
/* Feeds data; parameter sets are kept, slice segments are parsed immediately. */
int hc_parser_push(hc_parser* p, const uint8_t* data, size_t size, int stream_format);
/* Returns the records of the picture parsed so far and resets the parser for the next picture
 * (parameter sets stay). NULL + HC_ERR_BITSTREAM text if no complete picture is available. */
hc_records* hc_parser_take_picture(hc_parser* p);

void hc_records_free(hc_records* r);
const hc_pic* hc_records_pic(const hc_records* r);
const hc_ctu* hc_records_ctus(const hc_records* r, size_t* count);
const hc_blk* hc_records_blks(const hc_records* r, size_t* count);
const hc_tb* hc_records_tbs(const hc_records* r, size_t* count);
const hc_coeff* hc_records_coeffs(const hc_records* r, size_t* count);
const uint8_t* hc_records_edge_map(const hc_records* r, size_t* bytes);
const int8_t* hc_records_qp_map(const hc_records* r, size_t* bytes);
const uint8_t* hc_records_scaling(const hc_records* r, size_t* bytes); /* NULL if flat */
/* total bytes of all record arrays (the `R` term of the roofline: bytes uploaded per picture) */
size_t hc_records_upload_bytes(const hc_records* r);

/* ---- K0: CABAC parse on the device --------------------------------------------------------------------
 * For pictures K0 accepts (no HEVC tiles / pcm / transquant bypass ...; csrc/kernels/k0_core.cuh) only the
 * parameter sets and slice headers are parsed on the host; the slice data is unescaped and handed to the engine as
 * bytes, and kernel K0 (one warp per WPP row / per picture, wavefront-synchronised) writes the records straight
 * into HBM. hc_k0_prepare never fails for a well-formed picture: check hc_k0_eligible and fall back to
 * hc_parse_picture + hc_batch_add_picture otherwise. */
typedef struct hc_k0_picture hc_k0_picture;
hc_k0_picture* hc_k0_prepare(const uint8_t* data, size_t size, int stream_format);
void hc_k0_free(hc_k0_picture* k);
int hc_k0_eligible(const hc_k0_picture* k);
const char* hc_k0_why_not(const hc_k0_picture* k);
const hc_pic* hc_k0_pic(const hc_k0_picture* k);          /* header fields only (sizes, formats, VUI) */
size_t hc_k0_upload_bytes(const hc_k0_picture* k);        /* bytes this picture adds to the H2D copy */
/* Same result through the K0 core — the DEVICE CABAC parser (csrc/kernels/k0_core.cuh) — executed on the CPU:
 * the scaffold the tests use to validate K0 record by record. NULL + "not eligible for K0: ..." for pictures K0
 * leaves to the host parser (HEVC tiles, pcm, transquant bypass, ...). */
hc_records* hc_parse_picture_k0(const uint8_t* data, size_t size, int stream_format);
/* One-call convenience: parse one coded picture (parameter sets + slice NALs). */
hc_records* hc_parse_picture(const uint8_t* data, size_t size, int stream_format);

/* ------------------------------------------------------------------ HEIF container -------- */
/* Minimal ISO-BMFF/HEIF item resolver used by the batch decode API (the plugin path gets NAL
 * units from libheif instead). Mirrors what libheif resolves before it calls the decoder plugin:
 * libheif/file.cc:1246-1536, libheif/context.cc:172-221,710-1240. */
typedef struct hc_heif hc_heif;

typedef struct hc_heif_image_info {
  uint32_t id;
  int32_t is_grid;
  int32_t width, height;       /* output size: grid output size or ispe of a single image       */
  int32_t rows, cols;          /* grid layout (1,1 for a single image)                          */
  uint32_t alpha_id;           /* alpha auxiliary image item, 0 if none                         */
  int32_t rot;                 /* irot: anti-clockwise quarter turns                            */
  int32_t mirror;              /* imir: -1 none, 0 vertical axis, 1 horizontal axis             */
  int32_t nclx_present;        /* container colr(nclx) overrides the bitstream VUI              */
  int32_t primaries, transfer, matrix, full_range;
  int32_t n_transforms;        /* irot / imir properties in ipma order (the order the reference applies them) */
  uint8_t transforms[8];       /* HC_XF_*                                                                     */
  int32_t has_clap;            /* number of clean-aperture (clap) properties, consumed in order by HC_XF_CLAP */
  uint32_t claps[4][8];        /* width num/den, height num/den, horizontal offset num/den, vertical offset num/den */
  int32_t premultiplied_alpha; /* a 'prem' reference marks the colour samples as premultiplied by alpha (context.cc:1150-1161) */
} hc_heif_image_info;
#define HC_XF_ROT90 1          /* anti-clockwise quarter turns, HeifPixelImage::rotate_ccw pixelimage.cc:539 */
#define HC_XF_ROT180 2
#define HC_XF_ROT270 3
#define HC_XF_MIRROR_H 4       /* heif_transform_mirror_direction_horizontal: every row reversed (:778-783)  */
#define HC_XF_MIRROR_V 5       /* ..._vertical: row order reversed (:784-789)                                */
#define HC_XF_CLAP 6           /* clean aperture crop (context.cc:1981-2015)                                  */

/* 'iovl' derived image item (ISO/IEC 23008-12 6.6.2.2; libheif ImageOverlay, context.cc:285-369) */
#define HC_OVERLAY_MAX_CHILDREN 16
typedef struct hc_heif_overlay_info {
  int32_t canvas_w, canvas_h;
  uint16_t background[4];      /* R, G, B, A, 16 bit each */
  int32_t n;                   /* referenced images ('dimg'), composed in this order */
  uint32_t children[HC_OVERLAY_MAX_CHILDREN];
  int32_t dx[HC_OVERLAY_MAX_CHILDREN], dy[HC_OVERLAY_MAX_CHILDREN];
} hc_heif_overlay_info;

/* `data` must stay valid until hc_heif_close. NULL + error text on malformed files. */
hc_heif* hc_heif_open(const uint8_t* data, size_t size);
void hc_heif_close(hc_heif* f);
uint32_t hc_heif_primary_id(const hc_heif* f);
/* writes up to `max` ids, returns the total number of top-level images */
int hc_heif_top_level_ids(const hc_heif* f, uint32_t* ids, int max);
/* HC_ERR_ARGUMENT when `id` is not an overlay item */
int hc_heif_get_overlay(const hc_heif* f, uint32_t id, hc_heif_overlay_info* info);
int hc_heif_get_image_info(const hc_heif* f, uint32_t id, hc_heif_image_info* info);
/* row-major tile item ids of a grid; returns rows*cols or a negative error */
int hc_heif_grid_tiles(const hc_heif* f, uint32_t id, uint32_t* tiles, int max);
/* The other images of a file (libheif's heif_image_handle_get_list_of_thumbnail_IDs / ..._auxiliary_image_IDs): the items
 * with a 'thmb' / 'auxl' reference to image `id`, in ascending item id. Writes up to `max` ids and returns the total count.
 * include_alpha = 0 leaves out the alpha images (heif_image_handle_get_list_of_auxiliary_image_IDs with
 * LIBHEIF_AUX_IMAGE_FILTER_OMIT_ALPHA). Any of these items can be decoded by naming it in hc_heic_job_create_items. */
int hc_heif_thumbnail_ids(const hc_heif* f, uint32_t id, uint32_t* ids, int max);
int hc_heif_auxiliary_ids(const hc_heif* f, uint32_t id, int include_alpha, uint32_t* ids, int max);
/* auxC type URN of an auxiliary image (heif_image_handle_get_auxiliary_type), e.g. "urn:mpeg:hevc:2015:auxid:2" for a depth
 * map: copied NUL-terminated into buf (truncated to len - 1 characters); returns its length, HC_ERR_ARGUMENT for an item
 * without auxC. */
int hc_heif_aux_type(const hc_heif* f, uint32_t id, char* buf, size_t len);
/* hvcC parameter sets + item data as 4-byte-length-prefixed NAL units (what libheif gives
 * heif_decoder_plugin::push_data). *out is malloc'ed; release with hc_free. */
int hc_heif_coded_stream(const hc_heif* f, uint32_t id, uint8_t** out, size_t* size);
void hc_free(void* p);

/* ------------------------------------------------------------------ colour conversion ----- */
/* output layouts == heif_chroma_interleaved_* (libheif/api/libheif/heif.h heif_chroma) */
#define HC_OUT_RGB 0
#define HC_OUT_RGBA 1
#define HC_OUT_RRGGBB_BE 2
#define HC_OUT_RRGGBBAA_BE 3
#define HC_OUT_RRGGBB_LE 4
#define HC_OUT_RRGGBBAA_LE 5
/* Native planar output, what heif_decode_image(..., heif_colorspace_undefined, heif_chroma_undefined, ...) returns: the
 * decoded planes as they are (after grid paste, limited->full rescale, irot / imir / clap and the alpha rescale), no colour
 * conversion, no depth change, no chroma resampling. Packed layout of one image: planes Y, Cb, Cr, A in that order, the planes
 * the image lacks left out (monochrome: Y only; A whenever the image has alpha), each plane tight (stride = plane width x
 * sample bytes) and right after the previous one; samples are 1 byte for 8-bit images and 2 bytes little-endian otherwise;
 * chroma planes are (w + 1) / 2 wide for 4:2:0 / 4:2:2 and (h + 1) / 2 high for 4:2:0. See hc_image_plane_layout. */
#define HC_OUT_YCBCR 6

#define HC_CSC_INT420 0 /* Op_YCbCr420_to_RGB24 / _RGB32: 8-bit fixed point      yuv2rgb.cc:260-495 */
#define HC_CSC_FLOAT 1  /* Op_YCbCr_to_RGB<> / Op_YCbCr420_to_RRGGBBaa: fp32     yuv2rgb.cc:28-254,498-643 */
#define HC_CSC_GBR 2    /* matrix_coefficients == 0                               yuv2rgb.cc:197-211 */
#define HC_CSC_YCGCO 3  /* matrix_coefficients == 8                               yuv2rgb.cc:212-226 */
#define HC_CSC_MONO 4   /* Op_mono_to_RGB24_32: R = G = B = Y                     monochrome.cc:150-260 */

/* bit-depth changing plane ops of the reference (hdr_sdr.cc:24-236), fused into K5 */
#define HC_DEPTH_NONE 0
#define HC_DEPTH_TO_SDR 1 /* Op_to_sdr_planes: v >> (depth - 8), no rounding                              */
#define HC_DEPTH_TO_HDR 2 /* Op_to_hdr_planes: (v << (t - 8)) | (v >> (16 - t)), 8 bit -> t bit           */

typedef struct hc_csc_params {
  int32_t mode;          /* HC_CSC_*                                                             */
  int32_t out_format;    /* HC_OUT_*                                                             */
  int32_t full_range;
  int32_t bit_depth;     /* depth the conversion arithmetic runs at (after pre_op)               */
  int32_t r_cr_i, g_cb_i, g_cr_i, b_cb_i; /* lround(256*coefficient), INT420 mode                */
  float r_cr, g_cb, g_cr, b_cb;           /* nclx.cc:151-171                                     */
  int32_t in_depth;      /* sample depth of the decoded planes                                   */
  int32_t out_depth;     /* depth of the written channels: 8 for RGB / RGBA, else the input depth (10 for 8-bit input) */
  int32_t pre_op;        /* HC_DEPTH_* applied to Y, Cb, Cr, A as they are loaded                */
  int32_t post_op;       /* HC_DEPTH_* applied to R, G, B, A before they are written             */
  int32_t premultiply;   /* RGBA 8-bit output only: R, G, B = (v * A + 128) >> 8 (pixelimage.cc:896-941), set by the job */
  int32_t upsampling;    /* HC_UPSAMPLE_*: how 4:2:0 / 4:2:2 chroma is brought to the luma grid                  */
  int32_t coeff_matrix;  /* matrix_coefficients the coefficients were derived from: an unspecified matrix (2) stays 2 —
                            the literal BT.601 defaults — when the matrix op is the first op of the reference's chain and
                            becomes 6 behind any other op (see csc_select.cc)                     */
} hc_csc_params;

/* HC_OUT_YCBCR is accepted for every chroma format, bit depth and matrix (11 / 14 included: nothing is converted) and gives
 * parameters that describe an identity: in_depth = out_depth = bit_depth = the image's bit depth, no pre / post op. */
/* Chooses the conversion the reference's pipeline would run with default decoding options
 * (colorconversion.cc:266-420, table in SURVEY.md 3.5) and fills the coefficients exactly as
 * nclx.cc:82-171 computes them. `matrix`/`primaries`/`full_range` are the image's nclx values
 * (pass matrix=2 for "unspecified": replaced by BT.601 like nclx.cc:346-359); matrix 12 / 13 derive Kr / Kb from the
 * chromaticities of `primaries` (nclx.cc:88-110). Every output format is available for every bit depth: the reference
 * inserts Op_to_sdr_planes / Op_to_hdr_planes (hdr_sdr.cc) before or after the matrix depending on the input — the chain
 * it picks (tools/csc_pipeline_probe.cc asks the unmodified reference; table in DESIGN.md) is encoded in pre_op / post_op.
 * Returns HC_ERR_UNSUPPORTED for combinations the reference cannot convert either (matrix 11/14). */
int hc_csc_select(int matrix, int primaries, int full_range, int chroma_format, int bit_depth,
                  int has_alpha, int out_format, hc_csc_params* out);
/* Chroma upsampling choice of heif_color_conversion_options (heif.h:1546-1562). NEAREST is what the reference's pipeline
 * search ends up with under its default options. BILINEAR mirrors `preferred_chroma_upsampling_algorithm = bilinear,
 * only_use_preferred_chroma_algorithm = true` (what heif-dec -C bilinear sets, examples/heif_dec.cc:502-509):
 * Op_YCbCr420/422_bilinear_to_YCbCr444 (chroma_sampling.cc:441-933, border rules included) in front of Op_YCbCr_to_RGB<>.
 * 4:4:4 images convert as usual; matrix_coefficients 0 with subsampled chroma has no pipeline in the reference either
 * (HC_ERR_UNSUPPORTED), nor has monochrome input to RRGGBB(AA) here. */
#define HC_UPSAMPLE_NEAREST 0
#define HC_UPSAMPLE_BILINEAR 1
int hc_csc_select_opt(int matrix, int primaries, int full_range, int chroma_format, int bit_depth,
                      int has_alpha, int out_format, int upsampling, hc_csc_params* out);

/* ------------------------------------------------------------------ device engine ---------- */
typedef struct hc_engine hc_engine;
typedef struct hc_batch hc_batch;

/* Creates the engine on CUDA device `device`. NULL + HC_ERR_NO_DEVICE text when no usable GPU is
 * present: there is deliberately no CPU fallback. */
hc_engine* hc_engine_create(int device);
void hc_engine_destroy(hc_engine* e);
/* Options: "device_parse" (default 1; environment HEIFCUDA_PARSER=host sets 0): hc_heic_job / hc_heic_decode_stream
 * let kernel K0 parse the slice data of every picture it accepts instead of the host CABAC parser.
 * "host_share_pct" (environment HEIFCUDA_HOST_SHARE): with device_parse, this percentage of the coded items of every job
 * is parsed by the host threads instead, which run while the GPU is busy with the previous batch of
 * hc_heic_decode_stream (hybrid parse). Default -1 = automatic: none for a single hc_heic_job, and in
 * hc_heic_decode_stream a share that follows the measured host / GPU time per batch.
 * "stream_depth" (environment HEIFCUDA_STREAM_DEPTH; default 0 = automatic): batches hc_heic_decode_stream keeps in flight,
 * 2..6. Automatic: 3, or 6 once a batch's read-back is measured to take more than 0.4 of the period between completions
 * (several GPUs reading back over one host link); the engine remembers the choice for its next call.
 * "chroma_upsampling" (default HC_UPSAMPLE_NEAREST): HC_UPSAMPLE_BILINEAR makes hc_heic_job / hc_heic_decode_stream convert
 * with bilinear chroma upsampling (see hc_csc_select_opt).
 * "premultiply_alpha" (default 0): 1 makes hc_heic_job / hc_heic_decode_stream multiply interleaved RGBA 8-bit output by its
 * alpha like heif_image_rgba_premultiply_alpha (heif.cc:1444-1490, pixelimage.cc:896-941: (v * A + 128) >> 8), fused into K5;
 * images the file already marks premultiplied ('prem') are left alone, as that call refuses them.
 * "k0_max_critical_ctbs" (default 160): K0 is serial per substream, so hc_heic_job only hands it pictures whose parse
 * critical path is at most this many CTBs (WPP: CTB columns + 2 x (CTB rows - 1); no WPP: all CTBs of the picture);
 * the others stay with the host parser.
 * "scale_max_side" (default 0 = off; negative: HC_ERR_ARGUMENT): hc_heic_job / hc_heic_decode_stream deliver every image
 * whose full-size output W x H (after irot / imir / clap and the alpha link: what hc_image_desc reported without the option)
 * has max(W, H) > S as a smaller image that fits S: W >= H -> S x max(1, H * S / W), else max(1, W * S / H) x S (integer
 * division). Images within S are delivered unchanged; the option never enlarges. This is the library's fit rule (no claim of
 * parity with any thumbnailer). The pixels are those of heif_image_scale_image (nearest neighbour, see
 * hc_batch_set_canvas_output_size) applied to the full-size output, which is never written: K5 / K7 convert only the
 * sampled pixels. hc_image_desc then reports the delivered size, and the stream's buffers, external-destination check and
 * stats follow it. Read when a job is created. Not available with HC_OUT_YCBCR (a job fails at creation,
 * hc_heic_decode_stream(_ext) fails the call with HC_ERR_UNSUPPORTED) nor for band jobs (hc_heic_job_create_band fails);
 * hc_heic_job_set_rgb_target and hc_heic_job_read_plane refuse a scaled image (HC_ERR_UNSUPPORTED). */
int hc_engine_set_option(hc_engine* e, const char* name, int value);
int hc_engine_get_option(const hc_engine* e, const char* name);

/* A batch = a set of parsed pictures placed on destination canvases (one canvas per output
 * image: a single picture, or a HEIF grid whose tiles are pasted at their offsets). */
hc_batch* hc_batch_create(hc_engine* e);
void hc_batch_destroy(hc_batch* b);
/* returns the canvas index (>= 0) */
int hc_batch_add_canvas(hc_batch* b, int width, int height, int chroma_format, int bit_depth, int with_alpha);
#define HC_ROLE_COLOUR 0
#define HC_ROLE_ALPHA 1 /* the picture's luma becomes the canvas' alpha plane (context.cc:2029-2078) */
#define HC_ROLE_LUMA 2  /* only the picture's luma is kept, as plane 0 of a (monochrome) canvas: an alpha image that is
                         * decoded on its own because its size differs from the colour image's (hc_batch_link_alpha) */
/* `rec` must stay alive until hc_batch_upload returns. (x,y): paste position of the picture's
 * conformance window on the canvas, luma samples. rescale_limited: apply the reference's
 * limited->full range rescale while pasting (grid tiles whose nclx is limited range). */
int hc_batch_add_picture(hc_batch* b, const hc_records* rec, int canvas, int x, int y, int role, int rescale_limited);
/* Adds a picture whose slice data is parsed by K0 on the device. `k` must stay alive until hc_batch_upload returns. */
int hc_batch_add_k0_picture(hc_batch* b, const hc_k0_picture* k, int canvas, int x, int y, int role, int rescale_limited);
int hc_batch_k0_pictures(const hc_batch* b);              /* pictures of the batch that K0 parses */
/* packs all records into one pinned arena and copies it to the device (async on the engine stream) */
int hc_batch_upload(hc_batch* b);
#define HC_STAGE_DEBLOCK 1
#define HC_STAGE_SAO 2
#define HC_STAGE_ALL 3
/* [K0 (device CABAC parse) ->] K1 (dequant+transform) -> K2 (intra wavefront) -> K3 (deblock) -> K4 (SAO+crop+paste).
 * Asynchronous for host-parsed batches; a batch with device-parsed pictures waits for K0's verdict so that malformed
 * slice data is reported here (HC_ERR_BITSTREAM). */
int hc_batch_reconstruct(hc_batch* b, int stages);
/* Same, never waits: a K0 parse error is reported by the next synchronising call on the batch (hc_batch_sync,
 * hc_batch_read_*, hc_batch_stage_ms). */
int hc_batch_reconstruct_async(hc_batch* b, int stages);
/* Geometric transform of a canvas between K4 and K5 (irot / imir of the reference, applied plane by plane like
 * HeifPixelImage::rotate_ccw / mirror_inplace): output sample (x', y') of a plane of w x h input samples is input
 * sample (sx, sy) with  !swap: sx = flip_x ? w-1-x' : x', sy = flip_y ? h-1-y' : y'   (output w x h)
 *                        swap: sx = flip_x ? w-1-y' : y', sy = flip_y ? h-1-x' : x'   (output h x w).
 * Call before hc_batch_upload. hc_batch_convert / read_rgb / read_plane then see the transformed canvas. */
int hc_batch_set_canvas_transform(hc_batch* b, int canvas, int swap, int flip_x, int flip_y);
/* General form: an ordered list of passes per canvas (set_canvas_transform replaces the list by one dihedral pass).
 * HC_PASS_DIHEDRAL: a0 = swap, a1 = flip_x, a2 = flip_y as above. HC_PASS_CROP: the window [a0, a2] x [a1, a3]
 * (left, top, right, bottom, inclusive, in pixels of the image at that point), scaled to every plane like
 * HeifPixelImage::crop does (pixelimage.cc:797-870) — the clap property of the reference. */
#define HC_PASS_DIHEDRAL 0
#define HC_PASS_CROP 1
int hc_batch_add_canvas_pass(hc_batch* b, int canvas, int kind, int a0, int a1, int a2, int a3);
/* The alpha plane of `canvas` (created with_alpha) is plane 0 of `alpha_canvas`, rescaled to the size of `canvas` by
 * nearest neighbour exactly like HeifPixelImage::scale_nearest_neighbor (pixelimage.cc:1156-1253: ix = x * in_w / out_w,
 * iy = y * in_h / out_h) as HeifContext::decode_image_planar does for an alpha image whose size differs from the colour
 * image's (context.cc:2064-2071). Both canvases are taken after their own geometric passes. Call before hc_batch_upload. */
int hc_batch_link_alpha(hc_batch* b, int canvas, int alpha_canvas);
/* Delivered size of a canvas (any width, height >= 1, smaller or larger): pixel (x, y) of the delivered image is pixel
 * (x * W / width, y * H / height) of the full-size interleaved image (W x H: the canvas after its passes; 64-bit products,
 * integer division) — HeifPixelImage::scale_nearest_neighbor (pixelimage.cc:1156-1253), i.e. heif_image_scale_image on the
 * converted image. Every per-pixel step of K5 / K7 runs at the source pixel as without it. Call before hc_batch_upload;
 * overlay canvases included. hc_batch_convert(_many), hc_batch_read_rgb(_async) and hc_batch_copy_rgb_device then see the
 * delivered size; hc_batch_read_plane(s) keep returning the full-size planes. HC_ERR_UNSUPPORTED for a canvas with an
 * external RGB target; a scaled canvas cannot be converted to HC_OUT_YCBCR nor take an external target either. */
int hc_batch_set_canvas_output_size(hc_batch* b, int canvas, int width, int height);
/* 'iovl' derived image (libheif context.cc:2579-2675): an output canvas without planes of its own. K7 fills it with the
 * background colour (16-bit R, G, B, A as stored in the item; the reference keeps the high byte of R, G, B) and overlays
 * the child canvases in the order they are added at (dx, dy) — copied, or alpha-blended when the child canvas has an alpha
 * plane — and writes the interleaved result (hc_batch_convert_many with this canvas; params[].out_format selects the
 * format, RGB(A) or RRGGBB(AA) at 10 bit like the reference). child_params: hc_csc_select(..., HC_OUT_RGB) of the child
 * (Op_YCbCr_to_RGB<uint8_t>). Children must be 8-bit 4:4:4 canvases (the reference converts nothing else) with offsets >= 0. */
int hc_batch_add_overlay_canvas(hc_batch* b, int width, int height, const uint16_t background[4]);
int hc_batch_overlay_add_child(hc_batch* b, int overlay_canvas, int child_canvas, int dx, int dy, const hc_csc_params* child_params);
/* K5 / K7 / K8 for n canvases (canvases[i] with params[i]) in as few launches as possible, async. K5 converts a canvas into
 * the batch's device RGB buffer, K7 composes an overlay canvas (hc_batch_add_overlay_canvas) there; a canvas whose params have
 * out_format == HC_OUT_YCBCR goes to K8 instead, which packs the canvas' output planes into the same buffer in the layout of
 * HC_OUT_YCBCR. Overlay canvases and canvases with an external RGB target (hc_batch_set_rgb_target) cannot be planar:
 * HC_ERR_UNSUPPORTED.
 * The buffer holds one block per canvas in canvas order, sized by the canvas' output format (8 bytes per pixel before its
 * first conversion). A call lays out anew the canvases it names and those not converted yet; a converted canvas it does not
 * name keeps its block and its bytes. When the new layout would move such a canvas, or the buffer would have to grow while one
 * exists, the call fails with HC_ERR_ARGUMENT and changes nothing: convert it again in the same call. */
int hc_batch_convert_many(hc_batch* b, int n, const int* canvases, const hc_csc_params* params);
/* hc_batch_convert_many for one canvas */
int hc_batch_convert(hc_batch* b, int canvas, const hc_csc_params* params);
int hc_batch_sync(hc_batch* b);
/* D2H reads (synchronous). plane: 0 Y, 1 Cb, 2 Cr, 3 alpha. Samples are 1 byte for 8-bit canvases,
 * 2 bytes little-endian otherwise. */
int hc_batch_read_plane(hc_batch* b, int canvas, int plane, void* dst, size_t dst_stride_bytes);
/* planes 0..nplanes-1 of a canvas with one synchronisation (pinned staging inside) */
int hc_batch_read_planes(hc_batch* b, int canvas, int nplanes, void* const* dst, const size_t* dst_strides);
/* The converted image of a canvas. For a canvas converted to HC_OUT_YCBCR these copy its packed planes with one 1-D copy
 * (hc_image_plane_layout bytes); dst_stride_bytes must then be the tight Y row (width x sample bytes), else HC_ERR_ARGUMENT. */
int hc_batch_read_rgb(hc_batch* b, int canvas, void* dst, size_t dst_stride_bytes);
int hc_batch_copy_rgb_device(hc_batch* b, int canvas, void* device_dst, size_t dst_stride_bytes);
/* same copy without the final synchronisation (dst should be pinned); pair with hc_batch_sync */
int hc_batch_read_rgb_async(hc_batch* b, int canvas, void* dst, size_t dst_stride_bytes);
/* residuals of picture `pic` as produced by K1 (resid_count int16) — used by the parity tests */
int hc_batch_read_residual(hc_batch* b, int pic, int16_t* dst, size_t count);
/* device time of the last run's stages in ms (CUDA events on the engine stream):
 * [0] H2D upload, [1] K1, [2] K2, [3] K3, [4] K4, [5] K5 / K8 (sum over convert calls), [6] D2H of the last read,
 * [7] K0 (device CABAC parse; runs once per upload, the records then stay resident) */
int hc_batch_stage_ms(hc_batch* b, float ms[8]);
/* CUDA-event stopwatch on the batch's stream: start records an event; stop records a second one,
 * waits for it and returns the device time between the two in ms (used by bench.py to time K
 * steps on the stream the kernels are launched on). */
int hc_batch_timer_start(hc_batch* b);
int hc_batch_timer_stop_ms(hc_batch* b, float* ms);
/* number of kernel launches issued by the last reconstruct + convert calls */
int hc_batch_launch_count(const hc_batch* b);
/* bytes of the packed record arena uploaded by hc_batch_upload */
size_t hc_batch_upload_bytes(const hc_batch* b);

/* ------------------------------------------------------------------ HEIC batch decode ------ */
/* The call a user of the reference makes is heif_decode_image(handle, &img, heif_colorspace_RGB,
 * heif_chroma_interleaved_*, opts) per file (libheif/api/libheif/heif.cc:1150), which walks
 * HeifContext::decode_image_user (context.cc:1516): container -> one decoder instance per coded
 * item -> paste -> colour conversion. hc_heic_job is the same walk for MANY files at once: all
 * coded items (single images, every grid tile, alpha auxiliary images) of all files are parsed by
 * a pool of host threads and reconstructed on the GPU as one batch. */
typedef struct hc_heic_job hc_heic_job;

typedef struct hc_image_desc {
  int32_t width, height;     /* output size in pixels (the delivered size under "scale_max_side") */
  int32_t chroma_format;     /* of the decoded YCbCr image                                        */
  int32_t bit_depth;
  int32_t has_alpha;
  int32_t out_format;        /* HC_OUT_* of this image (automatic: 8-bit -> RGB/RGBA, else RRGGBB(AA)_LE) */
  int32_t bytes_per_pixel;   /* HC_OUT_YCBCR: bytes per sample (1 or 2), so width * bytes_per_pixel is the Y row       */
  int32_t coded_pictures;    /* HEVC pictures decoded for this image (tiles + alpha)              */
  int32_t premultiplied_alpha; /* heif_image_is_premultiplied_alpha of the result: the file says so ('prem'), or the engine option
                                "premultiply_alpha" multiplied the RGBA output (heif_image_rgba_premultiply_alpha; never for
                                HC_OUT_YCBCR, which that call does not take) */
} hc_image_desc;

/* Packed layout of an HC_OUT_YCBCR image (see HC_OUT_YCBCR): byte offset, stride in bytes, width and height in samples of
 * planes 0 Y, 1 Cb, 2 Cr, 3 A; a plane the image lacks gets width, height and stride 0. Any of the arrays may be NULL.
 * Returns the total packed bytes, or 0 for a desc of another output format. */
size_t hc_image_plane_layout(const hc_image_desc* d, size_t offset[4], size_t stride[4], int32_t width[4], int32_t height[4]);

/* Parses `nfiles` HEIC files held in host memory (the primary image of each) with `threads` host
 * threads (<=0: hardware concurrency). The buffers must stay valid until hc_heic_job_destroy.
 * want_alpha: 0 -> interleaved RGB / RRGGBB_LE, 1 -> RGBA / RRGGBBAA_LE (8-bit images / deeper images), or
 * HC_OUTPUT_FORMAT(HC_OUT_*) -> that format for every image whatever its bit depth, like the `chroma` argument of
 * heif_decode_image (heif.cc:1150): a 10-bit image to interleaved RGB goes through the reference's Op_to_sdr_planes, an
 * 8-bit image to RRGGBB through Op_to_hdr_planes (10 bit), both fused into K5. The same encoding is accepted by
 * hc_heic_job_create_band and hc_heic_decode_stream.
 * HC_OUTPUT_FORMAT(HC_OUT_YCBCR): every image as its native planes (heif_colorspace_undefined / heif_chroma_undefined),
 * packed by K8; hc_heic_job_read_rgb then copies the packed planes (stride = the Y row). A is delivered whenever the image has
 * alpha. The "premultiply_alpha" and "chroma_upsampling" options do not apply. Overlay ('iovl') images, which the reference
 * composes in RGB, fail as unsupported images, and so does an image whose clean aperture (clap) leaves chroma planes of
 * another size than the packed layout: the reference scales the crop window to each plane by integer division, so a 4:2:0 /
 * 4:2:2 window at an odd column with an even width (4:2:0: or at an odd row with an even height) keeps one chroma sample
 * more than (w + 1) / 2 (h + 1) / 2. With error isolation (hc_heic_decode_stream_ext) each such file fails alone.
 * hc_heic_job_create_band and hc_heic_job_set_rgb_target refuse the format. */
#define HC_OUTPUT_FORMAT(fmt) (0x100 | (fmt))
hc_heic_job* hc_heic_job_create(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes,
                                int want_alpha, int threads);
/* Any image item, not only the primary one (heif_context_get_image_handle / heif_image_handle_get_thumbnail /
 * heif_image_handle_get_auxiliary_image_handle + heif_decode_image): image k of the job is item item_ids[k] of buffer k,
 * 0 = its primary image; item_ids == NULL is hc_heic_job_create. The same buffer may appear in several entries. The item is
 * decoded exactly as a primary image would be: its own irot / imir / clap, its own alpha image (an 'auxl' alpha referring to
 * it, at any size), its own colr, its 'prem' flag, grid and 'iovl' composition. Any 'hvc1', 'grid' or 'iovl' item may be
 * named: hidden items, thumbnails, auxiliary images (an alpha or depth image decodes as a monochrome image), grid tiles.
 * Any other item ('Exif', 'mime', 'iden', a missing id) fails the job with a text that names the item. */
hc_heic_job* hc_heic_job_create_items(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes,
                                      const uint32_t* item_ids, int want_alpha, int threads);
/* Multi-GPU decode of ONE huge grid image (BASELINE config C5): every GPU decodes a band of tile rows
 * [tile_row_begin, tile_row_end) of the primary grid image; the job's single output image is that band
 * (desc.height = band height). *first_output_row / *full_height place the band in the whole picture; the
 * caller stitches the bands into the owner GPU's buffer with peer copies (hc_heic_job_copy_rgb_device +
 * NCCL send/recv or cudaMemcpyPeer). HEIF grid tiles are independent pictures (context.cc:2407-2415), so no
 * data crosses GPUs before the stitch. */
hc_heic_job* hc_heic_job_create_band(hc_engine* e, const uint8_t* data, size_t size, int want_alpha, int threads,
                                     int tile_row_begin, int tile_row_end, int* first_output_row, int* full_height);
/* ---- one huge grid image on several GPUs (BASELINE config C5; reference: one process, std::async per tile,
 * libheif/context.cc:2120-2404) ----
 * The output lives in ONE device buffer on the owner GPU (hc_shared_image). Every GPU decodes a band of tile rows
 * (hc_heic_job_create_band) and its K5 writes the band's RGB rows straight into the owner's buffer: ordinary stores on the
 * owner, NVLink peer stores everywhere else (cudaDeviceEnablePeerAccess within one process, CUDA IPC between the
 * processes of a one-process-per-GPU launch). No collective, no staging copy. */
typedef struct hc_shared_image hc_shared_image;
#define HC_IPC_HANDLE_BYTES 64
/* owner: `height` rows of `width` pixels of `bytes_per_pixel` on the engine's device (rows padded for K5's 8-pixel units) */
hc_shared_image* hc_shared_image_create(hc_engine* e, int width, int height, int bytes_per_pixel);
/* another PROCESS: the owner exports 64 bytes, the peer opens them on its own engine's device */
int hc_shared_image_export(const hc_shared_image* s, uint8_t handle[HC_IPC_HANDLE_BYTES]);
hc_shared_image* hc_shared_image_open(hc_engine* e, const uint8_t handle[HC_IPC_HANDLE_BYTES], int width, int height, int bytes_per_pixel);
/* another engine (device) of the SAME process: enables peer access from e's device to the owner's */
hc_shared_image* hc_shared_image_attach(hc_engine* e, const hc_shared_image* owner);
void hc_shared_image_destroy(hc_shared_image* s);
void* hc_shared_image_device_ptr(const hc_shared_image* s);
size_t hc_shared_image_stride(const hc_shared_image* s);
/* owner: rows [first_row, first_row + rows) to host memory, synchronous (device-wide: call it after every writer's
 * hc_heic_job_sync and whatever barrier orders the writers before the reader) */
int hc_shared_image_read(hc_shared_image* s, int first_row, int rows, void* dst, size_t dst_stride_bytes);
/* K5 of image `image` writes its rows to rows [first_row, ...) of `dst` instead of the job's own RGB buffer. Call before
 * hc_heic_job_run; hc_heic_job_read_rgb is not available for such an image. HC_ERR_UNSUPPORTED for HC_OUT_YCBCR images. */
int hc_heic_job_set_rgb_target(hc_heic_job* j, int image, hc_shared_image* dst, int first_row);
/* same at batch level: any device pointer K5 may store to (peer-mapped or local), rows `stride_bytes` apart;
 * HC_ERR_UNSUPPORTED for a canvas converted to HC_OUT_YCBCR */
int hc_batch_set_rgb_target(hc_batch* b, int canvas, void* device_dst, size_t stride_bytes);
/* device-to-device copy of a converted image into caller-owned device memory (any device reachable from the job's: the copy
 * is a peer copy over NVLink then), synchronous */
int hc_heic_job_copy_rgb_device(hc_heic_job* j, int image, void* device_dst, size_t dst_stride_bytes);
void hc_heic_job_destroy(hc_heic_job* j);
int hc_heic_job_image_count(const hc_heic_job* j);
int hc_heic_job_image_desc(const hc_heic_job* j, int image, hc_image_desc* desc);
/* H2D upload of the packed records (async). */
int hc_heic_job_upload(hc_heic_job* j);
/* K1..K4 for all pictures + K5 for every image (async; may be called repeatedly after one upload). */
int hc_heic_job_run(hc_heic_job* j);
int hc_heic_job_sync(hc_heic_job* j);
/* copies image `image` to host memory (dst_stride_bytes >= width*bytes_per_pixel), synchronous */
int hc_heic_job_read_rgb(hc_heic_job* j, int image, void* dst, size_t dst_stride_bytes);
/* decoded planes of an image (0 Y, 1 Cb, 2 Cr, 3 alpha), as the plugin ABI would return them */
int hc_heic_job_read_plane(hc_heic_job* j, int image, int plane, void* dst, size_t dst_stride_bytes);
/* stage timings of the last run (see hc_batch_stage_ms), launches, uploaded bytes, host parse seconds */
int hc_heic_job_stage_ms(hc_heic_job* j, float ms[8]);
int hc_heic_job_timer_start(hc_heic_job* j);
int hc_heic_job_timer_stop_ms(hc_heic_job* j, float* ms);
int hc_heic_job_launch_count(const hc_heic_job* j);
size_t hc_heic_job_upload_bytes(const hc_heic_job* j);
double hc_heic_job_parse_seconds(const hc_heic_job* j);

/* Streaming form for long file lists (BASELINE config C4: thousands of files): the files are cut
 * into batches of `files_per_batch` (0: chosen by the library, about 800 MP of output per batch — 64 files of 12 MP, 384 of
 * 1080p: the device parser needs some 20,000 substreams in flight); while batch b is uploaded, reconstructed, converted and read
 * back, the host threads already parse batch b+1. Every finished image is handed to `on_image`
 * (called on the calling thread, in file order) as tightly strided rows in PINNED host memory that
 * stays valid until the callback returns. Returns HC_OK or the first error (hc_last_error). */
typedef void (*hc_image_callback)(void* user, int file_index, const hc_image_desc* desc, const void* pixels,
                                  size_t stride_bytes);
typedef struct hc_stream_stats {
  double seconds_total;      /* wall time of the call                                             */
  double seconds_parse;      /* sum over batches of the host parse phase (overlaps the GPU phase) */
  double seconds_gpu_phase;  /* sum over batches of upload + kernels + read-back (host wall time) */
  double device_ms;          /* sum over batches of K1..K5 device time                            */
  uint64_t bytes_h2d, bytes_d2h;
  int64_t pixels;            /* output pixels delivered                                           */
  int32_t batches, launches;
  int32_t files_failed;      /* files reported through file_status (hc_heic_decode_stream_ext)   */
  int32_t depth;             /* batches in flight at the end of the call (3, or 6 when read-backs are slow) */
} hc_stream_stats;
int hc_heic_decode_stream(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes, int want_alpha,
                          int threads, int files_per_batch, hc_image_callback on_image, void* user,
                          hc_stream_stats* stats);
/* External destinations (the reference's heif_decoding_options::ext_dst / heif_decoding_options_add_external_dest,
 * heif.h:1605-1615; HeifPixelImage::add_shared_rgba_plane, pixelimage.cc:221-266): dests[k] describes where the final
 * pixels of file k go — `len` bytes at `dst` (pinned memory makes the copy asynchronous), rows `stride` bytes apart. Like
 * the reference, a destination that is absent or too small (len < stride * (height - 1) + row bytes, or stride < row
 * bytes) is ignored and the image is delivered in the library's own pinned memory; the callback receives whichever pointer
 * and stride were used. dests may be NULL.
 * HC_OUT_YCBCR: the callback gets the base of the packed planes and stride_bytes = the Y row. A destination is used when
 * len >= hc_image_plane_layout(...) and stride is 0 or the Y row, and ignored otherwise. stats->bytes_d2h counts the packed
 * bytes.
 * Error isolation: with file_status == NULL the first file that cannot be decoded fails the whole call (hc_heic_decode_stream).
 * With file_status != NULL (nfiles entries) such a file gets its error code there and no callback, every other file is
 * delivered, and the call returns HC_OK unless something other than the content of a file went wrong (CUDA, memory);
 * stats->files_failed counts them and hc_last_error() describes the first. A damaged container, unsupported coding tools,
 * slice data the parser rejects and the device parser's capacity limit are all per-file errors. */
typedef struct hc_stream_dest {
  void* dst;
  size_t len;
  size_t stride;
} hc_stream_dest;
int hc_heic_decode_stream_ext(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes, int want_alpha,
                              int threads, int files_per_batch, const hc_stream_dest* dests, int* file_status,
                              hc_image_callback on_image, void* user, hc_stream_stats* stats);
/* hc_heic_decode_stream_ext over entries that name an image item each (see hc_heic_job_create_items): entry k is item
 * item_ids[k] of buffer k (0 = the primary image), and file_index, file_status[k] and dests[k] refer to entry k; item_ids ==
 * NULL is hc_heic_decode_stream_ext. The automatic batch size (files_per_batch == 0) follows the size of the named items, so
 * a list of thumbnails goes in large batches. An entry naming an item that cannot be decoded fails alone under error
 * isolation. */
int hc_heic_decode_stream_items(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes, const uint32_t* item_ids,
                                int want_alpha, int threads, int files_per_batch, const hc_stream_dest* dests, int* file_status,
                                hc_image_callback on_image, void* user, hc_stream_stats* stats);
/* pinned host memory for fast H2D/D2H in the caller (NULL when no CUDA engine) */
void* hc_host_alloc(size_t bytes);
void hc_host_free(void* p);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* HEIFCUDA_H */
