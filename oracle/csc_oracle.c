/*
 * csc_oracle.c — CPU restatement of the reference's YCbCr -> interleaved RGB conversion chain.
 *
 * TEST INFRASTRUCTURE ONLY (see hevc_recon_oracle.c). Parity status: PINNED against the unmodified
 * reference's heif_decode_image() output on its bundled HEIC files (golden MD5s, SURVEY.md §8c) and
 * against oracle/_ref on synthetic grids (tests/test_oracle_golden.py).
 *
 * Follows, with paths relative to /root/reference/libheif/:
 *   nclx.cc:82-171                 Kr/Kb and matrix coefficients
 *   colorconversion.cc:266-420     which op chain is chosen (resolved table: SURVEY.md §3.5)
 *   color-conversion/yuv2rgb.cc:260-495   Op_YCbCr420_to_RGB24 / _RGB32 (8-bit fixed point)
 *   color-conversion/yuv2rgb.cc:28-254    Op_YCbCr_to_RGB<Pixel> (fp32)
 *   color-conversion/yuv2rgb.cc:498-643   Op_YCbCr420_to_RRGGBBaa (fp32)
 *   color-conversion/rgb2rgb.cc:28-272,613-729  interleave / endianness ops
 *   color-conversion/hdr_sdr.cc:24-236    Op_to_hdr_planes / Op_to_sdr_planes (bit-depth changes)
 *   color-conversion/monochrome.cc:53-140  Op_mono_to_YCbCr420
 *   common_utils.h:56-79           clip helpers
 * Compile with -ffp-contract=off: every float product and sum is rounded separately, as in the
 * reference's SSE2 build.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include "oracle_counters.h"

static void count_clip(int lo, int maxi) {
  switch (maxi) {
    case 255: if (lo) HC_COUNT(k5_clip_lo_8); else HC_COUNT(k5_clip_hi_8); break;
    case 1023: if (lo) HC_COUNT(k5_clip_lo_10); else HC_COUNT(k5_clip_hi_10); break;
    case 4095: if (lo) HC_COUNT(k5_clip_lo_12); else HC_COUNT(k5_clip_hi_12); break;
    default: break;
  }
}
static uint16_t clip_f_u16(float fx, int32_t maxi) { /* common_utils.h:64-70 */
  long x = (long)(fx + 0.5f);
  if (x < 0) { count_clip(1, maxi); return 0; }
  if (x > maxi) { count_clip(0, maxi); return (uint16_t)maxi; }
  return (uint16_t)x;
}
static uint8_t clip_int_u8(int x) {
  if (x < 0 || x > 255) count_clip(x < 0, 255);
  return x < 0 ? 0 : (x > 255 ? 255 : (uint8_t)x);
}

typedef struct { float r_cr, g_cb, g_cr, b_cb; } coeffs_t;

/* nclx.cc:46-75 get_colour_primaries: {green x,y, blue x,y, red x,y, white x,y}; zeros when undefined */
static int get_primaries(int idx, float p[8]) {
  static const float tab[][9] = {
      {1, 0.300f, 0.600f, 0.150f, 0.060f, 0.640f, 0.330f, 0.3127f, 0.3290f}, {4, 0.21f, 0.71f, 0.14f, 0.08f, 0.67f, 0.33f, 0.310f, 0.316f},
      {5, 0.29f, 0.60f, 0.15f, 0.06f, 0.64f, 0.33f, 0.3127f, 0.3290f},       {6, 0.310f, 0.595f, 0.155f, 0.070f, 0.630f, 0.340f, 0.3127f, 0.3290f},
      {7, 0.310f, 0.595f, 0.155f, 0.070f, 0.630f, 0.340f, 0.3127f, 0.3290f}, {8, 0.243f, 0.692f, 0.145f, 0.049f, 0.681f, 0.319f, 0.310f, 0.316f},
      {9, 0.170f, 0.797f, 0.131f, 0.046f, 0.708f, 0.292f, 0.3127f, 0.3290f}, {10, 0.0f, 1.0f, 0.0f, 0.0f, 1.0f, 0.0f, 0.333333f, 0.33333f},
      {11, 0.265f, 0.690f, 0.150f, 0.060f, 0.680f, 0.320f, 0.314f, 0.351f},  {12, 0.265f, 0.690f, 0.150f, 0.060f, 0.680f, 0.320f, 0.3127f, 0.3290f},
      {22, 0.295f, 0.605f, 0.155f, 0.077f, 0.630f, 0.340f, 0.3127f, 0.3290f}};
  for (size_t i = 0; i < sizeof(tab) / sizeof(tab[0]); i++)
    if ((int)tab[i][0] == idx) { for (int k = 0; k < 8; k++) p[k] = tab[i][1 + k]; return 1; }
  for (int k = 0; k < 8; k++) p[k] = 0.f;
  return 0;
}

static coeffs_t get_coeffs(int matrix, int primaries) { /* nclx.cc:82-171 */
  float Kr = 0.f, Kb = 0.f;
  if (matrix == 12 || matrix == 13) { /* nclx.cc:88-110: Kr / Kb from the chromaticities of the colour primaries */
    float p[8];
    get_primaries(primaries, p);
    const float gx = p[0], gy = p[1], bx = p[2], by = p[3], rx = p[4], ry = p[5], wx = p[6], wy = p[7];
    const float zr = 1 - (rx + ry), zg = 1 - (gx + gy), zb = 1 - (bx + by), zw = 1 - (wx + wy);
    const float denom = wy * (rx * (gy * zb - by * zg) + gx * (by * zr - ry * zb) + bx * (ry * zg - gy * zr));
    if (denom != 0.0f) {
      Kr = (ry * (wx * (gy * zb - by * zg) + wy * (bx * zg - gx * zb) + zw * (gx * by - bx * gy))) / denom;
      Kb = (by * (wx * (ry * zg - gy * zr) + wy * (gx * zr - rx * zg) + zw * (rx * gy - gx * ry))) / denom;
    }
  } else {
    switch (matrix) {
      case 1: Kr = 0.2126f; Kb = 0.0722f; break;
      case 4: Kr = 0.30f; Kb = 0.11f; break;
      case 5: case 6: Kr = 0.299f; Kb = 0.114f; break;
      case 7: Kr = 0.212f; Kb = 0.087f; break;
      case 9: case 10: Kr = 0.2627f; Kb = 0.0593f; break;
      default: break;
    }
  }
  coeffs_t c;
  if (Kb != 0 || Kr != 0) {
    c.r_cr = 2 * (-Kr + 1);
    c.g_cb = 2 * Kb * (-Kb + 1) / (Kb + Kr - 1);
    c.g_cr = 2 * Kr * (-Kr + 1) / (Kb + Kr - 1);
    c.b_cb = 2 * (-Kb + 1);
  } else {
    c.r_cr = 1.402f; c.g_cb = -0.344136f; c.g_cr = -0.714136f; c.b_cb = 1.772f;
  }
  return c;
}

/* hdr_sdr.cc:54-97 Op_to_hdr_planes (8 -> out_bits) and :140-236 Op_to_sdr_planes (in_bits -> 8, no rounding) */
static int to_hdr(int v, int out_bits) { return ((v << (out_bits - 8)) | (v >> (16 - out_bits))) & 0xffff; }
static int to_sdr(int v, int in_bits) { return (v >> (in_bits - 8)) & 0xff; }

/* Op_YCbCr420_bilinear_to_YCbCr444 (chroma_sampling.cc:441-705) on one chroma plane, restated loop by loop: borders
 * first (the first / last row and column index the chroma row with cx / 2, as the reference does), then every 2x2 square
 * between four chroma samples. `in` has ((w+1)/2) x ((h+1)/2) samples, `out` w x h. */
void hc_oracle_bilinear_420(const uint16_t* in, int in_stride, uint16_t* out, int out_stride, int width, int height) {
  out[0] = in[0];
  for (int cx = 0; cx < (width - 1) / 2; cx++) {
    out[2 * cx + 1] = (uint16_t)((3 * in[cx / 2] + 1 * in[cx / 2 + 1] + 2) / 4);
    out[2 * cx + 2] = (uint16_t)((1 * in[cx / 2] + 3 * in[cx / 2 + 1] + 2) / 4);
  }
  if (width % 2 == 0) out[width - 1] = in[width / 2 - 1];
  for (int cy = 0; cy < (height - 1) / 2; cy++) {
    out[(2 * cy + 1) * out_stride] = (uint16_t)((3 * in[cy / 2 * in_stride] + 1 * in[(cy / 2 + 1) * in_stride] + 2) / 4);
    out[(2 * cy + 2) * out_stride] = (uint16_t)((1 * in[cy / 2 * in_stride] + 3 * in[(cy / 2 + 1) * in_stride] + 2) / 4);
  }
  if (height % 2 == 0) out[(height - 1) * out_stride] = in[(height / 2 - 1) * in_stride];
  if (width % 2 == 0)
    for (int cy = 0; cy < (height - 1) / 2; cy++) {
      out[(2 * cy + 1) * out_stride + width - 1] = (uint16_t)((3 * in[cy / 2 * in_stride + width / 2 - 1] + 1 * in[(cy / 2 + 1) * in_stride + width / 2 - 1] + 2) / 4);
      out[(2 * cy + 2) * out_stride + width - 1] = (uint16_t)((1 * in[cy / 2 * in_stride + width / 2 - 1] + 3 * in[(cy / 2 + 1) * in_stride + width / 2 - 1] + 2) / 4);
    }
  if (height % 2 == 0)
    for (int cx = 0; cx < (width - 1) / 2; cx++) {
      out[(height - 1) * out_stride + 2 * cx + 1] = (uint16_t)((3 * in[(height / 2 - 1) * in_stride + cx / 2] + 1 * in[(height / 2 - 1) * in_stride + cx / 2 + 1] + 2) / 4);
      out[(height - 1) * out_stride + 2 * cx + 2] = (uint16_t)((1 * in[(height / 2 - 1) * in_stride + cx / 2] + 3 * in[(height / 2 - 1) * in_stride + cx / 2 + 1] + 2) / 4);
    }
  if (width % 2 == 0 && height % 2 == 0) out[(height - 1) * out_stride + width - 1] = in[(height / 2 - 1) * in_stride + width / 2 - 1];
  for (int y = 1; y < height - 1; y += 2)
    for (int x = 1; x < width - 1; x += 2) {
      const int cx = x / 2, cy = y / 2;
      const int c00 = in[cy * in_stride + cx], c01 = in[cy * in_stride + cx + 1], c10 = in[(cy + 1) * in_stride + cx], c11 = in[(cy + 1) * in_stride + cx + 1];
      out[(y + 0) * out_stride + x + 0] = (uint16_t)((c00 * 3 * 3 + c01 * 1 * 3 + c10 * 3 * 1 + c11 * 1 * 1 + 8) / 16);
      out[(y + 0) * out_stride + x + 1] = (uint16_t)((c00 * 1 * 3 + c01 * 3 * 3 + c10 * 1 * 1 + c11 * 3 * 1 + 8) / 16);
      out[(y + 1) * out_stride + x + 0] = (uint16_t)((c00 * 3 * 1 + c01 * 1 * 1 + c10 * 3 * 3 + c11 * 1 * 3 + 8) / 16);
      out[(y + 1) * out_stride + x + 1] = (uint16_t)((c00 * 1 * 1 + c01 * 3 * 1 + c10 * 1 * 3 + c11 * 3 * 3 + 8) / 16);
    }
}

/* Op_YCbCr422_bilinear_to_YCbCr444 (chroma_sampling.cc:709-933): `in` has ((w+1)/2) x h samples */
void hc_oracle_bilinear_422(const uint16_t* in, int in_stride, uint16_t* out, int out_stride, int width, int height) {
  for (int y = 0; y < height; y++) out[y * out_stride] = in[y * in_stride];
  if (width % 2 == 0)
    for (int y = 0; y < height; y++) out[y * out_stride + width - 1] = in[y * in_stride + width / 2 - 1];
  for (int y = 0; y < height; y++)
    for (int x = 1; x < width - 1; x += 2) {
      const int cx = x / 2;
      const int c0 = in[y * in_stride + cx], c1 = in[y * in_stride + cx + 1];
      out[y * out_stride + x + 0] = (uint16_t)((c0 * 3 + c1 * 1 + 2) / 4);
      out[y * out_stride + x + 1] = (uint16_t)((c0 * 1 + c1 * 3 + 2) / 4);
    }
}

static int hc_oracle_csc_core(const uint16_t* y, const uint16_t* cb, const uint16_t* cr, const uint16_t* a, int y_stride,
                              int c_stride, int a_stride, int width, int height, int chroma_format, int bit_depth, int matrix,
                              int primaries, int full_range, int out_format, uint8_t* out, size_t out_stride, int bilinear_in);

/* upsampling 1 = the options heif-dec -C bilinear sets (bilinear chroma upsampling, only the preferred algorithm): the
 * chain is [plane op] Op_YCbCr42x_bilinear_to_YCbCr444 -> Op_YCbCr_to_RGB<> [plane op] -> interleaver
 * (tests/golden/csc_pipelines_bilinear.json); restated literally: upsample whole planes, then convert as 4:4:4. */
int hc_oracle_csc_opt(const uint16_t* y, const uint16_t* cb, const uint16_t* cr, const uint16_t* a, int y_stride,
                      int c_stride, int a_stride, int width, int height, int chroma_format, int bit_depth, int matrix,
                      int primaries, int full_range, int out_format, int upsampling, uint8_t* out, size_t out_stride) {
  if (!upsampling || (chroma_format != 1 && chroma_format != 2))
    return hc_oracle_csc_core(y, cb, cr, a, y_stride, c_stride, a_stride, width, height, chroma_format, bit_depth, matrix, primaries, full_range,
                              out_format, out, out_stride, 0);
  if (matrix == 0) return -1;
  const int out8 = out_format <= 1, to_alpha = out_format == 1 || out_format == 3 || out_format == 5, in8 = bit_depth == 8;
  const int op = (out8 && !in8) ? 1 : ((!out8 && in8) ? 2 : 0);
  const int pre = (a != NULL && !to_alpha) ? 0 : op;        /* the plane op goes behind the matrix when an alpha plane is dropped */
  const int target = out8 ? 8 : (in8 ? 10 : bit_depth);
  const int cw = (width + 1) / 2, ch = chroma_format == 1 ? (height + 1) / 2 : height;
  uint16_t* tmp = (uint16_t*)malloc(sizeof(uint16_t) * ((size_t)2 * cw * ch + (size_t)2 * width * height));
  if (!tmp) return -2;
  uint16_t *pcb = tmp, *pcr = tmp + (size_t)cw * ch, *ucb = pcr + (size_t)cw * ch, *ucr = ucb + (size_t)width * height;
  for (int yy = 0; yy < ch; yy++)
    for (int x = 0; x < cw; x++) {
      int vb = cb[(size_t)yy * c_stride + x], vr = cr[(size_t)yy * c_stride + x];
      if (pre == 1) { vb = to_sdr(vb, bit_depth); vr = to_sdr(vr, bit_depth); }
      else if (pre == 2) { vb = to_hdr(vb, target); vr = to_hdr(vr, target); }
      pcb[(size_t)yy * cw + x] = (uint16_t)vb;
      pcr[(size_t)yy * cw + x] = (uint16_t)vr;
    }
  if (chroma_format == 1) { hc_oracle_bilinear_420(pcb, cw, ucb, width, width, height); hc_oracle_bilinear_420(pcr, cw, ucr, width, width, height); }
  else { hc_oracle_bilinear_422(pcb, cw, ucb, width, width, height); hc_oracle_bilinear_422(pcr, cw, ucr, width, width, height); }
  /* bilinear_in: 1 = the chroma planes handed over already went through `pre` (luma and alpha have not), 2 = no plane op in front */
  const int rc = hc_oracle_csc_core(y, ucb, ucr, a, y_stride, width, a_stride, width, height, 3, bit_depth, matrix, primaries, full_range, out_format, out,
                                    out_stride, pre ? 1 : 2);
  free(tmp);
  return rc;
}

int hc_oracle_csc(const uint16_t* y, const uint16_t* cb, const uint16_t* cr, const uint16_t* a, int y_stride,
                  int c_stride, int a_stride, int width, int height, int chroma_format, int bit_depth, int matrix,
                  int primaries, int full_range, int out_format, uint8_t* out, size_t out_stride) {
  return hc_oracle_csc_core(y, cb, cr, a, y_stride, c_stride, a_stride, width, height, chroma_format, bit_depth, matrix, primaries, full_range, out_format,
                            out, out_stride, 0);
}

/* out_format: 0 RGB, 1 RGBA, 2 RRGGBB_BE, 3 RRGGBBAA_BE, 4 RRGGBB_LE, 5 RRGGBBAA_LE.
 * Planes are uint16 arrays (any bit depth), strides in samples. `a` may be NULL.
 * Returns 0, or -1 for combinations the reference cannot convert.
 *
 * Which ops run, for the default decoding options, was read off the unmodified reference with
 * tools/csc_pipeline_probe.cc (ColorConversionPipeline::construct_pipeline + debug_dump_pipeline; table in DESIGN.md):
 *   target interleaved RGB / RGBA (8 bit, colorconversion.cc:571-587):
 *     4:2:0 full range (matrix not 0 / 8):  [Op_to_sdr_planes on Y Cb Cr A]  Op_YCbCr420_to_RGB24 / _RGB32     (integer)
 *     monochrome:                           [Op_to_sdr_planes]               Op_mono_to_RGB24_32               (copy)
 *     everything else:      Op_YCbCr_to_RGB<> at the input depth (fp32)  [Op_to_sdr_planes on R G B A]  Op_RGB_to_RGB24_32
 *   target RRGGBB(AA) (input depth, or 10 bit for 8-bit input):
 *     4:2:0 or monochrome (Op_mono_to_YCbCr420: Cb = Cr = 128 << (bpp - 8)), matrix not 0 / 8, and the output has alpha
 *     only if the input has:                [Op_to_hdr_planes on Y Cb Cr A]  Op_YCbCr420_to_RRGGBBaa           (fp32)
 *     everything else:      Op_YCbCr_to_RGB<> at the input depth  [Op_to_hdr_planes on R G B A]  Op_RGB_HDR_to_RRGGBBaa_BE
 *                           [Op_RRGGBBaa_swap_endianness]; a missing alpha plane is filled with the maximum of the final depth */
static int hc_oracle_csc_core(const uint16_t* y, const uint16_t* cb, const uint16_t* cr, const uint16_t* a, int y_stride,
                              int c_stride, int a_stride, int width, int height, int chroma_format, int bit_depth, int matrix,
                              int primaries, int full_range, int out_format, uint8_t* out, size_t out_stride, int bilinear_in) {
  /* matrix 2 (unspecified) reaches the ops unchanged: Kr = Kb = 0 -> the literal BT.601 defaults
   * (nclx.cc:140-149,159-169), NOT the values computed from Kr/Kb of matrix 6 */
  if (matrix == 11 || matrix == 14) return -1;
  /* Op_mono_to_YCbCr420 hands on a fresh colour state (monochrome.cc:36-45: nothing copies the nclx), so whatever follows
   * it converts with the defaults of color_profile_nclx (nclx.h:165-168): full range, matrix unspecified */
  const int image_matrix = matrix, image_full = full_range;
  if (chroma_format == 0 && out_format > 1) { matrix = 2; full_range = 1; }
  const int to_alpha = out_format == 1 || out_format == 3 || out_format == 5;
  const int out8 = out_format <= 1;
  const int has_alpha = a != NULL;
  const int in8 = bit_depth == 8;
  const int special = matrix == 0 || matrix == 8;
  const int cls420 = chroma_format == 0 || chroma_format == 1;       /* monochrome goes through Op_mono_to_YCbCr420 */
  coeffs_t k = get_coeffs(matrix, primaries);
  const int shiftH = (chroma_format == 1 || chroma_format == 2) ? 1 : 0;
  const int shiftV = chroma_format == 1 ? 1 : 0;

  int pre = 0, post = 0;     /* 1: to_sdr, 2: to_hdr; pre on Y Cb Cr A, post on R G B A */
  int op;                    /* 0 integer 4:2:0, 1 fp32 general, 2 monochrome copy */
  const int target = out8 ? 8 : (in8 ? 10 : bit_depth);
  if (out8) {
    if (chroma_format == 0) { op = 2; pre = in8 ? 0 : 1; }
    else if (chroma_format == 1 && full_range && !special) { op = 0; pre = in8 ? 0 : 1; }
    else { op = 1; post = in8 ? 0 : 1; }
  } else {
    op = 1;
    if (cls420 && !special && (!to_alpha || has_alpha)) pre = in8 ? 2 : 0;
    else if (in8) {
      /* equal-cost alternatives "matrix at 8 bit, then Op_to_hdr_planes" / "Op_to_hdr_planes, then matrix at 10 bit": the
       * search's expansion order decides; read off the exhaustive table tests/golden/csc_pipelines.json */
      const int hdr_first = (has_alpha && !to_alpha && (chroma_format == 3 || image_matrix == 0)) ||
                            (chroma_format == 0 && !has_alpha && to_alpha && image_matrix == 0 && image_full);
      if (hdr_first) pre = 2; else post = 2;
    }
  }
  if (bilinear_in) {      /* behind the bilinear upsampling: general matrix op; plane op in front (1) or behind / absent (2) */
    const int opd = (out8 && !in8) ? 1 : ((!out8 && in8) ? 2 : 0);
    op = 1;
    pre = bilinear_in == 1 ? opd : 0;
    post = bilinear_in == 1 ? 0 : opd;
  }
  const int work = pre == 1 ? 8 : (pre == 2 ? target : bit_depth);   /* depth the conversion runs at */
  const int maxv = (1 << work) - 1;
  const int half = 1 << (work - 1);
  /* An op reads the nclx of the image it is handed (yuv2rgb.cc:121-128,598-603). The FIRST op of a chain gets the decoded
   * image with its own nclx — matrix 2 (unspecified) then means the literal BT.601 defaults (nclx.cc:140-149); every later
   * op gets an image stamped with the pipeline's colour state (colorconversion.cc:454-455), in which unspecified values
   * were replaced by matrix 6 / primaries 1 (colorconversion.cc:528, nclx.cc:346-359) — coefficients computed from Kr / Kb,
   * which differ from the literals in the last ulp. The matrix op is not first behind Op_drop_alpha_plane or a plane op. */
  if (chroma_format != 0 || out8) {
    /* Op_RGB_to_RGB24_32 ignores an alpha plane it does not need: no Op_drop_alpha_plane in front of the general 8-bit path */
    const int drops_alpha = has_alpha && !to_alpha && !(out8 && op == 1);
    const int matrix_first = !drops_alpha && pre == 0 && !bilinear_in;
    if (!matrix_first) {
      const coeffs_t k2 = get_coeffs(matrix == 2 ? 6 : matrix, primaries == 2 ? 1 : primaries);
      k = k2;
    }
  }
  const int r_cr = (int)lround(256 * k.r_cr), g_cr = (int)lround(256 * k.g_cr);
  const int g_cb = (int)lround(256 * k.g_cb), b_cb = (int)lround(256 * k.b_cb);
  const float lro = (float)(16 << (work - 8));
#define PRE(v) (pre == 1 ? to_sdr((v), bit_depth) : (pre == 2 ? to_hdr((v), target) : (v)))
#define POST(v) (post == 1 ? to_sdr((v), work) : (post == 2 ? to_hdr((v), target) : (v)))

  for (int yy = 0; yy < height; yy++)
    for (int x = 0; x < width; x++) {
      const int yv = PRE(y[(size_t)yy * y_stride + x]);
      int cbv, crv;
      if (chroma_format) {
        cbv = cb[(size_t)(yy >> shiftV) * c_stride + (x >> shiftH)];
        crv = cr[(size_t)(yy >> shiftV) * c_stride + (x >> shiftH)];
        if (bilinear_in != 1) { cbv = PRE(cbv); crv = PRE(crv); }
      } else {
        cbv = crv = PRE(128 << (bit_depth - 8));      /* monochrome.cc:99-100,128: the planes Op_mono_to_YCbCr420 adds */
      }
      int R, G, B;
      if (op == 2) {
        R = G = B = yv;
      } else if (op == 0) { /* yuv2rgb.cc:349-361 */
        const int cbi = cbv - 128, cri = crv - 128;
        R = clip_int_u8(yv + ((r_cr * cri + 128) >> 8));
        G = clip_int_u8(yv + ((g_cb * cbi + g_cr * cri + 128) >> 8));
        B = clip_int_u8(yv + ((b_cb * cbi + 128) >> 8));
      } else if (matrix == 0) { /* yuv2rgb.cc:197-211 */
        if (full_range) { R = crv; G = yv; B = cbv; }
        else {
          R = clip_f_u16((crv - lro) * 1.1429f, maxv);
          G = clip_f_u16((yv - lro) * 1.1689f, maxv);
          B = clip_f_u16((cbv - lro) * 1.1429f, maxv);
        }
      } else if (matrix == 8) { /* yuv2rgb.cc:212-226 */
        const int c1 = cbv - half, c2 = crv - half;
        R = clip_int_u8(yv - c1 + c2);
        G = clip_int_u8(yv + c1);
        B = clip_int_u8(yv - c1 - c2);
      } else { /* yuv2rgb.cc:227-244 */
        float fy = (float)yv, fcb = (float)(cbv - half), fcr = (float)(crv - half);
        if (!full_range) {
          fy = (fy - lro) * 1.1689f;
          fcb = fcb * 1.1429f;
          fcr = fcr * 1.1429f;
        }
        R = clip_f_u16(fy + k.r_cr * fcr, maxv);
        G = clip_f_u16(fy + k.g_cb * fcb + k.g_cr * fcr, maxv);
        B = clip_f_u16(fy + k.b_cb * fcb, maxv);
      }
      R = POST(R); G = POST(G); B = POST(B);
      /* alpha rides through the same plane ops; a missing plane is filled at the final depth (rgb2rgb.cc:251,264; 0xFF in
       * the 8-bit interleavers) */
      int A;
      if (has_alpha) { A = PRE(a[(size_t)yy * a_stride + x]); A = POST(A); }
      else A = (1 << target) - 1;
      uint8_t* o = out + (size_t)yy * out_stride;
      if (out_format == 0) {
        o[3 * x + 0] = (uint8_t)R; o[3 * x + 1] = (uint8_t)G; o[3 * x + 2] = (uint8_t)B;
      } else if (out_format == 1) {
        o[4 * x + 0] = (uint8_t)R; o[4 * x + 1] = (uint8_t)G; o[4 * x + 2] = (uint8_t)B; o[4 * x + 3] = (uint8_t)A;
      } else {
        const int le = out_format >= 4, ps = to_alpha ? 8 : 6;
        const int v[4] = {R, G, B, A};
        for (int c = 0; c < (to_alpha ? 4 : 3); c++) {
          o[ps * x + 2 * c + le] = (uint8_t)(v[c] >> 8);
          o[ps * x + 2 * c + 1 - le] = (uint8_t)(v[c] & 0xff);
        }
      }
    }
#undef PRE
#undef POST
  return 0;
}
