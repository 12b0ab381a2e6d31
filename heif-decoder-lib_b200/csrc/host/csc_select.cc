// csc_select.cc — which colour conversion the reference would run, and with which coefficients.
//
// Mirrors, for the default heif_decoding_options, the outcome of the reference's Dijkstra search
// over its ColorConversionOperation pool (libheif/color-conversion/colorconversion.cc:266-420;
// resolved table in SURVEY.md §3.5) and the coefficient derivation of libheif/nclx.cc:82-171.
// The float expressions are written in the same order as the reference's so that fp32 rounding is
// identical; this file is compiled with -ffp-contract=off.
#include "../capi/capi_internal.h"
#include <cmath>

namespace {

struct KrKb { float Kr = 0.f, Kb = 0.f; };

// nclx.cc:46-75 get_colour_primaries: green, blue, red, white chromaticities (zeros when the index is not tabulated)
struct Prim { int idx; float gx, gy, bx, by, rx, ry, wx, wy; };
const Prim kPrimaries[] = {
    {1, 0.300f, 0.600f, 0.150f, 0.060f, 0.640f, 0.330f, 0.3127f, 0.3290f}, {4, 0.21f, 0.71f, 0.14f, 0.08f, 0.67f, 0.33f, 0.310f, 0.316f},
    {5, 0.29f, 0.60f, 0.15f, 0.06f, 0.64f, 0.33f, 0.3127f, 0.3290f},       {6, 0.310f, 0.595f, 0.155f, 0.070f, 0.630f, 0.340f, 0.3127f, 0.3290f},
    {7, 0.310f, 0.595f, 0.155f, 0.070f, 0.630f, 0.340f, 0.3127f, 0.3290f}, {8, 0.243f, 0.692f, 0.145f, 0.049f, 0.681f, 0.319f, 0.310f, 0.316f},
    {9, 0.170f, 0.797f, 0.131f, 0.046f, 0.708f, 0.292f, 0.3127f, 0.3290f}, {10, 0.0f, 1.0f, 0.0f, 0.0f, 1.0f, 0.0f, 0.333333f, 0.33333f},
    {11, 0.265f, 0.690f, 0.150f, 0.060f, 0.680f, 0.320f, 0.314f, 0.351f},  {12, 0.265f, 0.690f, 0.150f, 0.060f, 0.680f, 0.320f, 0.3127f, 0.3290f},
    {22, 0.295f, 0.605f, 0.155f, 0.077f, 0.630f, 0.340f, 0.3127f, 0.3290f}};

// nclx.cc:82-138 get_Kr_Kb
KrKb kr_kb(int matrix, int primaries) {
  KrKb r;
  if (matrix == 12 || matrix == 13) {
    Prim p{0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (const Prim& q : kPrimaries)
      if (q.idx == primaries) p = q;
    const float zr = 1 - (p.rx + p.ry), zg = 1 - (p.gx + p.gy), zb = 1 - (p.bx + p.by), zw = 1 - (p.wx + p.wy);
    const float denom = p.wy * (p.rx * (p.gy * zb - p.by * zg) + p.gx * (p.by * zr - p.ry * zb) + p.bx * (p.ry * zg - p.gy * zr));
    if (denom == 0.0f) return r;
    r.Kr = (p.ry * (p.wx * (p.gy * zb - p.by * zg) + p.wy * (p.bx * zg - p.gx * zb) + zw * (p.gx * p.by - p.bx * p.gy))) / denom;
    r.Kb = (p.by * (p.wx * (p.ry * zg - p.gy * zr) + p.wy * (p.gx * zr - p.rx * zg) + zw * (p.rx * p.gy - p.gx * p.ry))) / denom;
    return r;
  }
  switch (matrix) {
    case 1: r.Kr = 0.2126f; r.Kb = 0.0722f; break;
    case 4: r.Kr = 0.30f; r.Kb = 0.11f; break;
    case 5:
    case 6: r.Kr = 0.299f; r.Kb = 0.114f; break;
    case 7: r.Kr = 0.212f; r.Kb = 0.087f; break;
    case 9:
    case 10: r.Kr = 0.2627f; r.Kb = 0.0593f; break;
    default: break;
  }
  return r;
}

}  // namespace

extern "C" int hc_csc_select(int matrix, int primaries, int full_range, int chroma_format, int bit_depth,
                             int has_alpha, int out_format, hc_csc_params* out) {
  return hc_csc_select_opt(matrix, primaries, full_range, chroma_format, bit_depth, has_alpha, out_format, HC_UPSAMPLE_NEAREST, out);
}

extern "C" int hc_csc_select_opt(int matrix, int primaries, int full_range, int chroma_format, int bit_depth,
                                 int has_alpha, int out_format, int upsampling, hc_csc_params* out) {
  if (!out || (upsampling != HC_UPSAMPLE_NEAREST && upsampling != HC_UPSAMPLE_BILINEAR) || out_format < HC_OUT_RGB || out_format > HC_OUT_YCBCR || bit_depth < 8 || bit_depth > 16 || chroma_format < 0 ||
      chroma_format > 3) {
    hc::set_last_error("hc_csc_select: bad argument");
    return HC_ERR_ARGUMENT;
  }
  if (out_format == HC_OUT_YCBCR) {
    // the planes as decoded (heif_colorspace_undefined / heif_chroma_undefined): no op at all, so any matrix goes
    hc_csc_params p{};
    p.mode = HC_CSC_FLOAT;
    p.out_format = HC_OUT_YCBCR;
    p.full_range = full_range ? 1 : 0;
    p.bit_depth = p.in_depth = p.out_depth = bit_depth;
    p.pre_op = p.post_op = HC_DEPTH_NONE;
    p.upsampling = HC_UPSAMPLE_NEAREST;
    p.coeff_matrix = matrix;
    *out = p;
    return HC_OK;
  }
  // matrix 2 (unspecified) reaches the conversion ops unchanged: Kr = Kb = 0 selects the literal
  // BT.601 defaults (nclx.cc:140-149,159-169), which differ in the last ulp from the values
  // computed for matrix 6.
  if (matrix == 11 || matrix == 14) {
    hc::set_last_error("matrix_coefficients 11/14 are not convertible (the reference rejects them too)");
    return HC_ERR_UNSUPPORTED;
  }
  // Monochrome images reach the RRGGBB(AA) targets through Op_mono_to_YCbCr420, whose output state is a fresh ColorState
  // (monochrome.cc:36-45): the ops behind it see the defaults of color_profile_nclx (nclx.h:165-168) — full range, matrix
  // unspecified — whatever the image's own nclx says.
  const int image_matrix = matrix, image_full = full_range;
  if (chroma_format == 0 && out_format != HC_OUT_RGB && out_format != HC_OUT_RGBA) { matrix = 2; full_range = 1; }
  hc_csc_params p;
  p.out_format = out_format;
  p.full_range = full_range ? 1 : 0;
  p.in_depth = bit_depth;
  p.upsampling = HC_UPSAMPLE_NEAREST;
  p.premultiply = 0;
  const bool bilinear = upsampling == HC_UPSAMPLE_BILINEAR && (chroma_format == 1 || chroma_format == 2);
  if (upsampling == HC_UPSAMPLE_BILINEAR && chroma_format == 0 && out_format != HC_OUT_RGB && out_format != HC_OUT_RGBA) {
    hc::set_last_error("monochrome images to RRGGBB(AA) with the bilinear-only option are not supported");
    return HC_ERR_UNSUPPORTED;
  }
  if (bilinear && matrix == 0) {
    hc::set_last_error("bilinear chroma upsampling of GBR-coded (matrix_coefficients 0) subsampled images: the reference finds no pipeline either");
    return HC_ERR_UNSUPPORTED;
  }

  // ---- which ops the reference's pipeline search ends up with (colorconversion.cc:266-420, default options), read off
  // the unmodified reference with tools/csc_pipeline_probe.cc for every input class x output format (table: DESIGN.md) ----
  const bool in8 = bit_depth == 8;
  const bool out8 = out_format == HC_OUT_RGB || out_format == HC_OUT_RGBA;
  const bool out_alpha = out_format == HC_OUT_RGBA || out_format == HC_OUT_RRGGBBAA_BE || out_format == HC_OUT_RRGGBBAA_LE;
  const bool special = matrix == 0 || matrix == 8;            // excluded from the 4:2:0 ops (yuv2rgb.cc:283,520)
  const int general = matrix == 0 ? HC_CSC_GBR : (matrix == 8 ? HC_CSC_YCGCO : HC_CSC_FLOAT);   // Op_YCbCr_to_RGB<>
  p.out_depth = out8 ? 8 : (in8 ? 10 : bit_depth);            // colorconversion.cc:571-587
  p.pre_op = p.post_op = HC_DEPTH_NONE;
  if (bilinear) {
    // only_use_preferred_chroma_algorithm rules the nearest-neighbour 4:2:0 ops out (yuv2rgb.cc:272-279,504-511): the chain
    // is always Op_YCbCr42x_bilinear_to_YCbCr444 -> Op_YCbCr_to_RGB<> -> interleaver, with the depth-changing plane op in
    // front of the upsampling — or behind the matrix when an alpha plane is dropped on the way
    // (tests/golden/csc_pipelines_bilinear.json, 2304 cases)
    p.mode = general;
    p.upsampling = HC_UPSAMPLE_BILINEAR;
    const int op = (out8 && !in8) ? HC_DEPTH_TO_SDR : ((!out8 && in8) ? HC_DEPTH_TO_HDR : HC_DEPTH_NONE);
    if (has_alpha && !out_alpha) p.post_op = op;
    else p.pre_op = op;
  } else if (out8) {
    if (chroma_format == 0) {                                 // [Op_to_sdr_planes] Op_mono_to_RGB24_32
      p.mode = HC_CSC_MONO;
      p.pre_op = in8 ? HC_DEPTH_NONE : HC_DEPTH_TO_SDR;
    } else if (chroma_format == 1 && full_range && !special) {   // [Op_to_sdr_planes] Op_YCbCr420_to_RGB24 / _RGB32
      p.mode = HC_CSC_INT420;
      p.pre_op = in8 ? HC_DEPTH_NONE : HC_DEPTH_TO_SDR;
    } else {                                                  // Op_YCbCr_to_RGB<> [Op_to_sdr_planes] Op_RGB_to_RGB24_32
      p.mode = general;
      p.post_op = in8 ? HC_DEPTH_NONE : HC_DEPTH_TO_SDR;
    }
  } else {
    p.mode = general;
    // Op_YCbCr420_to_RRGGBBaa (after Op_mono_to_YCbCr420 for monochrome input) keeps the input's alpha state, so it is
    // only on the cheapest path when no alpha plane has to be invented
    if ((chroma_format == 0 || chroma_format == 1) && !special && (!out_alpha || has_alpha)) p.pre_op = in8 ? HC_DEPTH_TO_HDR : HC_DEPTH_NONE;
    else if (in8) {
      // Op_YCbCr_to_RGB<uint8_t> [Op_to_hdr_planes] Op_RGB_HDR_to_RRGGBBaa_BE [swap] — or, at equal cost, Op_to_hdr_planes
      // first and Op_YCbCr_to_RGB<uint16_t> at 10 bit. Which one the search returns is decided by the order in which it
      // expands equal-cost states; the exhaustive table (tests/golden/csc_pipelines.json, 2304 cases) shows the plane op in
      // front exactly when an alpha plane is dropped first and the image is 4:4:4 or GBR, and for one monochrome corner.
      const bool hdr_first = (has_alpha && !out_alpha && (chroma_format == 3 || image_matrix == 0)) ||
                             (chroma_format == 0 && !has_alpha && out_alpha && image_matrix == 0 && image_full);
      if (hdr_first) p.pre_op = HC_DEPTH_TO_HDR;
      else p.post_op = HC_DEPTH_TO_HDR;
    }
  }
  p.bit_depth = p.pre_op == HC_DEPTH_TO_SDR ? 8 : (p.pre_op == HC_DEPTH_TO_HDR ? p.out_depth : bit_depth);

  // An op reads the nclx of the image it is handed (yuv2rgb.cc:121-128,598-603). The FIRST op of a chain gets the decoded
  // image with its own nclx: matrix 2 (unspecified) reaches it unchanged and Kr = Kb = 0 selects the literal BT.601 defaults
  // (nclx.cc:140-149,159-169). Every later op gets an image stamped with the pipeline's colour state
  // (colorconversion.cc:454-455), in which unspecified values were replaced by matrix 6 / primaries 1
  // (colorconversion.cc:528, nclx.cc:346-359): coefficients computed from Kr / Kb, different from the literals in the last
  // ulp. The matrix op is not the first one behind Op_drop_alpha_plane or a plane op. (Monochrome input of the RRGGBB
  // targets keeps the fresh state of Op_mono_to_YCbCr420, see above.)
  // Op_drop_alpha_plane only appears in front of the ops that keep the input's alpha state (the 4:2:0 ops and
  // Op_RGB_HDR_to_RRGGBBaa_BE's feeders); Op_RGB_to_RGB24_32 simply ignores an alpha plane it does not need.
  const bool fresh_state = chroma_format == 0 && !out8;
  const bool drops_alpha = has_alpha && !out_alpha && !(out8 && p.mode != HC_CSC_INT420);
  const bool matrix_first = !drops_alpha && p.pre_op == HC_DEPTH_NONE && !bilinear;
  if (!fresh_state && !matrix_first) {
    if (matrix == 2) matrix = 6;
    if (primaries == 2) primaries = 1;
  }
  p.coeff_matrix = matrix;
  // nclx.cc:151-171 get_YCbCr_to_RGB_coefficients (defaults :140-149 when Kr = Kb = 0)
  const KrKb k = kr_kb(matrix, primaries);
  if (k.Kb != 0 || k.Kr != 0) {
    p.r_cr = 2 * (-k.Kr + 1);
    p.g_cb = 2 * k.Kb * (-k.Kb + 1) / (k.Kb + k.Kr - 1);
    p.g_cr = 2 * k.Kr * (-k.Kr + 1) / (k.Kb + k.Kr - 1);
    p.b_cb = 2 * (-k.Kb + 1);
  } else {
    p.r_cr = 1.402f;
    p.g_cb = -0.344136f;
    p.g_cr = -0.714136f;
    p.b_cb = 1.772f;
  }
  // yuv2rgb.cc:331-334
  p.r_cr_i = (int)std::lround(256 * p.r_cr);
  p.g_cr_i = (int)std::lround(256 * p.g_cr);
  p.g_cb_i = (int)std::lround(256 * p.g_cb);
  p.b_cb_i = (int)std::lround(256 * p.b_cb);
  *out = p;
  return HC_OK;
}
