// k5_csc.cu — K5: libheif's YCbCr -> interleaved RGB colour-conversion chain fused into one
// output-writing kernel (chroma upsampling, matrix, range expansion, interleave, endianness,
// alpha merge).
//
// Replaces, depending on hc_csc_params::mode (selection mirrors ColorConversionPipeline::
// construct_pipeline, colorconversion.cc:266-420, for the default decoding options):
//   HC_CSC_INT420 : Op_YCbCr420_to_RGB24 / Op_YCbCr420_to_RGB32            yuv2rgb.cc:260-495
//   HC_CSC_FLOAT  : Op_YCbCr_to_RGB<uint8_t|uint16_t> (+ Op_RGB_to_RGB24_32, Op_RGB_HDR_to_RRGGBBaa_BE,
//                   Op_RRGGBBaa_swap_endianness) and Op_YCbCr420_to_RRGGBBaa  yuv2rgb.cc:28-254,498-643,
//                   rgb2rgb.cc:28-272,613-729 — each of which is a separate full-image pass with
//                   its own allocation in the reference
//   HC_CSC_GBR / HC_CSC_YCGCO : the matrix_coefficients 0 / 8 branches        yuv2rgb.cc:197-226
//   HC_CSC_MONO   : Op_mono_to_RGB24_32 (monochrome.cc:150-260); monochrome input of the other modes gets the constant
//                   chroma planes of Op_mono_to_YCbCr420 (monochrome.cc:53-140)
//   pre_op / post_op : Op_to_sdr_planes / Op_to_hdr_planes (hdr_sdr.cc:24-236) before or after the matrix, wherever the
//                   reference's pipeline search puts them — 10/12-bit images to RGB(A) 8, 8-bit images to RRGGBB(AA)
// Float arithmetic uses explicit round-to-nearest mul/add (no FMA contraction) and the
// reference's (long)(x + 0.5f) rounding (common_utils.h:64-70) so results are bit-exact.
//
// Mapping: one thread converts 8 horizontally adjacent pixels (8/16-byte plane loads) and writes them
// with 64-bit / 128-bit stores; a warp writes 768 (RGB) .. 2048 (RRGGBBAA) contiguous bytes. Pure streaming:
// algorithmic bytes = s*c (+s alpha) read + bytes-per-pixel written.
// Scaled output (heif_image_scale_image after the conversion, HeifPixelImage::scale_nearest_neighbor pixelimage.cc:1156-1253):
// every output pixel of the conversion depends on its own source pixel only, so converting just the sampled source pixels
// gives the same bytes as converting at full size and scaling the result. The thread mapping and the stores stay as above;
// the loads become per-pixel gathers (gather_px8).
#include <algorithm>
#include "launch.h"

namespace hc {

HC_D int clip_f(float fx, int maxi) {
  const long long x = (long long)__fadd_rn(fx, 0.5f);
  return x < 0 ? 0 : (x > maxi ? maxi : (int)x);
}

// MODE is a compile-time constant at every call site (the per-pixel loop is instantiated once per conversion mode)
template <typename Pixel, int MODE>
__device__ __forceinline__ void convert_px(const CscArgs& a, int yv, int cbv, int crv, int& r, int& g, int& b) {
  const hc_csc_params& p = a.p;
  const int bpp = p.bit_depth;
  const int maxv = (1 << bpp) - 1, half = 1 << (bpp - 1);
  if (MODE == HC_CSC_INT420) {
    const int cb = cbv - 128, cr = crv - 128;
    r = clip3i(0, 255, yv + ((p.r_cr_i * cr + 128) >> 8));
    g = clip3i(0, 255, yv + ((p.g_cb_i * cb + p.g_cr_i * cr + 128) >> 8));
    b = clip3i(0, 255, yv + ((p.b_cb_i * cb + 128) >> 8));
  } else if (MODE == HC_CSC_FLOAT) {
    float fy = (float)yv, cb = (float)(cbv - half), cr = (float)(crv - half);
    if (!p.full_range) {
      fy = __fmul_rn(__fsub_rn(fy, (float)(16 << (bpp - 8))), 1.1689f);
      cb = __fmul_rn(cb, 1.1429f);
      cr = __fmul_rn(cr, 1.1429f);
    }
    r = clip_f(__fadd_rn(fy, __fmul_rn(p.r_cr, cr)), maxv);
    g = clip_f(__fadd_rn(__fadd_rn(fy, __fmul_rn(p.g_cb, cb)), __fmul_rn(p.g_cr, cr)), maxv);
    b = clip_f(__fadd_rn(fy, __fmul_rn(p.b_cb, cb)), maxv);
  } else if (MODE == HC_CSC_GBR) {
    if (p.full_range) { r = crv; g = yv; b = cbv; }
    else {
      const float off = (float)(16 << (bpp - 8));
      r = clip_f(__fmul_rn(__fsub_rn((float)crv, off), 1.1429f), maxv);
      g = clip_f(__fmul_rn(__fsub_rn((float)yv, off), 1.1689f), maxv);
      b = clip_f(__fmul_rn(__fsub_rn((float)cbv, off), 1.1429f), maxv);
    }
  } else {  // HC_CSC_YCGCO (clip_int_u8 in the reference regardless of depth, yuv2rgb.cc:218-226)
    const int cb = cbv - half, cr = crv - half;
    r = clip3i(0, 255, yv - cb + cr);
    g = clip3i(0, 255, yv + cb);
    b = clip3i(0, 255, yv - cb - cr);
  }
}

template <typename Pixel>
HC_D void load_px8(const Pixel* p, int n, int v[8]);
template <>
HC_D void load_px8<uint8_t>(const uint8_t* p, int n, int v[8]) {
  if (n == 8 && (reinterpret_cast<uintptr_t>(p) & 7) == 0) {
    const uint2 w = *reinterpret_cast<const uint2*>(p);
#pragma unroll
    for (int k = 0; k < 4; k++) { v[k] = (w.x >> (8 * k)) & 0xff; v[4 + k] = (w.y >> (8 * k)) & 0xff; }
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = k < n ? (int)p[k] : 0;
  }
}
template <>
HC_D void load_px8<uint16_t>(const uint16_t* p, int n, int v[8]) {
  if (n == 8 && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    const uint4 w = *reinterpret_cast<const uint4*>(p);
    v[0] = w.x & 0xffff; v[1] = w.x >> 16; v[2] = w.y & 0xffff; v[3] = w.y >> 16;
    v[4] = w.z & 0xffff; v[5] = w.z >> 16; v[6] = w.w & 0xffff; v[7] = w.w >> 16;
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = k < n ? (int)p[k] : 0;
  }
}

template <typename Pixel>
HC_D void load_px4(const Pixel* p, int n, int fill, int v[8]) {
  constexpr int PS = (int)sizeof(Pixel);
  if (n == 4 && (reinterpret_cast<uintptr_t>(p) & (4 * PS - 1)) == 0) {
    if (PS == 1) {
      const uint32_t w = *reinterpret_cast<const uint32_t*>(p);
#pragma unroll
      for (int k = 0; k < 4; k++) v[k] = (w >> (8 * k)) & 0xff;
    } else {
      const uint2 w = *reinterpret_cast<const uint2*>(p);
      v[0] = w.x & 0xffff; v[1] = w.x >> 16; v[2] = w.y & 0xffff; v[3] = w.y >> 16;
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; k++) v[k] = k < n ? (int)p[k] : fill;
  }
}

// One thread converts 8 horizontally adjacent pixels: 8/16-byte plane loads, 8/16-byte interleaved stores
// (24 .. 64 bytes per thread, contiguous across the warp). Output rows are padded to a multiple of 8 pixels.
// Op_to_sdr_planes / Op_to_hdr_planes (hdr_sdr.cc:54-97,140-236) on one sample: `from` is the sample's depth for TO_SDR,
// `to` the target depth for TO_HDR (the input is 8 bit there)
HC_D int depth_op(int op, int v, int from, int to) {
  return op == HC_DEPTH_TO_SDR ? v >> (from - 8) : (op == HC_DEPTH_TO_HDR ? ((v << (to - 8)) | (v >> (16 - to))) : v);
}

// Op_YCbCr420_bilinear_to_YCbCr444 / Op_YCbCr422_bilinear_to_YCbCr444 (chroma_sampling.cc:441-705, :709-933) for ONE output
// sample (x, y) of one chroma plane: 3/4 - 1/4 weights between the surrounding chroma samples, chroma sited in the middle
// of its 2x2 (2x1) luma samples. The image border follows the reference statement by statement, including its
// `in[cx / 2]` indexing of the first / last row and column of 4:2:0 pictures (it halves the chroma index once more there).
// `pre` / `ind` / `outd`: the plane op in front of the upsampling is applied to every chroma sample that is read.
template <typename Pixel>
__device__ __forceinline__ int bilinear_chroma(const Pixel* P, int stride, int w, int h, int x, int y, bool v420, int pre, int ind, int outd) {
  auto S = [&](int cx, int cy) -> int { return depth_op(pre, (int)P[(size_t)cy * stride + cx], ind, outd); };
  const bool right = x == w - 1 && !(w & 1);
  if (!v420) {   // 4:2:2: horizontal only
    if (x == 0) return S(0, y);
    if (right) return S(w / 2 - 1, y);
    const int bx = (x & 1) ? x : x - 1, cx = bx >> 1;
    const int a0 = S(cx, y), a1 = S(cx + 1, y);
    return x == bx ? (a0 * 3 + a1 + 2) / 4 : (a0 + a1 * 3 + 2) / 4;
  }
  const bool bottom = y == h - 1 && !(h & 1);
  if (y == 0 || bottom) {
    const int cy = y == 0 ? 0 : h / 2 - 1;
    if (x == 0) return S(0, cy);
    if (right) return S(w / 2 - 1, cy);
    const int q = (((x & 1) ? x - 1 : x - 2) >> 1) / 2;     // "cx / 2" of the reference's border loops
    const int a0 = S(q, cy), a1 = S(q + 1, cy);
    return (x & 1) ? (3 * a0 + a1 + 2) / 4 : (a0 + 3 * a1 + 2) / 4;
  }
  if (x == 0 || right) {
    const int cx = x == 0 ? 0 : w / 2 - 1;
    const int q = (((y & 1) ? y - 1 : y - 2) >> 1) / 2;     // "cy / 2"
    const int a0 = S(cx, q), a1 = S(cx, q + 1);
    return (y & 1) ? (3 * a0 + a1 + 2) / 4 : (a0 + 3 * a1 + 2) / 4;
  }
  const int bx = (x & 1) ? x : x - 1, by = (y & 1) ? y : y - 1, cx = bx >> 1, cy = by >> 1;
  const int c00 = S(cx, cy), c01 = S(cx + 1, cy), c10 = S(cx, cy + 1), c11 = S(cx + 1, cy + 1);
  const int wx0 = x == bx ? 3 : 1, wx1 = 4 - wx0, wy0 = y == by ? 3 : 1, wy1 = 4 - wy0;
  return (c00 * wx0 * wy0 + c01 * wx1 * wy0 + c10 * wx0 * wy1 + c11 * wx1 * wy1 + 8) / 16;
}

// Gather form of the loads (CscArgs::gather): the 8 output pixels of a thread are converted from source pixels
// (ix, iy) = (x * src_w / width, y * src_h / height), 64-bit products. Y and A at (ix, iy), nearest chroma at
// (ix >> shiftH, iy >> shiftV), bilinear chroma evaluated at (ix, iy) of the source image. Padding lanes repeat the last pixel.
template <typename Pixel>
__device__ __noinline__ void gather_px8(const CscArgs& a, int y, int x0, bool bilinear, int shiftH, int shiftV, int half_in, int Y[8],
                                        int Cb[8], int Cr[8], int A[8]) {
  const int iy = (int)((long long)y * a.src_h / a.height);
  const Pixel* yr = reinterpret_cast<const Pixel*>(a.y) + (size_t)iy * a.y_stride;
  const Pixel* ar = a.a ? reinterpret_cast<const Pixel*>(a.a) + (size_t)iy * a.a_stride : nullptr;
  const size_t crow = (size_t)(iy >> shiftV) * a.c_stride;
  const int pre = a.p.pre_op, ind = a.p.in_depth, outd = a.p.out_depth;
#pragma unroll 1
  for (int k = 0; k < 8; k++) {
    const int ix = (int)((long long)min(x0 + k, a.width - 1) * a.src_w / a.width);
    Y[k] = yr[ix];
    A[k] = ar ? (int)ar[ix] : 0;
    if (bilinear) {
      Cb[k] = bilinear_chroma<Pixel>(reinterpret_cast<const Pixel*>(a.cb), a.c_stride, a.src_w, a.src_h, ix, iy, shiftV != 0, pre, ind, outd);
      Cr[k] = bilinear_chroma<Pixel>(reinterpret_cast<const Pixel*>(a.cr), a.c_stride, a.src_w, a.src_h, ix, iy, shiftV != 0, pre, ind, outd);
    } else if (a.chroma_format) {
      Cb[k] = reinterpret_cast<const Pixel*>(a.cb)[crow + (ix >> shiftH)];
      Cr[k] = reinterpret_cast<const Pixel*>(a.cr)[crow + (ix >> shiftH)];
    } else {
      Cb[k] = Cr[k] = half_in;
    }
  }
}

// GATHER: this instantiation also serves canvases whose CscArgs::gather is set (a CTA-uniform choice of the canvas);
// the instantiation without it is the plain same-size conversion.
template <typename Pixel, bool GATHER>
__device__ __forceinline__ void csc_unit(const CscArgs& a, unsigned tid) {
  const unsigned nq = (unsigned)(a.width + 7) >> 3;
  if (tid >= nq * (unsigned)a.height) return;
  const int y = (int)(tid / nq), x0 = (int)(tid - (unsigned)y * nq) << 3;
  const int n = min(8, a.width - x0);
  const int shiftH = (a.chroma_format == 1 || a.chroma_format == 2) ? 1 : 0;
  const int shiftV = a.chroma_format == 1 ? 1 : 0;
  const int fmt = a.p.out_format;
  const int ind = a.p.in_depth, outd = a.p.out_depth, pre = a.p.pre_op, post = a.p.post_op;
  // the neutral chroma value of the planes as stored: padding lanes, and the planes Op_mono_to_YCbCr420 adds to a
  // monochrome image (monochrome.cc:99-100,128)
  const int half_in = 128 << (ind - 8);

  int Y[8], Cb[8], Cr[8], A[8];
  const bool bilinear = a.p.upsampling == HC_UPSAMPLE_BILINEAR && shiftH;   // warp-uniform
  if (GATHER && a.gather) {
    gather_px8<Pixel>(a, y, x0, bilinear, shiftH, shiftV, half_in, Y, Cb, Cr, A);
  } else {
    load_px8<Pixel>(reinterpret_cast<const Pixel*>(a.y) + (size_t)y * a.y_stride + x0, n, Y);
    if (bilinear) {
#pragma unroll 1
      for (int k = 0; k < 8; k++) {
        const int x = min(x0 + k, a.width - 1);
        Cb[k] = bilinear_chroma<Pixel>(reinterpret_cast<const Pixel*>(a.cb), a.c_stride, a.width, a.height, x, y, shiftV != 0, pre, ind, outd);
        Cr[k] = bilinear_chroma<Pixel>(reinterpret_cast<const Pixel*>(a.cr), a.c_stride, a.width, a.height, x, y, shiftV != 0, pre, ind, outd);
      }
    } else if (a.chroma_format) {
      const size_t coff = (size_t)(y >> shiftV) * a.c_stride + (x0 >> shiftH);
      int cb[8], cr[8];
      const int nc = shiftH ? (n + 1) >> 1 : n;
      if (shiftH) {
        // 4 (or fewer) chroma samples cover the 8 pixels: nearest neighbour, cx = x >> 1 (yuv2rgb.cc:173-174)
        load_px4<Pixel>(reinterpret_cast<const Pixel*>(a.cb) + coff, nc, half_in, cb);
        load_px4<Pixel>(reinterpret_cast<const Pixel*>(a.cr) + coff, nc, half_in, cr);
#pragma unroll
        for (int k = 0; k < 8; k++) { Cb[k] = cb[k >> 1]; Cr[k] = cr[k >> 1]; }
      } else {
        load_px8<Pixel>(reinterpret_cast<const Pixel*>(a.cb) + coff, n, Cb);
        load_px8<Pixel>(reinterpret_cast<const Pixel*>(a.cr) + coff, n, Cr);
      }
    } else {
#pragma unroll
      for (int k = 0; k < 8; k++) Cb[k] = Cr[k] = half_in;
    }
    if (a.a) load_px8<Pixel>(reinterpret_cast<const Pixel*>(a.a) + (size_t)y * a.a_stride + x0, n, A);
  }
  if (pre != HC_DEPTH_NONE) {   // warp-uniform
#pragma unroll
    for (int k = 0; k < 8; k++) {
      Y[k] = depth_op(pre, Y[k], ind, outd);
      if (!bilinear) {          // the bilinear fetch applied it to the samples it read
        Cb[k] = depth_op(pre, Cb[k], ind, outd);
        Cr[k] = depth_op(pre, Cr[k], ind, outd);
      }
      A[k] = depth_op(pre, A[k], ind, outd);
    }
  }

  int R[8], G[8], B[8];
  if (a.p.mode == HC_CSC_MONO) {
#pragma unroll
    for (int k = 0; k < 8; k++) R[k] = G[k] = B[k] = Y[k];
  } else if (a.p.mode == HC_CSC_INT420) {
#pragma unroll
    for (int k = 0; k < 8; k++) convert_px<Pixel, HC_CSC_INT420>(a, Y[k], Cb[k], Cr[k], R[k], G[k], B[k]);
  } else if (a.p.mode == HC_CSC_FLOAT) {
#pragma unroll
    for (int k = 0; k < 8; k++) convert_px<Pixel, HC_CSC_FLOAT>(a, Y[k], Cb[k], Cr[k], R[k], G[k], B[k]);
  } else if (a.p.mode == HC_CSC_GBR) {
#pragma unroll
    for (int k = 0; k < 8; k++) convert_px<Pixel, HC_CSC_GBR>(a, Y[k], Cb[k], Cr[k], R[k], G[k], B[k]);
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++) convert_px<Pixel, HC_CSC_YCGCO>(a, Y[k], Cb[k], Cr[k], R[k], G[k], B[k]);
  }
  if (post != HC_DEPTH_NONE) {   // warp-uniform; the matrix ran at the input depth
#pragma unroll
    for (int k = 0; k < 8; k++) {
      R[k] = depth_op(post, R[k], ind, outd);
      G[k] = depth_op(post, G[k], ind, outd);
      B[k] = depth_op(post, B[k], ind, outd);
      A[k] = depth_op(post, A[k], ind, outd);
    }
  }
  if (!a.a) {   // a missing alpha plane is opaque at the final depth (yuv2rgb.cc:470, rgb2rgb.cc:251,264)
#pragma unroll
    for (int k = 0; k < 8; k++) A[k] = (1 << outd) - 1;
  }
  if (a.p.premultiply && fmt == HC_OUT_RGBA) {   // heif_image_rgba_premultiply_alpha, PREMULTI_PIXEL (pixelimage.cc:896-900)
#pragma unroll
    for (int k = 0; k < 8; k++) {
      R[k] = (R[k] * A[k] + 128) >> 8;
      G[k] = (G[k] * A[k] + 128) >> 8;
      B[k] = (B[k] * A[k] + 128) >> 8;
    }
  }

  uint8_t* orow = a.out + (size_t)y * a.out_stride;
  if (fmt == HC_OUT_RGB) {
    uint32_t w[6];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int k = 4 * h;
      w[3 * h + 0] = R[k] | (G[k] << 8) | (B[k] << 16) | (R[k + 1] << 24);
      w[3 * h + 1] = G[k + 1] | (B[k + 1] << 8) | (R[k + 2] << 16) | (G[k + 2] << 24);
      w[3 * h + 2] = B[k + 2] | (R[k + 3] << 8) | (G[k + 3] << 16) | (B[k + 3] << 24);
    }
    uint2* o = reinterpret_cast<uint2*>(orow + (size_t)x0 * 3);   // x0 * 3 is a multiple of 8
    o[0] = make_uint2(w[0], w[1]); o[1] = make_uint2(w[2], w[3]); o[2] = make_uint2(w[4], w[5]);
  } else if (fmt == HC_OUT_RGBA) {
    uint4* o = reinterpret_cast<uint4*>(orow + (size_t)x0 * 4);
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int k = 4 * h;
      uint4 v;
      v.x = R[k] | (G[k] << 8) | (B[k] << 16) | ((uint32_t)A[k] << 24);
      v.y = R[k + 1] | (G[k + 1] << 8) | (B[k + 1] << 16) | ((uint32_t)A[k + 1] << 24);
      v.z = R[k + 2] | (G[k + 2] << 8) | (B[k + 2] << 16) | ((uint32_t)A[k + 2] << 24);
      v.w = R[k + 3] | (G[k + 3] << 8) | (B[k + 3] << 16) | ((uint32_t)A[k + 3] << 24);
      o[h] = v;
    }
  } else {
    const bool le = (fmt == HC_OUT_RRGGBB_LE || fmt == HC_OUT_RRGGBBAA_LE);
    const bool alpha = (fmt == HC_OUT_RRGGBBAA_BE || fmt == HC_OUT_RRGGBBAA_LE);
    auto h16 = [&](int v) -> uint32_t { return le ? (uint32_t)v : (uint32_t)(((v & 0xff) << 8) | (v >> 8)); };
    if (alpha) {
      uint4* o = reinterpret_cast<uint4*>(orow + (size_t)x0 * 8);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        uint4 v;
        v.x = h16(R[2 * k]) | (h16(G[2 * k]) << 16);
        v.y = h16(B[2 * k]) | (h16(A[2 * k]) << 16);
        v.z = h16(R[2 * k + 1]) | (h16(G[2 * k + 1]) << 16);
        v.w = h16(B[2 * k + 1]) | (h16(A[2 * k + 1]) << 16);
        o[k] = v;
      }
    } else {
      uint32_t w[12];
#pragma unroll
      for (int h = 0; h < 4; h++) {
        const int k = 2 * h;
        w[3 * h + 0] = h16(R[k]) | (h16(G[k]) << 16);
        w[3 * h + 1] = h16(B[k]) | (h16(R[k + 1]) << 16);
        w[3 * h + 2] = h16(G[k + 1]) | (h16(B[k + 1]) << 16);
      }
      uint4* o = reinterpret_cast<uint4*>(orow + (size_t)x0 * 6);   // x0 * 6 is a multiple of 16
      o[0] = make_uint4(w[0], w[1], w[2], w[3]); o[1] = make_uint4(w[4], w[5], w[6], w[7]); o[2] = make_uint4(w[8], w[9], w[10], w[11]);
    }
  }
}

// All canvases of a batch in one launch (blockIdx.y = canvas): a 12 MP canvas is a ~10 us kernel at HBM speed, so
// per-canvas launches are dominated by launch gaps and tails.
template <typename Pixel, bool GATHER>
__global__ void __launch_bounds__(256) k5_csc_batch_kernel(CscBatch b) {
  __shared__ CscArgs sa;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&b.a[blockIdx.y]);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&sa);
    for (int i = threadIdx.x; i < (int)(sizeof(CscArgs) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  csc_unit<Pixel, GATHER>(sa, blockIdx.x * blockDim.x + threadIdx.x);
}

// Fast path of the common case — 8-bit 4:2:0, integer matrix (Op_YCbCr420_to_RGB24, yuv2rgb.cc:260-375), no alpha, RGB24,
// width a multiple of 8 and even height: one thread converts an 8 x 2 pixel block, so the four chroma pairs it needs
// are loaded and multiplied once for 16 pixels (the generic kernel spends ~45 instructions per pixel, this one ~16).
__global__ void __launch_bounds__(256) k5_int420_rgb24_kernel(CscBatch b) {
  __shared__ CscArgs sa;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&b.a[blockIdx.y]);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&sa);
    for (int i = threadIdx.x; i < (int)(sizeof(CscArgs) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const CscArgs& a = sa;
  const unsigned nq = (unsigned)a.width >> 3, rows2 = (unsigned)a.height >> 1;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= nq * rows2) return;
  const int y = (int)(tid / nq) << 1, x0 = (int)(tid % nq) << 3;
  const uint2 y0 = *reinterpret_cast<const uint2*>(a.y + (size_t)y * a.y_stride + x0);
  const uint2 y1 = *reinterpret_cast<const uint2*>(a.y + (size_t)(y + 1) * a.y_stride + x0);
  const size_t coff = (size_t)(y >> 1) * a.c_stride + (x0 >> 1);
  const uint32_t cbw = *reinterpret_cast<const uint32_t*>(a.cb + coff), crw = *reinterpret_cast<const uint32_t*>(a.cr + coff);
  const int r_cr = a.p.r_cr_i, g_cb = a.p.g_cb_i, g_cr = a.p.g_cr_i, b_cb = a.p.b_cb_i;
  int rc[4], gc[4], bc[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int cb = (int)((cbw >> (8 * k)) & 0xff) - 128, cr = (int)((crw >> (8 * k)) & 0xff) - 128;
    rc[k] = (r_cr * cr + 128) >> 8;
    gc[k] = (g_cb * cb + g_cr * cr + 128) >> 8;
    bc[k] = (b_cb * cb + 128) >> 8;
  }
#pragma unroll
  for (int row = 0; row < 2; row++) {
    const uint2 yw = row ? y1 : y0;
    uint32_t R[8], G[8], B[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int yv = (int)(((k < 4 ? yw.x : yw.y) >> (8 * (k & 3))) & 0xff);
      R[k] = (uint32_t)min(max(yv + rc[k >> 1], 0), 255);
      G[k] = (uint32_t)min(max(yv + gc[k >> 1], 0), 255);
      B[k] = (uint32_t)min(max(yv + bc[k >> 1], 0), 255);
    }
    uint32_t w[6];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int k = 4 * h;
      w[3 * h + 0] = R[k] | (G[k] << 8) | (B[k] << 16) | (R[k + 1] << 24);
      w[3 * h + 1] = G[k + 1] | (B[k + 1] << 8) | (R[k + 2] << 16) | (G[k + 2] << 24);
      w[3 * h + 2] = B[k + 2] | (R[k + 3] << 8) | (G[k + 3] << 16) | (B[k + 3] << 24);
    }
    uint2* o = reinterpret_cast<uint2*>(a.out + (size_t)(y + row) * a.out_stride + (size_t)x0 * 3);
    o[0] = make_uint2(w[0], w[1]); o[1] = make_uint2(w[2], w[3]); o[2] = make_uint2(w[4], w[5]);
  }
}

static bool k5_fast_path(const CscArgs& a, bool sixteen_bit) {
  return !sixteen_bit && !a.gather && a.chroma_format == 1 && a.p.mode == HC_CSC_INT420 && a.p.out_format == HC_OUT_RGB && a.a == nullptr &&
         a.p.pre_op == HC_DEPTH_NONE && a.p.post_op == HC_DEPTH_NONE && a.p.upsampling == HC_UPSAMPLE_NEAREST && !a.p.premultiply &&
         (a.width & 7) == 0 && (a.height & 1) == 0 && (a.y_stride & 7) == 0 && (a.c_stride & 3) == 0 &&
         (reinterpret_cast<uintptr_t>(a.y) & 7) == 0 && (reinterpret_cast<uintptr_t>(a.cb) & 3) == 0 && (reinterpret_cast<uintptr_t>(a.cr) & 3) == 0 &&
         (a.out_stride & 7) == 0 && (reinterpret_cast<uintptr_t>(a.out) & 7) == 0;
}

void launch_k5_batch(const CscBatch& b, bool sixteen_bit, cudaStream_t stream) {
  long long nmax = 0;
  for (int i = 0; i < b.n; i++) nmax = std::max(nmax, (long long)((b.a[i].width + 7) >> 3) * b.a[i].height);
  if (nmax <= 0 || b.n <= 0) return;
  bool fast = true, gather = false;
  for (int i = 0; i < b.n; i++) fast = fast && k5_fast_path(b.a[i], sixteen_bit);
  for (int i = 0; i < b.n; i++) gather = gather || b.a[i].gather;
  if (fast) {   // 16 pixels per thread
    k5_int420_rgb24_kernel<<<dim3((unsigned)((nmax / 2 + 255) / 256), (unsigned)b.n), 256, 0, stream>>>(b);
    return;
  }
  dim3 grid((unsigned)((nmax + 255) / 256), (unsigned)b.n);
  if (gather) {   // a scaled canvas in the launch: the instantiation with the gather form
    if (sixteen_bit) k5_csc_batch_kernel<uint16_t, true><<<grid, 256, 0, stream>>>(b);
    else k5_csc_batch_kernel<uint8_t, true><<<grid, 256, 0, stream>>>(b);
  } else {
    if (sixteen_bit) k5_csc_batch_kernel<uint16_t, false><<<grid, 256, 0, stream>>>(b);
    else k5_csc_batch_kernel<uint8_t, false><<<grid, 256, 0, stream>>>(b);
  }
}

}  // namespace hc
