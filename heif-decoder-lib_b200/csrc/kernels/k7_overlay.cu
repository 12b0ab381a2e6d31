// k7_overlay.cu — K7: 'iovl' derived images composed on the device, straight into the interleaved output.
//
// Replaces HeifContext::decode_overlay_image (context.cc:2579-2675) and HeifPixelImage::overlay (pixelimage.cc:1017-1150)
// plus the colour conversions around them: the reference fills an 8-bit planar RGB canvas with the background colour
// (fill_RGB_16bit, :943-1000: the high byte of the 16-bit values), converts every child image to planar RGB 4:4:4
// (Op_YCbCr_to_RGB<uint8_t>, yuv2rgb.cc:28-254 — it only finds a pipeline for 4:4:4 children), overlays the children in
// reference order — a copy, or (child * a + canvas * (255 - a)) / 255 when the child has an alpha plane — and finally
// interleaves the canvas (Op_RGB_to_RGB24_32, rgb2rgb.cc:28-143; Op_to_hdr_planes + Op_RGB_HDR_to_RRGGBBaa_BE [+ swap] for the
// RRGGBB(AA) targets). Here one thread owns one output pixel and walks the child list in the same order, so no planar
// canvas, no per-child pass and no extra allocation exist. Children are canvases of the batch after K4 / K6.
#include <algorithm>

#include "launch.h"

namespace hc {

HC_D int k7_clip_f(float fx, int maxi) {
  const long long x = (long long)__fadd_rn(fx, 0.5f);
  return x < 0 ? 0 : (x > maxi ? maxi : (int)x);
}

// SCALED: output pixel (x, y) of a band is the composition at canvas pixel (x * src_w / width, (row0 + y) * src_h / full_h)
// (HeifPixelImage::scale_nearest_neighbor of the composed image, pixelimage.cc:1156-1253); otherwise at (x, y) itself.
template <bool SCALED>
__global__ void __launch_bounds__(256) k7_overlay_kernel(OverlayArgs a) {
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= a.width || y >= a.height) return;
  int sx = x, sy = y;
  if (SCALED) {
    sx = (int)((long long)x * a.src_w / a.width);
    sy = (int)((long long)(a.row0 + y) * a.src_h / a.full_h);
  }
  int R = a.bkg[0], G = a.bkg[1], B = a.bkg[2];
  for (int k = 0; k < a.n; k++) {
    const OverlayChild& c = a.child[k];
    const int cx = sx - c.dx, cy = sy - c.dy;
    if (cx < 0 || cy < 0 || cx >= c.w || cy >= c.h) continue;
    const int yv = c.y[(size_t)cy * c.y_stride + cx], cbv = c.cb[(size_t)cy * c.c_stride + cx], crv = c.cr[(size_t)cy * c.c_stride + cx];
    int r, g, b;
    if (c.mode == HC_CSC_GBR) {            // yuv2rgb.cc:197-211
      if (c.full_range) { r = crv; g = yv; b = cbv; }
      else {
        r = k7_clip_f(__fmul_rn(__fsub_rn((float)crv, 16.f), 1.1429f), 255);
        g = k7_clip_f(__fmul_rn(__fsub_rn((float)yv, 16.f), 1.1689f), 255);
        b = k7_clip_f(__fmul_rn(__fsub_rn((float)cbv, 16.f), 1.1429f), 255);
      }
    } else if (c.mode == HC_CSC_YCGCO) {   // :212-226
      const int c1 = cbv - 128, c2 = crv - 128;
      r = clip3i(0, 255, yv - c1 + c2);
      g = clip3i(0, 255, yv + c1);
      b = clip3i(0, 255, yv - c1 - c2);
    } else {                               // :227-244
      float fy = (float)yv, fcb = (float)(cbv - 128), fcr = (float)(crv - 128);
      if (!c.full_range) {
        fy = __fmul_rn(__fsub_rn(fy, 16.f), 1.1689f);
        fcb = __fmul_rn(fcb, 1.1429f);
        fcr = __fmul_rn(fcr, 1.1429f);
      }
      r = k7_clip_f(__fadd_rn(fy, __fmul_rn(c.r_cr, fcr)), 255);
      g = k7_clip_f(__fadd_rn(__fadd_rn(fy, __fmul_rn(c.g_cb, fcb)), __fmul_rn(c.g_cr, fcr)), 255);
      b = k7_clip_f(__fadd_rn(fy, __fmul_rn(c.b_cb, fcb)), 255);
    }
    if (c.a) {                             // pixelimage.cc:1141-1143
      const int al = c.a[(size_t)cy * c.a_stride + cx];
      R = (r * al + R * (255 - al)) / 255;
      G = (g * al + G * (255 - al)) / 255;
      B = (b * al + B * (255 - al)) / 255;
    } else {
      R = r; G = g; B = b;
    }
  }
  uint8_t* o = a.out + (size_t)y * a.out_stride;
  const int fmt = a.out_format;
  if (fmt == HC_OUT_RGB) {
    o[3 * x] = (uint8_t)R; o[3 * x + 1] = (uint8_t)G; o[3 * x + 2] = (uint8_t)B;
  } else if (fmt == HC_OUT_RGBA) {
    *reinterpret_cast<uint32_t*>(o + 4 * x) = (uint32_t)R | ((uint32_t)G << 8) | ((uint32_t)B << 16) | 0xff000000u;
  } else {
    // Op_to_hdr_planes (8 -> 10 bit) on R, G, B; a missing alpha plane is opaque at 10 bit (rgb2rgb.cc:251,264)
    const bool le = fmt == HC_OUT_RRGGBB_LE || fmt == HC_OUT_RRGGBBAA_LE, alpha = fmt == HC_OUT_RRGGBBAA_BE || fmt == HC_OUT_RRGGBBAA_LE;
    const int v[4] = {(R << 2) | (R >> 6), (G << 2) | (G >> 6), (B << 2) | (B >> 6), 1023};
    const int ps = alpha ? 8 : 6;
    for (int c = 0; c < (alpha ? 4 : 3); c++) {
      o[ps * x + 2 * c + (le ? 1 : 0)] = (uint8_t)(v[c] >> 8);
      o[ps * x + 2 * c + (le ? 0 : 1)] = (uint8_t)(v[c] & 0xff);
    }
  }
}

void launch_k7(const OverlayArgs& a, cudaStream_t stream) {
  if (a.width <= 0 || a.height <= 0) return;
  // gridDim.y is at most 65,535 blocks of 8 rows: a taller image is composed in bands of delivered rows, each with its output
  // rows and the children's offsets shifted up by the band's first row (scaled: the band's first row is passed instead)
  const bool scaled = a.src_w != a.width || a.src_h != a.height;
  for (int r0 = 0; r0 < a.height; r0 += kMaxGridY * 8) {
    OverlayArgs b = a;
    b.height = std::min(a.height - r0, kMaxGridY * 8);
    b.out = a.out + r0 * a.out_stride;
    b.row0 = r0;
    b.full_h = a.height;
    const dim3 grid((unsigned)((a.width + 31) / 32), (unsigned)((b.height + 7) / 8));
    if (scaled) {
      k7_overlay_kernel<true><<<grid, 256, 0, stream>>>(b);
    } else {
      for (int k = 0; k < a.n; k++) b.child[k].dy = a.child[k].dy - r0;
      k7_overlay_kernel<false><<<grid, 256, 0, stream>>>(b);
    }
  }
}

}  // namespace hc
