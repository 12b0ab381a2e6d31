// k6_transform.cu — K6: geometric transformations of a decoded image (irot / imir item properties) on its planes,
// between K4 (SAO + paste) and K5 (colour conversion).
//
// Replaces HeifPixelImage::rotate_ccw (pixelimage.cc:539-741) and HeifPixelImage::mirror_inplace (:743-794) as
// HeifContext::decode_image_planar applies them in ipma order (context.cc:1955-1978). The reference transforms every
// plane by itself with that plane's own width / height (so odd sizes and subsampled chroma behave exactly as there);
// any sequence of rotations and mirrors of a plane is one of the eight dihedral maps, composed on the host
// (engine: hc_batch_set_canvas_transform).
//
// Mapping: one thread per output sample through a 32 x 32 shared tile when the map swaps the axes (reads and writes
// both coalesced), a plain gather otherwise. Algorithmic bytes: read s + write s per sample.
#include <algorithm>

#include "launch.h"

namespace hc {

template <typename Pixel>
__global__ void __launch_bounds__(256) k6_transform_kernel(XformArgs a) {
  __shared__ Pixel tile[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8 threads, 4 rows each
  const Pixel* __restrict__ src = reinterpret_cast<const Pixel*>(a.src);
  Pixel* __restrict__ dst = reinterpret_cast<Pixel*>(a.dst);
  const int ow = a.swap ? a.h : a.w, oh = a.swap ? a.w : a.h;
  const int ox0 = blockIdx.x * 32, oy0 = blockIdx.y * 32;
  if (!a.swap) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int ox = ox0 + tx, oy = oy0 + ty + 8 * r;
      if (ox < ow && oy < oh) {
        const int sx = a.flip_x ? a.w - 1 - ox : ox, sy = a.flip_y ? a.h - 1 - oy : oy;
        dst[(size_t)oy * a.dst_stride + ox] = src[(size_t)sy * a.src_stride + sx];
      }
    }
    return;
  }
  // swapped axes: output tile (ox0.., oy0..) comes from input columns sx(oy) and input rows sy(ox); read the input
  // tile row-wise (tx along input x), write the output tile row-wise (tx along output x)
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int j = ty + 8 * r;                 // input row index inside the tile <-> output x offset
    const int ox = ox0 + j, oy = oy0 + tx;    // this load serves output sample (ox0 + j, oy0 + tx)
    if (ox < ow && oy < oh) {
      const int sx = a.flip_x ? a.w - 1 - oy : oy, sy = a.flip_y ? a.h - 1 - ox : ox;
      tile[j][tx] = src[(size_t)sy * a.src_stride + sx];
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int i = ty + 8 * r;
    const int ox = ox0 + tx, oy = oy0 + i;
    if (ox < ow && oy < oh) dst[(size_t)oy * a.dst_stride + ox] = tile[tx][i];
  }
}

// Nearest-neighbour rescale of a plane: HeifPixelImage::scale_nearest_neighbor (pixelimage.cc:1231-1250), used by the
// reference for an alpha image whose size differs from its colour image's (context.cc:2064-2071).
template <typename Pixel>
__global__ void __launch_bounds__(256) k6_scale_kernel(const Pixel* __restrict__ src, int sw, int sh, int src_stride, Pixel* __restrict__ dst,
                                                       int dw, int dh, int dst_stride) {
  const int x = blockIdx.x * 32 + (threadIdx.x & 31);
  if (x >= dw) return;
  const int ix = (int)((long long)x * sw / dw);
  // gridDim.y is at most 65,535: taller planes are covered by striding over 32-row blocks
  for (int y0 = blockIdx.y * 32; y0 < dh; y0 += gridDim.y * 32) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int y = y0 + (threadIdx.x >> 5) + 8 * r;
      if (y >= dh) continue;
      const int iy = (int)((long long)y * sh / dh);
      dst[(size_t)y * dst_stride + x] = src[(size_t)iy * src_stride + ix];
    }
  }
}

void launch_k6_scale(const uint8_t* src, int sw, int sh, int src_stride, uint8_t* dst, int dw, int dh, int dst_stride, bool sixteen_bit,
                     cudaStream_t stream) {
  if (sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0) return;
  dim3 grid((unsigned)((dw + 31) / 32), (unsigned)std::min((dh + 31) / 32, kMaxGridY));
  if (sixteen_bit)
    k6_scale_kernel<uint16_t><<<grid, 256, 0, stream>>>(reinterpret_cast<const uint16_t*>(src), sw, sh, src_stride, reinterpret_cast<uint16_t*>(dst), dw, dh, dst_stride);
  else
    k6_scale_kernel<uint8_t><<<grid, 256, 0, stream>>>(src, sw, sh, src_stride, dst, dw, dh, dst_stride);
}

void launch_k6(const XformArgs& a, bool sixteen_bit, cudaStream_t stream) {
  if (a.w <= 0 || a.h <= 0) return;
  const int ow = a.swap ? a.h : a.w, oh = a.swap ? a.w : a.h;
  // gridDim.y is at most 65,535 blocks of 32 output rows. A taller output is transformed in bands of output rows; a band
  // is the same map on a sub-image of the input: rows of the input without swap, columns with swap (from the far end when
  // that axis is flipped).
  const size_t ps = sixteen_bit ? 2 : 1;
  for (int r0 = 0; r0 < oh; r0 += kMaxGridY * 32) {
    const int n = std::min(oh - r0, kMaxGridY * 32);
    XformArgs b = a;
    b.dst = a.dst + (size_t)r0 * a.dst_stride * ps;
    if (!a.swap) {
      b.h = n;
      b.src = a.src + (size_t)(a.flip_y ? a.h - r0 - n : r0) * a.src_stride * ps;
    } else {
      b.w = n;
      b.src = a.src + (size_t)(a.flip_x ? a.w - r0 - n : r0) * ps;
    }
    dim3 grid((unsigned)((ow + 31) / 32), (unsigned)((n + 31) / 32));
    if (sixteen_bit) k6_transform_kernel<uint16_t><<<grid, 256, 0, stream>>>(b);
    else k6_transform_kernel<uint8_t><<<grid, 256, 0, stream>>>(b);
  }
}

}  // namespace hc
