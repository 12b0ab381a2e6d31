// k8_planar.cu — K8: the output planes of canvases (Y, Cb, Cr, A in the plane pool, rows at 128-byte pitches) packed into
// HC_OUT_YCBCR images (tight rows, plane after plane), so that one image is one contiguous block that a single 1-D copy
// reads back. Pure byte movement: 8- and 16-bit samples are the same to it.
//
// A plane is rows x row_bytes bytes in the destination. Every thread writes one 16-byte-aligned chunk of it; the unaligned
// head (before the first aligned address) and the partial tail are written bytewise by the first and the last thread. A
// chunk whose 16 source bytes lie in one row is read with one 16-byte load when source and destination are equally
// aligned (the plane starts and rows of 8-bit 4:2:0 images with widths that are multiples of 32), else with four or five
// aligned 4-byte loads and funnel shifts; a chunk that straddles rows (row_bytes not a multiple of 16) gathers bytewise.
#include "launch.h"

namespace hc {

namespace {

__device__ __forceinline__ uint8_t src_byte(const PackPlane& p, unsigned i) {
  const unsigned row = i / p.row_bytes;
  return p.src[(size_t)row * p.src_pitch + (i - row * p.row_bytes)];
}

}  // namespace

__global__ void __launch_bounds__(256) k8_pack_kernel(PackBatch b) {
  const PackPlane& p = b.p[blockIdx.y];
  const unsigned n = p.row_bytes * p.rows;          // < 2^32: at most 32768 x 32768 samples of 2 bytes
  const unsigned head = min(n, (unsigned)((16 - (reinterpret_cast<uintptr_t>(p.dst) & 15)) & 15));
  const unsigned nchunks = (n - head + 15) / 16;
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > nchunks) return;
  if (t == 0) {                                     // unaligned head
    for (unsigned i = 0; i < head; i++) p.dst[i] = src_byte(p, i);
    return;
  }
  const unsigned i0 = head + (t - 1) * 16;
  if (i0 + 16 > n) {                                // partial tail
    for (unsigned i = i0; i < n; i++) p.dst[i] = src_byte(p, i);
    return;
  }
  uint4* out = reinterpret_cast<uint4*>(p.dst + i0);
  const unsigned row = i0 / p.row_bytes, col = i0 - row * p.row_bytes;
  if (col + 16 <= p.row_bytes) {
    const uint8_t* s = p.src + (size_t)row * p.src_pitch + col;
    const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(s) & 15);
    if (mis == 0) {
      *out = __ldg(reinterpret_cast<const uint4*>(s));
      return;
    }
    // the aligned words that hold s[0..15]; the fifth only when s is not 4-byte aligned (it then still holds s[15])
    const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(s) & ~(uintptr_t)3);
    const unsigned sh = (unsigned)(reinterpret_cast<uintptr_t>(s) & 3) * 8;
    const uint32_t w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2), w3 = __ldg(w + 3), w4 = sh ? __ldg(w + 4) : 0u;
    *out = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
    return;
  }
  uint32_t v[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    uint32_t x = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) x |= (uint32_t)src_byte(p, i0 + 4 * k + j) << (8 * j);
    v[k] = x;
  }
  *out = make_uint4(v[0], v[1], v[2], v[3]);
}

void launch_k8_batch(const PackBatch& b, cudaStream_t stream) {
  unsigned threads = 0;
  for (int i = 0; i < b.n; i++) {
    const unsigned n = b.p[i].row_bytes * b.p[i].rows;
    threads = max(threads, 1 + (n + 15) / 16);       // head thread + chunks (an upper bound)
  }
  if (b.n <= 0 || threads <= 1) return;
  k8_pack_kernel<<<dim3((threads + 255) / 256, (unsigned)b.n), 256, 0, stream>>>(b);
}

}  // namespace hc
