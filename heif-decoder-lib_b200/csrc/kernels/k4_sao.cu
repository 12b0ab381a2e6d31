// k4_sao.cu — K4: sample adaptive offset + conformance-window crop + paste into the destination
// image (own picture or HEIF grid canvas) in ONE pass.
//
// Replaces apply_sample_adaptive_offset_sequential (sao.cc:552-625: full-plane copy, then
// apply_sao_internal :261-488 with sao_band_filter / sao_edge_filter, fallback-postfilter.h:216-315),
// the conformance-window copy of convert_libde265_image_to_heif_image (decoder_libde265.cc:88-157)
// and the tile paste of decode_and_paste_tile_image (context.cc:2407-2539) including its
// limited->full range rescale of limited-range tiles (:2504-2528).
//
// The reference needs a deblocked copy of every plane because it filters in place; here the
// deblocked reconstruction planes are read-only input and the result is written straight to its
// final position, so the copy, the crop and the paste cost no extra memory pass.
//
// Mapping: one thread per 8 horizontally adjacent samples (8-aligned, so a unit never straddles a
// CTB: CTBs are >= 8 samples wide in every component); the unit's row and, for the edge classes,
// the rows above / below are fetched with one 8- or 16-byte load each. A warp covers a
// (CTB width) x (256 / CTB width) patch of ONE CTB, so SAO type, class and offsets are warp-uniform.
// Algorithmic bytes: read s + write s per sample (neighbour rows hit L1/L2).
#include "postfilter_core.cuh"

namespace hc {

// One CTB of one colour plane by one warp: the warp walks the CTB's row groups. lane -> (8-sample unit in the CTB row, row
// inside the group); a warp pass covers (CTB width / 8) units x (256 / CTB width) rows of ONE CTB, so the SAO type / class /
// offsets are warp-uniform and only the CTB-border handling differs between lanes.
template <typename Pixel>
__device__ __forceinline__ void sao_ctb(const BatchView& bv, const hc_pic& pic, int c, unsigned ctb, int lane) {
  SaoPlane<Pixel> P;
  P.init(bv, pic, c);
  const int lu = P.log2w - 3;                        // log2 units per CTB row (0..3)
  const int rows = 32 >> lu;                         // rows per warp pass
  const int ctby = (int)(ctb / pic.ctbs_w), ctbx = (int)(ctb - (unsigned)ctby * pic.ctbs_w);
  const int x0 = (ctbx << P.log2w) + ((lane & ((1 << lu) - 1)) << 3);
  if (x0 >= P.width) return;
  const Pixel* __restrict__ src = reinterpret_cast<const Pixel*>(bv.planes + pic.rec_off[c]);
  const int sstride = (int)pic.rec_stride[c];
  const int y_end = min(P.height, (ctby + 1) << P.log2h);
  for (int y = (ctby << P.log2h) + (lane >> lu); y < y_end; y += rows)
    sao_unit<Pixel>(bv, pic, P, x0, y, src + (size_t)y * sstride + x0, sstride);
}

// One warp per CTB (it walks the CTB's row groups), 8 CTBs per CTA, the picture descriptor staged in shared memory:
// a CTA moves 8 x 4 KB instead of 2 KB, so the pass is no longer bound by CTA launch rate and descriptor loads
// (the first version was: 147 K CTAs per 8 x 12 MP step, half of them empty chroma CTAs).
__global__ void __launch_bounds__(256, 5) k4_sao_kernel(BatchView bv) {
  __shared__ hc_pic spic;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(bv.pics + blockIdx.y);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&spic);
    for (int i = threadIdx.x; i < (int)(sizeof(hc_pic) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const hc_pic& pic = spic;
  const int c = blockIdx.z;
  if (c > 0 && pic.chroma_format == 0) return;
  if (pic.dst_flags & (HC_DST_SKIP_Y << c)) return;   // component not wanted at the destination
  const unsigned ctb = blockIdx.x * 8u + (threadIdx.x >> 5);
  if (ctb >= (unsigned)pic.ctbs_w * pic.ctbs_h) return;
  const int lane = threadIdx.x & 31;
  if (pic.bit_depth_y == 8 && pic.bit_depth_c == 8) sao_ctb<uint8_t>(bv, pic, c, ctb, lane);
  else sao_ctb<uint16_t>(bv, pic, c, ctb, lane);
}

// max_ctbs = max over pictures of the number of CTBs
void launch_k4(const BatchView& bv, long long max_ctbs, int planes, cudaStream_t stream) {
  if (max_ctbs <= 0 || bv.npics <= 0) return;
  dim3 grid((unsigned)((max_ctbs + 7) / 8), (unsigned)bv.npics, (unsigned)planes);
  k4_sao_kernel<<<grid, 256, 0, stream>>>(bv);
}

}  // namespace hc
