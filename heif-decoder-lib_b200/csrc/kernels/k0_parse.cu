// k0_parse.cu — K0 on the device: one warp (lane 0 walks the syntax) per substream chain, K0_WARPS chains per CTA.
//
// CABAC is serial inside a substream, so the parallelism is across substreams: the CTB rows of WPP pictures
// (wavefront-synchronised with the row above, kernels/k0_core.cuh) and across the pictures / grid tiles / files of a
// batch — a 12 MP iPhone-style grid image is 48 tiles x 8 rows = 384 chains; a batch of 8 such files keeps 3072
// chains in flight. Chains are ordered row-major across all pictures so that a chain only ever waits for a chain
// with a smaller index (scheduled no later than itself). Tables, context states and the picture / slice descriptors
// of a chain live in shared memory (k0_core.cuh: Scratch).
#include "launch.h"
#include "k0_core.cuh"

namespace hc {

// Chains per CTA: the warps of a CTA share one shared-memory copy of the parser tables; each warp owns a Scratch
// (context states, picture / slice descriptors, K1 list staging). Consecutive chains are the same CTB row of
// consecutive pictures, so the warps of a CTA run for about the same time.
constexpr int K0_WARPS = 4;

// K0_MIN_CTAS: CTAs per SM the register allocation must allow (5 -> 96 registers, 6 -> 80, 8 -> 64). A chain uses one
// lane, so resident chains per SM = 4 * K0_MIN_CTAS is limited by registers x 32 lanes: the value trades spills in a chain
// against chains in flight. Measured per 32 x 12 MP (DESIGN.md), v6 (one lane per chain): 5 -> 114 ms, 6 -> 109 ms,
// 8 -> 109 ms, 10 -> 116 ms, 12 -> 129 ms; v7 (warp-uniform chains): 5 -> 102.8, 6 -> 103.2, 7 -> 100.2, 8 -> 97.7,
// 9 -> 97.4, 10 -> 110.2, 12 -> 115.0, 16 -> 126.2 ms: 8 is the fastest up to noise. Ten or more CTAs per SM would also
// need more shared memory than the default carve-out offers (12.4 KB per CTA).
constexpr int K0_MIN_CTAS = 8;

__global__ void __launch_bounds__(32 * K0_WARPS, K0_MIN_CTAS) k0_parse_kernel(const k0::Tables* __restrict__ tables, const k0::Pic* __restrict__ pics,
                                                                             const k0::Sub* __restrict__ subs, const k0::Chain* __restrict__ chains,
                                                                             int nchains) {
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(tables);
    uint32_t* dst = reinterpret_cast<uint32_t*>(k0::k0_smem);
    for (int i = threadIdx.x; i < (int)(sizeof(k0::Tables) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  const int chain = blockIdx.x * K0_WARPS + warp;
  // ALL 32 lanes of the warp walk the chain's syntax with identical data (warp-uniform execution costs what one lane costs:
  // measured 112.6 ms with 32 lanes against 113.5 ms with one); the data-parallel parts of the parser — coefficient records,
  // map fills, context tables, K1 lists — are spread over the lanes (k0_core.cuh: K0_LANES / lane())
  if (chain >= nchains) return;
  const k0::Chain ch = chains[chain];
  k0::Parser ps;
  memset(&ps, 0, sizeof(ps));   // CuQpDeltaVal & co. are read even when the stream never codes them
  ps.wbase = (uint32_t)(k0::TABLE_BYTES + warp * k0::SCRATCH_BYTES);
#if defined(__CUDA_ARCH__)
  ps.cabac.ta = (uint32_t)__cvta_generic_to_shared(k0::k0_smem);
  ps.cabac.sa = ps.cabac.ta + ps.wbase;   // the Scratch starts with the decoder state
#endif
  ps.run_chain(pics, subs, ch.first_sub, ch.nsubs);
}

// Second, fully parallel half of K0: the neighbour availability masks of every block record (k0_core.cuh: finish_blk),
// one warp per CTB, the picture descriptor in shared memory.
__global__ void __launch_bounds__(256) k0_finish_kernel(const k0::Pic* __restrict__ pics) {
  __shared__ k0::Pic sp;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(pics + blockIdx.y);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&sp);
    for (int i = threadIdx.x; i < (int)(sizeof(k0::Pic) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int ctb = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (ctb >= sp.ctbs_w * sp.ctbs_h || *sp.error) return;
  k0::finish_ctb(sp, ctb, threadIdx.x & 31, 32);
}

void launch_k0_finish(const k0::Pic* pics, int npics, int max_ctbs, cudaStream_t stream) {
  if (npics <= 0 || max_ctbs <= 0) return;
  static_assert(sizeof(k0::Pic) % 4 == 0, "descriptor is copied word-wise");
  k0_finish_kernel<<<dim3((unsigned)((max_ctbs + 7) / 8), (unsigned)npics), 256, 0, stream>>>(pics);
}

void launch_k0(const k0::Tables* tables, const k0::Pic* pics, const k0::Sub* subs, const k0::Chain* chains, int nchains,
               cudaStream_t stream) {
  if (nchains <= 0) return;
  static_assert(sizeof(k0::Tables) % 4 == 0, "tables are copied word-wise");
  const int smem = k0::TABLE_BYTES + K0_WARPS * k0::SCRATCH_BYTES;
  const int grid = (nchains + K0_WARPS - 1) / K0_WARPS;
  k0_parse_kernel<<<grid, 32 * K0_WARPS, smem, stream>>>(tables, pics, subs, chains, nchains);
}

}  // namespace hc
