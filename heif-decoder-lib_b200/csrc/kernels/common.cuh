// common.cuh — shared definitions for the sm_100a reconstruction kernels.
#pragma once
#include <cstdint>
#include "../../../include/heifcuda_records.h"

#if defined(__CUDACC__)
#define HC_HD __host__ __device__ __forceinline__
#define HC_D __device__ __forceinline__
#else
#define HC_HD inline
#define HC_D inline
#endif

namespace hc {

HC_HD int clip3i(int lo, int hi, int v) { return v < lo ? lo : (v > hi ? hi : v); }
HC_HD int clip_bd(int v, int bd) { return clip3i(0, (1 << bd) - 1, v); }
HC_HD int iabs(int v) { return v < 0 ? -v : v; }
HC_HD int sat16(int v) { return clip3i(-32768, 32767, v); }

// Device-side view of one uploaded batch. All pointers are device pointers.
struct BatchView {
  const hc_pic* pics;
  const hc_ctu* ctus;
  const hc_blk* blks;
  const hc_tb* tbs;
  const hc_coeff* coeffs;
  const uint8_t* edge_map;
  const int8_t* qp_map;
  const uint8_t* scaling;
  int16_t* resid;          // residual buffer (K1 output, K2 input)
  uint8_t* planes;         // plane pool base: hc_pic::rec_off / dst_off are byte offsets from here
  int npics;
  int flags;               // HC_VIEW_*
};
constexpr int HC_VIEW_NO_SAO = 1;  // K4 only crops + pastes (parity tests of the earlier stages)

// One wavefront task of K2: a CTB row of one colour component of one picture.
struct RowTask {
  uint32_t pic;
  uint16_t row;
  uint8_t comp;
  uint8_t pad;
  int32_t dep;   // task index of the row above (same picture / component), -1 for row 0
  uint32_t smem_off;  // byte offset of this warp's slice of the CTA's dynamic shared memory
};
// The row tasks one warp of K2 runs one after the other (a CTA is three warps: two luma-class rows and one list of up to
// four subsampled chroma rows; see k2_intra_lists_kernel)
struct WarpWork {
  uint32_t task[4];
  uint32_t n;
};

#if defined(__CUDACC__)
// L2-coherent loads: neighbour samples and progress counters are produced by other SMs while
// this kernel runs, so they must not be served from a stale L1 line.
HC_D unsigned ld_cg_u8(const uint8_t* p) {
  unsigned v;
  asm volatile("ld.global.cg.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
HC_D unsigned ld_cg_u16(const uint16_t* p) {
  unsigned short v;
  asm volatile("ld.global.cg.u16 %0, [%1];" : "=h"(v) : "l"(p) : "memory");
  return v;
}
HC_D unsigned ld_sample_cg(const uint8_t* p) { return ld_cg_u8(p); }
HC_D unsigned ld_sample_cg(const uint16_t* p) { return ld_cg_u16(p); }
HC_D int ld_acquire_s32(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
HC_D void st_release_s32(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
#endif

}  // namespace hc
