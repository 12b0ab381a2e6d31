// k2_intra.cu — K2: intra prediction + residual add as a CTB wavefront over every picture of a
// batch at once, with the CTB under reconstruction resident in shared memory.
//
// Replaces decode_intra_prediction (intrapred.cc:337-362: border gather intrapred.h:838-984,
// reference smoothing :192-266, planar :269-293, DC :296-330, angular :338-441) and the
// "+= residual, clip" tail of the reference's transform functions.
//
// Parallel structure (nothing like the reference's per-TU call chain):
//   * one warp owns one CTB row of one colour component of one picture (RowTask); luma, Cb and Cr
//     are independent dependency chains and run concurrently;
//   * a row may process CTB x once the row above has finished CTB x+1 (left / top-left / top /
//     top-right neighbours): the classic 2-CTB wavefront, tracked with one acquire/release
//     counter per task in global memory;
//   * tasks are ordered row-major across ALL pictures, so every picture / grid tile of the batch
//     advances its own wavefront simultaneously and a task only ever waits on a task with a
//     smaller index (scheduled no later than itself -> forward progress);
//   * the block-to-block dependency chain inside a CTB never leaves the SM: the CTB's samples live
//     in a per-warp shared-memory tile (+ top halo row fetched once per CTB through L2, + left
//     halo column kept from the previous CTB); the finished CTB is written to HBM once, coalesced;
//   * block records are read 32 at a time (one 16-byte record per lane, broadcast by shuffle) two
//     batches ahead; the residuals of the small blocks of the NEXT batch are staged in shared
//     memory by TMA bulk copies (cp.async.bulk + mbarrier, one copy per block issued by the lane
//     that holds its record) while the current batch is being predicted; 16x16 / 32x32 blocks read
//     their residuals straight from global memory (L2-prefetched), their latency amortised over
//     >= 256 samples;
//   * slice/tile/z-scan availability was resolved by the host (hc_blk::avail_*), so the kernel
//     carries no bitstream-structure logic; substitution of unavailable reference samples is
//     folded into the gather (the substitute is itself a reconstructed sample of the tile).
//
// Bound: instruction issue / dependency latency of the per-block chain, not HBM; see DESIGN.md.
#include <atomic>
#include "launch.h"

namespace hc {

__device__ __constant__ int8_t c_intra_angle[35] = {0,   0,   32,  26,  21,  17,  13,  9,   5,  2,  0,  -2,
                                                    -5,  -9,  -13, -17, -21, -26, -32, -26, -21, -17, -13, -9,
                                                    -5,  -2,  0,   2,   5,   9,   13,  17,  21,  26,  32};
__device__ __constant__ int16_t c_inv_angle[15] = {-4096, -1638, -910, -630, -482, -390, -315, -256,
                                                   -315,  -390,  -482, -630, -910, -1638, -4096};

// ---- per-warp shared-memory layout (bytes; see k2_task_smem_bytes) ---------------------------------
// [0,16)    two mbarriers
// [16,..)   refA[REF_LEN] int16, refB[REF_LEN] int16      reference samples p[-64..64] (index + REF_OFF)
// then      corner (16 B slot), top[2*cw] Pixel, 16 B slot, tile[ch][cw*ps+4 bytes] (left halo in the row padding),
//           stage[2][cap] int16
constexpr int REF_OFF = 66;
constexpr int REF_LEN = 136;
constexpr int K2_REF_BYTES = 2 * REF_LEN * 2;   // 544
constexpr int K2_STAGE_MAX_ELEMS = 2048;        // 32 blocks of 8x8

HC_HD int k2_align16(int v) { return (v + 15) & ~15; }
HC_HD int k2_stage_elems(int cw, int ch) { return cw * ch < K2_STAGE_MAX_ELEMS ? cw * ch : K2_STAGE_MAX_ELEMS; }

int k2_task_smem_bytes(int ctb_w, int ctb_h, int pixel_bytes) {
  int o = 16 + K2_REF_BYTES;
  o += 16 + k2_align16(2 * ctb_w * pixel_bytes);                  // corner slot + top row
  o += 16 + k2_align16(ctb_h * (ctb_w * pixel_bytes + 4));        // left-halo slot of row 0 + tile rows
  o += 2 * k2_stage_elems(ctb_w, ctb_h) * 2;                      // two residual stage buffers
  return k2_align16(o);
}

// ---- mbarrier / TMA bulk copy primitives -------------------------------------------------------------
HC_D uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
HC_D void mbar_init(uint32_t bar, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
HC_D void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
HC_D void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
HC_D void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
               "r"(bar)
               : "memory");
}
HC_D void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
HC_D void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
HC_D void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
HC_D uint2 ld_cg_v2(const void* p) {
  uint2 v;
  asm volatile("ld.global.cg.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}

// Per-warp geometry of the shared-memory CTB tile. All *_off values are byte offsets from the
// warp's shared-memory base `sm`.
//   top row  : sample (x,-1) at top_off + x*PS, x = -1 (corner) .. 2*cw-1
//   tile     : sample (x,y)  at tile_off + y*pitch + x*PS; the left halo column x = -1 lives in the
//              4 padding bytes that end the previous row (pitch = cw*PS + 4)
struct Geo {
  uint8_t* sm;
  int16_t* refA;
  int16_t* refB;
  int top_off, tile_off, pitch;
  int bit_depth;
  bool strong;   // strong_intra_smoothing applies to this component (luma, sps flag)
};

// Per-block parameters, computed once per batch by the lane that holds the record (32 blocks in
// parallel) and broadcast by shuffle in the block loop:
//   w0 : left_off | top_off << 16     byte offsets of ref sample (-1, 0) resp. corner (-1,-1) of the block
//   w1 : store_off | mode << 16 | (log2-2) << 22 | BP_* bits
//   w2 : lo & 0xff | (hi & 0xff) << 8 | staged residual byte offset << 16     (lo..hi: the available run)
//   w3 : avail_left | avail_top << 16                        (general substitution only)
//   w4 : int16 index in the residual buffer                  (16x16 / 32x32 blocks only)
constexpr uint32_t BP_HAS_RES = 1u << 24, BP_PCM = 1u << 25, BP_FILT = 1u << 26, BP_EDGE = 1u << 27, BP_NOEDGEFLT = 1u << 28,
                   BP_NONE_AVAIL = 1u << 29, BP_GENERAL = 1u << 30, BP_TL = 1u << 31;

template <typename Pixel>
HC_D int ld_px(const uint8_t* sm, int off) { return (int)*reinterpret_cast<const Pixel*>(sm + off); }

// slot (4-sample unit in scan order) -> first / last reference index it covers
HC_D int slot_first(int s, int nu) { return s < nu ? -(4 * (nu - 1 - s) + 4) : (s == nu ? 0 : 4 * (s - nu - 1) + 1); }
HC_D int slot_last(int s, int nu) { return s < nu ? -(4 * (nu - 1 - s) + 1) : (s == nu ? 0 : 4 * (s - nu - 1) + 4); }

// One prediction block. All 32 lanes run every statement (no divergent lane guards): lanes beyond
// the block's sample count recompute a sample another lane owns and store the identical value.
template <typename Pixel, int LOG2>
__device__ __forceinline__ void process_block(const Geo& g, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, const int16_t* __restrict__ res,
                                              int lane) {
  constexpr int PS = (int)sizeof(Pixel);
  constexpr int nT = 1 << LOG2, nref = 4 * nT + 1, nu = nT >> 1;
  constexpr int NS = nT * nT;                       // samples
  constexpr int ITER = NS >= 32 ? NS / 32 : 1;      // sample passes of the warp
  constexpr int RPI = 32 >> LOG2;                   // block rows covered per pass (8x8: 4, 16x16: 2, 32x32: 1)
  constexpr int GIT = (nref + 31) / 32;             // gather passes
  const int store_off = w1 & 0xffff, mode = (w1 >> 16) & 63;
  const int pitch = g.pitch;
  const int maxv = (1 << g.bit_depth) - 1;
  // this lane's sample of pass 0: s0 = lane (4x4: lane & 15), x = s0 % nT, y = s0 / nT
  const int s0 = NS >= 32 ? lane : (lane & (NS - 1));
  const int x = s0 & (nT - 1), yb = s0 >> LOG2;
  uint8_t* out = g.sm + store_off + yb * pitch + x * PS;

  if (w1 & BP_PCM) {
#pragma unroll 1
    for (int j = 0; j < ITER; j++) *reinterpret_cast<Pixel*>(out + j * RPI * pitch) = (Pixel)(uint16_t)res[s0 + 32 * j];
    __syncwarp();
    return;
  }
  // The residual add is the last step of the block, but its operands do not depend on the prediction: ncu put 27 % of the
  // kernel's stall samples on the `v + res[...]` lines (the load is issued behind the warp barriers of the gather / filter
  // phases and every sample pass waits for it). Small blocks (staged in shared memory) read theirs now, into registers;
  // 16x16 / 32x32 blocks (read from global memory, one 64-byte row group per pass) pull their lines into L1 now.
  const bool has_res = w1 & BP_HAS_RES;
  int rpre0 = 0, rpre1 = 0;
  if (has_res) {
    if (LOG2 <= 3) {
      rpre0 = res[s0];
      if (ITER == 2) rpre1 = res[s0 + 32];
    } else if (lane * 128 < NS * 2 + 128) {
      prefetch_l1(reinterpret_cast<const char*>(res) + lane * 128);
    }
  }
  auto residual = [&](int j) -> int { return LOG2 <= 3 ? (j == 0 ? rpre0 : rpre1) : (int)res[s0 + 32 * j]; };

  // ---- 1. gather reference samples p[-2nT..2nT]; substitution folded in (intrapred.h:838-984) ----
  const int left_off = w0 & 0xffff, top_off = w0 >> 16;
  if (!(w1 & (BP_NONE_AVAIL | BP_GENERAL))) {
    // the available units form one run in scan order: unavailable samples take the nearest end of it
    const int lo = (int)(int8_t)(w2 & 0xff), hi = (int)(int8_t)((w2 >> 8) & 0xff);
#pragma unroll
    for (int j = 0; j < GIT; j++) {
      const int idx = min(lane + 32 * j, nref - 1);
      const int i = idx - 2 * nT;
      const int src = min(max(i, lo), hi);
      const int off = src < 0 ? left_off - (src + 1) * pitch : top_off + src * PS;
      g.refA[REF_OFF + i] = (int16_t)ld_px<Pixel>(g.sm, off);
    }
  } else if (w1 & BP_NONE_AVAIL) {
#pragma unroll
    for (int j = 0; j < GIT; j++) g.refA[REF_OFF + min(lane + 32 * j, nref - 1) - 2 * nT] = (int16_t)(1 << (g.bit_depth - 1));
  } else {
    // general case (slice / tile corners): nearest available unit before, else the first available
    const unsigned availL = w3 & 0xffff, availT = w3 >> 16;
    const unsigned long long tl = (w1 & BP_TL) ? 1ull : 0ull;
    unsigned long long A;
    if (nu == 16) A = (unsigned long long)(__brev(availL) >> 16) | (tl << 16) | ((unsigned long long)availT << 17);
    else A = (unsigned long long)(__brev(availL) >> (32 - nu)) | (tl << nu) | ((unsigned long long)(availT & ((1u << nu) - 1u)) << (nu + 1));
    for (int idx = lane; idx < nref; idx += 32) {
      const int i = idx - 2 * nT;
      const int s = i < 0 ? nu - 1 - ((-i - 1) >> 2) : (i == 0 ? nu : nu + 1 + ((i - 1) >> 2));
      int src = i;
      if (!((A >> s) & 1)) {
        const unsigned long long below = A & ((1ull << s) - 1ull);
        if (below) src = slot_last(63 - __clzll((long long)below), nu);
        else src = slot_first(__ffsll((long long)A) - 1, nu);
      }
      const int off = src < 0 ? left_off - (src + 1) * pitch : top_off + src * PS;
      g.refA[REF_OFF + i] = (int16_t)ld_px<Pixel>(g.sm, off);
    }
  }
  __syncwarp();

  // ---- 2. reference smoothing (intrapred.h:192-266); the mode/size rule was evaluated in the pre-pass ----
  const int16_t* p = g.refA + REF_OFF;
  if (LOG2 > 2 && (w1 & BP_FILT)) {
    bool bi = false;
    if (LOG2 == 5 && g.strong) {
      const int thr = 1 << (g.bit_depth - 5);
      bi = iabs(p[0] + p[64] - 2 * p[32]) < thr && iabs(p[0] + p[-64] - 2 * p[-32]) < thr;
    }
    int16_t* q = g.refB + REF_OFF;
#pragma unroll
    for (int j = 0; j < GIT; j++) {
      const int idx = min(lane + 32 * j, nref - 1);
      const int i = idx - 2 * nT;
      int v;
      if (i == -2 * nT || i == 2 * nT) v = p[i];
      else if (LOG2 == 5 && bi) {
        if (i == 0) v = p[0];
        else if (i < 0) v = p[0] + (((-i) * (p[-64] - p[0]) + 32) >> 6);
        else v = p[0] + ((i * (p[64] - p[0]) + 32) >> 6);
      } else {
        v = (p[i + 1] + 2 * p[i] + p[i - 1] + 2) >> 2;
      }
      q[i] = (int16_t)v;
    }
    __syncwarp();
    p = q;
  }

  // ---- 3. prediction + residual + store into the tile --------------------------------------------
  const bool edge_ok = w1 & BP_EDGE;
  if (mode == 0) {
    const int tr = p[1 + nT], bl = p[-1 - nT];
    const int top = p[1 + x], hx = (x + 1) * tr + nT;
#pragma unroll 1
    for (int j = 0; j < ITER; j++) {
      const int y = yb + j * RPI;
      int v = ((nT - 1 - x) * p[-1 - y] + hx + (nT - 1 - y) * top + (y + 1) * bl) >> (LOG2 + 1);
      if (has_res) v = clip3i(0, maxv, v + residual(j));
      *reinterpret_cast<Pixel*>(out + j * RPI * pitch) = (Pixel)v;
    }
  } else if (mode == 1) {
    const int ln = lane & (nT - 1);
    int sum = p[ln + 1] + p[-ln - 1];
#pragma unroll
    for (int o = nT >> 1; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const int dc = (sum + nT) >> (LOG2 + 1);
    const int top = (p[x + 1] + 3 * dc + 2) >> 2;
#pragma unroll 1
    for (int j = 0; j < ITER; j++) {
      const int y = yb + j * RPI;
      int v = dc;
      if (edge_ok) {
        if (y == 0) v = x == 0 ? (p[-1] + 2 * dc + p[1] + 2) >> 2 : top;
        else if (x == 0) v = (p[-y - 1] + 3 * dc + 2) >> 2;
      }
      if (has_res) v = clip3i(0, maxv, v + residual(j));
      *reinterpret_cast<Pixel*>(out + j * RPI * pitch) = (Pixel)v;
    }
  } else {
    // vertical modes walk the top row (ref[k] = p[k]); horizontal modes the left column (ref[k] = p[-k]);
    // u runs along the reference, w away from it
    const int angle = c_intra_angle[mode];
    const bool vertical = mode >= 18;
    const int sgn = vertical ? 1 : -1;
    if (angle == 0) {
      // modes 10 / 26: copy the reference, optional boundary filter on the first row / column
      const bool edge_flt = edge_ok && !(w1 & BP_NOEDGEFLT);
      const int p0 = p[0], p1 = p[sgn];
#pragma unroll 1
      for (int j = 0; j < ITER; j++) {
        const int y = yb + j * RPI;
        const int u = vertical ? x : y, w = vertical ? y : x;
        int v = p[sgn * (u + 1)];
        if (edge_flt && u == 0) v = clip3i(0, maxv, p1 + ((p[-sgn * (1 + w)] - p0) >> 1));
        if (has_res) v = clip3i(0, maxv, v + residual(j));
        *reinterpret_cast<Pixel*>(out + j * RPI * pitch) = (Pixel)v;
      }
    } else if (angle > 0) {
      // the reference index never goes negative; (32a + 16) >> 5 == a covers iFact == 0
#pragma unroll 1
      for (int j = 0; j < ITER; j++) {
        const int y = yb + j * RPI;
        const int u = vertical ? x : y, w = vertical ? y : x;
        const int t = (w + 1) * angle;
        const int k0 = u + (t >> 5) + 1, f = t & 31;
        int v = ((32 - f) * p[sgn * k0] + f * p[sgn * (k0 + 1)] + 16) >> 5;
        if (has_res) v = clip3i(0, maxv, v + residual(j));
        *reinterpret_cast<Pixel*>(out + j * RPI * pitch) = (Pixel)v;
      }
    } else {
      // negative angles: indices below zero project onto the other reference through the inverse angle
      const int inv = c_inv_angle[mode - 11];
#pragma unroll 1
      for (int j = 0; j < ITER; j++) {
        const int y = yb + j * RPI;
        const int u = vertical ? x : y, w = vertical ? y : x;
        const int t = (w + 1) * angle;
        const int k0 = u + (t >> 5) + 1, k1 = k0 + 1, f = t & 31;
        const int i0 = k0 >= 0 ? sgn * k0 : -sgn * ((k0 * inv + 128) >> 8);
        const int i1 = k1 >= 0 ? sgn * k1 : -sgn * ((k1 * inv + 128) >> 8);
        int v = ((32 - f) * p[i0] + f * p[i1] + 16) >> 5;
        if (has_res) v = clip3i(0, maxv, v + residual(j));
        *reinterpret_cast<Pixel*>(out + j * RPI * pitch) = (Pixel)v;
      }
    }
  }
  // make the block visible to the lanes that gather the next block's references
  __syncwarp();
}

// One batch = up to 32 consecutive block records of one CTB (lane k holds record k).
struct Batch {
  int cx;      // CTB column
  int j;       // first record inside the CTB's list
  int n;       // records in this batch
  int count;   // records in the CTB's list
};

template <typename Pixel>
__device__ void run_row(const BatchView& bv, const hc_pic& pic, const RowTask task, int* progress, int my_index, uint8_t* smem, int lane) {
  constexpr int PS = (int)sizeof(Pixel);
  const int comp = task.comp;
  const int subw = (comp && (pic.chroma_format == 1 || pic.chroma_format == 2)) ? 1 : 0;
  const int subh = (comp && pic.chroma_format == 1) ? 1 : 0;
  const int cw = (1 << pic.log2_ctb) >> subw, ch = (1 << pic.log2_ctb) >> subh;
  const int plane_w = pic.width >> subw, plane_h = pic.height >> subh;
  Pixel* plane = reinterpret_cast<Pixel*>(bv.planes + pic.rec_off[comp]);
  const int stride = (int)pic.rec_stride[comp];
  const int16_t* resid = bv.resid + pic.resid_base;
  const uint4* blks = reinterpret_cast<const uint4*>(bv.blks + pic.blk_base);
  const hc_ctu* ctus = bv.ctus + pic.ctu_base + (size_t)task.row * pic.ctbs_w;
  const int W = pic.ctbs_w;
  const int y0 = task.row * ch;
  const int pic_flags = pic.flags, chroma_format = pic.chroma_format;

  // ---- carve the per-warp shared memory (k2_task_smem_bytes) ----
  Geo g;
  g.sm = smem;
  const uint32_t bar0 = smem_u32(smem), bar1 = bar0 + 8;
  int o = 16;
  g.refA = reinterpret_cast<int16_t*>(smem + o);
  g.refB = g.refA + REF_LEN;
  o += K2_REF_BYTES;
  g.top_off = o + 16;                      // corner at top_off - PS
  o += 16 + k2_align16(2 * cw * PS);
  g.tile_off = o + 16;                     // left halo of row 0 at tile_off - PS
  g.pitch = cw * PS + 4;
  o += 16 + k2_align16(ch * g.pitch);
  const int cap = k2_stage_elems(cw, ch);
  const int stage_off0 = o, stage_off1 = o + cap * 2;
  g.bit_depth = comp == 0 ? pic.bit_depth_y : pic.bit_depth_c;
  g.strong = (pic_flags & HC_PIC_STRONG_INTRA) && comp == 0;

  if (lane == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_proxy_async();
  __syncwarp();

  // CTB -> (first record, record count) of this component: lane k caches CTB k (rows are short: 8 CTBs
  // for a 512 tile, 30 for 1080p); wider rows fall back to a global load. Both are warp-uniform calls.
  const uint32_t my_first = lane < W ? ctus[lane].blk_first[comp] : 0u;
  const int my_count = lane < W ? (int)ctus[lane].blk_count[comp] : 0;
  auto ctb_first = [&](int cx) -> uint32_t {
    const uint32_t v = __shfl_sync(0xffffffffu, my_first, cx & 31);
    return cx < 32 ? v : ctus[cx].blk_first[comp];
  };
  auto ctb_count = [&](int cx) -> int {
    const int v = __shfl_sync(0xffffffffu, my_count, cx & 31);
    return cx < 32 ? v : (int)ctus[cx].blk_count[comp];
  };

  auto first_batch = [&]() -> Batch {
    Batch b;
    b.cx = 0; b.j = 0;
    b.count = ctb_count(0);
    b.n = b.count < 32 ? b.count : 32;
    return b;
  };
  auto next_batch = [&](const Batch& a) -> Batch {   // a.cx == W marks the end
    Batch b = a;
    if (a.cx >= W) return b;
    b.j = a.j + 32;
    if (b.j >= a.count) {
      b.cx = a.cx + 1;
      b.j = 0;
      b.count = b.cx < W ? ctb_count(b.cx) : 0;
    }
    b.n = b.count - b.j < 32 ? b.count - b.j : 32;
    return b;
  };
  auto load_recs = [&](const Batch& b) -> uint4 {
    uint4 r = make_uint4(0, 0, 0, 0);
    if (b.cx >= W) return r;                      // warp-uniform
    const uint32_t first = ctb_first(b.cx);
    if (lane < b.n) r = __ldg(blks + first + b.j + lane);
    return r;
  };
  // residual elements of a record that are staged in shared memory (small blocks)
  auto staged_elems = [&](const Batch& b, const uint4& r) -> int {
    if (b.cx >= W || lane >= b.n) return 0;
    const int log2 = r.y & 0xff, flags = (r.y >> 16) & 0xff;
    if (!(flags & (HC_BLK_HAS_RESID | HC_BLK_PCM))) return 0;
    return log2 <= 3 ? 1 << (2 * log2) : 0;
  };
  // issues the staging copies of batch b into stage buffer `buf`; returns this lane's element offset
  // inside the buffer and the batch total through `total`
  auto issue_stage = [&](const Batch& b, const uint4& r, int buf, int& total) -> int {
    const int sz = staged_elems(b, r);
    int incl = sz;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    total = __shfl_sync(0xffffffffu, incl, 31);
    const int off = incl - sz;
    const uint32_t bar = buf ? bar1 : bar0;
    if (total > 0) {
      if (lane == 0) mbar_expect_tx(bar, (uint32_t)total * 2u);
      __syncwarp();
      if (sz > 0) bulk_g2s(bar0 + (uint32_t)(buf ? stage_off1 : stage_off0) + (uint32_t)off * 2u, resid + r.w, (uint32_t)sz * 2u, bar);
    }
    // large blocks: pull their residual lines into L2 ahead of use
    if (b.cx < W && lane < b.n) {
      const int log2 = r.y & 0xff, flags = (r.y >> 16) & 0xff;
      if (log2 >= 4 && (flags & (HC_BLK_HAS_RESID | HC_BLK_PCM))) {
        const char* src = reinterpret_cast<const char*>(resid + r.w);
        const int bytes = 2 << (2 * log2);
        for (int k = 0; k < bytes; k += 128) prefetch_l2(src + k);
      }
    }
    return off;
  };
  // pre-pass: this lane's record -> the block parameter words (see above)
  auto block_params = [&](const Batch& b, const uint4& r, int stage_off, int off_elems, uint32_t& w0, uint32_t& w1, uint32_t& w2, uint32_t& w4) {
    const int log2 = r.y & 0xff, nT = 1 << log2, mode = (r.y >> 8) & 0xff, flags = (r.y >> 16) & 0xff;
    const int lx = (int)(r.x & 0xffff) - b.cx * cw, ly = (int)(r.x >> 16) - y0;
    const int left_off = g.tile_off + ly * g.pitch + (lx - 1) * PS;
    const int top_off = (ly == 0 ? g.top_off : g.tile_off + (ly - 1) * g.pitch) + (lx - 1) * PS;
    w0 = (uint32_t)left_off | ((uint32_t)top_off << 16);
    const int store_off = g.tile_off + ly * g.pitch + lx * PS;
    uint32_t bits = 0;
    if (flags & HC_BLK_HAS_RESID) bits |= BP_HAS_RES;
    if (flags & HC_BLK_PCM) bits |= BP_PCM;
    if (flags & HC_BLK_AVAIL_TL) bits |= BP_TL;
    if (flags & HC_BLK_NO_EDGE_FLT) bits |= BP_NOEDGEFLT;
    if (comp == 0 && nT < 32) bits |= BP_EDGE;
    if (!(pic_flags & HC_PIC_NO_INTRA_SMOOTH) && (comp == 0 || chroma_format == 3) && mode != 1 && nT != 4) {
      const int d1 = iabs(mode - 26), d2 = iabs(mode - 10);
      const int minDist = d1 < d2 ? d1 : d2;
      if (nT == 8 ? minDist > 7 : nT == 16 ? minDist > 1 : minDist > 0) bits |= BP_FILT;
    }
    // availability in scan order: left units bottom->top, top-left, top units left->right
    const unsigned availL = r.z & 0xffff, availT = r.z >> 16;
    const int nu = nT >> 1;
    const unsigned long long tl = (flags & HC_BLK_AVAIL_TL) ? 1ull : 0ull;
    unsigned long long A;
    if (nu == 16) A = (unsigned long long)(__brev(availL) >> 16) | (tl << 16) | ((unsigned long long)availT << 17);
    else A = (unsigned long long)(__brev(availL) >> (32 - nu)) | (tl << nu) | ((unsigned long long)(availT & ((1u << nu) - 1u)) << (nu + 1));
    int lo = 0, hi = 0;
    if (A == 0) bits |= BP_NONE_AVAIL;
    else {
      const int fs = __ffsll((long long)A) - 1, ls = 63 - __clzll((long long)A);
      const unsigned long long run = A >> fs;
      if (run & (run + 1)) bits |= BP_GENERAL;
      lo = slot_first(fs, nu);
      hi = slot_last(ls, nu);
    }
    w1 = (uint32_t)store_off | ((uint32_t)mode << 16) | ((uint32_t)(log2 - 2) << 22) | bits;
    w2 = (uint32_t)(lo & 0xff) | ((uint32_t)(hi & 0xff) << 8) | ((uint32_t)(stage_off + off_elems * 2) << 16);
    w4 = r.w;
  };

  // ---- software pipeline: records two batches ahead, staged residuals one batch ahead ----
  Batch cur = first_batch();
  Batch nxt = next_batch(cur);
  uint4 rec_cur = load_recs(cur);
  uint4 rec_nxt = load_recs(nxt);
  int total_cur = 0, total_nxt = 0;
  int off_cur = issue_stage(cur, rec_cur, 0, total_cur);
  int off_nxt = 0;
  uint32_t phase0 = 0, phase1 = 0;
  int buf = 0;

  while (cur.cx < W) {
    const Batch nn = next_batch(nxt);
    const uint4 rec_nn = load_recs(nn);              // in flight during this whole batch
    // the other stage buffer was last read by the previous batch (its trailing __syncwarp is behind us)
    fence_proxy_async();
    off_nxt = issue_stage(nxt, rec_nxt, buf ^ 1, total_nxt);

    uint32_t w0, w1, w2, w4;
    block_params(cur, rec_cur, buf ? stage_off1 : stage_off0, off_cur, w0, w1, w2, w4);
    const uint32_t w3 = rec_cur.z;

    const int cx = cur.cx;
    const int x0 = cx * cw;
    if (cur.j == 0) {
      // ---- CTB prologue: left halo from the previous CTB, wavefront wait, top halo through L2 ----
      if (cx > 0)
        for (int r = lane; r < ch; r += 32)
          *reinterpret_cast<Pixel*>(smem + g.tile_off + r * g.pitch - PS) = *reinterpret_cast<const Pixel*>(smem + g.tile_off + r * g.pitch + (cw - 1) * PS);
      if (task.dep >= 0) {
        const int need = cx + 2 < W ? cx + 2 : W;
        if (lane == 0)
          while (ld_acquire_s32(progress + task.dep) < need) __nanosleep(100);
        __syncwarp();
        const Pixel* above = plane + (size_t)(y0 - 1) * stride + x0;
        const int units = (2 * cw * PS) >> 3;       // 8-byte units, <= 32
        if (lane < units) reinterpret_cast<uint2*>(smem + g.top_off)[lane] = ld_cg_v2(reinterpret_cast<const uint8_t*>(above) + lane * 8);
        if (lane == 31 && cx > 0) *reinterpret_cast<Pixel*>(smem + g.top_off - PS) = (Pixel)ld_sample_cg(above - 1);
      }
      __syncwarp();
    }

    // ---- the blocks of this batch ----
    if (total_cur > 0) {
      mbar_wait(buf ? bar1 : bar0, buf ? phase1 : phase0);
      if (buf) phase1 ^= 1; else phase0 ^= 1;
    }
    // the parameter words of block k+1 are broadcast while block k is being predicted
    uint32_t n0 = __shfl_sync(0xffffffffu, w0, 0), n1 = __shfl_sync(0xffffffffu, w1, 0), n2 = __shfl_sync(0xffffffffu, w2, 0);
    for (int k = 0; k < cur.n; k++) {
      const uint32_t b0 = n0, b1 = n1, b2 = n2;
      const int kn = k + 1 < cur.n ? k + 1 : k;
      n0 = __shfl_sync(0xffffffffu, w0, kn); n1 = __shfl_sync(0xffffffffu, w1, kn); n2 = __shfl_sync(0xffffffffu, w2, kn);
      uint32_t b3 = 0;
      if (b1 & BP_GENERAL) b3 = __shfl_sync(0xffffffffu, w3, k);   // warp-uniform branch
      const int lg = (b1 >> 22) & 3;
      if (lg == 0) process_block<Pixel, 2>(g, b0, b1, b2, b3, reinterpret_cast<const int16_t*>(smem + (b2 >> 16)), lane);
      else if (lg == 1) process_block<Pixel, 3>(g, b0, b1, b2, b3, reinterpret_cast<const int16_t*>(smem + (b2 >> 16)), lane);
      else {
        const uint32_t b4 = __shfl_sync(0xffffffffu, w4, k);
        if (lg == 2) process_block<Pixel, 4>(g, b0, b1, b2, b3, resid + b4, lane);
        else process_block<Pixel, 5>(g, b0, b1, b2, b3, resid + b4, lane);
      }
    }

    if (cur.j + cur.n >= cur.count) {
      // ---- CTB epilogue: tile -> HBM (4-byte units), publish progress ----
      const int w = min(cw, plane_w - x0), h = min(ch, plane_h - y0);
      const int upr = (w * PS) >> 2;   // coded plane widths are multiples of 4 samples
      uint8_t* dst = reinterpret_cast<uint8_t*>(plane + (size_t)y0 * stride + x0);
      const size_t dpitch = (size_t)stride * PS;
      if (upr == 16) {
        for (int u = lane; u < 16 * h; u += 32) {
          const int r = u >> 4, q = u & 15;
          *reinterpret_cast<uint32_t*>(dst + r * dpitch + q * 4) = *reinterpret_cast<const uint32_t*>(smem + g.tile_off + r * g.pitch + q * 4);
        }
      } else {
        for (int u = lane; u < upr * h; u += 32) {
          const int r = u / upr, q = u - r * upr;
          *reinterpret_cast<uint32_t*>(dst + r * dpitch + q * 4) = *reinterpret_cast<const uint32_t*>(smem + g.tile_off + r * g.pitch + q * 4);
        }
      }
      __threadfence();
      __syncwarp();
      if (lane == 0) st_release_s32(progress + my_index, cx + 1);
    }

    cur = nxt; nxt = nn;
    rec_cur = rec_nxt; rec_nxt = rec_nn;
    off_cur = off_nxt; total_cur = total_nxt;
    buf ^= 1;
  }
  // a warp may run several chroma rows one after the other in the same shared memory (k2_intra_lists_kernel): the
  // mbarriers are re-initialised by the next row, which requires them to be invalidated first
  __syncwarp();
  if (lane == 0) {
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar0) : "memory");
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar1) : "memory");
  }
  __syncwarp();
}

// A CTA is three warps, each running the row tasks of its list one after the other. The host builds the lists (engine.cu):
// a luma-class row takes a warp of its own, and up to four units of subsampled chroma rows (a 4:2:0 row is one unit, a
// 4:2:2 row two) share the third warp, since a luma row takes about as long as the four chroma rows of 4:2:0 together.
// Lists are filled in task order, a luma-class list holds one task and all chroma rows of a CTA share one warp, so a task
// only waits for a task in an earlier CTA, in another warp's single-task list, or earlier in its own list: forward progress
// holds as for one task per warp.
__global__ void __launch_bounds__(96, 6)
k2_intra_lists_kernel(BatchView bv, const RowTask* __restrict__ tasks, const WarpWork* __restrict__ work, int* progress) {
  extern __shared__ __align__(16) uint8_t k2_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const WarpWork ww = work[blockIdx.x * 3 + warp];
#pragma unroll 1
  for (uint32_t k = 0; k < ww.n; k++) {
    const int index = (int)ww.task[k];
    const RowTask task = tasks[index];
    const hc_pic& pic = bv.pics[task.pic];
    if (pic.bit_depth_y == 8 && pic.bit_depth_c == 8)
      run_row<uint8_t>(bv, pic, task, progress, index, k2_smem + task.smem_off, lane);
    else
      run_row<uint16_t>(bv, pic, task, progress, index, k2_smem + task.smem_off, lane);
    __syncwarp();
  }
}

void launch_k2(const BatchView& bv, const RowTask* tasks, const WarpWork* work, int nctas, int smem_bytes, int* progress, cudaStream_t stream) {
  if (nctas <= 0) return;
  // per device attribute: raised only when a launch needs more than any earlier one on this device (the plugin launches
  // K2 once per tile from many threads, and every CUDA call serialises on the context)
  {
    static std::atomic<int> max_set[64];
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (smem_bytes > max_set[dev].load(std::memory_order_relaxed)) {
      cudaFuncSetAttribute(k2_intra_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
      int cur = max_set[dev].load();
      while (smem_bytes > cur && !max_set[dev].compare_exchange_weak(cur, smem_bytes)) {}
    }
  }
  k2_intra_lists_kernel<<<nctas, 96, smem_bytes, stream>>>(bv, tasks, work, progress);
}

}  // namespace hc
