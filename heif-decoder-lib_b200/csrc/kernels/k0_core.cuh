// k0_core.cuh — K0: CABAC slice-data parse of HEVC intra pictures as host/device code.
//
// The same statements compile for the GPU (k0_parse.cu: one warp per substream chain, lane 0 walks the
// syntax) and for the CPU (capi: hc_parse_picture_k0, used by the tests to check this parser record by
// record against the reconstruction oracle before it ever runs on a GPU). It emits the records of
// include/heifcuda_records.h directly into device memory, so a picture parsed here needs no record upload at all:
// only its RBSP bytes (~0.2 B/px) cross PCIe.
//
// It replaces the same reference code as host/hevc_parse.cc — read_coding_tree_unit slice.cc:3026, read_sao :2886,
// read_coding_quadtree :4905, read_coding_unit :4568, read_transform_tree :4139, read_transform_unit :3867,
// residual_coding :3118, decode_quantization_parameters transform.cc:31 — and is written from the same text
// (H.265 7.3.8, 9.3, 8.4.2, 8.6.1, 6.4.1). Parallel structure the reference does not have:
//   * WPP pictures: one chain per CTB row; a row may parse CTB x once the row above has parsed CTB x+1
//     (context hand-over after the 2nd CTB, 9.3.2.2, plus the split/SAO-merge neighbours), tracked by the same
//     acquire/release counters K2 uses; all rows of all pictures of a batch are in flight;
//   * other pictures: one chain per picture (every slice segment in order).
// Not handled here (the host parser takes such pictures): HEVC tiles, pcm, transquant bypass,
// cu_chroma_qp_offset, persistent_rice_adaptation, slice segments that start inside a CTB row of a WPP picture.
//
// Layout of a K0 picture: every CTB owns fixed-capacity slices of the picture's blk / tb / coeff / residual
// regions (worst case of a CTB), so chains never allocate.
#pragma once
#include <cstring>
#include "common.cuh"

// functions that stay real calls: those with several call sites (the parser is instruction-fetch bound, so each has one
// copy), and the per-CTB / per-CU steps of the syntax walk
#if defined(__CUDACC__)
#define K0_FN __host__ __device__ __noinline__
#else
#define K0_FN __attribute__((noinline))
#endif
// Loops are not unrolled on the device: the parser is one thread per warp and bound by instruction fetch
// (ncu: "no_instruction" was the top stall of the running warps), so code size matters more than loop overhead.
#if defined(__CUDA_ARCH__)
#define K0_LOOP _Pragma("unroll 1")
#else
#define K0_LOOP
#endif

namespace hc {
namespace k0 {

// ---- context table layout: identical to host/hevc_cabac.h (CtxIdx) -------------------------------------------
enum : int {
  CX_SAO_MERGE = 0, CX_SAO_TYPE = 1, CX_SPLIT_CU = 2, CX_TQ_BYPASS = 5, CX_PART_MODE = 6, CX_PREV_INTRA_LUMA = 7,
  CX_INTRA_CHROMA = 8, CX_CBF_LUMA = 9, CX_CBF_CHROMA = 11, CX_SPLIT_TRANSFORM = 15, CX_CU_QP_DELTA = 18,
  CX_TSKIP = 20, CX_LAST_X = 22, CX_LAST_Y = 40, CX_CSBF = 58, CX_SIG = 62, CX_G1 = 106, CX_G2 = 130,
  CX_COUNT = 136   // the range-extension contexts behind G2 are never touched by the streams K0 accepts
};
constexpr int CTX_BYTES = 160;   // padded

// All read-only tables of the parser in one block (constant memory on the device).
struct alignas(16) Tables {
  uint32_t recip[256];             // floor(2^34 / (256 + i)) + 1: x / range == (x * recip) >> 34 for x < 2^25 (bypass strings)
  uint8_t range_lps[64][4];
  uint8_t next_state[128][2];      // [state][is_lps]
  uint8_t ctx_init[CX_COUNT];      // initValue per context (initType 0)
  uint8_t sig_b4[2][3][16];        // [chroma][scanIdx][k]
  uint8_t sig_sb[2][3][2][4][3][16];
  uint8_t scan_pos[3][16];         // 4x4 scan: x | y << 2
  uint8_t scan_sub[4][3][64];      // sub-block scan for log2 (0..3) grids: x | y << 3
  uint8_t inv_sub[4][3][64];       // [log2][scanIdx][x + (y << log2)] -> scan index
  uint8_t inv_pos[3][16];
  uint8_t mode422[35];
  int8_t qpc420[14];
};

struct Slice {
  int32_t segment_address, slice_addr_rs, slice_qp_y;
  uint32_t data_begin, data_end;     // slice_segment_data bytes inside Pic::bytes (data_end excludes the padding)
  int8_t cb_qp_offset, cr_qp_offset, beta_offset, tc_offset;
  uint8_t dependent, sao_luma, sao_chroma, deblocking_disabled, loop_filter_across_slices, pad[3];
};

struct Pic {
  // geometry / parameter sets (flattened Sps / Pps, host/hevc_params.h)
  int32_t W, H, w8, h8, w4, h4, ctbs_w, ctbs_h;
  int32_t log2_ctb, log2_min_cb, log2_min_tb, log2_max_tb, max_th_depth_intra;
  int32_t chroma_array_type, sub_w, sub_h, bit_depth_y, bit_depth_c, qp_bd_offset_y, qp_bd_offset_c;
  int32_t log2_max_transform_skip_size, log2_min_cu_qp_delta_size, pps_cb_qp_offset, pps_cr_qp_offset;
  int32_t log2_sao_offset_scale_luma, log2_sao_offset_scale_chroma;
  uint8_t transform_skip_enabled, sign_data_hiding, cu_qp_delta_enabled, entropy_coding_sync;
  uint8_t implicit_rdpcm, tskip_rotation, tskip_context, pps_loop_filter_across_slices;
  int32_t nslices;                   // slice segments of the picture (1: no per-CTB slice lookups)
  uint32_t pic_index;                // picture index in the batch (hc_tb::pic)
  uint32_t tb_global_base;           // index of this picture's first hc_tb in the batch array
  // per-CTB capacities
  uint32_t blk_cap[3], blk_cap_ctb, tb_cap_ctb, coeff_cap_ctb, resid_cap_ctb;
  // inputs
  const uint8_t* bytes;
  const Slice* slices;
  const int32_t* ctb_slice;          // per CTB (RS): index into slices
  const uint8_t* ctu_static;         // per CTB: sao_nb, sao_nb_c, flags, 0
  // scratch maps
  uint8_t* ct_depth;                 // per 8x8
  uint8_t* ipm;                      // per 4x4
  uint8_t* ipm_c;
  uint8_t* wpp_ctx;                  // ctbs_h * CTX_BYTES
  int* progress;                     // per CTB row: CTBs parsed
  int* error;
  // outputs
  int8_t* qp_map;                    // per 8x8 (is QP_Y while parsing)
  uint8_t* edge_map;                 // per 4x4
  hc_ctu* ctus;
  hc_blk* blks;
  hc_tb* tbs;
  hc_coeff* coeffs;
  uint32_t* tb_lists[4];             // batch-global K1 launch lists
  unsigned int* tb_counts;           // 4 counters
};

// One substream: CTBs [first_ctb, end_ctb) of one slice segment, starting at byte `byte_begin` of Pic::bytes
// (byte_begin == 0xffffffff: continue where the previous substream of the chain stopped).
struct Sub {
  uint32_t pic, slice;
  int32_t first_ctb, end_ctb;
  uint32_t byte_begin;
  uint32_t flags;                    // SUB_*
};
constexpr uint32_t SUB_ROW_CHAIN = 1;   // parallel mode: this substream is one CTB row, synchronised with the row above
struct Chain { uint32_t first_sub, nsubs; };

constexpr int ERR_NONE = 0, ERR_BITSTREAM = 1, ERR_CAPACITY = 2;

// ---- platform glue ------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
HC_D int k0_clz(unsigned v) { return __clz((int)v); }
HC_D int k0_popc(unsigned v) { return __popc(v); }
HC_D int k0_ctz(unsigned v) { return __ffs((int)v) - 1; }
HC_D int progress_load(const int* p) { return ld_acquire_s32(p); }
// the lanes of the chain's warp have all written parts of the row's maps / records: every lane fences its own writes, the
// warp meets, one lane publishes
HC_D void progress_store(int* p, int v) {
  __threadfence();
  __syncwarp();
  if ((threadIdx.x & 31) == 0) st_release_s32(p, v);
}
// A waiting chain polls a progress word of the row above. A CTB takes milliseconds to parse, so the poll interval grows
// to ~16 us: the first version polled every ~80 ns (__nanosleep(400) returns much earlier than asked), and the wait loops
// of the chains that cannot start yet issued as many instructions — and L2 requests on a handful of hot words — as all
// working chains together (ncu: 14.3 G of 29.7 G warp instructions of an 8 x 12 MP batch).
HC_D void backoff(unsigned& ns) { __nanosleep(ns); if (ns < 16384u) ns <<= 1; }
HC_D void far_wait() { __nanosleep(200000u); }
#else
HC_HD int k0_clz(unsigned v) { return __builtin_clz(v); }
HC_HD int k0_popc(unsigned v) { return __builtin_popcount(v); }
HC_HD int k0_ctz(unsigned v) { return __builtin_ctz(v); }
HC_HD int progress_load(const int* p) { return *p; }
HC_HD void progress_store(int* p, int v) { *p = v; }
HC_HD void backoff(unsigned&) {}
HC_HD void far_wait() {}
#endif

// Per-chain scratch. On the device it lives in shared memory next to ONE copy of the tables per CTA (k0_parse.cu),
// so every table lookup, context-state access and parameter read of the hot loops is an LDS / STS with a
// compile-time-known address space; on the host it is a member of the parser.
constexpr int TB_CAP_MAX = 768;      // transform blocks of one CTB: 64x64 4:4:4 in 4x4 blocks
// Device build: the arithmetic decoder's registers live HERE, not in the parser object (see CabacDev below).
struct alignas(16) CabState {
  unsigned long long value;          // offset + look-ahead bits, as in Cabac
  uint32_t range;
  int avail;
  const uint8_t* next;               // next byte of the substream to move into `value`
  const uint8_t* start;
  const uint8_t* end;
  uint32_t pad[2];
};
// The parse state of the chain: CTB position, record counters of the current CTB, QG / QP and CU state. It lives in the
// Scratch rather than in the parser object: the parser's syntax functions are real calls, and a stack object reached
// through `this` turns every access into a local- or generic-memory one (run_chain zeroes it).
struct ChainState {
  int err;
  int ctb_rs, ctb_x, ctb_y;
  uint32_t nblk[3], ntb, ncoeff, nresid;       // used inside the current CTB
  int IsCuQpDeltaCoded, CuQpDeltaVal;
  int currentQG_x, currentQG_y, lastQPYinPreviousQG, currentQPY;
  int qPYPrime, qPCbPrime, qPCrPrime;
  int cu_x0, cu_y0;
  int tt_x, tt_y;                              // the transform-tree node being parsed
  uint32_t tt_cbf;                             // nibble l: cbf_cb | cbf_cr << 2 the open level above hands to nodes of log2 l
  uint8_t cu_log2, tt_log2;
  uint8_t cu_max_trafo_depth, cu_intra_split;  // of the current CU, read by every level of its transform tree
  uint8_t filterLeftCbEdge, filterTopCbEdge;
  uint8_t tt_flags, tt_mode;                  // of the transform unit being parsed: transform_tree_flags, intra mode of the block
};
struct Scratch {
  CabState cab;
  ChainState cs;
  uint8_t ctx[CTX_BYTES];            // CABAC context states
  Pic pic;                           // copy of the picture descriptor
  Slice slice;                       // copy of the current slice segment descriptor
  uint8_t tb_size[TB_CAP_MAX];       // log2 - 2 of every transform block of the current CTB (K1 list flush, decode_ctu)
  int32_t rem[16];                   // coeff_abs_level_remaining of the coefficients of the current sub-block (residual_coding)
};
constexpr int TABLE_BYTES = (int)((sizeof(Tables) + 15) & ~(size_t)15);
constexpr int SCRATCH_BYTES = (int)((sizeof(Scratch) + 15) & ~(size_t)15);
#if defined(__CUDACC__)
extern __shared__ __align__(16) uint8_t k0_smem[];   // [Tables][Scratch x warps of the CTA]
// Byte offset of the calling warp's Scratch in k0_smem. The device parser derives every address from it instead of
// keeping one in the parser object: that object is a stack variable of the kernel, so each syntax function (a real call)
// had to read it back from local memory and keep `this` live across its calls.
HC_D uint32_t scratch_offset() { return (uint32_t)TABLE_BYTES + (threadIdx.x >> 5) * (uint32_t)SCRATCH_BYTES; }
#endif

// ---- arithmetic decoder: same design as host/hevc_cabac.h (offset + look-ahead in one 64-bit register) --------
// The hot functions copy this struct into a local (registers), decode, and write it back (see Parser).
struct Cabac {
  const uint8_t* start;
  const uint8_t* end;
  unsigned long long value;
  uint32_t range;
  int avail;
  uint32_t pos;                      // bytes of the substream already moved into `value`
  // device: the bitstream is read as aligned 32-bit words, one word ahead of its use, so that a refill never waits
  // for memory (w_hi holds the word the next byte comes from, w_lo the one after)
  const uint32_t* wp;
  uint32_t w_hi, w_lo, wshift;

  HC_HD static uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
  HC_HD uint32_t next32() {
#if defined(__CUDA_ARCH__)
    const uint32_t r = __funnelshift_l(w_lo, w_hi, wshift);
    w_hi = w_lo;
    w_lo = __byte_perm(__ldg(wp), 0, 0x0123);
    wp++;
#else
    // never read behind the substream: damaged slice data can ask for any number of bins before the next overrun() check
    // (found by the ASAN run of the fuzz inputs); the missing bytes read as zero, like the reference's decoder at the end
    // of its buffer (cabac.cc:230-243)
    const uint8_t* q = start + pos;
    uint32_t r = 0;
    if (q + 4 <= end) r = be32(q);
    else
      for (int k = 0; k < 4; k++)
        if (q + k < end) r |= (uint32_t)q[k] << (24 - 8 * k);
#endif
    pos += 4;
    return r;
  }
  HC_HD void refill() {
    if (__builtin_expect(avail < 16, 0)) {
      value = (value << 32) | next32();
      avail += 32;
    }
  }
  HC_HD void init(const uint8_t* p, const uint8_t* e) {
    start = p; end = e;
    range = 510;
    pos = 0;
#if defined(__CUDA_ARCH__)
    const unsigned a = (unsigned)(reinterpret_cast<uintptr_t>(p) & 3);
    wp = reinterpret_cast<const uint32_t*>(p - a);
    wshift = 8 * a;
    w_hi = __byte_perm(__ldg(wp), 0, 0x0123);
    w_lo = __byte_perm(__ldg(wp + 1), 0, 0x0123);
    wp += 2;
#else
    wp = nullptr; w_hi = w_lo = wshift = 0;
#endif
    value = next32();
    avail = 32 - 9;
  }
  HC_HD const uint8_t* position() const {
    const long long shifts = (long long)pos * 8 - 9 - avail;
    return start + 2 + (shifts >> 3);
  }
  HC_HD bool overrun() const { return position() > end; }
  HC_HD int bin(const Tables& t, uint8_t& state) {
    const uint32_t st = state;
    const uint32_t lps = t.range_lps[st >> 1][(range >> 6) & 3];
    const uint32_t nxt = *reinterpret_cast<const uint16_t*>(t.next_state[st]);   // both successors; picked below
    const uint32_t rmps = range - lps;
    const unsigned long long scaled = (unsigned long long)rmps << avail;
    const uint32_t is_lps = value >= scaled;
    if (is_lps) value -= scaled;
    const uint32_t r = is_lps ? lps : rmps;
    const int n = k0_clz(r) - 23;
    range = r << n;
    avail -= n;
    state = (uint8_t)(is_lps ? nxt >> 8 : nxt);
    refill();
    return (int)((st & 1) ^ is_lps);
  }
  HC_HD int bin(const Tables& t, uint8_t* ctx, int i) { return bin(t, ctx[i]); }
  HC_HD int bypass() {
    avail--;
    const unsigned long long scaled = (unsigned long long)range << avail;
    int b = 0;
    if (value >= scaled) { value -= scaled; b = 1; }
    refill();
    return b;
  }
  // x / range for x < 2^25, by the reciprocal table (an integer division is ~25 instructions on the device)
  HC_HD uint32_t div_range(const Tables& t, uint32_t x) const { return (uint32_t)(((unsigned long long)x * t.recip[range - 256]) >> 34); }
  HC_HD uint32_t bypass_bits(const Tables& t, int n) {
    uint32_t out = 0;
    while (n > 0) {
      const int k = n > 16 ? 16 : n;
      avail -= k;
      const uint32_t q = div_range(t, (uint32_t)(value >> avail));
      value -= (unsigned long long)(q * range) << avail;
      out = (out << k) | q;
      refill();
      n -= k;
    }
    return out;
  }
  HC_HD uint32_t peek16(const Tables& t) const { return div_range(t, (uint32_t)(value >> (avail - 16))); }
  HC_HD void consume(int n, uint32_t bins) {
    avail -= n;
    value -= (unsigned long long)(bins * range) << avail;
    refill();
  }
  HC_HD int terminate() {
    range -= 2;
    const unsigned long long scaled = (unsigned long long)range << avail;
    if (value >= scaled) return 1;
    if (range < 256) { range <<= 1; avail--; }
    refill();
    return 0;
  }
};


#if defined(__CUDACC__)
// ---- device form of the arithmetic decoder -------------------------------------------------------------------
// K0 is one lane per warp and, with every resident chain working, bound by INSTRUCTION FETCH (ncu at 32 files per batch:
// no_instruction is 49 % of the stall samples, and the kernel takes the same 143 ms at 16, 20, 24, 28 and 32 chains per
// SM): every warp of an SM partition walks its own part of a 40 KB hot path, so the 6 KB L0 / 32 KB L1.5 instruction
// caches miss all the time. 42 % of the executed instructions were copies of bin() + refill() inlined at 27 call sites.
// Here the decoder is a handful of small functions that are NOT inlined and keep their state (value / range / avail /
// byte pointer) in the chain's shared-memory scratch: one copy of the hot code for all call sites and all warps, and no
// decoder registers held across the syntax functions.
// Explicit shared-space accesses with 32-bit addresses: through a generic pointer every function recomputed the shared
// window (two S2R + LEA) before its first access.
HC_D uint4 lds128(uint32_t a) { uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory"); return v; }
HC_D void sts128(uint32_t a, uint4 v) { asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory"); }
HC_D uint2 lds64(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory"); return v; }
HC_D void sts64(uint32_t a, uint2 v) { asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory"); }
HC_D uint32_t lds32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
HC_D uint32_t lds16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
HC_D uint32_t lds8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
HC_D void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// `sa` = shared-space address of the chain's CabState (the Scratch starts with it), `ta` = of the CTA's Tables
constexpr uint32_t CAB_NEXT = (uint32_t)offsetof(CabState, next), CAB_END = (uint32_t)offsetof(CabState, end), CAB_CTX = (uint32_t)offsetof(Scratch, ctx);
constexpr uint32_t TAB_LPS = (uint32_t)offsetof(Tables, range_lps), TAB_NEXT = (uint32_t)offsetof(Tables, next_state), TAB_RECIP = (uint32_t)offsetof(Tables, recip);

static __device__ __noinline__ uint32_t cab_next32(uint32_t sa) {
  const uint2 pv = lds64(sa + CAB_NEXT);
  const unsigned long long pa = ((unsigned long long)pv.y << 32) | pv.x;
  {
    // behind the end of the substream (damaged slice data between two overrun() checks) the decoder reads zeros and the
    // read pointer stops: no load ever leaves the picture's bytes by more than the 8 bytes of the aligned pair below
    const uint2 ev = lds64(sa + CAB_END);
    const unsigned long long ea = ((unsigned long long)ev.y << 32) | ev.x;
    if (pa >= ea) {   // keep counting (position() / overrun() follow the pointer), stop loading
      const unsigned long long pe = pa + 4;
      sts64(sa + CAB_NEXT, make_uint2((uint32_t)pe, (uint32_t)(pe >> 32)));
      return 0u;
    }
  }
  const unsigned a = pv.x & 3u;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(pa - a);
  const uint32_t hi = __byte_perm(__ldg(w), 0, 0x0123), lo = __byte_perm(__ldg(w + 1), 0, 0x0123);
  const unsigned long long pn = pa + 4;
  sts64(sa + CAB_NEXT, make_uint2((uint32_t)pn, (uint32_t)(pn >> 32)));
  return __funnelshift_l(lo, hi, 8 * a);
}
#define K0_CAB_LOAD  const uint4 s_ = lds128(sa); unsigned long long value = ((unsigned long long)s_.y << 32) | s_.x; uint32_t range = s_.z; int avail = (int)s_.w;
#define K0_CAB_REFILL if (avail < 16) { value = (value << 32) | cab_next32(sa); avail += 32; }
#define K0_CAB_STORE sts128(sa, make_uint4((uint32_t)value, (uint32_t)(value >> 32), range, (uint32_t)avail));

static __device__ __noinline__ int cab_bin(uint32_t sa, uint32_t ta, int ci) {
  const uint32_t sp = sa + CAB_CTX + (uint32_t)ci;
  const uint32_t st = lds8(sp);
  K0_CAB_LOAD
  const uint32_t lps = lds8(ta + TAB_LPS + ((st >> 1) << 2) + ((range >> 6) & 3));
  const uint32_t nxt = lds16(ta + TAB_NEXT + (st << 1));   // both successors; picked below
  const uint32_t rmps = range - lps;
  const unsigned long long scaled = (unsigned long long)rmps << avail;
  const uint32_t is_lps = value >= scaled;
  if (is_lps) value -= scaled;
  const uint32_t r = is_lps ? lps : rmps;
  const int n = __clz((int)r) - 23;
  range = r << n;
  avail -= n;
  sts8(sp, is_lps ? nxt >> 8 : nxt & 0xffu);
  K0_CAB_REFILL
  K0_CAB_STORE
  return (int)((st & 1) ^ is_lps);
}
// The sig_coeff_flag run of one sub-block (scan positions last_coeff .. 1) in one call. Lane k holds the context index
// and the context state of position k; per bin the state comes by shuffle instead of a shared-memory load, the decoder
// registers stay in registers, and a decoded bin updates every lane that holds the same context. The states go back to
// shared memory once, at the end (lanes with the same context hold the same state).
static __device__ __noinline__ uint32_t cab_sig_run(uint32_t sa, uint32_t ta, uint32_t myci, int last_coeff) {
  const uint32_t sp = sa + CAB_CTX + myci;
  uint32_t myst = lds8(sp);
  K0_CAB_LOAD
  uint32_t sig = 0;
  K0_LOOP for (int k = last_coeff; k > 0; k--) {
    const uint32_t st = __shfl_sync(0xffffffffu, myst, k);
    const uint32_t ci = __shfl_sync(0xffffffffu, myci, k);
    const uint32_t lps = lds8(ta + TAB_LPS + ((st >> 1) << 2) + ((range >> 6) & 3));
    const uint32_t nxt = lds16(ta + TAB_NEXT + (st << 1));
    const uint32_t rmps = range - lps;
    const unsigned long long scaled = (unsigned long long)rmps << avail;
    const uint32_t is_lps = value >= scaled;
    if (is_lps) value -= scaled;
    const uint32_t r = is_lps ? lps : rmps;
    const int n = __clz((int)r) - 23;
    range = r << n;
    avail -= n;
    const uint32_t ns = is_lps ? nxt >> 8 : nxt & 0xffu;
    if (myci == ci) myst = ns;
    sig |= ((st & 1u) ^ is_lps) << k;
    K0_CAB_REFILL
  }
  sts8(sp, myst);
  K0_CAB_STORE
  return sig;
}
static __device__ __noinline__ int cab_bypass(uint32_t sa) {
  K0_CAB_LOAD
  avail--;
  const unsigned long long scaled = (unsigned long long)range << avail;
  int b = 0;
  if (value >= scaled) { value -= scaled; b = 1; }
  K0_CAB_REFILL
  K0_CAB_STORE
  return b;
}
static __device__ __noinline__ uint32_t cab_bypass_bits(uint32_t sa, uint32_t ta, int n) {
  K0_CAB_LOAD
  const unsigned long long recip = lds32(ta + TAB_RECIP + ((range - 256) << 2));
  uint32_t out = 0;
  K0_LOOP while (n > 0) {
    const int k = n > 16 ? 16 : n;
    avail -= k;
    const uint32_t q = (uint32_t)(((unsigned long long)(uint32_t)(value >> avail) * recip) >> 34);
    value -= (unsigned long long)(q * range) << avail;
    out = (out << k) | q;
    K0_CAB_REFILL
    n -= k;
  }
  K0_CAB_STORE
  return out;
}
static __device__ __noinline__ uint32_t cab_peek16(uint32_t sa, uint32_t ta) {
  const uint4 s_ = lds128(sa);
  const unsigned long long value = ((unsigned long long)s_.y << 32) | s_.x;
  const unsigned long long recip = lds32(ta + TAB_RECIP + ((s_.z - 256) << 2));
  return (uint32_t)(((unsigned long long)(uint32_t)(value >> ((int)s_.w - 16)) * recip) >> 34);
}
static __device__ __noinline__ void cab_consume(uint32_t sa, int n, uint32_t bins) {
  K0_CAB_LOAD
  avail -= n;
  value -= (unsigned long long)(bins * range) << avail;
  K0_CAB_REFILL
  K0_CAB_STORE
}
static __device__ __noinline__ int cab_terminate(uint32_t sa) {
  K0_CAB_LOAD
  range -= 2;
  const unsigned long long scaled = (unsigned long long)range << avail;
  int r = 1;
  if (value < scaled) {
    r = 0;
    if (range < 256) { range <<= 1; avail--; }
    K0_CAB_REFILL
  }
  K0_CAB_STORE
  return r;
}
#undef K0_CAB_LOAD
#undef K0_CAB_REFILL
#undef K0_CAB_STORE

// Same interface as Cabac, without state of its own: `sa` = shared-space address of the warp's CabState (the Scratch
// starts with it), `ta` = of the CTA's Tables. Copying it in and out of the hot functions is free.
struct CabacDev {
  HC_D static uint32_t ta() { return (uint32_t)__cvta_generic_to_shared(k0_smem); }
  HC_D static uint32_t sa() { return ta() + scratch_offset(); }
  HC_D CabState& state() const { return *reinterpret_cast<CabState*>(k0_smem + scratch_offset()); }
  HC_D void init(const uint8_t* p, const uint8_t* e) {
    CabState& c = state();
    c.start = p; c.end = e; c.next = p;
    c.range = 510;
    c.value = cab_next32(sa());
    c.avail = 32 - 9;
  }
  HC_D const uint8_t* position() const {
    const CabState& c = state();
    const long long shifts = (long long)(c.next - c.start) * 8 - 9 - c.avail;
    return c.start + 2 + (shifts >> 3);
  }
  HC_D bool overrun() const { return position() > state().end; }
  HC_D int bin(const Tables&, uint8_t*, int i) { return cab_bin(sa(), ta(), i); }
  HC_D int bypass() { return cab_bypass(sa()); }
  HC_D uint32_t bypass_bits(const Tables&, int n) { return cab_bypass_bits(sa(), ta(), n); }
  HC_D uint32_t peek16(const Tables&) const { return cab_peek16(sa(), ta()); }
  HC_D void consume(int n, uint32_t bins) { cab_consume(sa(), n, bins); }
  HC_D int terminate() { return cab_terminate(sa()); }
};
#endif
#if defined(__CUDA_ARCH__)
typedef CabacDev CabacT;
#else
typedef Cabac CabacT;
#endif

HC_HD uint8_t ctx_init_state(int init_value, int slice_qp) {
  const int slope = init_value >> 4, offs = init_value & 15;
  const int m = slope * 5 - 45, n = (offs << 3) - 16;
  const int q = slice_qp < 0 ? 0 : (slice_qp > 51 ? 51 : slice_qp);
  int pre = ((m * q) >> 4) + n;
  pre = pre < 1 ? 1 : (pre > 126 ? 126 : pre);
  const int mps = pre <= 63 ? 0 : 1;
  const int st = mps ? pre - 64 : 63 - pre;
  return (uint8_t)((st << 1) | mps);
}

HC_HD int morton4(int x, int y) {   // interleave 4 bits of x (even positions) and 4 bits of y (odd positions)
  unsigned v = (unsigned)(x & 15) | ((unsigned)(y & 15) << 8);
  v = (v | (v << 2)) & 0x3333u;
  v = (v | (v << 1)) & 0x5555u;
  return (int)((v & 0xffu) | (v >> 7));
}

// ---- neighbour availability of one prediction block (intrapred.h:443-543, :838-940), no tiles: TS == RS ---------
// Fills avail_left / avail_top / HC_BLK_AVAIL_TL of a record emitted by Parser::emit_blk. `p` may live anywhere.
HC_HD void finish_blk(const Pic& p, hc_blk& b) {
  const int cIdx = b.cidx, xB = b.x, yB = b.y, log2 = b.log2;
  const int nT = 1 << log2;
  const int SubW = cIdx == 0 ? 1 : p.sub_w, SubH = cIdx == 0 ? 1 : p.sub_h;
  const int xBL = xB * SubW, yBL = yB * SubH;
  const int l2c = p.log2_ctb, cw = p.ctbs_w;
  const int sh2 = l2c - p.log2_min_tb, mask = (1 << l2c) - 1;
  auto zs = [&](int x, int y) { return ((((x >> l2c) + (y >> l2c) * cw)) << (2 * sh2)) + morton4((x & mask) >> p.log2_min_tb, (y & mask) >> p.log2_min_tb); };
  auto sa_of = [&](int n) { return p.nslices == 1 ? 0 : p.slices[p.ctb_slice[n]].slice_addr_rs; };
  bool aL = true, aT = true, aTR = true, aTL = true;
  if (xBL == 0) { aL = false; aTL = false; }
  if (yBL == 0) { aT = false; aTL = false; aTR = false; }
  if (xBL + nT * SubW >= p.W) aTR = false;
  if (p.nslices != 1) {
    const int xCur = xBL >> l2c, yCur = yBL >> l2c;
    const int xLeft = (xBL - 1) >> l2c, xRight = (xBL + nT * SubW) >> l2c, yTop = (yBL - 1) >> l2c;
    const int sa = sa_of(xCur + yCur * cw);
    if (aL && sa_of(xLeft + yCur * cw) != sa) aL = false;
    if (aT && sa_of(xCur + yTop * cw) != sa) aT = false;
    if (aTL && sa_of(xLeft + yTop * cw) != sa) aTL = false;
    if (aTR && sa_of(xRight + yTop * cw) != sa) aTR = false;
  }
  int nBottom = (p.H - yBL + SubH - 1) / SubH;
  if (nBottom > 2 * nT) nBottom = 2 * nT;
  int nRight = (p.W - xBL + SubW - 1) / SubW;
  if (nRight > 2 * nT) nRight = 2 * nT;
  const int currAddr = zs(xBL, yBL);
  unsigned left = 0, top = 0;
  if (aL) {
    for (int y = nBottom - 1; y >= 0; y -= 4)
      if (zs((xB - 1) * SubW, (yB + y) * SubH) <= currAddr) left |= 1u << (y >> 2);
  }
  bool tl = false;
  if (aTL) tl = zs((xB - 1) * SubW, (yB - 1) * SubH) <= currAddr;
  for (int x = 0; x < nRight; x += 4) {
    const bool ba = x < nT ? aT : aTR;
    if (ba && zs((xB + x) * SubW, (yB - 1) * SubH) <= currAddr) top |= 1u << (x >> 2);
  }
  b.flags = (uint8_t)((b.flags & ~HC_BLK_AVAIL_TL) | (tl ? HC_BLK_AVAIL_TL : 0));
  b.avail_left = (uint16_t)left;
  b.avail_top = (uint16_t)top;
}

// All blocks of one CTB, lanes [lane, lane + stride, ...] (host: lane 0, stride 1).
HC_HD void finish_ctb(const Pic& p, int ctb, int lane, int stride) {
  const hc_ctu& ctu = p.ctus[ctb];
  for (int c = 0; c < 3; c++)
    for (int k = lane; k < (int)ctu.blk_count[c]; k += stride) finish_blk(p, p.blks[ctu.blk_first[c] + k]);
}

// One 16-byte record (hc_tb, hc_blk) from four words held in registers: one vector store on the device.
HC_HD void store_rec16(void* dst, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<uint4*>(dst) = make_uint4(w0, w1, w2, w3);   // the record arrays are 16-byte aligned
#else
  const uint32_t w[4] = {w0, w1, w2, w3};
  memcpy(dst, w, 16);
#endif
}
static_assert(sizeof(hc_tb) == 16 && sizeof(hc_blk) == 16, "records are stored as four words");

// ---- the parser of one chain ---------------------------------------------------------------------------------
// All parse state is in the chain's Scratch (cs()).
struct Parser {
  // host build: the tables and the scratch are reached through these pointers and the decoder is a member; the device
  // build finds its copies in shared memory from the warp index (scratch_offset()), and CabacDev is empty
  const Tables* T;
  Scratch* S;
  CabacT cabac;

  // Device: the 32 lanes of a warp execute the parser with identical data (warp-uniform: one instruction issue serves all
  // of them) and share out the data-parallel loops: `for (i = lane(); i < n; i += K0_LANES)`. After such a loop whose
  // results later lanes read from memory, lanes_sync() orders the writes. Host: one lane.
#if defined(__CUDA_ARCH__)
  static constexpr int K0_LANES = 32;
  HC_HD int lane() const { return (int)(threadIdx.x & 31); }
  HC_HD void lanes_sync() const { __syncwarp(); }
  HC_HD const Tables& tab() const { return *reinterpret_cast<const Tables*>(k0_smem); }
  HC_HD Scratch& scratch() const { return *reinterpret_cast<Scratch*>(k0_smem + scratch_offset()); }
#else
  static constexpr int K0_LANES = 1;
  HC_HD int lane() const { return 0; }
  HC_HD void lanes_sync() const {}
  HC_HD const Tables& tab() const { return *T; }
  HC_HD Scratch& scratch() const { return *S; }
#endif
  HC_HD const Pic& pic() const { return scratch().pic; }
  HC_HD const Slice& slice() const { return scratch().slice; }
  HC_HD uint8_t* ctxs() const { return scratch().ctx; }
  HC_HD ChainState& cs() const { return scratch().cs; }

  HC_HD int bin(int c) { return cabac.bin(tab(), ctxs(), c); }
  HC_HD int err() const { return cs().err; }
  HC_HD void fail(int code) { ChainState& c = cs(); if (!c.err) c.err = code; }
  HC_HD void init_contexts() {
    const Tables& t = tab();
    uint8_t* ctx = ctxs();
    const int qp = slice().slice_qp_y;
    K0_LOOP for (int i = lane(); i < CX_COUNT; i += K0_LANES) ctx[i] = ctx_init_state(t.ctx_init[i], qp);
    lanes_sync();
  }

  // ---- availability (no tiles: TS == RS) ----
  HC_HD int ctb_of(int x, int y) const { const Pic& p = pic(); return (x >> p.log2_ctb) + (y >> p.log2_ctb) * p.ctbs_w; }
  // pictures with one slice (the usual case) never look at the per-CTB slice table
  HC_HD int slice_addr_of_ctb(int n) const { const Pic& p = pic(); return p.nslices == 1 ? 0 : p.slices[p.ctb_slice[n]].slice_addr_rs; }
  HC_HD bool ctb_available(int xC, int yC, int xN, int yN) const {
    const Pic& p = pic();
    if (xN < 0 || yN < 0 || xN >= p.W || yN >= p.H) return false;
    if (p.nslices == 1) return true;
    return slice_addr_of_ctb(ctb_of(xN, yN)) == slice_addr_of_ctb(ctb_of(xC, yC));
  }
  HC_HD int zs_addr(int x, int y) const {
    const Pic& p = pic();
    const int sh2 = p.log2_ctb - p.log2_min_tb, mask = (1 << p.log2_ctb) - 1;
    return (ctb_of(x, y) << (2 * sh2)) + morton4((x & mask) >> p.log2_min_tb, (y & mask) >> p.log2_min_tb);
  }
  HC_HD bool available_zscan(int xC, int yC, int xN, int yN) const {
    const Pic& p = pic();
    if (xN < 0 || yN < 0 || xN >= p.W || yN >= p.H) return false;
    if (zs_addr(xN, yN) > zs_addr(xC, yC)) return false;
    return ctb_available(xC, yC, xN, yN);
  }

  // ---- 7.3.8.3 SAO ----
  K0_FN void read_sao() {
    const Pic& p = pic();
    const Tables& t = tab();
    uint8_t* const ctx = ctxs();
    CabacT cb = cabac;
    const int ctb_rs = cs().ctb_rs;
    hc_ctu& ctu = p.ctus[ctb_rs];
    bool merge_left = false, merge_up = false;
    if (cs().ctb_x > 0 && slice_addr_of_ctb(ctb_rs - 1) == slice().slice_addr_rs) merge_left = cb.bin(t, ctx, CX_SAO_MERGE);
    if (cs().ctb_y > 0 && !merge_left && slice_addr_of_ctb(ctb_rs - p.ctbs_w) == slice().slice_addr_rs) merge_up = cb.bin(t, ctx, CX_SAO_MERGE);
    if (merge_left || merge_up) {
      const hc_ctu& src = p.ctus[merge_left ? ctb_rs - 1 : ctb_rs - p.ctbs_w];
      K0_LOOP for (int c = 0; c < 3; c++) {
        ctu.sao_type[c] = src.sao_type[c];
        ctu.sao_band_or_class[c] = src.sao_band_or_class[c];
        K0_LOOP for (int i = 0; i < 4; i++) ctu.sao_offset[c][i] = src.sao_offset[c][i];
      }
      if (!slice().sao_luma) ctu.sao_type[0] = 0;
      if (!slice().sao_chroma) ctu.sao_type[1] = ctu.sao_type[2] = 0;
      cabac = cb;
      return;
    }
    const int ncomp = p.chroma_array_type != 0 ? 3 : 1;
    K0_LOOP for (int c = 0; c < ncomp; c++) {
      if (!((slice().sao_luma && c == 0) || (slice().sao_chroma && c > 0))) { ctu.sao_type[c] = 0; continue; }
      if (c < 2) {
        int ty = 0;
        if (cb.bin(t, ctx, CX_SAO_TYPE)) ty = cb.bypass() ? 2 : 1;
        ctu.sao_type[c] = (uint8_t)ty;
      } else {
        ctu.sao_type[2] = ctu.sao_type[1];
      }
      if (ctu.sao_type[c] == 0) continue;
      const int bitDepth = c == 0 ? p.bit_depth_y : p.bit_depth_c;
      const int cMax = (1 << ((bitDepth < 10 ? bitDepth : 10) - 5)) - 1;
      uint32_t absv = 0;   // the four magnitudes (<= 31), 8 bits each
      K0_LOOP for (int i = 0; i < 4; i++) {
        int v = 0;
        K0_LOOP while (v < cMax && cb.bypass()) v++;
        absv |= (uint32_t)v << (8 * i);
      }
      const int scale = c == 0 ? p.log2_sao_offset_scale_luma : p.log2_sao_offset_scale_chroma;
      if (ctu.sao_type[c] == 1) {
        uint32_t sign = 0;   // bit i: offset i is negative
        K0_LOOP for (int i = 0; i < 4; i++)
          if ((absv >> (8 * i)) & 0xffu) sign |= (uint32_t)cb.bypass() << i;
        ctu.sao_band_or_class[c] = (uint8_t)cb.bypass_bits(t, 5);
        K0_LOOP for (int i = 0; i < 4; i++) {
          const int a = (int)((absv >> (8 * i)) & 0xffu);
          ctu.sao_offset[c][i] = (int8_t)((((sign >> i) & 1u) ? -a : a) * (1 << scale));
        }
      } else {
        if (c < 2) ctu.sao_band_or_class[c] = (uint8_t)cb.bypass_bits(t, 2);
        else ctu.sao_band_or_class[2] = ctu.sao_band_or_class[1];
        K0_LOOP for (int i = 0; i < 4; i++) {
          const int a = (int)((absv >> (8 * i)) & 0xffu);
          ctu.sao_offset[c][i] = (int8_t)((i < 2 ? a : -a) * (1 << scale));
        }
      }
    }
    cabac = cb;
  }

  // ---- 8.6.1 QP derivation (transform.cc:31-210 bookkeeping) ----
  K0_FN void derive_qp(int xCU, int yCU) {
    const Pic& p = pic();
    ChainState& s = cs();
    const int qgmask = (1 << p.log2_min_cu_qp_delta_size) - 1;
    const int xQG = xCU - (xCU & qgmask), yQG = yCU - (yCU & qgmask);
    if (xQG != s.currentQG_x || yQG != s.currentQG_y) {
      s.lastQPYinPreviousQG = s.currentQPY;
      s.currentQG_x = xQG;
      s.currentQG_y = yQG;
    }
    const int ctbmask = (1 << p.log2_ctb) - 1;
    const bool firstInCTBRow = (xQG == 0 && (yQG & ctbmask) == 0);
    const int sx = (slice().slice_addr_rs % p.ctbs_w) << p.log2_ctb, sy = (slice().slice_addr_rs / p.ctbs_w) << p.log2_ctb;
    const bool firstQGInSlice = (sx == xQG && sy == yQG);
    int pred = (firstQGInSlice || (firstInCTBRow && p.entropy_coding_sync)) ? slice().slice_qp_y : s.lastQPYinPreviousQG;
    int qA = pred, qB = pred;
    if (available_zscan(xQG, yQG, xQG - 1, yQG) && ctb_of(xQG - 1, yQG) == s.ctb_rs) qA = p.qp_map[((xQG - 1) >> 3) + (yQG >> 3) * p.w8];
    if (available_zscan(xQG, yQG, xQG, yQG - 1) && ctb_of(xQG, yQG - 1) == s.ctb_rs) qB = p.qp_map[(xQG >> 3) + ((yQG - 1) >> 3) * p.w8];
    pred = (qA + qB + 1) >> 1;
    const int QPY = ((pred + s.CuQpDeltaVal + 52 + 2 * p.qp_bd_offset_y) % (52 + p.qp_bd_offset_y)) - p.qp_bd_offset_y;
    s.qPYPrime = QPY + p.qp_bd_offset_y < 0 ? 0 : QPY + p.qp_bd_offset_y;
    const int qPiCb = clip3i(-p.qp_bd_offset_c, 57, QPY + p.pps_cb_qp_offset + slice().cb_qp_offset);
    const int qPiCr = clip3i(-p.qp_bd_offset_c, 57, QPY + p.pps_cr_qp_offset + slice().cr_qp_offset);
    int qPCb = qPiCb, qPCr = qPiCr;   // the reference does not cap non-4:2:0 at 51 (transform.cc:175-178)
    if (p.chroma_array_type == 1) {
      qPCb = qPiCb < 30 ? qPiCb : (qPiCb >= 44 ? qPiCb - 6 : tab().qpc420[qPiCb - 30]);
      qPCr = qPiCr < 30 ? qPiCr : (qPiCr >= 44 ? qPiCr - 6 : tab().qpc420[qPiCr - 30]);
    }
    s.qPCbPrime = qPCb + p.qp_bd_offset_c < 0 ? 0 : qPCb + p.qp_bd_offset_c;
    s.qPCrPrime = qPCr + p.qp_bd_offset_c < 0 ? 0 : qPCr + p.qp_bd_offset_c;
    const int l8 = s.cu_log2 > 3 ? s.cu_log2 - 3 : 0, n8 = 1 << l8;
    K0_LOOP for (int i = lane(); i < n8 * n8; i += K0_LANES) {
      const int xx = (s.cu_x0 >> 3) + (i & (n8 - 1)), yy = (s.cu_y0 >> 3) + (i >> l8);
      if (xx < p.w8 && yy < p.h8) p.qp_map[xx + yy * p.w8] = (int8_t)QPY;
    }
    lanes_sync();
    s.currentQPY = QPY;
  }

  // every 4x4 unit belongs to exactly one transform unit and the map starts zeroed, so plain stores suffice
  HC_HD void mark_tu_edges(int x0, int y0, int log2) {
    if (slice().deblocking_disabled) return;
    const Pic& p = pic();
    const ChainState& s = cs();
    const int n4 = (1 << log2) >> 2;
    const int left = (x0 == s.cu_x0) ? s.filterLeftCbEdge : 1, top = (y0 == s.cu_y0) ? s.filterTopCbEdge : 1;
    uint8_t* e = p.edge_map + (x0 >> 2) + (y0 >> 2) * p.w4;
    const uint8_t fl = left ? HC_EDGE_V : 0, ft = top ? HC_EDGE_H : 0;
    if (fl | ft) e[0] = (uint8_t)(fl | ft);
    if (left) {
      K0_LOOP for (int k = 1 + lane(); k < n4; k += K0_LANES) e[k * p.w4] = HC_EDGE_V;
    }
    if (top) {
      K0_LOOP for (int k = 1 + lane(); k < n4; k += K0_LANES) e[k] = HC_EDGE_H;
    }
  }

  // One prediction block record. The neighbour availability masks (avail_left / avail_top / HC_BLK_AVAIL_TL) only
  // depend on the block geometry and the slice layout, not on the parse, so they are filled in afterwards by a
  // massively parallel pass (finish_blk below: k0_finish_kernel on the device) instead of by the serial chain.
  HC_HD void emit_blk(int cIdx, int xB, int yB, int log2, int mode, bool has_resid, uint32_t resid_off) {
    const Pic& p = pic();
    ChainState& s = cs();
    const uint32_t n = s.nblk[cIdx];
    if (n >= p.blk_cap[cIdx]) { fail(ERR_CAPACITY); return; }
    s.nblk[cIdx] = n + 1;
    uint32_t base = (uint32_t)s.ctb_rs * p.blk_cap_ctb;
    if (cIdx > 0) base += p.blk_cap[0];
    if (cIdx > 1) base += p.blk_cap[1];
    // hc_blk: x, y | log2, mode, flags, cidx | avail_left = avail_top = 0 | resid_off
    store_rec16(p.blks + base + n, ((uint32_t)xB & 0xffffu) | ((uint32_t)yB << 16),
                ((uint32_t)log2 & 0xffu) | (((uint32_t)mode & 0xffu) << 8) | ((has_resid ? HC_BLK_HAS_RESID : 0u) << 16) | ((uint32_t)cIdx << 24),
                0u, has_resid ? resid_off : 0u);
  }

  // ---- 7.3.8.11 residual_coding ----
  // The arithmetic decoder state is copied into a local for the duration of the call, and the per-sub-block lists
  // (scan positions, base levels, "escape possible" flags, coded-sub-block neighbours) are bit-packed scalars, so the
  // whole loop nest runs out of registers and shared memory.
  K0_FN uint32_t residual_coding(int log2, int cIdx, int pred_mode) {
    const Pic& p = pic();
    const Tables& t = tab();
    uint8_t* const ctx = ctxs();
    CabacT cb = cabac;
    bool tskip = false;
    if (p.transform_skip_enabled && log2 <= p.log2_max_transform_skip_size) tskip = cb.bin(t, ctx, CX_TSKIP + (cIdx ? 1 : 0));

    // last significant coefficient position
    int last_x = 0, last_y = 0;
    {
      const int cMax = (log2 << 1) - 1;
      int offset, shift;
      if (cIdx == 0) { offset = 3 * (log2 - 2) + ((log2 - 1) >> 2); shift = (log2 + 1) >> 2; }
      else { offset = 15; shift = log2 - 2; }
      K0_LOOP for (int d = 0; d < 2; d++) {
        int v = 0;
        const int base = (d ? CX_LAST_Y : CX_LAST_X) + offset;
        K0_LOOP while (v < cMax && cb.bin(t, ctx, base + (v >> shift))) v++;
        if (d) last_y = v;
        else last_x = v;
      }
    }
    int LastX = last_x, LastY = last_y;
    if (last_x > 3) { const int nb = (last_x >> 1) - 1; LastX = ((2 + (last_x & 1)) << nb) + (int)cb.bypass_bits(t, nb); }
    if (last_y > 3) { const int nb = (last_y >> 1) - 1; LastY = ((2 + (last_y & 1)) << nb) + (int)cb.bypass_bits(t, nb); }

    int scanIdx = 0;
    if (log2 == 2 || (log2 == 3 && (cIdx == 0 || p.chroma_array_type == 3))) {
      if (pred_mode >= 6 && pred_mode <= 14) scanIdx = 2;
      else if (pred_mode >= 22 && pred_mode <= 30) scanIdx = 1;
    }
    if (scanIdx == 2) { const int tmp = LastX; LastX = LastY; LastY = tmp; }
    const int nT = 1 << log2;
    if (LastX >= nT || LastY >= nT) { fail(ERR_BITSTREAM); return 0; }

    const int lsb = log2 - 2;
    const uint8_t* scanSub = t.scan_sub[lsb][scanIdx];
    const uint8_t* scanPos = t.scan_pos[scanIdx];
    const int lastSubBlock = t.inv_sub[lsb][scanIdx][(LastX >> 2) + ((LastY >> 2) << lsb)];
    const int lastScanPos = t.inv_pos[scanIdx][(LastX & 3) + ((LastY & 3) << 2)];

    // coded_sub_block_flag of the right / lower neighbour, one bit per sub-block at Sx + 8 * Sy
    unsigned long long csbf_right = 0, csbf_below = 0;

    {
      const ChainState& s = cs();
      if (s.ntb >= p.tb_cap_ctb || s.nresid + (uint32_t)(nT * nT) > p.resid_cap_ctb) { fail(ERR_CAPACITY); return 0; }
    }
    // the coefficient records of this block start at cs().ncoeff, which stays put until the block's record is written
    hc_coeff* out = p.coeffs + ((uint32_t)cs().ctb_rs * p.coeff_cap_ctb + cs().ncoeff);

    uint32_t type = (uint32_t)cIdx;
    if (tskip) type |= HC_TB_TSKIP;
    else if (log2 == 2 && cIdx == 0) type |= HC_TB_DST;
    if (p.implicit_rdpcm && tskip && (pred_mode == 10 || pred_mode == 26)) type |= (pred_mode == 26) ? HC_TB_RDPCM_V : HC_TB_RDPCM_H;
    if (p.tskip_rotation && log2 == 2 && tskip) type |= HC_TB_ROTATE;

    const bool ts_ctx = p.tskip_context && tskip;
    const bool sign_hiding_possible = p.sign_data_hiding && !(p.implicit_rdpcm && tskip && (pred_mode == 10 || pred_mode == 26));
    int c1 = 1;
    uint32_t ncoeff_total = 0;
    const int chroma = cIdx ? 1 : 0;
    const int ts_c = chroma ? 43 : 42;
    const int sig_size = log2 == 3 ? (scanIdx == 0 ? 0 : 1) : 2;

    K0_LOOP for (int i = lastSubBlock; i >= 0; i--) {
      const int sxy = scanSub[i];
      const int Sx = sxy & 7, Sy = sxy >> 3;
      const int prevCsbf = (int)((csbf_right >> sxy) & 1) | ((int)((csbf_below >> sxy) & 1) << 1);
      int inferSbDc = 0, coded = 1;
      if (i < lastSubBlock && i > 0) {
        coded = cb.bin(t, ctx, CX_CSBF + (prevCsbf ? 1 : 0) + (cIdx ? 2 : 0));
        inferSbDc = 1;
      }
      if (!coded) continue;
      if (Sx > 0) csbf_right |= 1ull << (sxy - 1);
      if (Sy > 0) csbf_below |= 1ull << (sxy - 8);

      // significance map of this sub-block: bit k = coefficient at scan position k; decoding order is from the
      // highest position down
      uint32_t sig = 0;
      const int xS0 = Sx << 2, yS0 = Sy << 2;
      const uint8_t* sigtab = log2 == 2 ? t.sig_b4[chroma][scanIdx] : t.sig_sb[chroma][sig_size][(Sx | Sy) ? 1 : 0][prevCsbf][scanIdx];
      const int dc_ctx = ts_ctx ? ts_c : ((log2 == 2 || i > 0) ? sigtab[0] : (chroma ? 27 : 0));

      const int last_coeff = (i == lastSubBlock) ? lastScanPos - 1 : 15;
      if (i == lastSubBlock) sig = 1u << lastScanPos;
#if defined(__CUDA_ARCH__)
      if (last_coeff > 0) sig |= cab_sig_run(cb.sa(), cb.ta(), (uint32_t)(CX_SIG + (ts_ctx ? ts_c : sigtab[lane() & 15])), last_coeff);
#else
      if (ts_ctx) {
        K0_LOOP for (int k = last_coeff; k > 0; k--) sig |= (uint32_t)cb.bin(t, ctx, CX_SIG + ts_c) << k;
      } else {
        K0_LOOP for (int k = last_coeff; k > 0; k--) sig |= (uint32_t)cb.bin(t, ctx, CX_SIG + sigtab[k]) << k;
      }
#endif
      if (last_coeff >= 0) {
        if (sig != 0 || !inferSbDc) sig |= (uint32_t)cb.bin(t, ctx, CX_SIG + dc_ctx);
        else sig = 1;
      }
      if (sig == 0) continue;
#if defined(__CUDA_ARCH__)
      const int n = __popc(sig);
#else
      const int n = __builtin_popcount(sig);
#endif

      int ctxSet = (i == 0 || cIdx > 0) ? 0 : 2;
      if (c1 == 0) ctxSet++;
      c1 = 1;
      int firstG1 = 16;
      const int ng1 = n < 8 ? n : 8;
      const int g1base = CX_G1 + ctxSet * 4 + (cIdx > 0 ? 16 : 0);
      uint32_t g1mask = 0;              // coefficient c has abs level >= 2
      K0_LOOP for (int c = 0; c < ng1; c++) {
        const int b = cb.bin(t, ctx, g1base + c1);
        g1mask |= (uint32_t)b << c;
        if (b && c < firstG1) firstG1 = c;
        c1 = b ? 0 : ((c1 > 0 && c1 < 3) ? c1 + 1 : c1);
      }
      // escape (coeff_abs_level_remaining) follows when the base level is at its maximum: 3 for the first "greater 1"
      // coefficient with greater2 set, 2 for the other greater-1 coefficients of the first eight, 1 beyond them
      uint32_t escmask = (g1mask | ~((1u << ng1) - 1u)) & ((1u << n) - 1u);
      int g2 = 0;
      if (firstG1 < 16) {
        g2 = cb.bin(t, ctx, CX_G2 + ctxSet + (cIdx > 0 ? 4 : 0));
        if (!g2) escmask &= ~(1u << firstG1);
      }

      const int pos_first = 31 - k0_clz(sig), pos_last = 31 - k0_clz(sig & (0u - sig));
      const bool signHidden = sign_hiding_possible && (pos_first - pos_last > 3);
      const int nsign = signHidden ? n - 1 : n;
      const uint32_t signs = cb.bypass_bits(t, nsign) << (16 - nsign);

      if (cs().ncoeff + ncoeff_total + (uint32_t)n > p.coeff_cap_ctb) { fail(ERR_CAPACITY); return 0; }
      // (1) serial: coeff_abs_level_remaining of the coefficients that have one, in coding order (Rice adaptation)
      int32_t* remv = scratch().rem;
      int sumRem = 0, rice = 0;
      uint32_t em = escmask;
      K0_LOOP while (em) {
        const int c = k0_ctz(em);
        em &= em - 1;
        const int base = 1 + (int)((g1mask >> c) & 1) + ((c == firstG1) ? g2 : 0);
        int rem = 0;
        const uint32_t q16 = cb.peek16(t);
        const int ones = q16 == 0xffffu ? 16 : k0_clz(~(q16 << 16));
        const int suffix_len = ones <= 3 ? rice : ones - 3 + rice;
        const int len = ones + 1 + suffix_len;
        if (len <= 16) {
          const uint32_t bins = q16 >> (16 - len);
          const int suffix = (int)(bins & ((1u << suffix_len) - 1u));
          rem = ones <= 3 ? (ones << rice) + suffix : (((1 << (ones - 3)) + 3 - 1) << rice) + suffix;
          cb.consume(len, bins);
        } else {
          int prefix = 0;
          K0_LOOP while (prefix < 32 && cb.bypass()) prefix++;
          if (prefix >= 32) { fail(ERR_BITSTREAM); return 0; }
          if (prefix <= 3) rem = (prefix << rice) + (int)cb.bypass_bits(t, rice);
          else rem = (((1 << (prefix - 3)) + 3 - 1) << rice) + (int)cb.bypass_bits(t, prefix - 3 + rice);
        }
        if (base + rem > 3 * (1 << rice)) { rice++; if (rice > 4) rice = 4; }
        remv[c] = rem;
        sumRem += rem;
      }
      // (2) lane-parallel: scan position k of the sub-block -> its record. Coefficient index c (coding order: from the
      // highest position down) = number of significant positions above k; sign-data hiding flips the LAST coefficient when
      // the sum of all absolute levels is odd — the sum of the base levels follows from the masks.
      const int sumAbs = n + k0_popc(g1mask & ((1u << n) - 1u)) + (firstG1 < 16 ? g2 : 0) + sumRem;
      const int pos0 = xS0 + (yS0 << log2);
      K0_LOOP for (int k = 15 - lane(); k >= 0; k -= K0_LANES) {
        if (!((sig >> k) & 1)) continue;
        const int c = k0_popc(sig >> (k + 1));
        int level = 1 + (int)((g1mask >> c) & 1) + ((c == firstG1) ? g2 : 0);
        if ((escmask >> c) & 1) level += remv[c];
        bool neg = (c < nsign) ? ((signs >> (15 - c)) & 1) : false;
        if (signHidden && c == n - 1 && (sumAbs & 1)) neg = !neg;
        const int sp = scanPos[k];
        hc_coeff co;
        co.pos = (uint16_t)(pos0 + (sp & 3) + ((sp >> 2) << log2));
        co.level = (int16_t)(neg ? -level : level);
        out[ncoeff_total + c] = co;
      }
      ncoeff_total += (uint32_t)n;
    }
    cabac = cb;
    ChainState& s = cs();
    const uint32_t ctb = (uint32_t)s.ctb_rs, ntb = s.ntb;
    const uint32_t resid_off = ctb * p.resid_cap_ctb + s.nresid;
    const uint32_t qp = (uint32_t)(cIdx == 0 ? s.qPYPrime : (cIdx == 1 ? s.qPCbPrime : s.qPCrPrime));
    // hc_tb: coeff_off | resid_off | ncoeff, pic | log2, qp, type, matrix_id
    store_rec16(p.tbs + (ctb * p.tb_cap_ctb + ntb), ctb * p.coeff_cap_ctb + s.ncoeff, resid_off,
                (ncoeff_total & 0xffffu) | (p.pic_index << 16),
                (uint32_t)log2 | ((qp & 0xffu) << 8) | (type << 16) | ((log2 == 5 ? 0u : (uint32_t)cIdx) << 24));
    scratch().tb_size[ntb] = (uint8_t)(log2 - 2);
    s.ntb = ntb + 1;
    s.ncoeff += ncoeff_total;
    s.nresid += (uint32_t)(nT * nT);
    return resid_off;
  }

  // ---- 7.3.8.10 transform_unit (record emission in the reference's reconstruction order, slice.cc:3979-4118) ----
  // The unit is the transform-tree node in cs(): tt_x, tt_y, tt_log2, and tt_flags from transform_tree_flags. Inlined into
  // the transform-tree walk, its only caller. residual_coding needs nearly all registers, so across its calls this keeps
  // only the chroma block index; the rest is read again from cs() and pic().
  HC_HD void transform_unit() {
    const Pic& p = pic();
    if ((cs().tt_flags & 0x3e) && p.cu_qp_delta_enabled && !cs().IsCuQpDeltaCoded) {
      int v = 0;
      if (bin(CX_CU_QP_DELTA)) {
        v = 1;
        K0_LOOP while (v < 5 && bin(CX_CU_QP_DELTA + 1)) v++;
        if (v == 5) {
          int k = 0;
          K0_LOOP while (k < 32 && cabac.bypass()) k++;
          if (k >= 32) { fail(ERR_BITSTREAM); return; }
          v += ((1 << k) - 1) + (int)cabac.bypass_bits(tab(), k);
        }
      }
      int sign = 0;
      if (v) sign = cabac.bypass();
      ChainState& s = cs();
      s.IsCuQpDeltaCoded = 1;
      s.CuQpDeltaVal = sign ? -v : v;
      derive_qp(s.cu_x0, s.cu_y0);
    }
    ChainState& s = cs();
    mark_tu_edges(s.tt_x, s.tt_y, s.tt_log2);
    s.tt_mode = p.ipm[(s.tt_x >> 2) + (s.tt_y >> 2) * p.w4];
    uint32_t roff = 0;
    if (s.tt_flags & 0x20) roff = residual_coding(s.tt_log2, 0, s.tt_mode);
    if (err()) return;
    emit_blk(0, s.tt_x, s.tt_y, s.tt_log2, s.tt_mode, (s.tt_flags & 0x20) != 0, roff);
    const int cat = p.chroma_array_type;
    if (cat == 0) return;
    // chroma of this TU; else the parent's 8x8 chroma with the 4th 4x4 luma block (blkIdx 3: bit 2 of x and y set — a 4x4
    // TU always has a parent, CUs are at least 8x8)
    if (!(s.tt_log2 > 2 || cat == 3) && !(s.tt_x & s.tt_y & 4)) return;
    K0_LOOP for (int k = 0; k < (cat == 2 ? 4 : 2); k++) {
      int c, xB, yB, l2;
      bool coded = chroma_block(k, c, xB, yB, l2);
      const int lx = xB * p.sub_w, ly = yB * p.sub_h;   // mode lookup position of the reference (slice.cc:3760-3763)
      s.tt_mode = p.ipm_c[((lx < p.W - 1 ? lx : p.W - 1) >> 2) + ((ly < p.H - 1 ? ly : p.H - 1) >> 2) * p.w4];
      uint32_t ro = 0;
      if (coded) ro = residual_coding(l2, c, s.tt_mode);
      if (err()) return;
      coded = chroma_block(k, c, xB, yB, l2);
      emit_blk(c, xB, yB, l2, s.tt_mode, coded, ro);
    }
  }

  // Chroma block k of the transform unit in cs() — Cb, then Cr; with 4:2:2 each as an upper and a lower square: its
  // component, position and size; returns its cbf. Evaluated again after the block's residual_coding call instead of
  // being held in registers across it.
  HC_HD bool chroma_block(int k, int& c, int& xB, int& yB, int& l2) const {
    const Pic& p = pic();
    const ChainState& s = cs();
    const int cat = p.chroma_array_type, log2 = s.tt_log2;
    const bool own = log2 > 2 || cat == 3;
    const int t = cat == 2 ? k & 1 : 0;
    c = cat == 2 ? 1 + (k >> 1) : 1 + k;
    l2 = cat == 3 ? log2 : (log2 > 2 ? log2 - 1 : 2);
    xB = (own ? s.tt_x : s.tt_x - 4) / p.sub_w;
    yB = (own ? s.tt_y : s.tt_y - 4) / p.sub_h + (t << l2);
    return (s.tt_flags >> (2 * c - 1 + t)) & 1;
  }

  // ---- 7.3.8.8 transform_tree ----
  // The flags of one node. `parent_cbf`: cbf_cb | cbf_cr << 2 of the parent; returns
  // split | cbf_cb << 1 | cbf_cr << 3 | cbf_luma << 5
  HC_HD int transform_tree_flags(int log2, int depth, int parent_cbf) {
    const Pic& p = pic();
    const Tables& t = tab();
    uint8_t* const ctx = ctxs();
    const int max_depth = cs().cu_max_trafo_depth, intra_split = cs().cu_intra_split;
    const int parent_cbf_cb = parent_cbf & 3, parent_cbf_cr = parent_cbf >> 2;
    CabacT cb = cabac;
    int split;
    if (log2 <= p.log2_max_tb && log2 > p.log2_min_tb && depth < max_depth && !(intra_split && depth == 0)) split = cb.bin(t, ctx, CX_SPLIT_TRANSFORM + 5 - log2);
    else split = (log2 > p.log2_max_tb || (intra_split && depth == 0)) ? 1 : 0;
    int cbf_cb = -1, cbf_cr = -1;
    if ((log2 > 2 && p.chroma_array_type != 0) || p.chroma_array_type == 3) {
      const bool second = p.chroma_array_type == 2 && (!split || log2 == 3);
      if (parent_cbf_cb) {
        cbf_cb = cb.bin(t, ctx, CX_CBF_CHROMA + depth);
        if (second) cbf_cb |= cb.bin(t, ctx, CX_CBF_CHROMA + depth) << 1;
      }
      if (parent_cbf_cr) {
        cbf_cr = cb.bin(t, ctx, CX_CBF_CHROMA + depth);
        if (second) cbf_cr |= cb.bin(t, ctx, CX_CBF_CHROMA + depth) << 1;
      }
    }
    if (cbf_cb < 0) cbf_cb = (depth > 0 && log2 == 2) ? parent_cbf_cb : 0;
    if (cbf_cr < 0) cbf_cr = (depth > 0 && log2 == 2) ? parent_cbf_cr : 0;
    int cbf_luma = 0;
    if (!split) cbf_luma = cb.bin(t, ctx, CX_CBF_LUMA + (depth == 0 ? 1 : 0));
    cabac = cb;
    return split | (cbf_cb << 1) | (cbf_cr << 3) | (cbf_luma << 5);
  }

  // The transform tree of the current CU (position, size, depth limit and intra split in cs()), walked in z-order by a
  // loop rather than by recursion, so that a node costs no call and no call frame in local memory: the parser is
  // instruction-fetch bound. The walk's state is the node (tt_x, tt_y, tt_log2) and the chroma cbfs each open level
  // hands to its children (tt_cbf); a node's position says which child it is. It lives in cs(), not in registers,
  // because residual_coding needs nearly all of them.
  HC_HD void transform_tree() {
    {
      ChainState& s = cs();
      s.tt_x = s.cu_x0; s.tt_y = s.cu_y0; s.tt_log2 = s.cu_log2;
      s.tt_cbf = 5u << (4 * s.cu_log2);   // the root inherits cbf_cb = cbf_cr = 1
    }
    K0_LOOP for (;;) {
      if (err()) return;
      ChainState& s = cs();
      const int log2 = s.tt_log2;
      const int f = transform_tree_flags(log2, s.cu_log2 - log2, (s.tt_cbf >> (4 * log2)) & 15);
      if (f & 1) {
        if (log2 == 2) { fail(ERR_BITSTREAM); return; }
        s.tt_cbf = (s.tt_cbf & ~(15u << (4 * (log2 - 1)))) | ((uint32_t)((f >> 1) & 15) << (4 * (log2 - 1)));
        s.tt_log2 = (uint8_t)(log2 - 1);
        continue;   // first child: same position
      }
      s.tt_flags = (uint8_t)f;
      transform_unit();
      // next node: the next sibling, or up while this node is its parent's 4th child
      int x = s.tt_x, y = s.tt_y, l = s.tt_log2;
      const int cu_log2 = s.cu_log2;
      K0_LOOP for (;;) {
        if (l == cu_log2) return;
        const int h = 1 << l;
        if (!(x & h)) { x += h; break; }           // child 0 -> 1, 2 -> 3
        if (!(y & h)) { x -= h; y += h; break; }   // child 1 -> 2
        x -= h; y -= h; l++;
      }
      s.tt_x = x; s.tt_y = y; s.tt_log2 = (uint8_t)l;
    }
  }

  // ---- 7.3.8.5 coding_unit (I slices) ----
  // size-independent part: everything up to the transform tree; leaves the CU's transform depth limit and intra split in cs()
  K0_FN void coding_unit_modes(int LOG2, int x0, int y0, int depth) {
    const Pic& p = pic();
    const int nCbS = 1 << LOG2;
    {
      ChainState& s = cs();
      s.cu_x0 = x0; s.cu_y0 = y0; s.cu_log2 = (uint8_t)LOG2;
    }
    {
      const int l8 = LOG2 - 3, n8 = nCbS >> 3;     // CUs are at least 8 x 8
      K0_LOOP for (int i = lane(); i < n8 * n8; i += K0_LANES)
        p.ct_depth[((x0 >> 3) + (i & (n8 - 1))) + ((y0 >> 3) + (i >> l8)) * p.w8] = (uint8_t)depth;
      lanes_sync();
    }
    // deblocking: which CU edges may be filtered (deblock.cc:165-215)
    {
      int filterLeftCbEdge = x0 != 0, filterTopCbEdge = y0 != 0;
      const int ctbmask = (1 << p.log2_ctb) - 1;
      if (x0 && (x0 & ctbmask) == 0 && !slice().loop_filter_across_slices && slice_addr_of_ctb(ctb_of(x0 - 1, y0)) != slice().slice_addr_rs) filterLeftCbEdge = 0;
      if (y0 && (y0 & ctbmask) == 0 && !slice().loop_filter_across_slices && slice_addr_of_ctb(ctb_of(x0, y0 - 1)) != slice().slice_addr_rs) filterTopCbEdge = 0;
      ChainState& s = cs();
      s.filterLeftCbEdge = (uint8_t)filterLeftCbEdge;
      s.filterTopCbEdge = (uint8_t)filterTopCbEdge;
    }
    derive_qp(x0, y0);

    const Tables& t = tab();
    uint8_t* const ctx = ctxs();
    CabacT cb = cabac;
    bool nxn = false;
    if (LOG2 == p.log2_min_cb) {
      nxn = !cb.bin(t, ctx, CX_PART_MODE);
      if (nxn && LOG2 <= p.log2_min_tb) { fail(ERR_BITSTREAM); return; }
    }
    // ---- intra prediction modes ----
    const int pbOffset = nxn ? nCbS / 2 : nCbS;
    const int nparts = nxn ? 4 : 1;
    uint32_t prev_flag = 0;   // bit i: prev_intra_luma_pred_flag of partition i
    uint32_t idx_rem = 0;     // bits 8i..8i+7: mpm_idx or rem_intra_luma_pred_mode of partition i
    K0_LOOP for (int i = 0; i < nparts; i++) prev_flag |= (uint32_t)cb.bin(t, ctx, CX_PREV_INTRA_LUMA) << i;
    K0_LOOP for (int i = 0; i < nparts; i++) {
      uint32_t v = 0;
      if ((prev_flag >> i) & 1u) {
        K0_LOOP while (v < 2 && cb.bypass()) v++;
      } else {
        v = cb.bypass_bits(t, 5);
      }
      idx_rem |= v << (8 * i);
    }
    const bool availA0 = ctb_available(x0, y0, x0 - 1, y0), availB0 = ctb_available(x0, y0, x0, y0 - 1);
    uint32_t luma_modes = 0;  // bits 8i..8i+7: IntraPredModeY of partition i
    K0_LOOP for (int idx = 0; idx < nparts; idx++) {
      const int i = (idx & 1) * pbOffset, j = (idx >> 1) * pbOffset;
      const int x = x0 + i, y = y0 + j;
      const bool availA = availA0 || i > 0, availB = availB0 || j > 0;
      int candA = 1, candB = 1;
      if (availA) candA = p.ipm[((x - 1) >> 2) + (y >> 2) * p.w4];
      if (availB && !(y - 1 < ((y >> p.log2_ctb) << p.log2_ctb))) candB = p.ipm[(x >> 2) + ((y - 1) >> 2) * p.w4];
      int cand0, cand1, cand2;
      if (candA == candB) {
        if (candA < 2) { cand0 = 0; cand1 = 1; cand2 = 26; }
        else { cand0 = candA; cand1 = 2 + ((candA - 2 - 1 + 32) % 32); cand2 = 2 + ((candA - 2 + 1) % 32); }
      } else {
        cand0 = candA; cand1 = candB;
        if (candA != 0 && candB != 0) cand2 = 0;
        else if (candA != 1 && candB != 1) cand2 = 1;
        else cand2 = 26;
      }
      const int v = (int)((idx_rem >> (8 * idx)) & 0xffu);
      int mode;
      if ((prev_flag >> idx) & 1u) {
        mode = v == 0 ? cand0 : (v == 1 ? cand1 : cand2);
      } else {
        int t;
        if (cand0 > cand1) { t = cand0; cand0 = cand1; cand1 = t; }
        if (cand0 > cand2) { t = cand0; cand0 = cand2; cand2 = t; }
        if (cand1 > cand2) { t = cand1; cand1 = cand2; cand2 = t; }
        mode = v;
        if (mode >= cand0) mode++;
        if (mode >= cand1) mode++;
        if (mode >= cand2) mode++;
      }
      luma_modes |= (uint32_t)mode << (8 * idx);
      const int n4 = pbOffset >> 2, l4 = k0_ctz((unsigned)n4);
      K0_LOOP for (int i = lane(); i < n4 * n4; i += K0_LANES)
        p.ipm[((x >> 2) + (i & (n4 - 1))) + ((y >> 2) + (i >> l4)) * p.w4] = (uint8_t)mode;
      lanes_sync();     // the next partition's candidate modes read this one's
    }
    const int cat = p.chroma_array_type;
    if (cat != 0) {
      const int nchroma = cat == 3 ? nparts : 1;
      K0_LOOP for (int idx = 0; idx < nchroma; idx++) {
        int icpm = 4;
        if (cb.bin(t, ctx, CX_INTRA_CHROMA)) icpm = (int)cb.bypass_bits(t, 2);
        const int luma = (int)((luma_modes >> (8 * idx)) & 0xffu);
        int m = luma;
        if (icpm != 4) {
          m = icpm == 0 ? 0 : (icpm == 1 ? 26 : (icpm == 2 ? 10 : 1));
          if (m == luma) m = 34;
        }
        if (cat == 2) m = tab().mode422[m];
        const int i = cat == 3 ? (idx & 1) * pbOffset : 0, j = cat == 3 ? (idx >> 1) * pbOffset : 0;
        const int n4 = (cat == 3 ? pbOffset : nCbS) >> 2, l4 = k0_ctz((unsigned)n4);
        K0_LOOP for (int q = lane(); q < n4 * n4; q += K0_LANES)
          p.ipm_c[(((x0 + i) >> 2) + (q & (n4 - 1))) + (((y0 + j) >> 2) + (q >> l4)) * p.w4] = (uint8_t)m;
      }
      lanes_sync();     // transform_unit reads the chroma mode of its position
    }
    cabac = cb;
    ChainState& s = cs();
    s.cu_max_trafo_depth = (uint8_t)(p.max_th_depth_intra + (nxn ? 1 : 0));
    s.cu_intra_split = nxn ? 1 : 0;
  }

  // ---- 7.3.8.4 coding_quadtree ----
  HC_HD int coding_quadtree_split(int log2, int x0, int y0, int depth) {
    const Pic& p = pic();
    const int size = 1 << log2;
    int split;
    if (x0 + size <= p.W && y0 + size <= p.H && log2 > p.log2_min_cb) {
      int condL = 0, condA = 0;
      if (ctb_available(x0, y0, x0 - 1, y0) && p.ct_depth[((x0 - 1) >> 3) + (y0 >> 3) * p.w8] > depth) condL = 1;
      if (ctb_available(x0, y0, x0, y0 - 1) && p.ct_depth[(x0 >> 3) + ((y0 - 1) >> 3) * p.w8] > depth) condA = 1;
      split = bin(CX_SPLIT_CU + condL + condA);
    } else {
      split = log2 > p.log2_min_cb;
    }
    if (p.cu_qp_delta_enabled && log2 >= p.log2_min_cu_qp_delta_size) { ChainState& s = cs(); s.IsCuQpDeltaCoded = 0; s.CuQpDeltaVal = 0; }
    return split;
  }

  // The coding quadtree of the current CTB, walked in z-order by a loop like transform_tree. Children that lie outside the
  // picture are skipped: the right ones when x + h >= W, the lower ones when y + h >= H. Every node first checks the
  // chain's error state and the bitstream position; an error ends the walk. After a CU the walk resumes from the CU's
  // position in cs(), so that nothing of it is held in registers across the CU's transform tree.
  HC_HD void coding_quadtree() {
    int log2 = pic().log2_ctb, x = cs().ctb_x << log2, y = cs().ctb_y << log2;
    K0_LOOP for (;;) {
      if (err() || cabac.overrun()) { fail(ERR_BITSTREAM); return; }
      const int depth = pic().log2_ctb - log2;
      if (coding_quadtree_split(log2, x, y, depth)) {
        if (log2 <= 3) { fail(ERR_BITSTREAM); return; }
        log2--;
        continue;   // first child: same position, always inside the picture
      }
      // 7.3.8.5 coding_unit
      coding_unit_modes(log2, x, y, depth);
      if (err()) return;
      transform_tree();
      const Pic& p = pic();
      x = cs().cu_x0; y = cs().cu_y0; log2 = cs().cu_log2;
      K0_LOOP for (;;) {
        if (log2 == p.log2_ctb) return;
        const int h = 1 << log2;
        if (!(x & h) && x + h < p.W) { x += h; break; }             // child 0 -> 1, 2 -> 3
        if (!(y & h) && y + h < p.H) { x &= ~h; y += h; break; }    // child 0 -> 2 when 1 is outside, 1 -> 2
        x &= ~h; y &= ~h; log2++;
      }
    }
  }

  // ---- one CTU ----
  K0_FN void decode_ctu() {
    const Pic& p = pic();
    {
      ChainState& s = cs();
      s.nblk[0] = s.nblk[1] = s.nblk[2] = 0;
      s.ntb = s.ncoeff = s.nresid = 0;
      hc_ctu& ctu = p.ctus[s.ctb_rs];
      K0_LOOP for (int c = 0; c < 3; c++) { ctu.sao_type[c] = 0; ctu.sao_band_or_class[c] = 0; for (int i = 0; i < 4; i++) ctu.sao_offset[c][i] = 0; }
    }
    if (slice().sao_luma || slice().sao_chroma) read_sao();
    coding_quadtree();
    const ChainState& s = cs();
    const int ctb_rs = s.ctb_rs;
    const uint32_t ntb = s.ntb;
    hc_ctu& ctu = p.ctus[ctb_rs];
    // K1 launch lists: one reservation per size class and CTB instead of one atomic per transform block
    if (ntb) {
      const uint8_t* ts = scratch().tb_size;
      const uint32_t tb0 = p.tb_global_base + (uint32_t)ctb_rs * p.tb_cap_ctb;
      unsigned long long packed = 0;   // four 16-bit counters
#if defined(__CUDA_ARCH__)
      // lane-parallel: count, lane l < 4 reserves the entries of size class l, then an order-preserving compaction 32
      // blocks at a time
      K0_LOOP for (uint32_t t = (uint32_t)lane(); t < ntb; t += K0_LANES) packed += 1ull << (16 * ts[t]);
      K0_LOOP for (int o = 16; o > 0; o >>= 1) packed += __shfl_xor_sync(0xffffffffu, packed, o);
      unsigned mine = 0;
      if (lane() < 4) {
        const unsigned n = (unsigned)(packed >> (16 * lane())) & 0xffffu;
        if (n) mine = atomicAdd(p.tb_counts + lane(), n);
      }
      unsigned slot[4];
#pragma unroll
      for (int l = 0; l < 4; l++) slot[l] = __shfl_sync(0xffffffffu, mine, l);
      const unsigned below = (1u << lane()) - 1u;
      K0_LOOP for (uint32_t t0 = 0; t0 < ntb; t0 += K0_LANES) {
        const uint32_t t = t0 + (uint32_t)lane();
        const int sz = t < ntb ? (int)ts[t] : -1;
#pragma unroll
        for (int l = 0; l < 4; l++) {
          const unsigned m = __ballot_sync(0xffffffffu, sz == l);
          if (sz == l) p.tb_lists[l][slot[l] + (unsigned)__popc(m & below)] = tb0 + t;
          slot[l] += (unsigned)__popc(m);
        }
      }
#else
      K0_LOOP for (uint32_t t = 0; t < ntb; t++) packed += 1ull << (16 * ts[t]);
      K0_LOOP for (int l = 0; l < 4; l++) {
        const unsigned n = (unsigned)(packed >> (16 * l)) & 0xffffu;
        if (!n) continue;
        unsigned slot = p.tb_counts[l];
        p.tb_counts[l] += n;
        K0_LOOP for (uint32_t t = 0; t < ntb; t++)
          if (ts[t] == l) p.tb_lists[l][slot++] = tb0 + t;
      }
#endif
    }
    uint32_t base = (uint32_t)ctb_rs * p.blk_cap_ctb;
    K0_LOOP for (int c = 0; c < 3; c++) {
      ctu.blk_first[c] = base;
      ctu.blk_count[c] = (uint16_t)s.nblk[c];
      base += p.blk_cap[c];
    }
    ctu.beta_offset = slice().beta_offset;
    ctu.tc_offset = slice().tc_offset;
    const uint8_t* st = p.ctu_static + 4 * ctb_rs;
    ctu.sao_nb = st[0];
    ctu.sao_nb_c = st[1];
    ctu.flags = (uint8_t)(st[2] | (slice().deblocking_disabled ? HC_CTU_DEBLOCK_OFF : 0));
    ctu.pad[0] = ctu.pad[1] = ctu.pad[2] = 0;
  }

  // ---- a chain of substreams (decode_slice_segment loop of the host parser) ----
  K0_FN void run_chain(const Pic* pics, const Sub* subs, uint32_t first_sub, uint32_t nsubs) {
    ChainState& c = cs();
    {
      uint32_t* w = reinterpret_cast<uint32_t*>(&c);   // CuQpDeltaVal & co. are read even when the stream never codes them
      K0_LOOP for (int i = lane(); i < (int)(sizeof(ChainState) / 4); i += K0_LANES) w[i] = 0;
      lanes_sync();
    }
    uint32_t loaded_pic = 0xffffffffu;
    uint8_t* const ctx = ctxs();
    K0_LOOP for (uint32_t s = 0; s < nsubs && !c.err; s++) {
      const Sub sub = subs[first_sub + s];
      if (sub.pic != loaded_pic) { scratch().pic = pics[sub.pic]; loaded_pic = sub.pic; }
      const Pic& p = pic();
      scratch().slice = p.slices[sub.slice];
      const uint8_t* seg_end = p.bytes + slice().data_end;
      if (sub.byte_begin != 0xffffffffu) cabac.init(p.bytes + sub.byte_begin, seg_end);
      const bool row_chain = sub.flags & SUB_ROW_CHAIN;
      c.ctb_rs = sub.first_ctb;
      c.currentQG_x = c.currentQG_y = -1;
      c.currentQPY = 0;
      if (s == 0) { c.IsCuQpDeltaCoded = 0; c.CuQpDeltaVal = 0; c.lastQPYinPreviousQG = 0; }
      if (!row_chain && sub.first_ctb == slice().segment_address && slice().segment_address > 0) {
        // thread-context initialisation of the reference (decctx.cc:467-506)
        const int prev = slice().segment_address - 1;
        int x = (((prev % p.ctbs_w) + 1) << p.log2_ctb) - 1, y = (((prev / p.ctbs_w) + 1) << p.log2_ctb) - 1;
        if (x > p.W - 1) x = p.W - 1;
        if (y > p.H - 1) y = p.H - 1;
        c.currentQPY = p.qp_map[(x >> 3) + (y >> 3) * p.w8];
      }
      // 9.3.1: context initialisation at the start of the slice segment (dependent segments of a serial chain keep
      // the table of the previous segment; rows of a WPP picture synchronise below)
      const bool segment_start = sub.first_ctb == slice().segment_address;
      if (segment_start && !slice().dependent) init_contexts();
      bool first_of_independent = segment_start && !slice().dependent;

      c.ctb_x = c.ctb_rs % p.ctbs_w;
      c.ctb_y = c.ctb_rs / p.ctbs_w;
      K0_LOOP while (c.ctb_rs < sub.end_ctb && !c.err) {
        const int ctb_x = c.ctb_x, ctb_y = c.ctb_y;
        if (row_chain && ctb_y > 0) {
          // wavefront: the row above must be two CTBs ahead (its context table, split depths and SAO parameters)
          const int need = ctb_x + 2 < p.ctbs_w ? ctb_x + 2 : p.ctbs_w;
          // a CTB of the row above takes milliseconds: while that row is two or more CTBs short of what this one needs
          // (the chains of rows 1, 2 of a batch start long before their turn) the chain sleeps in long steps; within one CTB
          // of its turn it polls with the short exponential back-off. The polling of the early rows was 6.7 % of all issued
          // instructions of the kernel (profiles/r02_k0_v7_ncu.txt).
          unsigned ns = 256;
          K0_LOOP for (;;) {
            const int have = progress_load(p.progress + ctb_y - 1);
            if (have >= need) break;
            if (need - have >= 2) far_wait(); else backoff(ns);
          }
        }
        if (p.entropy_coding_sync && ctb_x == 0 && ctb_y >= 1 && !(first_of_independent && c.ctb_rs == slice().segment_address)) {
          if (p.ctbs_w > 1) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(p.wpp_ctx + (size_t)(ctb_y - 1) * CTX_BYTES);
            uint32_t* dst = reinterpret_cast<uint32_t*>(ctx);
            K0_LOOP for (int i = lane(); i < CTX_BYTES / 4; i += K0_LANES) dst[i] = src[i];
            lanes_sync();
          } else {
            init_contexts();
          }
        }
        decode_ctu();
        if (c.err) break;
        if (cabac.overrun()) { fail(ERR_BITSTREAM); break; }
        if (p.entropy_coding_sync && ctb_x == 1 && ctb_y < p.ctbs_h - 1) {
          uint32_t* dst = reinterpret_cast<uint32_t*>(p.wpp_ctx + (size_t)ctb_y * CTX_BYTES);
          const uint32_t* src = reinterpret_cast<const uint32_t*>(ctx);
          K0_LOOP for (int i = lane(); i < CTX_BYTES / 4; i += K0_LANES) dst[i] = src[i];
        }
        if (row_chain) progress_store(p.progress + ctb_y, ctb_x + 1);
        const int end_of_slice_segment = cabac.terminate();
        const int next_rs = ++c.ctb_rs;
        if (ctb_x + 1 == p.ctbs_w) { c.ctb_x = 0; c.ctb_y = ctb_y + 1; }
        else c.ctb_x = ctb_x + 1;
        if (end_of_slice_segment) break;
        if (next_rs >= p.ctbs_w * p.ctbs_h) { fail(ERR_BITSTREAM); break; }
        if (p.entropy_coding_sync && c.ctb_x == 0) {
          if (!cabac.terminate()) { fail(ERR_BITSTREAM); break; }   // end_of_subset_one_bit
          if (row_chain) break;                                       // the next row is another chain
          const uint8_t* np = cabac.position();
          if (np >= seg_end) { fail(ERR_BITSTREAM); break; }
          cabac.init(np, seg_end);
          first_of_independent = false;
        }
      }
      if (!c.err && row_chain && c.ctb_rs != sub.end_ctb) fail(ERR_BITSTREAM);
    }
    if (c.err) {
      // unblock every waiter of this picture, then report
      if (loaded_pic == 0xffffffffu) scratch().pic = pics[subs[first_sub].pic];
      const Pic& p = pic();
      K0_LOOP for (int r = 0; r < p.ctbs_h; r++) progress_store(p.progress + r, 1 << 30);
      *p.error = c.err;
    }
  }
};

}  // namespace k0
}  // namespace hc
