// hevc_intra_enc.cc — synthetic-content generator: a small closed-loop HEVC intra (still picture)
// ENCODER used only to produce test and benchmark bitstreams.
//
// Why it exists: the reference's own content path (heif-enc + x265) is not available in this
// environment and the vendored enc265 crashes (SURVEY.md §0, §7 "hard parts"), so the configs of
// BASELINE.json (512x512 grid tiles, 4:2:2 10/12-bit, 1080p batches, ...) are generated here.
// TEST INFRASTRUCTURE: never loaded by the product. Every stream it writes is validated by decoding
// it with the unmodified reference (oracle/_ref/dec265) in tests/test_generated_streams.py.
//
// It is a real encoder (prediction from its own reconstruction, transform, quantisation, CABAC)
// with simple variance-driven block decisions and a seeded RNG for variety, so that decoded
// pictures look like the source and every syntax path the decoder supports can be switched on:
// chroma 4:0:0/4:2:0/4:2:2/4:4:4, 8-12 bit, CTB 16-64, TU 4-32 with RQT, NxN, SAO, deblocking
// offsets, cu_qp_delta, sign data hiding, transform skip, WPP, tiles, (dependent) slices, PCM,
// transquant bypass, scaling lists, strong intra smoothing, VUI, the SPS / PPS range extensions (transform skip up
// to 32x32, implicit RDPCM, rotation, transform-skip contexts, intra smoothing disabled, persistent Rice adaptation,
// CU chroma QP offset lists, SAO offset scale). A stress mode (hevc_enc_params::stress) pushes levels,
// intra modes, QPs and SAO parameters to the limits of their legal ranges for the parser tests, and counts what it wrote.
// Reconstruction inside the loop calls the CPU oracle's block functions (oracle/hevc_recon_oracle.c)
// so that encoder-side and decoder-side arithmetic cannot drift apart.
//
// Written from ITU-T H.265 §7.3 (syntax), §9.3 (CABAC encoding, §9.3.4.5 flush).
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/heifcuda_records.h"
#include "../../heif-decoder-lib_b200/csrc/host/hevc_cabac.h"
#include "../../heif-decoder-lib_b200/csrc/host/hevc_scan.h"

extern "C" {
void hc_oracle_predict_block(const hc_pic* pic, const hc_blk* b, uint16_t* plane, int stride, uint16_t* dst);
void hc_oracle_residual_block(const hc_pic* pic, const hc_tb* tb, const hc_coeff* coeffs, const uint8_t* scaling,
                              int32_t* res);

typedef struct hevc_enc_params {
  int32_t width, height;     // visible size (coded size is rounded up to a multiple of 8)
  int32_t chroma_format;     // 0..3
  int32_t bit_depth;         // 8..12
  int32_t qp;                // 0..51
  int32_t log2_ctb;          // 4..6
  int32_t log2_min_tb, log2_max_tb;
  int32_t max_th_depth;      // max_transform_hierarchy_depth_intra
  int32_t sao;
  int32_t deblock_disable, beta_offset_div2, tc_offset_div2;
  int32_t sign_hiding;
  int32_t cu_qp_delta;       // 0 off, else diff_cu_qp_delta_depth + 1
  int32_t transform_skip;
  int32_t wpp;
  int32_t tile_cols, tile_rows;
  int32_t slice_ctbs;        // 0: one slice, else CTBs per slice segment
  int32_t dependent_slices;  // every second slice segment is dependent
  int32_t strong_intra;
  int32_t scaling_list;      // 0 off, 1 default lists, 2 custom lists in the SPS
  int32_t pcm;
  int32_t transquant_bypass;
  int32_t vui, full_range, matrix, primaries, transfer;
  int32_t cb_qp_offset, cr_qp_offset;
  int32_t loop_filter_across_slices, loop_filter_across_tiles;
  int32_t stress;            // HEVC_ENC_STRESS_* bit mask; 0: ordinary content
  // range extensions (SPS / PPS range extension syntax); all 0: no extension is written
  int32_t transform_skip_rotation, transform_skip_context, implicit_rdpcm, intra_smoothing_disabled;
  int32_t persistent_rice_adaptation;
  int32_t extended_precision, cabac_bypass_alignment;  // flags only: the slice data ignores them (refused streams)
  int32_t log2_max_transform_skip_minus2;               // 0..3
  int32_t cross_component_prediction;                   // flag only (refused streams)
  int32_t chroma_qp_offset_list_len;                    // 0 off, else 1..6 entries with offsets drawn in -12..12
  int32_t diff_cu_chroma_qp_offset_depth;
  int32_t log2_sao_offset_scale_luma, log2_sao_offset_scale_chroma;
  uint32_t seed;
} hevc_enc_params;
}

// Stress mode: syntax values at the limits of their legal ranges, for parser tests. With stress == 0 the encoder
// makes exactly the draws of its RNG it always made, so every stream it wrote before is reproduced byte for byte.
enum {
  HEVC_ENC_STRESS_LEVELS = 1,   // per TB: keep the levels, or rewrite them sparse or dense with extreme values
  HEVC_ENC_STRESS_MODES = 2,    // luma modes uniform over 0..34, NxN more often, intra_chroma_pred_mode uniform over 0..4
  HEVC_ENC_STRESS_QP = 4,       // QG QP uniform over [-QpBdOffsetY, 51], reached through the wrap of 8.6.1
  HEVC_ENC_STRESS_SAO = 8,      // SAO offsets uniform over 0..cMax, more merges
  HEVC_ENC_STRESS_DENSE = 16,   // with LEVELS: every TB dense (every coefficient non-zero)
};

// Counters of what the encoder wrote (hevc_enc_encode_ex). X(name, n): n > 1 is an array, named name_0 .. name_<n-1>.
// Two groups: the syntax extremes of the stress mode, then the range-extension tools (from hevc_enc_rext_stat_first()
// on), which only streams with those tools switched on reach.
#define HEVC_ENC_STATS(X)                                                                                               \
  X(level_min, 1) X(level_max, 1) X(escape_long, 1) X(escape_prefix16, 1) X(rice4, 1)                                  \
  X(sb_16_sig, 1) X(sb_beyond_8, 1) X(sign_hidden_even, 1) X(sign_hidden_odd, 1) X(sign_string_16, 1)                   \
  X(last_suffix, 1) X(last_31, 1) X(inferred_sb_dc, 1) X(tskip_coded, 1)                                                \
  X(ctb_coeff_full, 1) X(ctb_tb_full, 1)                                                                                \
  X(qp_delta_ge5, 1) X(qp_delta_min, 1) X(qp_delta_max, 1) X(qp_wrap_below, 1) X(qp_wrap_above, 1) X(qp_y_neg, 1)       \
  X(qp_y_51, 1) X(chroma_qpi_clip_lo, 1) X(chroma_qpi_clip_hi, 1)                                                       \
  X(luma_mode, 35) X(mpm_idx, 3) X(rem_mode, 1) X(nxn_4_modes, 1) X(chroma_pred_mode, 5) X(chroma_mode_34, 1)           \
  X(mode422, 35)                                                                                                        \
  X(sao_offset_cmax_hbd, 1) X(sao_band_ge29, 1) X(sao_eo_class, 4) X(sao_merge_left, 1) X(sao_merge_up, 1)

#define HEVC_ENC_REXT_STATS(X)                                                                                          \
  X(rdpcm_h_tskip, 1) X(rdpcm_v_tskip, 1) X(rdpcm_h_bypass, 1) X(rdpcm_v_bypass, 1)                                     \
  X(rotate_tskip, 1) X(rotate_bypass, 1) X(tskip_log2, 4) X(sig_ctx_42, 1) X(sig_ctx_43, 1) X(sdh_off_rdpcm, 1)          \
  X(rice_init_gt0, 1) X(rice_gt4, 1) X(wpp_stat_coeff_restored, 1)                                                      \
  X(cu_chroma_qp_offset_off, 1) X(cu_chroma_qp_offset_idx, 6)                                                            \
  X(sao_offset_scaled_cmax, 1) X(no_edge_flt, 1) X(smoothing_skipped, 1) X(smoothing_skipped_strong, 1)

enum {
#define HEVC_ENC_STAT_ENUM(name, n) ST_##name, ST_##name##_end_ = ST_##name + (n) - 1,
  HEVC_ENC_STATS(HEVC_ENC_STAT_ENUM)
  ST_REXT_FIRST_,
  ST_REXT_BEFORE_ = ST_REXT_FIRST_ - 1,
  HEVC_ENC_REXT_STATS(HEVC_ENC_STAT_ENUM)
#undef HEVC_ENC_STAT_ENUM
  ST_COUNT
};

namespace {

using namespace hc;

inline int clip3(int lo, int hi, int v) { return v < lo ? lo : (v > hi ? hi : v); }

struct Rng {
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed * 0x9E3779B97F4A7C15ull + 0x1234567ull) {}
  uint32_t next() {
    s ^= s << 13; s ^= s >> 7; s ^= s << 17;
    return (uint32_t)(s >> 16);
  }
  int below(int n) { return (int)(next() % (uint32_t)n); }
  bool chance(int percent) { return below(100) < percent; }
};

// ------------------------------------------------------------------------------------------------
struct BitWriter {
  std::vector<uint8_t> bytes;
  uint32_t cur = 0;
  int nbits = 0;
  void put(uint32_t v, int n) {
    for (int i = n - 1; i >= 0; i--) {
      cur = (cur << 1) | ((v >> i) & 1);
      if (++nbits == 8) { bytes.push_back((uint8_t)cur); cur = 0; nbits = 0; }
    }
  }
  void ue(uint32_t v) {
    uint32_t x = v + 1;
    int len = 0;
    while ((x >> len) > 1) len++;
    put(0, len);
    put(x, len + 1);
  }
  void se(int v) { ue(v > 0 ? (uint32_t)(2 * v - 1) : (uint32_t)(-2 * v)); }
  void trailing() {
    put(1, 1);
    while (nbits) put(0, 1);
  }
  bool aligned() const { return nbits == 0; }
};

void append_nal(std::vector<uint8_t>& out, int nal_type, const std::vector<uint8_t>& rbsp) {
  std::vector<uint8_t> nal;
  nal.push_back((uint8_t)(nal_type << 1));
  nal.push_back(1);  // layer 0, temporal id plus1 = 1
  int zeros = 0;
  for (uint8_t b : rbsp) {
    if (zeros >= 2 && b <= 3) { nal.push_back(3); zeros = 0; }
    nal.push_back(b);
    zeros = b == 0 ? zeros + 1 : 0;
  }
  uint32_t n = (uint32_t)nal.size();
  out.push_back((uint8_t)(n >> 24)); out.push_back((uint8_t)(n >> 16)); out.push_back((uint8_t)(n >> 8)); out.push_back((uint8_t)n);
  out.insert(out.end(), nal.begin(), nal.end());
}

// ------------------------------------------------------------------------------------------------
// CABAC encoding engine (H.265 §9.3.4.5; carry propagation with a buffered-byte counter)
struct CabacEnc {
  std::vector<uint8_t>* out = nullptr;
  uint32_t low = 0, range = 510;
  int bits_left = 23, num_buffered = 0;
  uint32_t buffered_byte = 0xff;
  void start(std::vector<uint8_t>* o) { out = o; low = 0; range = 510; bits_left = 23; num_buffered = 0; buffered_byte = 0xff; }
  void write_out() {
    uint32_t lead = low >> (24 - bits_left);
    bits_left += 8;
    low &= 0xffffffffu >> bits_left;
    if (lead == 0xff) { num_buffered++; return; }
    if (num_buffered > 0) {
      uint32_t carry = lead >> 8;
      out->push_back((uint8_t)(buffered_byte + carry));
      buffered_byte = lead & 0xff;
      uint8_t fill = (uint8_t)((0xff + carry) & 0xff);
      while (num_buffered > 1) { out->push_back(fill); num_buffered--; }
    } else {
      num_buffered = 1;
      buffered_byte = lead;
    }
  }
  void test_write() { if (bits_left < 12) write_out(); }
  void bin(uint8_t& state, int v) {
    const detail::Transitions& tr = detail::kTransitions;
    uint32_t st = state;
    uint32_t lps = detail::kRangeLps[st >> 1][(range >> 6) & 3];
    range -= lps;
    if (v != (int)(st & 1)) {
      int nb = 0;
      uint32_t l = lps;
      while (l < 256) { l <<= 1; nb++; }
      low = (low + range) << nb;
      range = lps << nb;
      state = tr.lps[st];
      bits_left -= nb;
    } else {
      state = tr.mps[st];
      if (range >= 256) return;
      low <<= 1;
      range <<= 1;
      bits_left--;
    }
    test_write();
  }
  void bypass(int v) {
    low <<= 1;
    if (v) low += range;
    bits_left--;
    test_write();
  }
  void bypass_bits(uint32_t v, int n) { for (int i = n - 1; i >= 0; i--) bypass((v >> i) & 1); }
  void terminate(int v) {
    range -= 2;
    if (v) {
      low += range;
      low <<= 7;
      range = 2 << 7;
      bits_left -= 7;
    } else if (range >= 256) {
      return;
    } else {
      low <<= 1;
      range <<= 1;
      bits_left--;
    }
    test_write();
  }
  // flush + the terminating '1' bit + zero bits up to the byte boundary
  void finish() {
    if (low >> (32 - bits_left)) {
      out->push_back((uint8_t)(buffered_byte + 1));
      while (num_buffered > 1) { out->push_back(0x00); num_buffered--; }
      low -= 1u << (32 - bits_left);
    } else {
      if (num_buffered > 0) out->push_back((uint8_t)buffered_byte);
      while (num_buffered > 1) { out->push_back(0xff); num_buffered--; }
    }
    // remaining bits of low, then stop bit and alignment
    int n = 24 - bits_left;
    uint32_t v = low >> 8;
    uint32_t acc = 0;
    int nb = 0;
    auto putbit = [&](int b) {
      acc = (acc << 1) | (uint32_t)b;
      if (++nb == 8) { out->push_back((uint8_t)acc); acc = 0; nb = 0; }
    };
    for (int i = n - 1; i >= 0; i--) putbit((v >> i) & 1);
    putbit(1);
    while (nb) putbit(0);
  }
};

// ------------------------------------------------------------------------------------------------
const uint8_t kMode422[35] = {0,  1,  2,  2,  2,  2,  3,  5,  7,  8,  10, 12, 13, 15, 17, 18, 19, 20,
                              21, 22, 23, 23, 24, 24, 25, 25, 26, 27, 27, 28, 28, 29, 29, 30, 31};
const uint8_t kSigCtx4x4[16] = {0, 1, 4, 5, 2, 3, 4, 5, 6, 6, 8, 8, 7, 7, 8, 8};
const int kQuantScale[6] = {26214, 23302, 20560, 18396, 16384, 14564};
const uint8_t kDefault8x8Intra[64] = {
    16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 17, 16, 17, 16, 17, 18, 17, 18, 18, 17, 18, 21,
    19, 20, 21, 20, 19, 21, 24, 22, 22, 24, 24, 22, 22, 24, 25, 25, 27, 30, 27, 25, 25, 29,
    31, 35, 35, 31, 29, 36, 41, 44, 41, 36, 47, 54, 54, 47, 65, 70, 65, 88, 88, 115};
const uint8_t kDefault8x8Inter[64] = {
    16, 16, 16, 16, 16, 16, 16, 16, 16, 16, 17, 17, 17, 17, 17, 18, 18, 18, 18, 18, 18, 20,
    20, 20, 20, 20, 20, 20, 24, 24, 24, 24, 24, 24, 24, 24, 25, 25, 25, 25, 25, 25, 25, 28,
    28, 28, 28, 28, 28, 33, 33, 33, 33, 33, 41, 41, 41, 41, 54, 54, 54, 71, 71, 91};

int qpc_table_420(int qPi) {
  static const int8_t t[14] = {29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37, 37};
  if (qPi < 30) return qPi;
  if (qPi >= 44) return qPi - 6;
  return t[qPi - 30];
}

int dct_coef(int k, int n) {
  static const int t[32] = {64, 90, 90, 90, 89, 88, 87, 85, 83, 82, 80, 78, 75, 73, 70, 67,
                            64, 61, 57, 54, 50, 46, 43, 38, 36, 31, 25, 22, 18, 13, 9,  4};
  if (k == 0) return 64;
  int a = (k * (2 * n + 1)) % 128, s = 1;
  if (a > 64) a = 128 - a;
  if (a > 32) { a = 64 - a; s = -1; }
  return a == 32 ? 0 : s * t[a];
}
const int kDst[4][4] = {{29, 55, 74, 84}, {74, 74, 0, -74}, {84, -29, -74, 55}, {55, -84, 74, -29}};

struct TuData {
  bool coded = false;
  bool tskip = false;
  int rdpcm = 0;                // implicit RDPCM: 0 none, 1 horizontal, 2 vertical
  bool rotate = false;
  std::vector<int16_t> levels;  // nT*nT, raster
};

struct Node {
  int x0, y0, xBase, yBase, log2, depth, blkIdx;
  bool split = false;
  int cbf_cb = 0, cbf_cr = 0;   // as coded at this node (bit 1 = second 4:2:2 block)
  int cbf_luma = 0;
  std::unique_ptr<Node> child[4];
  TuData luma;
  TuData chroma[2][2];          // [cb/cr][block]
  int nchroma = 0;              // chroma blocks per component coded at this leaf (0, 1 or 2)
  int log2C = 0;
  int cxB = 0, cyB = 0;         // chroma block position (first block)
};

struct Enc {
  hevc_enc_params P;
  Rng rng;
  int W, H;                     // coded size
  int cf, bd, SubW, SubH;
  int log2_ctb, ctb, ctbs_w, ctbs_h, nctb;
  int log2_min_cb = 3;
  int log2_min_tb, log2_max_tb;
  int w8, h8, w4, h4;
  int tbs_w, tbs_h;
  int qp_bd_offset;
  std::vector<int> col_bd, row_bd, rs2ts, ts2rs, tile_id;
  std::vector<uint8_t> tile_start;
  std::vector<int> zs;
  std::vector<uint16_t> orig[3], rec[3];
  int pw[3], ph[3];
  std::vector<uint8_t> ct_depth, cu_flags, ipm;
  std::vector<int8_t> qp_y;
  std::vector<int> ctb_slice;
  hc_pic pic;
  std::vector<uint8_t> scaling;  // blob like the records' one
  uint8_t sl4[6][16], sl8[6][64], sl16[6][64], sl32[2][64];  // coded lists (diag order)
  int sl16_dc[6], sl32_dc[2];

  // slice / entropy state
  CabacEnc cabac;
  CtxSet ctx;
  std::vector<CtxSet> wpp_ctx;
  CtxSet dep_ctx;
  // StatCoeff (9.3.2.2 persistent Rice adaptation), stored and synchronised together with the context variables
  uint8_t stat_coeff[4] = {0, 0, 0, 0};
  std::vector<std::array<uint8_t, 4>> wpp_stat;
  std::array<uint8_t, 4> dep_stat = {{0, 0, 0, 0}};
  std::vector<uint8_t> slice_data;
  std::vector<uint32_t> entry_points;
  size_t substream_start = 0;
  int slice_addr_rs = 0, slice_qp = 26;
  bool slice_sao_luma = false, slice_sao_chroma = false;
  int ctb_addr_ts = 0, ctb_addr_rs = 0;
  bool IsCuQpDeltaCoded = false;
  int CuQpDeltaVal = 0;
  int qg_target_qp = 26;
  int currentQG_x = -1, currentQG_y = -1, lastQPYinPreviousQG = 0, currentQPY = 0;
  int cur_qp_y = 26;            // QP the current CU quantises with
  bool cu_bypass = false;
  int cu_x0 = 0, cu_y0 = 0, cu_log2 = 0;
  int log2_min_cu_qp_delta = 6;
  // cu_chroma_qp_offset: the decision of a chroma quantisation group is drawn when the group starts, takes effect at its
  // first TU with a coded chroma block (pass A) and is written there (pass B, in the same order)
  int log2_min_cu_chroma_qp_offset = 6, max_tskip_log2 = 2;
  int cqo_cb[6] = {}, cqo_cr[6] = {};
  bool cqo_coded_a = false, cqo_coded_b = false;
  int cqo_next = 0;                 // drawn for the current group: 0 flag off, k > 0 list entry k - 1
  int cqo_cur_cb = 0, cqo_cur_cr = 0;
  std::vector<int> cqo_queue;
  size_t cqo_read = 0;
  struct Sao { uint8_t type[3], boc[3]; int8_t off[3][4]; };
  std::vector<Sao> sao;
  uint64_t stats[ST_COUNT] = {};
  int ctb_ntb = 0, ctb_ncoeff = 0;  // coded TBs / coefficients of the current CTB

  explicit Enc(const hevc_enc_params& p) : P(p), rng(p.seed) {}

  inline void bin(int c, int v) { cabac.bin(ctx.s[c], v); }
  bool stress(int bit) const { return (P.stress & bit) != 0; }

  // ---- geometry helpers -------------------------------------------------------------------------
  int ctb_of(int x, int y) const { return (x >> log2_ctb) + (y >> log2_ctb) * ctbs_w; }
  int zs_addr(int x, int y) const { return zs[(x >> log2_min_tb) + (size_t)(y >> log2_min_tb) * tbs_w]; }
  bool ctb_available(int xC, int yC, int xN, int yN) const {
    if (xN < 0 || yN < 0 || xN >= W || yN >= H) return false;
    int c = ctb_of(xC, yC), n = ctb_of(xN, yN);
    if (ctb_slice[n] < 0 || ctb_slice[n] != ctb_slice[c]) return false;
    return tile_id[n] == tile_id[c];
  }
  bool available_zscan(int xC, int yC, int xN, int yN) const {
    if (xN < 0 || yN < 0 || xN >= W || yN >= H) return false;
    if (zs_addr(xN, yN) > zs_addr(xC, yC)) return false;
    return ctb_available(xC, yC, xN, yN);
  }

  void setup();
  void write_parameter_sets(std::vector<uint8_t>& out);
  void write_scaling_list_data(BitWriter& bw);
  void encode_picture(std::vector<uint8_t>& out);
  void init_contexts() { ctx_init_all(ctx, slice_qp); memset(stat_coeff, 0, sizeof(stat_coeff)); }
  bool rext_sps() const {
    return P.transform_skip_rotation || P.transform_skip_context || P.implicit_rdpcm || P.intra_smoothing_disabled ||
           P.persistent_rice_adaptation || P.extended_precision || P.cabac_bypass_alignment;
  }
  bool rext_pps() const {
    return P.log2_max_transform_skip_minus2 || P.cross_component_prediction || P.chroma_qp_offset_list_len ||
           P.log2_sao_offset_scale_luma || P.log2_sao_offset_scale_chroma;
  }
  void encode_ctu();
  void code_sao(int rx, int ry);
  void coding_quadtree(int x0, int y0, int log2, int depth);
  void coding_unit(int x0, int y0, int log2, int depth);
  double variance(int x0, int y0, int size) const;
  int choose_mode(int x0, int y0, int log2);
  hc_blk make_blk(int cIdx, int xB, int yB, int log2, int mode, bool no_edge) const;
  void build_tree(Node& n, int max_depth, int intra_split, const int* luma_modes, const int* chroma_modes);
  void process_tb(int cIdx, int xB, int yB, int log2, int mode, TuData& tu);
  void write_tree(Node& n, int max_depth, int intra_split, int parent_cbf_cb, int parent_cbf_cr, const int* luma_modes,
                  const int* chroma_modes);
  void write_tu(Node& n, const int* luma_modes, const int* chroma_modes);
  void residual_coding(const TuData& tu, int log2, int cIdx, int pred_mode);
  void derive_qp_pred(int xCU, int yCU, int& pred);
  void set_cu_qp(int qpy);
  int chroma_qp(int qpy, int c, int cu_off) const;
  int cu_chroma_offset(int c) const;
  int mode_for(const int* modes, int x, int y) const;
};

void Enc::setup() {
  cf = P.chroma_format; bd = P.bit_depth;
  SubW = (cf == 1 || cf == 2) ? 2 : 1;
  SubH = cf == 1 ? 2 : 1;
  W = (P.width + 7) & ~7;
  H = (P.height + 7) & ~7;
  log2_ctb = P.log2_ctb; ctb = 1 << log2_ctb;
  ctbs_w = (W + ctb - 1) / ctb; ctbs_h = (H + ctb - 1) / ctb; nctb = ctbs_w * ctbs_h;
  log2_min_tb = P.log2_min_tb; log2_max_tb = std::min(P.log2_max_tb, std::min(5, log2_ctb));
  w8 = W >> 3; h8 = H >> 3; w4 = W >> 2; h4 = H >> 2;
  tbs_w = ctbs_w << (log2_ctb - log2_min_tb); tbs_h = ctbs_h << (log2_ctb - log2_min_tb);
  qp_bd_offset = 6 * (bd - 8);
  // tiles (uniform spacing)
  int tc = std::max(1, std::min(P.tile_cols, ctbs_w)), trw = std::max(1, std::min(P.tile_rows, ctbs_h));
  P.tile_cols = tc; P.tile_rows = trw;
  col_bd.assign(tc + 1, 0); row_bd.assign(trw + 1, 0);
  for (int i = 0; i < tc; i++) col_bd[i + 1] = ((i + 1) * ctbs_w) / tc;
  for (int i = 0; i < trw; i++) row_bd[i + 1] = ((i + 1) * ctbs_h) / trw;
  rs2ts.assign(nctb, 0); ts2rs.assign(nctb, 0); tile_id.assign(nctb, 0); tile_start.assign(nctb, 0);
  for (int rs = 0; rs < nctb; rs++) {
    int tbX = rs % ctbs_w, tbY = rs / ctbs_w, tileX = 0, tileY = 0;
    for (int i = 0; i < tc; i++) if (tbX >= col_bd[i]) tileX = i;
    for (int j = 0; j < trw; j++) if (tbY >= row_bd[j]) tileY = j;
    int ts = 0;
    for (int i = 0; i < tileX; i++) ts += (row_bd[tileY + 1] - row_bd[tileY]) * (col_bd[i + 1] - col_bd[i]);
    for (int j = 0; j < tileY; j++) ts += ctbs_w * (row_bd[j + 1] - row_bd[j]);
    ts += (tbY - row_bd[tileY]) * (col_bd[tileX + 1] - col_bd[tileX]) + tbX - col_bd[tileX];
    rs2ts[rs] = ts; ts2rs[ts] = rs; tile_id[rs] = tileY * tc + tileX;
    if (tbX == col_bd[tileX] && tbY == row_bd[tileY]) tile_start[rs] = 1;
  }
  int shift = log2_ctb - log2_min_tb;
  zs.assign((size_t)tbs_w * tbs_h, 0);
  for (int y = 0; y < tbs_h; y++)
    for (int x = 0; x < tbs_w; x++) {
      int v = rs2ts[ctbs_w * (y >> shift) + (x >> shift)] << (shift * 2);
      for (int i = 0; i < shift; i++) { int m = 1 << i; v += (m & x ? m * m : 0) + (m & y ? 2 * m * m : 0); }
      zs[x + (size_t)y * tbs_w] = v;
    }
  ct_depth.assign((size_t)w8 * h8, 0); cu_flags.assign((size_t)w8 * h8, 0); qp_y.assign((size_t)w8 * h8, 0);
  ipm.assign((size_t)w4 * h4, 1);
  ctb_slice.assign(nctb, -1);
  wpp_ctx.assign(ctbs_h, CtxSet());
  sao.assign(nctb, Sao());
  memset(&pic, 0, sizeof(pic));
  pic.width = W; pic.height = H; pic.chroma_format = (uint8_t)cf; pic.bit_depth_y = pic.bit_depth_c = (uint8_t)bd;
  pic.log2_ctb = (uint8_t)log2_ctb; pic.ctbs_w = (uint16_t)ctbs_w; pic.ctbs_h = (uint16_t)ctbs_h;
  if (P.strong_intra) pic.flags |= HC_PIC_STRONG_INTRA;
  if (P.intra_smoothing_disabled) pic.flags |= HC_PIC_NO_INTRA_SMOOTH;
  wpp_stat.assign(ctbs_h, std::array<uint8_t, 4>{{0, 0, 0, 0}});
  max_tskip_log2 = P.transform_skip ? 2 + P.log2_max_transform_skip_minus2 : 2;
  log2_min_cu_chroma_qp_offset = log2_ctb - P.diff_cu_chroma_qp_offset_depth;
  for (int i = 0; i < P.chroma_qp_offset_list_len; i++) { cqo_cb[i] = rng.below(25) - 12; cqo_cr[i] = rng.below(25) - 12; }
  log2_min_cu_qp_delta = P.cu_qp_delta ? log2_ctb - std::min(P.cu_qp_delta - 1, log2_ctb - 3) : log2_ctb;

  // scaling lists
  if (P.scaling_list) {
    pic.flags |= HC_PIC_SCALING_LIST;
    for (int m = 0; m < 6; m++) {
      for (int i = 0; i < 16; i++) sl4[m][i] = 16;
      for (int i = 0; i < 64; i++) {
        sl8[m][i] = m < 3 ? kDefault8x8Intra[i] : kDefault8x8Inter[i];
        sl16[m][i] = sl8[m][i];
      }
      sl16_dc[m] = 16;
    }
    for (int m = 0; m < 2; m++) { for (int i = 0; i < 64; i++) sl32[m][i] = m == 0 ? kDefault8x8Intra[i] : kDefault8x8Inter[i]; sl32_dc[m] = 16; }
    if (P.scaling_list == 2) {
      for (int m = 0; m < 6; m++) {
        for (int i = 0; i < 16; i++) sl4[m][i] = (uint8_t)(8 + rng.below(40));
        for (int i = 0; i < 64; i++) { sl8[m][i] = (uint8_t)(8 + rng.below(60)); sl16[m][i] = (uint8_t)(8 + rng.below(80)); }
        sl16_dc[m] = 8 + rng.below(30);
      }
      for (int m = 0; m < 2; m++) { for (int i = 0; i < 64; i++) sl32[m][i] = (uint8_t)(8 + rng.below(100)); sl32_dc[m] = 8 + rng.below(30); }
    }
    scaling.assign(HC_SCALING_BLOB_BYTES, 16);
    const ScanTables& st = scan_tables();
    uint8_t* b = scaling.data();
    for (int m = 0; m < 6; m++) for (int i = 0; i < 16; i++) b[m * 16 + st.order[2][0][i].x + 4 * st.order[2][0][i].y] = sl4[m][i];
    b += 96;
    for (int m = 0; m < 6; m++) for (int i = 0; i < 64; i++) b[m * 64 + st.order[3][0][i].x + 8 * st.order[3][0][i].y] = sl8[m][i];
    b += 384;
    for (int m = 0; m < 6; m++) {
      for (int i = 0; i < 64; i++)
        for (int dy = 0; dy < 2; dy++) for (int dx = 0; dx < 2; dx++)
          b[m * 256 + (2 * st.order[3][0][i].x + dx) + 16 * (2 * st.order[3][0][i].y + dy)] = sl16[m][i];
      b[m * 256] = (uint8_t)sl16_dc[m];
    }
    b += 1536;
    for (int m = 0; m < 2; m++) {
      for (int i = 0; i < 64; i++)
        for (int dy = 0; dy < 4; dy++) for (int dx = 0; dx < 4; dx++)
          b[m * 1024 + (4 * st.order[3][0][i].x + dx) + 32 * (4 * st.order[3][0][i].y + dy)] = sl32[m][i];
      b[m * 1024] = (uint8_t)sl32_dc[m];
    }
  }
}

// ---- parameter sets ------------------------------------------------------------------------------
static void write_ptl(BitWriter& bw, int profile_idc) {
  bw.put(0, 2); bw.put(0, 1); bw.put((uint32_t)profile_idc, 5);
  for (int i = 0; i < 32; i++) bw.put(i == profile_idc || (profile_idc == 1 && i == 2) ? 1 : 0, 1);
  bw.put(1, 1); bw.put(0, 1); bw.put(0, 1); bw.put(1, 1);
  bw.put(0, 32); bw.put(0, 11);  // 43 reserved bits
  bw.put(0, 1);
  bw.put(186, 8);  // level 6.2
}

void Enc::write_scaling_list_data(BitWriter& bw) {
  // every list coded explicitly (scaling_list_pred_mode_flag = 1)
  for (int sizeId = 0; sizeId < 4; sizeId++)
    for (int m = 0; m < (sizeId == 3 ? 2 : 6); m++) {
      bw.put(1, 1);
      const uint8_t* l = sizeId == 0 ? sl4[m] : sizeId == 1 ? sl8[m] : sizeId == 2 ? sl16[m] : sl32[m];
      int n = sizeId == 0 ? 16 : 64, next = 8;
      if (sizeId > 1) {
        int dc = sizeId == 2 ? sl16_dc[m] : sl32_dc[m];
        bw.se(dc - 8);
        next = dc;
      }
      for (int i = 0; i < n; i++) {
        int d = l[i] - next;
        if (d > 127) d -= 256;
        if (d < -128) d += 256;
        bw.se(d);
        next = l[i];
      }
    }
}

void Enc::write_parameter_sets(std::vector<uint8_t>& out) {
  int profile = rext_sps() || rext_pps() ? 4 : (cf == 1 && bd == 8) ? 1 : (cf == 1 && bd <= 10) ? 2 : 4;
  {  // VPS
    BitWriter bw;
    bw.put(0, 4); bw.put(1, 1); bw.put(1, 1); bw.put(0, 6); bw.put(0, 3); bw.put(1, 1); bw.put(0xffff, 16);
    write_ptl(bw, profile);
    bw.put(1, 1); bw.ue(0); bw.ue(0); bw.ue(0);
    bw.put(0, 6); bw.ue(0); bw.put(0, 1); bw.put(0, 1);
    bw.trailing();
    append_nal(out, 32, bw.bytes);
  }
  {  // SPS
    BitWriter bw;
    bw.put(0, 4); bw.put(0, 3); bw.put(1, 1);
    write_ptl(bw, profile);
    bw.ue(0);
    bw.ue((uint32_t)cf);
    if (cf == 3) bw.put(0, 1);
    bw.ue((uint32_t)W); bw.ue((uint32_t)H);
    bool crop = W != P.width || H != P.height;
    bw.put(crop, 1);
    if (crop) { bw.ue(0); bw.ue((uint32_t)((W - P.width) / SubW)); bw.ue(0); bw.ue((uint32_t)((H - P.height) / SubH)); }
    bw.ue((uint32_t)(bd - 8)); bw.ue((uint32_t)(bd - 8));
    bw.ue(4);  // log2_max_pic_order_cnt_lsb_minus4
    bw.put(1, 1); bw.ue(0); bw.ue(0); bw.ue(0);
    bw.ue((uint32_t)(log2_min_cb - 3)); bw.ue((uint32_t)(log2_ctb - log2_min_cb));
    bw.ue((uint32_t)(log2_min_tb - 2)); bw.ue((uint32_t)(log2_max_tb - log2_min_tb));
    bw.ue(0); bw.ue((uint32_t)P.max_th_depth);
    bw.put(P.scaling_list ? 1 : 0, 1);
    if (P.scaling_list) {
      bw.put(P.scaling_list == 2, 1);
      if (P.scaling_list == 2) write_scaling_list_data(bw);
    }
    bw.put(0, 1);                    // amp
    bw.put(P.sao ? 1 : 0, 1);
    bw.put(P.pcm ? 1 : 0, 1);
    if (P.pcm) {
      bw.put((uint32_t)(bd - 1), 4); bw.put((uint32_t)(bd - 1), 4);
      bw.ue(0); bw.ue((uint32_t)(std::min(5, log2_ctb) - 3)); bw.put(0, 1);
    }
    bw.ue(0);                        // num_short_term_ref_pic_sets
    bw.put(0, 1);                    // long_term_ref_pics_present
    bw.put(0, 1);                    // temporal mvp
    bw.put(P.strong_intra ? 1 : 0, 1);
    bw.put(P.vui ? 1 : 0, 1);
    if (P.vui) {
      bw.put(0, 1); bw.put(0, 1);
      bw.put(1, 1); bw.put(5, 3); bw.put(P.full_range ? 1 : 0, 1); bw.put(1, 1);
      bw.put((uint32_t)P.primaries, 8); bw.put((uint32_t)P.transfer, 8); bw.put((uint32_t)P.matrix, 8);
      bw.put(0, 1); bw.put(0, 3); bw.put(0, 1); bw.put(0, 1); bw.put(0, 1);
    }
    bw.put(rext_sps(), 1);           // sps_extension_present
    if (rext_sps()) {
      bw.put(1, 1); bw.put(0, 7);    // sps_range_extension_flag, no multilayer / 3d / scc / 4 bits
      bw.put(P.transform_skip_rotation ? 1 : 0, 1);
      bw.put(P.transform_skip_context ? 1 : 0, 1);
      bw.put(P.implicit_rdpcm ? 1 : 0, 1);
      bw.put(0, 1);                  // explicit_rdpcm (inter only)
      bw.put(P.extended_precision ? 1 : 0, 1);
      bw.put(P.intra_smoothing_disabled ? 1 : 0, 1);
      bw.put(0, 1);                  // high_precision_offsets (inter only)
      bw.put(P.persistent_rice_adaptation ? 1 : 0, 1);
      bw.put(P.cabac_bypass_alignment ? 1 : 0, 1);
    }
    bw.trailing();
    append_nal(out, 33, bw.bytes);
  }
  {  // PPS
    BitWriter bw;
    bw.ue(0); bw.ue(0);
    bw.put(P.dependent_slices ? 1 : 0, 1);
    bw.put(0, 1); bw.put(0, 3);
    bw.put(P.sign_hiding ? 1 : 0, 1);
    bw.put(0, 1);
    bw.ue(0); bw.ue(0);
    bw.se(0);                        // init_qp_minus26
    bw.put(0, 1);
    bw.put(P.transform_skip ? 1 : 0, 1);
    bw.put(P.cu_qp_delta ? 1 : 0, 1);
    if (P.cu_qp_delta) bw.ue((uint32_t)(log2_ctb - log2_min_cu_qp_delta));
    bw.se(P.cb_qp_offset); bw.se(P.cr_qp_offset);
    bw.put(0, 1);
    bw.put(0, 1); bw.put(0, 1);
    bw.put(P.transquant_bypass ? 1 : 0, 1);
    bool tiles = P.tile_cols > 1 || P.tile_rows > 1;
    bw.put(tiles, 1);
    bw.put(P.wpp ? 1 : 0, 1);
    if (tiles) {
      bw.ue((uint32_t)(P.tile_cols - 1)); bw.ue((uint32_t)(P.tile_rows - 1));
      bw.put(1, 1);
      bw.put(P.loop_filter_across_tiles ? 1 : 0, 1);
    }
    bw.put(P.loop_filter_across_slices ? 1 : 0, 1);
    bool dbk_ctrl = P.deblock_disable || P.beta_offset_div2 || P.tc_offset_div2;
    bw.put(dbk_ctrl, 1);
    if (dbk_ctrl) {
      bw.put(0, 1);
      bw.put(P.deblock_disable ? 1 : 0, 1);
      if (!P.deblock_disable) { bw.se(P.beta_offset_div2); bw.se(P.tc_offset_div2); }
    }
    bw.put(0, 1);                    // pps_scaling_list_data_present
    bw.put(0, 1);
    bw.ue(0);
    bw.put(0, 1);
    bw.put(rext_pps(), 1);           // pps_extension_present
    if (rext_pps()) {
      bw.put(1, 1); bw.put(0, 7);    // pps_range_extension_flag, no multilayer / 3d / scc / 4 bits
      if (P.transform_skip) bw.ue((uint32_t)P.log2_max_transform_skip_minus2);
      bw.put(P.cross_component_prediction ? 1 : 0, 1);
      bw.put(P.chroma_qp_offset_list_len ? 1 : 0, 1);
      if (P.chroma_qp_offset_list_len) {
        bw.ue((uint32_t)P.diff_cu_chroma_qp_offset_depth);
        bw.ue((uint32_t)(P.chroma_qp_offset_list_len - 1));
        for (int i = 0; i < P.chroma_qp_offset_list_len; i++) { bw.se(cqo_cb[i]); bw.se(cqo_cr[i]); }
      }
      bw.ue((uint32_t)P.log2_sao_offset_scale_luma);
      bw.ue((uint32_t)P.log2_sao_offset_scale_chroma);
    }
    bw.trailing();
    append_nal(out, 34, bw.bytes);
  }
}

// ---- analysis helpers ------------------------------------------------------------------------------
double Enc::variance(int x0, int y0, int size) const {
  double s = 0, s2 = 0;
  int n = 0;
  for (int y = y0; y < std::min(y0 + size, H); y++)
    for (int x = x0; x < std::min(x0 + size, W); x++) {
      double v = orig[0][x + (size_t)y * pw[0]];
      s += v; s2 += v * v; n++;
    }
  if (!n) return 0;
  double m = s / n;
  return s2 / n - m * m;
}

hc_blk Enc::make_blk(int cIdx, int xB, int yB, int log2, int mode, bool no_edge) const {
  const int nT = 1 << log2;
  const int sw = cIdx == 0 ? 1 : SubW, sh = cIdx == 0 ? 1 : SubH;
  const int xBL = xB * sw, yBL = yB * sh;
  bool aL = true, aT = true, aTR = true, aTL = true;
  if (xBL == 0) { aL = false; aTL = false; }
  if (yBL == 0) { aT = false; aTL = false; aTR = false; }
  if (xBL + nT * sw >= W) aTR = false;
  int xCur = xBL >> log2_ctb, yCur = yBL >> log2_ctb;
  int xLeft = (xBL - 1) >> log2_ctb, xRight = (xBL + nT * sw) >> log2_ctb, yTop = (yBL - 1) >> log2_ctb;
  int cur = xCur + yCur * ctbs_w;
  auto same = [&](int cx, int cy) { int n = cx + cy * ctbs_w; return ctb_slice[n] == ctb_slice[cur] && tile_id[n] == tile_id[cur]; };
  if (aL && !same(xLeft, yCur)) aL = false;
  if (aT && !same(xCur, yTop)) aT = false;
  if (aTL && !same(xLeft, yTop)) aTL = false;
  if (aTR && !same(xRight, yTop)) aTR = false;
  int nBottom = std::min(2 * nT, (H - yBL + sh - 1) / sh), nRight = std::min(2 * nT, (W - xBL + sw - 1) / sw);
  const int currAddr = zs_addr(xBL, yBL);
  uint16_t left = 0, top = 0;
  if (aL) for (int y = nBottom - 1; y >= 0; y -= 4) if (zs_addr((xB - 1) * sw, (yB + y) * sh) <= currAddr) left |= (uint16_t)(1u << (y >> 2));
  bool tl = aTL && zs_addr((xB - 1) * sw, (yB - 1) * sh) <= currAddr;
  for (int x = 0; x < nRight; x += 4) {
    bool ba = x < nT ? aT : aTR;
    if (ba && zs_addr((xB + x) * sw, (yB - 1) * sh) <= currAddr) top |= (uint16_t)(1u << (x >> 2));
  }
  hc_blk b;
  memset(&b, 0, sizeof(b));
  b.x = (uint16_t)xB; b.y = (uint16_t)yB; b.log2 = (uint8_t)log2; b.mode = (uint8_t)mode; b.cidx = (uint8_t)cIdx;
  b.flags = (uint8_t)((tl ? HC_BLK_AVAIL_TL : 0) | (no_edge ? HC_BLK_NO_EDGE_FLT : 0));
  b.avail_left = left; b.avail_top = top;
  return b;
}

int Enc::choose_mode(int x0, int y0, int log2) {
  if (stress(HEVC_ENC_STRESS_MODES)) return rng.below(35);
  int l = std::min(log2, 5);
  int nT = 1 << l;
  int cands[12] = {0, 1, 10, 26, 2, 18, 34, 6, 14, 22, 30, 2 + rng.below(33)};
  int best = 1;
  long best_cost = -1;
  uint16_t pred[32 * 32];
  for (int k = 0; k < 12; k++) {
    hc_blk b = make_blk(0, x0, y0, l, cands[k], false);
    hc_oracle_predict_block(&pic, &b, rec[0].data(), pw[0], pred);
    long cost = 0;
    for (int y = 0; y < nT; y++)
      for (int x = 0; x < nT; x++) cost += std::abs((int)pred[x + y * nT] - (int)orig[0][(x0 + x) + (size_t)(y0 + y) * pw[0]]);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = cands[k]; }
  }
  if (rng.chance(8)) best = rng.below(35);  // variety: sometimes a random mode
  return best;
}

int Enc::chroma_qp(int qpy, int c, int cu_off) const {
  int off = (c == 1 ? P.cb_qp_offset : P.cr_qp_offset) + cu_off;
  int qPi = clip3(-qp_bd_offset, 57, qpy + off);
  int q = cf == 1 ? qpc_table_420(qPi) : qPi;
  return std::max(0, q + qp_bd_offset);
}

// CuQpOffsetCb / Cr a coded chroma block of the current TU is quantised with: the group's decision once it took effect,
// else the one drawn for the group (a TU with a coded chroma block is where it takes effect)
int Enc::cu_chroma_offset(int c) const {
  if (!P.chroma_qp_offset_list_len) return 0;
  if (cqo_coded_a) return c == 1 ? cqo_cur_cb : cqo_cur_cr;
  if (!cqo_next) return 0;
  return c == 1 ? cqo_cb[cqo_next - 1] : cqo_cr[cqo_next - 1];
}

// forward transform + quantisation of one block, then the decoder-exact reconstruction
void Enc::process_tb(int cIdx, int xB, int yB, int log2, int mode, TuData& tu) {
  const int nT = 1 << log2;
  uint16_t* plane = rec[cIdx].data();
  const int stride = pw[cIdx];
  uint16_t pred[32 * 32];
  // disableIntraBoundaryFilter as the decoder derives it: the bypass flag at the block's component coordinates
  const bool no_edge = P.implicit_rdpcm &&
                       (cu_flags[(std::min(xB, W - 1) >> 3) + (size_t)(std::min(yB, H - 1) >> 3) * w8] & 2);
  if (no_edge && cIdx == 0 && (mode == 10 || mode == 26) && nT < 32) stats[ST_no_edge_flt]++;
  if (P.intra_smoothing_disabled && (cIdx == 0 || cf == 3) && mode != 1 && nT != 4) {
    const int minDist = std::min(std::abs(mode - 26), std::abs(mode - 10));
    if (nT == 8 ? minDist > 7 : nT == 16 ? minDist > 1 : minDist > 0) {
      stats[ST_smoothing_skipped]++;
      if (cIdx == 0 && nT == 32 && P.strong_intra) stats[ST_smoothing_skipped_strong]++;
    }
  }
  hc_blk blk = make_blk(cIdx, xB, yB, log2, mode, no_edge);
  hc_oracle_predict_block(&pic, &blk, plane, stride, pred);
  int res[32 * 32];
  for (int y = 0; y < nT; y++)
    for (int x = 0; x < nT; x++) res[x + y * nT] = (int)orig[cIdx][(xB + x) + (size_t)(yB + y) * stride] - (int)pred[x + y * nT];

  const int cu_off = cIdx ? cu_chroma_offset(cIdx) : 0;
  const int qpP = cIdx == 0 ? cur_qp_y + qp_bd_offset : chroma_qp(cur_qp_y, cIdx, cu_off);
  tu.levels.assign((size_t)nT * nT, 0);
  tu.tskip = false;
  tu.coded = false;
  tu.rdpcm = 0;
  tu.rotate = false;
  // implicit RDPCM (8.6.2: intra, transform-skipped or bypass, mode 10 or 26) codes the differences along the
  // accumulation direction; rotation (nTbS = 4) codes the block turned by 180 degrees, i.e. in reversed raster order
  const int rdpcm = P.implicit_rdpcm && (mode == 10 || mode == 26) ? (mode == 26 ? 2 : 1) : 0;
  auto differences = [&](const int* r, int* d) {
    for (int y = 0; y < nT; y++)
      for (int x = 0; x < nT; x++) {
        const int i = x + y * nT;
        d[i] = r[i] - (rdpcm == 1 && x ? r[i - 1] : rdpcm == 2 && y ? r[i - nT] : 0);
      }
  };
  const bool rotate = P.transform_skip_rotation && log2 == 2;
  if (cu_bypass) {
    int d[32 * 32];
    differences(res, d);
    bool any = false;
    for (int i = 0; i < nT * nT; i++) { tu.levels[i] = (int16_t)d[rotate ? nT * nT - 1 - i : i]; any |= res[i] != 0; }
    tu.coded = any;
    tu.rdpcm = rdpcm;
    tu.rotate = rotate;
  } else {
    bool tskip = P.transform_skip && log2 <= max_tskip_log2 && rng.chance(25);
    long long coef[32 * 32];
    const int tshift = 15 - bd - log2;
    if (tskip) {
      int d[32 * 32];
      differences(res, d);
      for (int i = 0; i < nT * nT; i++) {
        const int v = d[rotate ? nT * nT - 1 - i : i];
        coef[i] = tshift >= 0 ? ((long long)v << tshift) : ((long long)v >> -tshift);
      }
    } else {
      const bool dst = log2 == 2 && cIdx == 0;
      const int fact = 1 << (5 - log2);
      long long tmp[32 * 32];
      const int s1 = log2 + bd - 9, s2 = log2 + 6;
      // columns then rows of T * R * T^T
      for (int k = 0; k < nT; k++)
        for (int x = 0; x < nT; x++) {
          long long a = 0;
          for (int y = 0; y < nT; y++) a += (long long)(dst ? kDst[k][y] : dct_coef(fact * k, y)) * res[x + y * nT];
          tmp[x + k * nT] = s1 > 0 ? (a + (1ll << (s1 - 1))) >> s1 : a;
        }
      for (int k = 0; k < nT; k++)
        for (int l = 0; l < nT; l++) {
          long long a = 0;
          for (int x = 0; x < nT; x++) a += (long long)(dst ? kDst[l][x] : dct_coef(fact * l, x)) * tmp[x + k * nT];
          coef[l + k * nT] = (a + (1ll << (s2 - 1))) >> s2;
        }
    }
    const int qbits = 14 + qpP / 6 + tshift;
    const long long add = (171ll << qbits) >> 9;
    bool any = false;
    for (int i = 0; i < nT * nT; i++) {
      long long scale = kQuantScale[qpP % 6];
      if (P.scaling_list) {
        const uint8_t* sc = scaling.data();
        int mid = log2 == 5 ? 0 : cIdx;
        int m = log2 == 2 ? sc[mid * 16 + i] : log2 == 3 ? sc[96 + mid * 64 + i] : log2 == 4 ? sc[480 + mid * 256 + i] : sc[2016 + i];
        scale = scale * 16 / std::max(1, m);
      }
      long long a = coef[i] < 0 ? -coef[i] : coef[i];
      long long lv = (a * scale + add) >> qbits;
      if (lv > 32767) lv = 32767;
      int16_t v = (int16_t)(coef[i] < 0 ? -lv : lv);
      tu.levels[i] = v;
      any |= v != 0;
    }
    tu.coded = any;
    tu.tskip = tskip && any;
    if (tskip) { tu.rdpcm = rdpcm; tu.rotate = rotate; }
    if (stress(HEVC_ENC_STRESS_LEVELS)) {
      // 0: keep the quantised levels, 1 / 2: sparse, 3: dense; values from the ends of TransCoeffLevel's range
      const int kind = stress(HEVC_ENC_STRESS_DENSE) ? 3 : rng.below(4);
      if (kind) {
        static const int kValues[8] = {1, -1, 2, -2, 3, -3, 32767, -32768};
        any = false;
        for (int i = 0; i < nT * nT; i++) {
          int v = 0;
          if (kind == 3 || rng.chance(30)) {
            const int r = rng.below(10);
            v = r < 8 ? kValues[r] : (int)(rng.next() & 0xffff) - 32768;
            if (kind == 3 && v == 0) v = 1;
          }
          tu.levels[i] = (int16_t)v;
          any |= v != 0;
        }
        tu.coded = any;
        tu.tskip = tskip && any;
      }
    }
  }
  if (!tu.tskip && !cu_bypass) { tu.rdpcm = 0; tu.rotate = false; }
  if (tu.coded && cIdx && !cu_bypass) {
    const int qPi = cur_qp_y + (cIdx == 1 ? P.cb_qp_offset : P.cr_qp_offset) + cu_off;
    if (qPi < -qp_bd_offset) stats[ST_chroma_qpi_clip_lo]++;
    if (qPi > 57) stats[ST_chroma_qpi_clip_hi]++;
  }

  // sign data hiding: fix the parity of every 4x4 sub-block that will hide a sign (never to +32768: -32768 becomes -32767)
  int scanIdx = 0;
  if (log2 == 2 || (log2 == 3 && (cIdx == 0 || cf == 3))) {
    if (mode >= 6 && mode <= 14) scanIdx = 2;
    else if (mode >= 22 && mode <= 30) scanIdx = 1;
  }
  if (tu.coded && P.sign_hiding && !cu_bypass && !(tu.tskip && tu.rdpcm)) {
    const ScanTables& st = scan_tables();
    const ScanPos* sp = st.order[2][scanIdx];
    for (int sy = 0; sy < nT / 4; sy++)
      for (int sx = 0; sx < nT / 4; sx++) {
        int first = -1, last = -1, sum = 0;
        for (int n = 0; n < 16; n++) {
          int v = tu.levels[(sx * 4 + sp[n].x) + (sy * 4 + sp[n].y) * nT];
          if (v) { if (first < 0) first = n; last = n; sum += std::abs(v); }
        }
        if (first < 0 || last - first <= 3) continue;
        int16_t& f = tu.levels[(sx * 4 + sp[first].x) + (sy * 4 + sp[first].y) * nT];
        bool neg = f < 0;
        if ((sum & 1) != (neg ? 1 : 0)) {
          // change the magnitude of the first coefficient by one (never to zero)
          int a = std::abs((int)f);
          a = a >= 32767 ? a - 1 : a + 1;
          f = (int16_t)(neg ? -a : a);
        }
      }
  }

  // decoder-exact reconstruction
  if (tu.coded) {
    std::vector<hc_coeff> co;
    for (int i = 0; i < nT * nT; i++)
      if (tu.levels[i]) { hc_coeff c; c.pos = (uint16_t)i; c.level = tu.levels[i]; co.push_back(c); }
    hc_tb tb;
    memset(&tb, 0, sizeof(tb));
    tb.ncoeff = (uint16_t)co.size();
    tb.log2 = (uint8_t)log2;
    tb.qp = (uint8_t)qpP;
    tb.matrix_id = (uint8_t)(log2 == 5 ? 0 : cIdx);
    uint8_t type = (uint8_t)cIdx;
    if (cu_bypass) type |= HC_TB_BYPASS;
    else if (tu.tskip) type |= HC_TB_TSKIP;
    else if (log2 == 2 && cIdx == 0) type |= HC_TB_DST;
    if (tu.rdpcm) type |= tu.rdpcm == 2 ? HC_TB_RDPCM_V : HC_TB_RDPCM_H;
    if (tu.rotate) type |= HC_TB_ROTATE;
    tb.type = type;
    int32_t r[32 * 32];
    hc_oracle_residual_block(&pic, &tb, co.data(), scaling.empty() ? nullptr : scaling.data(), r);
    for (int y = 0; y < nT; y++)
      for (int x = 0; x < nT; x++)
        plane[(xB + x) + (size_t)(yB + y) * stride] = (uint16_t)clip3(0, (1 << bd) - 1, (int)pred[x + y * nT] + r[x + y * nT]);
  } else {
    for (int y = 0; y < nT; y++)
      for (int x = 0; x < nT; x++) plane[(xB + x) + (size_t)(yB + y) * stride] = pred[x + y * nT];
  }
}

int Enc::mode_for(const int* modes, int x, int y) const {
  // modes[] holds up to 4 PU modes of the current CU (NxN: quadrants)
  if (modes[4] == 0) return modes[0];
  int half = (1 << cu_log2) >> 1;
  return modes[((y - cu_y0) >= half ? 2 : 0) + ((x - cu_x0) >= half ? 1 : 0)];
}

// pass A: decide the transform tree and reconstruct it in decoding order
void Enc::build_tree(Node& n, int max_depth, int intra_split, const int* luma_modes, const int* chroma_modes) {
  const int log2 = n.log2;
  bool can_choose = log2 <= log2_max_tb && log2 > log2_min_tb && n.depth < max_depth && !(intra_split && n.depth == 0);
  if (can_choose) {
    double v = variance(n.x0, n.y0, 1 << log2);
    n.split = v > 60.0 * (1 << (2 * (log2 - 2))) / 4.0 ? rng.chance(70) : rng.chance(12);
  } else {
    n.split = log2 > log2_max_tb || (intra_split && n.depth == 0);
  }
  if (n.split) {
    int h = 1 << (log2 - 1);
    for (int i = 0; i < 4; i++) {
      n.child[i].reset(new Node);
      Node& c = *n.child[i];
      c.x0 = n.x0 + (i & 1) * h; c.y0 = n.y0 + (i >> 1) * h; c.xBase = n.x0; c.yBase = n.y0;
      c.log2 = log2 - 1; c.depth = n.depth + 1; c.blkIdx = i;
      build_tree(c, max_depth, intra_split, luma_modes, chroma_modes);
    }
    // chroma flags of this node
    if (cf != 0) {
      if (log2 == 3 && cf != 3) {
        // children are 4x4 luma: the chroma blocks of this node were coded with child 3
        Node& c3 = *n.child[3];
        n.cbf_cb = n.cbf_cr = 0;
        for (int t = 0; t < c3.nchroma; t++) {
          if (c3.chroma[0][t].coded) n.cbf_cb |= 1 << t;
          if (c3.chroma[1][t].coded) n.cbf_cr |= 1 << t;
        }
      } else {
        n.cbf_cb = n.cbf_cr = 0;
        for (int i = 0; i < 4; i++) { if (n.child[i]->cbf_cb) n.cbf_cb = 1; if (n.child[i]->cbf_cr) n.cbf_cr = 1; }
      }
    }
    return;
  }
  // leaf: luma
  int modeY = mode_for(luma_modes, n.x0, n.y0);
  process_tb(0, n.x0, n.y0, log2, modeY, n.luma);
  n.cbf_luma = n.luma.coded;
  if (cf == 0) return;
  if (log2 > 2 || cf == 3) {
    n.log2C = std::max(2, cf == 3 ? log2 : log2 - 1);
    n.nchroma = cf == 2 ? 2 : 1;
    n.cxB = n.x0 / SubW; n.cyB = n.y0 / SubH;
  } else if (n.blkIdx == 3) {
    n.log2C = 2;
    n.nchroma = cf == 2 ? 2 : 1;
    n.cxB = n.xBase / SubW; n.cyB = n.yBase / SubH;
  } else {
    n.nchroma = 0;
  }
  int modeC = mode_for(chroma_modes, n.nchroma && log2 == 2 && cf != 3 ? n.xBase : n.x0, n.nchroma && log2 == 2 && cf != 3 ? n.yBase : n.y0);
  for (int c = 1; c <= 2; c++)
    for (int t = 0; t < n.nchroma; t++) process_tb(c, n.cxB, n.cyB + t * (1 << n.log2C), n.log2C, modeC, n.chroma[c - 1][t]);
  if (P.chroma_qp_offset_list_len && !cu_bypass && !cqo_coded_a) {
    bool any = false;
    for (int c = 0; c < 2; c++) for (int t = 0; t < n.nchroma; t++) any |= n.chroma[c][t].coded;
    if (any) {
      cqo_cur_cb = cu_chroma_offset(1);
      cqo_cur_cr = cu_chroma_offset(2);
      cqo_coded_a = true;
      cqo_queue.push_back(cqo_next);
    }
  }
  if (log2 > 2 || cf == 3) {
    n.cbf_cb = n.cbf_cr = 0;
    for (int t = 0; t < n.nchroma; t++) {
      if (n.chroma[0][t].coded) n.cbf_cb |= 1 << t;
      if (n.chroma[1][t].coded) n.cbf_cr |= 1 << t;
    }
  }
}

void Enc::derive_qp_pred(int xCU, int yCU, int& pred_out) {
  int qgmask = (1 << log2_min_cu_qp_delta) - 1;
  int xQG = xCU - (xCU & qgmask), yQG = yCU - (yCU & qgmask);
  if (xQG != currentQG_x || yQG != currentQG_y) {
    lastQPYinPreviousQG = currentQPY;
    currentQG_x = xQG; currentQG_y = yQG;
  }
  int ctbmask = ctb - 1;
  bool firstInCTBRow = (xQG == 0 && (yQG & ctbmask) == 0);
  int sx = (slice_addr_rs % ctbs_w) << log2_ctb, sy = (slice_addr_rs / ctbs_w) << log2_ctb;
  bool firstQGInSlice = (sx == xQG && sy == yQG);
  bool firstQGInTile = false;
  if ((P.tile_cols > 1 || P.tile_rows > 1) && (xQG & ctbmask) == 0 && (yQG & ctbmask) == 0) firstQGInTile = tile_start[ctb_of(xQG, yQG)] != 0;
  int pred = (firstQGInSlice || firstQGInTile || (firstInCTBRow && P.wpp)) ? slice_qp : lastQPYinPreviousQG;
  int shiftc = 2 * (log2_ctb - log2_min_tb);
  int qA = pred, qB = pred;
  if (available_zscan(xQG, yQG, xQG - 1, yQG) && (zs_addr(xQG - 1, yQG) >> shiftc) == ctb_addr_ts) qA = qp_y[((xQG - 1) >> 3) + (size_t)(yQG >> 3) * w8];
  if (available_zscan(xQG, yQG, xQG, yQG - 1) && (zs_addr(xQG, yQG - 1) >> shiftc) == ctb_addr_ts) qB = qp_y[(xQG >> 3) + (size_t)((yQG - 1) >> 3) * w8];
  pred_out = (qA + qB + 1) >> 1;
}

void Enc::set_cu_qp(int qpy) {
  int n8 = std::max(1, (1 << cu_log2) >> 3);
  for (int y = 0; y < n8; y++)
    for (int x = 0; x < n8; x++) {
      int xx = (cu_x0 >> 3) + x, yy = (cu_y0 >> 3) + y;
      if (xx < w8 && yy < h8) qp_y[xx + (size_t)yy * w8] = (int8_t)qpy;
    }
  currentQPY = qpy;
}

// ---- pass B: syntax ------------------------------------------------------------------------------
void Enc::residual_coding(const TuData& tu, int log2, int cIdx, int pred_mode) {
  const ScanTables& st = scan_tables();
  const int nT = 1 << log2;
  if (P.transform_skip && !cu_bypass && log2 <= max_tskip_log2) bin(CTX_TSKIP + (cIdx ? 1 : 0), tu.tskip ? 1 : 0);
  if (tu.tskip) { stats[ST_tskip_coded]++; stats[ST_tskip_log2 + log2 - 2]++; }
  if (tu.rdpcm) stats[cu_bypass ? (tu.rdpcm == 1 ? ST_rdpcm_h_bypass : ST_rdpcm_v_bypass) : (tu.rdpcm == 1 ? ST_rdpcm_h_tskip : ST_rdpcm_v_tskip)]++;
  if (tu.rotate) stats[cu_bypass ? ST_rotate_bypass : ST_rotate_tskip]++;
  const bool ts_ctx = P.transform_skip_context && (cu_bypass || tu.tskip);   // sig_coeff_flag contexts 42 / 43 (9.3.4.2.5)
  const int sbType = (cIdx == 0 ? 2 : 0) + (cu_bypass || tu.tskip ? 1 : 0);
  ctb_ntb++;
  for (int i = 0; i < nT * nT; i++) {
    ctb_ncoeff += tu.levels[i] != 0;
    if (tu.levels[i] == -32768) stats[ST_level_min]++;
    if (tu.levels[i] == 32767) stats[ST_level_max]++;
  }
  int scanIdx = 0;
  if (log2 == 2 || (log2 == 3 && (cIdx == 0 || cf == 3))) {
    if (pred_mode >= 6 && pred_mode <= 14) scanIdx = 2;
    else if (pred_mode >= 22 && pred_mode <= 30) scanIdx = 1;
  }
  const ScanPos* scanSub = st.order[log2 - 2][scanIdx];
  const ScanPos* scanPos = st.order[2][scanIdx];
  const int sbW = 1 << (log2 - 2);
  // last significant coefficient in scan order
  int lastSub = -1, lastPos = -1;
  for (int i = sbW * sbW - 1; i >= 0 && lastSub < 0; i--)
    for (int k = 15; k >= 0; k--) {
      int x = scanSub[i].x * 4 + scanPos[k].x, y = scanSub[i].y * 4 + scanPos[k].y;
      if (tu.levels[x + y * nT]) { lastSub = i; lastPos = k; break; }
    }
  int LastX = scanSub[lastSub].x * 4 + scanPos[lastPos].x, LastY = scanSub[lastSub].y * 4 + scanPos[lastPos].y;
  int cx = LastX, cy = LastY;
  if (scanIdx == 2) std::swap(cx, cy);
  // last_sig_coeff prefix/suffix: v < 4 -> prefix v; else v = ((2 + (p&1)) << ((p>>1)-1)) + suffix
  auto prefix_of = [](int v, int& prefix, int& suffix, int& nbits) {
    if (v < 4) { prefix = v; suffix = 0; nbits = 0; return; }
    for (int p = 4;; p++) {
      int n = (p >> 1) - 1, base = (2 + (p & 1)) << n;
      if (v >= base && v < base + (1 << n)) { prefix = p; suffix = v - base; nbits = n; return; }
    }
  };
  int px, sx, nx, py, sy, ny;
  prefix_of(cx, px, sx, nx);
  prefix_of(cy, py, sy, ny);
  auto code_prefix = [&](int base, int v) {
    int cMax = (log2 << 1) - 1, offset, shift;
    if (cIdx == 0) { offset = 3 * (log2 - 2) + ((log2 - 1) >> 2); shift = (log2 + 1) >> 2; }
    else { offset = 15; shift = log2 - 2; }
    for (int i = 0; i < v; i++) bin(base + offset + (i >> shift), 1);
    if (v < cMax) bin(base + offset + (v >> shift), 0);
  };
  code_prefix(CTX_LAST_X, px);
  code_prefix(CTX_LAST_Y, py);
  if (px > 3 || py > 3) stats[ST_last_suffix]++;
  if (LastX == 31 || LastY == 31) stats[ST_last_31]++;
  if (px > 3) cabac.bypass_bits((uint32_t)sx, nx);
  if (py > 3) cabac.bypass_bits((uint32_t)sy, ny);

  uint8_t csbf_nb[64];
  memset(csbf_nb, 0, sizeof(csbf_nb));
  const bool sign_hiding_possible = P.sign_hiding && !cu_bypass && !(tu.tskip && tu.rdpcm);
  int c1 = 1;
  for (int i = lastSub; i >= 0; i--) {
    const int Sx = scanSub[i].x, Sy = scanSub[i].y, xS0 = Sx << 2, yS0 = Sy << 2;
    bool any = false;
    for (int k = 0; k < 16; k++) if (tu.levels[(xS0 + scanPos[k].x) + (yS0 + scanPos[k].y) * nT]) any = true;
    int inferSbDc = 0;
    int coded;
    if (i < lastSub && i > 0) {
      coded = any;
      bin(CTX_CSBF + (csbf_nb[Sx + Sy * sbW] ? 1 : 0) + (cIdx ? 2 : 0), coded);
      inferSbDc = 1;
    } else {
      coded = 1;
    }
    if (coded) {
      if (Sx > 0) csbf_nb[Sx - 1 + Sy * sbW] |= 1;
      if (Sy > 0) csbf_nb[Sx + (Sy - 1) * sbW] |= 2;
    }
    if (!coded) continue;
    const int prevCsbf = csbf_nb[Sx + Sy * sbW];
    auto sig_ctx = [&](int xC, int yC) -> int {
      if (ts_ctx) { stats[cIdx ? ST_sig_ctx_43 : ST_sig_ctx_42]++; return cIdx ? 43 : 42; }
      int sigCtx;
      if (log2 == 2) sigCtx = kSigCtx4x4[(yC << 2) + xC];
      else if (xC + yC == 0) sigCtx = 0;
      else {
        int xP = xC & 3, yP = yC & 3;
        switch (prevCsbf) {
          case 0: sigCtx = (xP + yP >= 3) ? 0 : (xP + yP > 0) ? 1 : 2; break;
          case 1: sigCtx = (yP == 0) ? 2 : (yP == 1) ? 1 : 0; break;
          case 2: sigCtx = (xP == 0) ? 2 : (xP == 1) ? 1 : 0; break;
          default: sigCtx = 2; break;
        }
        if (cIdx == 0) { if ((xC >> 2) + (yC >> 2) > 0) sigCtx += 3; sigCtx += (log2 == 3) ? (scanIdx == 0 ? 9 : 15) : 21; }
        else sigCtx += (log2 == 3) ? 9 : 12;
      }
      return cIdx == 0 ? sigCtx : 27 + sigCtx;
    };
    int value[16], spos[16], n = 0;
    int last_coeff = (i == lastSub) ? lastPos - 1 : 15;
    if (i == lastSub) { spos[n] = lastPos; value[n] = tu.levels[LastX + LastY * nT]; n++; }
    for (int k = last_coeff; k > 0; k--) {
      int xC = xS0 + scanPos[k].x, yC = yS0 + scanPos[k].y;
      int v = tu.levels[xC + yC * nT];
      bin(CTX_SIG + sig_ctx(xC, yC), v != 0);
      if (v) { spos[n] = k; value[n] = v; n++; inferSbDc = 0; }
    }
    if (last_coeff >= 0) {
      int v = tu.levels[xS0 + yS0 * nT];
      if (!inferSbDc) {
        bin(CTX_SIG + sig_ctx(xS0, yS0), v != 0);
        if (v) { spos[n] = 0; value[n] = v; n++; }
      } else {
        // inferred significant: the encoder must really have a non-zero DC here
        spos[n] = 0; value[n] = v; n++;
        stats[ST_inferred_sb_dc]++;
      }
    }
    if (n == 0) continue;
    int ctxSet = (i == 0 || cIdx > 0) ? 0 : 2;
    if (c1 == 0) ctxSet++;
    c1 = 1;
    int firstG1 = -1;
    int ng1 = std::min(8, n);
    int base[16];
    for (int c = 0; c < n; c++) base[c] = 1;
    for (int c = 0; c < ng1; c++) {
      int a = std::abs(value[c]);
      int g1 = a > 1;
      bin(CTX_G1 + ctxSet * 4 + c1 + (cIdx > 0 ? 16 : 0), g1);
      if (g1) { base[c] = 2; c1 = 0; if (firstG1 < 0) firstG1 = c; }
      else if (c1 < 3 && c1 > 0) c1++;
    }
    if (firstG1 >= 0) {
      int g2 = std::abs(value[firstG1]) > 2;
      bin(CTX_G2 + ctxSet + (cIdx > 0 ? 4 : 0), g2);
      if (g2) base[firstG1] = 3;
    }
    bool signHidden = sign_hiding_possible && (spos[0] - spos[n - 1] > 3);
    if (P.sign_hiding && tu.tskip && tu.rdpcm && spos[0] - spos[n - 1] > 3) stats[ST_sdh_off_rdpcm]++;
    int nsign = signHidden ? n - 1 : n;
    if (n == 16) stats[ST_sb_16_sig]++;
    if (n > 8) stats[ST_sb_beyond_8]++;
    if (signHidden) stats[value[n - 1] < 0 ? ST_sign_hidden_odd : ST_sign_hidden_even]++;
    if (nsign == 16) stats[ST_sign_string_16]++;
    for (int c = 0; c < nsign; c++) cabac.bypass(value[c] < 0);
    // persistent Rice adaptation (9.3.3.11): the sub-block starts at StatCoeff / 4, which its first
    // coeff_abs_level_remaining updates; the parameter then rises without the cap at 4
    int rice = P.persistent_rice_adaptation ? stat_coeff[sbType] / 4 : 0;
    if (rice > 0) stats[ST_rice_init_gt0]++;
    bool first_remaining = true;
    for (int c = 0; c < n; c++) {
      const int a = std::abs(value[c]);
      // which coefficients carry coeff_abs_level_remaining (mirror of the decoder's base levels):
      //   first 8: greater1 = 0 -> level 1, nothing more;  greater1 = 1 and not the greater2 carrier ->
      //   base 2 + remaining;  the greater2 carrier: greater2 = 0 -> level 2, else base 3 + remaining;
      //   from the 9th coefficient on: base 1 + remaining
      int baseLevel;
      if (c < ng1) {
        if (a == 1) continue;
        if (c == firstG1) { if (a == 2) continue; baseLevel = 3; }
        else baseLevel = 2;
      } else {
        baseLevel = 1;
      }
      const int rem = a - baseLevel;
      if (rice == 4) stats[ST_rice4]++;
      if (rem < (3 << rice)) {
        int len = rem >> rice;
        if (len + 1 + rice > 16) stats[ST_escape_long]++;
        for (int k = 0; k < len; k++) cabac.bypass(1);
        cabac.bypass(0);
        cabac.bypass_bits((uint32_t)(rem & ((1 << rice) - 1)), rice);
      } else {
        int length = rice, code = rem - (3 << rice);
        while (code >= (1 << length)) { code -= 1 << length; length++; }
        int ones = 3 + length - rice;
        if (ones + 1 + length > 16) stats[ST_escape_long]++;
        if (ones >= 16) stats[ST_escape_prefix16]++;
        for (int k = 0; k < ones; k++) cabac.bypass(1);
        cabac.bypass(0);
        cabac.bypass_bits((uint32_t)code, length);
      }
      if (P.persistent_rice_adaptation && first_remaining) {
        uint8_t& sc = stat_coeff[sbType];
        if (rem >= (3 << (sc / 4))) sc++;
        else if (2 * rem < (1 << (sc / 4)) && sc > 0) sc--;
      }
      first_remaining = false;
      if (baseLevel + rem > 3 * (1 << rice)) rice = P.persistent_rice_adaptation ? rice + 1 : std::min(rice + 1, 4);
      if (rice > 4) stats[ST_rice_gt4]++;
    }
  }
}

void Enc::write_tu(Node& n, const int* luma_modes, const int* chroma_modes) {
  const int log2 = n.log2;
  int cbfChroma = n.cbf_cb | n.cbf_cr;
  // chroma flags seen by this TU: own (log2>2 / 4:4:4) or inherited from the parent (4x4 luma)
  if (n.cbf_luma || cbfChroma) {
    if (P.cu_qp_delta && !IsCuQpDeltaCoded) {
      int pred;
      derive_qp_pred(cu_x0, cu_y0, pred);
      int delta = qg_target_qp - pred;
      // CuQpDeltaVal is in [-(26 + QpBdOffsetY / 2), 25 + QpBdOffsetY / 2]; a target further away is reached through the
      // wrap QpY = ((pred + delta + 52 + 2 * QpBdOffsetY) % (52 + QpBdOffsetY)) - QpBdOffsetY (8.6.1). Without the QP
      // stress the target stays within +-12 of the prediction and never wraps.
      const int dmin = -(26 + qp_bd_offset / 2), dmax = 25 + qp_bd_offset / 2;
      if (delta > dmax) delta -= 52 + qp_bd_offset;
      if (delta < dmin) delta += 52 + qp_bd_offset;
      if (std::abs(delta) >= 5) stats[ST_qp_delta_ge5]++;
      if (delta == dmin) stats[ST_qp_delta_min]++;
      if (delta == dmax) stats[ST_qp_delta_max]++;
      if (pred + delta < -qp_bd_offset) stats[ST_qp_wrap_below]++;
      if (pred + delta > 51) stats[ST_qp_wrap_above]++;
      if (qg_target_qp < 0) stats[ST_qp_y_neg]++;
      if (qg_target_qp == 51) stats[ST_qp_y_51]++;
      int a = std::abs(delta);
      bin(CTX_CU_QP_DELTA, a > 0);
      if (a > 0) {
        int pre = std::min(a, 5);
        for (int k = 1; k < pre; k++) bin(CTX_CU_QP_DELTA + 1, 1);
        if (pre < 5) bin(CTX_CU_QP_DELTA + 1, 0);
        if (a >= 5) {
          int v = a - 5, k = 0;
          while (v >= (1 << k)) { cabac.bypass(1); v -= 1 << k; k++; }
          cabac.bypass(0);
          cabac.bypass_bits((uint32_t)v, k);
        }
        cabac.bypass(delta < 0);
      }
      IsCuQpDeltaCoded = true;
      CuQpDeltaVal = delta;
      set_cu_qp(qg_target_qp);
    }
    if (P.chroma_qp_offset_list_len && cbfChroma && !cu_bypass && !cqo_coded_b) {
      // cu_chroma_qp_offset_flag, cu_chroma_qp_offset_idx: TR with cMax = chroma_qp_offset_list_len_minus1, one context
      const int k = cqo_queue.at(cqo_read++);
      bin(CTX_CHROMA_QP_OFFSET_FLAG, k > 0);
      if (k > 0 && P.chroma_qp_offset_list_len > 1) {
        const int idx = k - 1, cmax = P.chroma_qp_offset_list_len - 1;
        for (int i = 0; i < idx; i++) bin(CTX_CHROMA_QP_OFFSET_IDX, 1);
        if (idx < cmax) bin(CTX_CHROMA_QP_OFFSET_IDX, 0);
      }
      stats[k > 0 ? ST_cu_chroma_qp_offset_idx + k - 1 : ST_cu_chroma_qp_offset_off]++;
      cqo_coded_b = true;
    }
  }
  int modeY = mode_for(luma_modes, n.x0, n.y0);
  if (n.cbf_luma) residual_coding(n.luma, log2, 0, modeY);
  if (cf == 0 || n.nchroma == 0) return;
  int modeC = mode_for(chroma_modes, log2 == 2 && cf != 3 ? n.xBase : n.x0, log2 == 2 && cf != 3 ? n.yBase : n.y0);
  for (int c = 1; c <= 2; c++)
    for (int t = 0; t < n.nchroma; t++)
      if (n.chroma[c - 1][t].coded) residual_coding(n.chroma[c - 1][t], n.log2C, c, modeC);
}

void Enc::write_tree(Node& n, int max_depth, int intra_split, int parent_cbf_cb, int parent_cbf_cr, const int* luma_modes,
                     const int* chroma_modes) {
  const int log2 = n.log2;
  if (log2 <= log2_max_tb && log2 > log2_min_tb && n.depth < max_depth && !(intra_split && n.depth == 0))
    bin(CTX_SPLIT_TRANSFORM + 5 - log2, n.split);
  int cbf_cb = n.cbf_cb, cbf_cr = n.cbf_cr;
  if ((log2 > 2 && cf != 0) || cf == 3) {
    if (parent_cbf_cb) {
      bin(CTX_CBF_CHROMA + n.depth, cbf_cb & 1);
      if (cf == 2 && (!n.split || log2 == 3)) bin(CTX_CBF_CHROMA + n.depth, (cbf_cb >> 1) & 1);
    }
    if (parent_cbf_cr) {
      bin(CTX_CBF_CHROMA + n.depth, cbf_cr & 1);
      if (cf == 2 && (!n.split || log2 == 3)) bin(CTX_CBF_CHROMA + n.depth, (cbf_cr >> 1) & 1);
    }
  } else if (cf != 0) {
    // 4x4 luma blocks inherit the parent's chroma flags
    cbf_cb = parent_cbf_cb; cbf_cr = parent_cbf_cr;
    n.cbf_cb = cbf_cb; n.cbf_cr = cbf_cr;
  }
  if (n.split) {
    // at a split node with a single flag in 4:2:2 the value is "any child"; already aggregated
    for (int i = 0; i < 4; i++) write_tree(*n.child[i], max_depth, intra_split, cbf_cb, cbf_cr, luma_modes, chroma_modes);
  } else {
    bin(CTX_CBF_LUMA + (n.depth == 0 ? 1 : 0), n.cbf_luma);
    write_tu(n, luma_modes, chroma_modes);
  }
}

void Enc::coding_unit(int x0, int y0, int log2, int depth) {
  const int nCbS = 1 << log2;
  cu_x0 = x0; cu_y0 = y0; cu_log2 = log2;
  cu_bypass = P.transquant_bypass && rng.chance(10);
  cqo_queue.clear();
  cqo_read = 0;
  if (P.transquant_bypass) bin(CTX_TQ_BYPASS, cu_bypass);
  {
    int n8 = nCbS >> 3;
    for (int y = 0; y < n8; y++)
      for (int x = 0; x < n8; x++) {
        size_t i = ((x0 >> 3) + x) + (size_t)((y0 >> 3) + y) * w8;
        ct_depth[i] = (uint8_t)depth;
        cu_flags[i] = cu_bypass ? 2 : 0;
      }
  }
  // QP of this CU: predicted QP until a delta is coded (decoder behaviour), target QP for quantisation
  int pred;
  derive_qp_pred(x0, y0, pred);
  if (P.cu_qp_delta) {
    int qpy = IsCuQpDeltaCoded ? qg_target_qp : pred;
    set_cu_qp(qpy);
    cur_qp_y = qg_target_qp;
  } else {
    set_cu_qp(slice_qp);
    cur_qp_y = slice_qp;
  }

  bool nxn = false;
  if (log2 == log2_min_cb) {
    nxn = log2 > log2_min_tb && (stress(HEVC_ENC_STRESS_MODES) ? rng.chance(50) : variance(x0, y0, nCbS) > 200 ? rng.chance(60) : rng.chance(10));
    bin(CTX_PART_MODE, nxn ? 0 : 1);
  }
  bool pcm = false;
  if (!nxn && P.pcm && log2 >= 3 && log2 <= std::min(5, log2_ctb)) {
    pcm = rng.chance(6);
    cabac.terminate(pcm ? 1 : 0);
  }
  if (pcm) {
    int n8 = nCbS >> 3;
    for (int y = 0; y < n8; y++) for (int x = 0; x < n8; x++) cu_flags[((x0 >> 3) + x) + (size_t)((y0 >> 3) + y) * w8] |= 1;
    for (int y = 0; y < (nCbS >> 2); y++) for (int x = 0; x < (nCbS >> 2); x++) ipm[((x0 >> 2) + x) + (size_t)((y0 >> 2) + y) * w4] = 1;
    cabac.finish();
    // pcm samples: full bit depth
    uint32_t acc = 0; int nb = 0;
    auto put = [&](uint32_t v, int n) { for (int i = n - 1; i >= 0; i--) { acc = (acc << 1) | ((v >> i) & 1); if (++nb == 8) { slice_data.push_back((uint8_t)acc); acc = 0; nb = 0; } } };
    int ncomp = cf ? 3 : 1;
    for (int c = 0; c < ncomp; c++) {
      int w = c ? nCbS / SubW : nCbS, h = c ? nCbS / SubH : nCbS;
      int xb = c ? x0 / SubW : x0, yb = c ? y0 / SubH : y0;
      for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
          uint16_t v = orig[c][(xb + x) + (size_t)(yb + y) * pw[c]];
          put(v, bd);
          rec[c][(xb + x) + (size_t)(yb + y) * pw[c]] = v;
        }
    }
    while (nb) put(0, 1);
    cabac.start(&slice_data);
    return;
  }

  // ---- intra modes + pass A ----
  int nparts = nxn ? 4 : 1;
  int pb = nxn ? nCbS / 2 : nCbS;
  int luma_modes[5] = {1, 1, 1, 1, nxn ? 1 : 0}, chroma_modes[5] = {1, 1, 1, 1, (nxn && cf == 3) ? 1 : 0};
  int icpm[4] = {4, 4, 4, 4};
  int max_depth = P.max_th_depth + (nxn ? 1 : 0);
  Node root;
  root.x0 = x0; root.y0 = y0; root.xBase = x0; root.yBase = y0; root.log2 = log2; root.depth = 0; root.blkIdx = 0;
  auto derive_chroma = [&](int idx) {
    int ic = stress(HEVC_ENC_STRESS_MODES) ? rng.below(5) : rng.chance(65) ? 4 : rng.below(4);
    icpm[idx] = ic;
    static const int cands[4] = {0, 26, 10, 1};
    int m = ic == 4 ? luma_modes[idx] : (cands[ic] == luma_modes[idx] ? 34 : cands[ic]);
    stats[ST_chroma_pred_mode + ic]++;
    if (ic != 4 && cands[ic] == luma_modes[idx]) stats[ST_chroma_mode_34]++;
    if (cf == 2) { stats[ST_mode422 + m]++; m = kMode422[m]; }
    chroma_modes[idx] = m;
  };
  if (!nxn) {
    luma_modes[0] = choose_mode(x0, y0, log2);
    if (cf) derive_chroma(0);
    build_tree(root, max_depth, 0, luma_modes, chroma_modes);
  } else {
    // NxN: the tree is split at depth 0; decide each quadrant's mode right before reconstructing it
    root.split = true;
    int h = nCbS / 2;
    for (int i = 0; i < 4; i++) {
      int xx = x0 + (i & 1) * h, yy = y0 + (i >> 1) * h;
      luma_modes[i] = choose_mode(xx, yy, log2 - 1);
      if (cf == 3) derive_chroma(i);
      else if (cf && i == 0) { derive_chroma(0); chroma_modes[1] = chroma_modes[2] = chroma_modes[3] = chroma_modes[0]; }
      root.child[i].reset(new Node);
      Node& c = *root.child[i];
      c.x0 = xx; c.y0 = yy; c.xBase = x0; c.yBase = y0; c.log2 = log2 - 1; c.depth = 1; c.blkIdx = i;
      build_tree(c, max_depth, 1, luma_modes, chroma_modes);
    }
    if (cf != 0) {
      if (log2 == 3 && cf != 3) {
        Node& c3 = *root.child[3];
        for (int t = 0; t < c3.nchroma; t++) { if (c3.chroma[0][t].coded) root.cbf_cb |= 1 << t; if (c3.chroma[1][t].coded) root.cbf_cr |= 1 << t; }
      } else {
        for (int i = 0; i < 4; i++) { if (root.child[i]->cbf_cb) root.cbf_cb = 1; if (root.child[i]->cbf_cr) root.cbf_cr = 1; }
      }
    }
  }

  // ---- pass B: prediction mode syntax ----
  bool availA0 = ctb_available(x0, y0, x0 - 1, y0), availB0 = ctb_available(x0, y0, x0, y0 - 1);
  int prev_flag[4], mpm_idx[4], rem[4];
  for (int idx = 0; idx < nparts; idx++) {
    int i = (idx & 1) * pb, j = (idx >> 1) * pb, x = x0 + i, y = y0 + j;
    bool availA = availA0 || i > 0, availB = availB0 || j > 0;
    int candA = 1, candB = 1;
    if (availA) candA = (cu_flags[((x - 1) >> 3) + (size_t)(y >> 3) * w8] & 1) ? 1 : ipm[((x - 1) >> 2) + (size_t)(y >> 2) * w4];
    if (availB) {
      if (cu_flags[(x >> 3) + (size_t)((y - 1) >> 3) * w8] & 1) candB = 1;
      else if (y - 1 < ((y >> log2_ctb) << log2_ctb)) candB = 1;
      else candB = ipm[(x >> 2) + (size_t)((y - 1) >> 2) * w4];
    }
    int cand[3];
    if (candA == candB) {
      if (candA < 2) { cand[0] = 0; cand[1] = 1; cand[2] = 26; }
      else { cand[0] = candA; cand[1] = 2 + ((candA - 2 - 1 + 32) % 32); cand[2] = 2 + ((candA - 2 + 1) % 32); }
    } else {
      cand[0] = candA; cand[1] = candB;
      cand[2] = (candA != 0 && candB != 0) ? 0 : (candA != 1 && candB != 1) ? 1 : 26;
    }
    int mode = luma_modes[idx];
    prev_flag[idx] = 0; mpm_idx[idx] = 0; rem[idx] = 0;
    for (int k = 0; k < 3; k++) if (cand[k] == mode) { prev_flag[idx] = 1; mpm_idx[idx] = k; break; }
    if (!prev_flag[idx]) {
      std::sort(cand, cand + 3);
      int r = mode;
      for (int k = 2; k >= 0; k--) if (r > cand[k]) r--;
      rem[idx] = r;
    }
    stats[ST_luma_mode + mode]++;
    if (prev_flag[idx]) stats[ST_mpm_idx + mpm_idx[idx]]++;
    else stats[ST_rem_mode]++;
    int n4 = pb >> 2;
    for (int yy = 0; yy < n4; yy++) for (int xx = 0; xx < n4; xx++) ipm[((x >> 2) + xx) + (size_t)((y >> 2) + yy) * w4] = (uint8_t)mode;
  }
  if (nparts == 4) {
    bool distinct = true;
    for (int i = 0; i < 4; i++) for (int j = 0; j < i; j++) distinct &= luma_modes[i] != luma_modes[j];
    if (distinct) stats[ST_nxn_4_modes]++;
  }
  for (int idx = 0; idx < nparts; idx++) bin(CTX_PREV_INTRA_LUMA, prev_flag[idx]);
  for (int idx = 0; idx < nparts; idx++) {
    if (prev_flag[idx]) { cabac.bypass(mpm_idx[idx] > 0); if (mpm_idx[idx] > 0) cabac.bypass(mpm_idx[idx] > 1); }
    else cabac.bypass_bits((uint32_t)rem[idx], 5);
  }
  auto code_icpm = [&](int v) {
    bin(CTX_INTRA_CHROMA, v != 4);
    if (v != 4) cabac.bypass_bits((uint32_t)v, 2);
  };
  if (cf == 3) for (int idx = 0; idx < nparts; idx++) code_icpm(icpm[idx]);
  else if (cf != 0) code_icpm(icpm[0]);

  write_tree(root, max_depth, nxn ? 1 : 0, 1, 1, luma_modes, chroma_modes);
}

void Enc::coding_quadtree(int x0, int y0, int log2, int depth) {
  int size = 1 << log2;
  bool split;
  if (x0 + size <= W && y0 + size <= H && log2 > log2_min_cb) {
    double v = variance(x0, y0, size);
    double thr = 40.0 + 4.0 * P.qp;
    split = v > thr ? rng.chance(85) : rng.chance(log2 == 6 ? 50 : 15);
    int condL = 0, condA = 0;
    if (ctb_available(x0, y0, x0 - 1, y0) && ct_depth[((x0 - 1) >> 3) + (size_t)(y0 >> 3) * w8] > depth) condL = 1;
    if (ctb_available(x0, y0, x0, y0 - 1) && ct_depth[(x0 >> 3) + (size_t)((y0 - 1) >> 3) * w8] > depth) condA = 1;
    bin(CTX_SPLIT_CU + condL + condA, split);
  } else {
    split = log2 > log2_min_cb;
  }
  if (P.cu_qp_delta && log2 >= log2_min_cu_qp_delta) {
    IsCuQpDeltaCoded = false;
    CuQpDeltaVal = 0;
    // target QP of this quantisation group (kept within +-6 of the slice QP and the legal range)
    qg_target_qp = clip3(std::max(0, slice_qp - 6), std::min(51, slice_qp + 6), slice_qp + rng.below(7) - 3);
    if (stress(HEVC_ENC_STRESS_QP)) qg_target_qp = -qp_bd_offset + rng.below(52 + qp_bd_offset);
  }
  if (P.chroma_qp_offset_list_len && log2 >= log2_min_cu_chroma_qp_offset) {
    cqo_coded_a = cqo_coded_b = false;
    cqo_next = rng.chance(80) ? 1 + rng.below(P.chroma_qp_offset_list_len) : 0;
  }
  if (split) {
    int h = size >> 1, x1 = x0 + h, y1 = y0 + h;
    coding_quadtree(x0, y0, log2 - 1, depth + 1);
    if (x1 < W) coding_quadtree(x1, y0, log2 - 1, depth + 1);
    if (y1 < H) coding_quadtree(x0, y1, log2 - 1, depth + 1);
    if (x1 < W && y1 < H) coding_quadtree(x1, y1, log2 - 1, depth + 1);
  } else {
    coding_unit(x0, y0, log2, depth);
  }
}

void Enc::code_sao(int rx, int ry) {
  Sao& s = sao[ctb_addr_rs];
  memset(&s, 0, sizeof(s));
  bool merge_left = false, merge_up = false;
  if (rx > 0) {
    int left = ctb_addr_rs - 1;
    if (ctb_slice[left] == slice_addr_rs && tile_id[left] == tile_id[ctb_addr_rs]) { merge_left = rng.chance(stress(HEVC_ENC_STRESS_SAO) ? 35 : 20); bin(CTX_SAO_MERGE, merge_left); }
  }
  if (ry > 0 && !merge_left) {
    int up = ctb_addr_rs - ctbs_w;
    if (ctb_slice[up] == slice_addr_rs && tile_id[up] == tile_id[ctb_addr_rs]) { merge_up = rng.chance(stress(HEVC_ENC_STRESS_SAO) ? 35 : 20); bin(CTX_SAO_MERGE, merge_up); }
  }
  if (merge_left) { stats[ST_sao_merge_left]++; s = sao[ctb_addr_rs - 1]; return; }
  if (merge_up) { stats[ST_sao_merge_up]++; s = sao[ctb_addr_rs - ctbs_w]; return; }
  int ncomp = cf ? 3 : 1;
  for (int c = 0; c < ncomp; c++) {
    if (!((slice_sao_luma && c == 0) || (slice_sao_chroma && c > 0))) continue;
    if (c < 2) {
      int r = rng.below(100);
      s.type[c] = r < 35 ? 0 : r < 65 ? 1 : 2;
      bin(CTX_SAO_TYPE, s.type[c] != 0);
      if (s.type[c]) cabac.bypass(s.type[c] == 2);
    } else {
      s.type[2] = s.type[1];
    }
    if (!s.type[c]) continue;
    int cMax = (1 << (std::min(bd, 10) - 5)) - 1;
    int absv[4];
    for (int i = 0; i < 4; i++) {
      absv[i] = rng.below((stress(HEVC_ENC_STRESS_SAO) ? cMax : std::min(cMax, 4)) + 1);
      if (absv[i] == cMax && bd >= 10) stats[ST_sao_offset_cmax_hbd]++;
      if (absv[i] == cMax && (c ? P.log2_sao_offset_scale_chroma : P.log2_sao_offset_scale_luma)) stats[ST_sao_offset_scaled_cmax]++;
      for (int k = 0; k < absv[i]; k++) cabac.bypass(1);
      if (absv[i] < cMax) cabac.bypass(0);
    }
    if (s.type[c] == 1) {
      int sign[4];
      for (int i = 0; i < 4; i++) { sign[i] = 0; if (absv[i]) { sign[i] = rng.below(2); cabac.bypass(sign[i]); } }
      s.boc[c] = (uint8_t)rng.below(32);
      cabac.bypass_bits(s.boc[c], 5);
      if (s.boc[c] >= 29) stats[ST_sao_band_ge29]++;
      for (int i = 0; i < 4; i++) s.off[c][i] = (int8_t)(sign[i] ? -absv[i] : absv[i]);
    } else {
      if (c < 2) { s.boc[c] = (uint8_t)rng.below(4); cabac.bypass_bits(s.boc[c], 2); stats[ST_sao_eo_class + s.boc[c]]++; }
      else s.boc[2] = s.boc[1];
    }
  }
}

void Enc::encode_ctu() {
  int rx = ctb_addr_rs % ctbs_w, ry = ctb_addr_rs / ctbs_w;
  if (slice_sao_luma || slice_sao_chroma) code_sao(rx, ry);
  ctb_ntb = ctb_ncoeff = 0;
  coding_quadtree(rx * ctb, ry * ctb, log2_ctb, 0);
  // the records' per-CTB capacities: every sample a coefficient, every 4x4 block of every component a TB
  const int csamples = cf ? 2 * (ctb / SubW) * (ctb / SubH) : 0;
  if (ctb_ncoeff == ctb * ctb + csamples) stats[ST_ctb_coeff_full]++;
  if (ctb_ntb == (ctb * ctb + csamples) / 16) stats[ST_ctb_tb_full]++;
}

void Enc::encode_picture(std::vector<uint8_t>& out) {
  write_parameter_sets(out);
  const bool tiles = P.tile_cols > 1 || P.tile_rows > 1;
  int ts = 0;
  int seg_index = 0;
  int last_independent_addr = 0;
  while (ts < nctb) {
    int seg_len = P.slice_ctbs > 0 ? std::min(P.slice_ctbs, nctb - ts) : nctb;
    bool dependent = P.dependent_slices && (seg_index & 1) && ts > 0;
    int seg_addr = ts2rs[ts];
    if (!dependent) {
      last_independent_addr = seg_addr;
      slice_qp = P.qp;
      slice_sao_luma = P.sao != 0;
      slice_sao_chroma = P.sao != 0 && cf != 0;
    }
    slice_addr_rs = last_independent_addr;
    // ---- slice data ----
    slice_data.clear();
    entry_points.clear();
    substream_start = 0;
    cabac.start(&slice_data);
    currentQG_x = currentQG_y = -1;
    if (seg_addr > 0) {
      int prev = ts2rs[ts - 1];
      int x = std::min((((prev % ctbs_w) + 1) << log2_ctb) - 1, W - 1), y = std::min((((prev / ctbs_w) + 1) << log2_ctb) - 1, H - 1);
      currentQPY = qp_y[(x >> 3) + (size_t)(y >> 3) * w8];
    }
    if (dependent && !tile_start[seg_addr]) { ctx = dep_ctx; memcpy(stat_coeff, dep_stat.data(), 4); }
    else init_contexts();
    bool first_substream_of_independent = !dependent;
    for (int k = 0; k < seg_len; k++) {
      ctb_addr_ts = ts + k;
      ctb_addr_rs = ts2rs[ctb_addr_ts];
      int cxr = ctb_addr_rs % ctbs_w, cyr = ctb_addr_rs / ctbs_w;
      if (P.wpp && cxr == 0 && cyr >= 1 && !(first_substream_of_independent && ctb_addr_rs == seg_addr)) {
        if (ctbs_w > 1) {
          ctx = wpp_ctx[cyr - 1];
          if (memcmp(stat_coeff, wpp_stat[cyr - 1].data(), 4)) stats[ST_wpp_stat_coeff_restored]++;
          memcpy(stat_coeff, wpp_stat[cyr - 1].data(), 4);
        } else {
          init_contexts();
        }
      }
      ctb_slice[ctb_addr_rs] = slice_addr_rs;
      encode_ctu();
      if (P.wpp && cxr == 1 && cyr < ctbs_h - 1) { wpp_ctx[cyr] = ctx; memcpy(wpp_stat[cyr].data(), stat_coeff, 4); }
      bool last = k == seg_len - 1;
      cabac.terminate(last ? 1 : 0);
      if (last) {
        dep_ctx = ctx;
        memcpy(dep_stat.data(), stat_coeff, 4);
        cabac.finish();
        break;
      }
      int next_rs = ts2rs[ctb_addr_ts + 1];
      bool eoss = (tiles && tile_id[next_rs] != tile_id[ctb_addr_rs]) || (P.wpp && (next_rs / ctbs_w) != cyr);
      if (eoss) {
        cabac.terminate(1);
        cabac.finish();
        entry_points.push_back((uint32_t)(slice_data.size() - substream_start));
        substream_start = slice_data.size();
        cabac.start(&slice_data);
        first_substream_of_independent = false;
        if (tiles) init_contexts();
      }
    }
    // ---- slice header ----
    // entry_point_offset counts bytes of the escaped NAL payload. Every substream ends with a byte
    // holding the terminating '1' bit, so no zero run crosses a substream border and the escaped
    // size of each substream can be computed on its own.
    std::vector<uint32_t> esc_offsets;
    {
      size_t pos = 0;
      for (uint32_t len : entry_points) {
        int zeros = 0;
        uint32_t e = 0;
        for (size_t i = pos; i < pos + len; i++) {
          if (zeros >= 2 && slice_data[i] <= 3) { e++; zeros = 0; }
          e++;
          zeros = slice_data[i] == 0 ? zeros + 1 : 0;
        }
        esc_offsets.push_back(e);
        pos += len;
      }
    }
    BitWriter bw;
    bw.put(ts == 0 ? 1 : 0, 1);
    bw.put(0, 1);  // no_output_of_prior_pics_flag (IDR)
    bw.ue(0);
    if (ts != 0) {
      if (P.dependent_slices) bw.put(dependent, 1);
      int bits = 0;
      while ((1 << bits) < nctb) bits++;
      bw.put((uint32_t)seg_addr, bits);
    }
    if (!dependent) {
      bw.ue(2);  // I slice
      if (P.sao) { bw.put(slice_sao_luma, 1); if (cf) bw.put(slice_sao_chroma, 1); }
      bw.se(slice_qp - 26);
      if (P.chroma_qp_offset_list_len) bw.put(1, 1);  // cu_chroma_qp_offset_enabled_flag
      if (P.loop_filter_across_slices && (slice_sao_luma || slice_sao_chroma || !P.deblock_disable)) bw.put(1, 1);
    }
    std::vector<uint8_t> payload;
    if (tiles || P.wpp) {
      bw.ue((uint32_t)esc_offsets.size());
      if (!esc_offsets.empty()) {
        // minimal field width, like x265/HM: wide zero-filled fields would put emulation-prevention
        // bytes into the header, which the reference's offset correction does not expect
        // (nal-parser.cc:106-113 counts header bytes too)
        uint32_t mx = 0;
        for (uint32_t o : esc_offsets) mx = std::max(mx, o - 1);
        int len = 1;
        while (len < 32 && (mx >> len)) len++;
        bw.ue((uint32_t)(len - 1));
        for (uint32_t o : esc_offsets) bw.put(o - 1, len);
      }
    }
    bw.trailing();
    payload = bw.bytes;
    payload.insert(payload.end(), slice_data.begin(), slice_data.end());
    append_nal(out, 20 /* IDR_N_LP */, payload);
    ts += seg_len;
    seg_index++;
  }
}

}  // namespace

extern "C" {

// planes: uint16 samples of the visible picture (width x height, chroma subsampled), tightly
// packed strides given in samples. Output: 4-byte-length-prefixed NAL units (VPS, SPS, PPS, slices).
// recon (optional): per component a buffer of the coded size (width and height rounded up to a multiple of 8,
// chroma subsampled, tightly packed) that receives the encoder's reconstruction before the in-loop filters.
// stats (optional): hevc_enc_stat_count() counters of what was written (names: hevc_enc_stat_name; the range-extension
// group starts at hevc_enc_rext_stat_first()).
int hevc_enc_encode_ex(const hevc_enc_params* params, const uint16_t* const planes[3], const int strides[3], uint8_t** out,
                       size_t* out_size, uint16_t* const recon[3], uint64_t* stats) {
  if (!params || !planes || !out || !out_size) return -1;
  hevc_enc_params P = *params;
  if (P.width <= 0 || P.height <= 0 || P.chroma_format < 0 || P.chroma_format > 3 || P.bit_depth < 8 || P.bit_depth > 12) return -2;
  if (P.log2_ctb < 4 || P.log2_ctb > 6 || P.log2_min_tb < 2 || P.log2_max_tb > 5 || P.log2_min_tb > P.log2_max_tb) return -2;
  if (P.log2_min_tb >= 3) return -2;  // min CB is fixed at 8x8 here
  if (P.qp < -6 * (P.bit_depth - 8) || P.qp > 51) return -2;
  if (P.log2_max_transform_skip_minus2 < 0 || P.log2_max_transform_skip_minus2 > 3) return -2;
  if (P.chroma_qp_offset_list_len < 0 || P.chroma_qp_offset_list_len > 6) return -2;
  if (P.diff_cu_chroma_qp_offset_depth < 0 || P.diff_cu_chroma_qp_offset_depth > P.log2_ctb - 3) return -2;
  const int max_sao_scale = std::max(0, P.bit_depth - 10);
  if (P.log2_sao_offset_scale_luma < 0 || P.log2_sao_offset_scale_luma > max_sao_scale) return -2;
  if (P.log2_sao_offset_scale_chroma < 0 || P.log2_sao_offset_scale_chroma > max_sao_scale) return -2;
  Enc enc(P);
  enc.setup();
  const int ncomp = enc.cf ? 3 : 1;
  for (int c = 0; c < ncomp; c++) {
    int w = c ? enc.W / enc.SubW : enc.W, h = c ? enc.H / enc.SubH : enc.H;
    int vw = c ? (P.width + enc.SubW - 1) / enc.SubW : P.width, vh = c ? (P.height + enc.SubH - 1) / enc.SubH : P.height;
    enc.pw[c] = w; enc.ph[c] = h;
    enc.orig[c].assign((size_t)w * h, 0);
    enc.rec[c].assign((size_t)w * h, 0);
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) enc.orig[c][x + (size_t)y * w] = planes[c][std::min(x, vw - 1) + (size_t)std::min(y, vh - 1) * strides[c]];
  }
  std::vector<uint8_t> bytes;
  enc.encode_picture(bytes);
  uint8_t* p = (uint8_t*)malloc(bytes.size() ? bytes.size() : 1);
  if (!p) return -3;
  memcpy(p, bytes.data(), bytes.size());
  *out = p;
  *out_size = bytes.size();
  if (recon)
    for (int c = 0; c < ncomp; c++)
      if (recon[c]) memcpy(recon[c], enc.rec[c].data(), enc.rec[c].size() * sizeof(uint16_t));
  if (stats) memcpy(stats, enc.stats, sizeof(enc.stats));
  return 0;
}

int hevc_enc_encode(const hevc_enc_params* params, const uint16_t* const planes[3], const int strides[3], uint8_t** out,
                    size_t* out_size) {
  return hevc_enc_encode_ex(params, planes, strides, out, out_size, nullptr, nullptr);
}

int hevc_enc_stat_count(void) { return ST_COUNT; }

int hevc_enc_rext_stat_first(void) { return ST_REXT_FIRST_; }

const char* hevc_enc_stat_name(int i) {
  static const std::vector<std::string> names = [] {
    std::vector<std::string> v;
#define HEVC_ENC_STAT_NAME(name, n) \
  for (int k = 0; k < (n); k++) v.push_back((n) == 1 ? std::string(#name) : std::string(#name) + "_" + std::to_string(k));
    HEVC_ENC_STATS(HEVC_ENC_STAT_NAME)
    HEVC_ENC_REXT_STATS(HEVC_ENC_STAT_NAME)
#undef HEVC_ENC_STAT_NAME
    return v;
  }();
  return i >= 0 && i < (int)names.size() ? names[(size_t)i].c_str() : nullptr;
}

void hevc_enc_free(void* p) { free(p); }

}  // extern "C"
