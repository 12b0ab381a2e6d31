// hevc_parse.cc — CABAC slice-data parse of HEVC intra pictures into reconstruction records.
//
// Written from ITU-T H.265 (04/2015): §7.3.8 (slice data syntax), §9.3 (CABAC), §8.4.2 (luma intra
// mode derivation), §8.4.3 (chroma mode), §8.6.1 (QP derivation), §6.4.1 (z-scan availability),
// §8.7.2.2/8.7.2.3 (deblocking edge derivation for intra pictures).  No sample is reconstructed
// here: every block is emitted as a record for the GPU (include/heifcuda_records.h).
//
// Where the reference decoder (third-party/libde265) deviates from the text and the deviation is
// observable in decoded pictures, the reference is followed and cited:
//   - non-4:2:0 chroma QP is not capped at 51 for dequantisation      transform.cc:171-178
//   - 4:2:2 chroma mode remap table                                    slice.cc:4563-4566
//   - WPP context hand-over uses the row above's stored table whenever the picture is wider
//     than one CTB (no top-right availability test)                    slice.cc:5195-5217
//   - coefficient levels wrap to int16                                 slice.cc:3671
//   - deblock slice/tile edge tests only at CTB boundaries             deblock.cc:180-215
#include "hevc_parse.h"
#include "k0_host.h"
#include "hevc_cabac.h"
#include "hevc_scan.h"
#include <algorithm>
#include <array>
#include <cstdlib>

namespace hc {

namespace {

inline int clip3(int lo, int hi, int v) { return v < lo ? lo : (v > hi ? hi : v); }

// H.265 Table 8-10 (ChromaArrayType == 1)
inline int qpc_table_420(int qPi) {
  static const int8_t t[14] = {29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37, 37};
  if (qPi < 30) return qPi;
  if (qPi >= 44) return qPi - 6;
  return t[qPi - 30];
}

// reference's Table 8-3 variant (slice.cc:4563-4566)
const uint8_t kMode422[35] = {0,  1,  2,  2,  2,  2,  3,  5,  7,  8,  10, 12, 13, 15, 17, 18, 19, 20,
                              21, 22, 23, 23, 24, 24, 25, 25, 26, 27, 27, 28, 28, 29, 29, 30, 31};

const uint8_t kSigCtx4x4[16] = {0, 1, 4, 5, 2, 3, 4, 5, 6, 6, 8, 8, 7, 7, 8, 8};

}  // namespace

struct HevcIntraParser::Impl {
  Sps sps_tab[16];
  Pps pps_tab[64];

  // ---- current picture ----
  bool started = false;
  const Sps* S = nullptr;
  const Pps* P = nullptr;
  Pps pps_copy;   // parameter sets may be re-sent between pictures: keep what this picture uses
  Sps sps_copy;
  std::unique_ptr<PictureRecords> rec;
  std::vector<SliceHeader> slices;
  SliceHeader prev_independent;
  bool have_prev_independent = false;
  int ctbs_done = 0;

  int W = 0, H = 0;           // luma size
  int w8 = 0, h8 = 0;         // size in 8x8 units
  int w4 = 0, h4 = 0;         // size in 4x4 units
  std::vector<uint8_t> ct_depth;   // per 8x8
  std::vector<uint8_t> cu_flags;   // per 8x8: 1 = pcm, 2 = transquant bypass
  std::vector<int8_t> qp_y;        // per 8x8
  std::vector<uint8_t> ipm;        // per 4x4 luma intra pred mode
  std::vector<uint8_t> ipm_c;      // per 4x4 chroma intra pred mode (already remapped)
  std::vector<int> ctb_slice_addr; // per CTB (RS): SliceAddrRs, -1 = not decoded
  std::vector<int> ctb_slice_idx;  // per CTB (RS): index into slices[]
  std::vector<hc_blk> ctu_blks[3];

  // ---- entropy decoding state ----
  Cabac cabac;
  CtxSet ctx;
  std::vector<CtxSet> wpp_ctx;     // per CTB row: table saved after the 2nd CTB of the row
  std::vector<uint8_t> wpp_ctx_valid;
  std::vector<std::array<uint8_t, 4>> wpp_stat_coeff;   // StatCoeff stored with the table (9.3.2.4, TableStatCoeffWpp)
  CtxSet dep_ctx;                  // table at the end of the previous slice segment
  bool dep_ctx_valid = false;
  uint8_t stat_coeff[4] = {0, 0, 0, 0};

  // ---- slice / CU state ----
  const SliceHeader* sh = nullptr;
  int sh_idx = 0;
  int ctb_addr_ts = 0, ctb_addr_rs = 0;
  bool IsCuQpDeltaCoded = false;
  int CuQpDeltaVal = 0;
  bool IsCuChromaQpOffsetCoded = false;
  int CuQpOffsetCb = 0, CuQpOffsetCr = 0;
  int currentQG_x = -1, currentQG_y = -1, lastQPYinPreviousQG = 0, currentQPY = 0;
  int qPYPrime = 0, qPCbPrime = 0, qPCrPrime = 0;
  bool cu_transquant_bypass = false;
  int cu_x0 = 0, cu_y0 = 0, cu_log2 = 0;
  int filterLeftCbEdge = 0, filterTopCbEdge = 0;
  std::string error;

  // ---- K0 preparation (collect-only mode) ----
  bool collect_only = false;
  std::vector<std::vector<uint8_t>> k0_rbsp;   // padded RBSP of every slice segment NAL
  std::vector<size_t> k0_rbsp_size;

  // =========================================================================================
  std::string start_picture(const SliceHeader& first);
  std::string decode_slice_segment(const uint8_t* data, size_t size, const SliceHeader& hdr);
  void finish_picture();

  // ---- helpers ----
  int ctb_of(int x, int y) const { return (x >> S->log2_ctb) + (y >> S->log2_ctb) * S->ctbs_w; }
  bool ctb_available(int xC, int yC, int xN, int yN) const {
    if (xN < 0 || yN < 0 || xN >= W || yN >= H) return false;
    int c = ctb_of(xC, yC), n = ctb_of(xN, yN);
    if (ctb_slice_addr[n] < 0 || ctb_slice_addr[n] != ctb_slice_addr[c]) return false;
    if (P->tile_id_rs[n] != P->tile_id_rs[c]) return false;
    return true;
  }
  int zs_addr(int x, int y) const {
    return P->min_tb_addr_zs[(x >> S->log2_min_tb) + (size_t)(y >> S->log2_min_tb) * S->tbs_w];
  }
  bool available_zscan(int xC, int yC, int xN, int yN) const {
    if (xN < 0 || yN < 0 || xN >= W || yN >= H) return false;
    if (zs_addr(xN, yN) > zs_addr(xC, yC)) return false;
    return ctb_available(xC, yC, xN, yN);
  }

  inline int bin(int c) { return cabac.decode_bin(ctx.s[c]); }

  void init_contexts() {
    ctx_init_all(ctx, sh->slice_qp_y);
    for (int i = 0; i < 4; i++) stat_coeff[i] = 0;
  }

  // ---- syntax ----
  void decode_ctu();
  void read_sao(int rx, int ry, hc_ctu& ctu);
  void coding_quadtree(int x0, int y0, int log2, int depth);
  void coding_unit(int x0, int y0, int log2, int depth);
  void pcm_sample(int x0, int y0, int log2);
  void transform_tree(int x0, int y0, int xBase, int yBase, int log2, int depth, int blkIdx,
                      int max_depth, int intra_split, int parent_cbf_cb, int parent_cbf_cr);
  void transform_unit(int x0, int y0, int xBase, int yBase, int log2, int depth, int blkIdx,
                      int cbf_luma, int cbf_cb, int cbf_cr);
  // returns the picture-relative residual offset of the coded block
  uint32_t residual_coding(int x0, int y0, int log2, int cIdx, int pred_mode);
  void derive_qp(int xCU, int yCU);
  void emit_blk(int cIdx, int xB, int yB, int log2, int mode, bool has_resid, uint32_t resid_off,
                uint8_t extra_flags);
  void mark_tu_edges(int x0, int y0, int log2);
};

// ---------------------------------------------------------------------------------------------
HevcIntraParser::HevcIntraParser() : impl_(new Impl) {}
HevcIntraParser::~HevcIntraParser() { delete impl_; }

bool HevcIntraParser::picture_started() const { return impl_->started; }
bool HevcIntraParser::picture_complete() const {
  return impl_->started && impl_->ctbs_done >= impl_->S->pic_size_in_ctbs;
}

std::unique_ptr<PictureRecords> HevcIntraParser::take_picture(std::string* err) {
  Impl& d = *impl_;
  if (!d.started) {
    if (err) *err = "no picture in the bitstream";
    return nullptr;
  }
  if (d.ctbs_done < d.S->pic_size_in_ctbs) {
    if (err) *err = "picture incomplete: not all coding tree blocks were present";
    d.started = false;
    d.rec.reset();
    return nullptr;
  }
  d.finish_picture();
  d.started = false;
  if (err) err->clear();
  return std::move(d.rec);
}

std::string HevcIntraParser::push_length_prefixed(const uint8_t* data, size_t size) {
  size_t pos = 0;
  while (pos + 4 <= size) {
    uint32_t len = ((uint32_t)data[pos] << 24) | ((uint32_t)data[pos + 1] << 16) |
                   ((uint32_t)data[pos + 2] << 8) | data[pos + 3];
    pos += 4;
    if (len > size - pos) return "NAL unit length exceeds the data size";
    std::string e = push_nal(data + pos, len);
    if (!e.empty()) return e;
    pos += len;
  }
  return "";
}

std::string HevcIntraParser::push_annexb(const uint8_t* data, size_t size) {
  // find start codes 00 00 01
  size_t i = 0;
  auto find_sc = [&](size_t from) -> size_t {
    for (size_t k = from; k + 3 <= size; k++)
      if (data[k] == 0 && data[k + 1] == 0 && data[k + 2] == 1) return k;
    return size;
  };
  i = find_sc(0);
  while (i < size) {
    size_t start = i + 3;
    size_t next = find_sc(start);
    size_t end = next;
    // trailing zero bytes belong to the next start code (00 00 00 01)
    while (end > start && data[end - 1] == 0) end--;
    if (end > start) {
      std::string e = push_nal(data + start, end - start);
      if (!e.empty()) return e;
    }
    i = next;
  }
  return "";
}

std::string HevcIntraParser::push_nal(const uint8_t* nal, size_t size) {
  Impl& d = *impl_;
  if (size < 2) return "";  // empty NAL units are ignored like the reference does
  int nal_type = (nal[0] >> 1) & 0x3F;
  int layer_id = ((nal[0] & 1) << 5) | (nal[1] >> 3);
  if (layer_id > 0) return "";  // decctx.cc:1220: only the base layer is decoded

  std::vector<uint8_t> rbsp;
  std::vector<uint32_t> skipped;
  nal_unescape(nal, size, rbsp, &skipped);
  const size_t rbsp_size = rbsp.size();
  rbsp.resize(rbsp_size + 16, 0);   // the CABAC engine refills 4 bytes at a time (hevc_cabac.h)

  if (nal_type == NAL_SPS) {
    Sps s;
    std::string e = parse_sps(rbsp.data() + 2, rbsp_size - 2, s);
    if (!e.empty()) return e;
    // parameter sets precede the first VCL NAL unit of their access unit (7.4.2.4.4); a picture in progress keeps its own
    // copies, but later slice headers of it would be read against the new tables
    if (d.started) return "SPS inside a picture";
    // a re-sent SPS invalidates every PPS that refers to it (their derived tables are sized by the old one; the reference
    // does the same, decctx.cc process_sps): a slice that still names such a PPS fails with "refers to a missing PPS"
    for (Pps& p : d.pps_tab)
      if (p.valid && p.sps_id == s.sps_id) p.valid = false;
    d.sps_tab[s.sps_id] = s;
    return "";
  }
  if (nal_type == NAL_PPS) {
    Pps p;
    std::string e = parse_pps(rbsp.data() + 2, rbsp_size - 2, d.sps_tab, p);
    if (!e.empty()) return e;
    if (d.started) return "PPS inside a picture";
    d.pps_tab[p.pps_id] = std::move(p);
    return "";
  }
  if (nal_type >= 32) return "";  // VPS, AUD, SEI, EOS ... carry nothing the intra path needs
  if (nal_type > NAL_RSV_IRAP_VCL23 || (nal_type > 9 && nal_type < 16)) return "";  // reserved

  // ---- slice segment ----
  SliceHeader hdr;
  std::string e = parse_slice_header(rbsp.data(), rbsp_size, nal_type, d.sps_tab, d.pps_tab,
                                     d.have_prev_independent ? &d.prev_independent : nullptr, skipped, hdr);
  if (!e.empty()) return e;
  if (hdr.first_slice_segment_in_pic) {
    if (d.started) return "a second picture starts before the first one was taken";
    e = d.start_picture(hdr);
    if (!e.empty()) return e;
  } else if (!d.started) {
    return "slice segment without the first slice segment of its picture";
  }
  if (!hdr.dependent) {
    d.prev_independent = hdr;
    d.have_prev_independent = true;
  }
  if (d.collect_only) {
    if (d.pps_tab[hdr.pps_id].pps_id != d.P->pps_id) return "slice segments of one picture refer to different PPSs";
    d.slices.push_back(hdr);
    d.k0_rbsp_size.push_back(rbsp_size);
    d.k0_rbsp.push_back(std::move(rbsp));
    return "";
  }
  return d.decode_slice_segment(rbsp.data(), rbsp_size, hdr);
}

void HevcIntraParser::set_collect_only(bool on) { impl_->collect_only = on; }

void HevcIntraParser::reset() {
  Impl& d = *impl_;
  for (Sps& s : d.sps_tab) s.valid = false;
  for (Pps& p : d.pps_tab) p.valid = false;
  d.started = false;
  d.S = nullptr;
  d.P = nullptr;
  d.rec.reset();
  d.slices.clear();
  d.have_prev_independent = false;
  d.ctbs_done = 0;
  d.k0_rbsp.clear();
  d.k0_rbsp_size.clear();
}

// Builds the K0 inputs from the collected slice segments (see kernels/k0_core.cuh for what K0 accepts).
std::string HevcIntraParser::take_k0(K0HostPicture& out) {
  Impl& d = *impl_;
  if (!d.started || d.slices.empty()) return "no picture in the bitstream";
  const Sps& S = *d.S;
  const Pps& P = *d.P;
  out = K0HostPicture();
  out.hpic = d.rec->pic;
  out.scaling = d.rec->scaling;
  const int nctb = S.pic_size_in_ctbs, cw = S.ctbs_w, chh = S.ctbs_h;
  auto no = [&](const char* why) { out.eligible = false; out.why_not = why; d.started = false; d.rec.reset(); d.slices.clear(); d.k0_rbsp.clear(); d.k0_rbsp_size.clear(); return std::string(); };
  if (P.tiles_enabled) return no("HEVC tiles");
  if (S.pcm_enabled) return no("pcm");
  if (P.transquant_bypass_enabled) return no("transquant bypass");
  if (S.persistent_rice_adaptation_enabled) return no("persistent_rice_adaptation");
  if (P.chroma_qp_offset_list_enabled) return no("cu_chroma_qp_offset");
  if (S.log2_ctb < 4 || S.log2_ctb > 6 || S.log2_min_cb < 3) return no("coding block sizes");
  for (auto& h : d.slices)
    if (h.cu_chroma_qp_offset_enabled) return no("cu_chroma_qp_offset");
  // coverage: segments in increasing address order, together covering the picture
  for (size_t k = 0; k < d.slices.size(); k++) {
    const int a = d.slices[k].segment_address, b = k + 1 < d.slices.size() ? d.slices[k + 1].segment_address : nctb;
    if ((k == 0 && a != 0) || b <= a || b > nctb) return no("slice segments do not cover the picture in order");
    if (d.slices[k].dependent && k == 0) return no("dependent first slice segment");
  }

  k0::Pic& p = out.pic;
  memset(&p, 0, sizeof(p));
  p.W = S.width; p.H = S.height; p.w8 = p.W >> 3; p.h8 = p.H >> 3; p.w4 = p.W >> 2; p.h4 = p.H >> 2;
  p.ctbs_w = cw; p.ctbs_h = chh;
  p.log2_ctb = S.log2_ctb; p.log2_min_cb = S.log2_min_cb; p.log2_min_tb = S.log2_min_tb; p.log2_max_tb = S.log2_max_tb;
  p.max_th_depth_intra = S.max_th_depth_intra;
  p.chroma_array_type = S.ChromaArrayType; p.sub_w = S.SubWidthC; p.sub_h = S.SubHeightC;
  p.bit_depth_y = S.bit_depth_y; p.bit_depth_c = S.bit_depth_c; p.qp_bd_offset_y = S.qp_bd_offset_y; p.qp_bd_offset_c = S.qp_bd_offset_c;
  p.log2_max_transform_skip_size = P.log2_max_transform_skip_size;
  p.log2_min_cu_qp_delta_size = P.log2_min_cu_qp_delta_size;
  p.pps_cb_qp_offset = P.cb_qp_offset; p.pps_cr_qp_offset = P.cr_qp_offset;
  p.log2_sao_offset_scale_luma = P.log2_sao_offset_scale_luma; p.log2_sao_offset_scale_chroma = P.log2_sao_offset_scale_chroma;
  p.transform_skip_enabled = P.transform_skip_enabled; p.sign_data_hiding = P.sign_data_hiding;
  p.cu_qp_delta_enabled = P.cu_qp_delta_enabled; p.entropy_coding_sync = P.entropy_coding_sync_enabled;
  p.implicit_rdpcm = S.implicit_rdpcm_enabled; p.tskip_rotation = S.transform_skip_rotation_enabled;
  p.tskip_context = S.transform_skip_context_enabled; p.pps_loop_filter_across_slices = P.loop_filter_across_slices;
  p.nslices = (int32_t)d.slices.size();
  const int ctb = 1 << S.log2_ctb;
  const int ccw = S.ChromaArrayType ? ctb / S.SubWidthC : 0, cch = S.ChromaArrayType ? ctb / S.SubHeightC : 0;
  p.blk_cap[0] = (uint32_t)(ctb / 4) * (ctb / 4);
  p.blk_cap[1] = p.blk_cap[2] = (uint32_t)(ccw * cch) / 16;
  p.blk_cap_ctb = p.tb_cap_ctb = p.blk_cap[0] + p.blk_cap[1] + p.blk_cap[2];
  p.coeff_cap_ctb = p.resid_cap_ctb = (uint32_t)(ctb * ctb + 2 * ccw * cch);

  // slices, bytes, per-CTB slice index
  out.ctb_slice.assign(nctb, 0);
  bool any_deblock = false, any_sao = false;
  for (size_t k = 0; k < d.slices.size(); k++) {
    const SliceHeader& h = d.slices[k];
    k0::Slice s;
    memset(&s, 0, sizeof(s));
    s.segment_address = h.segment_address; s.slice_addr_rs = h.slice_addr_rs; s.slice_qp_y = h.slice_qp_y;
    if (h.data_byte_offset >= d.k0_rbsp_size[k]) return "slice segment has no data";
    s.data_begin = (uint32_t)(out.bytes.size() + h.data_byte_offset);
    s.data_end = (uint32_t)(out.bytes.size() + d.k0_rbsp_size[k]);
    s.cb_qp_offset = (int8_t)h.cb_qp_offset; s.cr_qp_offset = (int8_t)h.cr_qp_offset;
    s.beta_offset = (int8_t)h.beta_offset; s.tc_offset = (int8_t)h.tc_offset;
    s.dependent = h.dependent; s.sao_luma = h.sao_luma; s.sao_chroma = h.sao_chroma;
    s.deblocking_disabled = h.deblocking_disabled; s.loop_filter_across_slices = h.loop_filter_across_slices;
    out.slices.push_back(s);
    out.bytes.insert(out.bytes.end(), d.k0_rbsp[k].begin(), d.k0_rbsp[k].end());
    const int b = k + 1 < d.slices.size() ? d.slices[k + 1].segment_address : nctb;
    for (int a = h.segment_address; a < b; a++) out.ctb_slice[a] = (int32_t)k;
    any_deblock |= !h.deblocking_disabled;
    any_sao |= h.sao_luma || h.sao_chroma;
  }
  if (any_deblock) out.hpic.flags |= HC_PIC_HAS_DEBLOCK;   // conservative: K3 / K4 look at the per-unit data anyway
  if (any_sao) out.hpic.flags |= HC_PIC_HAS_SAO;

  // SAO neighbour masks (the static part of finish_picture: no tiles, no pcm / bypass units)
  out.ctu_static.assign((size_t)nctb * 4, 0);
  {
    auto sa_of = [&](int n) { return d.slices[out.ctb_slice[n]].slice_addr_rs; };
    static const int dx[8] = {-1, 1, 0, 0, -1, 1, -1, 1};
    static const int dy[8] = {0, 0, -1, 1, -1, -1, 1, 1};
    const bool fast = P.loop_filter_across_slices;
    for (int cy = 0; cy < chh; cy++)
      for (int cx = 0; cx < cw; cx++) {
        const int a = cx + cy * cw;
        for (int comp = 0; comp < 2; comp++) {
          int sa = sa_of(a);
          if (comp == 1 && S.ChromaArrayType != 0 && S.ChromaArrayType != 3) {
            const int qx = (cx << S.log2_ctb) / S.SubWidthC, qy = (cy << S.log2_ctb) / S.SubHeightC;
            sa = sa_of((qx >> S.log2_ctb) + (qy >> S.log2_ctb) * cw);
          }
          uint8_t m = 0;
          for (int k = 0; k < 8; k++) {
            const int nx = cx + dx[k], ny = cy + dy[k];
            if (nx < 0 || ny < 0 || nx >= cw || ny >= chh) continue;
            const int n = nx + ny * cw;
            bool ok = true;
            if (!fast) {
              const int sn = sa_of(n);
              if (sn < sa && !d.slices[out.ctb_slice[a]].loop_filter_across_slices) ok = false;
              if (sn > sa && !d.slices[out.ctb_slice[n]].loop_filter_across_slices) ok = false;
            }
            if (ok) m |= (uint8_t)(1u << k);
          }
          out.ctu_static[(size_t)a * 4 + comp] = m;
          if (comp == 1 && !fast && sa_of(a) != sa && !d.slices[out.ctb_slice[a]].loop_filter_across_slices)
            out.ctu_static[(size_t)a * 4 + 2] |= HC_CTU_SAO_C_SELF;
        }
      }
  }

  // chains: one per CTB row when every segment starts a row and carries all its entry points, else one per picture
  bool rows = P.entropy_coding_sync_enabled;
  for (size_t k = 0; rows && k < d.slices.size(); k++) {
    const int a = d.slices[k].segment_address, b = k + 1 < d.slices.size() ? d.slices[k + 1].segment_address : nctb;
    if (a % cw) rows = false;
    else if ((int)d.slices[k].entry_points.size() != (b - 1) / cw - a / cw) rows = false;
  }
  for (size_t k = 0; k < d.slices.size(); k++) {
    const SliceHeader& h = d.slices[k];
    const int a = h.segment_address, b = k + 1 < d.slices.size() ? d.slices[k + 1].segment_address : nctb;
    if (rows) {
      for (int r = a / cw; r <= (b - 1) / cw; r++) {
        k0::Sub s;
        s.pic = 0; s.slice = (uint32_t)k; s.first_ctb = r * cw; s.end_ctb = (r + 1) * cw < b ? (r + 1) * cw : b;
        const int i = r - a / cw;
        s.byte_begin = out.slices[k].data_begin + (i == 0 ? 0u : h.entry_points[i - 1]);
        if (s.byte_begin >= out.slices[k].data_end) return "entry point outside the slice segment";
        s.flags = k0::SUB_ROW_CHAIN;
        out.chains.push_back({(uint32_t)out.subs.size(), 1u});
        out.subs.push_back(s);
      }
    } else {
      k0::Sub s;
      s.pic = 0; s.slice = (uint32_t)k; s.first_ctb = a; s.end_ctb = b;
      s.byte_begin = out.slices[k].data_begin;
      s.flags = 0;
      out.subs.push_back(s);
    }
  }
  if (!rows) out.chains.push_back({0u, (uint32_t)out.subs.size()});
  out.eligible = true;
  d.started = false;
  d.rec.reset();
  d.slices.clear();
  d.k0_rbsp.clear();
  d.k0_rbsp_size.clear();
  return "";
}

// ---------------------------------------------------------------------------------------------
std::string HevcIntraParser::Impl::start_picture(const SliceHeader& first) {
  pps_copy = pps_tab[first.pps_id];
  sps_copy = sps_tab[pps_copy.sps_id];
  S = &sps_copy;
  P = &pps_copy;
  if (S->extended_precision_processing)
    return "extended_precision_processing_flag is not supported (the reference hard-wires it to 0)";
  if (S->cabac_bypass_alignment_enabled) return "cabac_bypass_alignment_enabled_flag is not supported";
  if (P->cross_component_prediction_enabled)
    return "cross_component_prediction is not supported by the GPU reconstruction path";
  if (S->ChromaArrayType == 0 && S->chroma_format_idc == 3)
    return "separate_colour_plane_flag streams are not supported";

  W = S->width;
  H = S->height;
  w8 = W >> 3; h8 = H >> 3; w4 = W >> 2; h4 = H >> 2;
  if (!collect_only) {   // state of the host CABAC parse; K0 keeps its own on the device
    derive_min_tb_addr_zs(sps_copy, pps_copy);
    ct_depth.assign((size_t)w8 * h8, 0);
    cu_flags.assign((size_t)w8 * h8, 0);
    qp_y.assign((size_t)w8 * h8, 0);
    ipm.assign((size_t)w4 * h4, 1);
    ipm_c.assign((size_t)w4 * h4, 1);
    ctb_slice_addr.assign(S->pic_size_in_ctbs, -1);
    ctb_slice_idx.assign(S->pic_size_in_ctbs, -1);
    wpp_ctx.assign(S->ctbs_h, CtxSet());
    wpp_ctx_valid.assign(S->ctbs_h, 0);
    wpp_stat_coeff.assign(S->ctbs_h, std::array<uint8_t, 4>{{0, 0, 0, 0}});
  }
  dep_ctx_valid = false;
  slices.clear();
  slices.reserve(64);
  ctbs_done = 0;
  // Per-picture CU / quantisation-group state. A parser object is reused for many pictures (reset(), one per host thread):
  // CuQpDeltaVal and the chroma offsets are READ by every QP derivation but only WRITTEN when the stream codes them, so a
  // picture without cu_qp_delta decoded after one that ended on a non-zero delta got every QP shifted (found by a
  // single-item job after example.heic: the whole picture differed).
  currentQPY = 0;
  lastQPYinPreviousQG = 0;
  currentQG_x = currentQG_y = -1;
  IsCuQpDeltaCoded = false;
  CuQpDeltaVal = 0;
  IsCuChromaQpOffsetCoded = false;
  CuQpOffsetCb = CuQpOffsetCr = 0;
  cu_transquant_bypass = false;
  for (int i = 0; i < 4; i++) stat_coeff[i] = 0;
  error.clear();

  rec.reset(new PictureRecords);
  hc_pic& p = rec->pic;
  memset(&p, 0, sizeof(p));
  p.width = W;
  p.height = H;
  p.crop_x = S->conf_left * S->SubWidthC;
  p.crop_y = S->conf_top * S->SubHeightC;
  p.crop_w = W - (S->conf_left + S->conf_right) * S->SubWidthC;
  p.crop_h = H - (S->conf_top + S->conf_bottom) * S->SubHeightC;
  p.chroma_format = (uint8_t)S->ChromaArrayType;
  p.bit_depth_y = (uint8_t)S->bit_depth_y;
  p.bit_depth_c = (uint8_t)S->bit_depth_c;
  p.log2_ctb = (uint8_t)S->log2_ctb;
  p.ctbs_w = (uint16_t)S->ctbs_w;
  p.ctbs_h = (uint16_t)S->ctbs_h;
  p.flags = 0;
  if (S->strong_intra_smoothing) p.flags |= HC_PIC_STRONG_INTRA;
  if (S->intra_smoothing_disabled) p.flags |= HC_PIC_NO_INTRA_SMOOTH;
  if (!S->video_full_range) p.flags |= HC_PIC_LIMITED_RANGE;
  p.pps_cb_qp_offset = (int8_t)P->cb_qp_offset;
  p.pps_cr_qp_offset = (int8_t)P->cr_qp_offset;
  p.colour_primaries = (uint8_t)S->colour_primaries;
  p.transfer_characteristics = (uint8_t)S->transfer_characteristics;
  p.matrix_coeffs = (uint8_t)S->matrix_coeffs;
  p.full_range = (uint8_t)S->video_full_range;
  if (!collect_only) {
    rec->ctus.assign(S->pic_size_in_ctbs, hc_ctu());
    for (auto& c : rec->ctus) memset(&c, 0, sizeof(c));
    rec->edge_map.assign((size_t)w4 * h4, 0);
    rec->qp_map.assign((size_t)w8 * h8, 0);
  }
  if (S->scaling_list_enabled) {
    p.flags |= HC_PIC_SCALING_LIST;
    rec->scaling.resize(HC_SCALING_BLOB_BYTES);
    uint8_t* b = rec->scaling.data();
    const ScalingLists& L = P->scaling;
    memcpy(b, L.s4, 6 * 16); b += 6 * 16;
    memcpy(b, L.s8, 6 * 64); b += 6 * 64;
    memcpy(b, L.s16, 6 * 256); b += 6 * 256;
    memcpy(b, L.s32[0], 1024); b += 1024;
    memcpy(b, L.s32[3], 1024);
  }
  // a rough reservation: avoids most reallocations on typical content
  rec->blks.reserve((size_t)w8 * h8 * 2);
  rec->tbs.reserve((size_t)w8 * h8);
  rec->coeffs.reserve((size_t)W * H / 8);
  started = true;
  return "";
}

// ---------------------------------------------------------------------------------------------
std::string HevcIntraParser::Impl::decode_slice_segment(const uint8_t* data, size_t size,
                                                        const SliceHeader& hdr) {
  if (pps_tab[hdr.pps_id].pps_id != P->pps_id || !pps_tab[hdr.pps_id].valid)
    return "slice segments of one picture refer to different PPSs";
  slices.push_back(hdr);
  sh = &slices.back();
  sh_idx = (int)slices.size() - 1;
  error.clear();

  if (hdr.data_byte_offset >= size) return "slice segment has no data";
  cabac.init(data + hdr.data_byte_offset, data + size);

  ctb_addr_ts = P->ctb_addr_rs_to_ts[hdr.segment_address];
  ctb_addr_rs = hdr.segment_address;

  // thread-context initialisation of the reference (decctx.cc:467-506)
  currentQG_x = currentQG_y = -1;
  if (hdr.segment_address > 0) {
    int prev = P->ctb_addr_ts_to_rs[ctb_addr_ts - 1];
    int x = std::min((((prev % S->ctbs_w) + 1) << S->log2_ctb) - 1, W - 1);
    int y = std::min((((prev / S->ctbs_w) + 1) << S->log2_ctb) - 1, H - 1);
    currentQPY = qp_y[(x >> 3) + (size_t)(y >> 3) * w8];
  }

  // §9.3.1: context initialisation / synchronisation at the start of the slice segment
  if (hdr.dependent) {
    if (P->tile_start_ctb[ctb_addr_rs]) {
      init_contexts();
    } else {
      if (!dep_ctx_valid) return "dependent slice segment without stored CABAC state";
      ctx = dep_ctx;
    }
  } else {
    init_contexts();
  }

  bool first_substream_of_independent = !hdr.dependent;
  const int ctbW = S->ctbs_w;

  while (true) {
    int ctbx = ctb_addr_rs % ctbW, ctby = ctb_addr_rs / ctbW;

    // WPP: take over the table stored after the 2nd CTB of the row above (slice.cc:5195-5217)
    if (P->entropy_coding_sync_enabled && ctbx == 0 && ctby >= 1 &&
        !(first_substream_of_independent && ctb_addr_rs == hdr.segment_address)) {
      if (ctbW > 1) {
        if (!wpp_ctx_valid[ctby - 1]) return "WPP: context table of the row above is missing";
        ctx = wpp_ctx[ctby - 1];
        memcpy(stat_coeff, wpp_stat_coeff[ctby - 1].data(), 4);
      } else {
        init_contexts();
      }
    }

    if (ctb_slice_addr[ctb_addr_rs] >= 0) return "coding tree block coded twice";
    ctb_slice_addr[ctb_addr_rs] = sh->slice_addr_rs;
    ctb_slice_idx[ctb_addr_rs] = sh_idx;

    decode_ctu();
    if (!error.empty()) return error;
    if (cabac.overrun()) return "slice data truncated";
    ctbs_done++;

    if (P->entropy_coding_sync_enabled && ctbx == 1 && ctby < S->ctbs_h - 1) {
      wpp_ctx[ctby] = ctx;
      memcpy(wpp_stat_coeff[ctby].data(), stat_coeff, 4);
      wpp_ctx_valid[ctby] = 1;
    }

    int end_of_slice_segment = cabac.decode_terminate();
    if (end_of_slice_segment) {
      if (P->dependent_slice_segments_enabled) {
        dep_ctx = ctx;
        dep_ctx_valid = true;
      }
      break;
    }

    ctb_addr_ts++;
    if (ctb_addr_ts >= S->pic_size_in_ctbs) return "slice data continues past the end of the picture";
    int next_rs = P->ctb_addr_ts_to_rs[ctb_addr_ts];
    bool end_of_substream = false;
    if (P->tiles_enabled && P->tile_id_rs[next_rs] != P->tile_id_rs[ctb_addr_rs]) end_of_substream = true;
    if (P->entropy_coding_sync_enabled && (next_rs / ctbW) != ctby) end_of_substream = true;
    ctb_addr_rs = next_rs;
    if (end_of_substream) {
      if (!cabac.decode_terminate()) return "end_of_subset_one_bit is not set";
      // the next substream starts at the byte after the last one fetched by the engine
      const uint8_t* p = cabac.position();
      if (p >= cabac.end) return "slice data truncated at a substream boundary";
      cabac.init(p, cabac.end);
      first_substream_of_independent = false;
      if (P->tiles_enabled) init_contexts();
    }
  }
  return "";
}

// ---------------------------------------------------------------------------------------------
void HevcIntraParser::Impl::decode_ctu() {
  const int ctb = 1 << S->log2_ctb;
  int rx = ctb_addr_rs % S->ctbs_w, ry = ctb_addr_rs / S->ctbs_w;
  hc_ctu& ctu = rec->ctus[ctb_addr_rs];
  for (int c = 0; c < 3; c++) ctu_blks[c].clear();

  if (sh->sao_luma || sh->sao_chroma) read_sao(rx, ry, ctu);

  coding_quadtree(rx * ctb, ry * ctb, S->log2_ctb, 0);
  if (!error.empty()) return;

  for (int c = 0; c < 3; c++) {
    ctu.blk_first[c] = (uint32_t)rec->blks.size();
    if (ctu_blks[c].size() > 65535) { error = "too many blocks in one CTB"; return; }
    ctu.blk_count[c] = (uint16_t)ctu_blks[c].size();
    rec->blks.insert(rec->blks.end(), ctu_blks[c].begin(), ctu_blks[c].end());
  }
  ctu.beta_offset = (int8_t)sh->beta_offset;
  ctu.tc_offset = (int8_t)sh->tc_offset;
  if (sh->deblocking_disabled) ctu.flags |= HC_CTU_DEBLOCK_OFF;
}

// §7.3.8.3 sample adaptive offset syntax
void HevcIntraParser::Impl::read_sao(int rx, int ry, hc_ctu& ctu) {
  bool merge_left = false, merge_up = false;
  if (rx > 0) {
    int left = ctb_addr_rs - 1;
    bool in_slice = ctb_slice_addr[left] == sh->slice_addr_rs;
    bool in_tile = P->tile_id_rs[left] == P->tile_id_rs[ctb_addr_rs];
    if (in_slice && in_tile) merge_left = bin(CTX_SAO_MERGE);
  }
  if (ry > 0 && !merge_left) {
    int up = ctb_addr_rs - S->ctbs_w;
    bool in_slice = ctb_slice_addr[up] == sh->slice_addr_rs;
    bool in_tile = P->tile_id_rs[up] == P->tile_id_rs[ctb_addr_rs];
    if (in_slice && in_tile) merge_up = bin(CTX_SAO_MERGE);
  }
  if (merge_left || merge_up) {
    const hc_ctu& src = rec->ctus[merge_left ? ctb_addr_rs - 1 : ctb_addr_rs - S->ctbs_w];
    memcpy(ctu.sao_type, src.sao_type, 3);
    memcpy(ctu.sao_band_or_class, src.sao_band_or_class, 3);
    memcpy(ctu.sao_offset, src.sao_offset, 12);
    // slice_sao_luma/chroma gating is per slice: re-apply for this CTB's slice
    if (!sh->sao_luma) ctu.sao_type[0] = 0;
    if (!sh->sao_chroma) ctu.sao_type[1] = ctu.sao_type[2] = 0;
    return;
  }
  int ncomp = S->ChromaArrayType != 0 ? 3 : 1;
  for (int c = 0; c < ncomp; c++) {
    if (!((sh->sao_luma && c == 0) || (sh->sao_chroma && c > 0))) {
      ctu.sao_type[c] = 0;
      continue;
    }
    if (c == 0 || c == 1) {
      int t = 0;
      if (bin(CTX_SAO_TYPE)) t = cabac.decode_bypass() ? 2 : 1;
      ctu.sao_type[c] = (uint8_t)t;
    } else {
      ctu.sao_type[2] = ctu.sao_type[1];
    }
    if (ctu.sao_type[c] == 0) continue;
    int bitDepth = c == 0 ? S->bit_depth_y : S->bit_depth_c;
    int cMax = (1 << (std::min(bitDepth, 10) - 5)) - 1;
    int absv[4];
    for (int i = 0; i < 4; i++) {
      int v = 0;
      while (v < cMax && cabac.decode_bypass()) v++;
      absv[i] = v;
    }
    int log2scale = c == 0 ? P->log2_sao_offset_scale_luma : P->log2_sao_offset_scale_chroma;
    if (ctu.sao_type[c] == 1) {
      int sign[4] = {0, 0, 0, 0};
      for (int i = 0; i < 4; i++)
        if (absv[i]) sign[i] = cabac.decode_bypass();
      ctu.sao_band_or_class[c] = (uint8_t)cabac.decode_bypass_bits(5);
      for (int i = 0; i < 4; i++)
        ctu.sao_offset[c][i] = (int8_t)((sign[i] ? -absv[i] : absv[i]) * (1 << log2scale));
    } else {
      if (c == 0 || c == 1) ctu.sao_band_or_class[c] = (uint8_t)cabac.decode_bypass_bits(2);
      else ctu.sao_band_or_class[2] = ctu.sao_band_or_class[1];
      ctu.sao_offset[c][0] = (int8_t)(absv[0] * (1 << log2scale));
      ctu.sao_offset[c][1] = (int8_t)(absv[1] * (1 << log2scale));
      ctu.sao_offset[c][2] = (int8_t)(-absv[2] * (1 << log2scale));
      ctu.sao_offset[c][3] = (int8_t)(-absv[3] * (1 << log2scale));
    }
  }
}

// §7.3.8.4
void HevcIntraParser::Impl::coding_quadtree(int x0, int y0, int log2, int depth) {
  if (!error.empty() || cabac.overrun()) return;
  int size = 1 << log2;
  bool split;
  if (x0 + size <= W && y0 + size <= H && log2 > S->log2_min_cb) {
    int condL = 0, condA = 0;
    if (ctb_available(x0, y0, x0 - 1, y0) && ct_depth[((x0 - 1) >> 3) + (size_t)(y0 >> 3) * w8] > depth) condL = 1;
    if (ctb_available(x0, y0, x0, y0 - 1) && ct_depth[(x0 >> 3) + (size_t)((y0 - 1) >> 3) * w8] > depth) condA = 1;
    split = bin(CTX_SPLIT_CU + condL + condA);
  } else {
    split = log2 > S->log2_min_cb;
  }
  if (P->cu_qp_delta_enabled && log2 >= P->log2_min_cu_qp_delta_size) {
    IsCuQpDeltaCoded = false;
    CuQpDeltaVal = 0;
  }
  if (sh->cu_chroma_qp_offset_enabled && log2 >= P->log2_min_cu_chroma_qp_offset_size)
    IsCuChromaQpOffsetCoded = false;
  if (split) {
    int h = size >> 1;
    int x1 = x0 + h, y1 = y0 + h;
    coding_quadtree(x0, y0, log2 - 1, depth + 1);
    if (x1 < W) coding_quadtree(x1, y0, log2 - 1, depth + 1);
    if (y1 < H) coding_quadtree(x0, y1, log2 - 1, depth + 1);
    if (x1 < W && y1 < H) coding_quadtree(x1, y1, log2 - 1, depth + 1);
  } else {
    coding_unit(x0, y0, log2, depth);
  }
}

// §8.6.1 with the bookkeeping of transform.cc:31-210
void HevcIntraParser::Impl::derive_qp(int xCU, int yCU) {
  int qgmask = (1 << P->log2_min_cu_qp_delta_size) - 1;
  int xQG = xCU - (xCU & qgmask), yQG = yCU - (yCU & qgmask);
  if (xQG != currentQG_x || yQG != currentQG_y) {
    lastQPYinPreviousQG = currentQPY;
    currentQG_x = xQG;
    currentQG_y = yQG;
  }
  int ctbmask = (1 << S->log2_ctb) - 1;
  bool firstInCTBRow = (xQG == 0 && (yQG & ctbmask) == 0);
  int sx = (sh->slice_addr_rs % S->ctbs_w) << S->log2_ctb;
  int sy = (sh->slice_addr_rs / S->ctbs_w) << S->log2_ctb;
  bool firstQGInSlice = (sx == xQG && sy == yQG);
  bool firstQGInTile = false;
  if (P->tiles_enabled && (xQG & ctbmask) == 0 && (yQG & ctbmask) == 0)
    firstQGInTile = P->tile_start_ctb[ctb_of(xQG, yQG)] != 0;
  int pred;
  if (firstQGInSlice || firstQGInTile || (firstInCTBRow && P->entropy_coding_sync_enabled)) pred = sh->slice_qp_y;
  else pred = lastQPYinPreviousQG;

  int shiftc = 2 * (S->log2_ctb - S->log2_min_tb);
  int qA = pred, qB = pred;
  if (available_zscan(xQG, yQG, xQG - 1, yQG)) {
    int ctbA = zs_addr(xQG - 1, yQG) >> shiftc;
    if (ctbA == ctb_addr_ts) qA = qp_y[((xQG - 1) >> 3) + (size_t)(yQG >> 3) * w8];
  }
  if (available_zscan(xQG, yQG, xQG, yQG - 1)) {
    int ctbB = zs_addr(xQG, yQG - 1) >> shiftc;
    if (ctbB == ctb_addr_ts) qB = qp_y[(xQG >> 3) + (size_t)((yQG - 1) >> 3) * w8];
  }
  pred = (qA + qB + 1) >> 1;
  int QPY = ((pred + CuQpDeltaVal + 52 + 2 * S->qp_bd_offset_y) % (52 + S->qp_bd_offset_y)) - S->qp_bd_offset_y;
  qPYPrime = std::max(0, QPY + S->qp_bd_offset_y);
  int qPiCb = clip3(-S->qp_bd_offset_c, 57, QPY + P->cb_qp_offset + sh->cb_qp_offset + CuQpOffsetCb);
  int qPiCr = clip3(-S->qp_bd_offset_c, 57, QPY + P->cr_qp_offset + sh->cr_qp_offset + CuQpOffsetCr);
  int qPCb, qPCr;
  if (S->ChromaArrayType == 1) {
    qPCb = qpc_table_420(qPiCb);
    qPCr = qpc_table_420(qPiCr);
  } else {  // reference: no Min(qPi,51) here (transform.cc:175-178)
    qPCb = qPiCb;
    qPCr = qPiCr;
  }
  qPCbPrime = std::max(0, qPCb + S->qp_bd_offset_c);
  qPCrPrime = std::max(0, qPCr + S->qp_bd_offset_c);
  // store QP_Y for the whole CU
  int n8 = std::max(1, (1 << cu_log2) >> 3);
  for (int y = 0; y < n8; y++)
    for (int x = 0; x < n8; x++) {
      int xx = (cu_x0 >> 3) + x, yy = (cu_y0 >> 3) + y;
      if (xx < w8 && yy < h8) qp_y[xx + (size_t)yy * w8] = (int8_t)QPY;
    }
  currentQPY = QPY;
}

// §7.3.8.5 (I slices)
void HevcIntraParser::Impl::coding_unit(int x0, int y0, int log2, int depth) {
  const int nCbS = 1 << log2;
  cu_x0 = x0; cu_y0 = y0; cu_log2 = log2;
  cu_transquant_bypass = false;
  if (P->transquant_bypass_enabled) cu_transquant_bypass = bin(CTX_TQ_BYPASS);

  // CU-level maps (8x8 granularity)
  {
    int n8 = nCbS >> 3;
    uint8_t fl = cu_transquant_bypass ? 2 : 0;
    for (int y = 0; y < n8; y++)
      for (int x = 0; x < n8; x++) {
        size_t i = ((x0 >> 3) + x) + (size_t)((y0 >> 3) + y) * w8;
        ct_depth[i] = (uint8_t)depth;
        cu_flags[i] = fl;
      }
  }

  // deblocking: which CU edges may be filtered (deblock.cc:165-215)
  filterLeftCbEdge = x0 != 0;
  filterTopCbEdge = y0 != 0;
  {
    int ctbmask = (1 << S->log2_ctb) - 1;
    if (x0 && (x0 & ctbmask) == 0) {
      int n = ctb_of(x0 - 1, y0);
      if (!sh->loop_filter_across_slices && ctb_slice_addr[n] >= 0 && ctb_slice_addr[n] != sh->slice_addr_rs)
        filterLeftCbEdge = 0;
      else if (!P->loop_filter_across_tiles && P->tile_id_rs[n] != P->tile_id_rs[ctb_of(x0, y0)])
        filterLeftCbEdge = 0;
    }
    if (y0 && (y0 & ctbmask) == 0) {
      int n = ctb_of(x0, y0 - 1);
      if (!sh->loop_filter_across_slices && ctb_slice_addr[n] >= 0 && ctb_slice_addr[n] != sh->slice_addr_rs)
        filterTopCbEdge = 0;
      else if (!P->loop_filter_across_tiles && P->tile_id_rs[n] != P->tile_id_rs[ctb_of(x0, y0)])
        filterTopCbEdge = 0;
    }
  }

  derive_qp(x0, y0);  // slice.cc:4593

  bool nxn = false;
  if (log2 == S->log2_min_cb) {
    // part_mode: one bin for intra CUs. NxN needs log2CbSize > MinTbLog2SizeY (§7.4.9.5).
    int b = bin(CTX_PART_MODE);
    nxn = !b;
    if (nxn && log2 <= S->log2_min_tb) { error = "PART_NxN in a coding block of minimum transform size"; return; }
  }

  bool pcm = false;
  if (!nxn && S->pcm_enabled && log2 >= S->log2_min_pcm_cb && log2 <= S->log2_max_pcm_cb)
    pcm = cabac.decode_terminate();

  if (pcm) {
    int n8 = nCbS >> 3;
    for (int y = 0; y < n8; y++)
      for (int x = 0; x < n8; x++) cu_flags[((x0 >> 3) + x) + (size_t)((y0 >> 3) + y) * w8] |= 1;
    // intra mode of a PCM CU reads as DC for its neighbours (§8.4.2)
    for (int y = 0; y < (nCbS >> 2); y++)
      for (int x = 0; x < (nCbS >> 2); x++) {
        ipm[((x0 >> 2) + x) + (size_t)((y0 >> 2) + y) * w4] = 1;
        ipm_c[((x0 >> 2) + x) + (size_t)((y0 >> 2) + y) * w4] = 1;
      }
    pcm_sample(x0, y0, log2);
    mark_tu_edges(x0, y0, log2);
    return;
  }

  // ---- intra prediction modes ----
  int pbOffset = nxn ? nCbS / 2 : nCbS;
  int nparts = nxn ? 4 : 1;
  int prev_flag[4], mpm_idx[4] = {0, 0, 0, 0}, rem[4] = {0, 0, 0, 0};
  for (int i = 0; i < nparts; i++) prev_flag[i] = bin(CTX_PREV_INTRA_LUMA);
  for (int i = 0; i < nparts; i++) {
    if (prev_flag[i]) {
      int v = 0;
      while (v < 2 && cabac.decode_bypass()) v++;
      mpm_idx[i] = v;
    } else {
      rem[i] = (int)cabac.decode_bypass_bits(5);
    }
  }
  bool availA0 = ctb_available(x0, y0, x0 - 1, y0);
  bool availB0 = ctb_available(x0, y0, x0, y0 - 1);
  int luma_modes[4];
  for (int idx = 0; idx < nparts; idx++) {
    int i = (idx & 1) * pbOffset, j = (idx >> 1) * pbOffset;
    int x = x0 + i, y = y0 + j;
    bool availA = availA0 || i > 0, availB = availB0 || j > 0;
    int candA = 1, candB = 1;
    if (availA) {
      if (cu_flags[((x - 1) >> 3) + (size_t)(y >> 3) * w8] & 1) candA = 1;
      else candA = ipm[((x - 1) >> 2) + (size_t)(y >> 2) * w4];
    }
    if (availB) {
      if (cu_flags[(x >> 3) + (size_t)((y - 1) >> 3) * w8] & 1) candB = 1;
      else if (y - 1 < ((y >> S->log2_ctb) << S->log2_ctb)) candB = 1;
      else candB = ipm[(x >> 2) + (size_t)((y - 1) >> 2) * w4];
    }
    int cand[3];
    if (candA == candB) {
      if (candA < 2) { cand[0] = 0; cand[1] = 1; cand[2] = 26; }
      else {
        cand[0] = candA;
        cand[1] = 2 + ((candA - 2 - 1 + 32) % 32);
        cand[2] = 2 + ((candA - 2 + 1) % 32);
      }
    } else {
      cand[0] = candA; cand[1] = candB;
      if (candA != 0 && candB != 0) cand[2] = 0;
      else if (candA != 1 && candB != 1) cand[2] = 1;
      else cand[2] = 26;
    }
    int mode;
    if (prev_flag[idx]) {
      mode = cand[mpm_idx[idx]];
    } else {
      if (cand[0] > cand[1]) std::swap(cand[0], cand[1]);
      if (cand[0] > cand[2]) std::swap(cand[0], cand[2]);
      if (cand[1] > cand[2]) std::swap(cand[1], cand[2]);
      mode = rem[idx];
      for (int n = 0; n < 3; n++)
        if (mode >= cand[n]) mode++;
    }
    luma_modes[idx] = mode;
    int n4 = pbOffset >> 2;
    for (int yy = 0; yy < n4; yy++)
      for (int xx = 0; xx < n4; xx++) ipm[((x >> 2) + xx) + (size_t)((y >> 2) + yy) * w4] = (uint8_t)mode;
  }

  auto chroma_mode = [&](int icpm, int luma) -> int {
    if (icpm == 4) return luma;
    static const int cands[4] = {0, 26, 10, 1};
    int m = cands[icpm];
    return m == luma ? 34 : m;
  };
  auto read_icpm = [&]() -> int {
    if (!bin(CTX_INTRA_CHROMA)) return 4;
    return (int)cabac.decode_bypass_bits(2);
  };
  if (S->ChromaArrayType == 3) {
    for (int idx = 0; idx < nparts; idx++) {
      int i = (idx & 1) * pbOffset, j = (idx >> 1) * pbOffset;
      int m = chroma_mode(read_icpm(), luma_modes[idx]);
      int n4 = pbOffset >> 2;
      for (int yy = 0; yy < n4; yy++)
        for (int xx = 0; xx < n4; xx++)
          ipm_c[(((x0 + i) >> 2) + xx) + (size_t)(((y0 + j) >> 2) + yy) * w4] = (uint8_t)m;
    }
  } else if (S->ChromaArrayType != 0) {
    int m = chroma_mode(read_icpm(), luma_modes[0]);
    if (S->ChromaArrayType == 2) m = kMode422[m];
    int n4 = nCbS >> 2;
    for (int yy = 0; yy < n4; yy++)
      for (int xx = 0; xx < n4; xx++) ipm_c[((x0 >> 2) + xx) + (size_t)((y0 >> 2) + yy) * w4] = (uint8_t)m;
  }

  int max_depth = S->max_th_depth_intra + (nxn ? 1 : 0);
  transform_tree(x0, y0, x0, y0, log2, 0, 0, max_depth, nxn ? 1 : 0, 1, 1);
}

// §7.3.8.7 pcm_sample(): samples are carried as a dense bypass-type block so that the GPU path
// needs no special input channel.
void HevcIntraParser::Impl::pcm_sample(int x0, int y0, int log2) {
  // PCM data starts at the byte after the last one fetched by the arithmetic decoder
  const uint8_t* p = cabac.position();
  BitReader br(p, (size_t)(cabac.end > p ? cabac.end - p : 0));
  int ncomp = S->ChromaArrayType != 0 ? 3 : 1;
  for (int c = 0; c < ncomp; c++) {
    int lw = log2, lh = log2;
    if (c > 0) {
      if (S->SubWidthC == 2) lw--;
      if (S->SubHeightC == 2) lh--;
    }
    int w = 1 << lw, h = 1 << lh;
    int pcm_bits = c == 0 ? S->pcm_bit_depth_y : S->pcm_bit_depth_c;
    int depth = c == 0 ? S->bit_depth_y : S->bit_depth_c;
    int shift = depth - pcm_bits;
    // split non-square (4:2:2 chroma: w x 2w) into square blocks of side w
    int nsq = h / w;
    std::vector<int> samples((size_t)w * h);
    for (int i = 0; i < w * h; i++) samples[i] = (int)br.u(pcm_bits) << shift;
    for (int s = 0; s < nsq; s++) {
      hc_tb tb;
      memset(&tb, 0, sizeof(tb));
      tb.coeff_off = (uint32_t)rec->coeffs.size();
      tb.resid_off = (uint32_t)rec->resid_count;
      tb.log2 = (uint8_t)lw;
      tb.type = (uint8_t)(c | HC_TB_BYPASS);
      int n = 0;
      for (int y = 0; y < w; y++)
        for (int x = 0; x < w; x++) {
          int v = samples[(size_t)(s * w + y) * w + x];
          if (v) {
            hc_coeff co;
            co.pos = (uint16_t)(x + y * w);
            co.level = (int16_t)v;
            rec->coeffs.push_back(co);
            n++;
          }
        }
      tb.ncoeff = (uint16_t)n;
      rec->tbs.push_back(tb);
      rec->tbs_by_size[tb.log2 - 2]++;
      rec->resid_count += (uint64_t)w * w;
      int xB = c == 0 ? x0 : x0 / S->SubWidthC;
      int yB = (c == 0 ? y0 : y0 / S->SubHeightC) + s * w;
      emit_blk(c, xB, yB, lw, 1, true, tb.resid_off, HC_BLK_PCM);
    }
  }
  if (br.overrun) { error = "PCM samples truncated"; return; }
  const uint8_t* np = p + br.byte_pos();
  cabac.init(np, cabac.end);
}

// marks the left/top edge of a transform block (deblock.cc:31-62) — bS is 2 everywhere in
// intra pictures (deblock.cc:275-277), so one bit per direction suffices.
void HevcIntraParser::Impl::mark_tu_edges(int x0, int y0, int log2) {
  if (sh->deblocking_disabled) return;
  int n4 = (1 << log2) >> 2;
  int left = (x0 == cu_x0) ? filterLeftCbEdge : 1;
  int top = (y0 == cu_y0) ? filterTopCbEdge : 1;
  if (left)
    for (int k = 0; k < n4; k++) rec->edge_map[(x0 >> 2) + (size_t)((y0 >> 2) + k) * w4] |= HC_EDGE_V;
  if (top)
    for (int k = 0; k < n4; k++) rec->edge_map[((x0 >> 2) + k) + (size_t)(y0 >> 2) * w4] |= HC_EDGE_H;
}

// §7.3.8.8
void HevcIntraParser::Impl::transform_tree(int x0, int y0, int xBase, int yBase, int log2, int depth,
                                           int blkIdx, int max_depth, int intra_split,
                                           int parent_cbf_cb, int parent_cbf_cr) {
  if (!error.empty() || cabac.overrun()) return;
  int split;
  if (log2 <= S->log2_max_tb && log2 > S->log2_min_tb && depth < max_depth && !(intra_split && depth == 0)) {
    split = bin(CTX_SPLIT_TRANSFORM + 5 - log2);
  } else {
    split = (log2 > S->log2_max_tb || (intra_split && depth == 0)) ? 1 : 0;
  }
  int cbf_cb = -1, cbf_cr = -1;
  if ((log2 > 2 && S->ChromaArrayType != 0) || S->ChromaArrayType == 3) {
    if (parent_cbf_cb) {
      cbf_cb = bin(CTX_CBF_CHROMA + depth);
      if (S->ChromaArrayType == 2 && (!split || log2 == 3)) cbf_cb |= bin(CTX_CBF_CHROMA + depth) << 1;
    }
    if (parent_cbf_cr) {
      cbf_cr = bin(CTX_CBF_CHROMA + depth);
      if (S->ChromaArrayType == 2 && (!split || log2 == 3)) cbf_cr |= bin(CTX_CBF_CHROMA + depth) << 1;
    }
  }
  if (cbf_cb < 0) cbf_cb = (depth > 0 && log2 == 2) ? parent_cbf_cb : 0;
  if (cbf_cr < 0) cbf_cr = (depth > 0 && log2 == 2) ? parent_cbf_cr : 0;

  if (split) {
    int h = 1 << (log2 - 1);
    transform_tree(x0, y0, x0, y0, log2 - 1, depth + 1, 0, max_depth, intra_split, cbf_cb, cbf_cr);
    transform_tree(x0 + h, y0, x0, y0, log2 - 1, depth + 1, 1, max_depth, intra_split, cbf_cb, cbf_cr);
    transform_tree(x0, y0 + h, x0, y0, log2 - 1, depth + 1, 2, max_depth, intra_split, cbf_cb, cbf_cr);
    transform_tree(x0 + h, y0 + h, x0, y0, log2 - 1, depth + 1, 3, max_depth, intra_split, cbf_cb, cbf_cr);
  } else {
    int cbf_luma = bin(CTX_CBF_LUMA + (depth == 0 ? 1 : 0));  // intra: always coded
    transform_unit(x0, y0, xBase, yBase, log2, depth, blkIdx, cbf_luma, cbf_cb, cbf_cr);
  }
}

// neighbour availability of one prediction block, in units of 4 component samples
// (mirror of intrapred.h:443-543 preproc + :838-940 z-scan tests)
void HevcIntraParser::Impl::emit_blk(int cIdx, int xB, int yB, int log2, int mode, bool has_resid,
                                     uint32_t resid_off, uint8_t extra_flags) {
  const int nT = 1 << log2;
  const int SubW = cIdx == 0 ? 1 : S->SubWidthC, SubH = cIdx == 0 ? 1 : S->SubHeightC;
  const int xBL = xB * SubW, yBL = yB * SubH;
  bool aL = true, aT = true, aTR = true, aTL = true;
  if (xBL == 0) { aL = false; aTL = false; }
  if (yBL == 0) { aT = false; aTL = false; aTR = false; }
  if (xBL + nT * SubW >= W) aTR = false;
  const int l2c = S->log2_ctb;
  int xCur = xBL >> l2c, yCur = yBL >> l2c;
  int xLeft = (xBL - 1) >> l2c, xRight = (xBL + nT * SubW) >> l2c, yTop = (yBL - 1) >> l2c;
  int cw = S->ctbs_w;
  int cur = xCur + yCur * cw;
  auto same = [&](int cx, int cy) -> bool {
    int n = cx + cy * cw;
    return ctb_slice_addr[n] == ctb_slice_addr[cur] && P->tile_id_rs[n] == P->tile_id_rs[cur];
  };
  if (aL && !same(xLeft, yCur)) aL = false;
  if (aT && !same(xCur, yTop)) aT = false;
  if (aTL && !same(xLeft, yTop)) aTL = false;
  if (aTR && !same(xRight, yTop)) aTR = false;

  int nBottom = (H - yBL + SubH - 1) / SubH;
  if (nBottom > 2 * nT) nBottom = 2 * nT;
  int nRight = (W - xBL + SubW - 1) / SubW;
  if (nRight > 2 * nT) nRight = 2 * nT;

  const int currAddr = zs_addr(xBL, yBL);
  uint16_t left = 0, top = 0;
  if (aL)
    for (int y = nBottom - 1; y >= 0; y -= 4)
      if (zs_addr((xB - 1) * SubW, (yB + y) * SubH) <= currAddr) left |= (uint16_t)(1u << (y >> 2));
  bool tl = false;
  if (aTL) tl = zs_addr((xB - 1) * SubW, (yB - 1) * SubH) <= currAddr;
  for (int x = 0; x < nRight; x += 4) {
    bool ba = x < nT ? aT : aTR;
    if (ba && zs_addr((xB + x) * SubW, (yB - 1) * SubH) <= currAddr) top |= (uint16_t)(1u << (x >> 2));
  }

  hc_blk b;
  b.x = (uint16_t)xB;
  b.y = (uint16_t)yB;
  b.log2 = (uint8_t)log2;
  b.mode = (uint8_t)mode;
  b.flags = (uint8_t)(extra_flags | (tl ? HC_BLK_AVAIL_TL : 0) | (has_resid ? HC_BLK_HAS_RESID : 0));
  b.cidx = (uint8_t)cIdx;
  b.avail_left = left;
  b.avail_top = top;
  b.resid_off = has_resid ? resid_off : 0;
  ctu_blks[cIdx].push_back(b);
}

// §7.3.8.10 transform_unit + record emission in the reference's reconstruction order
// (slice.cc:3979-4118)
void HevcIntraParser::Impl::transform_unit(int x0, int y0, int xBase, int yBase, int log2, int depth,
                                           int blkIdx, int cbf_luma, int cbf_cb, int cbf_cr) {
  (void)depth;
  const int cat = S->ChromaArrayType;
  int log2C = std::max(2, cat == 3 ? log2 : log2 - 1);
  int cbfChroma = cbf_cb | cbf_cr;
  if (cbf_luma || cbfChroma) {
    bool redo = false;
    if (P->cu_qp_delta_enabled && !IsCuQpDeltaCoded) {
      // cu_qp_delta_abs: prefix TU(5) with contexts 0,1,1,1,1 then EG0 suffix
      int v = 0;
      if (bin(CTX_CU_QP_DELTA)) {
        v = 1;
        while (v < 5 && bin(CTX_CU_QP_DELTA + 1)) v++;
        if (v == 5) {
          int k = 0;
          while (k < 32 && cabac.decode_bypass()) k++;
          if (k >= 32) { error = "cu_qp_delta_abs out of range"; return; }
          v += ((1 << k) - 1) + (int)cabac.decode_bypass_bits(k);
        }
      }
      int sign = 0;
      if (v) sign = cabac.decode_bypass();
      IsCuQpDeltaCoded = true;
      CuQpDeltaVal = sign ? -v : v;
      redo = true;
    }
    if (sh->cu_chroma_qp_offset_enabled && cbfChroma && !cu_transquant_bypass && !IsCuChromaQpOffsetCoded) {
      int flag = bin(CTX_CHROMA_QP_OFFSET_FLAG);
      int idx = 0;
      // cu_chroma_qp_offset_idx: truncated rice with cMax = chroma_qp_offset_list_len_minus1 and every bin in the one
      // context (H.265 9.3.3, as HM reads it); a single bin loses sync on lists of more than two entries
      if (flag) while (idx < P->chroma_qp_offset_list_len - 1 && bin(CTX_CHROMA_QP_OFFSET_IDX)) idx++;
      IsCuChromaQpOffsetCoded = true;
      if (flag) {
        CuQpOffsetCb = P->cb_qp_offset_list[idx];
        CuQpOffsetCr = P->cr_qp_offset_list[idx];
      } else {
        CuQpOffsetCb = CuQpOffsetCr = 0;
      }
      redo = true;
    }
    if (redo) derive_qp(cu_x0, cu_y0);
  }

  mark_tu_edges(x0, y0, log2);

  uint8_t noedge = 0;
  // disableIntraBoundaryFilter as evaluated by the reference: the bypass flag is looked up at the
  // block position in *component* coordinates (intrapred.cc:318-320)
  auto noedge_at = [&](int xB, int yB) -> uint8_t {
    if (!S->implicit_rdpcm_enabled) return 0;
    int xx = std::min(xB, W - 1), yy = std::min(yB, H - 1);
    return (cu_flags[(xx >> 3) + (size_t)(yy >> 3) * w8] & 2) ? HC_BLK_NO_EDGE_FLT : 0;
  };
  (void)noedge;

  // ---- luma ----
  int modeY = ipm[(x0 >> 2) + (size_t)(y0 >> 2) * w4];
  uint32_t roff = 0;
  if (cbf_luma) roff = residual_coding(x0, y0, log2, 0, modeY);
  if (!error.empty()) return;
  emit_blk(0, x0, y0, log2, modeY, cbf_luma != 0, roff, noedge_at(x0, y0));

  if (cat == 0) return;
  const int SubW = S->SubWidthC, SubH = S->SubHeightC;

  if (log2 > 2 || cat == 3) {
    int modeC = ipm_c[(x0 >> 2) + (size_t)(y0 >> 2) * w4];
    int nTC = 1 << log2C;
    for (int c = 1; c <= 2; c++) {
      int cbf = c == 1 ? cbf_cb : cbf_cr;
      int nblk = cat == 2 ? 2 : 1;
      for (int t = 0; t < nblk; t++) {
        int xB = x0 / SubW, yB = y0 / SubH + t * nTC;
        // chroma mode lookup position used by the reference for this block (slice.cc:3760-3763)
        int lx = xB * SubW, ly = yB * SubH;
        int m = ipm_c[(std::min(lx, W - 1) >> 2) + (size_t)(std::min(ly, H - 1) >> 2) * w4];
        (void)modeC;
        uint32_t ro = 0;
        bool coded = (cbf >> t) & 1;
        if (coded) ro = residual_coding(x0, y0 + t * nTC * SubH, log2C, c, m);
        if (!error.empty()) return;
        emit_blk(c, xB, yB, log2C, m, coded, ro, noedge_at(xB, yB));
      }
    }
  } else if (blkIdx == 3) {
    // 4x4 luma blocks: chroma of the parent 8x8 is coded with the last luma block
    int nTC = 4;
    for (int c = 1; c <= 2; c++) {
      int cbf = c == 1 ? cbf_cb : cbf_cr;
      int nblk = cat == 2 ? 2 : 1;
      for (int t = 0; t < nblk; t++) {
        int xB = xBase / SubW, yB = yBase / SubH + t * nTC;
        int lx = xB * SubW, ly = yB * SubH;
        int m = ipm_c[(std::min(lx, W - 1) >> 2) + (size_t)(std::min(ly, H - 1) >> 2) * w4];
        uint32_t ro = 0;
        bool coded = (cbf >> t) & 1;
        if (coded) ro = residual_coding(xBase, yBase + t * nTC * SubH, 2, c, m);
        if (!error.empty()) return;
        emit_blk(c, xB, yB, 2, m, coded, ro, noedge_at(xB, yB));
      }
    }
  }
}

// §7.3.8.11 residual_coding + §9.3.4.2.4-9.3.4.2.7 context selection
// sig_coeff_flag ctxInc (9.3.4.2.5) for every scan position, built once:
//   b4[chroma][scanIdx][k]                                   4x4 blocks (Table 9-50 ctxIdxMap)
//   sb[chroma][size class][sub-block != (0,0)][prevCsbf][scanIdx][k]   size class 0: 8x8 diagonal, 1: 8x8 hor/ver, 2: 16/32
//   ts[chroma][k]                                            transform_skip_context_enabled blocks
// (the DC position of sub-block (0,0) of blocks > 4x4 is context 0 and handled by the caller)
struct SigCtxTables {
  uint8_t b4[2][3][16];
  uint8_t sb[2][3][2][4][3][16];
  uint8_t ts[2][16];
  SigCtxTables() {
    const ScanTables& st = scan_tables();
    for (int c = 0; c < 2; c++) {
      for (int k = 0; k < 16; k++) ts[c][k] = (uint8_t)(c == 0 ? 42 : 43);
      for (int s = 0; s < 3; s++)
        for (int k = 0; k < 16; k++) {
          const int xP = st.order[2][s][k].x, yP = st.order[2][s][k].y;
          b4[c][s][k] = (uint8_t)((c ? 27 : 0) + kSigCtx4x4[(yP << 2) + xP]);
          for (int cls = 0; cls < 3; cls++)
            for (int nz = 0; nz < 2; nz++)
              for (int prev = 0; prev < 4; prev++) {
                int v;
                switch (prev) {
                  case 0: v = (xP + yP >= 3) ? 0 : (xP + yP > 0) ? 1 : 2; break;
                  case 1: v = (yP == 0) ? 2 : (yP == 1) ? 1 : 0; break;
                  case 2: v = (xP == 0) ? 2 : (xP == 1) ? 1 : 0; break;
                  default: v = 2; break;
                }
                if (c == 0) {
                  if (nz) v += 3;
                  v += cls == 0 ? 9 : (cls == 1 ? 15 : 21);
                } else {
                  v += cls == 2 ? 12 : 9;
                }
                sb[c][cls][nz][prev][s][k] = (uint8_t)((c ? 27 : 0) + v);
              }
        }
    }
  }
};
static const SigCtxTables& sig_ctx_tables() {
  static const SigCtxTables t;
  return t;
}

uint32_t HevcIntraParser::Impl::residual_coding(int x0, int y0, int log2, int cIdx, int pred_mode) {
  (void)x0; (void)y0;
  const ScanTables& st = scan_tables();
  bool tskip = false;
  if (P->transform_skip_enabled && !cu_transquant_bypass && log2 <= P->log2_max_transform_skip_size)
    tskip = bin(CTX_TSKIP + (cIdx ? 1 : 0));

  int sbType = cIdx == 0 ? 2 : 0;
  if (tskip || cu_transquant_bypass) sbType++;

  // last significant coefficient position
  auto last_prefix = [&](int base) -> int {
    int cMax = (log2 << 1) - 1;
    int offset, shift;
    if (cIdx == 0) { offset = 3 * (log2 - 2) + ((log2 - 1) >> 2); shift = (log2 + 1) >> 2; }
    else { offset = 15; shift = log2 - 2; }
    int v = 0;
    while (v < cMax && bin(base + offset + (v >> shift))) v++;
    return v;
  };
  int px = last_prefix(CTX_LAST_X);
  int py = last_prefix(CTX_LAST_Y);
  int LastX = px, LastY = py;
  if (px > 3) {
    int nb = (px >> 1) - 1;
    LastX = ((2 + (px & 1)) << nb) + (int)cabac.decode_bypass_bits(nb);
  }
  if (py > 3) {
    int nb = (py >> 1) - 1;
    LastY = ((2 + (py & 1)) << nb) + (int)cabac.decode_bypass_bits(nb);
  }

  int scanIdx = 0;
  if (log2 == 2 || (log2 == 3 && (cIdx == 0 || S->ChromaArrayType == 3))) {
    if (pred_mode >= 6 && pred_mode <= 14) scanIdx = 2;
    else if (pred_mode >= 22 && pred_mode <= 30) scanIdx = 1;
  }
  if (scanIdx == 2) std::swap(LastX, LastY);
  const int nT = 1 << log2;
  if (LastX >= nT || LastY >= nT) { error = "last significant coefficient outside the block"; return 0; }

  const ScanPos* scanSub = st.order[log2 - 2][scanIdx];
  const ScanPos* scanPos = st.order[2][scanIdx];
  const int sbW = 1 << (log2 - 2);

  // locate the last sub-block / position
  const int lastSubBlock = st.inverse[log2 - 2][scanIdx][(LastX >> 2) + ((LastY >> 2) << (log2 - 2))];
  const int lastScanPos = st.inverse[2][scanIdx][(LastX & 3) + ((LastY & 3) << 2)];

  uint8_t csbf_nb[64];
  memset(csbf_nb, 0, (size_t)sbW * sbW);

  hc_tb tb;
  memset(&tb, 0, sizeof(tb));
  tb.coeff_off = (uint32_t)rec->coeffs.size();
  tb.resid_off = (uint32_t)rec->resid_count;
  tb.log2 = (uint8_t)log2;
  tb.qp = (uint8_t)(cIdx == 0 ? qPYPrime : (cIdx == 1 ? qPCbPrime : qPCrPrime));
  tb.matrix_id = (uint8_t)(log2 == 5 ? 0 : cIdx);   // transform.cc:512-517 (intra)
  uint8_t type = (uint8_t)cIdx;
  if (cu_transquant_bypass) type |= HC_TB_BYPASS;
  else if (tskip) type |= HC_TB_TSKIP;
  else if (log2 == 2 && cIdx == 0) type |= HC_TB_DST;
  if (S->implicit_rdpcm_enabled && (cu_transquant_bypass || tskip) && (pred_mode == 10 || pred_mode == 26))
    type |= (pred_mode == 26) ? HC_TB_RDPCM_V : HC_TB_RDPCM_H;
  if (S->transform_skip_rotation_enabled && log2 == 2 && (cu_transquant_bypass || tskip)) type |= HC_TB_ROTATE;
  tb.type = type;

  const bool ts_ctx = S->transform_skip_context_enabled && (cu_transquant_bypass || tskip);
  const bool sign_hiding_possible =
      P->sign_data_hiding && !(cu_transquant_bypass ||
                               (S->implicit_rdpcm_enabled && tskip && (pred_mode == 10 || pred_mode == 26)));
  int c1 = 1;
  int ncoeff_total = 0;
  hc_coeff cbuf[1024];
  const SigCtxTables& sig = sig_ctx_tables();

  for (int i = lastSubBlock; i >= 0; i--) {
    const int Sx = scanSub[i].x, Sy = scanSub[i].y;
    int inferSbDc = 0;
    int coded = 0;
    if (i < lastSubBlock && i > 0) {
      int nb = csbf_nb[Sx + Sy * sbW];
      coded = bin(CTX_CSBF + (nb ? 1 : 0) + (cIdx ? 2 : 0));
      inferSbDc = 1;
    } else {
      coded = 1;
    }
    if (coded) {
      if (Sx > 0) csbf_nb[Sx - 1 + Sy * sbW] |= 1;
      if (Sy > 0) csbf_nb[Sx + (Sy - 1) * sbW] |= 2;
    }
    if (!coded) continue;

    int16_t value[16];
    int8_t spos[16];
    uint8_t maxbase[16];
    int n = 0;
    const int prevCsbf = csbf_nb[Sx + Sy * sbW];
    const int xS0 = Sx << 2, yS0 = Sy << 2;

    // sig_coeff_flag context per scan position of this sub-block (9.3.4.2.5), table driven
    const uint8_t* sigtab = ts_ctx ? sig.ts[cIdx ? 1 : 0]
                          : log2 == 2 ? sig.b4[cIdx ? 1 : 0][scanIdx]
                                      : sig.sb[cIdx ? 1 : 0][log2 == 3 ? (scanIdx == 0 ? 0 : 1) : 2][(Sx | Sy) ? 1 : 0][prevCsbf][scanIdx];
    const int dc_ctx = (ts_ctx || log2 == 2 || i > 0) ? sigtab[0] : (cIdx ? 27 : 0);

    // significant-coefficient flags: positions are written unconditionally and the count advances by the
    // decoded bin, so the (unpredictable) flag never steers a branch
    int last_coeff = (i == lastSubBlock) ? lastScanPos - 1 : 15;
    if (i == lastSubBlock) spos[n++] = (int8_t)lastScanPos;
    for (int k = last_coeff; k > 0; k--) {
      const int b = bin(CTX_SIG + sigtab[k]);
      spos[n] = (int8_t)k;
      n += b;
    }
    if (last_coeff >= 0) {
      if (n > 0 || !inferSbDc) {      // a significant flag was seen (or nothing can be inferred): DC flag is coded
        const int b = bin(CTX_SIG + dc_ctx);
        spos[n] = 0;
        n += b;
      } else {
        spos[n++] = 0;                // inferred: the only coefficient of a coded sub-block
      }
    }
    if (n == 0) continue;

    // greater1 / greater2 flags. base[c] = 1 + g1 (+ g2); a coefficient carries coeff_abs_level_remaining when its
    // base reached what the flags can express: 2 without g2, 3 for the one coefficient that had a g2 flag, 1 past the 8th
    int ctxSet = (i == 0 || cIdx > 0) ? 0 : 2;
    if (c1 == 0) ctxSet++;
    c1 = 1;
    int firstG1 = 16;
    const int ng1 = std::min(8, n);
    const int g1base = CTX_G1 + ctxSet * 4 + (cIdx > 0 ? 16 : 0);
    static const uint8_t c1next[8] = {0, 0, 2, 0, 3, 0, 3, 0};   // [c1 * 2 + bin]
    for (int c = 0; c < ng1; c++) {
      const int b = bin(g1base + c1);
      value[c] = (int16_t)(1 + b);
      maxbase[c] = (uint8_t)b;
      firstG1 = (b && c < firstG1) ? c : firstG1;
      c1 = c1next[c1 * 2 + b];
    }
    for (int c = ng1; c < n; c++) { value[c] = 1; maxbase[c] = 1; }
    if (firstG1 < 16) {
      int f = bin(CTX_G2 + ctxSet + (cIdx > 0 ? 4 : 0));
      value[firstG1] += f;
      maxbase[firstG1] = (uint8_t)f;
    }

    bool signHidden = sign_hiding_possible && (spos[0] - spos[n - 1] > 3);
    uint32_t signs = 0;
    int nsign = signHidden ? n - 1 : n;
    signs = cabac.decode_bypass_bits(nsign) << (16 - nsign);  // bit 15 = first coefficient

    int sumAbs = 0;
    int rice = S->persistent_rice_adaptation_enabled ? stat_coeff[sbType] / 4 : 0;
    bool firstRemaining = true;
    for (int c = 0; c < n; c++) {
      int base = value[c];
      int rem = 0;
      if (maxbase[c]) {
        // coeff_abs_level_remaining (§9.3.3.11): prefix of ones, TR / EGk suffix
        // fast path: prefix (ones + terminating zero) and suffix inside the next 16 bypass bins
        const uint32_t q16 = cabac.peek_bypass16();
        const int ones = q16 == 0xffffu ? 16 : __builtin_clz(~(q16 << 16));
        const int suffix_len = ones <= 3 ? rice : ones - 3 + rice;
        const int len = ones + 1 + suffix_len;
        if (len <= 16) {
          const uint32_t bins = q16 >> (16 - len);
          const int suffix = (int)(bins & ((1u << suffix_len) - 1u));
          rem = ones <= 3 ? (ones << rice) + suffix : (((1 << (ones - 3)) + 3 - 1) << rice) + suffix;
          cabac.consume_bypass(len, bins);
        } else {
          int prefix = 0;
          while (prefix < 32 && cabac.decode_bypass()) prefix++;
          if (prefix >= 32) { error = "coeff_abs_level_remaining prefix too long"; return 0; }
          if (prefix <= 3) rem = (prefix << rice) + (int)cabac.decode_bypass_bits(rice);
          else rem = (((1 << (prefix - 3)) + 3 - 1) << rice) + (int)cabac.decode_bypass_bits(prefix - 3 + rice);
        }
        if (base + rem > 3 * (1 << rice)) {
          rice++;
          if (!S->persistent_rice_adaptation_enabled && rice > 4) rice = 4;
        }
        if (S->persistent_rice_adaptation_enabled && firstRemaining) {
          if (rem >= (3 << (stat_coeff[sbType] / 4))) stat_coeff[sbType]++;
          else if (2 * rem < (1 << (stat_coeff[sbType] / 4)) && stat_coeff[sbType] > 0) stat_coeff[sbType]--;
        }
        firstRemaining = false;
      }
      int16_t level = (int16_t)(base + rem);  // int16 wrap like the reference (slice.cc:3671)
      bool neg = (c < nsign) ? ((signs >> (15 - c)) & 1) : false;
      if (neg) level = (int16_t)-level;
      if (signHidden) {
        sumAbs += base + rem;
        if (c == n - 1 && (sumAbs & 1)) level = (int16_t)-level;
      }
      int p = spos[c];
      hc_coeff co;
      co.pos = (uint16_t)((xS0 + scanPos[p].x) + (yS0 + scanPos[p].y) * nT);
      co.level = level;
      cbuf[ncoeff_total++] = co;
    }
  }
  rec->coeffs.insert(rec->coeffs.end(), cbuf, cbuf + ncoeff_total);
  tb.ncoeff = (uint16_t)ncoeff_total;
  rec->tbs.push_back(tb);
  rec->tbs_by_size[log2 - 2]++;
  rec->resid_count += (uint64_t)nT * nT;
  return tb.resid_off;
}

// ---------------------------------------------------------------------------------------------
// Picture-level post-pass: QP map, no-filter flags, SAO neighbour masks.
void HevcIntraParser::Impl::finish_picture() {
  hc_pic& p = rec->pic;
  for (size_t i = 0; i < qp_y.size(); i++) rec->qp_map[i] = qp_y[i];

  bool any_edge = false;
  for (uint8_t e : rec->edge_map)
    if (e & (HC_EDGE_V | HC_EDGE_H)) { any_edge = true; break; }
  if (any_edge) p.flags |= HC_PIC_HAS_DEBLOCK;

  // pcm / transquant-bypass units: needed by SAO (sao.cc:349-356) and by the reference's special
  // deblocking path for such streams (deblock.cc:755-790)
  if ((S->pcm_enabled && S->pcm_loop_filter_disabled) || P->transquant_bypass_enabled) p.flags |= HC_PIC_PCMF;
  if (S->pcm_enabled && S->pcm_loop_filter_disabled) p.flags |= HC_PIC_PCM_LF_DISABLED;
  if (S->pcm_enabled || P->transquant_bypass_enabled) {
    for (int y8 = 0; y8 < h8; y8++)
      for (int x8 = 0; x8 < w8; x8++) {
        uint8_t f = cu_flags[x8 + (size_t)y8 * w8];
        if (!f) continue;
        uint8_t bits = (uint8_t)(((f & 1) ? HC_EDGE_PCM : 0) | ((f & 2) ? HC_EDGE_BYPASS : 0));
        for (int dy = 0; dy < 2; dy++)
          for (int dx = 0; dx < 2; dx++) rec->edge_map[(x8 * 2 + dx) + (size_t)(y8 * 2 + dy) * w4] |= bits;
        rec->ctus[ctb_of(x8 << 3, y8 << 3)].flags |= HC_CTU_HAS_NOFILTER;
      }
  }

  // SAO neighbour masks, mirroring apply_sao_internal (sao.cc:323-423) including two quirks of the
  // reference: (a) its fast path ignores slice-level loop_filter_across_slices flags altogether,
  // (b) for chroma its "current slice address" is looked up at chroma coordinates taken as luma.
  bool any_sao = false;
  const int cw = S->ctbs_w, chh = S->ctbs_h;
  static const int dx[8] = {-1, 1, 0, 0, -1, 1, -1, 1};
  static const int dy[8] = {0, 0, -1, 1, -1, -1, 1, 1};
  for (int cy = 0; cy < chh; cy++)
    for (int cx = 0; cx < cw; cx++) {
      const int a = cx + cy * cw;
      hc_ctu& ctu = rec->ctus[a];
      if (ctu.sao_type[0] | ctu.sao_type[1] | ctu.sao_type[2]) any_sao = true;
      const bool fast = P->loop_filter_across_slices && !P->tiles_enabled && !(ctu.flags & HC_CTU_HAS_NOFILTER);
      for (int comp = 0; comp < 2; comp++) {
        // slice address the reference compares against
        int sa = ctb_slice_addr[a];
        if (comp == 1 && S->ChromaArrayType != 0 && S->ChromaArrayType != 3) {
          int qx = (cx << S->log2_ctb) / S->SubWidthC, qy = (cy << S->log2_ctb) / S->SubHeightC;
          sa = ctb_slice_addr[ctb_of(qx, qy)];
        }
        uint8_t m = 0;
        for (int k = 0; k < 8; k++) {
          int nx = cx + dx[k], ny = cy + dy[k];
          if (nx < 0 || ny < 0 || nx >= cw || ny >= chh) continue;
          int n = nx + ny * cw;
          if (ctb_slice_idx[n] < 0 || ctb_slice_idx[a] < 0) continue;
          bool ok = true;
          if (!fast) {
            int sn = ctb_slice_addr[n];
            if (sn < sa && !slices[ctb_slice_idx[a]].loop_filter_across_slices) ok = false;
            if (sn > sa && !slices[ctb_slice_idx[n]].loop_filter_across_slices) ok = false;
            if (!P->loop_filter_across_tiles && P->tile_id_rs[n] != P->tile_id_rs[a]) ok = false;
          }
          if (ok) m |= (uint8_t)(1u << k);
        }
        if (comp == 0) ctu.sao_nb = m;
        else {
          ctu.sao_nb_c = m;
          if (!fast && ctb_slice_addr[a] != sa && !slices[ctb_slice_idx[a]].loop_filter_across_slices)
            ctu.flags |= HC_CTU_SAO_C_SELF;
        }
      }
    }
  if (any_sao) p.flags |= HC_PIC_HAS_SAO;

  p.blk_count = (uint32_t)rec->blks.size();
  p.tb_count = (uint32_t)rec->tbs.size();
  p.coeff_count = (uint32_t)rec->coeffs.size();
  p.resid_count = rec->resid_count;
}

}  // namespace hc
