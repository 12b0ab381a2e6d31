// postfilter_core.cuh — the per-unit arithmetic of the in-loop filters: deblocking (k3_deblock.cu) and SAO + crop + paste
// (k4_sao.cu), one pass over global memory each.
//
// Deblocking replaces edge_filtering_luma_internal (deblock.cc:708-792) + loop_filter_luma (fallback-postfilter.h:31-135)
// and edge_filtering_chroma_internal (:1607-1772) + loop_filter_chroma (:138-179); SAO replaces apply_sao_internal
// (sao.cc:261-488) with sao_band_filter / sao_edge_filter (fallback-postfilter.h:216-315), the conformance-window copy
// (decoder_libde265.cc:88-157) and the tile paste with its limited->full rescale (context.cc:2407-2539).
#pragma once
#include "launch.h"

namespace hc {

static __device__ __constant__ uint8_t c_beta_tab[52] = {0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  6,  7,
                                                  8,  9,  10, 11, 12, 13, 14, 15, 16, 17, 18, 20, 22, 24, 26, 28, 30, 32,
                                                  34, 36, 38, 40, 42, 44, 46, 48, 50, 52, 54, 56, 58, 60, 62, 64};
static __device__ __constant__ uint8_t c_tc_tab[54] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,  0,  0,  0,  0,
                                                1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3,  3,  3,  3,  4,
                                                4, 4, 5, 5, 6, 6, 7, 8, 9, 10, 11, 13, 14, 16, 18, 20, 22, 24};

HC_D int qpc_from_qpi_420(int qPi) {
  // H.265 Table 8-10
  if (qPi < 30) return qPi;
  if (qPi >= 44) return qPi - 6;
  // 30..43 -> 29,30,31,32,33,33,34,34,35,35,36,36,37,37
  const int d = qPi - 30;
  return d < 4 ? 29 + d : 33 + ((d - 4) >> 1);
}

// Luma: 4 lines x 8 samples (p3 p2 p1 p0 | q0 q1 q2 q3) held in registers.
template <typename Pixel>
__device__ void deblock_luma_unit(Pixel* __restrict__ pix, ptrdiff_t xs, ptrdiff_t ys, int beta, int tc, bool no_p,
                                  bool no_q, int bit_depth) {
  int s[4][8];
#pragma unroll
  for (int k = 0; k < 4; k++)
#pragma unroll
    for (int i = 0; i < 8; i++) s[k][i] = pix[(ptrdiff_t)(i - 4) * xs + (ptrdiff_t)k * ys];

  const int dp0 = iabs(s[0][1] - 2 * s[0][2] + s[0][3]), dq0 = iabs(s[0][6] - 2 * s[0][5] + s[0][4]);
  const int dp3 = iabs(s[3][1] - 2 * s[3][2] + s[3][3]), dq3 = iabs(s[3][6] - 2 * s[3][5] + s[3][4]);
  const int d0 = dp0 + dq0, d3 = dp3 + dq3;
  if (d0 + d3 >= beta) return;

  const int beta_3 = beta >> 3, beta_2 = beta >> 2, tc25 = (tc * 5 + 1) >> 1;
  const bool strong = iabs(s[0][0] - s[0][3]) + iabs(s[0][7] - s[0][4]) < beta_3 && iabs(s[0][3] - s[0][4]) < tc25 &&
                      iabs(s[3][0] - s[3][3]) + iabs(s[3][7] - s[3][4]) < beta_3 && iabs(s[3][3] - s[3][4]) < tc25 &&
                      (d0 << 1) < beta_2 && (d3 << 1) < beta_2;
  const int maxv = (1 << bit_depth) - 1;
  if (strong) {
    const int tc2 = tc << 1;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int p3 = s[k][0], p2 = s[k][1], p1 = s[k][2], p0 = s[k][3];
      const int q0 = s[k][4], q1 = s[k][5], q2 = s[k][6], q3 = s[k][7];
      Pixel* l = pix + (ptrdiff_t)k * ys;
      if (!no_p) {
        l[-1 * xs] = (Pixel)(p0 + clip3i(-tc2, tc2, ((p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3) - p0));
        l[-2 * xs] = (Pixel)(p1 + clip3i(-tc2, tc2, ((p2 + p1 + p0 + q0 + 2) >> 2) - p1));
        l[-3 * xs] = (Pixel)(p2 + clip3i(-tc2, tc2, ((2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3) - p2));
      }
      if (!no_q) {
        l[0] = (Pixel)(q0 + clip3i(-tc2, tc2, ((p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3) - q0));
        l[1 * xs] = (Pixel)(q1 + clip3i(-tc2, tc2, ((p0 + q0 + q1 + q2 + 2) >> 2) - q1));
        l[2 * xs] = (Pixel)(q2 + clip3i(-tc2, tc2, ((2 * q3 + 3 * q2 + q1 + q0 + p0 + 4) >> 3) - q2));
      }
    }
  } else {
    const int side_thr = (beta + (beta >> 1)) >> 3;
    const bool two_p = dp0 + dp3 < side_thr, two_q = dq0 + dq3 < side_thr;
    const int tc_2 = tc >> 1;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int p2 = s[k][1], p1 = s[k][2], p0 = s[k][3];
      const int q0 = s[k][4], q1 = s[k][5], q2 = s[k][6];
      int delta = (9 * (q0 - p0) - 3 * (q1 - p1) + 8) >> 4;
      if (iabs(delta) >= 10 * tc) continue;
      delta = clip3i(-tc, tc, delta);
      Pixel* l = pix + (ptrdiff_t)k * ys;
      if (!no_p) {
        l[-1 * xs] = (Pixel)clip3i(0, maxv, p0 + delta);
        if (two_p) l[-2 * xs] = (Pixel)clip3i(0, maxv, p1 + clip3i(-tc_2, tc_2, (((p2 + p0 + 1) >> 1) - p1 + delta) >> 1));
      }
      if (!no_q) {
        l[0] = (Pixel)clip3i(0, maxv, q0 - delta);
        if (two_q) l[1 * xs] = (Pixel)clip3i(0, maxv, q1 + clip3i(-tc_2, tc_2, (((q2 + q0 + 1) >> 1) - q1 - delta) >> 1));
      }
    }
  }
}

// One 4-line unit of one edge. (x, y): plane position of the unit's first q0 sample; `pix` points at that sample (K3 filters
// the plane in place), `stride` is the plane's pitch in samples. Edge flags / QP / slice offsets are looked up by picture
// position.
template <typename Pixel>
__device__ __forceinline__ void deblock_unit_at(const BatchView& bv, const hc_pic& pic, int plane_idx, bool vertical, int x, int y, Pixel* pix,
                                                int stride) {
  const int W = pic.width, H = pic.height;
  const int w4 = W >> 2, w8 = W >> 3;
  const uint8_t* __restrict__ edge = bv.edge_map + pic.edge_base;
  const int8_t* __restrict__ qp = bv.qp_map + pic.qp_base;
  const hc_ctu* __restrict__ ctus = bv.ctus + pic.ctu_base;
  const int mask = vertical ? HC_EDGE_V : HC_EDGE_H;

  if (plane_idx == 0) {
    const int e = edge[(x >> 2) + (size_t)(y >> 2) * w4];
    if (!(e & mask)) return;
    // QP / offsets are taken at the first unit of the 8-sample segment (deblock.cc:731-752)
    const int sx = vertical ? x : (x & ~7), sy = vertical ? (y & ~7) : y;
    const int QP_Q = qp[(sx >> 3) + (size_t)(sy >> 3) * w8];
    const int QP_P = vertical ? qp[((sx - 1) >> 3) + (size_t)(sy >> 3) * w8] : qp[(sx >> 3) + (size_t)((sy - 1) >> 3) * w8];
    const int qPL = (QP_Q + QP_P + 1) >> 1;
    const hc_ctu& ctu = ctus[(sx >> pic.log2_ctb) + (sy >> pic.log2_ctb) * pic.ctbs_w];
    const int bd = pic.bit_depth_y;
    const int beta = c_beta_tab[clip3i(0, 51, qPL + ctu.beta_offset)] * (1 << (bd - 8));
    const int tc = c_tc_tab[clip3i(0, 53, qPL + 2 + ctu.tc_offset)] * (1 << (bd - 8));
    // Streams with pcm(+loop filter disabled) / transquant bypass: mirror of the reference's
    // special path as its default build behaves (deblock.cc:755-790, see oracle/hevc_recon_oracle.c)
    bool no_p = false, no_q = false;
    if (pic.flags & HC_PIC_PCMF) {
      bool normal[2][2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int qx = vertical ? sx : sx + 4 * u, qy = vertical ? sy + 4 * u : sy;
        const int px = vertical ? qx - 1 : qx, py = vertical ? qy : qy - 1;
        normal[u][0] = !(edge[(px >> 2) + (size_t)(py >> 2) * w4] & (HC_EDGE_PCM | HC_EDGE_BYPASS));
        normal[u][1] = !(edge[(qx >> 2) + (size_t)(qy >> 2) * w4] & (HC_EDGE_PCM | HC_EDGE_BYPASS));
      }
      const int j = vertical ? ((y >> 2) & 1) : ((x >> 2) & 1);
      if (normal[0][0] && normal[0][1] && normal[1][0] && normal[1][1]) no_p = no_q = bd > 8;
      else { no_p = normal[j][0]; no_q = normal[j][1]; }
    }
    if (vertical) deblock_luma_unit<Pixel>(pix, 1, stride, beta, tc, no_p, no_q, bd);
    else deblock_luma_unit<Pixel>(pix, stride, 1, beta, tc, no_p, no_q, bd);
    return;
  }

  // ---- chroma: edges on the 8-sample chroma grid, bS == 2 only, 1 sample each side ----------------
  const int SubW = (pic.chroma_format == 1 || pic.chroma_format == 2) ? 2 : 1;
  const int SubH = pic.chroma_format == 1 ? 2 : 1;
  const int xc = x, yc = y;
  const int lx = xc * SubW, ly = yc * SubH;  // luma position of this 4-sample unit
  const int e = edge[(lx >> 2) + (size_t)(ly >> 2) * w4];
  if (!(e & mask)) return;
  const int QP_Q = qp[(lx >> 3) + (size_t)(ly >> 3) * w8];
  const int QP_P = vertical ? qp[((lx - 1) >> 3) + (size_t)(ly >> 3) * w8] : qp[(lx >> 3) + (size_t)((ly - 1) >> 3) * w8];
  const int cQpPicOffset = plane_idx == 1 ? pic.pps_cb_qp_offset : pic.pps_cr_qp_offset;
  const int qPi = ((QP_Q + QP_P + 1) >> 1) + cQpPicOffset;
  const int QpC = pic.chroma_format == 1 ? qpc_from_qpi_420(qPi) : (qPi < 51 ? qPi : 51);
  // tc offset of the slice at the start of the 8-sample chroma segment (deblock.cc:1700-1701)
  const int sxc = vertical ? xc : (xc & ~7), syc = vertical ? (yc & ~7) : yc;
  const hc_ctu& ctu = ctus[((sxc * SubW) >> pic.log2_ctb) + ((syc * SubH) >> pic.log2_ctb) * pic.ctbs_w];
  const int bd = pic.bit_depth_c;
  const int tc = c_tc_tab[clip3i(0, 53, QpC + 2 + ctu.tc_offset)] * (1 << (bd - 8));
  const int maxv = (1 << bd) - 1;
  const ptrdiff_t xs = vertical ? 1 : stride, ys = vertical ? stride : 1;
  bool no_p = false, no_q = false;
  if (pic.flags & HC_PIC_PCMF) {
    // deblock.cc:1716-1755 + loop_filter_chroma_c (fallback-postfilter.h:138-179)
    bool normal[2][2];
    const bool lfd = pic.flags & HC_PIC_PCM_LF_DISABLED;
    const int slx = sxc * SubW, sly = syc * SubH;  // luma position of the segment start
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const int ux = vertical ? slx : slx + 4 * u * SubW, uy = vertical ? sly + 4 * u * SubH : sly;
      if (ux >= W || uy >= H) { normal[u][0] = normal[u][1] = true; continue; }
      const int upx = vertical ? ux - 1 : ux, upy = vertical ? uy : uy - 1;
      const int ep = edge[(upx >> 2) + (size_t)(upy >> 2) * w4], eq = edge[(ux >> 2) + (size_t)(uy >> 2) * w4];
      normal[u][0] = !((lfd && (ep & HC_EDGE_PCM)) || (ep & HC_EDGE_BYPASS));
      normal[u][1] = !((lfd && (eq & HC_EDGE_PCM)) || (eq & HC_EDGE_BYPASS));
    }
    if (!(normal[0][0] && normal[0][1] && normal[1][0] && normal[1][1])) {
      const int j = vertical ? ((yc >> 2) & 1) : ((xc >> 2) & 1);
      no_p = !normal[j][0];
      no_q = vertical ? !normal[j][0] : !normal[j][1];
    }
  }
#pragma unroll
  for (int k = 0; k < 4; k++) {
    Pixel* l = pix + (ptrdiff_t)k * ys;
    const int p1 = l[-2 * xs], p0 = l[-1 * xs], q0 = l[0], q1 = l[xs];
    const int delta = clip3i(-tc, tc, (((q0 - p0) * 4) + p1 - q1 + 4) >> 3);
    if (!no_p) l[-1 * xs] = (Pixel)clip3i(0, maxv, p0 + delta);
    if (!no_q) l[0] = (Pixel)clip3i(0, maxv, q0 - delta);
  }
}

// ---- SAO ---------------------------------------------------------------------------------------------------------
HC_D int sign3(int v) { return (v > 0) - (v < 0); }

template <typename Pixel>
HC_D void load8(const Pixel* p, int v[8]);
template <>
HC_D void load8<uint8_t>(const uint8_t* p, int v[8]) {
  const uint2 w = *reinterpret_cast<const uint2*>(p);
#pragma unroll
  for (int k = 0; k < 4; k++) { v[k] = (w.x >> (8 * k)) & 0xff; v[4 + k] = (w.y >> (8 * k)) & 0xff; }
}
template <>
HC_D void load8<uint16_t>(const uint16_t* p, int v[8]) {
  const uint4 w = *reinterpret_cast<const uint4*>(p);
  v[0] = w.x & 0xffff; v[1] = w.x >> 16; v[2] = w.y & 0xffff; v[3] = w.y >> 16;
  v[4] = w.z & 0xffff; v[5] = w.z >> 16; v[6] = w.w & 0xffff; v[7] = w.w >> 16;
}
HC_D void store8(uint8_t* p, const int v[8]) {
  uint2 w;
  w.x = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
  w.y = v[4] | (v[5] << 8) | (v[6] << 16) | (v[7] << 24);
  *reinterpret_cast<uint2*>(p) = w;
}
HC_D void store8(uint16_t* p, const int v[8]) {
  uint4 w;
  w.x = v[0] | (v[1] << 16); w.y = v[2] | (v[3] << 16); w.z = v[4] | (v[5] << 16); w.w = v[6] | (v[7] << 16);
  *reinterpret_cast<uint4*>(p) = w;
}

// Geometry of one colour plane of one picture for the SAO + crop + paste step (context.cc:2467-2497 for the windows)
template <typename Pixel>
struct SaoPlane {
  int c, sw, sh, width, height, log2w, log2h;
  int cx0, cy0, copy_w, copy_h, dx0, dy0;
  Pixel* dst;
  int dstride, bit_depth, maxv;
  __device__ __forceinline__ void init(const BatchView& bv, const hc_pic& pic, int comp) {
    c = comp;
    sw = (c && (pic.chroma_format == 1 || pic.chroma_format == 2)) ? 1 : 0;   // log2 subsampling
    sh = (c && pic.chroma_format == 1) ? 1 : 0;
    const int SubW = 1 << sw, SubH = 1 << sh;
    width = pic.width >> sw; height = pic.height >> sh;   // coded plane size (multiples of 4)
    log2w = pic.log2_ctb - sw; log2h = pic.log2_ctb - sh;
    cx0 = pic.crop_x >> sw; cy0 = pic.crop_y >> sh;
    const int cw = (pic.crop_w + SubW - 1) >> sw, ch = (pic.crop_h + SubH - 1) >> sh;
    dx0 = (pic.dst_x + SubW - 1) >> sw; dy0 = (pic.dst_y + SubH - 1) >> sh;
    const int dw = (pic.dst_w + SubW - 1) >> sw, dh = (pic.dst_h + SubH - 1) >> sh;
    copy_w = min(cw, dw - dx0); copy_h = min(ch, dh - dy0);
    dst = reinterpret_cast<Pixel*>(bv.planes + pic.dst_off[c]);
    dstride = (int)pic.dst_stride[c];
    bit_depth = c == 0 ? pic.bit_depth_y : pic.bit_depth_c;
    maxv = (1 << bit_depth) - 1;
  }
};

// One unit: 8 horizontally adjacent samples (x0 8-aligned, so inside one CTB) of row y. `row` points at sample (x0, y) of
// the deblocked plane, `sstride` is its pitch in samples.
template <typename Pixel>
__device__ __forceinline__ void sao_unit(const BatchView& bv, const hc_pic& pic, const SaoPlane<Pixel>& P, int x0, int y, const Pixel* row,
                                         int sstride) {
  const int c = P.c, width = P.width, height = P.height, log2w = P.log2w, log2h = P.log2h, bit_depth = P.bit_depth, maxv = P.maxv;
  const int SubW = 1 << P.sw, SubH = 1 << P.sh;
  const int ox0 = x0 - P.cx0;                         // destination column of sample 0 of the unit
  const int copy_w = P.copy_w;
  if (ox0 + 8 <= 0 || ox0 >= copy_w) return;
  const int oy = y - P.cy0;
  if (oy < 0 || oy >= P.copy_h) return;
  const int ctbx = x0 >> log2w, ctby = y >> log2h;
  const hc_ctu& ctu = bv.ctus[pic.ctu_base + ctbx + ctby * pic.ctbs_w];
  const int nvalid = min(8, width - x0);            // 4 or 8
  int v[8];
  if (nvalid == 8) load8<Pixel>(row, v);
  else {
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = k < nvalid ? (int)row[k] : 0;
  }

  const int type = (bv.flags & HC_VIEW_NO_SAO) ? 0 : ctu.sao_type[c];
  if (type) {
    // samples of pcm (with pcm_loop_filter_disabled) / transquant-bypass CUs are left alone (sao.cc:288-300)
    unsigned skip = 0;
    if (ctu.flags & HC_CTU_HAS_NOFILTER) {
      const uint8_t* __restrict__ edge = bv.edge_map + pic.edge_base;
      const int w4 = pic.width >> 2;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        if (k >= nvalid) continue;
        const int e = edge[(((x0 + k) * SubW) >> 2) + (size_t)((y * SubH) >> 2) * w4];
        if (((pic.flags & HC_PIC_PCM_LF_DISABLED) && (e & HC_EDGE_PCM)) || (e & HC_EDGE_BYPASS)) skip |= 1u << k;
      }
    }
    const int8_t* offs = ctu.sao_offset[c];
    const int o0 = offs[0], o1 = offs[1], o2 = offs[2], o3 = offs[3];
    if (type == 1) {
      // bandShift >= 8 leaves the sample untouched in the reference (sao.cc:461)
      if (bit_depth - 5 < 8) {
        const int pos = ctu.sao_band_or_class[c];
#pragma unroll
        for (int k = 0; k < 8; k++) {
          const int k4 = ((v[k] >> (bit_depth - 5)) - pos) & 31;
          if (k4 < 4 && !((skip >> k) & 1)) v[k] = clip3i(0, maxv, v[k] + (k4 == 0 ? o0 : k4 == 1 ? o1 : k4 == 2 ? o2 : o3));
        }
      }
    } else {
      const int cls = ctu.sao_band_or_class[c];
      const int hx = cls == 1 ? 0 : (cls == 3 ? 1 : -1);   // first neighbour (x+hx, y+vy), second (x-hx, y-vy)
      const int vy = cls == 0 ? 0 : -1;
      // rows of the two neighbours, columns x0-1 .. x0+8 (index + 1)
      int ra[10], rb[10];
      const bool have_up = y > 0, have_dn = y + 1 < height;
      const Pixel* rowa = vy ? row - sstride : row;
      const Pixel* rowb = vy ? row + sstride : row;
      const bool oka = vy ? have_up : true, okb = vy ? have_dn : true;
#pragma unroll
      for (int k = 0; k < 10; k++) { ra[k] = 0; rb[k] = 0; }
      if (vy == 0) {
#pragma unroll
        for (int k = 0; k < 8; k++) { ra[k + 1] = v[k]; rb[k + 1] = v[k]; }
      } else {
        if (oka) {
          if (nvalid == 8) load8<Pixel>(rowa, ra + 1);
          else for (int k = 0; k < nvalid; k++) ra[k + 1] = rowa[k];
        }
        if (okb) {
          if (nvalid == 8) load8<Pixel>(rowb, rb + 1);
          else for (int k = 0; k < nvalid; k++) rb[k + 1] = rowb[k];
        }
      }
      if (hx) {
        if (x0 > 0) { if (oka) ra[0] = rowa[-1]; if (okb) rb[0] = rowb[-1]; }
        if (x0 + 8 < width) { if (oka) ra[9] = rowa[8]; if (okb) rb[9] = rowb[8]; }   // nvalid == 8 here
      }
      const unsigned nb = c ? ctu.sao_nb_c : ctu.sao_nb;
      const bool self_quirk = c && (ctu.flags & HC_CTU_SAO_C_SELF);
      const int mw = (1 << log2w) - 1, mh = (1 << log2h) - 1;
      const int orig[8] = {v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]};
      // offsets for edgeIdx -2,-1,(0),1,2 packed as bytes (sao.cc:312-317)
      const unsigned long long packed = (unsigned long long)(uint8_t)o0 | ((unsigned long long)(uint8_t)o1 << 8) |
                                        ((unsigned long long)(uint8_t)o2 << 24) | ((unsigned long long)(uint8_t)o3 << 32);
      // interior unit: no sample's neighbour leaves the CTB (or the picture) in the direction of this class
      const bool in_x = hx == 0 || ((x0 & mw) != 0 && ((x0 + 8) & mw) != 0 && x0 + 8 < width);
      const bool in_y = vy == 0 || ((y & mh) != 0 && ((y + 1) & mh) != 0 && y + 1 < height);
      // One arithmetic path for every unit of the warp: an interior unit uses all eight samples, a border unit only those
      // whose neighbours are usable (okmask). The first version ran a fast loop for interior units and a second, branchy
      // loop for border units — a warp holds both kinds (units 0 and 7 of every 64-sample CTB row are border units for
      // three of the four edge classes), so it executed both loops one after the other.
      unsigned okmask = 0;
      if (nvalid == 8 && skip == 0 && in_x && in_y && !self_quirk) {
        okmask = 0xffu;
      } else {
        const int lwid = min(1 << log2w, width - (ctbx << log2w)), lhei = min(1 << log2h, height - (ctby << log2h));
        const int ly = y & mh;
        // may sample x0 + k use both of its neighbours? (picture edge, neighbouring CTB not usable, reference quirk)
        auto sample_ok = [&](int k) -> bool {
          const int x = x0 + k;
          bool ok = true;
#pragma unroll
          for (int n = 0; n < 2; n++) {
            const int xs = n == 0 ? x + hx : x - hx, ys = n == 0 ? y + vy : y - vy;
            if (xs < 0 || ys < 0 || xs >= width || ys >= height) { ok = false; continue; }
            const int dxc = (xs >> log2w) - ctbx, dyc = (ys >> log2h) - ctby;
            if (dxc | dyc) {
              int bit;
              if (dyc == 0) bit = dxc < 0 ? HC_NB_L : HC_NB_R;
              else if (dxc == 0) bit = dyc < 0 ? HC_NB_T : HC_NB_B;
              else if (dyc < 0) bit = dxc < 0 ? HC_NB_TL : HC_NB_TR;
              else bit = dxc < 0 ? HC_NB_BL : HC_NB_BR;
              if (!(nb & bit)) ok = false;
            } else if (self_quirk) {
              // reference quirk (sao.cc:283): border samples of this CTB also lose their in-CTB neighbours
              const int lx = x & mw;
              if (lx == 0 || ly == 0 || lx == lwid - 1 || ly == lhei - 1) ok = false;
            }
          }
          return ok;
        };
        if (nvalid == 8 && !self_quirk) {
          // A full unit lies inside one CTB column. Which CTB does a neighbour fall into? 3 x 3 bits, (dy + 1) * 3 + dx + 1,
          // the centre (this CTB) always usable, the others from the CTB's neighbour mask (a CTB beyond the picture edge
          // has no bit; the edge of a partial CTB counts as its border). Samples 1..6 can only leave the CTB vertically,
          // sample 0 also to the left, sample 7 also to the right.
          const unsigned grid9 = 0x10u | ((nb & HC_NB_TL) ? 0x001u : 0u) | ((nb & HC_NB_T) ? 0x002u : 0u) | ((nb & HC_NB_TR) ? 0x004u : 0u) |
                                 ((nb & HC_NB_L) ? 0x008u : 0u) | ((nb & HC_NB_R) ? 0x020u : 0u) | ((nb & HC_NB_BL) ? 0x040u : 0u) |
                                 ((nb & HC_NB_B) ? 0x080u : 0u) | ((nb & HC_NB_BR) ? 0x100u : 0u);
          const int cy1 = (vy && ly == 0) ? -1 : 0, cy2 = (vy && ly == lhei - 1) ? 1 : 0;   // first neighbour looks up, second down
          auto okbit = [&](int cx, int cy) -> unsigned { return (grid9 >> ((cy + 1) * 3 + cx + 1)) & 1u; };
          okmask = (okbit(0, cy1) & okbit(0, cy2)) ? 0xffu : 0u;
          if (hx) {
            const int lx0 = x0 & mw;
            if (lx0 == 0) {
              const unsigned o0 = hx < 0 ? (okbit(-1, cy1) & okbit(0, cy2)) : (okbit(0, cy1) & okbit(-1, cy2));
              okmask = (okmask & ~1u) | o0;
            }
            if (lx0 + 8 == lwid) {
              const unsigned o7 = hx > 0 ? (okbit(1, cy1) & okbit(0, cy2)) : (okbit(0, cy1) & okbit(1, cy2));
              okmask = (okmask & ~0x80u) | (o7 << 7);
            }
          }
        } else {
#pragma unroll
          for (int k = 0; k < 8; k++)
            if (k < nvalid && sample_ok(k)) okmask |= 1u << k;
        }
        okmask &= ~skip;
      }
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int a = hx < 0 ? ra[k] : (hx == 0 ? ra[k + 1] : ra[k + 2]);
        const int b = hx < 0 ? rb[k + 2] : (hx == 0 ? rb[k + 1] : rb[k]);
        const int e = sign3(orig[k] - a) + sign3(orig[k] - b);   // -2..2; the packed table holds 0 for e == 0
        const int off = (int)(int8_t)(packed >> (8 * (e + 2)));
        const int r = clip3i(0, maxv, orig[k] + off);
        v[k] = ((okmask >> k) & 1) ? r : orig[k];
      }
    }
  }
  if (pic.dst_flags & HC_DST_RESCALE_LIMITED) {
    // context.cc:2504-2528: bytewise float rescale of limited-range tiles, no FMA contraction
    const float ratio = c == 0 ? 1.1689f : 1.1429f;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const float full = __fmul_rn(__fsub_rn((float)v[k], (float)(16 << (bit_depth - 8))), ratio);
      const long r = (long)__fadd_rn(full, 0.5f);
      v[k] = r < 0 ? 0 : (r > 255 ? 255 : (int)r);
    }
  }
  Pixel* out = P.dst + (size_t)(P.dy0 + oy) * P.dstride + P.dx0 + ox0;
  if (nvalid == 8 && ox0 >= 0 && ox0 + 8 <= copy_w && ((P.dx0 + ox0) & 7) == 0) {
    store8(out, v);
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (k < nvalid && ox0 + k >= 0 && ox0 + k < copy_w) out[k] = (Pixel)v[k];
  }
}

}  // namespace hc
