/*
 * hevc_recon_oracle.c — CPU restatement of the reference's HEVC-intra reconstruction path.
 *
 * TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg
 * may build, load or call this file; the product (heif-decoder-lib_b200/) never does.
 *
 * Parity status: PINNED.  Fed with the records of the product's host parser this file reproduces
 * the reference decoder's output bit-exactly on every bitstream bundled with the reference
 * (golden MD5s of SURVEY.md §8c, checked in tests/test_oracle_golden.py against both the committed
 * MD5s and the unmodified reference built into oracle/_ref by oracle/Makefile.ref).
 *
 * Each function follows the reference file:line named above it (paths relative to
 * /root/reference/third-party/libde265/libde265/).  It is written as straightforward scalar loops
 * over whole pictures; the CUDA kernels it checks are organised completely differently.
 */
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include "../include/heifcuda_records.h"
#include "oracle_counters.h"

uint64_t hc_oracle_counter[HC_CNT_COUNT];
static const char* const kCounterNames[HC_CNT_COUNT] = {
#define X(n) #n,
    HC_ORACLE_COUNTERS
#undef X
};

void hc_oracle_counters_reset(void) { memset(hc_oracle_counter, 0, sizeof(hc_oracle_counter)); }
/* Copies up to n counters to out; returns the number of counters. */
int hc_oracle_counters(uint64_t* out, int n) {
  for (int i = 0; i < n && i < HC_CNT_COUNT; i++) out[i] = hc_oracle_counter[i];
  return HC_CNT_COUNT;
}
const char* hc_oracle_counter_name(int i) { return i >= 0 && i < HC_CNT_COUNT ? kCounterNames[i] : NULL; }

static inline int clip3i(int lo, int hi, int v) { return v < lo ? lo : (v > hi ? hi : v); }
static inline int clip_bd(int v, int bd) { return clip3i(0, (1 << bd) - 1, v); }
static inline int iabs(int v) { return v < 0 ? -v : v; }
static inline int isign(int v) { return (v > 0) - (v < 0); }

/* ------------------------------------------------------------------------------------------ */
/* fallback-dct.cc:300-305 (DST-VII 4x4) and :554-589 (DCT matrix; rows 0..31, generated from the
 * first column by the cosine symmetries of the standard's matrix, H.265 eq. 8-xx) */
static const int8_t kDst[4][4] = {{29, 55, 74, 84}, {74, 74, 0, -74}, {84, -29, -74, 55}, {55, -84, 74, -29}};
static const int8_t kDctCol0[32] = {64, 90, 90, 90, 89, 88, 87, 85, 83, 82, 80, 78, 75, 73, 70, 67,
                                    64, 61, 57, 54, 50, 46, 43, 38, 36, 31, 25, 22, 18, 13, 9,  4};
static int8_t g_dct[32][32];
static int g_dct_ready = 0;
static void init_dct(void) {
  if (g_dct_ready) return;
  for (int k = 0; k < 32; k++)
    for (int n = 0; n < 32; n++) {
      if (k == 0) { g_dct[k][n] = 64; continue; }
      int a = (k * (2 * n + 1)) % 128; /* angle in units of pi/64 */
      int s = 1;
      if (a > 64) a = 128 - a;
      if (a > 32) { a = 64 - a; s = -1; }
      g_dct[k][n] = (int8_t)(s * (a == 32 ? 0 : kDctCol0[a]));
    }
  g_dct_ready = 1;
}

static const int kLevelScale[6] = {40, 45, 51, 57, 64, 72};

/* transform.cc:386-689 scale_coefficients_internal + fallback-dct.cc transforms.
 * Produces the residual block (before adding to the prediction) of one coded TB. */
static void oracle_tb_residual(const hc_pic* pic, const hc_tb* tb, const hc_coeff* coeffs, const uint8_t* scaling,
                               int32_t* res /* nT*nT */) {
  const int log2 = tb->log2, nT = 1 << log2, cIdx = tb->type & HC_TB_CIDX_MASK;
  const int bitDepth = cIdx == 0 ? pic->bit_depth_y : pic->bit_depth_c;
  int16_t coeff[32 * 32];
  memset(coeff, 0, sizeof(int16_t) * nT * nT);

  if (tb->type & HC_TB_BYPASS) { /* transform.cc:426-460 */
    for (int i = 0; i < tb->ncoeff; i++) coeff[coeffs[i].pos] = coeffs[i].level;
    if (tb->type & HC_TB_ROTATE) /* fallback-dct.cc:292-298 */
      for (int y = 0; y < nT / 2; y++)
        for (int x = 0; x < nT; x++) {
          int16_t t = coeff[y * nT + x];
          coeff[y * nT + x] = coeff[(nT - 1 - y) * nT + nT - 1 - x];
          coeff[(nT - 1 - y) * nT + nT - 1 - x] = t;
        }
    if (tb->type & HC_TB_RDPCM_V) {
      for (int x = 0; x < nT; x++) { int sum = 0; for (int y = 0; y < nT; y++) { sum += coeff[x + y * nT]; res[y * nT + x] = sum; } }
    } else if (tb->type & HC_TB_RDPCM_H) {
      for (int y = 0; y < nT; y++) { int sum = 0; for (int x = 0; x < nT; x++) { sum += coeff[x + y * nT]; res[y * nT + x] = sum; } }
    } else {
      for (int i = 0; i < nT * nT; i++) res[i] = coeff[i];
    }
    return;
  }

  /* dequantisation, transform.cc:473-546 */
  int bdShift = bitDepth + log2 - 5;
  const int qP = tb->qp;
  if (!(pic->flags & HC_PIC_SCALING_LIST)) {
    bdShift -= 4;
    const int offset = 1 << (bdShift - 1);
    const int fact = kLevelScale[qP % 6] << (qP / 6);
    for (int i = 0; i < tb->ncoeff; i++) {
      int32_t c = coeffs[i].level;
      /* int32 arithmetic with wrap, as in the reference (SURVEY hazard 1) */
      const int64_t exact = ((int64_t)c * fact + offset) >> bdShift;
      c = (int32_t)((uint32_t)c * (uint32_t)fact + (uint32_t)offset) >> bdShift;
      if (exact != c) HC_COUNT(k1_flat_dequant_wrap);
      if (c < -32768 || c > 32767) HC_COUNT(k1_dequant_clip16);
      coeff[coeffs[i].pos] = (int16_t)clip3i(-32768, 32767, c);
    }
  } else {
    const int offset = 1 << (bdShift - 1);
    const uint8_t* sc;
    switch (log2) {
      case 2: sc = scaling + tb->matrix_id * 16; break;
      case 3: sc = scaling + 6 * 16 + tb->matrix_id * 64; break;
      case 4: sc = scaling + 6 * 16 + 6 * 64 + tb->matrix_id * 256; break;
      default: sc = scaling + 6 * 16 + 6 * 64 + 6 * 256 + (tb->matrix_id ? 1024 : 0); break;
    }
    for (int i = 0; i < tb->ncoeff; i++) {
      int pos = coeffs[i].pos;
      int fact = (sc[pos] * kLevelScale[qP % 6]) << (qP / 6);
      if (sc[pos] >= 200) HC_COUNT(k1_scaled_factor_ge200);
      int64_t c = coeffs[i].level;
      c = (c * fact + offset) >> bdShift;
      if (c < -32768 || c > 32767) HC_COUNT(k1_dequant_clip16);
      coeff[pos] = (int16_t)(c < -32768 ? -32768 : (c > 32767 ? 32767 : c));
    }
  }

  if (tb->type & HC_TB_TSKIP) { /* transform.cc:566-650, fallback-dct.cc:84-108,232-260 */
    int bd2 = 20 - bitDepth; if (bd2 < 0) bd2 = 0;
    int tsShift = 5 + log2;
    int rnd = 1 << (bd2 - 1);
    if (tb->type & HC_TB_ROTATE)
      for (int y = 0; y < nT / 2; y++)
        for (int x = 0; x < nT; x++) {
          int16_t t = coeff[y * nT + x];
          coeff[y * nT + x] = coeff[(nT - 1 - y) * nT + nT - 1 - x];
          coeff[(nT - 1 - y) * nT + nT - 1 - x] = t;
        }
    if (tb->type & HC_TB_RDPCM_V) {
      for (int x = 0; x < nT; x++) { int sum = 0; for (int y = 0; y < nT; y++) { int c = coeff[x + y * nT] << tsShift; sum += (c + rnd) >> bd2; res[y * nT + x] = sum; } }
    } else if (tb->type & HC_TB_RDPCM_H) {
      for (int y = 0; y < nT; y++) { int sum = 0; for (int x = 0; x < nT; x++) { int c = coeff[x + y * nT] << tsShift; sum += (c + rnd) >> bd2; res[y * nT + x] = sum; } }
    } else {
      for (int i = 0; i < nT * nT; i++) { int c = coeff[i] << tsShift; res[i] = (c + rnd) >> bd2; }
    }
    return;
  }

  const int postShift = 20 - bitDepth;
  const int rnd1 = 1 << 6, rnd2 = 1 << (postShift - 1);
  int16_t g[32 * 32];
  if (tb->type & HC_TB_DST) { /* fallback-dct.cc:309-378 */
    for (int c = 0; c < 4; c++)
      for (int i = 0; i < 4; i++) {
        int sum = 0;
        for (int j = 0; j < 4; j++) sum += kDst[j][i] * coeff[c + j * 4];
        if (((sum + rnd1) >> 7) < -32768 || ((sum + rnd1) >> 7) > 32767) HC_COUNT(k1_dst_pass1_clip);
        g[i * 4 + c] = (int16_t)clip3i(-32768, 32767, (sum + rnd1) >> 7);
      }
    for (int y = 0; y < 4; y++)
      for (int i = 0; i < 4; i++) {
        int sum = 0;
        for (int j = 0; j < 4; j++) sum += kDst[j][i] * g[y * 4 + j];
        if (((sum + rnd2) >> postShift) < -32768 || ((sum + rnd2) >> postShift) > 32767) HC_COUNT(k1_dst_pass2_clip);
        res[y * 4 + i] = clip3i(-32768, 32767, (sum + rnd2) >> postShift);
      }
    return;
  }
  /* fallback-dct.cc:593-733 transform_idct_add */
  init_dct();
  const int fact = 1 << (5 - log2);
  for (int c = 0; c < nT; c++)
    for (int i = 0; i < nT; i++) {
      int sum = 0;
      for (int j = 0; j < nT; j++) sum += g_dct[fact * j][i] * coeff[c + j * nT];
      if (((sum + rnd1) >> 7) < -32768 || ((sum + rnd1) >> 7) > 32767) HC_COUNT(k1_dct_pass1_clip);
      g[c + i * nT] = (int16_t)clip3i(-32768, 32767, (sum + rnd1) >> 7);
    }
  for (int y = 0; y < nT; y++)
    for (int i = 0; i < nT; i++) {
      int sum = 0;
      for (int j = 0; j < nT; j++) sum += g_dct[fact * j][i] * g[y * nT + j];
      res[y * nT + i] = (sum + rnd2) >> postShift; /* not clipped to int16 (fallback-dct.cc:723) */
    }
}

/* ------------------------------------------------------------------------------------------ */
static const int kIntraPredAngle[35] = {0,   0,   32,  26,  21,  17, 13, 9,  5,  2,  0,  -2, -5, -9, -13, -17, -21, -26,
                                        -32, -26, -21, -17, -13, -9, -5, -2, 0,  2,  5,  9,  13, 17, 21,  26,  32};
static const int kInvAngle[15] = {-4096, -1638, -910, -630, -482, -390, -315, -256, -315, -390, -482, -630, -910, -1638, -4096};

/* intrapred.cc:337-362 decode_intra_prediction: border fill (intrapred.h:838-984 with the
 * host-resolved availability bits), smoothing (:192-266), planar/DC/angular (:269-441). */
static void oracle_predict(const hc_pic* pic, const hc_blk* b, uint16_t* plane, int stride, uint16_t* dst /* nT*nT */) {
  const int nT = 1 << b->log2, cIdx = b->cidx;
  const int bitDepth = cIdx == 0 ? pic->bit_depth_y : pic->bit_depth_c;
  int border_mem[4 * 32 + 1];
  uint8_t avail_mem[4 * 32 + 1];
  int* p = border_mem + 2 * 32;
  uint8_t* av = avail_mem + 2 * 32;
  memset(avail_mem, 0, sizeof(avail_mem));
  const int xB = b->x, yB = b->y;
  int nAvail = 0, firstValue = 0, haveFirst = 0;

  /* left column, bottom to top (intrapred.h:857-884) */
  for (int k = 2 * nT / 4 - 1; k >= 0; k--)
    if (b->avail_left & (1u << k)) {
      for (int i = 0; i < 4; i++) {
        int y = 4 * k + 3 - i;
        p[-y - 1] = plane[(xB - 1) + (size_t)(yB + y) * stride];
        av[-y - 1] = 1;
      }
      if (!haveFirst) { firstValue = plane[(xB - 1) + (size_t)(yB + 4 * k + 3) * stride]; haveFirst = 1; }
      nAvail += 4;
    }
  if (b->flags & HC_BLK_AVAIL_TL) {
    p[0] = plane[(xB - 1) + (size_t)(yB - 1) * stride];
    av[0] = 1;
    if (!haveFirst) { firstValue = p[0]; haveFirst = 1; }
    nAvail++;
  }
  for (int k = 0; k < 2 * nT / 4; k++)
    if (b->avail_top & (1u << k)) {
      for (int i = 0; i < 4; i++) {
        p[4 * k + i + 1] = plane[(xB + 4 * k + i) + (size_t)(yB - 1) * stride];
        av[4 * k + i + 1] = 1;
      }
      if (!haveFirst) { firstValue = p[4 * k + 1]; haveFirst = 1; }
      nAvail += 4;
    }
  /* reference_sample_substitution (intrapred.h:944-984) */
  if (nAvail != 4 * nT + 1) {
    if (nAvail == 0) {
      for (int i = -2 * nT; i <= 2 * nT; i++) p[i] = 1 << (bitDepth - 1);
    } else {
      if (!av[-2 * nT]) p[-2 * nT] = firstValue;
      for (int i = -2 * nT + 1; i <= 2 * nT; i++)
        if (!av[i]) p[i] = p[i - 1];
    }
  }

  const int mode = b->mode;
  /* intrapred.cc:307-311 + intrapred.h:192-266 */
  if (!(pic->flags & HC_PIC_NO_INTRA_SMOOTH) && (cIdx == 0 || pic->chroma_format == 3)) {
    int filterFlag = 0;
    if (mode != 1 && nT != 4) {
      int d1 = iabs(mode - 26), d2 = iabs(mode - 10);
      int minDist = d1 < d2 ? d1 : d2;
      if (nT == 8) filterFlag = minDist > 7;
      else if (nT == 16) filterFlag = minDist > 1;
      else if (nT == 32) filterFlag = minDist > 0;
    }
    if (filterFlag) {
      int pF_mem[4 * 32 + 1];
      int* pF = pF_mem + 2 * 32;
      int biInt = (pic->flags & HC_PIC_STRONG_INTRA) && cIdx == 0 && nT == 32 &&
                  iabs(p[0] + p[64] - 2 * p[32]) < (1 << (pic->bit_depth_y - 5)) &&
                  iabs(p[0] + p[-64] - 2 * p[-32]) < (1 << (pic->bit_depth_y - 5));
      pF[-2 * nT] = p[-2 * nT];
      pF[2 * nT] = p[2 * nT];
      if (biInt) {
        HC_COUNT(k2_strong_smoothing);
        pF[0] = p[0];
        for (int i = 1; i <= 63; i++) {
          pF[-i] = p[0] + ((i * (p[-64] - p[0]) + 32) >> 6);
          pF[i] = p[0] + ((i * (p[64] - p[0]) + 32) >> 6);
        }
      } else {
        HC_COUNT(k2_121_smoothing);
        for (int i = -(2 * nT - 1); i <= 2 * nT - 1; i++) pF[i] = (p[i + 1] + 2 * p[i] + p[i - 1] + 2) >> 2;
      }
      for (int i = -2 * nT; i <= 2 * nT; i++) p[i] = pF[i];
    }
  }

  if (mode <= 34) hc_oracle_counter[HC_CNT_k2_mode_0 + mode]++;
  if (mode == 0) { /* planar, intrapred.h:269-293 */
    for (int y = 0; y < nT; y++)
      for (int x = 0; x < nT; x++)
        dst[x + y * nT] = (uint16_t)(((nT - 1 - x) * p[-1 - y] + (x + 1) * p[1 + nT] + (nT - 1 - y) * p[1 + x] +
                                      (y + 1) * p[-1 - nT] + nT) >> (b->log2 + 1));
  } else if (mode == 1) { /* DC, intrapred.h:296-330 */
    int dc = 0;
    for (int i = 0; i < nT; i++) dc += p[i + 1] + p[-i - 1];
    dc = (dc + nT) >> (b->log2 + 1);
    for (int i = 0; i < nT * nT; i++) dst[i] = (uint16_t)dc;
    if (cIdx == 0 && nT < 32) {
      dst[0] = (uint16_t)((p[-1] + 2 * dc + p[1] + 2) >> 2);
      for (int x = 1; x < nT; x++) dst[x] = (uint16_t)((p[x + 1] + 3 * dc + 2) >> 2);
      for (int y = 1; y < nT; y++) dst[y * nT] = (uint16_t)((p[-y - 1] + 3 * dc + 2) >> 2);
    }
  } else { /* angular, intrapred.h:338-441 */
    int ref_mem[4 * 32 + 1];
    int* ref = ref_mem + 2 * 32;
    const int angle = kIntraPredAngle[mode];
    const int noEdge = (b->flags & HC_BLK_NO_EDGE_FLT) != 0;
    if (mode >= 18) {
      for (int x = 0; x <= nT; x++) ref[x] = p[x];
      if (angle < 0) {
        int inv = kInvAngle[mode - 11];
        if (((nT * angle) >> 5) < -1)
          for (int x = (nT * angle) >> 5; x <= -1; x++) ref[x] = p[0 - ((x * inv + 128) >> 8)];
      } else {
        for (int x = nT + 1; x <= 2 * nT; x++) ref[x] = p[x];
      }
      for (int y = 0; y < nT; y++)
        for (int x = 0; x < nT; x++) {
          int iIdx = ((y + 1) * angle) >> 5, iFact = ((y + 1) * angle) & 31;
          dst[x + y * nT] = (uint16_t)(iFact ? ((32 - iFact) * ref[x + iIdx + 1] + iFact * ref[x + iIdx + 2] + 16) >> 5
                                             : ref[x + iIdx + 1]);
        }
      if (mode == 26 && cIdx == 0 && nT < 32 && !noEdge)
        for (int y = 0; y < nT; y++) dst[y * nT] = (uint16_t)clip_bd(p[1] + ((p[-1 - y] - p[0]) >> 1), bitDepth);
    } else {
      for (int x = 0; x <= nT; x++) ref[x] = p[-x];
      if (angle < 0) {
        int inv = kInvAngle[mode - 11];
        if (((nT * angle) >> 5) < -1)
          for (int x = (nT * angle) >> 5; x <= -1; x++) ref[x] = p[(x * inv + 128) >> 8];
      } else {
        for (int x = nT + 1; x <= 2 * nT; x++) ref[x] = p[-x];
      }
      for (int y = 0; y < nT; y++)
        for (int x = 0; x < nT; x++) {
          int iIdx = ((x + 1) * angle) >> 5, iFact = ((x + 1) * angle) & 31;
          dst[x + y * nT] = (uint16_t)(iFact ? ((32 - iFact) * ref[y + iIdx + 1] + iFact * ref[y + iIdx + 2] + 16) >> 5
                                             : ref[y + iIdx + 1]);
        }
      if (mode == 10 && cIdx == 0 && nT < 32 && !noEdge)
        for (int x = 0; x < nT; x++) dst[x] = (uint16_t)clip_bd(p[-1] + ((p[1 + x] - p[0]) >> 1), bitDepth);
    }
  }
}

/* ------------------------------------------------------------------------------------------ */
static const uint8_t kBetaTab[52] = {0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  6,  7,
                                     8,  9,  10, 11, 12, 13, 14, 15, 16, 17, 18, 20, 22, 24, 26, 28, 30, 32,
                                     34, 36, 38, 40, 42, 44, 46, 48, 50, 52, 54, 56, 58, 60, 62, 64};
static const uint8_t kTcTab[54] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,  0,  0,  0,  0,
                                   1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3,  3,  3,  3,  4,
                                   4, 4, 5, 5, 6, 6, 7, 8, 9, 10, 11, 13, 14, 16, 18, 20, 22, 24};
/* clip3(0, 53, idx) of the tc table index */
static int count_tc_idx(int idx) {
  if (idx < 0) HC_COUNT(k3_tc_idx_clamp_lo);
  if (idx > 53) HC_COUNT(k3_tc_idx_clamp_hi);
  return clip3i(0, 53, idx);
}
static int qpc_420(int qPi) { /* H.265 Table 8-10 / transform.cc table8_22 */
  static const int8_t t[14] = {29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37, 37};
  if (qPi < 30) return qPi;
  if (qPi >= 44) return qPi - 6;
  return t[qPi - 30];
}

typedef struct {
  const hc_pic* pic;
  const hc_ctu* ctus;
  const uint8_t* edge;
  const int8_t* qp;
  int w4, w8;
} dbk_ctx;

static inline int edge_at(const dbk_ctx* d, int x, int y) { return d->edge[(x >> 2) + (size_t)(y >> 2) * d->w4]; }
static inline int qp_at(const dbk_ctx* d, int x, int y) { return d->qp[(x >> 3) + (size_t)(y >> 3) * d->w8]; }
static inline const hc_ctu* ctu_at(const dbk_ctx* d, int x, int y) {
  return &d->ctus[(x >> d->pic->log2_ctb) + (y >> d->pic->log2_ctb) * d->pic->ctbs_w];
}

/* deblock.cc:708-792 edge_filtering_luma_internal + fallback-postfilter.h:31-135 loop_filter_luma.
 * Streams with (pcm && pcm_loop_filter_disabled) or transquant_bypass_enabled take the reference's
 * special path (deblock.cc:755-790), restated here exactly as its default (SIMD) build behaves, which
 * is NOT what the standard says: an 8-sample segment touching no pcm/bypass CU is filtered normally
 * for 8-bit pictures (SIMD kernel ignores the flags) and not at all for deeper ones (the scalar
 * template tests "!no_p" while the caller passes true for "filter"); in a segment that does touch
 * one, only the pcm/bypass sides are modified. */
static void oracle_deblock_luma(const dbk_ctx* d, uint16_t* plane, int stride, int vertical) {
  const hc_pic* pic = d->pic;
  const int bd = pic->bit_depth_y;
  const int mask = vertical ? HC_EDGE_V : HC_EDGE_H;
  for (int y = 0; y < pic->height; y += 8)
    for (int x = 0; x < pic->width; x += 8) {
      int bs0 = (edge_at(d, x, y) & mask) ? 2 : 0;
      int bs1 = ((vertical ? edge_at(d, x, y + 4) : edge_at(d, x + 4, y)) & mask) ? 2 : 0;
      if (!bs0 && !bs1) continue;
      int QP_Q = qp_at(d, x, y);
      int QP_P = vertical ? qp_at(d, x - 1, y) : qp_at(d, x, y - 1);
      int qPL = (QP_Q + QP_P + 1) >> 1;
      const hc_ctu* ctu = ctu_at(d, x, y);
      if (qPL + ctu->beta_offset < 0 || qPL + ctu->beta_offset > 51) HC_COUNT(k3_beta_idx_clamp);
      int beta = kBetaTab[clip3i(0, 51, qPL + ctu->beta_offset)] * (1 << (bd - 8));
      int tcs[2];
      tcs[0] = bs0 ? kTcTab[count_tc_idx(qPL + 2 * (bs0 - 1) + ctu->tc_offset)] * (1 << (bd - 8)) : 0;
      tcs[1] = bs1 ? kTcTab[count_tc_idx(qPL + 2 * (bs1 - 1) + ctu->tc_offset)] * (1 << (bd - 8)) : 0;
      const ptrdiff_t xs = vertical ? 1 : stride, ys = vertical ? stride : 1;
      uint16_t* pix = plane + x + (size_t)y * stride;
      for (int j = 0; j < 2; j++, pix += 4 * ys) {
        const int tc = tcs[j];
        int no_p = 0, no_q = 0; /* 1 = leave that side untouched */
        if (pic->flags & HC_PIC_PCMF) {
          int normal[2][2];
          for (int u = 0; u < 2; u++) {
            int px = vertical ? x - 1 : x + 4 * u, py = vertical ? y + 4 * u : y - 1;
            int qx = vertical ? x : x + 4 * u, qy = vertical ? y + 4 * u : y;
            normal[u][0] = !(edge_at(d, px, py) & (HC_EDGE_PCM | HC_EDGE_BYPASS));
            normal[u][1] = !(edge_at(d, qx, qy) & (HC_EDGE_PCM | HC_EDGE_BYPASS));
          }
          if (normal[0][0] && normal[0][1] && normal[1][0] && normal[1][1]) no_p = no_q = (bd > 8);
          else { no_p = normal[j][0]; no_q = normal[j][1]; }
        }
#define PX(i, k) pix[(ptrdiff_t)(i) * xs + (ptrdiff_t)(k) * ys]
        const int dp0 = iabs(PX(-3, 0) - 2 * PX(-2, 0) + PX(-1, 0)), dq0 = iabs(PX(2, 0) - 2 * PX(1, 0) + PX(0, 0));
        const int dp3 = iabs(PX(-3, 3) - 2 * PX(-2, 3) + PX(-1, 3)), dq3 = iabs(PX(2, 3) - 2 * PX(1, 3) + PX(0, 3));
        const int d0 = dp0 + dq0, d3 = dp3 + dq3;
        if (d0 + d3 >= beta) continue;
        const int beta_3 = beta >> 3, beta_2 = beta >> 2, tc25 = (tc * 5 + 1) >> 1;
        if (iabs(PX(-4, 0) - PX(-1, 0)) + iabs(PX(3, 0) - PX(0, 0)) < beta_3 && iabs(PX(-1, 0) - PX(0, 0)) < tc25 &&
            iabs(PX(-4, 3) - PX(-1, 3)) + iabs(PX(3, 3) - PX(0, 3)) < beta_3 && iabs(PX(-1, 3) - PX(0, 3)) < tc25 &&
            (d0 << 1) < beta_2 && (d3 << 1) < beta_2) {
          const int tc2 = tc << 1;
          HC_COUNT(k3_luma_strong);
          for (int k = 0; k < 4; k++) {
            const int p3 = PX(-4, k), p2 = PX(-3, k), p1 = PX(-2, k), p0 = PX(-1, k);
            const int q0 = PX(0, k), q1 = PX(1, k), q2 = PX(2, k), q3 = PX(3, k);
            if (!no_p) {
              PX(-1, k) = (uint16_t)(p0 + clip3i(-tc2, tc2, ((p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3) - p0));
              PX(-2, k) = (uint16_t)(p1 + clip3i(-tc2, tc2, ((p2 + p1 + p0 + q0 + 2) >> 2) - p1));
              PX(-3, k) = (uint16_t)(p2 + clip3i(-tc2, tc2, ((2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3) - p2));
            }
            if (!no_q) {
              PX(0, k) = (uint16_t)(q0 + clip3i(-tc2, tc2, ((p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3) - q0));
              PX(1, k) = (uint16_t)(q1 + clip3i(-tc2, tc2, ((p0 + q0 + q1 + q2 + 2) >> 2) - q1));
              PX(2, k) = (uint16_t)(q2 + clip3i(-tc2, tc2, ((2 * q3 + 3 * q2 + q1 + q0 + p0 + 4) >> 3) - q2));
            }
          }
        } else {
          int nd_p = 1, nd_q = 1;
          const int tc_2 = tc >> 1;
          if (dp0 + dp3 < ((beta + (beta >> 1)) >> 3)) nd_p = 2;
          if (dq0 + dq3 < ((beta + (beta >> 1)) >> 3)) nd_q = 2;
          HC_COUNT(k3_luma_weak);
          if (nd_p > 1 || nd_q > 1) HC_COUNT(k3_luma_weak_nd2);
          for (int k = 0; k < 4; k++) {
            const int p2 = PX(-3, k), p1 = PX(-2, k), p0 = PX(-1, k);
            const int q0 = PX(0, k), q1 = PX(1, k), q2 = PX(2, k);
            int delta0 = (9 * (q0 - p0) - 3 * (q1 - p1) + 8) >> 4;
            if (iabs(delta0) < 10 * tc) {
              delta0 = clip3i(-tc, tc, delta0);
              if (!no_p) PX(-1, k) = (uint16_t)clip_bd(p0 + delta0, bd);
              if (!no_q) PX(0, k) = (uint16_t)clip_bd(q0 - delta0, bd);
              if (!no_p && nd_p > 1) PX(-2, k) = (uint16_t)clip_bd(p1 + clip3i(-tc_2, tc_2, (((p2 + p0 + 1) >> 1) - p1 + delta0) >> 1), bd);
              if (!no_q && nd_q > 1) PX(1, k) = (uint16_t)clip_bd(q1 + clip3i(-tc_2, tc_2, (((q2 + q0 + 1) >> 1) - q1 - delta0) >> 1), bd);
            }
          }
        }
#undef PX
      }
    }
}

/* deblock.cc:1607-1772 edge_filtering_chroma_internal + fallback-postfilter.h:138-179 */
static void oracle_deblock_chroma(const dbk_ctx* d, uint16_t* plane, int stride, int vertical, int cplane) {
  const hc_pic* pic = d->pic;
  const int SubW = (pic->chroma_format == 1 || pic->chroma_format == 2) ? 2 : 1;
  const int SubH = pic->chroma_format == 1 ? 2 : 1;
  const int bd = pic->bit_depth_c;
  const int mask = vertical ? HC_EDGE_V : HC_EDGE_H;
  const int cQpPicOffset = cplane == 0 ? pic->pps_cb_qp_offset : pic->pps_cr_qp_offset;
  const int stepx = 8 * SubW, stepy = 8 * SubH; /* luma step: edges on the 8-sample chroma grid */
  for (int ly = 0; ly < pic->height; ly += stepy)
    for (int lx = 0; lx < pic->width; lx += stepx) {
      int l1x = vertical ? lx : lx + 4 * SubW, l1y = vertical ? ly + 4 * SubH : ly;
      int bS0 = (edge_at(d, lx, ly) & mask) ? 2 : 0;
      int bS1 = (l1x < pic->width && l1y < pic->height && (edge_at(d, l1x, l1y) & mask)) ? 2 : 0;
      if (bS0 != 2 && bS1 != 2) continue;
      int tcv[2];
      for (int j = 0; j < 2; j++) {
        int qx = j ? l1x : lx, qy = j ? l1y : ly;
        if (qx >= pic->width || qy >= pic->height) { tcv[j] = 0; continue; }
        int QP_Q = qp_at(d, qx, qy);
        int QP_P = vertical ? qp_at(d, qx - 1, qy) : qp_at(d, qx, qy - 1);
        int qPi = ((QP_Q + QP_P + 1) >> 1) + cQpPicOffset;
        if (qPi >= 30 && qPi <= 43) HC_COUNT(k3_chroma_qpi_30_43);
        if (qPi < 0) HC_COUNT(k3_chroma_qpi_neg);
        int QpC = pic->chroma_format == 1 ? qpc_420(qPi) : (qPi < 51 ? qPi : 51);
        int tc_offset = ctu_at(d, lx, ly)->tc_offset;
        int tcPrime = kTcTab[count_tc_idx(QpC + 2 + tc_offset)];
        tcv[j] = ((j ? bS1 : bS0) == 2) ? tcPrime * (1 << (bd - 8)) : 0;
      }
      const int xDi = lx / SubW, yDi = ly / SubH;
      uint16_t* ptr = plane + xDi + (size_t)yDi * stride;
      for (int k = 0; k < 8; k++) {
        const int j = k >> 2;
        const int tc = tcv[j];
        int lqx = vertical ? lx : lx + k * SubW, lqy = vertical ? ly + k * SubH : ly;
        if (lqx >= pic->width || lqy >= pic->height) continue;
        int no_p = 0, no_q = 0;
        if (pic->flags & HC_PIC_PCMF) {
          /* deblock.cc:1716-1755: flags of the two 4-line units of this 8-sample segment */
          int normal[2][2];
          const int lfd = (pic->flags & HC_PIC_PCM_LF_DISABLED) != 0;
          for (int u = 0; u < 2; u++) {
            int ux = vertical ? lx : lx + 4 * u * SubW, uy = vertical ? ly + 4 * u * SubH : ly;
            int upx = vertical ? lx - 1 : ux, upy = vertical ? uy : ly - 1;
            if (ux >= pic->width || uy >= pic->height) { normal[u][0] = normal[u][1] = 1; continue; }
            int ep = edge_at(d, upx, upy), eq = edge_at(d, ux, uy);
            normal[u][0] = !((lfd && (ep & HC_EDGE_PCM)) || (ep & HC_EDGE_BYPASS));
            normal[u][1] = !((lfd && (eq & HC_EDGE_PCM)) || (eq & HC_EDGE_BYPASS));
          }
          if (!(normal[0][0] && normal[0][1] && normal[1][0] && normal[1][1])) {
            /* loop_filter_chroma_c (fallback-postfilter.h:138-179): the vertical branch tests the P
             * flag for both sides */
            no_p = !normal[j][0];
            no_q = vertical ? !normal[j][0] : !normal[j][1];
          }
        }
        uint16_t *q0p, *q1p, *p0p, *p1p;
        if (vertical) { q0p = ptr + (size_t)k * stride; q1p = q0p + 1; p0p = q0p - 1; p1p = q0p - 2; }
        else { q0p = ptr + k; q1p = q0p + stride; p0p = q0p - stride; p1p = q0p - 2 * stride; }
        int delta = clip3i(-tc, tc, ((((*q0p - *p0p) * 4) + *p1p - *q1p + 4) >> 3));
        int np = clip_bd(*p0p + delta, bd), nq = clip_bd(*q0p - delta, bd);
        if (!no_p) *p0p = (uint16_t)np;
        if (!no_q) *q0p = (uint16_t)nq;
      }
    }
}

/* sao.cc:349-356,441-445: pcm samples (when pcm_loop_filter_disabled) and bypass samples keep their value */
static int sao_sample_skipped(const hc_pic* pic, int e) {
  return ((pic->flags & HC_PIC_PCM_LF_DISABLED) && (e & HC_EDGE_PCM)) || (e & HC_EDGE_BYPASS);
}

static void count_sao_clip(int v, int maxv) {
  if (v < 0) HC_COUNT(k4_clip_lo);
  else if (v > maxv) HC_COUNT(k4_clip_hi);
}

/* sao.cc:261-488 apply_sao_internal, :552-625 driver. in = deblocked copy, out = picture. */
static void oracle_sao_plane(const hc_pic* pic, const hc_ctu* ctus, const uint8_t* edge, int cIdx, const uint16_t* in,
                             uint16_t* out, int stride) {
  const int SubW = (cIdx && (pic->chroma_format == 1 || pic->chroma_format == 2)) ? 2 : 1;
  const int SubH = (cIdx && pic->chroma_format == 1) ? 2 : 1;
  const int width = pic->width / SubW, height = pic->height / SubH;
  const int bitDepth = cIdx == 0 ? pic->bit_depth_y : pic->bit_depth_c;
  const int maxv = (1 << bitDepth) - 1;
  const int nSW = (1 << pic->log2_ctb) / SubW, nSH = (1 << pic->log2_ctb) / SubH;
  const int w4 = pic->width >> 2;
  for (int yCtb = 0; yCtb < pic->ctbs_h; yCtb++)
    for (int xCtb = 0; xCtb < pic->ctbs_w; xCtb++) {
      const hc_ctu* ctu = &ctus[xCtb + yCtb * pic->ctbs_w];
      const int type = ctu->sao_type[cIdx];
      if (!type) continue;
      const int xC = xCtb * nSW, yC = yCtb * nSH;
      const int ctbW = xC + nSW > width ? width - xC : nSW, ctbH = yC + nSH > height ? height - yC : nSH;
      const int nofilt = (ctu->flags & HC_CTU_HAS_NOFILTER) != 0;
      if (type == 2) {
        int hPos[2], vPos[2];
        switch (ctu->sao_band_or_class[cIdx]) {
          case 0: hPos[0] = -1; hPos[1] = 1; vPos[0] = 0; vPos[1] = 0; break;
          case 1: hPos[0] = 0; hPos[1] = 0; vPos[0] = -1; vPos[1] = 1; break;
          case 2: hPos[0] = -1; hPos[1] = 1; vPos[0] = -1; vPos[1] = 1; break;
          default: hPos[0] = 1; hPos[1] = -1; vPos[0] = -1; vPos[1] = 1; break;
        }
        int8_t off[5];
        off[0] = ctu->sao_offset[cIdx][0]; off[1] = ctu->sao_offset[cIdx][1]; off[2] = 0;
        off[3] = ctu->sao_offset[cIdx][2]; off[4] = ctu->sao_offset[cIdx][3];
        for (int j = 0; j < ctbH; j++)
          for (int i = 0; i < ctbW; i++) {
            const int x = xC + i, y = yC + j;
            if (nofilt && sao_sample_skipped(pic, edge[((x * SubW) >> 2) + (size_t)((y * SubH) >> 2) * w4])) { HC_COUNT(k4_skip_nofilter); continue; }
            int skip = 0;
            const int on_border = (i == 0 || j == 0 || i == ctbW - 1 || j == ctbH - 1);
            for (int k = 0; k < 2 && !skip; k++) {
              int xS = x + hPos[k], yS = y + vPos[k];
              if (xS < 0 || yS < 0 || xS >= width || yS >= height) { skip = 1; break; }
              /* neighbouring CTB usable? (sao.cc:377-395, resolved per CTB by the host) */
              int dx = (xS < xC) ? -1 : (xS >= xC + nSW ? 1 : 0), dy = (yS < yC) ? -1 : (yS >= yC + nSH ? 1 : 0);
              if (dx || dy) {
                int bit;
                if (dy == 0) bit = dx < 0 ? HC_NB_L : HC_NB_R;
                else if (dx == 0) bit = dy < 0 ? HC_NB_T : HC_NB_B;
                else if (dy < 0) bit = dx < 0 ? HC_NB_TL : HC_NB_TR;
                else bit = dx < 0 ? HC_NB_BL : HC_NB_BR;
                if (!((cIdx ? ctu->sao_nb_c : ctu->sao_nb) & bit)) skip = 1;
              } else if (cIdx && on_border && (ctu->flags & HC_CTU_SAO_C_SELF)) {
                skip = 1; /* reference quirk: see HC_CTU_SAO_C_SELF */
              }
            }
            if (skip) continue;
            const int c = in[x + (size_t)y * stride];
            const int e = isign(c - in[(x + hPos[0]) + (size_t)(y + vPos[0]) * stride]) +
                          isign(c - in[(x + hPos[1]) + (size_t)(y + vPos[1]) * stride]);
            count_sao_clip(c + off[e + 2], maxv);
            out[x + (size_t)y * stride] = (uint16_t)clip3i(0, maxv, c + off[e + 2]);
          }
      } else {
        const int bandShift = bitDepth - 5;
        int bandTable[32];
        memset(bandTable, 0, sizeof(bandTable));
        for (int k = 0; k < 4; k++) bandTable[(k + ctu->sao_band_or_class[cIdx]) & 31] = k + 1;
        for (int j = 0; j < ctbH; j++)
          for (int i = 0; i < ctbW; i++) {
            const int x = xC + i, y = yC + j;
            if (nofilt && sao_sample_skipped(pic, edge[((x * SubW) >> 2) + (size_t)((y * SubH) >> 2) * w4])) { HC_COUNT(k4_skip_nofilter); continue; }
            const int c = in[x + (size_t)y * stride];
            const int bandIdx = bandTable[c >> bandShift];
            if (bandIdx > 0) {
              if (bandIdx - 1 + ctu->sao_band_or_class[cIdx] > 31) HC_COUNT(k4_band_wrap);
              count_sao_clip(c + ctu->sao_offset[cIdx][bandIdx - 1], maxv);
              out[x + (size_t)y * stride] = (uint16_t)clip3i(0, maxv, c + ctu->sao_offset[cIdx][bandIdx - 1]);
            }
          }
      }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Stage selection, for testing kernels one at a time */
#define HC_ORACLE_STAGE_DEBLOCK 1
#define HC_ORACLE_STAGE_SAO 2

/* Reconstructs one picture. planes[c] must hold stride[c]*plane_height(c) uint16 samples.
 * Returns 0 on success. If `residual_out` is not NULL it receives pic->resid_count int16
 * residuals exactly as the K1 kernel must produce them (saturated to int16). */
int hc_oracle_reconstruct(const hc_pic* pic, const hc_ctu* ctus, const hc_blk* blks, const hc_tb* tbs,
                          const hc_coeff* coeffs, const uint8_t* edge_map, const int8_t* qp_map,
                          const uint8_t* scaling, int stages, uint16_t* planes[3], const int strides[3],
                          int16_t* residual_out) {
  const int ncomp = pic->chroma_format ? 3 : 1;
  int16_t* resid = residual_out;
  int own_resid = 0;
  if (!resid) {
    resid = (int16_t*)malloc(sizeof(int16_t) * (size_t)(pic->resid_count ? pic->resid_count : 1));
    if (!resid) return -1;
    own_resid = 1;
  }
  /* K1 equivalent */
  for (uint32_t t = 0; t < pic->tb_count; t++) {
    const hc_tb* tb = &tbs[t];
    int32_t r[32 * 32];
    const int n = 1 << (2 * tb->log2);
    oracle_tb_residual(pic, tb, coeffs + tb->coeff_off, scaling, r);
    for (int i = 0; i < n; i++) {
      if (r[i] < -32768 || r[i] > 32767) {
        if (tb->type & (HC_TB_RDPCM_H | HC_TB_RDPCM_V)) HC_COUNT(k1_rdpcm_clip);
        else if (tb->type & HC_TB_TSKIP) HC_COUNT(k1_tskip_clip);
        else if (!(tb->type & (HC_TB_BYPASS | HC_TB_DST))) HC_COUNT(k1_dct_store_clip);
      }
      resid[tb->resid_off + i] = (int16_t)clip3i(-32768, 32767, r[i]);
    }
  }
  /* K2 equivalent: CTBs in raster order, component chains independent */
  for (int a = 0; a < pic->ctbs_w * pic->ctbs_h; a++)
    for (int c = 0; c < ncomp; c++) {
      const hc_ctu* ctu = &ctus[a];
      for (uint32_t k = 0; k < ctu->blk_count[c]; k++) {
        const hc_blk* b = &blks[ctu->blk_first[c] + k];
        const int nT = 1 << b->log2;
        const int bd = c == 0 ? pic->bit_depth_y : pic->bit_depth_c;
        uint16_t pred[32 * 32];
        uint16_t* pl = planes[c];
        const int st = strides[c];
        if (b->flags & HC_BLK_PCM) {
          for (int y = 0; y < nT; y++)
            for (int x = 0; x < nT; x++) pl[(b->x + x) + (size_t)(b->y + y) * st] = (uint16_t)resid[b->resid_off + x + y * nT];
          continue;
        }
        oracle_predict(pic, b, pl, st, pred);
        for (int y = 0; y < nT; y++)
          for (int x = 0; x < nT; x++) {
            int v = pred[x + y * nT];
            if (b->flags & HC_BLK_HAS_RESID) {
              const int s = v + resid[b->resid_off + x + y * nT];
              if (s < 0) HC_COUNT(k2_add_clip_lo);
              else if (s > (1 << bd) - 1) HC_COUNT(k2_add_clip_hi);
              v = clip_bd(s, bd);
            }
            pl[(b->x + x) + (size_t)(b->y + y) * st] = (uint16_t)v;
          }
      }
    }
  if (own_resid) free(resid);

  /* K3 equivalent: deblock.cc:1921-1959 — all vertical edges, then all horizontal edges */
  if ((stages & HC_ORACLE_STAGE_DEBLOCK) && (pic->flags & HC_PIC_HAS_DEBLOCK)) {
    dbk_ctx d;
    d.pic = pic; d.ctus = ctus; d.edge = edge_map; d.qp = qp_map; d.w4 = pic->width >> 2; d.w8 = pic->width >> 3;
    for (int vertical = 1; vertical >= 0; vertical--) {
      oracle_deblock_luma(&d, planes[0], strides[0], vertical);
      if (ncomp == 3) {
        oracle_deblock_chroma(&d, planes[1], strides[1], vertical, 0);
        oracle_deblock_chroma(&d, planes[2], strides[2], vertical, 1);
      }
    }
  }
  /* K4 equivalent */
  if ((stages & HC_ORACLE_STAGE_SAO) && (pic->flags & HC_PIC_HAS_SAO)) {
    for (int c = 0; c < ncomp; c++) {
      const int SubH = (c && pic->chroma_format == 1) ? 2 : 1;
      const size_t n = (size_t)strides[c] * (pic->height / SubH);
      uint16_t* copy = (uint16_t*)malloc(n * sizeof(uint16_t));
      if (!copy) return -1;
      memcpy(copy, planes[c], n * sizeof(uint16_t));
      oracle_sao_plane(pic, ctus, edge_map, c, copy, planes[c], strides[c]);
      free(copy);
    }
  }
  return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* Block-level entry points used by the test-content generator (tools/hevc_enc) to keep its
 * encoding loop closed (its reconstruction is by construction what a conforming decoder yields). */
void hc_oracle_predict_block(const hc_pic* pic, const hc_blk* b, uint16_t* plane, int stride, uint16_t* dst) {
  oracle_predict(pic, b, plane, stride, dst);
}
void hc_oracle_residual_block(const hc_pic* pic, const hc_tb* tb, const hc_coeff* coeffs, const uint8_t* scaling,
                              int32_t* res) {
  oracle_tb_residual(pic, tb, coeffs, scaling, res);
}
