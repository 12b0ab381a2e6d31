/*
 * oracle_counters.h — branch counters of the CPU oracle (hevc_recon_oracle.c, csc_oracle.c).
 *
 * TEST INFRASTRUCTURE ONLY. Each counter counts how often a value-dependent branch of the oracle was
 * taken: a clip, a wrap, a filter decision, a table index clamped at its end. The kernels have the same
 * branches, so a test corpus that leaves a counter at 0 cannot show that the kernels take that branch
 * correctly (tests/test_record_extremes.py). Counting never changes an output.
 */
#ifndef HC_ORACLE_COUNTERS_H
#define HC_ORACLE_COUNTERS_H

#include <stdint.h>

#define HC_ORACLE_INTRA_MODE_COUNTERS                                                                                \
  X(k2_mode_0) X(k2_mode_1) X(k2_mode_2) X(k2_mode_3) X(k2_mode_4) X(k2_mode_5) X(k2_mode_6) X(k2_mode_7)           \
  X(k2_mode_8) X(k2_mode_9) X(k2_mode_10) X(k2_mode_11) X(k2_mode_12) X(k2_mode_13) X(k2_mode_14) X(k2_mode_15)     \
  X(k2_mode_16) X(k2_mode_17) X(k2_mode_18) X(k2_mode_19) X(k2_mode_20) X(k2_mode_21) X(k2_mode_22) X(k2_mode_23)   \
  X(k2_mode_24) X(k2_mode_25) X(k2_mode_26) X(k2_mode_27) X(k2_mode_28) X(k2_mode_29) X(k2_mode_30) X(k2_mode_31)   \
  X(k2_mode_32) X(k2_mode_33) X(k2_mode_34)

#define HC_ORACLE_COUNTERS                                                                                        \
  X(k1_flat_dequant_wrap)      /* flat dequantisation result wrapped in int32 */                                   \
  X(k1_dequant_clip16)         /* dequantised coefficient clipped to int16 (flat or scaled) */                     \
  X(k1_scaled_factor_ge200)    /* scaled dequantisation with a scaling factor >= 200 */                            \
  X(k1_dct_pass1_clip)         /* DCT first (column) pass clipped to int16 */                                      \
  X(k1_dct_store_clip)         /* DCT second pass result clipped to int16 when stored */                           \
  X(k1_dst_pass1_clip)         /* DST first pass clipped to int16 */                                               \
  X(k1_dst_pass2_clip)         /* DST second pass clipped to int16 */                                              \
  X(k1_tskip_clip)             /* transform-skip residual clipped to int16 when stored */                          \
  X(k1_rdpcm_clip)             /* RDPCM accumulation (transform skip or bypass) clipped to int16 when stored */    \
  X(k2_add_clip_lo)            /* prediction + residual clipped to 0 */                                            \
  X(k2_add_clip_hi)            /* prediction + residual clipped to the maximum sample value */                     \
  X(k2_strong_smoothing)       /* bilinear strong intra smoothing of a 32x32 luma reference */                     \
  X(k2_121_smoothing)          /* [1 2 1] reference smoothing */                                                   \
  HC_ORACLE_INTRA_MODE_COUNTERS                                                                                    \
  X(k3_luma_strong)            /* luma strong filter applied to a 4-line segment */                                \
  X(k3_luma_weak)              /* luma weak filter applied to a 4-line segment */                                  \
  X(k3_luma_weak_nd2)          /* ... with nDp > 1 or nDq > 1 */                                                   \
  X(k3_tc_idx_clamp_lo)        /* tc table index clamped at 0 */                                                   \
  X(k3_tc_idx_clamp_hi)        /* tc table index clamped at 53 */                                                  \
  X(k3_beta_idx_clamp)         /* beta table index clamped at 0 or 51 */                                           \
  X(k3_chroma_qpi_30_43)       /* chroma qPi inside the 30..43 region of the 4:2:0 table */                       \
  X(k3_chroma_qpi_neg)         /* chroma qPi < 0 */                                                                \
  X(k4_band_wrap)              /* band offset applied through a band index that wrapped past 31 */                 \
  X(k4_clip_lo)                /* SAO result clipped to 0 */                                                       \
  X(k4_clip_hi)                /* SAO result clipped to the maximum sample value */                                \
  X(k4_skip_nofilter)          /* SAO sample left untouched because it is pcm (loop filter off) or bypass */       \
  X(k5_clip_lo_8) X(k5_clip_hi_8)     /* colour conversion output clipped, by the depth of the clip */            \
  X(k5_clip_lo_10) X(k5_clip_hi_10)                                                                                \
  X(k5_clip_lo_12) X(k5_clip_hi_12)

enum hc_oracle_counter_id {
#define X(n) HC_CNT_##n,
  HC_ORACLE_COUNTERS
#undef X
  HC_CNT_COUNT
};

extern uint64_t hc_oracle_counter[HC_CNT_COUNT];   /* defined in hevc_recon_oracle.c */
#define HC_COUNT(n) (hc_oracle_counter[HC_CNT_##n]++)

#endif
