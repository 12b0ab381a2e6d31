"""The range-extension corpus: small pictures from the synthetic-content encoder (tools/hevc_enc) with the HEVC range
extension coding tools switched on (SPS / PPS range extension syntax): transform skip up to 32 x 32, implicit RDPCM,
transform-skip rotation and contexts, intra smoothing disabled, persistent Rice adaptation, CU chroma QP offset lists and
the SAO offset scale, plus three streams with tools the decoder refuses. Generated at test time from fixed seeds, not
committed; the encoder's own reconstruction and the host parser are the references (test_rext_tools.py). Kept apart
from stress_streams.CONFIGS so that the parametrizations of test_syntax_extremes.py do not change.
"""
import functools
import sys

from conftest import ROOT

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tools import hevcenc  # noqa: E402

ALL, DENSE = hevcenc.STRESS_ALL, hevcenc.STRESS_ALL | hevcenc.STRESS_DENSE
NATURAL_MODES = ALL & ~hevcenc.STRESS_MODES     # the encoder's own mode decisions: modes 10 and 26 are frequent
SEEDS = (1, 2)

# every residual tool of the SPS / PPS range extensions that a transform-skipped block can carry
TS = dict(transform_skip=1, transform_skip_rotation=1, transform_skip_context=1, implicit_rdpcm=1)
TS32 = dict(TS, log2_max_transform_skip_minus2=3)

# name -> (width, height, encoder options); stress=ALL unless given
CONFIGS = {
    # the device parser (K0) takes these
    "ts32_420_8":       (96, 64, dict(TS32, stress=NATURAL_MODES)),
    "ts32_420_8_modes": (96, 64, dict(TS32)),
    "ts_422_10_wpp":    (128, 64, dict(TS32, chroma_format=2, bit_depth=10, wpp=1, log2_ctb=5)),
    "nosmooth_444_12":  (128, 96, dict(TS, chroma_format=3, bit_depth=12, intra_smoothing_disabled=1, strong_intra=1,
                                       stress=hevcenc.STRESS_SAO)),
    "nosmooth_420_10":  (128, 96, dict(intra_smoothing_disabled=1, strong_intra=1, bit_depth=10, stress=0)),
    "mono_12_sao2":     (96, 64, dict(TS32, chroma_format=0, bit_depth=12, log2_sao_offset_scale_luma=2, log2_ctb=4)),
    "sao_scale_444_12": (96, 64, dict(chroma_format=3, bit_depth=12, log2_sao_offset_scale_luma=1,
                                      log2_sao_offset_scale_chroma=2, log2_ctb=4)),
    # custom scaling lists on transform-skipped blocks up to 32 x 32 (DESIGN 4: which ScalingFactor they take)
    "scaling_ts32":     (96, 64, dict(TS32, scaling_list=2, stress=NATURAL_MODES)),
    "scaling_ts32_422": (96, 64, dict(TS32, scaling_list=2, chroma_format=2, bit_depth=12)),
    # every coefficient non-zero: RDPCM accumulation leaves the int16 range
    "dense_rdpcm_12":   (64, 64, dict(TS32, bit_depth=12, stress=DENSE)),
    "dense_rdpcm_444":  (64, 64, dict(TS32, chroma_format=3, stress=DENSE & ~hevcenc.STRESS_MODES)),
    "odd_ctb16":        (131, 75, dict(TS, log2_max_transform_skip_minus2=2, log2_ctb=4, bit_depth=10)),
    "odd_ctb32_444":    (101, 67, dict(TS32, chroma_format=3, log2_ctb=5, cu_qp_delta=2)),
    # the host parser only: transquant bypass, persistent Rice adaptation, CU chroma QP offsets
    "bypass_420":       (96, 64, dict(TS32, transquant_bypass=1, stress=NATURAL_MODES)),
    "bypass_422":       (96, 64, dict(TS32, transquant_bypass=1, chroma_format=2, bit_depth=10, stress=NATURAL_MODES)),
    "rice_wpp_dep":     (160, 96, dict(TS32, persistent_rice_adaptation=1, wpp=1, log2_ctb=5, slice_ctbs=5,
                                       dependent_slices=1, bit_depth=10)),
    "rice_tiles":       (136, 96, dict(TS, persistent_rice_adaptation=1, tile_cols=2, tile_rows=2, log2_ctb=4,
                                       chroma_format=3)),
    "cqo_lists":        (160, 96, dict(chroma_qp_offset_list_len=6, diff_cu_chroma_qp_offset_depth=2, cu_qp_delta=2,
                                       cb_qp_offset=-3, cr_qp_offset=4)),
    "cqo_422_len1":     (96, 64, dict(chroma_qp_offset_list_len=1, diff_cu_chroma_qp_offset_depth=2, cu_qp_delta=3,
                                      chroma_format=2, bit_depth=10, transquant_bypass=1)),
}
K0_DECLINED = {"bypass_420": "transquant bypass", "bypass_422": "transquant bypass",
               "rice_wpp_dep": "persistent_rice_adaptation", "rice_tiles": "HEVC tiles",
               "cqo_lists": "cu_chroma_qp_offset", "cqo_422_len1": "transquant bypass"}

# streams the decoder refuses, and the flag the refusal names
REFUSED = {
    "extended_precision":     (64, 64, dict(extended_precision=1, chroma_format=3, bit_depth=12),
                               "extended_precision_processing_flag"),
    "cabac_bypass_alignment": (64, 64, dict(cabac_bypass_alignment=1, chroma_format=2, bit_depth=10),
                               "cabac_bypass_alignment_enabled_flag"),
    "cross_component":        (64, 64, dict(cross_component_prediction=1, chroma_format=3), "cross_component_prediction"),
}

NAMES = ["%s#%d" % (n, s) for n in CONFIGS for s in SEEDS]
ELIGIBLE = [n for n in NAMES if n.split("#")[0] not in K0_DECLINED]
DECLINED = [n for n in NAMES if n not in ELIGIBLE]
REFUSED_NAMES = ["%s#%d" % (n, s) for n in REFUSED for s in SEEDS]


def options(name):
    base, seed = name.split("#")
    w, h, kw = CONFIGS[base] if base in CONFIGS else REFUSED[base][:3]
    kw = dict(kw, seed=int(seed))
    kw.setdefault("stress", ALL)
    return w, h, kw


@functools.lru_cache(maxsize=None)
def stream(name):
    """(bytes, {"recon": coded-size planes, "stats" / "rext_stats": counters}) of one corpus entry, e.g. "ts32_420_8#1"."""
    w, h, kw = options(name)
    cf, bd = kw.get("chroma_format", 1), kw.get("bit_depth", 8)
    planes = hevcenc.synth_image(w, h, cf, bd, kw["seed"])
    return hevcenc.encode(planes, want=("recon", "stats"), **kw)


def data(name):
    return stream(name)[0]
