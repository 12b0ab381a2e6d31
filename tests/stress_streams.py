"""The stress corpus: small pictures from the synthetic-content encoder (tools/hevc_enc) in stress mode, whose syntax
values sit at the limits of their legal ranges (levels of -32768 and 32767, long escape codes, dense sub-blocks, TB and
coefficient counts at the per-CTB capacity, QPs over the whole legal range with the wrap of 8.6.1, uniform intra modes,
the full SAO offset range). Generated at test time from fixed seeds; not committed, because no reference decoder
pins their output: the encoder's own reconstruction and the host parser are the references (test_syntax_extremes.py).
"""
import functools
import sys

from conftest import ROOT

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tools import hevcenc  # noqa: E402

ALL, DENSE = hevcenc.STRESS_ALL, hevcenc.STRESS_ALL | hevcenc.STRESS_DENSE
SEEDS = (1, 2)

# name -> (width, height, encoder options); stress=ALL unless given
CONFIGS = {
    "mono_8":          (96, 64, dict(chroma_format=0)),
    "mono_12_qg":      (120, 72, dict(chroma_format=0, bit_depth=12, cu_qp_delta=2)),
    "c420_8":          (96, 64, dict()),
    "c420_10_wpp_qg":  (120, 72, dict(bit_depth=10, cu_qp_delta=3, wpp=1)),
    "c420_12_ctb16":   (120, 72, dict(bit_depth=12, cu_qp_delta=1, log2_ctb=4)),
    "c422_8":          (96, 64, dict(chroma_format=2)),
    "c422_10_qg":      (96, 64, dict(chroma_format=2, bit_depth=10, cu_qp_delta=2)),
    "c422_12_qg":      (120, 72, dict(chroma_format=2, bit_depth=12, cu_qp_delta=3)),
    "c444_8_qg":       (96, 64, dict(chroma_format=3, cu_qp_delta=3)),
    "c444_10_ctb32":   (96, 64, dict(chroma_format=3, bit_depth=10, log2_ctb=5)),
    "c444_12":         (96, 64, dict(chroma_format=3, bit_depth=12)),
    # every TB 4x4 and every coefficient non-zero: full CTBs reach their TB and coefficient capacity (768 TBs at 64 x 64
    # 4:4:4, the parser's TB_CAP_MAX)
    "dense_444_ctb64": (128, 64, dict(chroma_format=3, log2_max_tb=2, stress=DENSE)),
    "dense_422_wpp":   (128, 64, dict(chroma_format=2, bit_depth=10, log2_ctb=5, log2_max_tb=2, wpp=1, stress=DENSE)),
    "wpp_dep_slices":  (160, 96, dict(wpp=1, log2_ctb=5, slice_ctbs=5, dependent_slices=1, cu_qp_delta=2, bit_depth=10)),
    "slices":          (136, 96, dict(log2_ctb=4, slice_ctbs=7, cu_qp_delta=1)),
    "one_ctb_wide":    (40, 136, dict(wpp=1, log2_ctb=5, cu_qp_delta=2)),
    "odd_420":         (131, 75, dict(bit_depth=10, cu_qp_delta=2)),
    "odd_444":         (101, 67, dict(chroma_format=3, log2_ctb=4)),
    "no_sign_hiding":  (96, 64, dict(sign_hiding=0, cu_qp_delta=3)),
    "no_sdh_dense":    (64, 64, dict(sign_hiding=0, chroma_format=2, log2_max_tb=3, stress=DENSE)),
    "tskip_12":        (96, 64, dict(transform_skip=1, bit_depth=12, cu_qp_delta=2)),
    "scaling_422_12":  (96, 64, dict(scaling_list=2, chroma_format=2, bit_depth=12)),
    "qp_low_12":       (96, 64, dict(bit_depth=12, qp=-24, cu_qp_delta=3, cb_qp_offset=12, cr_qp_offset=-12)),
    "qp51_8":          (96, 64, dict(qp=51, cu_qp_delta=1, cb_qp_offset=12, cr_qp_offset=12)),
    "qp_offsets_10":   (96, 64, dict(bit_depth=10, cu_qp_delta=3, cb_qp_offset=-12, cr_qp_offset=12, beta_offset_div2=6,
                                     tc_offset_div2=-6)),
    "dbk_offsets_444": (96, 64, dict(chroma_format=3, bit_depth=10, beta_offset_div2=-6, tc_offset_div2=6, cu_qp_delta=2)),
    # coding tools the device parser leaves to the host parser
    "tiles":           (136, 96, dict(tile_cols=2, tile_rows=2, log2_ctb=4, cu_qp_delta=2)),
    "pcm":             (96, 64, dict(pcm=1, bit_depth=10)),
    "bypass_422":      (96, 64, dict(transquant_bypass=1, chroma_format=2)),
}
K0_DECLINED = {"tiles", "pcm", "bypass_422"}

NAMES = ["%s#%d" % (n, s) for n in CONFIGS for s in SEEDS]
ELIGIBLE = [n for n in NAMES if n.split("#")[0] not in K0_DECLINED]


def options(name):
    base, seed = name.split("#")
    w, h, kw = CONFIGS[base]
    kw = dict(kw, seed=int(seed))
    kw.setdefault("stress", ALL)
    return w, h, kw


@functools.lru_cache(maxsize=None)
def stream(name):
    """(bytes, {"recon": coded-size planes, "stats": counters}) of one corpus entry, e.g. "c420_8#1"."""
    w, h, kw = options(name)
    cf, bd = kw.get("chroma_format", 1), kw.get("bit_depth", 8)
    planes = hevcenc.synth_image(w, h, cf, bd, kw["seed"])
    return hevcenc.encode(planes, want=("recon", "stats"), **kw)


def data(name):
    return stream(name)[0]
