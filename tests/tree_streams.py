"""The coding-tree geometry corpus: small pictures from the synthetic-content encoder (tools/hevc_enc) over the coding
and transform tree parameters the SPS can signal for intra pictures: min CB 8 .. 64, min TB 4 .. 32, max TB from the min
TB up to min(CTB, 32), max_transform_hierarchy_depth_intra 0 .. 4, quantisation groups of one min CB, and conformance
windows wider than 7 samples. Every other corpus has min CB 8 and min TB 4. Generated at test time from fixed seeds, not
committed; the encoder's own reconstruction and QP map, the host parser and a restatement of the deblocking edge rule are
the references (test_tree_geometry.py). Kept apart from the other corpora so that their parametrizations do not change.
"""
import functools
import sys

from conftest import ROOT

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tools import hevcenc  # noqa: E402

ALL = hevcenc.STRESS_ALL
SEEDS = (1, 2)


def tree(ctb, min_cb, min_tb, max_tb, depth):
    """Encoder options of one geometry, in log2 sizes."""
    return dict(log2_ctb=ctb, log2_min_cb=min_cb, log2_min_tb=min_tb, log2_max_tb=max_tb, max_th_depth=depth)


# name -> (width, height, encoder options); stress=ALL unless given. Every entry has min TB < min CB <= CTB,
# max TB <= min(CTB, 5), depth <= CTB - min TB and cu_qp_delta - 1 <= CTB - min CB; subsampled chroma has even sizes,
# because the conformance window counts chroma samples.
CONFIGS = {
    # the device parser (K0) takes these
    "cb16_ctb16_wpp":      (120, 72, dict(tree(4, 4, 2, 4, 2), wpp=1, cu_qp_delta=1)),    # no split_cu_flag anywhere
    "cb16_tb8_10":         (120, 72, dict(tree(5, 4, 3, 5, 2), bit_depth=10, cu_qp_delta=2)),
    "cb32_tb16_422_12":    (144, 96, dict(tree(6, 5, 4, 5, 1), chroma_format=2, bit_depth=12, cu_qp_delta=2)),
    # 56-sample crop; CU 64 split by max TB beyond depth 0; NxN gives 32 x 32 PBs
    "cb64_tb32_444_d0":    (200, 136, dict(tree(6, 6, 5, 5, 0), chroma_format=3)),
    "cb64_tb8_d3_wpp":     (184, 120, dict(tree(6, 6, 3, 5, 3), wpp=1)),
    "depth4_420_10":       (128, 72, dict(tree(6, 3, 2, 5, 4), bit_depth=10, cu_qp_delta=3)),
    "depth4_422":          (96, 64, dict(tree(6, 6, 2, 5, 4), chroma_format=2)),         # every CU 64 x 64
    "depth0_mono_12":      (96, 64, dict(tree(5, 3, 2, 4, 0), chroma_format=0, bit_depth=12)),
    "tb8_only":            (96, 64, dict(tree(5, 4, 3, 3, 2))),                           # no split_transform_flag coded
    # slice segments of one CTB row; WPP forbids a segment that starts inside a row from leaving it
    "cb32_slices_dep_wpp": (256, 160, dict(tree(6, 5, 2, 5, 2), wpp=1, slice_ctbs=4, dependent_slices=1, cu_qp_delta=2)),
    "tskip8_mintb8":       (96, 64, dict(tree(4, 4, 3, 4, 1), transform_skip=1, log2_max_transform_skip_minus2=1)),
    # the host parser only
    "tiles_cb32":          (256, 192, dict(tree(6, 5, 3, 5, 2), tile_cols=2, tile_rows=2)),
    "pcm_cb16":            (96, 64, dict(tree(5, 4, 2, 5, 2), bit_depth=10, pcm=1)),
    "bypass_cb16_444":     (96, 64, dict(tree(5, 4, 3, 5, 2), chroma_format=3, transquant_bypass=1)),
}
K0_DECLINED = {"tiles_cb32": "HEVC tiles", "pcm_cb16": "pcm", "bypass_cb16_444": "transquant bypass"}

NAMES = ["%s#%d" % (n, s) for n in CONFIGS for s in SEEDS]
ELIGIBLE = [n for n in NAMES if n.split("#")[0] not in K0_DECLINED]
DECLINED = [n for n in NAMES if n not in ELIGIBLE]


def options(name):
    base, seed = name.split("#")
    w, h, kw = CONFIGS[base]
    kw = dict(kw, seed=int(seed))
    kw.setdefault("stress", ALL)
    return w, h, kw


@functools.lru_cache(maxsize=None)
def stream(name):
    """(bytes, {"recon": coded-size planes, "qp": QpY per 8 x 8, "stats" / "rext_stats" / "tree_stats": counters}) of
    one corpus entry, e.g. "cb16_tb8_10#1"."""
    w, h, kw = options(name)
    cf, bd = kw.get("chroma_format", 1), kw.get("bit_depth", 8)
    planes = hevcenc.synth_image(w, h, cf, bd, kw["seed"])
    return hevcenc.encode(planes, want=("recon", "qp", "stats"), **kw)


def data(name):
    return stream(name)[0]
