"""ctypes binding of the synthetic-content generator (tools/hevc_enc: closed-loop HEVC intra encoder).
Test / benchmark infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "hevc_enc", "_build", "libhevcenc.so")

FIELDS = ["width", "height", "chroma_format", "bit_depth", "qp", "log2_ctb", "log2_min_tb", "log2_max_tb", "max_th_depth",
          "sao", "deblock_disable", "beta_offset_div2", "tc_offset_div2", "sign_hiding", "cu_qp_delta", "transform_skip",
          "wpp", "tile_cols", "tile_rows", "slice_ctbs", "dependent_slices", "strong_intra", "scaling_list", "pcm",
          "transquant_bypass", "vui", "full_range", "matrix", "primaries", "transfer", "cb_qp_offset", "cr_qp_offset",
          "loop_filter_across_slices", "loop_filter_across_tiles", "stress",
          # range extensions (SPS / PPS range extension syntax); all 0: no extension is written
          "transform_skip_rotation", "transform_skip_context", "implicit_rdpcm", "intra_smoothing_disabled",
          "persistent_rice_adaptation", "extended_precision", "cabac_bypass_alignment", "log2_max_transform_skip_minus2",
          "cross_component_prediction", "chroma_qp_offset_list_len", "diff_cu_chroma_qp_offset_depth",
          "log2_sao_offset_scale_luma", "log2_sao_offset_scale_chroma"]

# stress bits (hevc_enc_params::stress): syntax values at the limits of their legal ranges, for parser tests
STRESS_LEVELS, STRESS_MODES, STRESS_QP, STRESS_SAO, STRESS_DENSE = 1, 2, 4, 8, 16
STRESS_ALL = STRESS_LEVELS | STRESS_MODES | STRESS_QP | STRESS_SAO


class Params(C.Structure):
    _fields_ = [(f, C.c_int32) for f in FIELDS] + [("seed", C.c_uint32)]


DEFAULTS = dict(chroma_format=1, bit_depth=8, qp=26, log2_ctb=6, log2_min_tb=2, log2_max_tb=5, max_th_depth=2, sao=1,
                sign_hiding=1, tile_cols=1, tile_rows=1, strong_intra=1, vui=1, full_range=1, matrix=6, primaries=1,
                transfer=13, loop_filter_across_slices=1, loop_filter_across_tiles=1, seed=1)

_lib = None


def build(force=False):
    src = os.path.join(HERE, "hevc_enc", "hevc_intra_enc.cc")
    if force or not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", os.path.join(HERE, "hevc_enc")], stdout=subprocess.DEVNULL)
    return SO


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.hevc_enc_encode.restype = C.c_int
        _lib.hevc_enc_encode_ex.restype = C.c_int
        _lib.hevc_enc_stat_name.restype = C.c_char_p
        _lib.hevc_enc_free.argtypes = [C.c_void_p]
    return _lib


def _all_stat_names():
    L = lib()
    return [L.hevc_enc_stat_name(i).decode() for i in range(L.hevc_enc_stat_count())]


def stat_names():
    """Counters of the syntax extremes the stress mode writes."""
    return _all_stat_names()[:lib().hevc_enc_rext_stat_first()]


def rext_stat_names():
    """Counters of the range-extension coding tools (the range-extension fields of the encoder options)."""
    return _all_stat_names()[lib().hevc_enc_rext_stat_first():]


def encode(planes, want=(), **kw):
    """planes: list of 2-D integer arrays (Y[,Cb,Cr]) of the visible picture. Returns bytes:
    4-byte-length-prefixed NAL units (VPS, SPS, PPS, slice segments).
    want: any of "recon" (the encoder's reconstruction before the in-loop filters: uint16 planes of the coded size,
    width and height rounded up to a multiple of 8) and "stats" ({counter name: count} of what was written: the stress
    counters under "stats", the range-extension ones under "rext_stats"). With a
    non-empty want the result is (bytes, {name: value})."""
    L = lib()
    opts = dict(DEFAULTS)
    opts.update(kw)
    p = Params()
    for k, v in opts.items():
        setattr(p, k, int(v))
    p.height, p.width = planes[0].shape
    pl = [np.ascontiguousarray(a, np.uint16) for a in planes]
    pp = (C.c_void_p * 3)(*([a.ctypes.data for a in pl] + [None] * (3 - len(pl))))
    st = (C.c_int * 3)(*([a.shape[1] for a in pl] + [0] * (3 - len(pl))))
    out, size = C.c_void_p(), C.c_size_t()
    recon = rp = stats = None
    if "recon" in want:
        cf = p.chroma_format
        w8, h8 = (p.width + 7) & ~7, (p.height + 7) & ~7
        sw, sh = (2 if cf in (1, 2) else 1), (2 if cf == 1 else 1)
        recon = [np.zeros(d, np.uint16) for d in [(h8, w8)] + ([(h8 // sh, w8 // sw)] * 2 if cf else [])]
        rp = (C.c_void_p * 3)(*([a.ctypes.data for a in recon] + [None] * (3 - len(recon))))
    if "stats" in want:
        stats = (C.c_uint64 * L.hevc_enc_stat_count())()
    rc = L.hevc_enc_encode_ex(C.byref(p), pp, st, C.byref(out), C.byref(size), rp, stats)
    if rc != 0:
        raise RuntimeError("hevc_enc_encode failed: %d" % rc)
    data = C.string_at(out, size.value)
    L.hevc_enc_free(out)
    if not want:
        return data
    extra = {}
    if recon is not None:
        extra["recon"] = recon
    if stats is not None:
        first = L.hevc_enc_rext_stat_first()
        counts = dict(zip(_all_stat_names(), (int(v) for v in stats)))
        extra["stats"] = {k: counts[k] for k in _all_stat_names()[:first]}
        extra["rext_stats"] = {k: counts[k] for k in _all_stat_names()[first:]}
    return data, extra


def split_nals(stream):
    """length-prefixed stream -> list of NAL unit byte strings"""
    nals, pos = [], 0
    while pos + 4 <= len(stream):
        n = int.from_bytes(stream[pos:pos + 4], "big")
        nals.append(stream[pos + 4:pos + 4 + n])
        pos += 4 + n
    return nals


def to_annexb(stream):
    return b"".join(b"\x00\x00\x00\x01" + n for n in split_nals(stream))


def synth_image(width, height, chroma_format=1, bit_depth=8, seed=0):
    """Seeded synthetic picture: smooth gradients + band-limited noise + sharp edges (SURVEY.md 8d)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:height, 0:width].astype(np.float32)
    maxv = (1 << bit_depth) - 1
    base = 0.5 + 0.25 * np.sin(xx / (37.0 + seed % 7)) * np.cos(yy / 53.0) + 0.2 * (xx / max(width, 1) - 0.5)
    # band-limited noise: blur white noise with a small box filter
    noise = rng.normal(0, 1, (height, width)).astype(np.float32)
    k = 3
    noise = sum(np.roll(np.roll(noise, i, 0), j, 1) for i in range(-k, k + 1) for j in range(-k, k + 1)) / (2 * k + 1) ** 2
    img = base + 0.35 * noise
    # sharp edges: rectangles and a diagonal
    for _ in range(max(2, width * height // 60000)):
        x0, y0 = rng.integers(0, width), rng.integers(0, height)
        w, h = rng.integers(8, max(9, width // 4)), rng.integers(8, max(9, height // 4))
        img[y0:y0 + h, x0:x0 + w] += rng.uniform(-0.3, 0.3)
    img[(xx + yy).astype(np.int32) % 97 < 2] += 0.25
    img += rng.normal(0, 6.0 / 255.0, img.shape)
    y = np.clip(img * maxv, 0, maxv).astype(np.uint16)
    if chroma_format == 0:
        return [y]
    sw = 2 if chroma_format in (1, 2) else 1
    sh = 2 if chroma_format == 1 else 1
    cw, ch = (width + sw - 1) // sw, (height + sh - 1) // sh
    cy, cx = np.mgrid[0:ch, 0:cw].astype(np.float32)
    cb = 0.5 + 0.2 * np.sin(cx / 29.0 + seed) + 0.1 * np.cos(cy / 41.0) + rng.normal(0, 3.0 / 255.0, (ch, cw))
    cr = 0.5 + 0.2 * np.cos(cx / 31.0) * np.sin(cy / 23.0 + seed) + rng.normal(0, 3.0 / 255.0, (ch, cw))
    return [y, np.clip(cb * maxv, 0, maxv).astype(np.uint16), np.clip(cr * maxv, 0, maxv).astype(np.uint16)]
