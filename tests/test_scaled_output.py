"""Scaled output: images delivered at a bounded size (engine option "scale_max_side") or at any size per canvas
(hc_batch_set_canvas_output_size), with the nearest-neighbour sampling of heif_image_scale_image
(HeifPixelImage::scale_nearest_neighbor, pixelimage.cc:1156-1253) fused into K5 and K7.
Every GPU comparison is pinned the same way: the engine's full-size output of a file has its golden MD5 (or equals the
restatement), and the scaled output equals scale_nearest of that full-size output viewed as (H, W, bytes per pixel).
CPU tests: scale_nearest on interleaved pixels, and the fit rule restated here (the GPU tests use the same restatement)."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import pytest

import heif_b200 as hb
import heic_oracle as ho
from conftest import ROOT
from heif_b200 import api
from heif_b200._lib import CscParams

sys.path.insert(0, ROOT)

DIR = os.path.join(ROOT, "tests", "golden", "heic")
META = json.load(open(os.path.join(ROOT, "tests", "golden", "heic.json")))
FMETA = json.load(open(os.path.join(ROOT, "tests", "golden", "heic_formats.json")))
BMETA = json.load(open(os.path.join(ROOT, "tests", "golden", "heic_formats_bilinear.json")))
IMETA = json.load(open(os.path.join(ROOT, "tests", "golden", "iovl.json")))
NAMES = sorted(META)
FORMATS = {"rgb": hb.OUT_RGB, "rgba": hb.OUT_RGBA, "rrggbb_be": hb.OUT_RRGGBB_BE, "rrggbbaa_be": hb.OUT_RRGGBBAA_BE,
           "rrggbb_le": hb.OUT_RRGGBB_LE, "rrggbbaa_le": hb.OUT_RRGGBBAA_LE}
BPP = api.OUT_BYTES_PER_PIXEL
ERR_ARGUMENT, ERR_UNSUPPORTED = -2, -6


def load(name):
    return open(os.path.join(DIR, name + ".heic"), "rb").read()


def load_iovl(name):
    return open(os.path.join(ROOT, "tests", "golden", "iovl", name + ".heic"), "rb").read()


def md5(b):
    return hashlib.md5(b).hexdigest()


def fit(W, H, S):
    """the fit rule of "scale_max_side" (include/heifcuda.h): delivered size of a W x H image"""
    if S <= 0 or max(W, H) <= S:
        return W, H
    if W >= H:
        return S, max(1, H * S // W)
    return max(1, W * S // H), S


def scale_rows(rows, bpp, w, h):
    """scale_nearest of interleaved rows (H x W * bpp bytes) viewed as (H, W, bpp): whole pixels are copied"""
    H = rows.shape[0]
    px = rows.reshape(H, -1, bpp)
    return ho.scale_nearest(px, w, h).reshape(h, w * bpp)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("bpp", [3, 4, 6, 8])
def test_scale_nearest_copies_whole_pixels(bpp):
    rng = np.random.default_rng(bpp)
    for (H, W), (h, w) in [((7, 5), (3, 2)), ((5, 7), (11, 13)), ((1, 9), (1, 4)), ((9, 1), (4, 1)), ((13, 17), (13, 17)),
                           ((2, 3), (1, 1)), ((31, 29), (8, 33))]:
        src = rng.integers(0, 256, (H, W, bpp), dtype=np.uint8)
        want = np.empty((h, w, bpp), np.uint8)
        for y in range(h):
            for x in range(w):
                want[y, x, :] = src[y * H // h, x * W // w, :]
        assert np.array_equal(ho.scale_nearest(src, w, h), want), ((H, W), (h, w))
        assert np.array_equal(scale_rows(src.reshape(H, W * bpp), bpp, w, h), want.reshape(h, w * bpp))


def test_fit_rule():
    assert fit(4032, 3024, 512) == (512, 384)
    assert fit(3024, 4032, 512) == (384, 512)
    assert fit(640, 384, 97) == (97, 58)          # 384 * 97 / 640 = 58.2
    assert fit(300, 300, 7) == (7, 7)
    assert fit(1, 1000, 7) == (1, 7) and fit(1000, 1, 7) == (7, 1)
    assert fit(8, 200, 20) == (1, 20) and fit(200, 8, 20) == (20, 1)      # 0.8 rounds to 0 and becomes 1
    assert fit(640, 384, 640) == (640, 384) and fit(640, 384, 645) == (640, 384) and fit(640, 384, 0) == (640, 384)
    for W in range(1, 40):
        for H in range(1, 40):
            for S in (1, 2, 7, 16):
                w, h = fit(W, H, S)
                assert 1 <= w <= W and 1 <= h <= H and max(w, h) == min(max(W, H), S), (W, H, S)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    yield e
    e.close()


class Options:
    """engine options for the duration of a with-block, restored to their defaults afterwards"""
    DEFAULTS = {"scale_max_side": 0, "device_parse": 1, "host_share_pct": -1, "chroma_upsampling": 0, "premultiply_alpha": 0}

    def __init__(self, engine, **opts):
        self.engine, self.opts = engine, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.engine.set_option(k, v)

    def __exit__(self, *exc):
        for k in self.opts:
            self.engine.set_option(k, self.DEFAULTS[k])


def run_job(engine, files, fmt, **opts):
    """(descs, rows of every image) of one hc_heic_job under the given engine options"""
    with Options(engine, **opts):
        job = hb.HeicJob(engine, files, threads=4, out_format=fmt)
    try:
        job.upload()
        job.run()
        return list(job.descs), [job.read_rgb(i) for i in range(len(files))]
    finally:
        job.close()


def check_scaled(full, descs, rows, fmt, S, labels):
    """every image of a scaled job against scale_nearest of its full-size output"""
    bad = []
    for k, (f, d, r) in enumerate(zip(full, descs, rows)):
        H, W = f.shape[0], f.shape[1] // BPP[fmt]
        w, h = fit(W, H, S)
        assert (d.width, d.height, d.out_format, d.bytes_per_pixel) == (w, h, fmt, BPP[fmt]), (labels[k], S)
        if not np.array_equal(r, scale_rows(f, BPP[fmt], w, h)):
            bad.append((labels[k], S))
    return bad


def scale_values(names, sizes):
    """S of the fixed set and, per longest side M, M - 1 (scaled by one pixel), M and M + 5 (unchanged)"""
    groups = {}
    for n, (W, H) in zip(names, sizes):
        groups.setdefault(max(W, H), []).append(n)
    return [(S, names) for S in (1, 7, 64, 97)] + [(S, g) for M, g in sorted(groups.items()) for S in (M - 1, M, M + 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("device_parse", [1, 0])
@pytest.mark.parametrize("key", sorted(FORMATS))
def test_gpu_every_fixture_and_format_scaled(engine, key, device_parse):
    fmt = FORMATS[key]
    names = [n for n in NAMES if key + "_md5" in FMETA[n]]
    assert len(names) == 53
    descs, full = run_job(engine, [load(n) for n in names], fmt, device_parse=device_parse, host_share_pct=0)
    assert [md5(r.tobytes()) for r in full] == [FMETA[n][key + "_md5"] for n in names]
    by_name = dict(zip(names, full))
    bad = []
    for S, group in scale_values(names, [(d.width, d.height) for d in descs]):
        d, rows = run_job(engine, [load(n) for n in group], fmt, scale_max_side=S, device_parse=device_parse, host_share_pct=0)
        bad += check_scaled([by_name[n] for n in group], d, rows, fmt, S, group)
        for n, r in zip(group, rows):
            if S >= max(by_name[n].shape[0], by_name[n].shape[1] // BPP[fmt]):
                assert md5(r.tobytes()) == FMETA[n][key + "_md5"], (n, S)      # within S: the golden itself
    assert not bad, bad[:20]


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["rgb", "rgba", "rrggbb_le", "rrggbbaa_be"])
def test_gpu_bilinear_upsampling_scaled(engine, key):
    fmt = FORMATS[key]
    names = [n for n in NAMES if key + "_md5" in BMETA[n] and not (n.startswith("single_mono") and fmt > hb.OUT_RGBA)]
    _, full = run_job(engine, [load(n) for n in names], fmt, chroma_upsampling=1)
    assert [md5(r.tobytes()) for r in full] == [BMETA[n][key + "_md5"] for n in names]
    for S in (1, 7, 33, 97, 255):
        d, rows = run_job(engine, [load(n) for n in names], fmt, chroma_upsampling=1, scale_max_side=S)
        bad = check_scaled(full, d, rows, fmt, S, names)
        assert not bad, bad


@pytest.mark.gpu
def test_gpu_premultiplied_alpha_scaled(engine):
    names = [n for n in NAMES if "rgba_premultiplied_md5" in FMETA[n]]
    descs, full = run_job(engine, [load(n) for n in names], hb.OUT_RGBA, premultiply_alpha=1)
    want = [FMETA[n]["rgba_md5"] if n == "alpha_prem_420_8" else FMETA[n]["rgba_premultiplied_md5"] for n in names]
    assert [md5(r.tobytes()) for r in full] == want
    for S in (1, 7, 97):
        d, rows = run_job(engine, [load(n) for n in names], hb.OUT_RGBA, premultiply_alpha=1, scale_max_side=S)
        assert all(x.premultiplied_alpha == 1 for x in d)
        bad = check_scaled(full, d, rows, hb.OUT_RGBA, S, names)
        assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("key", sorted(FORMATS))
def test_gpu_overlays_scaled(engine, key):
    """K7 samples the composed 'iovl' image; the children stay full size"""
    fmt = FORMATS[key]
    names = sorted(IMETA)
    _, full = run_job(engine, [load_iovl(n) for n in names], fmt)
    assert [md5(r.tobytes()) for r in full] == [IMETA[n][key + "_md5"] for n in names]
    M = max(max(IMETA[n]["canvas"]) for n in names)
    for S in (1, 7, 97, M - 1, M):
        d, rows = run_job(engine, [load_iovl(n) for n in names], fmt, scale_max_side=S)
        bad = check_scaled(full, d, rows, fmt, S, names)
        assert not bad, bad


# ---- stream --------------------------------------------------------------------------------------------------------
STREAM_S = 50


def _full_rgb(engine, names):
    descs, full = run_job(engine, [load(n) for n in names], None)
    key = {hb.OUT_RGB: "rgb", hb.OUT_RGBA: "rgba", hb.OUT_RRGGBB_LE: "rrggbb_le", hb.OUT_RRGGBBAA_LE: "rrggbbaa_le"}
    assert [md5(r.tobytes()) for r in full] == [META[n][key[d.out_format] + "_md5"] for n, d in zip(names, descs)]
    return [(d.out_format, r) for d, r in zip(descs, full)]


def _want(full, S):
    out = []
    for fmt, f in full:
        w, h = fit(f.shape[1] // BPP[fmt], f.shape[0], S)
        out.append(scale_rows(f, BPP[fmt], w, h))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("host_share", [0, 100])
def test_gpu_stream_scaled(engine, host_share):
    names = NAMES
    want = _want(_full_rgb(engine, names), STREAM_S)
    for per_batch in (1, 3, 7):
        got = {}

        def on_image(index, desc, rows):
            got[index] = ((desc.width, desc.height), np.array(rows[:, :desc.width * desc.bytes_per_pixel]))

        with Options(engine, scale_max_side=STREAM_S, host_share_pct=host_share):
            st = hb.decode_stream(engine, [load(n) for n in names], on_image, threads=4, files_per_batch=per_batch)
        assert sorted(got) == list(range(len(names)))
        bad = [names[k] for k in got if got[k][1].shape != want[k].shape or not np.array_equal(got[k][1], want[k])]
        assert not bad, (per_batch, bad)
        assert st["bytes_d2h"] == sum(w.size for w in want)
        assert st["pixels"] == sum(g[0][0] * g[0][1] for g in got.values())
        assert st["batches"] == (len(names) + per_batch - 1) // per_batch


@pytest.mark.gpu
def test_gpu_stream_scaled_external_destinations(engine):
    """Destinations sized for the scaled image are used; one byte too small (or a stride under the scaled row) is ignored
    and the image arrives in the library's memory, still scaled."""
    names = NAMES[:16]
    want = _want(_full_rgb(engine, names), STREAM_S)
    dests, kinds = [], []
    for k, w in enumerate(want):
        kind = ("exact", "wide", "small", "none")[k % 4]
        h, row = w.shape
        if kind == "exact":
            dests.append(np.zeros((h, row), np.uint8))
        elif kind == "wide":
            dests.append(np.zeros((h, row + 40), np.uint8))
        elif kind == "small":     # one row short, or (a single row) one byte short
            dests.append(np.zeros((h - 1, row), np.uint8) if h > 1 else np.zeros((1, row - 1), np.uint8))
        else:
            dests.append(None)
        kinds.append(kind)
    seen = {}

    def on_image(index, desc, rows):
        ext = dests[index] is not None and rows.ctypes.data == dests[index].ctypes.data
        row = desc.width * desc.bytes_per_pixel
        seen[index] = (ext, np.array_equal(rows[:, :row], want[index]))

    with Options(engine, scale_max_side=STREAM_S):
        hb.decode_stream(engine, [load(n) for n in names], on_image, threads=2, files_per_batch=4, dests=dests)
    for k, kind in enumerate(kinds):
        ext, ok = seen[k]
        assert ok, (names[k], kind)
        assert ext == (kind in ("exact", "wide")), (names[k], kind)
        if ext:
            h, row = want[k].shape
            assert np.array_equal(dests[k][:, :row], want[k])


@pytest.mark.gpu
def test_gpu_stream_scaled_isolates_a_damaged_file(engine):
    names = NAMES[:7]
    want = _want(_full_rgb(engine, names), STREAM_S)
    files = [load(n) for n in names]
    files.insert(3, files[3][:len(files[3]) // 3])          # truncated in the middle of the list
    for per_batch in (1, 3, 7):
        got = {}
        with Options(engine, scale_max_side=STREAM_S):
            st = hb.decode_stream(engine, files, lambda i, d, r: got.__setitem__(i, np.array(r[:, :d.width * d.bytes_per_pixel])),
                                  files_per_batch=per_batch, isolate_errors=True)
        assert [k for k, v in enumerate(st["file_status"]) if v != 0] == [3], (per_batch, st["file_status"])
        assert sorted(got) == [k for k in range(len(files)) if k != 3]
        for k, w in enumerate(want):
            assert np.array_equal(got[k if k < 3 else k + 1], w), (per_batch, names[k])
        assert st["bytes_d2h"] == sum(w.size for w in want)


# ---- geometry ------------------------------------------------------------------------------------------------------
def _place(b, name):
    hf = hb.HeifFile(load(name))
    canvas, (matrix, primaries, full_range), has_alpha, bd, cf = api._place_image(hf, b, hf.primary_id)
    return canvas, (matrix, primaries, full_range, cf, bd, has_alpha)


@pytest.mark.gpu
@pytest.mark.parametrize("name,key", [("single_420_8_novui", "rgb"), ("alpha_422_10", "rrggbbaa_le"), ("single_444_8_bt2020", "rgba"),
                                      ("single_mono_12_full", "rrggbb_be")])
def test_gpu_batch_output_sizes_in_one_batch(engine, name, key):
    """Delivered widths 1..33 (K5's 8-pixel units and their tails), upscales and non-integer ratios: all canvases of ONE
    batch, whose output blocks lie back to back, so that a store outside a canvas' block corrupts its neighbour. The first
    canvas is full size and carries the golden MD5; every other one is compared in full against its restatement."""
    fmt = FORMATS[key]
    b = engine.batch()
    try:
        full_c, (m, prim, fr, cf, bd, alpha) = _place(b, name)
        W, H = META[name]["width"], META[name]["height"]
        sizes = [(w, 1 + (w * 7) % H) for w in range(1, 34)]
        sizes += [(2 * W + 3, 3 * H - 1), (W + 1, H - 1), (W * 5 // 3, max(1, H * 2 // 7)), (W - 1, H + 1), (1, 3 * H), (3 * W, 1)]
        canvases = []
        for w, h in sizes:
            c, _ = _place(b, name)
            b.set_output_size(c, w, h)
            canvases.append(c)
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        params = hb.csc_select(m, prim, fr, cf, bd, alpha, fmt)
        allc = [full_c] + canvases
        api.check(b._L, b._L.hc_batch_convert_many(b._h, len(allc), (C.c_int * len(allc))(*allc), (CscParams * len(allc))(*[params] * len(allc))),
                  "convert_many")
        full = b.read_rgb(full_c, fmt)
        assert md5(full.tobytes()) == FMETA[name][key + "_md5"]
        bad = [(w, h) for c, (w, h) in zip(canvases, sizes) if not np.array_equal(b.read_rgb(c, fmt), scale_rows(full, BPP[fmt], w, h))]
        assert not bad, bad
        # the planes stay full size
        assert b.read_plane(canvases[0], 0).shape == (H, W)
    finally:
        b.close()


def _synthetic(w, h):
    from tools import heif_writer, hevcenc
    s = hevcenc.encode(hevcenc.synth_image(w, h, 1, 8, seed=w + h), chroma_format=1, bit_depth=8, seed=5)
    return heif_writer.single_image(s, w, h, 1, 8)


@pytest.mark.gpu
def test_gpu_one_pixel_short_sides(engine):
    """8 x 200 and 200 x 8 images at S = 20: the short side (0.8) rounds to 0 and becomes 1; through the job and the stream"""
    files = [_synthetic(8, 200), _synthetic(200, 8)]
    for fmt in (hb.OUT_RGB, hb.OUT_RRGGBBAA_LE):
        _, full = run_job(engine, files, fmt)
        assert all(np.array_equal(f, ho.decode_rgb(data, fmt)) for f, data in zip(full, files))
        d, rows = run_job(engine, files, fmt, scale_max_side=20)
        assert [(x.width, x.height) for x in d] == [(1, 20), (20, 1)]
        assert not check_scaled(full, d, rows, fmt, 20, ["8x200", "200x8"])
    got = {}
    with Options(engine, scale_max_side=20):
        hb.decode_stream(engine, files, lambda i, d, r: got.__setitem__(i, ((d.width, d.height), np.array(r[:, :d.width * 3]))), files_per_batch=1)
    _, full = run_job(engine, files, hb.OUT_RGB)
    assert got[0][0] == (1, 20) and np.array_equal(got[0][1], scale_rows(full[0], 3, 1, 20))
    assert got[1][0] == (20, 1) and np.array_equal(got[1][1], scale_rows(full[1], 3, 20, 1))


@pytest.mark.gpu
def test_gpu_tall_flip_and_alpha_link_scaled(engine):
    """The 8 x 2,100,000 flip_y canvas with an alpha plane linked from 8 x 700,001 (test_geometry_extremes), delivered as
    13 x 1,999,999 RGBA: y * H reaches 4.2e12, past 32-bit products"""
    from test_geometry_extremes import PASS_DIHEDRAL, add_pass
    from tools import hevcenc
    import oracle_lib
    stream = hevcenc.encode(hevcenc.synth_image(8, 4096, 0, 8, seed=15), chroma_format=0, bit_depth=8)
    rec = hb.parse_picture(stream)
    tile = oracle_lib.reconstruct(rec)[0][0]
    H, HA, w, h = 2100000, 700001, 13, 1999999
    b = engine.batch()
    try:
        c = b.add_canvas(8, H, 0, 8, True)
        a = b.add_canvas(8, HA, 0, 8)
        for y in range(0, H, 4096):
            b.add_picture(rec, c, 0, y)
        for y in range(0, HA, 4096):
            b.add_picture(rec, a, 0, y)
        add_pass(b, c, PASS_DIHEDRAL, (0, 0, 1))
        api.check(b._L, b._L.hc_batch_link_alpha(b._h, c, a), "link_alpha")
        b.set_output_size(c, w, h)
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        b.convert(c, hb.csc_select(2, 2, 1, 0, 8, True, hb.OUT_RGBA))
        stacked = np.tile(tile, ((H + 4095) // 4096, 1))
        y_full = ho.dihedral(stacked[:H], 0, 0, 1)
        a_full = ho.scale_nearest(stacked[:HA], 8, H)
        full = np.stack([y_full, y_full, y_full, a_full], axis=2).astype(np.uint8)      # Op_mono_to_RGB24_32 with alpha
        want = ho.scale_nearest(full, w, h).reshape(h, w * 4)
        got = b.read_rgb(c, hb.OUT_RGBA)
        n = int((got != want).sum())
        assert n == 0, "13 x 1999999 from 8 x 2100000: %d bytes differ, first at %s" % (n, np.argwhere(got != want)[0])
    finally:
        b.close()


@pytest.mark.gpu
def test_gpu_tall_overlay_scaled(engine):
    """The 8 x 530,000 overlay (test_geometry_extremes) delivered as 11 x 600,001: two of K7's bands of delivered rows"""
    from test_geometry_extremes import BACKGROUND, _child_rgb, picture
    rec, planes = picture(3, 8, seed=14)
    W, H, w, h = 8, 530000, 11, 600001
    b = engine.batch()
    try:
        c = b.add_canvas(200, 120, 3, 8)
        b.add_picture(rec, c)
        conv = (1, 1, 0)
        rgb = _child_rgb(planes, conv)
        o = b._L.hc_batch_add_overlay_canvas(b._h, W, H, (C.c_uint16 * 4)(*BACKGROUND))
        assert o >= 0
        offs = [(0, 0), (3, 300001), (1, H - 50)]
        params = hb.csc_select(conv[0], conv[1], conv[2], 3, 8, False, hb.OUT_RGB)
        for dx, dy in offs:
            api.check(b._L, b._L.hc_batch_overlay_add_child(b._h, o, c, dx, dy, C.byref(params)), "overlay_add_child")
        api.check(b._L, b._L.hc_batch_set_canvas_output_size(b._h, o, w, h), "set_canvas_output_size")
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        api.check(b._L, b._L.hc_batch_convert_many(b._h, 1, (C.c_int * 1)(o), (CscParams * 1)(hb.csc_select(2, 2, 1, 3, 8, False, hb.OUT_RGB))),
                  "hc_batch_convert_many")
        want = scale_rows(ho.compose_overlay([rgb] * 3, [None] * 3, offs, BACKGROUND, W, H, hb.OUT_RGB), 3, w, h)
        got = np.empty_like(want)
        api.check(b._L, b._L.hc_batch_read_rgb(b._h, o, got.ctypes.data, got.strides[0]), "read_rgb")
        n = int((got != want).sum())
        assert n == 0, "overlay 11 x 600001 from 8 x 530000: %d bytes differ, first at %s" % (n, np.argwhere(got != want)[0])
    finally:
        b.close()


# ---- refusals and defaults -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_scaled_refusals_and_defaults(engine):
    L = engine._L
    name = "grid_640x384_t128_wpp"
    data = load(name)
    assert L.hc_engine_set_option(engine._h, b"scale_max_side", -1) == ERR_ARGUMENT
    assert engine.get_option("scale_max_side") == 0
    shared = L.hc_shared_image_create(engine._h, 97, 58, 3)
    assert shared
    try:
        with Options(engine, scale_max_side=97):
            assert engine.get_option("scale_max_side") == 97
            # HC_OUT_YCBCR: the job fails at creation, the stream fails the call (with error isolation too)
            with pytest.raises(hb.HeifCudaError, match="HC_OUT_YCBCR"):
                hb.HeicJob(engine, [data], threads=1, out_format=hb.OUT_YCBCR)
            for isolate in (False, True):
                with pytest.raises(hb.HeifCudaError, match=r"\(-6\)"):
                    hb.decode_stream(engine, [data, data], None, files_per_batch=1, out_format=hb.OUT_YCBCR, isolate_errors=isolate)
            # band jobs
            first, full = C.c_int(), C.c_int()
            assert not L.hc_heic_job_create_band(engine._h, data, len(data), 0, 1, 0, 1, C.byref(first), C.byref(full))
            # shared-image targets and plane reads of a scaled image
            job = hb.HeicJob(engine, [data], threads=1)
            try:
                d = job.descs[0]
                assert (d.width, d.height) == fit(640, 384, 97) == (97, 58)
                assert L.hc_heic_job_set_rgb_target(job._h, 0, shared, 0) == ERR_UNSUPPORTED
                job.upload()
                job.run()
                out = np.zeros((384, 640), np.uint8)
                assert L.hc_heic_job_read_plane(job._h, 0, 0, out.ctypes.data, out.strides[0]) == ERR_UNSUPPORTED
            finally:
                job.close()
        # an image whose longer side equals S is not scaled: its golden MD5 and its planes stay available
        small = "single_420_8_novui"
        W, H = META[small]["width"], META[small]["height"]
        with Options(engine, scale_max_side=max(W, H)):
            job = hb.HeicJob(engine, [load(small)], threads=1)
        try:
            assert (job.descs[0].width, job.descs[0].height) == (W, H)
            job.upload()
            job.run()
            assert md5(job.read_rgb(0).tobytes()) == META[small]["rgb_md5"]
            assert job.read_plane(0, 0).shape == (H, W)
        finally:
            job.close()
        # batch level: bad sizes, external targets either way round, HC_OUT_YCBCR of a scaled canvas
        b = engine.batch()
        try:
            c, (m, prim, fr, cf, bd, alpha) = _place(b, small)
            c2, _ = _place(b, small)
            for w, h in ((0, 5), (5, 0), (-1, 5)):
                assert L.hc_batch_set_canvas_output_size(b._h, c, w, h) == ERR_ARGUMENT
            assert L.hc_batch_set_canvas_output_size(b._h, 99, 5, 5) == ERR_ARGUMENT
            ptr = L.hc_shared_image_device_ptr(shared)
            stride = L.hc_shared_image_stride(shared)
            assert L.hc_batch_set_rgb_target(b._h, c2, ptr, stride) == 0
            assert L.hc_batch_set_canvas_output_size(b._h, c2, 5, 5) == ERR_UNSUPPORTED
            assert L.hc_batch_set_rgb_target(b._h, c2, None, 0) == 0
            b.set_output_size(c, 5, 5)
            assert L.hc_batch_set_rgb_target(b._h, c, ptr, stride) == ERR_UNSUPPORTED
            b.upload()
            b.reconstruct(hb.STAGE_ALL)
            ycbcr = hb.csc_select(m, prim, fr, cf, bd, alpha, hb.OUT_YCBCR)
            assert L.hc_batch_convert(b._h, c, C.byref(ycbcr)) == ERR_UNSUPPORTED
            assert L.hc_batch_convert_many(b._h, 1, (C.c_int * 1)(c), (CscParams * 1)(ycbcr)) == ERR_UNSUPPORTED
        finally:
            b.close()
    finally:
        L.hc_shared_image_destroy(shared)
    # S back to 0: the golden MD5s again
    _, rows = run_job(engine, [data, load("alpha_420_8")], hb.OUT_RGB)
    assert [md5(r.tobytes()) for r in rows] == [FMETA[name]["rgb_md5"], FMETA["alpha_420_8"]["rgb_md5"]]
