"""Everything after reconstruction that decides where a sample ends up, against the restatement at the limits of its
geometry: K4's crop + paste + limited->full rescale, K6 (dihedral maps), the crop pass, the alpha rescale, K7 (overlay)
and K8 (planar packing).

The fixtures reach these stages only at a handful of sizes, with every picture at (0, 0) of its own canvas. Here pictures
(fixture records mutated by record_mutation.mutate, so that pasted samples reach 0 and the maximum) are placed anywhere
on canvases cut at every residue, passes and alpha links are chained, and the results are compared with the plane-level
functions of heic_oracle (paste, dihedral, crop_planes, scale_nearest, compose_overlay), which
test_plane_helpers_reproduce_reference and the MD5 tests of test_heic_files / test_overlay pin to the reference.

Uncovered canvas memory is undefined (the plane pool is reused), so every comparison covers only what the restatement
says was written."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import heic_oracle as ho
import heif_b200 as hb
from heif_b200 import api
import oracle_lib
import record_mutation as rm
from conftest import ROOT
from heif_b200._lib import CscParams, ImageDesc

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GEN_DIR = os.path.join(ROOT, "tests", "golden", "generated")
HEIC_DIR = os.path.join(ROOT, "tests", "golden", "heic")
ROLE_LUMA = 2
PASS_DIHEDRAL, PASS_CROP = 0, 1
# one 200 x 120 (264 x 200 for 4:2:2 12 bit) fixture picture per (chroma format, bit depth); None: encoded at test time
PICTURES = {(0, 8): "mono_8", (0, 10): None, (0, 12): "mono_12", (1, 8): "qp51", (1, 10): "c420_10", (1, 12): "c420_12",
            (2, 8): "c422_8", (2, 10): "scaling_custom_10", (2, 12): "c422_12", (3, 8): "c444_8", (3, 10): "c444_10", (3, 12): None}
MAPS = [(s, fx, fy) for s in (0, 1) for fx in (0, 1) for fy in (0, 1)]
K6_EDGES = (1, 31, 32, 33, 63, 64, 65)


# ---------------------------------------------------------------------------------------------------------------- CPU
def _fuse(ops):
    """A run of irot / imir ops as the single dihedral map hc_batch_set_canvas_transform takes: found by applying the ops
    to a 2 x 3 array of distinct values and asking which of the eight maps gives the same array."""
    probe = np.arange(6).reshape(2, 3)
    want = probe
    for op in ops:
        want = ho.dihedral(want, *ho._DIHEDRAL[op])
    for m in MAPS:
        got = ho.dihedral(probe, *m)
        if got.shape == want.shape and np.array_equal(got, want):
            return m
    raise AssertionError(ops)


def _as_passes(planes, info):
    """irot / imir / clap as the engine runs them: consecutive rotations and mirrors fused into one dihedral pass, each clap a
    crop pass on the image as it is at that point"""
    run, nclap = [], 0
    for k in range(info.n_transforms + 1):
        op = info.transforms[k] if k < info.n_transforms else None
        if op in ho._DIHEDRAL:
            run.append(op)
            continue
        if run:
            m = _fuse(run)
            planes = [ho.dihedral(p, *m) for p in planes]
            run = []
        if op == 6:
            H, W = planes[0].shape
            planes = ho.crop_planes(planes, ho.clap_window(list(info.claps[nclap]), W, H))
            nclap += 1
    return planes


def _xform_fixtures():
    import json
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "heic.json")))
    out = []
    for name in sorted(meta):
        hf = hb.HeifFile(open(os.path.join(HEIC_DIR, name + ".heic"), "rb").read(), host_only=True)
        info = hf.image_info(hf.primary_id)
        ainfo = hf.image_info(info.alpha_id) if info.alpha_id else None
        if info.n_transforms or (ainfo and (ainfo.n_transforms or (ainfo.width, ainfo.height) != (info.width, info.height))):
            out.append((name, meta[name]["planes_md5"]))
    return out


def test_plane_helpers_reproduce_reference():
    """dihedral / crop_planes / scale_nearest on their own terms (fused dihedral passes, crop passes, the alpha rescale)
    applied to the oracle's planes of every fixture with irot / imir / clap or an alpha image of another size reproduce the
    reference's planes."""
    import hashlib
    cases = _xform_fixtures()
    assert len(cases) >= 20
    for name, want in cases:
        data = open(os.path.join(HEIC_DIR, name + ".heic"), "rb").read()
        planes, alpha, _, bd, _ = ho.decode_planes(data, transform=_as_passes)
        dt = np.uint8 if bd == 8 else np.dtype("<u2")
        got = hashlib.md5(b"".join(p.astype(dt).tobytes() for p in planes + ([alpha] if alpha is not None else []))).hexdigest()
        assert got == want, name


def test_fused_maps_are_the_engine_maps():
    """The eight maps close under composition, and a quarter turn is the map the engine's header documents."""
    a = np.arange(12).reshape(3, 4)
    assert np.array_equal(ho.dihedral(a, *ho._DIHEDRAL[1]), np.rot90(a, 1))
    assert np.array_equal(ho.dihedral(a, *ho._DIHEDRAL[3]), np.rot90(a, 3))
    for m1 in MAPS:
        for m2 in MAPS:
            ho_m = ho.dihedral(ho.dihedral(a, *m1), *m2)
            assert any(np.array_equal(ho_m, ho.dihedral(a, *m)) for m in MAPS)


def test_restated_rescale_clips_deep_tiles_to_255():
    """the reference's rescale keeps 8-bit output whatever the tile depth: 10 / 12-bit tiles are clipped to 255"""
    for bd in (8, 10, 12):
        p = np.array([[0, 16 << (bd - 8), 235, (1 << bd) - 1]], np.uint16)
        r = ho._rescale_limited(p, False, bd)
        assert r[0, 0] == 0 and r[0, 1] == 0 and r.max() <= 255
        assert (r[0, 3] == 255) and (bd > 8 or r[0, 2] == 255)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    yield e
    e.close()


_cache = {}


def picture(cf, bd, seed=1, crop=None):
    """(records, oracle planes) of the (cf, bd) picture, mutated with every family; crop = (x, y, w, h) edits the
    conformance window first"""
    name = PICTURES[(cf, bd)]
    if name is None:
        key = ("enc", cf, bd)
        if key not in _cache:
            from tools import hevcenc
            _cache[key] = hevcenc.encode(hevcenc.synth_image(200, 120, cf, bd, seed=cf * 16 + bd), chroma_format=cf, bit_depth=bd)
        rec = hb.parse_picture(_cache[key])
    else:
        rec = hb.parse_picture(open(os.path.join(GEN_DIR, name + ".hevc"), "rb").read())
    rm.mutate(rec, "all", seed)
    if crop is not None:
        p = rec.pic
        p.crop_x, p.crop_y, p.crop_w, p.crop_h = crop
    return rec, oracle_lib.reconstruct(rec)[0]


def dtype_of(bd):
    return np.uint8 if bd == 8 else np.uint16


def read_plane(b, canvas, plane, shape, bd):
    """one plane of a canvas' output view (after its passes) through the C ABI"""
    out = np.empty(shape, dtype_of(bd))
    api.check(b._L, b._L.hc_batch_read_plane(b._h, canvas, plane, out.ctypes.data, out.strides[0]), "read_plane")
    return out


def add_pass(b, canvas, kind, args):
    a = list(args) + [0] * (4 - len(args))
    api.check(b._L, b._L.hc_batch_add_canvas_pass(b._h, canvas, kind, *a), "add_canvas_pass")


def first_diff(got, want):
    bad = np.argwhere(got != want)
    return len(bad), (tuple(int(v) for v in bad[0]) if len(bad) else None)


def check_plane(got, want, what, plane, mask=None):
    assert got.shape == want.shape, "%s plane %d: shape %s, want %s" % (what, plane, got.shape, want.shape)
    g, w = got.astype(np.int64), want.astype(np.int64)
    if mask is not None:
        g, w = np.where(mask, g, 0), np.where(mask, w, 0)
    n, at = first_diff(g, w)
    assert n == 0, "%s plane %d: %d samples differ, first at (y,x)=%s: got %d want %d" % (
        what, plane, n, at, g[at], w[at])


# ---- paste / rescale ----------------------------------------------------------------------------------------------
def _tile_crop(cf, r):
    """conformance window of a tile of width 40 + r, height 24 + r, starting at a nonzero multiple of SubW / SubH"""
    sw, sh = ho.subsampling(cf)
    x, y = sw * (1 + r // 2), sh * (1 + r // 4)
    return x, y, 40 + r, 24 + r


@pytest.mark.gpu
@pytest.mark.parametrize("cf,bd", sorted(PICTURES))
def test_gpu_paste_and_rescale_at_every_cut(engine, cf, bd):
    """Grids of one tile size (width 40 + r, r = 0, 2, 4, 6: the store8 and the per-sample path of K4) on canvases that cut
    the last tile column and row at 1..7 samples; rescale off / on / mixed per tile; 1 x N and N x 1 grids; a canvas
    smaller than its one tile; a picture at an odd position; the alpha role (plain) and the luma role (rescaled)."""
    b = engine.batch()
    cases = []   # (label, canvas, want planes, written masks, has alpha)
    try:
        abd = 8 if bd == 8 else 12
        for r in (0, 2, 4, 6):
            crop = _tile_crop(cf, r)
            rec, tile = picture(cf, bd, seed=1 + r, crop=crop)
            arec, atile = picture(0, abd, seed=11 + r, crop=crop)
            tw, th = crop[2], crop[3]

            def grid(W, H, cols, rows, rescale_of, label, alpha=False, luma=False):
                ccf = 0 if luma else cf
                c = b.add_canvas(W, H, ccf, bd, alpha)
                want = ho.new_canvas(W, H, ccf)
                mask = ho.new_canvas(W, H, ccf, bool)
                if alpha:
                    want.append(np.zeros((H, W), np.uint16))
                    mask.append(np.zeros((H, W), bool))
                for j in range(rows):
                    for i in range(cols):
                        x, y, res = i * tw, j * th, rescale_of(i + j * cols)
                        if x >= W or y >= H:
                            continue
                        if luma:
                            b.add_picture(rec, c, x, y, ROLE_LUMA, res)
                            ho.paste(want, tile[:1], x, y, 0, res, bd)
                            ho.paste(mask, [np.ones_like(tile[0], bool)], x, y, 0, False, bd)
                            continue
                        b.add_picture(rec, c, x, y, api.ROLE_COLOUR, res)
                        ho.paste(want, tile, x, y, cf, res, bd)
                        ho.paste(mask, [np.ones_like(p, bool) for p in tile], x, y, cf, False, bd)
                        if alpha:
                            b.add_picture(arec, c, x, y, api.ROLE_ALPHA, False)
                            ho.paste(want[-1:], atile[:1], x, y, 0, False, abd)
                            ho.paste(mask[-1:], [np.ones_like(atile[0], bool)], x, y, 0, False, abd)
                cases.append(("%s tile=%dx%d crop=%s canvas=%dx%d" % (label, tw, th, crop[:2], W, H), c, want, mask, alpha))

            for k in range(1, 8):
                mode = k % 3
                grid(2 * tw + k, th + k, 3, 2, lambda i, m=mode: m == 1 or (m == 2 and i % 2 == 0),
                     "grid 3x2 cut=%d rescale=%s" % (k, ("off", "on", "mixed")[mode]))
            grid(tw - 3, 3 * th + 1, 1, 4, lambda i: i % 2 == 1, "grid 1x4")
            grid(3 * tw + 1, th - 1, 4, 1, lambda i: i % 2 == 0, "grid 4x1")
            grid(tw - 5, th - 3, 1, 1, lambda i: True, "one tile larger than its canvas")
            grid(2 * tw + 3, th + 5, 3, 2, lambda i: False, "alpha role", alpha=True)
            grid(2 * tw + 5, th + 2, 3, 2, lambda i: i != 1, "luma role rescaled", luma=True)
            # a picture at an odd position, not covering its canvas
            W, H = tw + 9, th + 7
            c = b.add_canvas(W, H, cf, bd)
            b.add_picture(rec, c, 3, 5, api.ROLE_COLOUR, r == 2)
            want, mask = ho.new_canvas(W, H, cf), ho.new_canvas(W, H, cf, bool)
            ho.paste(want, tile, 3, 5, cf, r == 2, bd)
            ho.paste(mask, [np.ones_like(p, bool) for p in tile], 3, 5, cf, False, bd)
            cases.append(("picture at (3, 5) tile=%dx%d canvas=%dx%d" % (tw, th, W, H), c, want, mask, False))
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        for label, c, want, mask, alpha in cases:
            what = "cf=%d bd=%d %s" % (cf, bd, label)
            for k, (w, m) in enumerate(zip(want, mask)):
                plane = 3 if alpha and k == len(want) - 1 else k
                check_plane(read_plane(b, c, plane, w.shape, bd), w, what, plane, m)
    finally:
        b.close()


# ---- passes: K6 and the crop pass ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bd", [8, 12])
def test_gpu_dihedral_maps_at_k6_tile_edges(engine, bd):
    """Planes of 1, 31, 32, 33, 63, 64 and 65 samples in each dimension (cut by a crop pass at an odd position) through all
    eight dihedral maps, 8- and 16-bit samples."""
    rec, planes = picture(0, bd, seed=3)
    b = engine.batch()
    cases = []
    try:
        for w in K6_EDGES:
            for h in K6_EDGES:
                win = (3, 5, 3 + w - 1, 5 + h - 1)
                for m in MAPS:
                    c = b.add_canvas(200, 120, 0, bd)
                    b.add_picture(rec, c)
                    add_pass(b, c, PASS_CROP, win)
                    add_pass(b, c, PASS_DIHEDRAL, m)
                    cases.append((w, h, m, c, ho.dihedral(ho.crop_planes(planes, win)[0], *m)))
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        for w, h, m, c, want in cases:
            check_plane(read_plane(b, c, 0, want.shape, bd), want, "bd=%d plane %dx%d map(swap,fx,fy)=%s" % (bd, w, h, m), 0)
    finally:
        b.close()


def _window(kind, W, H):
    if kind == "full":
        return 0, 0, W - 1, H - 1
    if kind == "1x1":
        return W // 2, H // 3, W // 2, H // 3
    if kind == "even":
        l, t = min(2, W - 1) & ~1, min(2, H - 1) & ~1
        return l, t, max(l, W - 4), max(t, H - 3)
    l, t = min(3, W - 1), min(1, H - 1)                  # odd
    return l, t, max(l, W - 2), max(t, H - 4)


WINDOWS = ("even", "odd", "1x1", "full")


@pytest.mark.gpu
@pytest.mark.parametrize("cf,bd", [(cf, bd) for cf in (0, 1, 2, 3) for bd in (8, 10)])
def test_gpu_pass_chains(engine, cf, bd):
    """dihedral -> crop -> dihedral -> crop, every map first, crop windows at even and odd positions, 1 x 1 and the full
    image. 4:2:2 quarter turns (which hc_heic_job refuses) included: planes only."""
    rec, planes = picture(cf, bd, seed=5)
    b = engine.batch()
    cases = []
    try:
        for i, m1 in enumerate(MAPS):
            for j in range(2):
                m2 = MAPS[(3 * i + 5 * j + 1) % 8]
                k1, k2 = WINDOWS[(i + j) % 4], WINDOWS[(i + 2 * j + 1) % 4]
                c = b.add_canvas(200, 120, cf, bd)
                b.add_picture(rec, c)
                want = [ho.dihedral(p, *m1) for p in planes]
                add_pass(b, c, PASS_DIHEDRAL, m1)
                w1 = _window(k1, want[0].shape[1], want[0].shape[0])
                want = ho.crop_planes(want, w1)
                add_pass(b, c, PASS_CROP, w1)
                want = [ho.dihedral(p, *m2) for p in want]
                add_pass(b, c, PASS_DIHEDRAL, m2)
                w2 = _window(k2, want[0].shape[1], want[0].shape[0])
                want = ho.crop_planes(want, w2)
                add_pass(b, c, PASS_CROP, w2)
                cases.append(("map%s crop%s map%s crop%s" % (m1, w1, m2, w2), c, want))
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        for label, c, want in cases:
            for k, w in enumerate(want):
                check_plane(read_plane(b, c, k, w.shape, bd), w, "cf=%d bd=%d %s" % (cf, bd, label), k)
    finally:
        b.close()


# ---- alpha link ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bd", [8, 12])
def test_gpu_alpha_link_scales(engine, bd):
    """An alpha canvas rescaled into a colour canvas by nearest neighbour: up and down by non-integer ratios, 1 x 1 -> large,
    large -> 1 x 1, 1 x N <-> N x 1, both canvases with passes of their own. Planes, and one K5 conversion with alpha."""
    rec, planes = picture(1, bd, seed=7)
    arec, aplanes = picture(0, bd, seed=8)
    # (colour passes, alpha passes): crop = (1, window), dihedral = (0, map)
    cases_def = [
        ([], [(1, (4, 3, 80, 55))]),                                   # 200 x 120 <- 77 x 53
        ([(1, (2, 6, 62, 42))], []),                                   # 61 x 37 <- 200 x 120
        ([(1, (0, 0, 149, 99))], [(1, (9, 9, 9, 9))]),                 # 1 x 1 -> 150 x 100
        ([(1, (8, 5, 8, 5))], []),                                     # 200 x 120 -> 1 x 1
        ([(1, (6, 0, 6, 99))], [(1, (0, 7, 99, 7))]),                  # N x 1 -> 1 x N
        ([(1, (0, 7, 99, 7))], [(1, (6, 0, 6, 99))]),                  # 1 x N -> N x 1
        ([(0, (1, 1, 0)), (1, (3, 4, 100, 180))], [(1, (5, 1, 150, 90)), (0, (0, 1, 1))]),
    ]
    b = engine.batch()
    cases = []
    try:
        for cp, ap in cases_def:
            c = b.add_canvas(200, 120, 1, bd, True)
            b.add_picture(rec, c)
            a = b.add_canvas(200, 120, 0, bd)
            b.add_picture(arec, a)
            want, alpha = list(planes), list(aplanes)
            for kind, args in cp:
                add_pass(b, c, kind, args)
                want = [ho.dihedral(p, *args) for p in want] if kind == 0 else ho.crop_planes(want, args)
            for kind, args in ap:
                add_pass(b, a, kind, args)
                alpha = [ho.dihedral(p, *args) for p in alpha] if kind == 0 else ho.crop_planes(alpha, args)
            api.check(b._L, b._L.hc_batch_link_alpha(b._h, c, a), "link_alpha")
            want.append(ho.scale_nearest(alpha[0], want[0].shape[1], want[0].shape[0]))
            cases.append(("colour passes %s alpha passes %s" % (cp, ap), c, want))
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        for label, c, want in cases:
            for k, w in enumerate(want):
                check_plane(read_plane(b, c, 3 if k == 3 else k, w.shape, bd), w, "bd=%d %s" % (bd, label), 3 if k == 3 else k)
        label, c, want = cases[-1]
        p = rec.pic
        fmt = hb.OUT_RGBA if bd == 8 else hb.OUT_RRGGBBAA_LE
        b.convert(c, hb.csc_select(p.matrix_coeffs, p.colour_primaries, p.full_range, 1, bd, True, fmt))
        h, w = want[0].shape
        got = np.empty((h, w * api.OUT_BYTES_PER_PIXEL[fmt]), np.uint8)
        api.check(b._L, b._L.hc_batch_read_rgb(b._h, c, got.ctypes.data, got.strides[0]), "read_rgb")
        exp = ho.csc(want[:3], 1, bd, p.matrix_coeffs, p.full_range, fmt, want[3], p.colour_primaries)
        n, at = first_diff(got, exp)
        assert n == 0, "bd=%d %s K5 with alpha: %d bytes differ, first at %s" % (bd, label, n, at)
    finally:
        b.close()


# ---- K8 ------------------------------------------------------------------------------------------------------------
K8_WIDTHS = list(range(1, 34)) + [250, 251, 252, 253, 254, 255, 256]


@pytest.mark.gpu
@pytest.mark.parametrize("sixteen", [False, True])
def test_gpu_planar_packing_of_every_width(engine, sixteen):
    """HC_OUT_YCBCR of canvases 1..33 and 250..256 samples wide, every chroma format, with and without alpha, after a crop
    (and for odd widths a mirror) pass, all in one hc_batch_convert_many (more than 24 canvases: K8 flushes mid-call).
    Expected bytes: the restated planes packed as hc_image_plane_layout says."""
    b = engine.batch()
    cases = []
    try:
        for cf in (0, 1, 2, 3):
            bd = 8 if not sixteen else (12 if cf != 2 else 10)
            rec, planes = picture(cf, bd, seed=9)
            abd = 8 if bd == 8 else 12
            arec, aplanes = picture(0, abd, seed=10)
            full = ho.new_canvas(400, 120, cf)
            for x in (0, 200):
                ho.paste(full, planes, x, 0, cf, False, bd)
            afull = ho.new_canvas(400, 120, 0)
            for x in (0, 200):
                ho.paste(afull, aplanes[:1], x, 0, 0, False, abd)
            for w in K8_WIDTHS:
                for alpha in (False, True):
                    h = 3 + (w * 7 + alpha) % 6
                    c = b.add_canvas(400, 120, cf, bd, alpha)
                    for x in (0, 200):
                        b.add_picture(rec, c, x, 0)
                        if alpha:
                            b.add_picture(arec, c, x, 0, api.ROLE_ALPHA)
                    want = list(full) + (afull if alpha else [])
                    if w % 2:
                        add_pass(b, c, PASS_DIHEDRAL, (0, 1, w % 4 == 1))
                        want = [ho.dihedral(p, 0, 1, w % 4 == 1) for p in want]
                    win = (2 * (w % 5), 2 * (w % 3), 2 * (w % 5) + w - 1, 2 * (w % 3) + h - 1)
                    add_pass(b, c, PASS_CROP, win)
                    want = ho.crop_planes(want, win)
                    cases.append(("cf=%d bd=%d %dx%d alpha=%s window=%s" % (cf, bd, w, h, alpha, win), c, want, cf, bd, alpha))
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        params = [hb.csc_select(2, 2, 1, cf, bd, alpha, hb.OUT_YCBCR) for _, _, _, cf, bd, alpha in cases]
        n = len(cases)
        api.check(b._L, b._L.hc_batch_convert_many(b._h, n, (C.c_int * n)(*[c[1] for c in cases]), (CscParams * n)(*params)),
                  "hc_batch_convert_many")
        for label, c, want, cf, bd, alpha in cases:
            h, w = want[0].shape
            d = ImageDesc()
            d.width, d.height, d.chroma_format, d.bit_depth, d.has_alpha = w, h, cf, bd, int(alpha)
            d.out_format, d.bytes_per_pixel = hb.OUT_YCBCR, 1 if bd == 8 else 2
            total, _ = hb.plane_layout(d)
            exp = np.frombuffer(b"".join(p.astype(np.uint8 if bd == 8 else "<u2").tobytes() for p in want), np.uint8)
            assert total == exp.size, label
            got = np.empty(total, np.uint8)
            api.check(b._L, b._L.hc_batch_read_rgb(b._h, c, got.ctypes.data, w * d.bytes_per_pixel), "read_rgb")
            nd, at = first_diff(got, exp)
            assert nd == 0, "%s: %d packed bytes differ, first at byte %s" % (label, nd, at)
    finally:
        b.close()


# ---- K7 ------------------------------------------------------------------------------------------------------------
# (matrix, primaries, full_range) of the children: GBR, YCgCo and matrix mode, full and limited range
CHILD_CONVERSIONS = ((0, 1, 1), (0, 1, 0), (8, 1, 1), (8, 1, 0), (1, 1, 1), (1, 1, 0), (6, 1, 0), (9, 9, 1))
BACKGROUND = (0x12ab, 0x80ff, 0xfe01, 0x7777)


def _child(b, rec, planes, arec, aplanes, window, alpha):
    """a 4:4:4 8-bit child canvas cut to `window` by a crop pass; returns (canvas, planes, alpha plane or None)"""
    c = b.add_canvas(200, 120, 3, 8, alpha)
    b.add_picture(rec, c)
    if alpha:
        b.add_picture(arec, c, 0, 0, api.ROLE_ALPHA)
    add_pass(b, c, PASS_CROP, window)
    pl = ho.crop_planes(list(planes) + ([aplanes[0]] if alpha else []), window)
    return c, pl[:3], (pl[3] if alpha else None)


def _child_rgb(planes, conv):
    m, prim, full = conv
    rgba = ho.csc(planes, 3, 8, m, full, hb.OUT_RGBA, None, prim)     # Op_YCbCr_to_RGB<uint8_t>: the general fp32 op
    return rgba.reshape(rgba.shape[0], -1, 4)[:, :, :3]


def _overlay_layouts():
    """(W, H, [(window, alpha, dx, dy)]) of the overlay canvases"""
    W, H = 150, 90
    kids = [((0, 0, 199, 119), False, 0, 0),                            # covers the canvas
            ((10, 10, 49, 39), True, 5, 5),
            ((7, 7, 7, 7), False, 0, 0),                                # 1 x 1
            ((0, 0, 29, 19), False, W - 1, 10),                         # 1 column left
            ((0, 0, 29, 19), True, 20, H - 1),                          # 1 row left
            ((0, 0, 29, 19), False, W, 0),                              # wholly outside: 0 columns left
            ((0, 0, 29, 19), False, 0, H),
            ((3, 5, 70, 60), True, 30, 20)]
    for k in range(8):                                                  # up to 16 overlapping children
        kids.append(((k, 2 * k, 40 + 9 * k, 30 + 5 * k), k % 2 == 1, 11 * k + 3, 7 * k + 1))
    return [(W, H, kids),
            (1, 77, [((0, 0, 9, 99), False, 0, 3), ((5, 5, 5, 5), True, 0, 76), ((0, 0, 0, 9), True, 0, 0)]),
            (77, 1, [((0, 0, 99, 9), True, 2, 0), ((5, 5, 5, 5), False, 76, 0), ((0, 0, 9, 0), False, 0, 0)])]


@pytest.mark.gpu
def test_gpu_overlay_geometry_and_blending(engine):
    """K7: children clipped at the right / bottom edge with 1 and 0 samples left, a 1 x 1 child, children wholly outside,
    16 overlapping children in order, alpha children (mutated alpha: 0, 255 and between), GBR / YCgCo / matrix children in
    full and limited range, background words whose low bytes are dropped, 1 x N and N x 1 canvases, every interleaved
    output format."""
    rec, planes = picture(3, 8, seed=12)
    arec, aplanes = picture(0, 8, seed=13)
    assert aplanes[0].min() == 0 and aplanes[0].max() == 255
    b = engine.batch()
    jobs = []
    try:
        layouts = []
        for W, H, kids in _overlay_layouts():
            children = []
            for k, (win, alpha, dx, dy) in enumerate(kids):
                c, pl, a = _child(b, rec, planes, arec, aplanes, win, alpha)
                conv = CHILD_CONVERSIONS[k % len(CHILD_CONVERSIONS)]
                children.append((c, _child_rgb(pl, conv), a, dx, dy, conv))
            layouts.append((W, H, children))
        for fmt in range(6):
            for W, H, children in layouts:
                o = b._L.hc_batch_add_overlay_canvas(b._h, W, H, (C.c_uint16 * 4)(*BACKGROUND))
                assert o >= 0
                for c, _, _, dx, dy, (m, prim, full) in children:
                    params = hb.csc_select(m, prim, full, 3, 8, False, hb.OUT_RGB)
                    api.check(b._L, b._L.hc_batch_overlay_add_child(b._h, o, c, dx, dy, C.byref(params)), "overlay_add_child")
                want = ho.compose_overlay([ch[1] for ch in children], [ch[2] for ch in children], [ch[3:5] for ch in children],
                                          BACKGROUND, W, H, fmt)
                jobs.append((o, fmt, W, H, want, [ch[3:6] for ch in children]))
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        n = len(jobs)
        params = [hb.csc_select(2, 2, 1, 3, 8, False, j[1]) for j in jobs]
        api.check(b._L, b._L.hc_batch_convert_many(b._h, n, (C.c_int * n)(*[j[0] for j in jobs]), (CscParams * n)(*params)),
                  "hc_batch_convert_many")
        for o, fmt, W, H, want, kids in jobs:
            got = np.empty_like(want)
            api.check(b._L, b._L.hc_batch_read_rgb(b._h, o, got.ctypes.data, got.strides[0]), "read_rgb")
            nd, at = first_diff(got, want)
            assert nd == 0, "overlay %dx%d format %d children (dx, dy, conversion)=%s: %d bytes differ, first at %s" % (
                W, H, fmt, kids, nd, at)
    finally:
        b.close()


# ---- tall images (gridDim.y is limited to 65,535) ------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_overlay_taller_than_the_k7_grid(engine):
    """an overlay canvas of 8 x 530,000 (K7's 8-row blocks: 66,250 of them)"""
    rec, planes = picture(3, 8, seed=14)
    W, H = 8, 530000
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
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        api.check(b._L, b._L.hc_batch_convert_many(b._h, 1, (C.c_int * 1)(o), (CscParams * 1)(hb.csc_select(2, 2, 1, 3, 8, False, hb.OUT_RGB))),
                  "hc_batch_convert_many")
        want = ho.compose_overlay([rgb] * 3, [None] * 3, offs, BACKGROUND, W, H, hb.OUT_RGB)
        got = np.empty_like(want)
        api.check(b._L, b._L.hc_batch_read_rgb(b._h, o, got.ctypes.data, got.strides[0]), "read_rgb")
        nd, at = first_diff(got, want)
        assert nd == 0, "overlay 8 x 530000: %d bytes differ, first at %s" % (nd, at)
    finally:
        b.close()


@pytest.mark.gpu
def test_gpu_passes_taller_than_the_k6_grid(engine):
    """a monochrome 8-bit canvas of 8 x 2,100,000 (K6's 32-row blocks: 65,625 of them) covered by stacked 8 x 4096 pictures,
    with a flip_y pass and an alpha plane linked from an 8 x 700,001 canvas"""
    from tools import hevcenc
    stream = hevcenc.encode(hevcenc.synth_image(8, 4096, 0, 8, seed=15), chroma_format=0, bit_depth=8)
    rec = hb.parse_picture(stream)
    tile = oracle_lib.reconstruct(rec)[0][0]
    H, HA = 2100000, 700001
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
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        stacked = np.tile(tile, ((H + 4095) // 4096, 1))
        want = ho.dihedral(stacked[:H], 0, 0, 1)
        check_plane(read_plane(b, c, 0, want.shape, 8), want, "8 x 2100000 flip_y", 0)
        walpha = ho.scale_nearest(stacked[:HA], 8, H)
        check_plane(read_plane(b, c, 3, walpha.shape, 8), walpha, "8 x 2100000 alpha linked from 8 x 700001", 3)
    finally:
        b.close()


# ---- whole files ---------------------------------------------------------------------------------------------------
def _enc(w, h, cf, bd, seed):
    from tools import hevcenc
    return hevcenc.encode(hevcenc.synth_image(w, h, cf, bd, seed), chroma_format=cf, bit_depth=bd, seed=seed)


def _files():
    """name -> HEIC bytes, generated at test time"""
    from tools import heif_writer as Wr
    files = {}
    for cf, bd in ((2, 10), (3, 12)):
        tiles = [_enc(64, 48, cf, bd, 20 + k) for k in range(6)]
        # 2 x 3 tiles of 64 x 48 cut to 129 x 49: 1-sample remnants in the last column and row
        files["grid_limited_%d_%d" % (cf, bd)] = Wr.grid_image(tiles, 2, 3, 64, 48, 129, 49, cf, bd, tile_nclx=(1, 13, 1, 0))
    files["clap_irot_clap_420"] = Wr.single_image(_enc(64, 48, 1, 8, 30), 64, 48, 1, 8, transforms=(
        Wr.clap(61, 1, 45, 1, -3, 2, 1, 2), Wr.irot(1), Wr.clap(37, 1, 51, 1, 1, 1, -1, 2)))
    # windows at (1, 2) and (5, 6): chroma planes one sample larger than the packed layout of 36 x 50, refused as planes
    files["clap_irot_clap_420_wide_chroma"] = Wr.single_image(_enc(64, 48, 1, 8, 35), 64, 48, 1, 8, transforms=(
        Wr.clap(60, 1, 45, 1, -1, 1, 1, 2), Wr.irot(1), Wr.clap(36, 1, 50, 1, 1, 2, 1, 1)))
    files["clap_irot_clap_444"] = Wr.single_image(_enc(64, 48, 3, 8, 31), 64, 48, 3, 8, transforms=(
        Wr.clap(60, 1, 45, 1, -1, 1, 1, 2), Wr.irot(3), Wr.clap(37, 1, 51, 1, 1, 1, -1, 2)))
    files["alpha_other_size_irot"] = Wr.single_image(_enc(64, 48, 1, 8, 32), 64, 48, 1, 8, alpha_stream=_enc(40, 30, 0, 8, 33),
                                                     alpha_size=(40, 30), transforms=(Wr.irot(1),))
    bld = Wr.HeifBuilder()
    kids = [bld.add_hevc_image(_enc(64, 64, 3, 8, 34 + k), 64, 64, 3, 8, hidden=True) for k in range(2)]
    bld.primary = bld.add_overlay(kids, 16, 600000, [(0, 0), (5, 599970)], background=BACKGROUND)
    files["iovl_16x600000"] = bld.serialize()
    return files


def _want_rgb(data, fmt):
    if _is_overlay(hb.HeifFile(data, host_only=True)):
        import test_overlay
        return test_overlay.compose(data, fmt)
    return ho.decode_rgb(data, fmt)


def _is_overlay(hf):
    try:
        hf.overlay(hf.primary_id)
        return True
    except hb.HeifCudaError:
        return False


@pytest.fixture(scope="module")
def files():
    return _files()


@pytest.mark.gpu
@pytest.mark.parametrize("device_parse", [1, 0])
def test_gpu_files_rgb_job_and_stream(engine, files, device_parse):
    """Limited-range grids at 10 / 12 bit in 4:2:2 / 4:4:4 with 1-sample remnants, clap -> irot -> clap at odd windows, an
    alpha image of another size under a rotation and a 16 x 600,000 overlay: hc_heic_job and hc_heic_decode_stream (host
    shares 0 and 100) against the oracle."""
    names = sorted(files)
    fmt = hb.OUT_RRGGBBAA_LE
    want = {n: _want_rgb(files[n], fmt) for n in names}
    engine.set_option("device_parse", device_parse)
    try:
        job = hb.HeicJob(engine, [files[n] for n in names], threads=2, out_format=fmt)
        job.upload()
        job.run()
        for i, n in enumerate(names):
            got = job.read_rgb(i)
            nd, at = first_diff(got, want[n])
            assert nd == 0, "job device_parse=%d %s: %d bytes differ, first at %s" % (device_parse, n, nd, at)
        job.close()
        for share in (0, 100):
            engine.set_option("host_share_pct", share)
            seen = {}
            hb.decode_stream(engine, [files[n] for n in names],
                             lambda i, d, rows: seen.__setitem__(i, first_diff(rows[:, :d.width * d.bytes_per_pixel], want[names[i]])),
                             threads=2, files_per_batch=3, out_format=fmt)
            assert sorted(seen) == list(range(len(names)))
            bad = {names[i]: v for i, v in seen.items() if v[0]}
            assert not bad, "stream device_parse=%d host_share=%d: (bytes differing, first) %s" % (device_parse, share, bad)
    finally:
        engine.set_option("device_parse", 1)
        engine.set_option("host_share_pct", -1)


@pytest.mark.gpu
def test_gpu_files_planar_job_and_stream(engine, files):
    """The same files as native planes; the 4:2:0 clap chain whose chroma planes outgrow the packed layout is refused as
    today, file by file."""
    names = [n for n in sorted(files) if not n.startswith("iovl")]
    refused = "clap_irot_clap_420_wide_chroma"
    ok = [n for n in names if n != refused]
    with pytest.raises(hb.HeifCudaError, match="clean aperture"):
        hb.HeicJob(engine, [files[refused]], threads=1, out_format=hb.OUT_YCBCR)
    want = {}
    for n in ok:
        planes, alpha, _, bd, _ = ho.decode_planes(files[n])
        want[n] = b"".join(p.astype(np.uint8 if bd == 8 else "<u2").tobytes() for p in planes + ([alpha] if alpha is not None else []))
    job = hb.HeicJob(engine, [files[n] for n in ok], threads=2, out_format=hb.OUT_YCBCR)
    job.upload()
    job.run()
    for i, n in enumerate(ok):
        got = b"".join(np.ascontiguousarray(p).tobytes() for p in job.read_planes(i))
        assert got == want[n], "planar job %s" % n
    job.close()
    for share in (0, 100):
        engine.set_option("host_share_pct", share)
        try:
            seen = {}
            st = hb.decode_stream(engine, [files[n] for n in names],
                                  lambda i, d, p: seen.__setitem__(i, b"".join(np.ascontiguousarray(q).tobytes() for q in p)),
                                  threads=2, files_per_batch=2, out_format=hb.OUT_YCBCR, isolate_errors=True)
        finally:
            engine.set_option("host_share_pct", -1)
        assert [names[i] for i, s in enumerate(st["file_status"]) if s] == [refused], st["file_status"]
        assert {names[i]: v == want[names[i]] for i, v in seen.items()} == {n: True for n in ok}, share
