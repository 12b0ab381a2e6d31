"""Native planar output (HC_OUT_YCBCR): what heif_decode_image(handle, &img, heif_colorspace_undefined,
heif_chroma_undefined, NULL) returns — the decoded Y / Cb / Cr (/ A) planes at their own bit depth, after paste, rescale and
transformations — delivered through the batch, job and stream APIs as one packed block per image (kernel K8).
CPU tests: the packed layout and the identity conversion parameters.
GPU tests: every fixture bit-exact against the reference's planes (tests/golden/heic.json planes_md5) through every API."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import pytest

import heif_b200 as hb
import heic_oracle
from conftest import ROOT
from heif_b200._lib import CscParams, ImageDesc

sys.path.insert(0, ROOT)

DIR = os.path.join(ROOT, "tests", "golden", "heic")
META = json.load(open(os.path.join(ROOT, "tests", "golden", "heic.json")))
NAMES = sorted(META)
YCBCR = 0x100 | hb.OUT_YCBCR     # HC_OUTPUT_FORMAT(HC_OUT_YCBCR)
PREM = {"alpha_prem_420_8"}      # the fixture whose alpha image is referenced by 'prem'


def load(name):
    return open(os.path.join(DIR, name + ".heic"), "rb").read()


def md5(b):
    return hashlib.md5(b).hexdigest()


def desc_of(w, h, cf, bd, alpha):
    d = ImageDesc()
    d.width, d.height, d.chroma_format, d.bit_depth, d.has_alpha = w, h, cf, bd, int(alpha)
    d.out_format, d.bytes_per_pixel = hb.OUT_YCBCR, 1 if bd == 8 else 2
    return d


def packed_md5(planes):
    return md5(b"".join(np.ascontiguousarray(p).tobytes() for p in planes))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("cf", [0, 1, 2, 3])
@pytest.mark.parametrize("size", [(64, 48), (65, 47), (1, 1), (301, 199)])
@pytest.mark.parametrize("bd", [8, 10, 12])
@pytest.mark.parametrize("alpha", [False, True])
def test_plane_layout(cf, size, bd, alpha):
    w, h = size
    ps = 1 if bd == 8 else 2
    cw = {0: 0, 1: (w + 1) // 2, 2: (w + 1) // 2, 3: w}[cf]
    ch = {0: 0, 1: (h + 1) // 2, 2: h, 3: h}[cf]
    want_wh = [(w, h), (cw, ch), (cw, ch), (w, h) if alpha else (0, 0)]
    total, planes = hb.plane_layout(desc_of(w, h, cf, bd, alpha), host_only=True)
    off = 0
    for k, (o, s, pw, ph) in enumerate(planes):
        assert (pw, ph) == want_wh[k], k
        assert s == pw * ps and o == off, k
        off += s * ph
    assert total == off == (w * h * (2 if alpha else 1) + 2 * cw * ch) * ps


def test_plane_layout_is_zero_for_interleaved_descs():
    d = desc_of(64, 48, 1, 8, False)
    for fmt in range(6):
        d.out_format = fmt
        assert hb.plane_layout(d, host_only=True)[0] == 0


@pytest.mark.parametrize("bd", [-1, 0, 7, 17])
def test_plane_layout_is_zero_for_impossible_depths(bd):
    assert hb.plane_layout(desc_of(64, 48, 1, bd, False), host_only=True)[0] == 0


@pytest.mark.parametrize("name", NAMES)
def test_plane_layout_matches_oracle_planes(name):
    planes, alpha, cf, bd, _ = heic_oracle.decode_planes(load(name))
    allp = planes + ([alpha] if alpha is not None else [])
    h, w = planes[0].shape
    total, layout = hb.plane_layout(desc_of(w, h, cf, bd, alpha is not None), host_only=True)
    assert total == sum(p.size for p in allp) * (1 if bd == 8 else 2)
    assert [(ph, pw) for _, _, pw, ph in layout if pw] == [p.shape for p in allp]


@pytest.mark.parametrize("cf", [0, 1, 2, 3])
@pytest.mark.parametrize("bd", [8, 10, 12, 16])
def test_csc_select_ycbcr_is_an_identity(cf, bd):
    for matrix in range(15):
        for full in (0, 1):
            for alpha in (False, True):
                for up in (hb.api.UPSAMPLE_NEAREST, hb.api.UPSAMPLE_BILINEAR):
                    p = hb.csc_select(matrix, 2, full, cf, bd, alpha, hb.OUT_YCBCR, host_only=True, upsampling=up)
                    assert (p.out_format, p.in_depth, p.out_depth, p.bit_depth) == (hb.OUT_YCBCR, bd, bd, bd), matrix
                    assert (p.pre_op, p.post_op, p.premultiply, p.upsampling) == (0, 0, 0, 0), matrix


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    yield e
    e.close()


def check_desc(d, name):
    m = META[name]
    assert (d.width, d.height, d.bit_depth, bool(d.has_alpha)) == (m["width"], m["height"], m["bit_depth"], m["has_alpha"]), name
    assert d.out_format == hb.OUT_YCBCR and d.bytes_per_pixel == (1 if d.bit_depth == 8 else 2), name
    assert d.premultiplied_alpha == (1 if name in PREM else 0), name


@pytest.mark.gpu
@pytest.mark.parametrize("device_parse", [1, 0])
def test_gpu_job_planes_match_reference(engine, device_parse):
    """All fixtures in one job: grids, limited-range tiles, 4:2:2 / 4:4:4 / mono, 10 / 12 bit, alpha of every kind,
    irot / imir / clap and prem. Each image's packed bytes are the reference's planes."""
    engine.set_option("device_parse", device_parse)
    engine.set_option("host_share_pct", 0)
    try:
        job = hb.HeicJob(engine, [load(n) for n in NAMES], threads=4, out_format=hb.OUT_YCBCR)
    finally:
        engine.set_option("device_parse", 1)
        engine.set_option("host_share_pct", -1)
    job.upload()
    job.run()
    ms = job.stage_ms()
    bad = []
    for i, name in enumerate(NAMES):
        d = job.descs[i]
        check_desc(d, name)
        planes = job.read_planes(i)
        assert len(planes) == (3 if d.chroma_format else 1) + (1 if d.has_alpha else 0), name
        if packed_md5(planes) != META[name]["planes_md5"]:
            bad.append(name)
    assert ms["k5_csc"] > 0      # K8 is timed in the K5 slot
    job.close()
    assert not bad, bad


def stream_checker(names):
    seen = []

    def on_image(index, desc, planes):
        name = names[index]
        check_desc(desc, name)
        seen.append((index, packed_md5(planes) == META[name]["planes_md5"], hb.plane_layout(desc)[0]))
    return seen, on_image


def packed_size(name):
    planes, alpha, cf, bd, _ = heic_oracle.decode_planes(load(name))
    return sum(p.size for p in planes + ([alpha] if alpha is not None else [])) * (1 if bd == 8 else 2)


@pytest.mark.gpu
@pytest.mark.parametrize("host_share", [-1, 0, 100])
def test_gpu_stream_planes_match_reference(engine, host_share):
    names = NAMES * 2
    seen, on_image = stream_checker(names)
    engine.set_option("host_share_pct", host_share)
    try:
        st = hb.decode_stream(engine, [load(n) for n in names], on_image, threads=4, files_per_batch=4, out_format=hb.OUT_YCBCR)
    finally:
        engine.set_option("host_share_pct", -1)
    assert [s[0] for s in seen] == list(range(len(names)))
    assert all(s[1] for s in seen), [names[s[0]] for s in seen if not s[1]]
    assert st["batches"] == (len(names) + 3) // 4
    assert st["bytes_d2h"] == sum(s[2] for s in seen)
    assert st["pixels"] == 2 * sum(META[n]["width"] * META[n]["height"] for n in NAMES)


@pytest.mark.gpu
@pytest.mark.parametrize("nbatches", [1, 2, 3, 4])
def test_gpu_stream_planes_fill_and_drain(engine, nbatches):
    names = (NAMES * 2)[:3 * nbatches - 1]
    seen, on_image = stream_checker(names)
    st = hb.decode_stream(engine, [load(n) for n in names], on_image, threads=2, files_per_batch=3, out_format=hb.OUT_YCBCR)
    assert [s[0] for s in seen] == list(range(len(names))) and all(s[1] for s in seen)
    assert st["batches"] == nbatches


@pytest.mark.gpu
def test_gpu_stream_planes_automatic_batch_size(engine):
    names = NAMES * 2
    seen, on_image = stream_checker(names)
    st = hb.decode_stream(engine, [load(n) for n in names], on_image, threads=4, files_per_batch=0, out_format=hb.OUT_YCBCR)
    assert [s[0] for s in seen] == list(range(len(names))) and all(s[1] for s in seen)
    assert st["batches"] == 1


@pytest.mark.gpu
def test_gpu_stream_planes_external_destinations(engine):
    """A 1-D destination of at least the packed size is used (the callback's planes live in it); one byte too small, or a
    2-D destination whose stride is not the Y row, is ignored and the planes arrive in the library's memory."""
    names = NAMES[:12]
    dests, kinds = [], []
    for k, n in enumerate(names):
        size = packed_size(n)
        kind = ("large", "small", "stride", "none")[k % 4]
        if kind == "large":
            dests.append(np.zeros(size + 100, np.uint8))
        elif kind == "small":
            dests.append(np.zeros(size - 1, np.uint8))
        elif kind == "stride":
            row = META[n]["width"] * (1 if META[n]["bit_depth"] == 8 else 2)
            dests.append(np.zeros((size // row + 2, row + 16), np.uint8))
        else:
            dests.append(None)
        kinds.append(kind)
    seen = {}

    def on_image(index, desc, planes):
        ext = dests[index] is not None and planes[0].ctypes.data == dests[index].ctypes.data
        seen[index] = (ext, packed_md5(planes) == META[names[index]]["planes_md5"])

    hb.decode_stream(engine, [load(n) for n in names], on_image, threads=2, files_per_batch=4, dests=dests, out_format=hb.OUT_YCBCR)
    for k, kind in enumerate(kinds):
        ext, ok = seen[k]
        assert ok, names[k]
        assert ext == (kind == "large"), (names[k], kind)
        if kind == "large":
            size = packed_size(names[k])
            assert md5(dests[k][:size].tobytes()) == META[names[k]]["planes_md5"]


@pytest.mark.gpu
def test_gpu_stream_planes_isolate_bad_files(engine):
    """Planar mode with file_status: a non-HEIC buffer, an 'iovl' file (the reference composes overlays in RGB) and a file
    whose slice data K0 rejects fail; every other file is delivered bit-exact."""
    from test_heic_files import _heic_with_rejected_slice_data, _iovl_file
    bad_slices, good_twin = _heic_with_rejected_slice_data()
    files = [load(NAMES[0]), b"not a heic file at all", load(NAMES[1]), _iovl_file(3), bad_slices, good_twin, load(NAMES[2])]
    planes, alpha, _, bd, _ = heic_oracle.decode_planes(good_twin)
    want = {0: META[NAMES[0]]["planes_md5"], 2: META[NAMES[1]]["planes_md5"], 5: packed_md5([p.astype(np.uint8 if bd == 8 else "<u2") for p in planes]),
            6: META[NAMES[2]]["planes_md5"]}
    expect_bad = {1, 3, 4}
    got = {}
    for per_batch in (3, 7, 1):
        got.clear()
        st = hb.decode_stream(engine, files, lambda i, d, p: got.__setitem__(i, packed_md5(p)), files_per_batch=per_batch,
                              isolate_errors=True, out_format=hb.OUT_YCBCR)
        assert {k for k, v in enumerate(st["file_status"]) if v != 0} == expect_bad, (per_batch, st["file_status"])
        assert st["files_failed"] == 3 and st["first_error"]
        assert got == want, per_batch


def _clap_file(clap_w, clap_h):
    """64 x 48 8-bit 4:2:0 with a centred clean aperture of clap_w x clap_h"""
    from tools import heif_writer as W, hevcenc
    s = hevcenc.encode(hevcenc.synth_image(64, 48, 1, 8, 31), chroma_format=1, bit_depth=8, seed=31)
    return W.single_image(s, 64, 48, 1, 8, transforms=(W.clap(clap_w, 1, clap_h, 1, 0, 1, 0, 1),))


@pytest.mark.gpu
def test_gpu_stream_planes_isolate_clap_with_wider_chroma(engine):
    """A centred clap of 62 x 48 (or 64 x 46) starts at an odd column (row): the reference's crop leaves 32 chroma samples
    per row (24 rows), one more than the packed layout's (w + 1) / 2 (h + 1) / 2. Such a file fails on its own as an
    unsupported image; 61 x 48 and 64 x 47 fit the layout and are delivered bit-exact, as is every other file."""
    files = [load(NAMES[0]), _clap_file(62, 48), _clap_file(61, 48), _clap_file(64, 46), _clap_file(64, 47), load(NAMES[1])]
    want = {0: META[NAMES[0]]["planes_md5"], 5: META[NAMES[1]]["planes_md5"]}
    for k in (2, 4):
        planes, _, _, _, _ = heic_oracle.decode_planes(files[k])
        want[k] = packed_md5([p.astype(np.uint8) for p in planes])
    got = {}
    for per_batch in (6, 2):
        got.clear()
        st = hb.decode_stream(engine, files, lambda i, d, p: got.__setitem__(i, packed_md5(p)), files_per_batch=per_batch,
                              isolate_errors=True, out_format=hb.OUT_YCBCR)
        assert {k for k, v in enumerate(st["file_status"]) if v != 0} == {1, 3}, (per_batch, st["file_status"])
        assert "clean aperture" in st["first_error"]
        assert got == want, per_batch
    with pytest.raises(hb.HeifCudaError, match="clean aperture"):
        hb.HeicJob(engine, [files[1]], threads=1, out_format=hb.OUT_YCBCR)


@pytest.mark.gpu
def test_gpu_planar_ignores_premultiply_and_upsampling_options(engine):
    names = [n for n in NAMES if META[n]["has_alpha"] or n.startswith("single_42")]
    engine.set_option("premultiply_alpha", 1)
    engine.set_option("chroma_upsampling", 1)
    try:
        job = hb.HeicJob(engine, [load(n) for n in names], threads=4, out_format=hb.OUT_YCBCR)
    finally:
        engine.set_option("premultiply_alpha", 0)
        engine.set_option("chroma_upsampling", 0)
    job.upload()
    job.run()
    for i, n in enumerate(names):
        check_desc(job.descs[i], n)
        assert packed_md5(job.read_planes(i)) == META[n]["planes_md5"], n
    job.close()


def _c3_file(bit_depth):
    from tools import heif_writer, hevcenc
    w, h = 2048, 1536
    colour = hevcenc.encode(hevcenc.synth_image(w, h, 2, bit_depth, seed=11), chroma_format=2, bit_depth=bit_depth, qp=24, wpp=1, sao=1,
                            log2_ctb=6, seed=3)
    alpha = hevcenc.encode([hevcenc.synth_image(w, h, 0, bit_depth, seed=12)[0]], chroma_format=0, bit_depth=bit_depth, qp=30, wpp=1,
                           log2_ctb=6, seed=4)
    return heif_writer.single_image(colour, w, h, 2, bit_depth, alpha_stream=alpha)


@pytest.mark.gpu
def test_gpu_full_size_planes_match_oracle(engine):
    """A 4032 x 3024 grid of 512 x 512 tiles (8-bit 4:2:0) and a 2048 x 1536 4:2:2 10-bit image with alpha."""
    from tools import heif_writer
    files = [heif_writer.synth_grid_heic(4032, 3024, tile=512, seed=7, qp=26, wpp=1, sao=1, log2_ctb=6), _c3_file(10)]
    job = hb.HeicJob(engine, files, threads=0, out_format=hb.OUT_YCBCR)
    job.upload()
    job.run()
    for i, data in enumerate(files):
        planes, alpha, _, bd, _ = heic_oracle.decode_planes(data)
        want = planes + ([alpha] if alpha is not None else [])
        got = job.read_planes(i)
        assert len(got) == len(want), i
        for k, (g, w) in enumerate(zip(got, want)):
            assert g.dtype == (np.uint8 if bd == 8 else np.dtype("<u2")) and np.array_equal(g.astype(np.uint16), w), (i, k)
    job.close()


@pytest.mark.gpu
def test_gpu_planar_refuses_what_it_does_not_do(engine):
    L = engine._L
    name = "grid_300x200_t128"
    data = load(name)
    # band jobs
    first, full = C.c_int(), C.c_int()
    assert not L.hc_heic_job_create_band(engine._h, data, len(data), YCBCR, 1, 0, 1, C.byref(first), C.byref(full))
    assert b"HC_OUT_YCBCR" in L.hc_last_error()
    # shared-image targets and a read with the wrong stride
    job = hb.HeicJob(engine, [data], threads=1, out_format=hb.OUT_YCBCR)
    d = job.descs[0]
    shared = L.hc_shared_image_create(engine._h, d.width, d.height, 3)
    assert shared
    assert L.hc_heic_job_set_rgb_target(job._h, 0, shared, 0) == -6      # HC_ERR_UNSUPPORTED
    L.hc_shared_image_destroy(shared)
    job.upload()
    job.run()
    total, _ = hb.plane_layout(d)
    buf = np.zeros(total + 64, np.uint8)
    assert L.hc_heic_job_read_rgb(job._h, 0, buf.ctypes.data, d.width + 1) == -2      # HC_ERR_ARGUMENT
    assert L.hc_heic_job_read_rgb(job._h, 0, buf.ctypes.data, d.width) == 0
    assert md5(buf[:total].tobytes()) == META[name]["planes_md5"] and not buf[total:].any()
    with pytest.raises(hb.HeifCudaError):
        job.read_rgb(0)
    job.close()
    # batch level: an overlay canvas cannot be planar; a planar canvas takes no external RGB target and reads back packed
    hf = hb.HeifFile(load("single_420_8_novui"))
    rec = hb.parse_picture(hf.coded_stream(hf.primary_id))
    b = engine.batch()
    p = rec.pic
    c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y)
    b.add_picture(rec, c)
    ov = L.hc_batch_add_overlay_canvas(b._h, 64, 64, (C.c_uint16 * 4)(0, 0, 0, 0xffff))
    assert ov >= 0
    b.upload()
    b.reconstruct(hb.STAGE_ALL)
    params = hb.csc_select(2, 2, 1, p.chroma_format, p.bit_depth_y, False, hb.OUT_YCBCR)
    assert L.hc_batch_convert_many(b._h, 1, (C.c_int * 1)(ov), (CscParams * 1)(params)) == -6
    assert L.hc_batch_convert(b._h, ov, C.byref(params)) == -6
    # a convert_many call that fails on one canvas leaves the others as they were: c stays RGB
    rgb_params = hb.csc_select(p.matrix_coeffs, p.colour_primaries, p.full_range, p.chroma_format, p.bit_depth_y, False, hb.OUT_RGB)
    b.convert(c, rgb_params)
    rgb = b.read_rgb(c, hb.OUT_RGB)
    assert L.hc_batch_convert_many(b._h, 2, (C.c_int * 2)(c, ov), (CscParams * 2)(params, params)) == -6
    assert np.array_equal(b.read_rgb(c, hb.OUT_RGB), rgb)
    b.convert(c, params)
    assert L.hc_batch_set_rgb_target(b._h, c, None, 0) == -6
    d = desc_of(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y, False)
    total, _ = hb.plane_layout(d)
    buf = np.zeros(total, np.uint8)
    assert L.hc_batch_read_rgb(b._h, c, buf.ctypes.data, p.crop_w * 2) == -2
    assert L.hc_batch_read_rgb(b._h, c, buf.ctypes.data, p.crop_w) == 0
    assert md5(buf.tobytes()) == packed_md5([b.read_plane(c, k) for k in range(3)]) == META["single_420_8_novui"]["planes_md5"]
    b.close()
