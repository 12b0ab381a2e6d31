"""GPU parity tests (run with -m gpu on the B200 box): the sm_100a kernels, called through the C ABI,
against the CPU oracle on the same records, stage by stage, and against the committed golden MD5s of
the unmodified reference."""
import hashlib
import json
import os

import numpy as np
import pytest

import heif_b200 as hb
import oracle_lib
from conftest import ROOT, read_stream

pytestmark = pytest.mark.gpu
GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))


def md5(b):
    return hashlib.md5(b).hexdigest()


@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)   # raises if the CUDA engine is missing: no fallback
    yield e
    e.close()


def all_pictures():
    """(label, Records) of every bundled picture."""
    out = []
    for name in sorted(GOLDEN["yuv_md5"]):
        out.append((name, hb.parse_picture(read_stream(name), hb.STREAM_ANNEXB)))
    for fname in sorted(GOLDEN["heic"]):
        hf = hb.HeifFile(read_stream(fname))
        for item in sorted(GOLDEN["heic"][fname]):
            out.append(("%s#%s" % (fname, item), hb.parse_picture(hf.coded_stream(int(item)))))
    return out


@pytest.fixture(scope="module")
def pictures():
    return all_pictures()


def gpu_planes(engine, rec, stages):
    b = engine.batch()
    p = rec.pic
    c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y)
    b.add_picture(rec, c)
    b.upload()
    b.reconstruct(stages)
    planes = [b.read_plane(c, k) for k in range(3 if p.chroma_format else 1)]
    resid = b.read_residual(0, int(p.resid_count))
    b.close()
    return planes, resid


def test_k1_residuals_match_oracle(engine, pictures):
    for label, rec in pictures:
        _, want = oracle_lib.reconstruct(rec, 0, want_residual=True)
        _, got = gpu_planes(engine, rec, 0)
        n = int(rec.pic.resid_count)
        assert np.array_equal(got[:n], want[:n]), label


@pytest.mark.parametrize("stages", [0, hb.STAGE_DEBLOCK, hb.STAGE_ALL])
def test_planes_match_oracle_per_stage(engine, pictures, stages):
    for label, rec in pictures:
        want, _ = oracle_lib.reconstruct(rec, stages)
        got, _ = gpu_planes(engine, rec, stages)
        for k, (g, w) in enumerate(zip(got, want)):
            bad = np.argwhere(g.astype(np.uint16) != w)
            assert bad.size == 0, "%s stages=%d plane %d: %d samples differ, first at (y,x)=%s" % (
                label, stages, k, len(bad), tuple(bad[0]))


def test_full_decode_matches_reference_golden(engine, pictures):
    for label, rec in pictures:
        got, _ = gpu_planes(engine, rec, hb.STAGE_ALL)
        digest = md5(b"".join(p.tobytes() for p in got))
        if "#" in label:
            fname, item = label.split("#")
            assert digest == GOLDEN["heic"][fname][item]["planes_md5"], label
        else:
            assert digest == GOLDEN["yuv_md5"][label], label


def test_one_batch_with_all_pictures(engine, pictures):
    """All pictures in flight at once: one upload, one launch sequence."""
    b = engine.batch()
    canvases = []
    for _, rec in pictures:
        p = rec.pic
        c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y)
        b.add_picture(rec, c)
        canvases.append(c)
    b.upload()
    b.reconstruct(hb.STAGE_ALL)
    for (label, rec), c in zip(pictures, canvases):
        want, _ = oracle_lib.reconstruct(rec, hb.STAGE_ALL)
        for k in range(3):
            assert np.array_equal(b.read_plane(c, k).astype(np.uint16), want[k]), (label, k)
    assert b.launch_count >= 5
    b.close()


@pytest.mark.parametrize("fname", sorted(GOLDEN["heic"]))
def test_heic_to_rgb_matches_reference_golden(engine, fname):
    data = read_stream(fname)
    for item, g in GOLDEN["heic"][fname].items():
        rgb = hb.decode_heic(engine, data, hb.OUT_RGB, int(item))
        assert rgb.shape == (g["height"], g["width"] * 3)
        assert md5(rgb.tobytes()) == g["rgb_md5"], (fname, item)
        rgba = hb.decode_heic(engine, data, hb.OUT_RGBA, int(item))
        assert md5(rgba.tobytes()) == g["rgba_md5"], (fname, item)
