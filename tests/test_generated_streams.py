"""Synthetic bitstream fixtures (tests/golden/generated/, made by the content generator in tools/hevc_enc
and decoded by the unmodified reference: tests/golden/make_generated.py) through the product's host
front-end + the CPU oracle (CPU test) and through the CUDA path (GPU test).

They cover what the reference's bundled streams do not: 4:0:0 / 4:2:2 / 4:4:4, 10 and 12 bit, CTB 16/32,
tiles, (dependent) slices with and without cross-boundary loop filtering, cu_qp_delta, transform skip,
scaling lists, PCM, transquant bypass, deblocking offsets, odd sizes with a conformance window."""
import hashlib
import json
import os

import numpy as np
import pytest

import heif_b200 as hb
import oracle_lib
from conftest import ROOT

GEN_DIR = os.path.join(ROOT, "tests", "golden", "generated")
META = json.load(open(os.path.join(ROOT, "tests", "golden", "generated.json")))
NAMES = sorted(META)


def stream(name):
    return open(os.path.join(GEN_DIR, name + ".hevc"), "rb").read()


def md5(b):
    return hashlib.md5(b).hexdigest()


@pytest.mark.parametrize("name", NAMES)
def test_host_parser_and_oracle_match_reference(name):
    rec = hb.parse_picture(stream(name), host_only=True)
    pic = rec.pic
    assert (pic.crop_w, pic.crop_h) == (META[name]["width"], META[name]["height"])
    planes, _ = oracle_lib.reconstruct(rec)
    assert md5(oracle_lib.planes_bytes(planes, pic.bit_depth_y)) == META[name]["yuv_md5"]


@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    yield e
    e.close()


def gpu_decode(engine, recs, stages=hb.STAGE_ALL):
    b = engine.batch()
    canvases = []
    for rec in recs:
        p = rec.pic
        c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y)
        b.add_picture(rec, c)
        canvases.append(c)
    b.upload()
    b.reconstruct(stages)
    out = []
    for rec, c in zip(recs, canvases):
        out.append([b.read_plane(c, k) for k in range(3 if rec.pic.chroma_format else 1)])
    resid = [b.read_residual(i, int(r.pic.resid_count)) for i, r in enumerate(recs)]
    b.close()
    return out, resid


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_matches_reference_and_oracle(engine, name):
    rec = hb.parse_picture(stream(name))
    (got,), (resid,) = gpu_decode(engine, [rec])
    want, want_resid = oracle_lib.reconstruct(rec, want_residual=True)
    n = int(rec.pic.resid_count)
    assert np.array_equal(resid[:n], want_resid[:n]), "K1 residuals differ"
    for k, (g, w) in enumerate(zip(got, want)):
        bad = np.argwhere(g.astype(np.uint16) != w)
        assert bad.size == 0, "%s plane %d: %d samples differ, first at (y,x)=%s" % (name, k, len(bad), tuple(bad[0]))
    dt = np.uint8 if rec.pic.bit_depth_y == 8 else np.dtype("<u2")
    assert md5(b"".join(p.astype(dt).tobytes() for p in got)) == META[name]["yuv_md5"]


@pytest.mark.gpu
@pytest.mark.parametrize("stages", [0, hb.STAGE_DEBLOCK])
def test_gpu_intermediate_stages_match_oracle(engine, stages):
    for name in NAMES:
        rec = hb.parse_picture(stream(name))
        (got,), _ = gpu_decode(engine, [rec], stages)
        want, _ = oracle_lib.reconstruct(rec, stages)
        for k, (g, w) in enumerate(zip(got, want)):
            assert np.array_equal(g.astype(np.uint16), w), (name, stages, k)


@pytest.mark.gpu
def test_gpu_mixed_batch(engine):
    """Every fixture in ONE batch: mixed sizes, chroma formats and bit depths in flight together."""
    recs = [hb.parse_picture(stream(n)) for n in NAMES]
    got, _ = gpu_decode(engine, recs)
    for name, rec, planes in zip(NAMES, recs, got):
        dt = np.uint8 if rec.pic.bit_depth_y == 8 else np.dtype("<u2")
        assert md5(b"".join(p.astype(dt).tobytes() for p in planes)) == META[name]["yuv_md5"], name
