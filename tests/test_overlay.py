"""'iovl' derived images (SURVEY 8f N3; libheif context.cc:2579-2675, pixelimage.cc:1017-1150): fixtures made by
tests/golden/make_iovl.py and decoded by the unmodified reference in every interleaved format.
CPU: container reader + a numpy restatement of the reference's composition reproduce the reference's MD5s.
GPU: the native job (children on canvases of their own, kernel K7 composing straight into the interleaved output)."""
import hashlib
import json
import os

import pytest

import heif_b200 as hb
import heic_oracle
from conftest import ROOT

DIR = os.path.join(ROOT, "tests", "golden", "iovl")
META = json.load(open(os.path.join(ROOT, "tests", "golden", "iovl.json")))
NAMES = sorted(META)
FORMATS = {"rgb": hb.OUT_RGB, "rgba": hb.OUT_RGBA, "rrggbb_be": hb.OUT_RRGGBB_BE, "rrggbbaa_be": hb.OUT_RRGGBBAA_BE,
           "rrggbb_le": hb.OUT_RRGGBB_LE, "rrggbbaa_le": hb.OUT_RRGGBBAA_LE}


def load(name):
    return open(os.path.join(DIR, name + ".heic"), "rb").read()


def md5(b):
    return hashlib.md5(b).hexdigest()


def compose(data, out_format):
    """decode_overlay_image restated: every child converted like Op_YCbCr_to_RGB<uint8_t> (the csc oracle's general path),
    then heic_oracle.compose_overlay"""
    hf = hb.HeifFile(data, host_only=True)
    ov = hf.overlay(hf.primary_id)
    children, alphas = [], []
    for k in range(ov.n):
        rgba = heic_oracle.decode_rgb(data, hb.OUT_RGBA, item_id=int(ov.children[k]))       # 4:4:4 8 bit: the general fp32 op, alpha copied
        px = rgba.reshape(rgba.shape[0], -1, 4)
        children.append(px[:, :, :3])
        alphas.append(px[:, :, 3] if hf.image_info(int(ov.children[k])).alpha_id else None)
    offsets = [(ov.dx[k], ov.dy[k]) for k in range(ov.n)]
    return heic_oracle.compose_overlay(children, alphas, offsets, ov.background, ov.canvas_w, ov.canvas_h, out_format)


@pytest.mark.parametrize("name", NAMES)
def test_overlay_container_fields(name):
    hf = hb.HeifFile(load(name), host_only=True)
    ov = hf.overlay(hf.primary_id)
    m = META[name]
    assert [ov.canvas_w, ov.canvas_h] == m["canvas"] and list(ov.background) == m["background"]
    assert ov.n == len(m["children"])
    assert [[ov.dx[k], ov.dy[k]] for k in range(ov.n)] == [c[2:4] for c in m["children"]]
    with pytest.raises(hb.HeifCudaError):
        hf.overlay(int(ov.children[0]))


@pytest.mark.parametrize("name", NAMES)
def test_overlay_restatement_reproduces_reference(name):
    data = load(name)
    for key, fmt in FORMATS.items():
        assert md5(compose(data, fmt).tobytes()) == META[name][key + "_md5"], key


@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("key", sorted(FORMATS))
def test_gpu_overlay_job_matches_reference(engine, key):
    job = hb.HeicJob(engine, [load(n) for n in NAMES], threads=2, out_format=FORMATS[key])
    job.upload()
    job.run()
    for i, n in enumerate(NAMES):
        d = job.descs[i]
        assert [d.width, d.height] == META[n]["size"]
        assert md5(job.read_rgb(i).tobytes()) == META[n][key + "_md5"], (n, key)
    job.close()


@pytest.mark.gpu
def test_gpu_overlay_of_subsampled_children_is_refused_like_the_reference(engine):
    """the reference fails with "Unsupported color conversion" for 4:2:0 children (tests/test_heic_files.py asserts it)"""
    from tools import heif_writer as W, hevcenc
    b = W.HeifBuilder()
    kid = b.add_hevc_image(hevcenc.encode(hevcenc.synth_image(64, 64, 1, 8, 70), chroma_format=1, bit_depth=8, seed=70), 64, 64, 1, 8, hidden=True)
    b.primary = b.add_overlay([kid], 100, 80, [(3, 5)])
    with pytest.raises(hb.HeifCudaError, match="Unsupported color conversion"):
        hb.HeicJob(engine, [b.serialize()], threads=1)
