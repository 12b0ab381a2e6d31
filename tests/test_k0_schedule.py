"""K0's schedule: one warp per substream chain, four chains per CTA, the chains in the order the engine sorts them (CTB
row first, the chain with the most slice data first within a row, then the order of the pictures). Which warp parses
which chain, and when, must not change a single record.

GPU: a batch with several times more chains than the 4,736 warps K0 keeps on a B200 (WPP and non-WPP pictures, grid and
single-image files, 1080p pictures of 17 rows of 30 CTBs) equals the oracle file by file; one file of one chain (one CTA,
three of its warps without work) too; one damaged picture in the middle of a large batch is reported by index while the
kernel finishes and every other picture stays bit-exact."""
import hashlib
import os

import numpy as np
import pytest

import heic_oracle
import heif_b200 as hb
from test_fuzz import GEN_DIR, GEN_META, _fmt, corrupt

from tools import heif_writer, hevcenc  # noqa: E402

# resident K0 warps of a B200: 148 SMs x 8 CTAs x 4 warps
SLOTS = 4736

_files = {}


def files():
    """name -> (HEIC bytes, K0 chains of its coded pictures)"""
    if not _files:
        enc = dict(qp=26, sao=1, log2_ctb=6)
        _files["grid_wpp_2048x1024"] = (heif_writer.synth_grid_heic(2048, 1024, tile=512, seed=21, wpp=1, **enc), 8 * 8)
        _files["grid_nowpp_1024x1024"] = (heif_writer.synth_grid_heic(1024, 1024, tile=512, seed=22, wpp=0, **enc), 4 * 1)
        s = hevcenc.encode(hevcenc.synth_image(1920, 1080, 1, 8, 23), wpp=1, seed=23, **enc)
        _files["single_wpp_1920x1080"] = (heif_writer.single_image(s, 1920, 1080, 1, 8), 17)
        s = hevcenc.encode(hevcenc.synth_image(512, 512, 1, 8, 24), wpp=0, seed=24, **enc)
        _files["single_nowpp_512"] = (heif_writer.single_image(s, 512, 512, 1, 8), 1)
    return _files


_want = {}


def want_rgb(name):
    if name not in _want:
        _want[name] = heic_oracle.decode_rgb(files()[name][0], hb.OUT_RGB)
    return _want[name]


@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    e.set_option("host_share_pct", 0)     # every coded item goes to K0
    yield e
    e.close()


def run_job(engine, names):
    job = hb.HeicJob(engine, [files()[n][0] for n in names])
    try:
        job.upload()
        job.run()
        assert job.stage_ms()["k0_parse"] > 0
        bad = [i for i, n in enumerate(names) if not np.array_equal(job.read_rgb(i), want_rgb(n))]
    finally:
        job.close()
    assert not bad, "files %s differ from the oracle" % [(i, names[i]) for i in bad[:8]]


@pytest.mark.gpu
def test_gpu_k0_many_more_chains_than_warps(engine):
    """The chain order crosses pictures, files and rows many times; files of four kinds interleaved."""
    kinds = sorted(files())
    names = [kinds[i % len(kinds)] for i in range(180 * len(kinds))]
    assert sum(files()[n][1] for n in names) >= 3 * SLOTS
    run_job(engine, names)


@pytest.mark.gpu
def test_gpu_k0_one_file_of_one_chain(engine):
    run_job(engine, ["single_nowpp_512"])


def _damaged():
    """The first corruption of test_fuzz's seeds for the 512 x 512 WPP tile that K0 rejects in its slice data."""
    data = open(os.path.join(GEN_DIR, "tile_512.hevc"), "rb").read()
    for seed in range(12):
        bad = corrupt(data, seed * 104729 + len("tile_512"))
        try:
            k = hb.K0Picture(bad, _fmt(bad))
        except hb.HeifCudaError:
            continue                                   # header damage: rejected on the host
        if not k.eligible:
            continue
        try:
            hb.parse_picture_k0(bad, _fmt(bad), host_only=True)
        except hb.HeifCudaError:
            return k                                   # the CPU build of the same parser core rejects it
    pytest.fail("no corruption of tile_512 is rejected in its slice data")


@pytest.mark.gpu
def test_gpu_k0_damaged_picture_in_a_large_batch(engine):
    """A failing chain raises its picture's progress words, so the chains below it in its picture end too: the batch
    finishes, the damaged picture is named, all others are bit-exact."""
    good = ["tile_512", "wpp", "wpp_slices", "base_420_8", "slices_dep", "c422_10"]
    names = [good[i % len(good)] for i in range(6 * len(good))] + ["tile_512"] * 720
    middle = len(names) // 2
    b = engine.batch()
    items = []
    for i, n in enumerate(names):
        if i == middle:
            k = _damaged()
            c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
            b.add_k0_picture(k, c)
            items.append((None, c, k))
        data = open(os.path.join(GEN_DIR, n + ".hevc"), "rb").read()
        k = hb.K0Picture(data, _fmt(data))
        assert k.eligible, (n, k.why_not)
        c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
        b.add_k0_picture(k, c)
        items.append((n, c, k))
    try:
        b.upload()
        with pytest.raises(hb.HeifCudaError) as ei:
            b.reconstruct(hb.STAGE_ALL)
        assert "picture %d:" % middle in str(ei.value), str(ei.value)
        bad = []
        for n, c, k in items:
            if n is None:
                continue
            pic = k.pic
            planes = [b.read_plane(c, i) for i in range(3 if pic.chroma_format else 1)]
            dt = np.uint8 if pic.bit_depth_y == 8 else np.dtype("<u2")
            if hashlib.md5(b"".join(p.astype(dt).tobytes() for p in planes)).hexdigest() != GEN_META[n]["yuv_md5"]:
                bad.append(n)
        assert not bad, bad
    finally:
        b.close()
