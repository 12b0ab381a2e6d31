"""K0, the device CABAC parser, against the host parser on bitstreams pushed to the limits of their syntax.

The fixtures of the other tests are natural content from the synthetic-content encoder at ordinary settings, so the
long escape path, Rice parameter 4, 16-sign bypass strings, levels of -32768, wrapped QPs, the full SAO offset range and
CTBs at their TB / coefficient capacity are reached by chance or not at all. Here the encoder's stress mode
(tools/hevc_enc, stress_streams.py) writes them on purpose.

CPU: the encoder still reproduces the committed fixtures with the stress off; every stress stream carries what the
encoder meant (the oracle on the host parser's records equals the encoder's own reconstruction), so the host parser is
a valid reference; the CPU build of K0 equals the host parser record for record; the encoder's counters prove the
corpus reaches every extreme.
GPU: the device K0 (lane-parallel writers, CabacDev, capacity slices) in batches of every shape and through the stream
API, compared with the oracle on the host parser's records stage by stage."""
import hashlib
import os
import sys

import numpy as np
import pytest

import heic_oracle
import heif_b200 as hb
import oracle_lib
import stress_streams as ss
from conftest import ROOT
from test_k0_parser import DECLINED, GEN, GEN_DIR, GEN_META, _fmt, _planes_md5, arrays, check_equal

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_generated  # noqa: E402

from tools import hevcenc, heif_writer  # noqa: E402

FMT = hb.STREAM_LENGTH_PREFIXED
STAGES = (0, hb.STAGE_DEBLOCK, hb.STAGE_ALL)
DECLINED_NAMES = [n for n in ss.NAMES if n not in ss.ELIGIBLE]

# Encoder counters the corpus cannot reach, and why. They must stay at 0: a corpus that reaches one belongs in the
# main check.
UNREACHABLE = {}


def first_diff(got, want):
    bad = np.argwhere(got.astype(np.uint16) != want)
    return len(bad), (tuple(int(v) for v in bad[0]) if len(bad) else None)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", sorted(make_generated.CASES))
def test_stress_off_reproduces_committed_fixture(name):
    """With stress == 0 the encoder makes the same RNG draws as before: the committed streams (and the benchmark's
    content) come out byte for byte."""
    w, h, kw = make_generated.CASES[name]
    planes = hevcenc.synth_image(w, h, kw.get("chroma_format", 1), kw.get("bit_depth", 8), seed=kw.get("seed", 1))
    assert hevcenc.encode(planes, **kw) == open(os.path.join(GEN_DIR, name + ".hevc"), "rb").read(), name


@pytest.mark.parametrize("name", ss.NAMES)
def test_stress_stream_round_trip(name):
    """The oracle's pre-filter planes from the host parser's records equal the encoder's reconstruction."""
    data, extra = ss.stream(name)
    got, _ = oracle_lib.reconstruct(hb.parse_picture(data, FMT, host_only=True), 0)
    for k, (g, r) in enumerate(zip(got, extra["recon"])):
        n, at = first_diff(g, r[:g.shape[0], :g.shape[1]])
        assert n == 0, "%s plane %d: %d samples differ from the encoder's reconstruction, first at (y,x)=%s" % (name, k, n, at)


@pytest.mark.parametrize("name", ss.ELIGIBLE)
def test_k0_records_equal_host_parser_stress(name):
    check_equal(ss.data(name), FMT)


@pytest.mark.parametrize("name", DECLINED_NAMES)
def test_k0_declines_stress_stream(name):
    with pytest.raises(hb.HeifCudaError) as ei:
        hb.parse_picture_k0(ss.data(name), FMT, host_only=True)
    assert "not eligible" in str(ei.value)
    assert not hb.K0Picture(ss.data(name), FMT, host_only=True).eligible


def test_stress_corpus_reaches_every_extreme():
    """Summed over the corpus every encoder counter is > 0 (tools/hevc_enc HEVC_ENC_STATS); the ones listed in
    UNREACHABLE stay at 0."""
    total = dict.fromkeys(hevcenc.stat_names(), 0)
    for name in ss.NAMES:
        for k, v in ss.stream(name)[1]["stats"].items():
            total[k] += v
    assert set(UNREACHABLE) <= set(total)
    missed = sorted(k for k, v in total.items() if v == 0 and k not in UNREACHABLE)
    assert not missed, "extremes the stress corpus never writes: %s" % missed
    reached = sorted(k for k in UNREACHABLE if total[k])
    assert not reached, "counters listed as unreachable were reached: %s" % reached
    # the per-CTB capacities are reached by a device-parsed picture, not only by a declined one
    for key in ("ctb_coeff_full", "ctb_tb_full", "level_min", "escape_prefix16", "sign_string_16", "qp_wrap_below"):
        assert sum(ss.stream(n)[1]["stats"][key] for n in ss.ELIGIBLE), key


def test_stress_records_hold_the_extremes():
    """What the counters claim is in the parsed records: levels of -32768 and 32767 and QP_Y below 0, from the host
    parser; a 64 x 64 4:4:4 CTB with TB_CAP_MAX (768) transform blocks."""
    levels, qps = [], []
    for name in ss.NAMES:
        x = arrays(hb.parse_picture(ss.data(name), FMT, host_only=True))
        levels.append(x["coeffs"].view(np.int16)[1::2])     # hc_coeff: pos, level
        qps.append(x["qp_map"].view(np.int8))
    lv = np.concatenate(levels)
    assert (lv == -32768).any() and (lv == 32767).any()
    assert np.concatenate(qps).min() < 0
    rec = hb.parse_picture(ss.data("dense_444_ctb64#1"), FMT, host_only=True)
    assert rec.pic.tb_count == 768 * rec.pic.ctbs_w * rec.pic.ctbs_h


def test_stress_is_deterministic():
    """Same seed, same bytes, reconstruction and counters; another seed, other bytes."""
    w, h, kw = ss.options("c422_12_qg#1")
    planes = hevcenc.synth_image(w, h, 2, 12, 1)
    a, ea = hevcenc.encode(planes, want=("recon", "stats"), **kw)
    b, eb = hevcenc.encode(planes, want=("recon", "stats"), **kw)
    assert a == b and ea["stats"] == eb["stats"]
    assert all(np.array_equal(x, y) for x, y in zip(ea["recon"], eb["recon"]))
    assert hevcenc.encode(planes, **dict(kw, seed=2)) != a


# ---------------------------------------------------------------------------------------------------------------- GPU

def check_planes(got, want, what, pic):
    """Names the first differing sample and the CTB it lies in."""
    sw = 2 if pic.chroma_format in (1, 2) else 1
    sh = 2 if pic.chroma_format == 1 else 1
    for k, (g, w) in enumerate(zip(got, want)):
        n, at = first_diff(g, w)
        if n:
            y, x = at
            cx, cy = (x * sw, y * sh) if k else (x, y)
            pytest.fail("%s plane %d: %d samples differ, first at (y,x)=(%d,%d) got %d want %d, in CTB (x,y)=(%d,%d)" % (
                what, k, n, y, x, int(g[y, x]), int(w[y, x]), cx >> pic.log2_ctb, cy >> pic.log2_ctb))


_want_cache = {}


def oracle_planes(name, stages):
    if (name, stages) not in _want_cache:
        _want_cache[(name, stages)] = oracle_lib.reconstruct(hb.parse_picture(ss.data(name), FMT, host_only=True), stages)[0]
    return _want_cache[(name, stages)]


@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)   # raises if the CUDA engine is missing: no fallback
    yield e
    e.close()


def k0_batch(engine, names, stages, data=ss.data):
    """One batch with every picture of names parsed by K0; data(name) gives the stream. Returns {name: (planes, pic)}."""
    b = engine.batch()
    items = []
    for name in names:
        k = hb.K0Picture(data(name), FMT)
        assert k.eligible, (name, k.why_not)
        p = k.pic
        c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y)
        b.add_k0_picture(k, c)
        items.append((name, c, k))
    try:
        b.upload()
        b.reconstruct(stages)
        return {name: ([b.read_plane(c, i) for i in range(3 if k.pic.chroma_format else 1)], k.pic) for name, c, k in items}
    finally:
        b.close()


@pytest.mark.gpu
def test_gpu_k0_stress_streams_in_one_batch(engine):
    """Every K0-eligible stress stream in one batch, at stage 0 (K0 + K1 + K2), deblocked and complete."""
    for stages in STAGES:
        got = k0_batch(engine, ss.ELIGIBLE, stages)
        for name in ss.ELIGIBLE:
            planes, pic = got[name]
            check_planes(planes, oracle_planes(name, stages), "%s stage=%d" % (name, stages), pic)


@pytest.mark.gpu
def test_gpu_k0_stress_streams_one_per_batch(engine):
    """One picture per batch: fewer chains, other scheduling of the wavefront waits."""
    for name in ss.ELIGIBLE:
        planes, pic = k0_batch(engine, [name], hb.STAGE_ALL)[name]
        check_planes(planes, oracle_planes(name, hb.STAGE_ALL), "%s alone" % name, pic)


@pytest.mark.gpu
def test_gpu_mixed_batch_stress_and_fixtures(engine):
    """Every stress stream host-parsed and (when eligible) K0-parsed, next to the 47 generated fixtures (K0 where
    eligible), all in one batch: capacity-full pictures beside ordinary ones."""
    b = engine.batch()
    items = []
    for name in ss.NAMES:
        rec = hb.parse_picture(ss.data(name), FMT)
        c = b.add_canvas(rec.pic.crop_w, rec.pic.crop_h, rec.pic.chroma_format, rec.pic.bit_depth_y)
        b.add_picture(rec, c)
        items.append(("stress", name + " host", name, c, rec.pic, rec))
        if name in ss.ELIGIBLE:
            k = hb.K0Picture(ss.data(name), FMT)
            c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
            b.add_k0_picture(k, c)
            items.append(("stress", name + " K0", name, c, k.pic, k))
    for name in GEN:
        data = open(os.path.join(GEN_DIR, name + ".hevc"), "rb").read()
        if name in DECLINED:
            r = hb.parse_picture(data, _fmt(name))
            c = b.add_canvas(r.pic.crop_w, r.pic.crop_h, r.pic.chroma_format, r.pic.bit_depth_y)
            b.add_picture(r, c)
            items.append(("gen", name, name, c, r.pic, r))
        else:
            k = hb.K0Picture(data, _fmt(name))
            c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
            b.add_k0_picture(k, c)
            items.append(("gen", name, name, c, k.pic, k))
    try:
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        bad = []
        for kind, what, name, c, pic, _ in items:
            if kind == "gen":
                if _planes_md5(b, c, pic) != GEN_META[name]["yuv_md5"]:
                    bad.append(what)
            else:
                planes = [b.read_plane(c, i) for i in range(3 if pic.chroma_format else 1)]
                check_planes(planes, oracle_planes(name, hb.STAGE_ALL), what + " (mixed batch)", pic)
        assert not bad, "generated fixtures that no longer match the reference: %s" % bad
    finally:
        b.close()


def _heic_files():
    """Single stress items (K0-eligible and not, every chroma format) and one 2 x 2 grid of 4:2:0 stress tiles."""
    files = []
    for name in ("c422_12_qg#1", "c444_10_ctb32#2", "mono_12_qg#1", "dense_444_ctb64#1", "qp_low_12#2", "odd_444#1",
                 "tiles#1"):
        w, h, kw = ss.options(name)
        files.append((name, heif_writer.single_image(ss.data(name), w, h, kw.get("chroma_format", 1), kw.get("bit_depth", 8))))
    tiles = [ss.data("c420_8#%d" % s) for s in (1, 2, 3, 4)]
    files.append(("grid c420_8#1..4", heif_writer.grid_image(tiles, 2, 2, 96, 64, 180, 120)))
    return files


@pytest.mark.gpu
@pytest.mark.parametrize("host_share", [0, 100])
def test_gpu_stream_planes_of_stress_heic(engine, host_share):
    """The production path: HEIC files of stress streams through decode_stream as native planes, device-parsed
    (host share 0) and host-parsed (100); the packed planes equal the oracle's."""
    files = _heic_files()
    want = {}
    for i, (name, data) in enumerate(files):
        planes, _, _, bd, _ = heic_oracle.decode_planes(data)
        dt = np.uint8 if bd == 8 else np.dtype("<u2")
        want[i] = hashlib.md5(b"".join(p.astype(dt).tobytes() for p in planes)).hexdigest()
    seen = {}

    def on_image(index, desc, planes):
        seen[index] = hashlib.md5(b"".join(np.ascontiguousarray(p).tobytes() for p in planes)).hexdigest()
    engine.set_option("host_share_pct", host_share)
    try:
        hb.decode_stream(engine, [d for _, d in files], on_image, threads=2, files_per_batch=4, out_format=hb.OUT_YCBCR)
    finally:
        engine.set_option("host_share_pct", -1)
    assert sorted(seen) == list(range(len(files)))
    bad = [files[i][0] for i in range(len(files)) if seen[i] != want[i]]
    assert not bad, "planes differ from the oracle: %s" % bad
