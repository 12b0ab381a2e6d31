"""K1..K5 against the CPU oracle on records pushed to the limits of their legal values.

The fixtures (47 generated streams, the three 1080p streams, the items of the bundled HEIC files) are natural
content: levels, QPs, intra modes and filter parameters stay in a narrow band, so the value-dependent branches of the
kernels are reached by chance or not at all. Here each fixture's records are rewritten by record_mutation.mutate()
(five families, two seeds) and the kernels are compared with the oracle on the result, stage by stage.
test_mutated_corpus_reaches_every_oracle_branch proves, with the oracle's branch counters, that the corpus reaches
the branches the GPU tests are meant for."""
import ctypes as C
import json
import os
import sys

import numpy as np
import pytest

import heic_oracle
import heif_b200 as hb
from heif_b200 import api
import oracle_lib
import record_mutation as rm
from conftest import ROOT, read_stream

GEN_DIR = os.path.join(ROOT, "tests", "golden", "generated")
GENERATED = sorted(json.load(open(os.path.join(ROOT, "tests", "golden", "generated.json"))))
GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))
FIXTURES = (["gen:" + n for n in GENERATED] + ["1080p:" + n for n in sorted(GOLDEN["yuv_md5"])] +
            ["heic:%s#%s" % (f, i) for f in sorted(GOLDEN["heic"]) for i in sorted(GOLDEN["heic"][f])])
SEEDS = (1, 2)
CASES = [(f, s) for f in rm.FAMILIES for s in SEEDS]
STAGES = (0, hb.STAGE_DEBLOCK, hb.STAGE_ALL)

# Counters the corpus cannot reach, and why. They must stay at 0: a corpus that reaches one belongs in the main check.
UNREACHABLE = {
    # |second-pass sum| <= 32768 * 242 (largest column sum of |DST|), shifted right by 20 - bitDepth >= 8: below 2^15
    "k1_dst_pass2_clip": "the DST second pass cannot leave int16 at bit depths up to 12",
}

# one picture per (chroma format, bit depth) the fixtures have, for K5
K5_PICTURES = ("mono_8", "mono_12", "base_420_8", "c420_10", "c420_12", "c422_8", "scaling_custom_10", "c422_12", "c444_8",
               "c444_10")
# (matrix_coefficients, colour_primaries): the primaries only matter to matrices 12 and 13
K5_MATRICES = ((0, 1), (1, 1), (2, 1), (5, 1), (6, 1), (9, 1), (10, 1), (12, 1), (12, 9), (13, 1), (13, 9))
# in any order: the K5 batch below has one canvas, and a convert lays out anew the block of the canvas it names
K5_OUT_FORMATS = (hb.OUT_RRGGBBAA_BE, hb.OUT_RRGGBBAA_LE, hb.OUT_RRGGBB_BE, hb.OUT_RRGGBB_LE, hb.OUT_RGBA, hb.OUT_RGB)


def load(label, host_only=False):
    """Records of one fixture picture; host_only=False gives the engine library's records, which a batch accepts."""
    kind, name = label.split(":", 1)
    if kind == "gen":
        return hb.parse_picture(open(os.path.join(GEN_DIR, name + ".hevc"), "rb").read(), host_only=host_only)
    if kind == "1080p":
        return hb.parse_picture(read_stream(name), hb.STREAM_ANNEXB, host_only=host_only)
    fname, item = name.split("#")
    hf = hb.HeifFile(read_stream(fname), host_only=host_only)
    return hb.parse_picture(hf.coded_stream(int(item)), host_only=host_only)


def mutated(label, family, seed, host_only=False):
    rec = load(label, host_only)
    rm.mutate(rec, family, seed)
    return rec


def csc_cases(chroma_format, bit_depth, has_alpha, host_only=False):
    """(matrix, primaries, full_range, out_format, upsampling) of every conversion csc_select accepts"""
    for out in K5_OUT_FORMATS:
        for matrix, primaries in K5_MATRICES:
            for full in (0, 1):
                for ups in (api.UPSAMPLE_NEAREST, api.UPSAMPLE_BILINEAR):
                    try:
                        params = hb.csc_select(matrix, primaries, full, chroma_format, bit_depth, has_alpha, out, host_only,
                                               upsampling=ups)
                    except hb.HeifCudaError:
                        continue
                    yield (matrix, primaries, full, out, ups), params


def oracle_rgb(planes, alpha, cf, bd, case):
    matrix, primaries, full, out, ups = case
    try:
        return heic_oracle.csc(planes, cf, bd, matrix, full, out, alpha, primaries, ups)
    except RuntimeError:
        return None


def alpha_stream(width, height, bit_depth):
    """A monochrome picture of the given size and depth from the synthetic-content encoder (tools/hevc_enc)."""
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from tools import hevcenc
    planes = hevcenc.synth_image(width, height, chroma_format=0, bit_depth=bit_depth, seed=width + height)
    return hevcenc.encode(planes, chroma_format=0, bit_depth=bit_depth)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("family", rm.FAMILIES)
def test_mutated_records_are_legal_and_reconstruct(family):
    for label in FIXTURES:
        for seed in SEEDS:
            rec = mutated(label, family, seed, host_only=True)
            rm.check_legal(rec)
            oracle_lib.reconstruct(rec, want_residual=True)


def test_unmutated_records_are_legal():
    for label in FIXTURES:
        rm.check_legal(load(label, host_only=True))


def test_mutation_is_deterministic_and_changes_values():
    label = "gen:c420_12"
    for family in rm.FAMILIES:
        a, b = mutated(label, family, 1, True), mutated(label, family, 1, True)
        va, vb, v0 = rm.views(a), rm.views(b), rm.views(load(label, True))
        for name in va:
            assert np.array_equal(va[name].view(np.uint8), vb[name].view(np.uint8)), (family, name)
        assert any(not np.array_equal(va[n].view(np.uint8), v0[n].view(np.uint8)) for n in va), family


def test_mutated_corpus_reaches_every_oracle_branch():
    """Every branch counter of the oracle is > 0 over the mutated corpus (K1..K4 over every fixture x family x seed,
    K5 over every conversion of the K5 pictures); the ones listed in UNREACHABLE stay at 0."""
    oracle_lib.counters_reset()
    for family, seed in CASES:
        for label in FIXTURES:
            oracle_lib.reconstruct(mutated(label, family, seed, host_only=True))
    for name in K5_PICTURES:
        rec = mutated("gen:" + name, "all", 1, host_only=True)
        planes, _ = oracle_lib.reconstruct(rec)
        p = rec.pic
        for case, _ in csc_cases(p.chroma_format, p.bit_depth_y, False, host_only=True):
            oracle_rgb(planes, None, p.chroma_format, p.bit_depth_y, case)
    counts = oracle_lib.counters()
    assert set(UNREACHABLE) <= set(counts)
    missed = sorted(k for k, v in counts.items() if v == 0 and k not in UNREACHABLE)
    assert not missed, "oracle branches the mutated corpus never takes: %s" % missed
    reached = sorted(k for k in UNREACHABLE if counts[k])
    assert not reached, "counters listed as unreachable were reached: %s" % reached


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)   # raises if the CUDA engine is missing: no fallback
    yield e
    e.close()


def gpu_run(engine, recs, stages, want_resid=False):
    """One batch holding every picture of recs. Returns (planes per picture, residuals per picture or None)."""
    b = engine.batch()
    canvases = []
    for rec in recs:
        p = rec.pic
        canvases.append(b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y))
        b.add_picture(rec, canvases[-1])
    b.upload()
    b.reconstruct(stages)
    planes = [[b.read_plane(c, k) for k in range(3 if r.pic.chroma_format else 1)] for r, c in zip(recs, canvases)]
    resid = [b.read_residual(i, int(r.pic.resid_count)) for i, r in enumerate(recs)] if want_resid else None
    b.close()
    return planes, resid


def first_diff(got, want):
    bad = np.argwhere(got != want)
    return len(bad), (tuple(int(v) for v in bad[0]) if len(bad) else None)


def check_planes(got, want, what):
    for k, (g, w) in enumerate(zip(got, want)):
        n, at = first_diff(g.astype(np.uint16), w)
        assert n == 0, "%s plane %d: %d samples differ, first at (y,x)=%s" % (what, k, n, at)


def check_residual(got, want, n, what):
    bad, at = first_diff(got[:n], want[:n])
    assert bad == 0, "%s: K1 residuals differ in %d of %d elements, first at %s" % (what, bad, n, at)


def check_corpus(engine, family, seed, stages_list, labels=FIXTURES, residuals=True):
    recs = [mutated(label, family, seed) for label in labels]
    for stages in stages_list:
        got, resid = gpu_run(engine, recs, stages, residuals and stages == stages_list[0])
        for i, (label, rec) in enumerate(zip(labels, recs)):
            what = "%s family=%s seed=%d stage=%d" % (label, family, seed, stages)
            want, want_resid = oracle_lib.reconstruct(rec, stages, want_residual=resid is not None)
            if resid is not None:
                check_residual(resid[i], want_resid, int(rec.pic.resid_count), what)
            check_planes(got[i], want, what)


@pytest.mark.gpu
@pytest.mark.parametrize("family,seed", CASES)
def test_gpu_stages_match_oracle_on_mutated_records(engine, family, seed):
    """Every mutated picture in one batch, at stage 0 (K1 + K2), deblocked (K3) and complete (K4)."""
    check_corpus(engine, family, seed, STAGES)


@pytest.mark.gpu
def test_gpu_single_picture_batches_match_oracle(engine):
    """One picture per batch: the launch geometry of a batch of one, for every fixture."""
    for label in FIXTURES:
        check_corpus(engine, "all", 1, (hb.STAGE_ALL,), [label])


def k5_batch(engine, name, with_alpha):
    """A batch with one mutated K5 picture on a canvas (and a mutated monochrome alpha picture of its size)."""
    rec = mutated("gen:" + name, "all", 1)
    p = rec.pic
    b = engine.batch()
    c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y, with_alpha)
    b.add_picture(rec, c)
    planes, _ = oracle_lib.reconstruct(rec)
    alpha = None
    if with_alpha:
        arec = hb.parse_picture(alpha_stream(p.crop_w, p.crop_h, p.bit_depth_y))
        rm.mutate(arec, "all", 2)
        b.add_picture(arec, c, role=api.ROLE_ALPHA)
        alpha = oracle_lib.reconstruct(arec)[0][0]
    b.upload()
    b.reconstruct(hb.STAGE_ALL)
    return b, c, rec, planes, alpha


@pytest.mark.gpu
@pytest.mark.parametrize("with_alpha", [False, True])
@pytest.mark.parametrize("name", K5_PICTURES)
def test_gpu_k5_every_conversion_matches_oracle(engine, name, with_alpha):
    b, c, rec, planes, alpha = k5_batch(engine, name, with_alpha)
    p = rec.pic
    cf, bd = p.chroma_format, p.bit_depth_y
    try:
        checked = 0
        for case, params in csc_cases(cf, bd, with_alpha):
            want = oracle_rgb(planes, alpha, cf, bd, case)
            if want is None:
                continue
            b.convert(c, params)
            got = b.read_rgb(c, case[3])
            n, at = first_diff(got, want)
            assert n == 0, "%s alpha=%s (matrix, primaries, full_range, out_format, upsampling)=%s: %d bytes differ, first at %s" % (
                name, with_alpha, case, n, at)
            checked += 1
        assert checked > 0
    finally:
        b.close()


def first_conversion(cases, planes, cf, out):
    """(params, oracle bytes) of the first of an 8-bit canvas' csc_cases to `out` that the oracle converts"""
    for case, params in cases:
        want = oracle_rgb(planes, None, cf, 8, case) if case[3] == out else None
        if want is not None:
            return params, want


@pytest.mark.gpu
def test_gpu_k5_convert_many_mixed_canvases(engine):
    """One hc_batch_convert_many call (the form hc_heic_job uses) over canvases of every format, depth and alpha, each
    with its own conversion; before it, single converts whose layout would move a canvas converted earlier."""
    b = engine.batch()
    jobs, seq = [], []
    for i, name in enumerate(K5_PICTURES):
        rec = mutated("gen:" + name, "all", 2)
        p = rec.pic
        with_alpha = i % 2 == 1
        c = b.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y, with_alpha)
        b.add_picture(rec, c)
        planes, _ = oracle_lib.reconstruct(rec)
        alpha = None
        if with_alpha:
            arec = hb.parse_picture(alpha_stream(p.crop_w, p.crop_h, p.bit_depth_y))
            rm.mutate(arec, "all", 3)
            b.add_picture(arec, c, role=api.ROLE_ALPHA)
            alpha = oracle_lib.reconstruct(arec)[0][0]
        cases = list(csc_cases(p.chroma_format, p.bit_depth_y, with_alpha))
        k = 7 * i
        while True:
            case, params = cases[k % len(cases)]
            want = oracle_rgb(planes, alpha, p.chroma_format, p.bit_depth_y, case)
            if want is not None:
                break
            k += 1
        jobs.append((name, c, case, params, want))
        if i in (0, 2):   # 8-bit canvases without alpha for the convert sequence below
            seq.append((c, {out: first_conversion(cases, planes, p.chroma_format, out) for out in (hb.OUT_RGBA, hb.OUT_RGB)}))
    try:
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        # convert c0 to RGBA, c1 to RGB, c0 to RGB: the narrower c0 would move c1's block, so the last call either fails and
        # changes nothing or leaves c1 where it was
        (c0, f0), (c1, f1) = seq
        b.convert(c0, f0[hb.OUT_RGBA][0])
        b.convert(c1, f1[hb.OUT_RGB][0])
        rc = engine._L.hc_batch_convert(b._h, c0, C.byref(f0[hb.OUT_RGB][0]))
        assert rc in (0, -2), rc      # HC_OK, HC_ERR_ARGUMENT
        assert np.array_equal(b.read_rgb(c1, hb.OUT_RGB), f1[hb.OUT_RGB][1])
        fmt0 = hb.OUT_RGB if rc == 0 else hb.OUT_RGBA
        assert np.array_equal(b.read_rgb(c0, fmt0), f0[fmt0][1])
        canv = (C.c_int * len(jobs))(*[j[1] for j in jobs])
        params = (hb.CscParams * len(jobs))(*[j[3] for j in jobs])
        api.check(engine._L, engine._L.hc_batch_convert_many(b._h, len(jobs), canv, params), "hc_batch_convert_many")
        for name, c, case, _, want in jobs:
            got = b.read_rgb(c, case[3])
            n, at = first_diff(got, want)
            assert n == 0, "%s %s: %d bytes differ, first at %s" % (name, case, n, at)
    finally:
        b.close()
