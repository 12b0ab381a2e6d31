"""The coding-tree geometry the SPS signals, from bitstream to pixels: min CB 16 .. 64, min TB 8 .. 32, max TB from the
min TB up to 32, transform depth 0 .. 4 (tree_streams.py). Every other stream of the suite has min CB 8 and min TB 4, so
the inferred splits and leaves of 7.3.8.4 and 7.3.8.8, part_mode at min CB, the quantisation groups of one min CB and the
wide conformance windows are reached here only.

CPU: every stream carries what the encoder meant (the oracle on the host parser's records equals the encoder's own
reconstruction); the CPU build of K0 equals the host parser record for record on every stream it takes and declines the
others for the right reason; the QP map of both parsers equals the encoder's own QpY map, the only independent check of
the QP of CUs without residual, which only deblocking sees; the deblocking edge bits of both parsers equal a numpy
restatement of 8.7.2 built from the luma blocks; SPS / PPS values one past each geometry limit are refused by name; the
encoder's counters prove the corpus reaches every case and the other corpora reach none of the new ones.
GPU: the device K0 + K1..K5 against the oracle in batches of every shape and through the stream API."""
import hashlib

import numpy as np
import pytest

import heic_oracle
import heif_b200 as hb
import oracle_lib
import record_mutation as rm
import tree_streams as ts
from test_k0_parser import DECLINED, GEN, GEN_DIR, GEN_META, _fmt, _planes_md5, check_equal
from test_syntax_extremes import check_planes, first_diff, k0_batch

from tools import heif_writer, hevcenc  # noqa: E402

FMT = hb.STREAM_LENGTH_PREFIXED
STAGES = (0, hb.STAGE_DEBLOCK, hb.STAGE_ALL)
# encoder counters that need min CB > 8, min TB > 4, transform depth 4 or a conformance offset of 8 or more: 0 over the
# stress and range-extension corpora, which is the gap this corpus closes
NEW_GEOMETRY = ["nxn_log2_1", "nxn_log2_2", "nxn_log2_3", "border_split_min_cb_0", "border_split_min_cb_1", "tu_depth_4",
                "leaf_at_min_tb_gt4", "qg_min_cb_gt8", "conf_offset_ge8"]


def records(name):
    return hb.parse_picture(ts.data(name), FMT, host_only=True)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", ts.NAMES)
def test_tree_stream_round_trip(name):
    """The oracle's pre-filter planes from the host parser's records equal the encoder's reconstruction."""
    data, extra = ts.stream(name)
    got, _ = oracle_lib.reconstruct(records(name), 0)
    for k, (g, r) in enumerate(zip(got, extra["recon"])):
        n, at = first_diff(g, r[:g.shape[0], :g.shape[1]])
        assert n == 0, "%s plane %d: %d samples differ from the encoder's reconstruction, first at (y,x)=%s" % (name, k, n, at)


@pytest.mark.parametrize("name", ts.ELIGIBLE)
def test_k0_records_equal_host_parser_tree(name):
    check_equal(ts.data(name), FMT)


@pytest.mark.parametrize("name", ts.DECLINED)
def test_k0_declines_tree_stream(name):
    k = hb.K0Picture(ts.data(name), FMT, host_only=True)
    assert not k.eligible
    assert k.why_not == ts.K0_DECLINED[name.split("#")[0]], k.why_not


def _parsed(name):
    """(parser name, records) of both parsers, K0 only where it takes the stream."""
    out = [("host", records(name))]
    if name in ts.ELIGIBLE:
        out.append(("K0", hb.parse_picture_k0(ts.data(name), FMT, host_only=True)))
    return out


@pytest.mark.parametrize("name", ts.NAMES)
def test_qp_map_equals_encoder(name):
    """QpY of every 8 x 8 block, as both parsers derive it (8.6.1), equals the QP the encoder coded with."""
    want = ts.stream(name)[1]["qp"]
    for parser, rec in _parsed(name):
        got = rm.views(rec)["qp_map"].reshape(want.shape)
        n, at = first_diff(got.view(np.uint8), want.view(np.uint8))
        assert n == 0, "%s %s: QpY of %d 8x8 blocks differs from the encoder's, first at (y8,x8)=%s got %d want %d" % (
            name, parser, n, at, got[at], want[at])


def restate_edges(pic, blks):
    """H.265 8.7.2 for an intra picture with default loop-filter flags: every transform and prediction block edge on the
    8 x 8 grid is filtered with bS 2, except at the picture's left and top edges. The luma blocks are the transform
    blocks (an NxN CU splits its transform tree at depth 0, so its PB edges are TB edges). Returns (H / 4, W / 4) bytes
    of EDGE_V / EDGE_H bits, the layout of hc_pic.edge_map, on the 8 x 8 grid only."""
    e = np.zeros((pic.height >> 2, pic.width >> 2), np.uint8)
    for b in blks[blks["cidx"] == 0]:
        x, y, n = int(b["x"]), int(b["y"]), 1 << int(b["log2"])
        if x and x % 8 == 0:
            e[y >> 2:(y + n) >> 2, x >> 2] |= rm.EDGE_V
        if y and y % 8 == 0:
            e[y >> 2, x >> 2:(x + n) >> 2] |= rm.EDGE_H
    return e


@pytest.mark.parametrize("name", ts.NAMES)
def test_edge_map_equals_restatement(name):
    for parser, rec in _parsed(name):
        v = rm.views(rec)
        want = restate_edges(rec.pic, v["blks"])
        got = v["edge_map"].reshape(want.shape).copy()
        # the parsers also mark the edges of 4 x 4 blocks between the grid lines; deblocking reads the grid only
        got[:, 1::2] &= ~np.uint8(rm.EDGE_V)
        got[1::2, :] &= ~np.uint8(rm.EDGE_H)
        got &= rm.EDGE_V | rm.EDGE_H
        n, at = first_diff(got, want)
        assert n == 0, "%s %s: %d 4x4 units with other edge bits, first at (y4,x4)=%s got %d want %d" % (
            name, parser, n, at, got[at], want[at])


def test_tree_corpus_reaches_every_case():
    """Every coding-tree counter of the encoder is > 0 over the corpus and over the K0-eligible streams alone; the
    counters of the new geometry are 0 over the stress and range-extension corpora."""
    import rext_streams as rs
    import stress_streams as ss
    total = dict.fromkeys(hevcenc.tree_stat_names(), 0)
    device = dict(total)
    for name in ts.NAMES:
        for k, v in ts.stream(name)[1]["tree_stats"].items():
            total[k] += v
            if name in ts.ELIGIBLE:
                device[k] += v
    assert set(NEW_GEOMETRY) <= set(total)
    assert not [k for k, v in total.items() if v == 0], total
    assert not [k for k, v in device.items() if v == 0], device
    for corpus in (ss, rs):
        for name in corpus.NAMES:
            st = corpus.stream(name)[1]["tree_stats"]
            assert not [k for k in NEW_GEOMETRY if st[k]], (name, {k: st[k] for k in NEW_GEOMETRY})


def test_tree_is_deterministic():
    """Same seed, same bytes; another seed, other bytes; log2_min_cb 0 stands for 3."""
    w, h, kw = ts.options("cb16_tb8_10#1")
    planes = hevcenc.synth_image(w, h, 1, 10, 1)
    a = hevcenc.encode(planes, **kw)
    assert a == hevcenc.encode(planes, **kw)
    assert hevcenc.encode(planes, **dict(kw, seed=2)) != a
    w, h, kw = ts.options("depth4_420_10#1")
    planes = hevcenc.synth_image(w, h, 1, 10, 1)
    assert hevcenc.encode(planes, **kw) == hevcenc.encode(planes, **dict(kw, log2_min_cb=0))


# ---- parameter sets one value past a geometry limit: the encoder's SPS / PPS with Exp-Golomb fields rewritten

def _rbsp(nal):
    out, zeros = bytearray(), 0
    for b in nal[2:]:
        if zeros >= 2 and b == 3:
            zeros = 0
            continue
        out.append(b)
        zeros = zeros + 1 if b == 0 else 0
    return nal[:2], "".join("{:08b}".format(b) for b in out)


def _nal(header, bits):
    bits = bits.rstrip("0")
    assert bits.endswith("1")                                   # rbsp_stop_one_bit
    bits += "0" * (-len(bits) % 8)
    out, zeros = bytearray(header), 0
    for i in range(0, len(bits), 8):
        b = int(bits[i:i + 8], 2)
        if zeros >= 2 and b <= 3:
            out.append(3)
            zeros = 0
        out.append(b)
        zeros = zeros + 1 if b == 0 else 0
    return bytes(out)


class _Bits:
    def __init__(self, bits):
        self.bits, self.pos, self.fields = bits, 0, {}

    def u(self, n):
        self.pos += n
        return int(self.bits[self.pos - n:self.pos], 2)

    def ue(self, name=None):
        start, lz = self.pos, 0
        while self.bits[self.pos] == "0":
            lz += 1
            self.pos += 1
        v = self.u(lz + 1) - 1
        if name:
            self.fields[name] = (start, self.pos, v)
        return v


def _sps_fields(bits):
    r = _Bits(bits)
    r.u(4)
    assert r.u(3) == 0, "one sub-layer"                        # sps_max_sub_layers_minus1
    r.u(1)
    r.u(96)                                                     # profile_tier_level(1, 0)
    r.ue()
    if r.ue() == 3:
        r.u(1)
    r.ue("pic_width_in_luma_samples")
    r.ue("pic_height_in_luma_samples")
    if r.u(1):
        for _ in range(4):
            r.ue()
    r.ue(), r.ue(), r.ue()
    assert r.u(1) == 1                                          # sub_layer_ordering_info_present_flag
    r.ue(), r.ue(), r.ue()
    for name in ("log2_min_luma_coding_block_size_minus3", "log2_diff_max_min_luma_coding_block_size",
                 "log2_min_luma_transform_block_size_minus2", "log2_diff_max_min_luma_transform_block_size",
                 "max_transform_hierarchy_depth_inter", "max_transform_hierarchy_depth_intra"):
        r.ue(name)
    return r.fields


def _pps_fields(bits):
    r = _Bits(bits)
    r.ue(), r.ue()
    r.u(7)                      # dependent_slice_segments_enabled .. cabac_init_present
    r.ue(), r.ue()
    r.ue()                      # init_qp_minus26 (se: same code length)
    r.u(2)
    if r.u(1):                  # cu_qp_delta_enabled_flag
        r.ue("diff_cu_qp_delta_depth")
    return r.fields


def _ue_bits(v):
    return "0" * ((v + 1).bit_length() - 1) + "{:b}".format(v + 1)


def rewrite(stream, changes):
    """The length-prefixed stream with SPS / PPS fields (name -> new value) rewritten, emulation prevention redone."""
    out = []
    for nal in hevcenc.split_nals(stream):
        typ = (nal[0] >> 1) & 0x3f
        if typ in (33, 34):
            header, bits = _rbsp(nal)
            fields = (_sps_fields if typ == 33 else _pps_fields)(bits)
            for name, (start, end, _) in sorted(fields.items(), key=lambda f: -f[1][0]):
                if name in changes:
                    bits = bits[:start] + _ue_bits(changes[name]) + bits[end:]
            nal = _nal(header, bits)
        out.append(len(nal).to_bytes(4, "big") + nal)
    return b"".join(out)


def fields(stream):
    nals = hevcenc.split_nals(stream)
    sps = next(n for n in nals if (n[0] >> 1) & 0x3f == 33)
    pps = next(n for n in nals if (n[0] >> 1) & 0x3f == 34)
    return {k: v[2] for k, v in list(_sps_fields(_rbsp(sps)[1]).items()) + list(_pps_fields(_rbsp(pps)[1]).items())}


# (stream, {field: value one past the limit}, message)
REFUSALS = {
    "min_tb_equals_min_cb": ("cb16_tb8_10#1", dict(log2_min_luma_transform_block_size_minus2=2,
                                                   log2_diff_max_min_luma_transform_block_size=1),
                             "SPS: min TB size must be below min CB size"),
    "max_tb_above_ctb16": ("cb16_ctb16_wpp#1", dict(log2_diff_max_min_luma_transform_block_size=3),
                           "SPS: max TB size out of range"),
    "max_tb_64": ("cb64_tb32_444_d0#1", dict(log2_diff_max_min_luma_transform_block_size=1),
                  "SPS: max TB size out of range"),
    "depth_above_ctb_minus_min_tb": ("depth4_420_10#1", dict(max_transform_hierarchy_depth_intra=5),
                                     "SPS: transform hierarchy depth out of range"),
    "width_not_multiple_of_min_cb": ("cb32_tb16_422_12#1", dict(pic_width_in_luma_samples=152),
                                     "SPS: picture size not a multiple of the min CB size"),
    "qp_delta_depth_above_ctb_minus_min_cb": ("cb32_tb16_422_12#1", dict(diff_cu_qp_delta_depth=2),
                                              "PPS: diff_cu_qp_delta_depth out of range"),
}


def test_rewrite_reproduces_the_stream():
    """With every field at its own value the rewrite gives back the encoder's bytes, and the fields are what the
    corpus asked for."""
    for name in {s for s, _, _ in REFUSALS.values()}:
        data = ts.data(name)
        f = fields(data)
        assert rewrite(data, f) == data, name
        kw = ts.options(name)[2]
        assert (f["log2_min_luma_coding_block_size_minus3"] + 3, f["log2_min_luma_transform_block_size_minus2"] + 2,
                f["max_transform_hierarchy_depth_intra"]) == (kw["log2_min_cb"], kw["log2_min_tb"], kw["max_th_depth"])


@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_geometry_past_limit_refused(case):
    """Both parsers refuse a parameter set one value past a limit of 7.4.3.2.1 / 7.4.3.3.1, and name it."""
    name, changes, message = REFUSALS[case]
    data = rewrite(ts.data(name), changes)
    got = fields(data)
    assert all(got[k] == v for k, v in changes.items())
    with pytest.raises(hb.HeifCudaError) as ei:
        hb.parse_picture(data, FMT, host_only=True)
    assert message in str(ei.value)
    with pytest.raises(hb.HeifCudaError) as ei:
        hb.K0Picture(data, FMT, host_only=True)
    assert message in str(ei.value)


# ---------------------------------------------------------------------------------------------------------------- GPU

_want_cache = {}


def oracle_planes(name, stages):
    if (name, stages) not in _want_cache:
        _want_cache[(name, stages)] = oracle_lib.reconstruct(records(name), stages)[0]
    return _want_cache[(name, stages)]


@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)   # raises if the CUDA engine is missing: no fallback
    yield e
    e.close()


@pytest.mark.gpu
def test_gpu_k0_tree_streams_in_one_batch(engine):
    """Every K0-eligible stream in one batch, at stage 0 (K0 + K1 + K2), deblocked and complete."""
    for stages in STAGES:
        got = k0_batch(engine, ts.ELIGIBLE, stages, ts.data)
        for name in ts.ELIGIBLE:
            planes, pic = got[name]
            check_planes(planes, oracle_planes(name, stages), "%s stage=%d" % (name, stages), pic)


@pytest.mark.gpu
def test_gpu_k0_tree_streams_one_per_batch(engine):
    for name in ts.ELIGIBLE:
        planes, pic = k0_batch(engine, [name], hb.STAGE_ALL, ts.data)[name]
        check_planes(planes, oracle_planes(name, hb.STAGE_ALL), "%s alone" % name, pic)


@pytest.mark.gpu
def test_gpu_mixed_batch_tree_stress_and_fixtures(engine):
    """Every stream of this corpus and of the stress corpus host-parsed and (when eligible) K0-parsed, next to the
    generated fixtures (against their reference MD5s), all in one batch."""
    import stress_streams as ss
    b = engine.batch()
    items = []
    for corpus in (ts, ss):
        for name in corpus.NAMES:
            rec = hb.parse_picture(corpus.data(name), FMT)
            c = b.add_canvas(rec.pic.crop_w, rec.pic.crop_h, rec.pic.chroma_format, rec.pic.bit_depth_y)
            b.add_picture(rec, c)
            items.append((corpus, name + " host", name, c, rec.pic, rec))
            if name in corpus.ELIGIBLE:
                k = hb.K0Picture(corpus.data(name), FMT)
                c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
                b.add_k0_picture(k, c)
                items.append((corpus, name + " K0", name, c, k.pic, k))
    for name in GEN:
        data = open(GEN_DIR + "/" + name + ".hevc", "rb").read()
        if name in DECLINED:
            r = hb.parse_picture(data, _fmt(name))
            c = b.add_canvas(r.pic.crop_w, r.pic.crop_h, r.pic.chroma_format, r.pic.bit_depth_y)
            b.add_picture(r, c)
            items.append((None, name, name, c, r.pic, r))
        else:
            k = hb.K0Picture(data, _fmt(name))
            c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
            b.add_k0_picture(k, c)
            items.append((None, name, name, c, k.pic, k))
    try:
        b.upload()
        b.reconstruct(hb.STAGE_ALL)
        bad = []
        for corpus, what, name, c, pic, _ in items:
            if corpus is None:
                if _planes_md5(b, c, pic) != GEN_META[name]["yuv_md5"]:
                    bad.append(what)
                continue
            want = oracle_planes(name, hb.STAGE_ALL) if corpus is ts else \
                oracle_lib.reconstruct(hb.parse_picture(ss.data(name), FMT, host_only=True), hb.STAGE_ALL)[0]
            planes = [b.read_plane(c, i) for i in range(3 if pic.chroma_format else 1)]
            check_planes(planes, want, what + " (mixed batch)", pic)
        assert not bad, "generated fixtures that no longer match the reference: %s" % bad
    finally:
        b.close()


def _heic_files():
    """Single images of every chroma format (K0-eligible and not) and a 2 x 2 grid of 4:4:4 min-CB-64 tiles cut by
    the canvas."""
    files = []
    for name in ("cb16_tb8_10#1", "cb32_tb16_422_12#2", "cb64_tb32_444_d0#1", "depth0_mono_12#1", "depth4_422#2",
                 "cb32_slices_dep_wpp#1", "tiles_cb32#1", "pcm_cb16#2", "bypass_cb16_444#1"):
        w, h, kw = ts.options(name)
        files.append((name, heif_writer.single_image(ts.data(name), w, h, kw.get("chroma_format", 1),
                                                     kw.get("bit_depth", 8))))
    w, h, _ = ts.options("cb64_tb32_444_d0#1")
    tiles = [ts.data("cb64_tb32_444_d0#%d" % s) for s in (1, 2, 3, 4)]
    files.append(("grid cb64_tb32_444_d0#1..4", heif_writer.grid_image(tiles, 2, 2, w, h, 2 * w - 24, 2 * h - 18,
                                                                       chroma_format=3)))
    return files


@pytest.mark.gpu
@pytest.mark.parametrize("host_share", [0, 100])
@pytest.mark.parametrize("out_format", [hb.OUT_YCBCR, hb.OUT_RGB])
def test_gpu_stream_of_tree_heic(engine, host_share, out_format):
    """HEIC files of this corpus through decode_stream, device-parsed (host share 0, where eligible) and host-parsed
    (100), as native planes (against the oracle's planes) and as RGB (against heic_oracle.decode_rgb)."""
    files = _heic_files()
    want = {}
    for i, (_, data) in enumerate(files):
        if out_format == hb.OUT_YCBCR:
            planes, _, _, bd, _ = heic_oracle.decode_planes(data)
            dt = np.uint8 if bd == 8 else np.dtype("<u2")
            want[i] = hashlib.md5(b"".join(p.astype(dt).tobytes() for p in planes)).hexdigest()
        else:
            want[i] = hashlib.md5(np.ascontiguousarray(heic_oracle.decode_rgb(data, out_format)).tobytes()).hexdigest()
    seen = {}

    def on_image(index, desc, out):
        if out_format == hb.OUT_YCBCR:
            seen[index] = hashlib.md5(b"".join(np.ascontiguousarray(p).tobytes() for p in out)).hexdigest()
        else:
            seen[index] = hashlib.md5(np.ascontiguousarray(out[:, :desc.width * desc.bytes_per_pixel]).tobytes()).hexdigest()
    engine.set_option("host_share_pct", host_share)
    try:
        hb.decode_stream(engine, [d for _, d in files], on_image, threads=2, files_per_batch=4, out_format=out_format)
    finally:
        engine.set_option("host_share_pct", -1)
    assert sorted(seen) == list(range(len(files)))
    bad = [files[i][0] for i in seen if seen[i] != want[i]]
    assert not bad, "differ from the oracle: %s" % bad
