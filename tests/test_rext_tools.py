"""The HEVC range-extension coding tools from bitstream to pixels: the synthetic-content encoder writes them
(rext_streams.py), both parsers read them, K0, K1 and K2 implement them, and the oracle restates them.

CPU: every stream carries what the encoder meant (the oracle on the host parser's records equals the encoder's own
reconstruction); the CPU build of K0 equals the host parser record for record on every stream it takes and declines the
others for the right reason; the three tools the decoder does not implement are refused by name; the encoder's counters
and the records prove the corpus reaches every tool; and a plain int64 restatement of the residual rules of H.265
(transform-skip shift, rotation, RDPCM accumulation, the scaling factor of transform-skipped blocks) agrees with the
oracle's residual on every transform-skipped and bypass block of the corpus, except in the one case named below.
GPU: the device K0 + K1..K5 against the oracle in batches of every shape and through the stream API."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import heic_oracle
import heif_b200 as hb
import oracle_lib
import record_mutation as rm
import rext_streams as rs
from test_k0_parser import DECLINED, GEN, GEN_DIR, GEN_META, _fmt, _planes_md5, check_equal
from test_syntax_extremes import check_planes, first_diff

from tools import heif_writer, hevcenc  # noqa: E402

FMT = hb.STREAM_LENGTH_PREFIXED
STAGES = (0, hb.STAGE_DEBLOCK, hb.STAGE_ALL)
TB_DST, TB_TSKIP, TB_BYPASS, TB_RDPCM_H, TB_RDPCM_V, TB_ROTATE = 0x04, 0x08, 0x10, 0x20, 0x40, 0x80
BLK_NO_EDGE_FLT, PIC_NO_INTRA_SMOOTH, PIC_SCALING_LIST = 0x04, 0x0002, 0x0010
# encoder counters of tools the device parser takes: reached by the K0-eligible streams alone
DEVICE_COUNTERS = (["rdpcm_h_tskip", "rdpcm_v_tskip", "rotate_tskip", "sig_ctx_42", "sig_ctx_43", "sdh_off_rdpcm",
                    "sao_offset_scaled_cmax", "smoothing_skipped", "smoothing_skipped_strong"] +
                   ["tskip_log2_%d" % k for k in range(4)])


def records(name):
    return hb.parse_picture(rs.data(name), FMT, host_only=True)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", rs.NAMES)
def test_rext_stream_round_trip(name):
    """The oracle's pre-filter planes from the host parser's records equal the encoder's reconstruction."""
    data, extra = rs.stream(name)
    got, _ = oracle_lib.reconstruct(records(name), 0)
    for k, (g, r) in enumerate(zip(got, extra["recon"])):
        n, at = first_diff(g, r[:g.shape[0], :g.shape[1]])
        assert n == 0, "%s plane %d: %d samples differ from the encoder's reconstruction, first at (y,x)=%s" % (name, k, n, at)


@pytest.mark.parametrize("name", rs.ELIGIBLE)
def test_k0_records_equal_host_parser_rext(name):
    check_equal(rs.data(name), FMT)


@pytest.mark.parametrize("name", rs.DECLINED)
def test_k0_declines_rext_stream(name):
    k = hb.K0Picture(rs.data(name), FMT, host_only=True)
    assert not k.eligible
    assert k.why_not == rs.K0_DECLINED[name.split("#")[0]], k.why_not


@pytest.mark.parametrize("name", rs.REFUSED_NAMES)
def test_refused_rext_stream(name):
    """Both parsers refuse a stream with a tool the decoder does not implement, and the message names it."""
    flag = rs.REFUSED[name.split("#")[0]][3]
    with pytest.raises(hb.HeifCudaError) as ei:
        hb.parse_picture(rs.data(name), FMT, host_only=True)
    assert flag in str(ei.value)
    with pytest.raises(hb.HeifCudaError) as ei:
        hb.K0Picture(rs.data(name), FMT, host_only=True)
    assert flag in str(ei.value)


def test_rext_corpus_reaches_every_tool():
    """Every range-extension counter of the encoder is > 0 over the corpus, and the ones of tools the device parser
    takes are > 0 over the K0-eligible streams alone."""
    total = dict.fromkeys(hevcenc.rext_stat_names(), 0)
    device = dict.fromkeys(DEVICE_COUNTERS, 0)
    for name in rs.NAMES:
        st = rs.stream(name)[1]["rext_stats"]
        for k in total:
            total[k] += st[k]
        if name in rs.ELIGIBLE:
            for k in device:
                device[k] += st[k]
    assert set(DEVICE_COUNTERS) <= set(total)
    assert not [k for k, v in total.items() if v == 0], total
    assert not [k for k, v in device.items() if v == 0], device
    # RDPCM accumulation that leaves the int16 range of the residual buffer, in a device-parsed picture
    oracle_lib.counters_reset()
    for name in rs.ELIGIBLE:
        oracle_lib.reconstruct(records(name), 0)
    assert oracle_lib.counters()["k1_rdpcm_clip"] > 0


def test_stress_corpus_writes_no_range_extension_tool():
    """With the range-extension options at 0 (the stress corpus) none of these tools is written; 4x4 transform skip
    needs no extension."""
    import stress_streams as ss
    for name in ss.NAMES:
        st = ss.stream(name)[1]["rext_stats"]
        assert not [k for k, v in st.items() if v and k != "tskip_log2_0"], name


def test_rext_records_carry_the_tools():
    types, blk_flags, pic_flags, tskip_log2, sao = [], [], 0, set(), set()
    for name in rs.NAMES:
        rec = records(name)
        v = rm.views(rec)
        types.append(v["tbs"]["type"].copy())
        blk_flags.append(v["blks"]["flags"][v["blks"]["cidx"] == 0].copy())
        pic_flags |= rec.pic.flags
        tskip_log2 |= set(v["tbs"]["log2"][(v["tbs"]["type"] & TB_TSKIP) != 0].tolist())
        base, _ = name.split("#")
        kw = rs.options(name)[2]
        scale = (kw.get("log2_sao_offset_scale_luma", 0), kw.get("log2_sao_offset_scale_chroma", 0))
        for c in range(3):
            if scale[min(c, 1)]:
                sao.update(("%s c%d" % (base, c), int(o)) for o in v["ctus"]["sao_offset"][:, c, :].reshape(-1)
                           if abs(int(o)) == 31 << scale[min(c, 1)])
    t = np.concatenate(types)
    for bit in (TB_RDPCM_H, TB_RDPCM_V, TB_ROTATE):
        assert ((t & bit) != 0).any(), hex(bit)
    assert (((t & (TB_RDPCM_H | TB_RDPCM_V | TB_ROTATE)) != 0) & ((t & (TB_TSKIP | TB_BYPASS)) == 0)).sum() == 0
    assert {3, 4, 5} <= tskip_log2, tskip_log2
    assert (np.concatenate(blk_flags) & BLK_NO_EDGE_FLT).any()
    assert pic_flags & PIC_NO_INTRA_SMOOTH
    assert any(o > 0 for _, o in sao) and any(o < 0 for _, o in sao), sorted(sao)


def _chroma_qp_without_cu_offset(rec, v):
    """Per coded non-bypass chroma TB: (qp in the record, qP' the TB would have without CuQpOffsetCb / Cr)."""
    pic = rec.pic
    sw = 2 if pic.chroma_format in (1, 2) else 1
    sh = 2 if pic.chroma_format == 1 else 1
    off = 6 * (pic.bit_depth_y - 8)
    blk_of = {int(b["resid_off"]): b for b in v["blks"] if b["flags"] & 0x02}
    w8 = pic.width >> 3
    out = []
    for tb in v["tbs"]:
        c = tb["type"] & 3
        if not c or tb["type"] & TB_BYPASS:
            continue
        b = blk_of[int(tb["resid_off"])]
        qpy = int(v["qp_map"][((b["y"] * sh) >> 3) * w8 + ((b["x"] * sw) >> 3)])
        qpi = min(57, max(-off, qpy + (pic.pps_cb_qp_offset if c == 1 else pic.pps_cr_qp_offset)))
        if pic.chroma_format == 1:
            qpi = qpi if qpi < 30 else qpi - 6 if qpi >= 44 else (29, 30, 31, 32, 33, 33, 34, 34, 35, 35, 36, 36, 37, 37)[qpi - 30]
        out.append((int(tb["qp"]), max(0, qpi + off)))
    return out


def test_rext_chroma_qp_carries_cu_offsets():
    """Chroma TBs of the streams with CU chroma QP offset lists take qP' shifted by the offsets; the same derivation
    without offsets holds for every other stream."""
    shifted = 0
    for name in rs.NAMES:
        rec = records(name)
        pairs = _chroma_qp_without_cu_offset(rec, rm.views(rec))
        n = sum(got != want for got, want in pairs)
        if rs.options(name)[2].get("chroma_qp_offset_list_len"):
            shifted += n
        else:
            assert n == 0, name
    assert shifted > 0


def test_no_edge_filter_lookup_position():
    """disableIntraBoundaryFilter: the records flag a chroma block by the bypass flag at its component coordinates
    in the luma CU map (the reference's lookup), which in 4:2:0 and 4:2:2 can be another CU than the one H.265 means.
    The flag only switches the luma edge filters, so the planes are the same under either rule (DESIGN 4)."""
    differ = 0
    for name in rs.NAMES:
        kw = rs.options(name)[2]
        if not (kw.get("transquant_bypass") and kw.get("implicit_rdpcm")) or kw.get("chroma_format", 1) not in (1, 2):
            continue
        rec = records(name)
        v = rm.views(rec)
        pic = rec.pic
        sw, sh = 2, 2 if pic.chroma_format == 1 else 1
        edge = v["edge_map"].reshape(pic.height >> 2, pic.width >> 2)
        bypass = (edge[::2, ::2] & 0x08) != 0           # per 8x8 luma unit (edge_map: HC_EDGE_BYPASS per 4x4)
        b = v["blks"]
        ch = b["cidx"] > 0
        spec = bypass[(b["y"][ch].astype(int) * sh) >> 3, (b["x"][ch].astype(int) * sw) >> 3]
        quirk = (b["flags"][ch] & BLK_NO_EDGE_FLT) != 0
        assert np.array_equal(quirk, bypass[np.minimum(b["y"][ch], pic.height - 1) >> 3,
                                            np.minimum(b["x"][ch], pic.width - 1) >> 3]), name
        differ += int((spec != quirk).sum())
        want, _ = oracle_lib.reconstruct(rec, hb.STAGE_ALL)
        b["flags"][ch] = np.where(spec, b["flags"][ch] | BLK_NO_EDGE_FLT, b["flags"][ch] & np.uint8(0xff ^ BLK_NO_EDGE_FLT))
        got, _ = oracle_lib.reconstruct(rec, hb.STAGE_ALL)
        for g, w in zip(got, want):
            assert np.array_equal(g, w), name
    assert differ > 0, "no chroma block where the two lookups pick different CUs"


# ---- an independent restatement of the residual rules (H.265 8.6.2, 8.6.4.2, 8.6.8 in the version with the range
# extensions), plain numpy in int64

LEVEL_SCALE = (40, 45, 51, 57, 64, 72)


def restate_residual(pic, tb, levels, scaling, tskip_factor_16):
    """Residual r of one transform-skipped or bypass block. levels: nT x nT TransCoeffLevel. tskip_factor_16: H.265's
    m = 16 for transform-skipped blocks larger than 4 x 4 (False: m from the scaling list, as the reference)."""
    log2 = int(tb["log2"])
    n = 1 << log2
    typ = int(tb["type"])
    bit_depth = pic.bit_depth_y if (typ & 3) == 0 else pic.bit_depth_c
    if typ & TB_BYPASS:
        r = levels.astype(np.int64)
        if typ & TB_ROTATE:
            r = r[::-1, ::-1]
    else:
        qp = int(tb["qp"])
        if not (pic.flags & PIC_SCALING_LIST) or (tskip_factor_16 and n > 4):
            m = np.full((n, n), 16, np.int64)
        else:
            start = {2: 0, 3: 96, 4: 96 + 384, 5: 96 + 384 + 1536}[log2]
            size = n * n
            mid = int(tb["matrix_id"]) if log2 < 5 else (1 if tb["matrix_id"] else 0)
            m = scaling[start + mid * size:start + (mid + 1) * size].astype(np.int64).reshape(n, n)
        bd_shift = bit_depth + log2 - 5
        fact = LEVEL_SCALE[qp % 6] << (qp // 6)
        if pic.flags & PIC_SCALING_LIST:
            d = (levels.astype(np.int64) * m * fact + (1 << (bd_shift - 1))) >> bd_shift
        else:
            # m = 16 taken out of the product, which the reference forms in int32 and lets wrap (DESIGN 4, quirks)
            t = levels.astype(np.int64) * fact + (1 << (bd_shift - 5))
            d = (((t + (1 << 31)) % (1 << 32)) - (1 << 31)) >> (bd_shift - 4)
        d = np.clip(d, -32768, 32767)
        if typ & TB_ROTATE:
            d = d[::-1, ::-1]
        ts_shift, bd2 = 5 + log2, max(20 - bit_depth, 0)
        r = ((d << ts_shift) + (1 << (bd2 - 1) if bd2 else 0)) >> bd2
    if typ & TB_RDPCM_H:
        r = np.cumsum(r, axis=1)
    elif typ & TB_RDPCM_V:
        r = np.cumsum(r, axis=0)
    return r


def test_residual_restatement_matches_oracle():
    """The restatement equals hc_oracle_residual_block on every transform-skipped and bypass block of the corpus.
    Named disagreement: transform-skipped blocks larger than 4 x 4 in a picture with scaling lists, where H.265 takes
    m = 16 and the oracle, K1 and the reference take the scaling list's factor (DESIGN 4); the restatement is run
    with both rules there and the case must be reached."""
    O = oracle_lib.lib()
    res = np.zeros(1024, np.int32)
    checked, factor_cases, kinds = 0, 0, set()
    for name in rs.NAMES:
        rec = records(name)
        pic = rec.pic
        v = rm.views(rec)
        scaling = v["scaling"]
        sc_ptr = C.c_void_p(rec.array("scaling")[0]) if len(scaling) else None
        coeffs = v["coeffs"]
        for tb in v["tbs"]:
            if not int(tb["type"]) & (TB_TSKIP | TB_BYPASS):
                continue
            n = 1 << int(tb["log2"])
            co = coeffs[int(tb["coeff_off"]):int(tb["coeff_off"]) + int(tb["ncoeff"])]
            levels = np.zeros(n * n, np.int64)
            levels[co["pos"].astype(np.int64)] = co["level"]
            levels = levels.reshape(n, n)
            tbc = np.array([tb], rm.TB)
            cc = np.ascontiguousarray(co)
            O.hc_oracle_residual_block(C.byref(pic), C.c_void_p(tbc.ctypes.data), C.c_void_p(cc.ctypes.data), sc_ptr,
                                       C.c_void_p(res.ctypes.data))
            got = res[:n * n].reshape(n, n).astype(np.int64)
            want = restate_residual(pic, tb, levels, scaling, tskip_factor_16=False)
            assert np.array_equal(got, want), (name, tb)
            h265 = restate_residual(pic, tb, levels, scaling, tskip_factor_16=True)
            if not np.array_equal(h265, want):
                assert (pic.flags & PIC_SCALING_LIST) and (int(tb["type"]) & TB_TSKIP) and n > 4, (name, tb)
                factor_cases += 1
            checked += 1
            kinds.add((int(tb["type"]) & (TB_TSKIP | TB_BYPASS | TB_RDPCM_H | TB_RDPCM_V | TB_ROTATE), n))
    assert factor_cases > 0
    for k in (TB_TSKIP | TB_RDPCM_H, TB_TSKIP | TB_RDPCM_V, TB_TSKIP | TB_ROTATE, TB_BYPASS | TB_ROTATE,
              TB_BYPASS | TB_RDPCM_H, TB_BYPASS | TB_RDPCM_V):
        assert any(t & k == k for t, _ in kinds), hex(k)
    assert {n for t, n in kinds if t & TB_RDPCM_V} >= {8, 16}, kinds


def test_rext_is_deterministic_and_off_by_default():
    """Same seed, same bytes; with every range-extension option at 0 the SPS and PPS carry no extension."""
    w, h, kw = rs.options("ts_422_10_wpp#1")
    planes = hevcenc.synth_image(w, h, 2, 10, 1)
    a = hevcenc.encode(planes, **kw)
    assert a == hevcenc.encode(planes, **kw)
    assert hevcenc.encode(planes, **dict(kw, seed=2)) != a
    plain = {k: v for k, v in kw.items() if k not in hevcenc.FIELDS[hevcenc.FIELDS.index("transform_skip_rotation"):]}
    rec = hb.parse_picture(hevcenc.encode(planes, **plain), FMT, host_only=True)
    v = rm.views(rec)
    assert not (v["tbs"]["type"] & (TB_RDPCM_H | TB_RDPCM_V | TB_ROTATE)).any()
    assert not (rec.pic.flags & PIC_NO_INTRA_SMOOTH)


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


def k0_batch(engine, names, stages):
    b = engine.batch()
    items = []
    for name in names:
        k = hb.K0Picture(rs.data(name), FMT)
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
def test_gpu_k0_rext_streams_in_one_batch(engine):
    """Every K0-eligible range-extension stream in one batch, at stage 0 (K0 + K1 + K2), deblocked and complete."""
    for stages in STAGES:
        got = k0_batch(engine, rs.ELIGIBLE, stages)
        for name in rs.ELIGIBLE:
            planes, pic = got[name]
            check_planes(planes, oracle_planes(name, stages), "%s stage=%d" % (name, stages), pic)


@pytest.mark.gpu
def test_gpu_k0_rext_streams_one_per_batch(engine):
    for name in rs.ELIGIBLE:
        planes, pic = k0_batch(engine, [name], hb.STAGE_ALL)[name]
        check_planes(planes, oracle_planes(name, hb.STAGE_ALL), "%s alone" % name, pic)


@pytest.mark.gpu
def test_gpu_mixed_batch_rext_and_fixtures(engine):
    """Every range-extension stream host-parsed and (when eligible) K0-parsed, next to the 47 generated fixtures,
    all in one batch."""
    b = engine.batch()
    items = []
    for name in rs.NAMES:
        rec = hb.parse_picture(rs.data(name), FMT)
        c = b.add_canvas(rec.pic.crop_w, rec.pic.crop_h, rec.pic.chroma_format, rec.pic.bit_depth_y)
        b.add_picture(rec, c)
        items.append(("rext", name + " host", name, c, rec.pic, rec))
        if name in rs.ELIGIBLE:
            k = hb.K0Picture(rs.data(name), FMT)
            c = b.add_canvas(k.pic.crop_w, k.pic.crop_h, k.pic.chroma_format, k.pic.bit_depth_y)
            b.add_k0_picture(k, c)
            items.append(("rext", name + " K0", name, c, k.pic, k))
    for name in GEN:
        data = open(GEN_DIR + "/" + name + ".hevc", "rb").read()
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


HEIC_NAMES = ("ts32_420_8#1", "ts_422_10_wpp#2", "nosmooth_444_12#1", "mono_12_sao2#1", "scaling_ts32_422#1",
              "dense_rdpcm_12#2", "odd_ctb32_444#1", "bypass_422#1", "rice_wpp_dep#1", "cqo_lists#2")


def _heic(name):
    w, h, kw = rs.options(name)
    return heif_writer.single_image(rs.data(name), w, h, kw.get("chroma_format", 1), kw.get("bit_depth", 8))


@pytest.mark.gpu
@pytest.mark.parametrize("host_share", [0, 100])
@pytest.mark.parametrize("out_format", [hb.OUT_YCBCR, hb.OUT_RGB])
def test_gpu_stream_of_rext_heic(engine, host_share, out_format):
    """HEIC files of range-extension streams through decode_stream, device-parsed (host share 0, where eligible) and
    host-parsed (100), as native planes (against the oracle's planes) and as RGB (against heic_oracle.csc). A refused
    file in the middle of the stream reports its error and every other file is still delivered bit-exact."""
    names = list(HEIC_NAMES[:5]) + ["extended_precision#1"] + list(HEIC_NAMES[5:])
    files = [_heic(n) for n in names]
    refused = names.index("extended_precision#1")
    want = {}
    for i, data in enumerate(files):
        if i == refused:
            continue
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
        st = hb.decode_stream(engine, files, on_image, threads=2, files_per_batch=4, out_format=out_format,
                              isolate_errors=True)
    finally:
        engine.set_option("host_share_pct", -1)
    assert [k for k, v in enumerate(st["file_status"]) if v != 0] == [refused], st["file_status"]
    assert "extended_precision_processing_flag" in st["first_error"], st["first_error"]
    assert sorted(seen) == [i for i in range(len(files)) if i != refused]
    bad = [names[i] for i in seen if seen[i] != want[i]]
    assert not bad, "differ from the oracle: %s" % bad
