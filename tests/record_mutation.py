"""Seeded mutation of one picture's records (include/heifcuda_records.h), in place.

The bundled and generated streams are natural content at moderate QP, so the value-dependent branches of the
kernels (int32 wrap and int16 clips of K1, clipping of the residual add, strong intra smoothing, the deblocking
decisions and table clamps, SAO band wrap and offset extremes) are reached by chance or not at all. mutate()
rewrites the values inside the records, never their layout, so that the oracle and the kernels can be compared on
content pushed to the limits of the legal ranges. Every value it writes is one a conforming bitstream could
produce for the same block structure; check_legal() asserts those ranges.

Test infrastructure (tests/test_record_extremes.py)."""
import ctypes as C
import zlib

import numpy as np

COEFF = np.dtype([("pos", "<u2"), ("level", "<i2")])
TB = np.dtype([("coeff_off", "<u4"), ("resid_off", "<u4"), ("ncoeff", "<u2"), ("pic", "<u2"), ("log2", "u1"), ("qp", "u1"),
               ("type", "u1"), ("matrix_id", "u1")])
BLK = np.dtype([("x", "<u2"), ("y", "<u2"), ("log2", "u1"), ("mode", "u1"), ("flags", "u1"), ("cidx", "u1"),
                ("avail_left", "<u2"), ("avail_top", "<u2"), ("resid_off", "<u4")])
CTU = np.dtype([("blk_first", "<u4", 3), ("blk_count", "<u2", 3), ("sao_type", "u1", 3), ("sao_band_or_class", "u1", 3),
                ("sao_offset", "i1", (3, 4)), ("beta_offset", "i1"), ("tc_offset", "i1"), ("sao_nb", "u1"), ("flags", "u1"),
                ("sao_nb_c", "u1"), ("pad", "u1", 3)])
assert (COEFF.itemsize, TB.itemsize, BLK.itemsize, CTU.itemsize) == (4, 16, 16, 44)
assert TB.fields["qp"][1] == 13 and BLK.fields["mode"][1] == 5 and CTU.fields["sao_type"][1] == 18
assert CTU.fields["sao_offset"][1] == 24 and CTU.fields["beta_offset"][1] == 36 and CTU.fields["tc_offset"][1] == 37

TB_CIDX, TB_BYPASS, TB_RDPCM = 0x03, 0x10, 0x60
BLK_HAS_RESID, BLK_PCM = 0x02, 0x08
EDGE_V, EDGE_H = 0x01, 0x02
PIC_HAS_DEBLOCK, PIC_HAS_SAO, PIC_SCALING_LIST = 0x0004, 0x0008, 0x0010
# host/hevc_parse.cc kMode422: 4:2:2 chroma intra modes after the remapping of H.265 Table 8-3
MODE_422 = (0, 1, 2, 2, 2, 2, 3, 5, 7, 8, 10, 12, 13, 15, 17, 18, 19, 20, 21, 22, 23, 23, 24, 24, 25, 25, 26, 27, 27, 28, 28,
            29, 29, 30, 31)
MODES_422 = np.array(sorted(set(MODE_422)), np.uint8)
FLAT_MODES = np.array([0, 1, 10, 26], np.uint8)   # planar, DC, pure horizontal, pure vertical: all in the 4:2:2 image
FAMILIES = ("levels", "modes", "flat", "filters", "all")


def views(rec):
    """Writable numpy views of the record arrays of one picture (the parser's own vectors)."""
    out = {}
    for name, dt in (("coeffs", COEFF), ("tbs", TB), ("blks", BLK), ("ctus", CTU), ("edge_map", np.uint8),
                     ("qp_map", np.int8), ("scaling", np.uint8)):
        p, n = rec.array(name)
        dt = np.dtype(dt)
        if not n or not p:
            out[name] = np.zeros(0, dt)
            continue
        raw = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n * dt.itemsize,))
        out[name] = raw.view(dt)
    return out


def _qp_bd_offsets(pic):
    return 6 * (pic.bit_depth_y - 8), 6 * (pic.bit_depth_c - 8)


def _pcm_tbs(v):
    """Transform blocks that carry PCM samples (a PCM hc_blk points at their residual)."""
    pcm_off = v["blks"]["resid_off"][(v["blks"]["flags"] & BLK_PCM) != 0]
    return np.isin(v["tbs"]["resid_off"], pcm_off)


def _tb_of_coeff(tbs, ncoeffs):
    idx = np.full(ncoeffs, -1, np.int64)
    lens = tbs["ncoeff"].astype(np.int64)
    t = np.repeat(np.arange(len(tbs)), lens)
    within = np.arange(len(t)) - np.repeat(np.cumsum(lens) - lens, lens)
    idx[tbs["coeff_off"][t].astype(np.int64) + within] = t
    return idx


def _mutable_blocks(v, pic):
    """Non-PCM blocks whose mode may change: a block coded with implicit RDPCM keeps the mode that selected it."""
    b = v["blks"]
    rdpcm_off = v["tbs"]["resid_off"][(v["tbs"]["type"] & TB_RDPCM) != 0]
    keep = ((b["flags"] & BLK_PCM) != 0) | (((b["flags"] & BLK_HAS_RESID) != 0) & np.isin(b["resid_off"], rdpcm_off))
    return ~keep


def _levels(v, pic, rng, tb_mask):
    tbs, co = v["tbs"], v["coeffs"]
    sel = tb_mask & ~_pcm_tbs(v)
    owner = _tb_of_coeff(tbs, len(co))
    cmask = (owner >= 0) & sel[np.maximum(owner, 0)]
    n = int(cmask.sum())
    kind = rng.integers(0, 5, n)
    lv = np.select([kind == 0, kind == 1, kind == 2, kind == 3], [1, -1, 32767, -32768], rng.integers(-32768, 32768, n))
    co["level"][cmask] = lv.astype(np.int16)
    off_y, off_c = _qp_bd_offsets(pic)
    cidx = tbs["type"] & TB_CIDX
    hi = np.where(cidx == 0, 51 + off_y, 51 + off_c)
    q = rng.integers(0, hi + 1)
    tbs["qp"][sel] = q[sel].astype(np.uint8)
    if (pic.flags & PIC_SCALING_LIST) and len(v["scaling"]):
        v["scaling"][:] = _scaling_blob(rng)


def _scaling_blob(rng):
    """ScalingFactor arrays (H.265 7.4.5) from random scaling lists: 4x4 and 8x8 lists as coded, 16x16 and 32x32
    upsampled from an 8x8 list with their own DC value; every entry in 1..255."""
    parts = [rng.integers(1, 256, (6, 16)), rng.integers(1, 256, (6, 64))]
    for count, rep in ((6, 2), (2, 4)):
        m = rng.integers(1, 256, (count, 8, 8)).repeat(rep, 1).repeat(rep, 2)
        m[:, 0, 0] = rng.integers(1, 256, count)
        parts.append(m.reshape(count, -1))
    return np.concatenate([p.reshape(-1) for p in parts]).astype(np.uint8)


def _flat(v, pic, rng, tb_mask, blk_mask):
    tbs, co = v["tbs"], v["coeffs"]
    sel = tb_mask & ~_pcm_tbs(v)
    owner = _tb_of_coeff(tbs, len(co))
    cmask = (owner >= 0) & sel[np.maximum(owner, 0)]
    co["level"][cmask] = np.where(co["pos"][cmask] == 0, rng.integers(-2, 3, int(cmask.sum())), 0).astype(np.int16)
    b = v["blks"]
    m = blk_mask & _mutable_blocks(v, pic)
    b["mode"][m] = rng.choice(FLAT_MODES, int(m.sum()))


def _modes(v, pic, rng, blk_mask):
    b = v["blks"]
    m = blk_mask & _mutable_blocks(v, pic)
    new = rng.integers(0, 35, len(b)).astype(np.uint8)
    if pic.chroma_format == 2:
        c = b["cidx"] != 0
        new[c] = rng.choice(MODES_422, int(c.sum()))
    b["mode"][m] = new[m]


def _sao_offset_max(bd):
    return (1 << (min(bd, 10) - 5)) - 1


def _filters(v, pic, rng):
    ctus = v["ctus"]
    n = len(ctus)
    ctus["beta_offset"] = 2 * rng.integers(-6, 7, n)
    ctus["tc_offset"] = 2 * rng.integers(-6, 7, n)
    ncomp = 3 if pic.chroma_format else 1
    # log2_sao_offset_scale_luma / _chroma (PPS range extension): 0..max(0, bitDepth - 10)
    scale = [int(rng.integers(0, max(0, pic.bit_depth_y - 10) + 1)), int(rng.integers(0, max(0, pic.bit_depth_c - 10) + 1))]
    for c in range(ncomp):
        bd = pic.bit_depth_y if c == 0 else pic.bit_depth_c
        if c == 2:   # Cr shares Cb's SAO type and edge class (sao_type_idx_chroma, sao_eo_class_chroma)
            typ = ctus["sao_type"][:, 1].copy()
            cls = ctus["sao_band_or_class"][:, 1].copy()
        else:
            typ = rng.integers(0, 3, n)
            cls = rng.integers(0, 4, n)
        band = np.where(rng.random(n) < 0.5, rng.integers(28, 32, n), rng.integers(0, 32, n))
        mag = rng.integers(0, _sao_offset_max(bd) + 1, (n, 4))
        sign = np.where(rng.random((n, 4)) < 0.5, -1, 1)
        band_off = sign * mag
        edge_off = mag * np.array([1, 1, -1, -1])
        off = np.where((typ == 1)[:, None], band_off, np.where((typ == 2)[:, None], edge_off, 0)) << scale[min(c, 1)]
        ctus["sao_type"][:, c] = typ
        ctus["sao_band_or_class"][:, c] = np.where(typ == 1, band, np.where(typ == 2, cls, 0))
        ctus["sao_offset"][:, c, :] = off.astype(np.int8)
    off_y = 6 * (pic.bit_depth_y - 8)
    v["qp_map"][:] = rng.integers(-off_y, 52, len(v["qp_map"])).astype(np.int8)
    w4, h4 = pic.width >> 2, pic.height >> 2
    e = v["edge_map"].reshape(h4, w4)
    flip = rng.integers(0, 4, e.shape).astype(np.uint8) & _edge_allowed(w4, h4)
    e ^= flip


def _edge_allowed(w4, h4):
    """Edge bits a unit may carry: vertical edges on interior columns, horizontal edges on interior rows of the 8x8 grid."""
    ux, uy = np.arange(w4), np.arange(h4)
    v = ((ux % 2 == 0) & (ux > 0))[None, :].astype(np.uint8) * EDGE_V
    h = ((uy % 2 == 0) & (uy > 0))[:, None].astype(np.uint8) * EDGE_H
    return (v | h).astype(np.uint8)


def _update_pic_flags(v, pic):
    ncomp = 3 if pic.chroma_format else 1
    flags = pic.flags & ~(PIC_HAS_DEBLOCK | PIC_HAS_SAO)
    if np.any(v["edge_map"] & (EDGE_V | EDGE_H)):
        flags |= PIC_HAS_DEBLOCK
    if np.any(v["ctus"]["sao_type"][:, :ncomp]):
        flags |= PIC_HAS_SAO
    pic.flags = flags


def mutate(rec, family, seed):
    """Rewrites the values of one picture's records in place (family: one of FAMILIES). Deterministic in (family, seed)."""
    if family not in FAMILIES:
        raise ValueError(family)
    rng = np.random.default_rng([seed, zlib.crc32(family.encode())])
    v = views(rec)
    pic = rec.pic
    ntb, nblk = len(v["tbs"]), len(v["blks"])
    if family == "levels":
        _levels(v, pic, rng, np.ones(ntb, bool))
    elif family == "modes":
        _modes(v, pic, rng, np.ones(nblk, bool))
    elif family == "flat":
        _flat(v, pic, rng, np.ones(ntb, bool), np.ones(nblk, bool))
    elif family == "filters":
        _filters(v, pic, rng)
    else:   # every family at once: each block and transform block is either extreme or flat
        flat_tb, flat_blk = rng.random(ntb) < 0.3, rng.random(nblk) < 0.3
        _levels(v, pic, rng, ~flat_tb)
        _modes(v, pic, rng, ~flat_blk)
        _flat(v, pic, rng, flat_tb, flat_blk)
        _filters(v, pic, rng)
    _update_pic_flags(v, pic)


def check_legal(rec):
    """Asserts that the records hold values a conforming bitstream could produce (the ranges mutate() draws from)."""
    v = views(rec)
    pic = rec.pic
    off_y, off_c = _qp_bd_offsets(pic)
    ncomp = 3 if pic.chroma_format else 1
    tbs, blks, ctus = v["tbs"], v["blks"], v["ctus"]
    cidx = tbs["type"] & TB_CIDX
    assert np.all(tbs["qp"] <= np.where(cidx == 0, 51 + off_y, 51 + off_c)), "qP' above 51 + QpBdOffset"
    pcm = _pcm_tbs(v)
    owner = _tb_of_coeff(tbs, len(v["coeffs"]))
    in_pcm = (owner >= 0) & pcm[np.maximum(owner, 0)]
    bd_of = np.where(cidx == 0, pic.bit_depth_y, pic.bit_depth_c)
    lv = v["coeffs"]["level"][in_pcm].astype(np.int64)
    assert np.all((lv >= 0) & (lv < (1 << bd_of[owner[in_pcm]]))), "PCM sample outside the sample range"
    assert np.all(blks["mode"] <= 34), "intra mode above 34"
    if pic.chroma_format == 2:
        assert np.all(np.isin(blks["mode"][blks["cidx"] != 0], MODES_422)), "4:2:2 chroma mode outside the image of Table 8-3"
    if (pic.flags & PIC_SCALING_LIST) and len(v["scaling"]):
        assert np.all(v["scaling"] >= 1), "scaling factor 0"
    assert np.all(ctus["beta_offset"] % 2 == 0) and np.all(np.abs(ctus["beta_offset"].astype(int)) <= 12), "beta offset"
    assert np.all(ctus["tc_offset"] % 2 == 0) and np.all(np.abs(ctus["tc_offset"].astype(int)) <= 12), "tc offset"
    typ, boc, off = ctus["sao_type"], ctus["sao_band_or_class"], ctus["sao_offset"].astype(int)
    assert np.all(typ[:, :ncomp] <= 2), "SAO type"
    if ncomp == 3:
        assert np.all(typ[:, 1] == typ[:, 2]), "Cb and Cr SAO types differ"
        edge = typ[:, 1] == 2
        assert np.all(boc[edge, 1] == boc[edge, 2]), "Cb and Cr edge classes differ"
    for c in range(ncomp):
        bd = pic.bit_depth_y if c == 0 else pic.bit_depth_c
        lim = _sao_offset_max(bd) << max(0, bd - 10)
        t = typ[:, c]
        assert np.all(boc[t == 1, c] <= 31) and np.all(boc[t == 2, c] <= 3), "band position / edge class"
        assert np.all(np.abs(off[:, c]) <= lim), "SAO offset magnitude"
        assert np.all(off[t == 0, c] == 0), "offsets of a component without SAO"
        eo = off[t == 2, c]
        assert np.all(eo[:, :2] >= 0) and np.all(eo[:, 2:] <= 0), "edge offset signs"
    assert np.all((v["qp_map"] >= -off_y) & (v["qp_map"] <= 51)), "QP_Y outside -QpBdOffsetY..51"
    w4, h4 = pic.width >> 2, pic.height >> 2
    e = v["edge_map"].reshape(h4, w4)
    # the parser also flags 4x4 transform edges, which no filter reads; none lies on the picture boundary
    assert not np.any(e[:, 0] & EDGE_V) and not np.any(e[0, :] & EDGE_H), "deblocking edge on the picture boundary"
    if np.any(e & (EDGE_V | EDGE_H)):
        assert pic.flags & PIC_HAS_DEBLOCK, "edges flagged but HC_PIC_HAS_DEBLOCK clear"
    if np.any(typ[:, :ncomp]):
        assert pic.flags & PIC_HAS_SAO, "SAO in use but HC_PIC_HAS_SAO clear"
