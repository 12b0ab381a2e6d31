"""Decoding any image item of a HEIF file, not only the primary one: thumbnails ('thmb'), auxiliary images ('auxl': alpha,
depth, gain maps), other top-level images, hidden items and grid tiles, through hc_heic_job_create_items,
hc_heic_decode_stream_items and decode_heic(item_id=...).
The corpus: every fixture of tests/golden/heic/, the reference's example.heic (two top-level images with a thumbnail each)
and three files written here from fixed seeds with tools/hevcenc + tools/heif_writer (a burst of three top-level images, a
phone-style photo with two thumbnails, a depth map, a gain map and an Exif item, and a 4096 x 4096 grid with a tiny
thumbnail).
CPU tests: the container reader's lists, and the oracle chain on the generated items.
GPU tests: every image item against heic_oracle (decode_planes / decode_rgb with the item's id), example.heic's second
image against the reference's golden MD5s, the stream's batch sizing and error isolation per entry."""
import functools
import hashlib
import json
import os
import struct
import sys

import numpy as np
import pytest

import heif_b200 as hb
import heic_oracle as ho
from conftest import ROOT, read_stream

sys.path.insert(0, ROOT)
from tools import heif_writer as W, hevcenc  # noqa: E402

DIR = os.path.join(ROOT, "tests", "golden", "heic")
FIXTURES = sorted(f[:-5] for f in os.listdir(DIR) if f.endswith(".heic"))
GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))["heic"]["example.heic"]
FORMATS = [hb.OUT_RGB, hb.OUT_RGBA, hb.OUT_RRGGBB_BE, hb.OUT_RRGGBBAA_BE, hb.OUT_RRGGBB_LE, hb.OUT_RRGGBBAA_LE, hb.OUT_YCBCR]
DEPTH_URN = "urn:mpeg:hevc:2015:auxid:2"
GAIN_URN = "urn:com:apple:photo:2020:aux:hdrgainmap"
MISSING = 999


def md5(b):
    return hashlib.md5(b).hexdigest()


def _coded(w, h, cf, bd, seed, **kw):
    return hevcenc.encode(hevcenc.synth_image(w, h, cf, bd, seed), chroma_format=cf, bit_depth=bd, seed=seed, **kw)


def _aux(urn):
    return W.fullbox(b"auxC", 0, 0, urn.encode() + b"\x00")


# ------------------------------------------------------------------------------------------------------ generated files
@functools.lru_cache(maxsize=None)
def burst():
    """Three top-level images: 4:2:0 8-bit with irot (item 1), 4:4:4 10-bit with an alpha image (items 2, 3; the primary)
    and monochrome 12-bit (item 4)."""
    b = W.HeifBuilder()
    b.add_hevc_image(_coded(96, 64, 1, 8, 11), 96, 64, 1, 8, extra_props=(W.irot(1),))
    second = b.add_hevc_image(_coded(80, 48, 3, 10, 12), 80, 48, 3, 10)
    b.add_alpha(second, _coded(80, 48, 0, 10, 13), 80, 48, 0, 10)
    b.add_hevc_image(_coded(64, 40, 0, 12, 14), 64, 40, 0, 12)
    b.primary = second
    return b.serialize()


PHONE = dict(grid=5, thumb=6, thumb_alpha=7, thumb_grid=10, depth=11, gain=12, exif=13)


@functools.lru_cache(maxsize=None)
def phone():
    """A phone photo: a rotated 2 x 2 grid (item 5, the primary); a thumbnail with the same irot and a half-size alpha image
    of its own (items 6, 7); a second thumbnail that is a 2 x 1 grid (item 10 over tiles 8, 9); a 10-bit monochrome depth
    map with a clap (item 11); a limited-range gain map whose colr overrides its VUI (item 12); an Exif item (13)."""
    b = W.HeifBuilder()
    tiles = [b.add_hevc_image(_coded(64, 64, 1, 8, 20 + k), 64, 64, 1, 8, hidden=True) for k in range(4)]
    grid = b.add_grid(tiles, 2, 2, 120, 100, extra_props=(W.irot(1),))
    thumb = b.add_hevc_image(_coded(48, 32, 1, 8, 30), 48, 32, 1, 8, extra_props=(W.irot(1),))
    b.add_alpha(thumb, _coded(24, 16, 0, 8, 31), 24, 16, 0, 8, extra_props=(W.irot(1),))
    b.refs.append((b"thmb", thumb, [grid]))
    ttiles = [b.add_hevc_image(_coded(32, 32, 1, 8, 32 + k), 32, 32, 1, 8, hidden=True) for k in range(2)]
    tgrid = b.add_grid(ttiles, 1, 2, 60, 30)
    b.refs.append((b"thmb", tgrid, [grid]))
    depth = b.add_hevc_image(_coded(96, 72, 0, 10, 40), 96, 72, 0, 10, hidden=True,
                             extra_props=(_aux(DEPTH_URN), W.clap(90, 1, 70, 1, 0, 1, 0, 1)))
    b.refs.append((b"auxl", depth, [grid]))
    gain = b.add_hevc_image(_coded(60, 50, 1, 8, 41), 60, 50, 1, 8, hidden=True, nclx=(1, 13, 1, 0), extra_props=(_aux(GAIN_URN),))
    b.refs.append((b"auxl", gain, [grid]))
    exif = b.add_item(b"Exif", struct.pack(">I", 0) + b"MM\x00\x2a\x00\x00\x00\x08\x00\x00", [], hidden=True)
    b.refs.append((b"cdsc", exif, [grid]))
    b.primary = grid
    got = dict(grid=grid, thumb=thumb, thumb_alpha=thumb + 1, thumb_grid=tgrid, depth=depth, gain=gain, exif=exif)
    assert got == PHONE, got
    return b.serialize()


BIG = dict(tile=1, grid=2, thumb=3)


@functools.lru_cache(maxsize=None)
def big():
    """A 4096 x 4096 grid whose 64 'dimg' references all name one 512 x 512 tile (item 1), with a 64 x 48 thumbnail."""
    b = W.HeifBuilder()
    tile = b.add_hevc_image(_coded(512, 512, 1, 8, 50), 512, 512, 1, 8, hidden=True)
    grid = b.add_grid([tile] * 64, 8, 8, 4096, 4096)
    thumb = b.add_hevc_image(_coded(64, 48, 1, 8, 51), 64, 48, 1, 8)
    b.refs.append((b"thmb", thumb, [grid]))
    b.primary = grid
    assert (tile, grid, thumb) == (BIG["tile"], BIG["grid"], BIG["thumb"])
    return b.serialize()


def sources():
    """label -> file bytes of every file of the corpus but the big one"""
    out = {n: open(os.path.join(DIR, n + ".heic"), "rb").read() for n in FIXTURES}
    out["example.heic"] = read_stream("example.heic")
    out["burst"] = burst()
    out["phone"] = phone()
    return out


def image_items(data):
    """Every image item reachable from the top-level images: the images themselves, their thumbnails and auxiliary images
    (alpha included), and the tiles of every grid among them, ascending."""
    hf = hb.HeifFile(data, host_only=True)
    todo, seen = list(hf.top_level_ids()), set()
    while todo:
        i = todo.pop()
        if i in seen:
            continue
        seen.add(i)
        todo += hf.thumbnail_ids(i) + hf.auxiliary_ids(i, include_alpha=True)
        if hf.image_info(i).is_grid:
            todo += hf.grid_tiles(i)
    return sorted(seen)


@functools.lru_cache(maxsize=None)
def oracle_planes(label, item):
    return ho.decode_planes(sources()[label], item)


def oracle_bytes(label, item, fmt):
    """what image `item` of a file must decode to in format `fmt` (packed planes for OUT_YCBCR), or None where the
    conversion does not exist"""
    planes, alpha, cf, bd, (matrix, full, primaries) = oracle_planes(label, item)
    if fmt == hb.OUT_YCBCR:
        dt = np.uint8 if bd == 8 else np.dtype("<u2")
        return b"".join(p.astype(dt).tobytes() for p in planes + ([alpha] if alpha is not None else []))
    try:
        return ho.csc(planes, cf, bd, matrix, full, fmt, alpha, primaries).tobytes()
    except RuntimeError:
        return None


@functools.lru_cache(maxsize=None)
def entries():
    """(label, item id) of one job: per file its primary as 0 and by id, then every other image item, so that entries
    repeat buffers and mix primary and non-primary items"""
    out = []
    for label, data in sources().items():
        primary = hb.HeifFile(data, host_only=True).primary_id
        out += [(label, 0), (label, primary)] + [(label, i) for i in image_items(data) if i != primary]
    return out


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_example_heic_thumbnails():
    hf = hb.HeifFile(read_stream("example.heic"), host_only=True)
    assert hf.top_level_ids() == [20004, 20006]
    assert hf.thumbnail_ids(20004) == [20005] and hf.thumbnail_ids(20006) == [20007]
    assert hf.thumbnail_ids(20005) == [] and hf.auxiliary_ids(20004, include_alpha=True) == []


def test_phone_like_thumbnail_and_gain_map():
    hf = hb.HeifFile(open(os.path.join(DIR, "phone_like_grid_irot90.heic"), "rb").read(), host_only=True)
    assert hf.primary_id == 7
    assert hf.thumbnail_ids(7) == [8]
    assert hf.auxiliary_ids(7) == [9] == hf.auxiliary_ids(7, include_alpha=True)
    assert hf.aux_type(9) == GAIN_URN
    with pytest.raises(hb.HeifCudaError, match="item 7 has no auxC"):
        hf.aux_type(7)


@pytest.mark.parametrize("name", FIXTURES)
def test_fixture_alpha_is_an_auxiliary_image(name):
    hf = hb.HeifFile(open(os.path.join(DIR, name + ".heic"), "rb").read(), host_only=True)
    pid = hf.primary_id
    alpha = hf.image_info(pid).alpha_id
    others = [9] if name == "phone_like_grid_irot90" else []     # its gain map
    assert hf.auxiliary_ids(pid) == others
    assert hf.auxiliary_ids(pid, include_alpha=True) == sorted(others + ([alpha] if alpha else []))
    if alpha:
        assert hf.aux_type(alpha) in ("urn:mpeg:hevc:2015:auxid:1", "urn:mpeg:mpegB:cicp:systems:auxiliary:alpha")


def test_generated_files_lists():
    hf = hb.HeifFile(burst(), host_only=True)
    assert hf.primary_id == 2 and hf.top_level_ids() == [1, 2, 4]
    assert hf.auxiliary_ids(2) == [] and hf.auxiliary_ids(2, include_alpha=True) == [3]
    assert all(hf.thumbnail_ids(i) == [] for i in (1, 2, 4))
    hf = hb.HeifFile(phone(), host_only=True)
    P = PHONE
    assert hf.primary_id == P["grid"] and hf.top_level_ids() == [P["grid"]]
    assert hf.thumbnail_ids(P["grid"]) == [P["thumb"], P["thumb_grid"]]
    assert hf.auxiliary_ids(P["grid"]) == hf.auxiliary_ids(P["grid"], include_alpha=True) == [P["depth"], P["gain"]]
    assert hf.auxiliary_ids(P["thumb"]) == [] and hf.auxiliary_ids(P["thumb"], include_alpha=True) == [P["thumb_alpha"]]
    assert (hf.aux_type(P["depth"]), hf.aux_type(P["gain"])) == (DEPTH_URN, GAIN_URN)
    assert hf.image_info(P["thumb"]).alpha_id == P["thumb_alpha"]
    hf = hb.HeifFile(big(), host_only=True)
    assert hf.thumbnail_ids(BIG["grid"]) == [BIG["thumb"]] and hf.grid_tiles(BIG["grid"]) == [BIG["tile"]] * 64


def test_generated_items_through_the_oracle():
    """The oracle chain on the generated items: sizes after each item's own transformations, alpha attached at the colour
    image's size."""
    P = PHONE
    want = {("burst", 0): (48, 80, True), ("burst", 1): (96, 64, False), ("burst", 3): (48, 80, False), ("burst", 4): (40, 64, False),
            ("phone", 0): (120, 100, False), ("phone", P["thumb"]): (48, 32, True), ("phone", P["thumb_alpha"]): (24, 16, False),
            ("phone", P["thumb_grid"]): (30, 60, False), ("phone", P["depth"]): (70, 90, False), ("phone", P["gain"]): (50, 60, False)}
    for (label, item), (h, w, has_alpha) in want.items():
        planes, alpha, *_ = oracle_planes(label, item)
        assert planes[0].shape == (h, w) and (alpha is not None) == has_alpha, (label, item)
        if has_alpha:
            assert alpha.shape == (h, w)
    assert set(image_items(phone())) == set(range(1, 13))
    assert image_items(burst()) == [1, 2, 3, 4]


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def engine():
    e = hb.Engine(0)
    yield e
    e.close()


class Options:
    DEFAULTS = {"scale_max_side": 0, "device_parse": 1, "host_share_pct": -1}

    def __init__(self, engine, **opts):
        self.engine, self.opts = engine, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.engine.set_option(k, v)

    def __exit__(self, *exc):
        for k in self.opts:
            self.engine.set_option(k, self.DEFAULTS[k])


def read(job, i):
    if job.descs[i].out_format == hb.OUT_YCBCR:
        return b"".join(np.ascontiguousarray(p).tobytes() for p in job.read_planes(i))
    return job.read_rgb(i).tobytes()


def run_job(engine, files, items, fmt, **opts):
    with Options(engine, **opts):
        job = hb.HeicJob(engine, files, threads=4, out_format=fmt, items=items)
    try:
        job.upload()
        job.run()
        return [read(job, i) for i in range(len(files))], list(job.descs)
    finally:
        job.close()


@pytest.mark.gpu
@pytest.mark.parametrize("device_parse", [1, 0])
def test_gpu_example_second_image_matches_reference(engine, device_parse):
    """example.heic item 20006 (not its primary) named in a job: the reference's own RGB, RGBA and planes."""
    data = read_stream("example.heic")
    g = GOLDEN["20006"]
    for fmt, key in ((hb.OUT_RGB, "rgb_md5"), (hb.OUT_RGBA, "rgba_md5"), (hb.OUT_YCBCR, "planes_md5")):
        got, descs = run_job(engine, [data, data], [20006, 0], fmt, device_parse=device_parse, host_share_pct=0)
        assert (descs[0].width, descs[0].height) == (g["width"], g["height"])
        assert md5(got[0]) == g[key], key
        assert md5(got[1]) == GOLDEN["20004"][key], key


@pytest.mark.gpu
@pytest.mark.parametrize("device_parse", [1, 0])
@pytest.mark.parametrize("fmt", FORMATS)
def test_gpu_every_image_item_matches_oracle(engine, fmt, device_parse):
    """Every image item of every file in ONE job, buffers repeated, primary and other items mixed; entries naming the
    primary (by 0 or by id) are byte-identical to hc_heic_job_create."""
    src = sources()
    ents = [(lb, it) for lb, it in entries() if oracle_bytes(lb, it, fmt) is not None]
    assert len(ents) > 150
    got, descs = run_job(engine, [src[lb] for lb, _ in ents], [it for _, it in ents], fmt, device_parse=device_parse, host_share_pct=0)
    bad = [(lb, it) for (lb, it), g in zip(ents, got) if g != oracle_bytes(lb, it, fmt)]
    assert not bad, bad
    labels = sorted(lb for lb, it in ents if it == 0)
    with Options(engine, device_parse=device_parse, host_share_pct=0):
        plain = hb.HeicJob(engine, [src[lb] for lb in labels], threads=4, out_format=fmt)
    plain.upload()
    plain.run()
    whole = {lb: read(plain, k) for k, lb in enumerate(labels)}
    plain.close()
    primary = {lb: hb.HeifFile(src[lb], host_only=True).primary_id for lb in labels}
    for (lb, it), g in zip(ents, got):
        if it in (0, primary[lb]):
            assert g == whole[lb], (lb, it)


def stream_entries():
    """the stream's corpus: every item of the generated files and of example.heic, and of four fixtures"""
    keep = {"burst", "phone", "example.heic", "alpha_half_420_8", "alpha_irot90_420_8", "grid_irot90_300x200", "single_mono_12_full"}
    return [(lb, it) for lb, it in entries() if lb in keep]


def fit(W, H, S):
    """the fit rule of "scale_max_side" (include/heifcuda.h)"""
    if S <= 0 or max(W, H) <= S:
        return W, H
    return (S, max(1, H * S // W)) if W >= H else (max(1, W * S // H), S)


def scaled(rows_bytes, w, h, bpp, S):
    """heif_image_scale_image's nearest-neighbour sampling of interleaved pixels to the fit within S"""
    px = np.frombuffer(rows_bytes, np.uint8).reshape(h, w, bpp)
    w2, h2 = fit(w, h, S)
    return np.ascontiguousarray(px[np.arange(h2) * h // h2][:, np.arange(w2) * w // w2]).tobytes()


def run_stream(engine, ents, fmt=hb.OUT_RGBA, **kw):
    src = sources()
    seen = {}

    def on_image(index, desc, rows):
        seen[index] = (desc.width, desc.height, rows[:, :desc.width * desc.bytes_per_pixel].tobytes())
    st = hb.decode_stream(engine, [src[lb] for lb, _ in ents], on_image, threads=4, out_format=fmt, items=[it for _, it in ents], **kw)
    return seen, st


@pytest.mark.gpu
@pytest.mark.parametrize("host_share", [0, 100])
@pytest.mark.parametrize("files_per_batch", [1, 3, 0])
def test_gpu_stream_items(engine, host_share, files_per_batch):
    ents = stream_entries()
    with Options(engine, host_share_pct=host_share):
        seen, st = run_stream(engine, ents, files_per_batch=files_per_batch)
    assert sorted(seen) == list(range(len(ents)))
    bad = [e for k, e in enumerate(ents) if seen[k][2] != oracle_bytes(*e, hb.OUT_RGBA)]
    assert not bad, bad
    if files_per_batch:
        assert st["batches"] == -(-len(ents) // files_per_batch)


@pytest.mark.gpu
def test_gpu_stream_items_external_destinations(engine):
    """dests[k] belongs to entry k: every other entry gets a destination of its own, with a padded stride"""
    src = sources()
    ents = stream_entries()
    fmt = hb.OUT_RRGGBB_LE
    sizes = [oracle_planes(lb, it)[0][0].shape for lb, it in ents]
    dests = [np.zeros((h, w * 6 + 16), np.uint8) if k % 2 == 0 else None for k, (h, w) in enumerate(sizes)]
    ext = {}

    def on_image(index, desc, rows):
        ext[index] = rows.ctypes.data == (dests[index].ctypes.data if dests[index] is not None else None)
    hb.decode_stream(engine, [src[lb] for lb, _ in ents], on_image, threads=4, files_per_batch=3, out_format=fmt, dests=dests,
                     items=[it for _, it in ents])
    assert sorted(ext) == list(range(len(ents))) and all(ext[k] == (k % 2 == 0) for k in ext)
    for k, (lb, it) in enumerate(ents):
        if dests[k] is not None:
            h, w = sizes[k]
            assert dests[k][:, :w * 6].tobytes() == oracle_bytes(lb, it, fmt), (lb, it)
            assert not dests[k][:, w * 6:].any()


@pytest.mark.gpu
def test_gpu_stream_items_scaled(engine):
    """scale_max_side = 80: the depth map (90 x 70 after its clap) and the primary grid are scaled, the thumbnails are not"""
    P, S = PHONE, 80
    ents = [("phone", i) for i in (0, P["thumb"], P["thumb_grid"], P["depth"], P["gain"], P["thumb_alpha"])] + [("burst", 1)]
    with Options(engine, scale_max_side=S):
        seen, _ = run_stream(engine, ents, files_per_batch=0)
    for k, (lb, it) in enumerate(ents):
        h, w = oracle_planes(lb, it)[0][0].shape
        assert seen[k][:2] == fit(w, h, S), (lb, it)
        assert seen[k][2] == scaled(oracle_bytes(lb, it, hb.OUT_RGBA), w, h, 4, S), (lb, it)
    assert seen[3][:2] != (90, 70) and seen[1][:2] == (32, 48) and seen[2][:2] == (60, 30)


@pytest.mark.gpu
@pytest.mark.parametrize("files_per_batch", [1, 3, 7])
def test_gpu_stream_isolates_an_entry_naming_no_image(engine, files_per_batch):
    """An entry naming the Exif item or an id the file lacks, at every position: it fails alone with a text naming the
    item, and every other entry (all of them non-primary items but one) stays bit-exact."""
    P = PHONE
    good = [("phone", P["thumb"]), ("burst", 1), ("phone", P["depth"]), ("phone", 0), ("phone", P["thumb_grid"]),
            ("burst", 4), ("phone", P["gain"])]
    for bad_item in (P["exif"], MISSING):
        for pos in range(len(good)):
            ents = list(good)
            ents[pos] = ("phone", bad_item)
            seen, st = run_stream(engine, ents, files_per_batch=files_per_batch, isolate_errors=True)
            assert st["files_failed"] == 1 and st["file_status"][pos] != 0, (bad_item, pos)
            assert "item %d" % bad_item in st["first_error"], st["first_error"]
            assert sorted(seen) == [k for k in range(len(ents)) if k != pos]
            for k in seen:
                assert seen[k][2] == oracle_bytes(*ents[k], hb.OUT_RGBA), (bad_item, pos, ents[k])


@pytest.mark.gpu
def test_gpu_automatic_batch_size_follows_the_named_item(engine):
    """100 entries of a 4096 x 4096 file: its 64 x 48 thumbnails go in one batch, its primary (16.8 MP, 47 entries per batch
    of about 800 MP) in three. scale_max_side keeps the read-back small; the batch size follows the coded size."""
    data = big()
    with Options(engine, scale_max_side=64):
        n = {}
        for item in (BIG["thumb"], 0):
            seen = []
            st = hb.decode_stream(engine, [data] * 100, lambda k, d, r: seen.append(k), threads=4, files_per_batch=0,
                                  out_format=hb.OUT_RGB, items=[item] * 100)
            assert sorted(seen) == list(range(100))
            n[item] = st["batches"]
    assert n == {BIG["thumb"]: 1, 0: 3}


@pytest.mark.gpu
def test_gpu_job_refuses_an_entry_that_is_no_image(engine):
    data = phone()
    for item, text in ((PHONE["exif"], "item %d is of type 'Exif'" % PHONE["exif"]), (MISSING, "item %d does not exist" % MISSING)):
        with pytest.raises(hb.HeifCudaError, match=text):
            hb.HeicJob(engine, [data, data], items=[0, item])


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [hb.OUT_RGB, hb.OUT_RGBA, hb.OUT_RRGGBBAA_LE])
def test_gpu_decode_heic_rotated_thumbnail_with_its_own_alpha(engine, fmt):
    """decode_heic(item_id=...) on a thumbnail that carries its own irot and a half-size alpha image"""
    got = hb.decode_heic(engine, phone(), fmt, item_id=PHONE["thumb"])
    assert got.shape == (48, 32 * api_bpp(fmt))
    assert got.tobytes() == oracle_bytes("phone", PHONE["thumb"], fmt)


def api_bpp(fmt):
    return hb.api.OUT_BYTES_PER_PIXEL[fmt]
