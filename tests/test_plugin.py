"""The drop-in boundary: libheif-cuda.so behind the UNMODIFIED reference libheif (oracle/_ref/libheifref.so).

The plugin implements struct heif_decoder_plugin (libheif/api/libheif/heif_plugin.h:53-112); the reference
library loads it with heif_load_plugin (init.cc:211-267 -> dlsym "plugin_info", plugins_unix.cc:95-110) and
the caller selects it with heif_decoding_options.decoder_id = "cuda" (plugin_registry.cc:231-255).

CPU tests: exported symbols / struct contents / registration with the reference / loud failure without a GPU.
GPU tests: heif_decode_image through the plugin reproduces the libde265 plugin's pixels (golden MD5s in
tests/golden/heic.json were produced by the reference with its own libde265 plugin).
Without the reference build the plugin is driven through its struct the way libheif drives a decoder plugin (one decoder
per coded item: new_decoder, push_data, decode_image, free_decoder), calling back into oracle/plugin_host.c, and
tests/heic_oracle.py does libheif's part (grid paste, alpha, transformations, colour conversion) on the images it returns."""
import concurrent.futures as cf
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import heic_oracle
import heif_b200 as hb
import oracle_lib
import refheif as R
from conftest import PKG_DIR, ROOT

PLUGIN = os.path.join(PKG_DIR, "plugins", "libheif-cuda.so")
META = json.load(open(os.path.join(ROOT, "tests", "golden", "heic.json")))
HEIC_DIR = os.path.join(ROOT, "tests", "golden", "heic")

needs_plugin = pytest.mark.skipif(not os.path.exists(PLUGIN), reason="plugin not built")
needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref (reference build) not present")


class Err(C.Structure):
    _fields_ = [("code", C.c_int), ("subcode", C.c_int), ("message", C.c_char_p)]


class DecoderPlugin(C.Structure):
    """hcp_decoder_plugin (include/heifcuda_plugin.h) == struct heif_decoder_plugin"""
    _fields_ = [("plugin_api_version", C.c_int),
                ("get_plugin_name", C.CFUNCTYPE(C.c_char_p)),
                ("init_plugin", C.CFUNCTYPE(None)),
                ("deinit_plugin", C.CFUNCTYPE(None)),
                ("does_support_format", C.CFUNCTYPE(C.c_int, C.c_int)),
                ("new_decoder", C.CFUNCTYPE(Err, C.POINTER(C.c_void_p), C.c_int)),
                ("free_decoder", C.CFUNCTYPE(None, C.c_void_p)),
                ("push_data", C.CFUNCTYPE(Err, C.c_void_p, C.c_char_p, C.c_size_t)),
                ("decode_image", C.CFUNCTYPE(Err, C.c_void_p, C.POINTER(C.c_void_p))),
                ("set_strict_decoding", C.CFUNCTYPE(None, C.c_void_p, C.c_int)),
                ("id_name", C.c_char_p)]


class PluginInfo(C.Structure):
    _fields_ = [("version", C.c_int), ("type", C.c_int), ("plugin", C.POINTER(DecoderPlugin)), ("internal_handle", C.c_void_p)]


def md5(b):
    return hashlib.md5(b).hexdigest()


_host = {}


def _plugin_and_host():
    """(plugin struct, oracle/plugin_host.c library): the plugin calls back into the stand-in through HEIFCUDA_LIBHEIF"""
    if not _host:
        oracle_lib.build()
        H = C.CDLL(oracle_lib.PLUGIN_HOST_SO)
        H.heif_image_get_plane.restype = C.c_void_p
        H.heif_image_get_plane.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        H.heif_image_release.argtypes = [C.c_void_p]
        H.ph_image_plane.argtypes = [C.c_void_p, C.c_int] + [C.POINTER(C.c_int)] * 4
        H.ph_image_nclx.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        os.environ["HEIFCUDA_LIBHEIF"] = oracle_lib.PLUGIN_HOST_SO
        _host.update(plugin=PluginInfo.in_dll(C.CDLL(PLUGIN), "plugin_info").plugin.contents, host=H)
    return _host["plugin"], _host["host"]


def _check(err, what):
    if err.code != 0:
        raise RuntimeError("%s: heif_error %d/%d %s" % (what, err.code, err.subcode, err.message))


def plugin_picture(stream, rec):
    """One coded picture through the plugin (decode_image_planar's life cycle of a decoder, context.cc): the cropped planes
    of the heif_image it returns; the nclx it attaches must be the VUI's (decoder_libde265.cc:339-362)."""
    p, H = _plugin_and_host()
    dec = C.c_void_p()
    _check(p.new_decoder(C.byref(dec), 1), "new_decoder")
    img = C.c_void_p()
    try:
        _check(p.push_data(dec, stream, len(stream)), "push_data")
        _check(p.decode_image(dec, C.byref(img)), "decode_image")
    finally:
        p.free_decoder(dec)
    try:
        planes = []
        for ch in range(3):
            w, h, bits, stride = C.c_int(), C.c_int(), C.c_int(), C.c_int()
            if not H.ph_image_plane(img, ch, C.byref(w), C.byref(h), C.byref(bits), C.byref(stride)):
                break
            dt = np.dtype(np.uint8) if bits.value <= 8 else np.dtype("<u2")
            buf = C.string_at(H.heif_image_get_plane(img, ch, None), stride.value * h.value)
            rows = np.frombuffer(buf, np.uint8).reshape(h.value, stride.value)[:, :w.value * dt.itemsize]
            planes.append(np.ascontiguousarray(rows).view(dt).astype(np.uint16))
        nclx = (C.c_int * 4)()
        assert H.ph_image_nclx(img, nclx)
        pic = rec.pic
        assert list(nclx) == [pic.colour_primaries, pic.transfer_characteristics, pic.matrix_coeffs, int(bool(pic.full_range))]
    finally:
        H.heif_image_release(img)
    return planes


TARGETS = {"rgb": hb.OUT_RGB, "rgba": hb.OUT_RGBA, "rrggbb_le": hb.OUT_RRGGBB_LE, "rrggbbaa_le": hb.OUT_RRGGBBAA_LE}


def host_decode(data, keys, threads=1):
    """{"planes": Y Cb Cr (A) bytes, key: interleaved bytes of TARGETS[key]} with every coded picture decoded by the plugin;
    `threads` decoders at once for the tiles of a grid (heif_context_set_threads: std::async per tile, context.cc:2361-2401)"""
    hf = hb.HeifFile(data, host_only=True)
    info = hf.image_info(hf.primary_id)
    streams = [hf.coded_stream(t) for t in hf.grid_tiles(hf.primary_id)] if info.is_grid else []
    hf.close()
    with cf.ThreadPoolExecutor(max_workers=threads) as pool:
        done = dict(zip(streams, pool.map(lambda s: plugin_picture(s, hb.parse_picture(s, host_only=True)), streams)))
    planes, alpha, cfmt, bd, (matrix, full, primaries) = heic_oracle.decode_planes(
        data, picture=lambda s, r: done[s] if s in done else plugin_picture(s, r))
    dt = np.uint8 if bd == 8 else np.dtype("<u2")
    out = {"planes": b"".join(p.astype(dt).tobytes() for p in planes + ([alpha] if alpha is not None else []))}
    for key in keys:
        out[key] = heic_oracle.csc(planes, cfmt, bd, matrix, full, TARGETS[key], alpha, primaries).tobytes()
    return out


def load(name):
    return open(os.path.join(HEIC_DIR, name + ".heic"), "rb").read()


@needs_plugin
def test_plugin_exports_the_reference_abi():
    L = C.CDLL(PLUGIN)
    info = PluginInfo.in_dll(L, "plugin_info")
    assert (info.version, info.type) == (1, 1)          # heif_plugin_type_decoder
    p = info.plugin.contents
    assert p.plugin_api_version == 3 and p.id_name == b"cuda"
    assert b"CUDA" in p.get_plugin_name()
    assert p.does_support_format(1) > 100               # heif_compression_HEVC outranks libde265's 100
    assert p.does_support_format(2) == 0 and p.does_support_format(4) == 0
    # decoder life cycle without any pixel work
    dec = C.c_void_p()
    assert p.new_decoder(C.byref(dec), 4).code == 0 and dec.value
    p.set_strict_decoding(dec, 1)
    e = p.push_data(dec, b"\x00\x00\x00", 3)            # truncated NAL length -> End_of_data like the reference
    assert (e.code, e.subcode) == (7, 100)
    e = p.push_data(dec, b"\x00\x00\x00\x09\x40\x01", 6)
    assert (e.code, e.subcode) == (7, 100)
    p.free_decoder(dec)


_loaded = {}


def reference_with_plugin():
    """The reference library with libheif-cuda.so registered through its own loader."""
    L = R.lib()
    if "info" not in _loaded:
        os.environ["HEIFCUDA_LIBHEIF"] = os.path.join(R.REF_DIR, "libheifref.so")   # ctypes loads libheif RTLD_LOCAL
        info = C.c_void_p()
        err = L.heif_load_plugin(PLUGIN.encode(), C.byref(info))
        assert err.code == 0, err.message
        _loaded["info"] = info
        R.FOREIGN_PLUGIN_LOADED = True
    return L


@needs_plugin
@needs_ref
def test_reference_loads_and_registers_the_plugin():
    L = reference_with_plugin()
    L.heif_have_decoder_for_format.argtypes = [C.c_int]
    assert L.heif_have_decoder_for_format(1)
    L.heif_get_decoder_descriptors.argtypes = [C.c_int, C.POINTER(C.c_void_p), C.c_int]
    L.heif_decoder_descriptor_get_id_name.restype = C.c_char_p
    L.heif_decoder_descriptor_get_id_name.argtypes = [C.c_void_p]
    descs = (C.c_void_p * 8)()
    n = L.heif_get_decoder_descriptors(1, descs, 8)
    ids = [L.heif_decoder_descriptor_get_id_name(descs[i]) for i in range(n)]
    assert b"cuda" in ids and b"libde265" in ids
    assert ids[0] == b"cuda"    # sorted by priority: the CUDA plugin is the default HEVC decoder now


def _has_gpu():
    # (no torch import needed for this)
    return os.path.exists("/dev/nvidiactl") or os.path.exists("/dev/nvidia0")


@needs_plugin
def test_plugin_fails_loudly_without_a_gpu():
    if _has_gpu():
        pytest.skip("a CUDA device is present")
    if not R.available():
        with pytest.raises(RuntimeError) as ei:
            host_decode(load("single_420_8_novui"), [])
        assert "decoder_cuda" in str(ei.value) or "CUDA" in str(ei.value)
        planes = heic_oracle.decode_planes(load("single_420_8_novui"))[0]
        assert md5(b"".join(p.astype(np.uint8).tobytes() for p in planes)) == META["single_420_8_novui"]["planes_md5"]
        return
    reference_with_plugin()
    with pytest.raises(RuntimeError) as ei:
        R.decode(load("single_420_8_novui"), R.COLORSPACE_UNDEFINED, R.CHROMA_UNDEFINED, decoder_id="cuda")
    assert "decoder_cuda" in str(ei.value) or "CUDA" in str(ei.value)
    # the reference's own decoder is still selectable next to it
    out = R.decode(load("single_420_8_novui"), R.COLORSPACE_UNDEFINED, R.CHROMA_UNDEFINED, decoder_id="libde265")
    assert md5(b"".join(out[k][0] for k in ("Y", "Cb", "Cr"))) == META["single_420_8_novui"]["planes_md5"]


@pytest.mark.gpu
@needs_plugin
@pytest.mark.parametrize("name", sorted(META))
def test_gpu_heif_decode_image_through_plugin(name):
    """heif_decode_image of the unmodified reference, decoder_id="cuda": planes and RGB == libde265 plugin."""
    m = META[name]
    data = load(name)
    if not R.available():
        keys = [k for k in (("rgb", "rgba") if m["bit_depth"] == 8 else ("rrggbb_le", "rrggbbaa_le")) if k + "_md5" in m]
        out = host_decode(data, keys)
        assert md5(out["planes"]) == m["planes_md5"]
        for key in keys:
            assert md5(out[key]) == m[key + "_md5"], key
        return
    reference_with_plugin()
    planes = R.decode(data, R.COLORSPACE_UNDEFINED, R.CHROMA_UNDEFINED, decoder_id="cuda")
    assert md5(b"".join(planes[k][0] for k in ("Y", "Cb", "Cr", "A") if k in planes)) == m["planes_md5"]
    targets = {"rgb": R.CHROMA_RGB, "rgba": R.CHROMA_RGBA} if m["bit_depth"] == 8 else {"rrggbb_le": R.CHROMA_RRGGBB_LE,
                                                                                       "rrggbbaa_le": R.CHROMA_RRGGBBAA_LE}
    for key, chroma in targets.items():
        if key + "_md5" in m:
            out = R.decode(data, R.COLORSPACE_RGB, chroma, decoder_id="cuda")
            assert md5(out["interleaved"][0]) == m[key + "_md5"], key


@pytest.mark.gpu
@needs_plugin
def test_gpu_plugin_default_selection_and_tile_threads():
    """No decoder_id: the plugin wins by priority; grid tiles decoded by concurrent decoder instances
    (heif_context_set_threads -> std::async per tile, context.cc:2361-2401)."""
    if not R.available():    # the priority itself is checked in test_plugin_exports_the_reference_abi
        for name in ("grid_300x200_t128", "example_1280x854"):
            if name in META:
                assert md5(host_decode(load(name), ["rgb"], threads=4)["rgb"]) == META[name]["rgb_md5"], name
        return
    reference_with_plugin()
    for name in ("grid_300x200_t128", "example_1280x854") :
        if name not in META:
            continue
        out = R.decode(load(name), R.COLORSPACE_RGB, R.CHROMA_RGB, threads=4, decoder_id="")
        assert md5(out["interleaved"][0]) == META[name]["rgb_md5"], name


@pytest.mark.gpu
@needs_plugin
def test_gpu_plugin_many_threads():
    """tests/test-race.go of the reference: many concurrent decodes of one file must not crash and agree."""
    import threading
    if R.available():
        reference_with_plugin()
    data = load("grid_300x200_t128")
    want = META["grid_300x200_t128"]["rgb_md5"]
    got = []

    def work():
        for _ in range(3):
            if R.available():
                got.append(md5(R.decode(data, R.COLORSPACE_RGB, R.CHROMA_RGB, decoder_id="cuda")["interleaved"][0]))
            else:
                got.append(md5(host_decode(data, ["rgb"])["rgb"]))

    ts = [threading.Thread(target=work) for _ in range(8)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert len(got) == 24 and set(got) == {want}
