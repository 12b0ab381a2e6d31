"""Loader for the CPU oracle (oracle/*.c -> oracle/_build/liboracle.so). Test infrastructure: the
checker, never the thing shipped or measured."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
SO = os.path.join(ORACLE_DIR, "_build", "liboracle.so")
SOURCES = ["hevc_recon_oracle.c", "csc_oracle.c"]
HEADERS = ["oracle_counters.h"]
# libheif's image / nclx callbacks for driving the decoder plugin without the reference libheif (oracle/plugin_host.c)
PLUGIN_HOST_SO = os.path.join(ORACLE_DIR, "_build", "libplugin_host.so")

STAGE_DEBLOCK, STAGE_SAO, STAGE_ALL = 1, 2, 3
_lib = None


def _compile(so, srcs, force, deps=()):
    if not force and os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(s) for s in list(srcs) + list(deps)):
        return
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", "-o", so] + srcs + ["-lm"])


def build(force=False):
    srcs = [os.path.join(ORACLE_DIR, s) for s in SOURCES if os.path.exists(os.path.join(ORACLE_DIR, s))]
    _compile(SO, srcs, force, [os.path.join(ORACLE_DIR, h) for h in HEADERS])
    _compile(PLUGIN_HOST_SO, [os.path.join(ORACLE_DIR, "plugin_host.c")], force)
    return SO


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.hc_oracle_reconstruct.restype = C.c_int
        _lib.hc_oracle_counters.restype = C.c_int
        _lib.hc_oracle_counter_name.restype = C.c_char_p
    return _lib


def counters_reset():
    lib().hc_oracle_counters_reset()


def counters():
    """{name: count} of the oracle's branch counters (oracle/oracle_counters.h) since the last counters_reset()"""
    O = lib()
    n = O.hc_oracle_counters(None, 0)
    out = (C.c_uint64 * n)()
    O.hc_oracle_counters(out, n)
    return {O.hc_oracle_counter_name(i).decode(): int(out[i]) for i in range(n)}


def plane_dims(pic):
    sw = 2 if pic.chroma_format in (1, 2) else 1
    sh = 2 if pic.chroma_format == 1 else 1
    dims = [(pic.width, pic.height)]
    if pic.chroma_format:
        dims += [(pic.width // sw, pic.height // sh)] * 2
    return dims, sw, sh


def reconstruct(rec, stages=STAGE_ALL, want_residual=False):
    """Runs the oracle on the records of one picture. Returns (list of cropped uint16 planes, residual or None)."""
    O = lib()
    pic = rec.pic
    dims, sw, sh = plane_dims(pic)
    planes = [np.zeros((h, w), np.uint16) for w, h in dims]
    pp = (C.c_void_p * 3)(*([p.ctypes.data for p in planes] + [None] * (3 - len(planes))))
    st = (C.c_int * 3)(*([w for w, h in dims] + [0] * (3 - len(planes))))
    ptr = {n: rec.array(n)[0] for n in ("ctus", "blks", "tbs", "coeffs", "edge_map", "qp_map", "scaling")}
    resid = np.zeros(max(int(pic.resid_count), 1), np.int16) if want_residual else None
    rc = O.hc_oracle_reconstruct(C.byref(pic), C.c_void_p(ptr["ctus"]), C.c_void_p(ptr["blks"]), C.c_void_p(ptr["tbs"]),
                                 C.c_void_p(ptr["coeffs"]), C.c_void_p(ptr["edge_map"]), C.c_void_p(ptr["qp_map"]),
                                 C.c_void_p(ptr["scaling"]), stages, pp, st,
                                 C.c_void_p(resid.ctypes.data) if want_residual else None)
    if rc != 0:
        raise RuntimeError("oracle failed: %d" % rc)
    out = []
    for i, p in enumerate(planes):
        cx, cy, cw, ch = pic.crop_x, pic.crop_y, pic.crop_w, pic.crop_h
        if i:
            cx //= sw
            cw = (cw + sw - 1) // sw
            cy //= sh
            ch = (ch + sh - 1) // sh
        out.append(np.ascontiguousarray(p[cy:cy + ch, cx:cx + cw]))
    return out, resid


def planes_bytes(planes, bit_depth):
    """Planar YUV bytes as dec265 -o / the plugin would return them (1 byte per sample for 8 bit, else LE16)."""
    dt = np.uint8 if bit_depth == 8 else np.dtype("<u2")
    return b"".join(p.astype(dt).tobytes() for p in planes)
