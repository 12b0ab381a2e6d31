"""Oracle-side HEIC decode: product container reader + host parser feed the CPU oracle; grid paste,
alpha attach and colour conversion are restated here following libheif/context.cc:1729-2539.
Test infrastructure (the checker)."""
import ctypes as C

import numpy as np

import heif_b200 as hb
import oracle_lib

OUT_BPP = {0: 3, 1: 4, 2: 6, 3: 8, 4: 6, 5: 8}


def csc(planes, chroma_format, bit_depth, matrix, full_range, out_format, alpha=None, primaries=2, upsampling=0):
    O = oracle_lib.lib()
    h, w = planes[0].shape
    out = np.zeros((h, w * OUT_BPP[out_format]), np.uint8)
    pl = [np.ascontiguousarray(p, np.uint16) for p in planes]
    a = np.ascontiguousarray(alpha, np.uint16) if alpha is not None else None
    rc = O.hc_oracle_csc_opt(C.c_void_p(pl[0].ctypes.data), C.c_void_p(pl[1].ctypes.data if len(pl) > 1 else None),
                         C.c_void_p(pl[2].ctypes.data if len(pl) > 2 else None), C.c_void_p(a.ctypes.data if a is not None else None),
                         pl[0].shape[1], pl[1].shape[1] if len(pl) > 1 else 0, a.shape[1] if a is not None else 0,
                         w, h, chroma_format, bit_depth, matrix, int(primaries), int(full_range), out_format, int(upsampling),
                         C.c_void_p(out.ctypes.data), C.c_size_t(out.strides[0]))
    if rc != 0:
        raise RuntimeError("oracle csc cannot convert this combination")
    return out


def _rescale_limited(plane, chroma, bit_depth):
    """context.cc:2504-2528: clip_f_u8((v - 16<<(bpp-8)) * ratio), byte-wise (8-bit tiles)"""
    ratio = np.float32(1.1429 if chroma else 1.1689)
    full = (plane.astype(np.float32) - np.float32(16 << (bit_depth - 8))) * ratio
    x = (full + np.float32(0.5)).astype(np.int64)  # (long)(fx + 0.5f): truncation toward zero
    return np.clip(x, 0, 255).astype(np.uint16)


def subsampling(chroma_format):
    """(SubWidthC, SubHeightC)"""
    return (2 if chroma_format in (1, 2) else 1), (2 if chroma_format == 1 else 1)


def new_canvas(W, H, chroma_format, dtype=np.uint16):
    """zeroed planes of a W x H canvas: Y [, Cb, Cr]"""
    sw, sh = subsampling(chroma_format)
    planes = [np.zeros((H, W), dtype)]
    if chroma_format:
        planes += [np.zeros(((H + sh - 1) // sh, (W + sw - 1) // sw), dtype) for _ in range(2)]
    return planes


def paste(canvas_planes, tile_planes, x, y, chroma_format, rescale, bit_depth):
    """Grid paste of one tile at luma position (x, y) (context.cc:2467-2528): chroma at ((x + SubW - 1) / SubW,
    (y + SubH - 1) / SubH), clipped at the canvas edge, limited-range tiles rescaled on the way. In place."""
    sw, sh = subsampling(chroma_format)
    for k, p in enumerate(tile_planes):
        if rescale:
            p = _rescale_limited(p, k > 0, bit_depth)
        xx, yy = (x, y) if k == 0 else ((x + sw - 1) // sw, (y + sh - 1) // sh)
        c = canvas_planes[k]
        hh, ww = min(p.shape[0], c.shape[0] - yy), min(p.shape[1], c.shape[1] - xx)
        if hh > 0 and ww > 0:
            c[yy:yy + hh, xx:xx + ww] = p[:hh, :ww]
    return canvas_planes


def dihedral(plane, swap, flip_x, flip_y):
    """The map of hc_batch_set_canvas_transform on one plane of w x h samples: output (x', y') is input (sx, sy) with
    !swap: sx = flip_x ? w-1-x' : x', sy = flip_y ? h-1-y' : y';  swap: sx = flip_x ? w-1-y' : y', sy = flip_y ? h-1-x' : x'.
    irot / imir of the reference (HeifPixelImage::rotate_ccw / mirror_inplace, pixelimage.cc:539-794) are such maps."""
    g = plane[::-1 if flip_y else 1, ::-1 if flip_x else 1]
    return np.ascontiguousarray(g.T if swap else g)


def crop_planes(planes, window):
    """HeifPixelImage::crop (pixelimage.cc:797-870): the inclusive window (left, top, right, bottom) of the image
    (planes[0]'s size) scaled to every plane by integer division (:820-823)"""
    l, t, r, b = window
    H, W = planes[0].shape
    out = []
    for p in planes:
        ph, pw = p.shape
        out.append(np.ascontiguousarray(p[t * ph // H:b * ph // H + 1, l * pw // W:r * pw // W + 1]))
    return out


def scale_nearest(plane, w, h):
    """HeifPixelImage::scale_nearest_neighbor (pixelimage.cc:1231-1250): out(x, y) = in(x * in_w / w, y * in_h / h)"""
    iy = np.arange(h, dtype=np.int64) * plane.shape[0] // h
    ix = np.arange(w, dtype=np.int64) * plane.shape[1] // w
    return np.ascontiguousarray(plane[iy][:, ix])


def compose_overlay(children_rgb, alphas, offsets, background, W, H, out_format):
    """decode_overlay_image (context.cc:2579-2675, pixelimage.cc:1017-1150): an 8-bit planar RGB canvas filled with the
    high bytes of the 16-bit background words; every child (h x w x 3 8-bit RGB) overlaid in order at its offset,
    clipped at the canvas edge — copied, or (child * a + canvas * (255 - a)) / 255 with an alpha plane; then the
    interleaver of the requested format. Returns the interleaved rows (H x W * bytes per pixel, uint8)."""
    canvas = np.empty((H, W, 3), np.int64)
    for k in range(3):
        canvas[:, :, k] = background[k] >> 8
    for px, a, (dx, dy) in zip(children_rgb, alphas, offsets):
        h, w = px.shape[:2]
        if dx >= W or dy >= H:
            continue
        ww, hh = min(w, W - dx), min(h, H - dy)
        src = px[:hh, :ww, :3].astype(np.int64)
        if a is not None:
            al = a[:hh, :ww, None].astype(np.int64)
            canvas[dy:dy + hh, dx:dx + ww] = (src * al + canvas[dy:dy + hh, dx:dx + ww] * (255 - al)) // 255
        else:
            canvas[dy:dy + hh, dx:dx + ww] = src
    rgb = canvas.astype(np.uint16)
    if out_format == 0:                                          # RGB
        return rgb.astype(np.uint8).reshape(H, W * 3)
    if out_format == 1:                                          # RGBA: opaque
        out = np.full((H, W, 4), 255, np.uint8)
        out[:, :, :3] = rgb
        return out.reshape(H, W * 4)
    v = (rgb << 2) | (rgb >> 6)                                  # Op_to_hdr_planes, 8 -> 10 bit
    if out_format in (3, 5):                                     # RRGGBBAA: opaque at 10 bit
        v = np.concatenate([v, np.full((H, W, 1), 1023, np.uint16)], axis=2)
    dt = "<u2" if out_format in (4, 5) else ">u2"
    return np.frombuffer(v.astype(dt).tobytes(), np.uint8).reshape(H, -1)


def _oracle_picture(stream, rec):
    return oracle_lib.reconstruct(rec)[0]


def decode_planes(data, item_id=None, picture=_oracle_picture, transform=None):
    """Returns (planes[list], alpha or None, chroma_format, bit_depth, (matrix, full_range, primaries)).
    picture(coded stream, its records) -> cropped planes of one coded picture: the oracle, or another HEVC decoder in
    the place libheif gives its decoder plugin. transform(planes, image info) -> the planes after the item's irot / imir /
    clap (default: _transform_all)."""
    transform = transform or _transform_all
    hf = hb.HeifFile(data, host_only=True)
    iid = item_id or hf.primary_id
    info = hf.image_info(iid)
    if info.is_grid:
        ids = hf.grid_tiles(iid)
        streams = [hf.coded_stream(t) for t in ids]
        recs = [hb.parse_picture(s, host_only=True) for s in streams]
        p0 = recs[0].pic
        cf, bd = p0.chroma_format, p0.bit_depth_y
        W, H = info.width, info.height
        canvas = new_canvas(W, H, cf)
        tw, th = p0.crop_w, p0.crop_h
        for i, (t, s, r) in enumerate(zip(ids, streams, recs)):
            tinfo = hf.image_info(t)
            full = tinfo.full_range if tinfo.nclx_present else r.pic.full_range
            matrix = tinfo.matrix if tinfo.nclx_present else r.pic.matrix_coeffs
            paste(canvas, picture(s, r), (i % info.cols) * tw, (i // info.cols) * th, cf, (not full) and matrix != 0, bd)
        nclx = (info.matrix, info.full_range, info.primaries) if info.nclx_present else (2, 1, 2)
        planes = canvas
    else:
        s = hf.coded_stream(iid)
        r = hb.parse_picture(s, host_only=True)
        planes = picture(s, r)
        cf, bd = r.pic.chroma_format, r.pic.bit_depth_y
        nclx = (info.matrix, info.full_range, info.primaries) if info.nclx_present else (r.pic.matrix_coeffs, r.pic.full_range, r.pic.colour_primaries)
    alpha = None
    if info.alpha_id:
        ainfo = hf.image_info(info.alpha_id)
        if ainfo.is_grid:     # the alpha image is decoded like any image item (context.cc:2040-2071): a grid of its own
            apl = [decode_planes(data, info.alpha_id, picture, transform)[0][0]]
            alpha = apl[0]    # decode_planes applied the alpha item's own transformations already
        else:
            s = hf.coded_stream(info.alpha_id)
            apl = picture(s, hb.parse_picture(s, host_only=True))
            alpha = transform([apl[0]], ainfo)[0]
    planes = transform(planes, info)
    if alpha is not None and alpha.shape != planes[0].shape:
        alpha = scale_nearest(alpha, planes[0].shape[1], planes[0].shape[0])     # context.cc:2064-2071
    return planes, alpha, cf, bd, nclx


def _tdiv(a, b):
    """C integer division (truncation toward zero)"""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b >= 0) else -q


class _Frac:
    """libheif's Fraction (box.cc:51-147): 32-bit numerator / denominator, halved until they fit, truncating division"""

    def __init__(self, n, d, wide=False):
        if wide:
            lo, hi = -(1 << 31), (1 << 31) - 1
            while n < lo or n > hi or d < lo or d > hi:
                n = _tdiv(n + (1 if n >= 0 else -1), 2)
                d = _tdiv(d + (1 if d >= 0 else -1), 2)
        else:
            while d > 0x10000 or d < -0x10000:
                n, d = _tdiv(n, 2), _tdiv(d, 2)
            while d > 1 and (n > 0x10000 or n < -0x10000):
                n, d = _tdiv(n, 2), _tdiv(d, 2)
        self.n, self.d = n, d

    def add(self, b):
        return _Frac(self.n + b.n, self.d, True) if self.d == b.d else _Frac(self.n * b.d + b.n * self.d, self.d * b.d, True)

    def sub(self, b):
        return _Frac(self.n - b.n, self.d, True) if self.d == b.d else _Frac(self.n * b.d - b.n * self.d, self.d * b.d, True)

    def addi(self, v):
        return _Frac(self.n + v * self.d, self.d, True)

    def divi(self, v):
        return _Frac(self.n, self.d * v, True)

    def round_down(self):
        return _tdiv(self.n, self.d)

    def round(self):
        return _tdiv(self.n + _tdiv(self.d, 2), self.d)


def _s32(v):
    return v - (1 << 32) if v >= (1 << 31) else v


def clap_window(c, w, h):
    """(left, top, right, bottom) of a clap box on a w x h image: Box_clap::*_rounded (box.cc:3771-3804) + context.cc:1990-2003"""
    caw, cah = _Frac(c[0], c[1]), _Frac(c[2], c[3])
    hoff, voff = _Frac(_s32(c[4]), c[5]), _Frac(_s32(c[6]), c[7])
    left = hoff.add(_Frac(w - 1, 2)).sub(caw.addi(-1).divi(2)).round_down()
    right = caw.addi(-1).addi(left).round()
    top = voff.add(_Frac(h - 1, 2)).sub(cah.addi(-1).divi(2)).round()
    bottom = cah.addi(-1).addi(top).round()
    return max(left, 0), max(top, 0), min(right, w - 1), min(bottom, h - 1)


# irot / imir as the dihedral map of hc_batch_set_canvas_transform: (swap, flip_x, flip_y)
_DIHEDRAL = {1: (1, 1, 0), 2: (0, 1, 1), 3: (1, 0, 1), 4: (0, 1, 0), 5: (0, 0, 1)}


def _transform_all(planes, info):
    """irot / imir / clap in ipma order, plane by plane (context.cc:1955-2016, pixelimage.cc:539-870); planes[0] has the
    image size"""
    nclap = 0
    for k in range(info.n_transforms):
        op = info.transforms[k]
        H, W = planes[0].shape
        if op in _DIHEDRAL:
            planes = [dihedral(p, *_DIHEDRAL[op]) for p in planes]
        elif op == 6:
            planes = crop_planes(planes, clap_window(list(info.claps[nclap]), W, H))
            nclap += 1
    return [np.ascontiguousarray(p) for p in planes]


def decode_rgb(data, out_format, item_id=None, upsampling=0, picture=_oracle_picture):
    planes, alpha, cf, bd, (matrix, full, primaries) = decode_planes(data, item_id, picture)
    return csc(planes, cf, bd, matrix, full, out_format, alpha, primaries, upsampling)
