"""Thin object wrappers over the C ABI. Names follow the reference's domain: pictures, tiles, grid
canvases, planes (libheif/context.cc, libheif/plugins/decoder_libde265.cc)."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import CscParams, HeifCudaError, HeifImageInfo, check

STREAM_LENGTH_PREFIXED, STREAM_ANNEXB, STREAM_SINGLE_NAL = 0, 1, 2
OUT_RGB, OUT_RGBA, OUT_RRGGBB_BE, OUT_RRGGBBAA_BE, OUT_RRGGBB_LE, OUT_RRGGBBAA_LE = range(6)
OUT_BYTES_PER_PIXEL = {OUT_RGB: 3, OUT_RGBA: 4, OUT_RRGGBB_BE: 6, OUT_RRGGBBAA_BE: 8, OUT_RRGGBB_LE: 6, OUT_RRGGBBAA_LE: 8}
OUT_YCBCR = 6    # native planes (heif_colorspace_undefined / heif_chroma_undefined), packed Y, Cb, Cr, A: see plane_layout
STAGE_DEBLOCK, STAGE_SAO, STAGE_ALL = 1, 2, 3
ROLE_COLOUR, ROLE_ALPHA = 0, 1


class Records:
    """Parsed records of one coded picture (hc_records)."""

    def __init__(self, L, handle):
        self._L, self._h = L, handle

    @property
    def pic(self):
        return self._L.hc_records_pic(self._h).contents

    def array(self, name):
        """(pointer, element count) of one record array: ctus, blks, tbs, coeffs, edge_map, qp_map, scaling"""
        n = C.c_size_t()
        p = getattr(self._L, "hc_records_" + name)(self._h, C.byref(n))
        return p, n.value

    @property
    def upload_bytes(self):
        return self._L.hc_records_upload_bytes(self._h)

    def close(self):
        if self._h:
            self._L.hc_records_free(self._h)
            self._h = None

    def __del__(self):
        self.close()


def parse_picture(data, stream_format=STREAM_LENGTH_PREFIXED, host_only=False):
    """Host front-end: NAL stream of one picture -> Records (serial CABAC parse on the CPU)."""
    L = _lib.load(host_only)
    h = L.hc_parse_picture(data, len(data), stream_format)
    if not h:
        raise HeifCudaError("bitstream: " + (L.hc_last_error() or b"").decode())
    return Records(L, h)


def parse_picture_k0(data, stream_format=STREAM_LENGTH_PREFIXED, host_only=False):
    """The K0 core (device CABAC parser) executed on the CPU -> Records in the host parser's form.
    Raises HeifCudaError("not eligible ...") for pictures K0 leaves to the host parser."""
    L = _lib.load(host_only)
    h = L.hc_parse_picture_k0(data, len(data), stream_format)
    if not h:
        raise HeifCudaError((L.hc_last_error() or b"").decode())
    return Records(L, h)


class K0Picture:
    """Headers of one picture prepared for K0, the device CABAC parser (hc_k0_picture)."""

    def __init__(self, data, stream_format=STREAM_LENGTH_PREFIXED, host_only=False):
        self._L = _lib.load(host_only)
        self._h = self._L.hc_k0_prepare(data, len(data), stream_format)
        if not self._h:
            raise HeifCudaError("bitstream: " + (self._L.hc_last_error() or b"").decode())

    @property
    def eligible(self):
        return bool(self._L.hc_k0_eligible(self._h))

    @property
    def why_not(self):
        return (self._L.hc_k0_why_not(self._h) or b"").decode()

    @property
    def pic(self):
        return self._L.hc_k0_pic(self._h).contents

    @property
    def upload_bytes(self):
        return self._L.hc_k0_upload_bytes(self._h)

    def close(self):
        if self._h:
            self._L.hc_k0_free(self._h)
            self._h = None

    def __del__(self):
        self.close()


class HeifFile:
    """ISO-BMFF/HEIF item resolver (hc_heif)."""

    def __init__(self, data, host_only=False):
        self._L = _lib.load(host_only)
        self._buf = C.create_string_buffer(data, len(data))  # must outlive the handle
        self._h = self._L.hc_heif_open(self._buf, len(data))
        if not self._h:
            raise HeifCudaError("container: " + (self._L.hc_last_error() or b"").decode())

    @property
    def primary_id(self):
        return self._L.hc_heif_primary_id(self._h)

    def top_level_ids(self):
        ids = (C.c_uint32 * 64)()
        n = self._L.hc_heif_top_level_ids(self._h, ids, 64)
        return list(ids[:min(n, 64)])

    def image_info(self, item_id):
        info = HeifImageInfo()
        check(self._L, self._L.hc_heif_get_image_info(self._h, item_id, C.byref(info)), "hc_heif_get_image_info")
        return info

    def overlay(self, item_id):
        """hc_heif_get_overlay: the 'iovl' description of an overlay item (raises for other items)"""
        from ._lib import HeifOverlayInfo
        info = HeifOverlayInfo()
        check(self._L, self._L.hc_heif_get_overlay(self._h, item_id, C.byref(info)), "hc_heif_get_overlay")
        return info

    def grid_tiles(self, item_id):
        tiles = (C.c_uint32 * 4096)()
        n = check(self._L, self._L.hc_heif_grid_tiles(self._h, item_id, tiles, 4096), "hc_heif_grid_tiles")
        return list(tiles[:n])

    def coded_stream(self, item_id):
        out, size = C.c_void_p(), C.c_size_t()
        check(self._L, self._L.hc_heif_coded_stream(self._h, item_id, C.byref(out), C.byref(size)), "hc_heif_coded_stream")
        data = C.string_at(out, size.value)
        self._L.hc_free(out)
        return data

    def close(self):
        if self._h:
            self._L.hc_heif_close(self._h)
            self._h = None

    def __del__(self):
        self.close()


UPSAMPLE_NEAREST, UPSAMPLE_BILINEAR = 0, 1


def csc_select(matrix, primaries, full_range, chroma_format, bit_depth, has_alpha, out_format, host_only=False, upsampling=UPSAMPLE_NEAREST):
    L = _lib.load(host_only)
    p = CscParams()
    check(L, L.hc_csc_select_opt(matrix, primaries, int(full_range), chroma_format, bit_depth, int(has_alpha), out_format, int(upsampling),
                                 C.byref(p)), "hc_csc_select")
    return p


def plane_layout(desc, host_only=False):
    """hc_image_plane_layout: (total bytes, [(offset, stride, width, height) of Y, Cb, Cr, A]) of an OUT_YCBCR image; planes the
    image lacks have width 0. total is 0 for a desc of another output format."""
    L = _lib.load(host_only)
    off, stride = (C.c_size_t * 4)(), (C.c_size_t * 4)()
    w, h = (C.c_int32 * 4)(), (C.c_int32 * 4)()
    total = L.hc_image_plane_layout(C.byref(desc), off, stride, w, h)
    return total, [(off[k], stride[k], w[k], h[k]) for k in range(4)]


def split_planes(desc, packed):
    """The planes of one packed OUT_YCBCR image (1-D uint8 array) as 2-D views: uint8, or little-endian uint16 above 8 bit."""
    total, planes = plane_layout(desc)
    dt = np.uint8 if desc.bit_depth == 8 else np.dtype("<u2")
    return [packed[o:o + s * h].view(dt).reshape(h, w) for o, s, w, h in planes if w]


class Engine:
    """Device engine on one GPU (hc_engine). Raises when no CUDA device / CUDA build is available."""

    def __init__(self, device=0):
        self._L = _lib.load(False)
        self._h = self._L.hc_engine_create(device)
        if not self._h:
            raise HeifCudaError("engine: " + (self._L.hc_last_error() or b"").decode())

    def batch(self):
        return Batch(self)

    def set_option(self, name, value):
        """"device_parse": 1 = K0 parses the slice data on the GPU (default), 0 = host CABAC parser; "scale_max_side": S > 0
        delivers HeicJob / decode_stream images whose longer side exceeds S scaled to fit S (include/heifcuda.h)"""
        check(self._L, self._L.hc_engine_set_option(self._h, name.encode(), int(value)), "set_option")

    def get_option(self, name):
        return self._L.hc_engine_get_option(self._h, name.encode())

    def close(self):
        if self._h:
            self._L.hc_engine_destroy(self._h)
            self._h = None


class Batch:
    """A set of pictures placed on destination canvases, reconstructed together (hc_batch)."""

    def __init__(self, engine):
        self._L, self._eng = engine._L, engine
        self._h = self._L.hc_batch_create(engine._h)
        if not self._h:
            raise HeifCudaError("batch: " + (self._L.hc_last_error() or b"").decode())
        self._canvases = []
        self._out_size = {}      # canvas -> delivered (width, height) set by set_output_size
        self._keep = []

    def add_canvas(self, width, height, chroma_format, bit_depth, with_alpha=False):
        c = check(self._L, self._L.hc_batch_add_canvas(self._h, width, height, chroma_format, bit_depth, int(with_alpha)), "add_canvas")
        self._canvases.append((width, height, chroma_format, bit_depth, with_alpha))
        return c

    def add_picture(self, rec, canvas, x=0, y=0, role=ROLE_COLOUR, rescale_limited=False):
        self._keep.append(rec)
        return check(self._L, self._L.hc_batch_add_picture(self._h, rec._h, canvas, x, y, role, int(rescale_limited)), "add_picture")

    def add_k0_picture(self, k0pic, canvas, x=0, y=0, role=ROLE_COLOUR, rescale_limited=False):
        """a picture whose slice data the GPU parses (K0)"""
        self._keep.append(k0pic)
        return check(self._L, self._L.hc_batch_add_k0_picture(self._h, k0pic._h, canvas, x, y, role, int(rescale_limited)), "add_k0_picture")

    def set_output_size(self, canvas, width, height):
        """hc_batch_set_canvas_output_size: deliver the canvas as width x height pixels sampled by nearest neighbour from its
        full-size converted image (heif_image_scale_image); read_plane keeps returning the full-size planes"""
        check(self._L, self._L.hc_batch_set_canvas_output_size(self._h, canvas, width, height), "set_output_size")
        self._out_size[canvas] = (width, height)

    def upload(self):
        check(self._L, self._L.hc_batch_upload(self._h), "upload")

    def reconstruct(self, stages=STAGE_ALL):
        check(self._L, self._L.hc_batch_reconstruct(self._h, stages), "reconstruct")

    def convert(self, canvas, params):
        check(self._L, self._L.hc_batch_convert(self._h, canvas, C.byref(params)), "convert")

    def sync(self):
        check(self._L, self._L.hc_batch_sync(self._h), "sync")

    def plane_shape(self, canvas, plane):
        w, h, cf, bd, _ = self._canvases[canvas]
        if plane in (1, 2):
            if cf in (1, 2):
                w = (w + 1) // 2
            if cf == 1:
                h = (h + 1) // 2
        return h, w

    def read_plane(self, canvas, plane):
        h, w = self.plane_shape(canvas, plane)
        dt = np.uint8 if self._canvases[canvas][3] == 8 else np.uint16
        out = np.empty((h, w), dt)
        check(self._L, self._L.hc_batch_read_plane(self._h, canvas, plane, out.ctypes.data, out.strides[0]), "read_plane")
        return out

    def read_rgb(self, canvas, out_format):
        w, h = self._out_size.get(canvas, self._canvases[canvas][:2])
        out = np.empty((h, w * OUT_BYTES_PER_PIXEL[out_format]), np.uint8)
        check(self._L, self._L.hc_batch_read_rgb(self._h, canvas, out.ctypes.data, out.strides[0]), "read_rgb")
        return out

    def read_residual(self, pic_index, count):
        out = np.empty(count, np.int16)
        check(self._L, self._L.hc_batch_read_residual(self._h, pic_index, out.ctypes.data, count), "read_residual")
        return out

    def stage_ms(self):
        ms = (C.c_float * 8)()
        check(self._L, self._L.hc_batch_stage_ms(self._h, ms), "stage_ms")
        return dict(zip(("h2d", "k1_transform", "k2_intra", "k3_deblock", "k4_sao", "k5_csc", "d2h", "k0_parse"), list(ms)[:8]))

    @property
    def launch_count(self):
        return self._L.hc_batch_launch_count(self._h)

    @property
    def upload_bytes(self):
        return self._L.hc_batch_upload_bytes(self._h)

    def close(self):
        if self._h:
            self._L.hc_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


def _place_image(hf, batch, item_id):
    """Adds one top-level HEIF image (single picture or grid + optional alpha) to a batch.
    Mirrors HeifContext::decode_image_planar / decode_full_grid_image (context.cc:1729-2404).
    Returns (canvas, effective nclx tuple (matrix, primaries, full_range), has_alpha, bit_depth, chroma_format)."""
    info = hf.image_info(item_id)
    # this stage-level helper places pictures only; the native job (hc_heic_job, HeicJob) is what applies irot / imir /
    # clap and rescales an alpha image of another size — refuse rather than return an untransformed image
    if info.n_transforms:
        raise HeifCudaError("item %d carries transformations: decode it through HeicJob" % item_id)
    if info.alpha_id and hf.image_info(info.alpha_id).n_transforms:
        raise HeifCudaError("the alpha image of item %d carries transformations: decode it through HeicJob" % item_id)
    recs, tiles = [], []
    if info.is_grid:
        ids = hf.grid_tiles(item_id)
        for t in ids:
            recs.append(parse_picture(hf.coded_stream(t)))
        p0 = recs[0].pic
        tw, th = p0.crop_w, p0.crop_h
        canvas = batch.add_canvas(info.width, info.height, p0.chroma_format, p0.bit_depth_y, bool(info.alpha_id))
        for i, r in enumerate(recs):
            x0, y0 = (i % info.cols) * tw, (i // info.cols) * th
            tinfo = hf.image_info(ids[i])
            full = tinfo.full_range if tinfo.nclx_present else r.pic.full_range
            matrix = tinfo.matrix if tinfo.nclx_present else r.pic.matrix_coeffs
            # context.cc:2504: tiles with limited-range nclx and matrix != 0 are rescaled while pasting
            batch.add_picture(r, canvas, x0, y0, ROLE_COLOUR, rescale_limited=(not full) and matrix != 0)
        # the grid canvas carries no nclx (SURVEY hazard 6) unless the grid item has a colr box
        nclx = (info.matrix, info.primaries, info.full_range) if info.nclx_present else (2, 2, 1)
        cf, bd = p0.chroma_format, p0.bit_depth_y
    else:
        r = parse_picture(hf.coded_stream(item_id))
        p = r.pic
        canvas = batch.add_canvas(p.crop_w, p.crop_h, p.chroma_format, p.bit_depth_y, bool(info.alpha_id))
        batch.add_picture(r, canvas, 0, 0, ROLE_COLOUR)
        # container colr(nclx) overrides the bitstream VUI (context.cc:1844-1847)
        nclx = (info.matrix, info.primaries, info.full_range) if info.nclx_present else (p.matrix_coeffs, p.colour_primaries, p.full_range)
        cf, bd = p.chroma_format, p.bit_depth_y
    if info.alpha_id:
        a = parse_picture(hf.coded_stream(info.alpha_id))
        cw, ch = (info.width, info.height) if info.is_grid else (recs[0].pic.crop_w if recs else p.crop_w, recs[0].pic.crop_h if recs else p.crop_h)
        if (a.pic.crop_w, a.pic.crop_h) != (cw, ch):
            raise HeifCudaError("the alpha image of item %d has another size: decode it through HeicJob" % item_id)
        batch.add_picture(a, canvas, 0, 0, ROLE_ALPHA)
    return canvas, nclx, bool(info.alpha_id), bd, cf


def decode_heic(engine, data, out_format=OUT_RGB, item_id=None):
    """HEIC file bytes -> interleaved RGB rows (numpy uint8 [h, w*bytes_per_pixel]), the Python
    twin of heif_decode_image(handle, &img, heif_colorspace_RGB, heif_chroma_interleaved_*, NULL).
    The primary image goes through the native job (hc_heic_job: transformations, alpha of any size, every output format);
    another item of the file (item_id) through the stage-level calls, which refuse what they do not apply."""
    hf = HeifFile(data)
    if item_id is None or item_id == hf.primary_id:
        hf.close()
        job = HeicJob(engine, [data], out_format=out_format)
        try:
            job.upload()
            job.run()
            return job.read_rgb(0)
        finally:
            job.close()
    batch = engine.batch()
    try:
        canvas, (matrix, primaries, full_range), has_alpha, bd, cf = _place_image(hf, batch, item_id or hf.primary_id)
        params = csc_select(matrix, primaries, full_range, cf, bd, has_alpha, out_format)
        batch.upload()
        batch.reconstruct(STAGE_ALL)
        batch.convert(canvas, params)
        return batch.read_rgb(canvas, out_format)
    finally:
        batch.close()
        hf.close()


class HeicJob:
    """Many HEIC files -> interleaved RGB through the native batch path (hc_heic_job): host threads
    parse every coded item, the GPU reconstructs all of them as one batch."""

    def __init__(self, engine, files, want_alpha=False, threads=0, out_format=None):
        """out_format: one of OUT_* for every image whatever its bit depth (HC_OUTPUT_FORMAT), default by bit depth"""
        from ._lib import ImageDesc
        if out_format is not None:
            want_alpha = 0x100 | int(out_format)
        self._L, self._eng = engine._L, engine
        self._bufs = [C.create_string_buffer(f, len(f)) for f in files]
        n = len(files)
        ptrs = (C.c_char_p * n)(*[C.cast(b, C.c_char_p) for b in self._bufs])
        sizes = (C.c_size_t * n)(*[len(f) for f in files])
        self._h = self._L.hc_heic_job_create(engine._h, n, ptrs, sizes, int(want_alpha), threads)
        if not self._h:
            raise HeifCudaError("heic job: " + (self._L.hc_last_error() or b"").decode())
        self.descs = []
        for i in range(self._L.hc_heic_job_image_count(self._h)):
            d = ImageDesc()
            check(self._L, self._L.hc_heic_job_image_desc(self._h, i, C.byref(d)), "image_desc")
            self.descs.append(d)

    def upload(self):
        check(self._L, self._L.hc_heic_job_upload(self._h), "upload")

    def run(self):
        check(self._L, self._L.hc_heic_job_run(self._h), "run")

    def sync(self):
        check(self._L, self._L.hc_heic_job_sync(self._h), "sync")

    def read_rgb(self, image, out=None):
        d = self.descs[image]
        if d.out_format == OUT_YCBCR:
            raise HeifCudaError("image %d is planar (OUT_YCBCR): read it with read_planes" % image)
        if out is None:
            out = np.empty((d.height, d.width * d.bytes_per_pixel), np.uint8)
        check(self._L, self._L.hc_heic_job_read_rgb(self._h, image, out.ctypes.data, out.strides[0]), "read_rgb")
        return out

    def read_planes(self, image):
        """OUT_YCBCR jobs: the planes of an image (Y, Cb, Cr, A as the image has them) from ONE read of its packed bytes"""
        d = self.descs[image]
        total, _ = plane_layout(d)
        if not total:
            raise HeifCudaError("image %d is not planar: create the job with out_format=OUT_YCBCR" % image)
        buf = np.empty(total, np.uint8)
        check(self._L, self._L.hc_heic_job_read_rgb(self._h, image, buf.ctypes.data, d.width * d.bytes_per_pixel), "read_planes")
        return split_planes(d, buf)

    def read_plane(self, image, plane):
        d = self.descs[image]
        w, h = d.width, d.height
        if plane in (1, 2):
            if d.chroma_format in (1, 2):
                w = (w + 1) // 2
            if d.chroma_format == 1:
                h = (h + 1) // 2
        out = np.empty((h, w), np.uint8 if d.bit_depth == 8 else np.uint16)
        check(self._L, self._L.hc_heic_job_read_plane(self._h, image, plane, out.ctypes.data, out.strides[0]), "read_plane")
        return out

    def stage_ms(self):
        ms = (C.c_float * 8)()
        check(self._L, self._L.hc_heic_job_stage_ms(self._h, ms), "stage_ms")
        return dict(zip(("h2d", "k1_transform", "k2_intra", "k3_deblock", "k4_sao", "k5_csc", "d2h", "k0_parse"), list(ms)[:8]))

    def timer_start(self):
        check(self._L, self._L.hc_heic_job_timer_start(self._h), "timer_start")

    def timer_stop_ms(self):
        ms = C.c_float()
        check(self._L, self._L.hc_heic_job_timer_stop_ms(self._h, C.byref(ms)), "timer_stop_ms")
        return ms.value

    @property
    def launch_count(self):
        return self._L.hc_heic_job_launch_count(self._h)

    @property
    def upload_bytes(self):
        return self._L.hc_heic_job_upload_bytes(self._h)

    @property
    def parse_seconds(self):
        return self._L.hc_heic_job_parse_seconds(self._h)

    def close(self):
        if self._h:
            self._L.hc_heic_job_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


def decode_stream(engine, files, on_image=None, want_alpha=False, threads=0, files_per_batch=8, out_format=None, dests=None,
                  isolate_errors=False):
    """Long file lists (hc_heic_decode_stream): host parse of batch b+1 overlaps upload + kernels + read-back of
    batch b. on_image(file_index, desc, rows) gets every image as a numpy view [h, w*bytes_per_pixel] of PINNED
    host memory that is only valid inside the callback; with out_format=OUT_YCBCR `rows` is instead the list of the image's
    planes (split_planes), views of the same kind. Returns the hc_stream_stats as a dict.
    dests: per file a writable uint8 array or None; [rows, stride] for interleaved output, 1-D (the packed bytes) for OUT_YCBCR.
    isolate_errors: a file that cannot be decoded does not fail the call; the dict gains "file_status" (one HC_* code per
    file, 0 = delivered) and "first_error" (text)."""
    from ._lib import IMAGE_CALLBACK, StreamStats
    L = engine._L
    if out_format is not None:
        want_alpha = 0x100 | int(out_format)    # HC_OUTPUT_FORMAT
    bufs = {}
    ptr_list = []
    for f in files:                         # identical bytes objects share one buffer
        if id(f) not in bufs:
            bufs[id(f)] = C.create_string_buffer(f, len(f))
        ptr_list.append(C.cast(bufs[id(f)], C.c_char_p))
    n = len(files)
    ptrs = (C.c_char_p * n)(*ptr_list)
    sizes = (C.c_size_t * n)(*[len(f) for f in files])

    def _cb(_user, index, desc, pixels, stride):
        if on_image is not None:
            d = desc.contents
            if d.out_format == OUT_YCBCR:
                total, _ = plane_layout(d)
                on_image(index, d, split_planes(d, np.ctypeslib.as_array((C.c_uint8 * total).from_address(pixels))))
                return
            rows = np.ctypeslib.as_array((C.c_uint8 * (stride * d.height)).from_address(pixels)).reshape(d.height, stride)
            on_image(index, d, rows)

    cb = IMAGE_CALLBACK(_cb)
    st = StreamStats()
    xd = None
    if dests is not None:    # external destinations: one writable uint8 numpy array (or None) per file
        from ._lib import StreamDest
        xd = (StreamDest * n)()
        for k, a in enumerate(dests):
            if a is not None:
                xd[k].dst, xd[k].len, xd[k].stride = a.ctypes.data, a.nbytes, a.strides[0] if a.ndim > 1 else 0
    status = (C.c_int * n)() if isolate_errors else None
    check(L, L.hc_heic_decode_stream_ext(engine._h, n, ptrs, sizes, int(want_alpha), threads, files_per_batch, xd, status, cb, None,
                                         C.byref(st)), "hc_heic_decode_stream")
    out = {k: getattr(st, k) for k, _ in StreamStats._fields_}
    if isolate_errors:
        out["file_status"] = list(status)
        out["first_error"] = (L.hc_last_error() or b"").decode() if st.files_failed else ""
    return out
