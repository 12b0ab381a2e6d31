#!/usr/bin/env python
"""bench.py — decoded MP/s HEIC -> RGB on B200 (BASELINE.json metric), one JSON line on stdout.

Workloads (--workload, config.workload names the one on the line):
  c2 (default) BASELINE config C2 — 4032x3024 "iPhone-style" grid of 48 (8x6) 512x512 HEVC intra tiles, 8-bit 4:2:0,
               CTB 64, WPP, SAO + deblocking, QP 26, full-range BT.601 VUI -> interleaved RGB; one step = `--images`
               files (default 32 = 1536 coded pictures in flight), `--distinct` different files (default 8)
  c4           BASELINE config C4 — a list of 1920x1080 single-picture HEIC files sharded by image across the ranks
               (same coding tools; a 1080p picture is 17 WPP rows of 30 CTBs); one step = `--images` files (default 192)
  c5           BASELINE config C5 — ONE 11520x8704 grid of 391 tiles, tile rows split across the ranks (strong scaling),
               every rank's K5 writing its band straight into rank 0's buffer over NVLink (hc_shared_image)
The default run also carries a short c4 and a c5 measurement as the keys "c4" / "c5" of the same line.
Content is synthetic (tools/hevc_enc closed-loop encoder + tools/heif_writer), generated untimed at start-up.

  value : whole-job MP/s of the device path as SURVEY 8(d) defines the metric — per step the H2D copy of the step's inputs
          (RBSP bytes + headers for the device parser, packed records for --parser host), K0 (device CABAC parse) and
          K1..K5, each timed with CUDA events on the stream it runs on; inputs in pinned host memory, outputs left in HBM.
          `value_reconstruction_only` is K1..K5 alone with the records resident (what round 1 called `value`).
  e2e   : the same metric through the C ABI (hc_heic_decode_stream) from HEIC bytes in host memory to RGB bytes in
          pinned host memory: container + header parse, slice-data parse (K0 on the GPU, plus the share the host
          threads take meanwhile; --parser host: host threads only), H2D, K1..K5 and D2H inside the timed region
  roofline     : the dominant reconstruction kernel's algorithmic bytes / its CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline : the unmodified reference (oracle/_ref: libheif + libde265, heif_decode_image -> RGB) on
                 the host cores, bounded sample of the same file

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c4|c5] [--dump-outputs DIR]
Every GPU measurement times exactly K steps. The content is seeded, so the same arguments give the same inputs on every run;
--dump-outputs DIR writes what the timed path computed in its last step, so that two builds can be compared output for output.
Launched under torchrun for N > 1 (one rank per GPU, NCCL only for the barrier / max-over-ranks / the C5 IPC handle).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "heif-decoder-lib_b200"), os.path.join(ROOT, "tests"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

GRID_W, GRID_H, TILE = 4032, 3024, 512
C4_W, C4_H = 1920, 1080
C5_W, C5_H = 11520, 8704
WORKLOADS = {
    "c2": "C2: 4032x3024 grid of 48 512x512 HEVC-intra tiles, 8-bit 4:2:0, CTB64 WPP SAO+deblock QP26 -> RGB24",
    "c4": "C4: list of 1920x1080 single-picture HEIC files sharded by image, 8-bit 4:2:0, CTB64 WPP SAO+deblock QP26 -> RGB24",
    "c5": "C5: one 11520x8704 grid of 391 512x512 tiles, tile rows split across the GPUs, K5 writes into rank 0's buffer over NVLink -> RGB24",
}
STREAM_DEPTH = 6     # the most batches hc_heic_decode_stream keeps in flight (3, or 6 when read-backs are slow: heic_job.cc)
METRIC = "decoded MP/s HEIC->RGB (device-timed)"
UNIT = "MP/s"
STAGES = ("k1_transform", "k2_intra", "k3_deblock", "k4_sao", "k5_csc")
DUMP_BYTES = 60 << 20    # --dump-outputs writes at most this much


def dump_outputs(out_dir, n, read_rgb):
    """--dump-outputs: the n interleaved RGB images of the last timed step (read_rgb(i) -> uint8 array, all of one size) as
    DIR/rgb.npy, float32, one row per image. Images too large for DUMP_BYTES are sampled at fixed, seeded byte positions,
    the same in every image, which go to DIR/rgb_positions.npy."""
    import numpy as np
    size = read_rgb(0).size
    per_image = min(size, DUMP_BYTES // (4 * n + 8))
    pos = np.arange(size) if per_image == size else np.sort(np.random.default_rng(0).choice(size, per_image, replace=False))
    out = np.empty((n, per_image), np.float32)
    for i in range(n):
        out[i] = read_rgb(i).reshape(-1)[pos]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rgb.npy"), out)
    np.save(os.path.join(out_dir, "rgb_positions.npy"), pos.astype(np.float64))


# ---------------------------------------------------------------------------------------------------------- content
def _gen_c2(job):
    i, path = job
    from tools import heif_writer
    wpp = 0 if "_nowpp" in os.path.basename(path) else 1      # --no-wpp: one substream per tile instead of one per CTB row
    data = heif_writer.synth_grid_heic(GRID_W, GRID_H, tile=TILE, seed=100 + i, qp=26, wpp=wpp, sao=1, log2_ctb=6)
    with open(path + ".tmp", "wb") as f:
        f.write(data)
    os.replace(path + ".tmp", path)


def _gen_c4(job):
    i, path = job
    from tools import heif_writer, hevcenc
    stream = hevcenc.encode(hevcenc.synth_image(C4_W, C4_H, 1, 8, 300 + i), qp=26, wpp=1, sao=1, log2_ctb=6, seed=300 + i)
    data = heif_writer.single_image(stream, C4_W, C4_H, 1, 8)
    with open(path + ".tmp", "wb") as f:
        f.write(data)
    os.replace(path + ".tmp", path)


def _make(gen, paths):
    """missing files are encoded in parallel child processes (the encoder is single-threaded, ~10 s per 12 MP file)"""
    todo = [(i, p) for i, p in enumerate(paths) if not os.path.exists(p)]
    limit = max(1, os.cpu_count() or 1)
    running = []
    for job in todo:
        while len(running) >= limit:
            running.pop(0).wait()
        code = "import sys; sys.path.insert(0, %r); import bench; bench.%s((%d, %r))" % (ROOT, gen.__name__, job[0], job[1])
        running.append(subprocess.Popen([sys.executable, "-c", code], stdout=subprocess.DEVNULL))
    for pr in running:
        pr.wait()
    missing = [p for p in paths if not os.path.exists(p)]
    if missing:
        raise RuntimeError("content generation failed for %s" % missing)
    return [open(p, "rb").read() for p in paths]


def make_content(n_distinct, cache_dir, wpp=True):
    """n_distinct synthetic 12 MP grid HEICs (cached on disk between runs of the same box)."""
    os.makedirs(cache_dir, exist_ok=True)
    return _make(_gen_c2, [os.path.join(cache_dir, "c2_%dx%d_t%d_seed%d%s.heic" % (GRID_W, GRID_H, TILE, i, "" if wpp else "_nowpp")) for i in range(n_distinct)])


def make_content_c4(n_distinct, cache_dir):
    os.makedirs(cache_dir, exist_ok=True)
    return _make(_gen_c4, [os.path.join(cache_dir, "c4_%dx%d_seed%d.heic" % (C4_W, C4_H, i)) for i in range(n_distinct)])


def make_content_c5(c2_files, cache_dir):
    """One 11520 x 8704 grid (23 x 17 = 391 tiles) built from the coded tiles of the C2 files, reused cyclically: every
    tile is its own item and its own HEVC picture for the decoder; no further encoding is needed."""
    import heif_b200 as hb
    from tools import heif_writer
    path = os.path.join(cache_dir, "c5_%dx%d_t%d_from%d.heic" % (C5_W, C5_H, TILE, len(c2_files)))
    if not os.path.exists(path):
        streams = []
        for data in c2_files:
            hf = hb.HeifFile(data, host_only=True)
            streams += [hf.coded_stream(t) for t in hf.grid_tiles(hf.primary_id)]
            hf.close()
        cols, rows = (C5_W + TILE - 1) // TILE, (C5_H + TILE - 1) // TILE
        tiles = [streams[k % len(streams)] for k in range(cols * rows)]
        data = heif_writer.grid_image(tiles, rows, cols, TILE, TILE, C5_W, C5_H)
        with open(path + ".tmp", "wb") as f:
            f.write(data)
        os.replace(path + ".tmp", path)
    return open(path, "rb").read()


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- reference arms
def reference_arm(files, steps, warmup, threads, mp):
    """The reference's own CPU implementation on all host cores, two ways, the better one is the value:
      (a) its own policy: heif_decode_image(..., RGB, interleaved_RGB) per file with
          heif_context_set_threads(ctx, handle, cores) (grid -> one thread per tile, heif.cc:499-514);
      (b) process-level data parallelism (BASELINE.md section 4): `cores` files decoded concurrently, one thread each."""
    import concurrent.futures as cf
    import refheif as R
    if not R.available():
        return None
    f0 = files[0]
    for _ in range(warmup):
        R.decode(f0, R.COLORSPACE_RGB, R.CHROMA_RGB, threads=threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        R.decode(f0, R.COLORSPACE_RGB, R.CHROMA_RGB, threads=threads)
    dt_a = (time.perf_counter() - t0) / steps
    with cf.ThreadPoolExecutor(max_workers=threads) as pool:   # ctypes releases the GIL inside heif_decode_image
        def one(k):
            R.decode(files[k % len(files)], R.COLORSPACE_RGB, R.CHROMA_RGB, threads=1)
        list(pool.map(one, range(threads)))                    # warm-up
        t0 = time.perf_counter()
        n = threads * max(1, min(steps, 2))
        list(pool.map(one, range(n)))
        dt_b = (time.perf_counter() - t0) / n
    best = min(dt_a, dt_b)
    return {"value": mp / best, "ms_per_step": best * 1e3,
            "sample": "one %.2f MP file: (a) %d decoder threads %.1f MP/s, (b) %d concurrent single-thread decodes %.1f MP/s" % (
                mp, threads, mp / dt_a, threads, mp / dt_b)}


def plugin_arm(files, threads):
    """Level-1 drop-in: the UNMODIFIED reference libheif (oracle/_ref) decodes the same file through its own
    heif_decode_image, with libheif-cuda.so loaded by heif_load_plugin and selected as decoder ("cuda"); the reference's
    libde265 plugin is timed through the very same call for comparison, and the two outputs are compared."""
    import ctypes as C
    import hashlib
    import refheif as R
    plugin = os.path.join(ROOT, "heif-decoder-lib_b200", "plugins", "libheif-cuda.so")
    if not R.available() or not os.path.exists(plugin):
        return None
    try:
        L = R.lib()
        os.environ["HEIFCUDA_LIBHEIF"] = os.path.join(R.REF_DIR, "libheifref.so")
        info = C.c_void_p()
        err = L.heif_load_plugin(plugin.encode(), C.byref(info))
        if err.code != 0:
            return {"error": (err.message or b"").decode()}
        R.FOREIGN_PLUGIN_LOADED = True
        f0 = files[0]
        mp = GRID_W * GRID_H / 1e6
        want = R.decode(f0, R.COLORSPACE_RGB, R.CHROMA_RGB, threads=threads, decoder_id="libde265")["interleaved"][0]
        got = R.decode(f0, R.COLORSPACE_RGB, R.CHROMA_RGB, threads=threads, decoder_id="cuda")["interleaved"][0]   # also the warm-up
        for _ in range(3):                                                                                          # pools, clocks
            R.decode(f0, R.COLORSPACE_RGB, R.CHROMA_RGB, threads=threads, decoder_id="cuda")
        def median_time(decoder, n=7):       # single decodes of one file vary by tens of per cent: the median of seven
            ts = []
            for _ in range(n):
                t0 = time.perf_counter()
                R.decode(f0, R.COLORSPACE_RGB, R.CHROMA_RGB, threads=threads, decoder_id=decoder)
                ts.append(time.perf_counter() - t0)
            return sorted(ts)[n // 2]
        dt = median_time("cuda")
        dt_ref = median_time("libde265")
        return {"value": mp / dt, "unit": UNIT, "ms_per_image": dt * 1e3, "tile_threads": threads,
                "libde265_plugin_same_call": {"value": mp / dt_ref, "ms_per_image": dt_ref * 1e3},
                "bit_exact_vs_libde265_plugin": hashlib.md5(got).digest() == hashlib.md5(want).digest(),
                "what": "unmodified reference libheif, heif_decode_image -> RGB, decoder plugin = libheif-cuda.so (one file at a time; "
                        "grid paste and colour conversion stay on the CPU inside libheif)"}
    except Exception as e:   # never fail the measurement on the optional arm
        return {"error": str(e)}


# ------------------------------------------------------------------------------------------------- GPU measurements
def measure_list(hb, eng, files, steps, warmup, threads, images, barrier, max_over_ranks, local_rank, sample_clocks=True, dump_dir=None):
    """Image-list workloads (c2, c4): device-timed figures and the e2e stream figure (times already max-ed over the ranks).
    dump_dir: where the RGB images of the last step of the `value` loop go (dump_outputs)."""
    import numpy as np
    job = hb.HeicJob(eng, files, want_alpha=False, threads=threads)
    job.upload()
    for _ in range(warmup):
        job.run()
    job.sync()
    stage = job.stage_ms()
    sampler = ClockSampler(local_rank) if sample_clocks else None
    if sampler:
        sampler.start()
        step_ms = max(1e-3, sum(stage[k] for k in STAGES))
        for _ in range(int(600.0 / step_ms) + 1):      # >= 0.6 s of load for nvidia-smi's polling
            job.run()
        job.sync()
    # (1) reconstruction only: K steps of K1..K5, records resident, one event pair around all of them
    barrier()
    job.timer_start()
    for _ in range(steps):
        job.run()
    recon_ms = max_over_ranks(job.timer_stop_ms()) / steps
    stage_recon = job.stage_ms()
    # (2) the metric as SURVEY 8(d) defines it: per step H2D of the step's inputs + K0 + K1..K5, each from the CUDA events
    # of the stream it runs on (the host-side packing between two steps is not device time and is not counted)
    barrier()
    dev_ms, acc, launches = 0.0, {}, 0
    for _ in range(steps):
        job.upload()
        job.run()
        st = job.stage_ms()           # synchronises
        dev_ms += st["h2d"] + st["k0_parse"] + sum(st[k] for k in STAGES)
        launches += job.launch_count
        for k, v in st.items():
            acc[k] = acc.get(k, 0.0) + v / steps
    barrier()
    dev_ms = max_over_ranks(dev_ms) / steps
    clocks = sampler.stop() if sampler else None
    upload_bytes = job.upload_bytes
    try:   # parity guard: the timed configuration still produces the reference's pixels (the oracle is only the checker)
        import heic_oracle
        check = bool(np.array_equal(job.read_rgb(0), heic_oracle.decode_rgb(files[0], hb.OUT_RGB)))
    except Exception as e:
        check = "unchecked: %s" % e
    if dump_dir:
        dump_outputs(dump_dir, len(files), job.read_rgb)
    job.close()

    # end to end: one call of the public streaming API. The figure is the STEADY-STATE period of the pipeline: deliveries of
    # the first and the last depth - 1 batches are left out (`depth` batches are in flight: the first delivery comes late
    # relative to the ones behind it, the last batches drain without successors — over 40 batches the first-to-last figure
    # is 6 % better than the middle of the run, tools/stream_depth_probe.py), so 2 * skip + 1 + e2e_steps batches are decoded.
    e2e_steps = steps
    skip = STREAM_DEPTH - 1   # deliveries left out at either end: the batches in flight behind / ahead of the window
    marks, checksum = [], [0]

    def on_image(index, desc, rows):
        if index % images == images - 1:
            marks.append(time.perf_counter())
        if index == 0:
            checksum[0] = int(rows[::97, ::389].astype(np.uint64).sum())   # touch the pinned result on the host

    # an untimed call first: the engine pins its output buffers (1.3 s per 2.6 GB), fills its device pools and settles how
    # many batches it keeps in flight (3, or 6 when the read-back is slow); a service's later calls look like the timed one
    hb.decode_stream(eng, files * (STREAM_DEPTH + 10), None, want_alpha=False, threads=threads, files_per_batch=images)
    barrier()
    t_start = time.perf_counter()
    st = hb.decode_stream(eng, files * (2 * skip + 1 + e2e_steps), on_image, want_alpha=False, threads=threads, files_per_batch=images)
    barrier()
    e2e_dt = max_over_ranks((marks[-1 - skip] - marks[skip]) / e2e_steps)
    e2e_first_to_last = max_over_ranks((marks[-1] - marks[0]) / (len(marks) - 1))
    return {"dev_ms": dev_ms, "recon_ms": recon_ms, "stage": acc, "stage_recon": stage_recon, "launches": launches, "clocks": clocks,
            "upload_bytes": upload_bytes, "parity": check, "e2e_dt": e2e_dt, "e2e_steps": e2e_steps, "first_batch_s": marks[0] - t_start,
            "e2e_first_to_last": e2e_first_to_last,
            "stream": st}


def measure_c5(hb, eng, data, steps, warmup, threads, rank, world, dist, barrier, max_over_ranks, dump_dir=None):
    """One huge grid, tile rows split across the ranks, every K5 writing its band into rank 0's hc_shared_image.
    dump_dir: where rank 0 writes the stitched image of the last timed step (dump_outputs)."""
    import hashlib
    import torch
    from heif_b200.multigpu import BandJob, SharedImage
    from heif_b200._lib import check
    L = eng._L
    t0 = time.perf_counter()
    job = BandJob(eng, data, rank, world, 0, threads)        # container + headers of this rank's tiles (K0 parses the slice data)
    parse_s = max_over_ranks(time.perf_counter() - t0)
    bpp = 3
    handle = [None]
    shared = None
    if rank == 0:
        shared = SharedImage(eng, job.width, job.full_height, bpp)
        handle[0] = shared.export()
    if world > 1:
        dist.broadcast_object_list(handle, src=0)
        if rank != 0:
            shared = SharedImage(eng, job.width, job.full_height, bpp, handle=handle[0])
    has = job._h is not None
    if has:
        check(L, L.hc_heic_job_set_rgb_target(job._h, 0, shared._h, job.first_row), "hc_heic_job_set_rgb_target")

    def run(upload=False):
        if has:
            if upload:
                check(L, L.hc_heic_job_upload(job._h), "upload")
            check(L, L.hc_heic_job_run(job._h), "run")

    def sync():
        if has:
            check(L, L.hc_heic_job_sync(job._h), "sync")

    # first pass: H2D + K0 + K1..K5 (the device parse happens once per upload), wall clock between two barriers
    barrier()
    t0 = time.perf_counter()
    run(True)
    sync()
    barrier()
    first_s = max_over_ranks(time.perf_counter() - t0)
    st_first = job.stage_ms() if has else {}
    for _ in range(max(0, warmup - 1)):
        run()
    sync()
    barrier()
    if has:
        check(L, L.hc_heic_job_timer_start(job._h), "timer_start")
    for _ in range(steps):
        run()
    ms = ctypes.c_float(0.0)
    if has:
        check(L, L.hc_heic_job_timer_stop_ms(job._h, ctypes.byref(ms)), "timer_stop")
    barrier()
    recon_ms = max_over_ranks(ms.value) / steps
    st = job.stage_ms() if has else {}
    k5_ms = max_over_ranks(st.get("k5_csc", 0.0))
    md5, d2h_s = None, 0.0
    if rank == 0:
        t0 = time.perf_counter()
        full = shared.read()
        d2h_s = time.perf_counter() - t0
        md5 = hashlib.md5(full.tobytes()).hexdigest()
        if dump_dir:
            dump_outputs(dump_dir, 1, lambda i: full)
        del full
    barrier()
    band_rows = job.desc.height if has else 0
    remote = 0.0 if rank == 0 else float(band_rows * job.width * bpp)
    if world > 1:
        t = torch.tensor([remote], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        remote = float(t.item())
    job.close()
    out = {"first_pass_ms": first_s * 1e3, "recon_ms": recon_ms, "k0_ms": max_over_ranks(st_first.get("k0_parse", 0.0)), "k5_ms": k5_ms,
           "parse_s": parse_s, "d2h_s": d2h_s, "md5": md5, "remote_bytes": remote,
           "stage_ms_rank0": {k: round(v, 4) for k, v in st.items()} if rank == 0 else None}
    if rank == 0 and world > 1:    # the stitched image against the whole file decoded as one job on this GPU (untimed)
        j1 = hb.HeicJob(eng, [data], threads=threads)
        j1.upload()
        j1.run()
        out["bit_exact_vs_single_gpu"] = hashlib.md5(j1.read_rgb(0).tobytes()).hexdigest() == md5
        out["k5_ms_single_gpu_local"] = j1.stage_ms()["k5_csc"]
        j1.close()
    barrier()
    shared.close()
    return out


def c5_report(c5, world):
    mp5 = C5_W * C5_H / 1e6
    return {"workload": WORKLOADS["c5"], "scaling": "strong", "value": mp5 / (c5["recon_ms"] * 1e-3), "unit": UNIT, "ms_per_step": c5["recon_ms"],
            "value_what": "K1..K5 of every rank's band, K5 writing into rank 0's buffer, records resident; max over ranks",
            "first_pass_ms_incl_upload_and_k0": c5["first_pass_ms"], "k0_ms": c5["k0_ms"],
            "bit_exact_vs_single_gpu": c5.get("bit_exact_vs_single_gpu"), "md5": c5["md5"],
            "stitch": {"how": "K5 stores its band into rank 0's buffer (hc_shared_image: CUDA IPC mapping, NVLink peer stores) — there is no "
                              "separate stitch pass, so its cost is the difference between K5 with peer writes and K5 with local writes",
                       "remote_bytes_per_step": c5["remote_bytes"], "k5_ms_with_peer_writes_max_over_ranks": c5["k5_ms"],
                       "k5_ms_whole_image_one_gpu_local": c5.get("k5_ms_single_gpu_local"), "nvlink_peak_GBps_per_direction": 900.0,
                       "remote_write_GBps_per_writer": (c5["remote_bytes"] / max(1, world - 1)) / (c5["k5_ms"] * 1e-3) / 1e9
                       if c5["k5_ms"] > 0 and world > 1 else None},
            "stage_ms_rank0": c5["stage_ms_rank0"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every GPU measurement")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--images", type=int, default=0, help="files per step and GPU (default: 64 for c2 — K0 is a wavefront per picture, its ramps "
                    "amortise better over 64 files than 32: value 3.6 -> 3.9 GP/s — and 384 for c4)")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic files (replicated to --images)")
    ap.add_argument("--threads", type=int, default=0, help="host parse threads (0 = all cores)")
    ap.add_argument("--host-share", type=int, default=-1, help="with --parser device: %% of the coded items parsed by the host threads "
                    "meanwhile in the e2e arm (default: engine default)")
    ap.add_argument("--parser", default="device", choices=["device", "host"],
                    help="where the CABAC slice data is parsed: K0 on the GPU (default) or the host parser")
    ap.add_argument("--no-wpp", action="store_true", help="c2 content without wavefront substreams (one CABAC chain per 512 x 512 tile): "
                    "what K0's throughput depends on; not the BASELINE configuration")
    ap.add_argument("--no-numa", action="store_true", help="multi-GPU runs: do not bind a rank's threads to the CPUs next to its GPU")
    ap.add_argument("--skip-baselines", action="store_true", help="kernel experiments: leave out the cpu_baseline and plugin_dropin arms")
    ap.add_argument("--skip-extras", action="store_true", help="leave out the c4 / c5 side measurements of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the RGB images the workload's timed path computed in its last step "
                    "(rank 0's) to DIR/rgb.npy as float32, sampled at the seeded byte positions in DIR/rgb_positions.npy when "
                    "they exceed 60 MiB in all")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    wl = args.workload
    images = args.images or (384 if wl == "c4" else 64)
    if not args.images and wl == "c2":
        # 64 files per step need ~8 GB of pinned host memory per rank in the stream API (three output buffers in flight); a box
        # that cannot give every rank three times that runs 32 files per step. Same answer on every rank of the box.
        try:
            import psutil
            if psutil.virtual_memory().available / max(1, int(os.environ.get("WORLD_SIZE", "1"))) < 24e9:
                images = 32
        except ImportError:
            pass

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    numa = None
    if world > 1 and args.impl != "reference" and not args.no_numa:
        # one rank per GPU on a two-socket box: keep the rank's threads (and with them its pinned buffers, which are placed
        # where they are first touched) on the CPUs next to its GPU, so that uploads and read-backs do not cross the socket link
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (cores + 63) // 64)
            cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
            cpus &= set(os.sched_getaffinity(0))
            if cpus and len(cpus) < cores:
                os.sched_setaffinity(0, cpus)
                numa = "%d cpus next to GPU %d" % (len(cpus), local_rank)
        except Exception as e:      # no NVML, one socket, containers without the right: run unpinned
            numa = "unpinned (%s)" % type(e).__name__
    # the synthetic content is cached outside the tree, which may be read-only; one directory per user, shared by the ranks
    cache = os.path.join(tempfile.gettempdir(), "heif_b200_bench_content_%d" % os.getuid())
    file_mp = {"c2": GRID_W * GRID_H / 1e6, "c4": C4_W * C4_H / 1e6, "c5": C5_W * C5_H / 1e6}[wl]

    if args.impl == "reference":
        if rank != 0:
            return 0
        files = make_content_c4(min(args.distinct, 4), cache) if wl == "c4" else make_content(min(args.distinct, 2), cache)
        if wl == "c5":
            files = [make_content_c5(files, cache)]
        r = reference_arm(files, max(1, min(args.steps, 5 if wl != "c5" else 2)), 1, cores, file_mp)
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref (reference build) is missing"}))
            return 0
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong" if wl == "c5" else "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": WORKLOADS[wl]},
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "reference", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # stdout carries exactly one JSON line: NCCL's version / debug lines go to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    import torch
    import heif_b200 as hb

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the reconstruction path has no CPU fallback")
    torch.cuda.set_device(local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- content (untimed; rank 0 generates, the others read the cache) ----
    def content(fn, *a):
        if rank == 0:
            fn(*a)
        barrier()
        return fn(*a)

    extras = wl == "c2" and not args.skip_extras and not args.no_wpp
    c2_files = content(make_content, args.distinct, cache, not args.no_wpp) if wl in ("c2", "c5") else None
    c4_files = content(make_content_c4, args.distinct, cache) if wl == "c4" or extras else None
    c5_file = content(make_content_c5, c2_files, cache) if wl == "c5" or extras else None

    eng = hb.Engine(local_rank)
    eng.set_option("device_parse", 1 if args.parser == "device" else 0)
    if args.host_share >= 0:
        eng.set_option("host_share_pct", args.host_share)
    threads = args.threads or max(1, cores // max(1, world))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic"}

    if wl in ("c2", "c4"):
        distinct = c2_files if wl == "c2" else c4_files
        files = [distinct[(i + rank) % len(distinct)] for i in range(images)]
        mp_per_step = images * file_mp
        # R: bytes of packed records per output pixel as the host parser emits them (what K1 / K2 read from HBM either way)
        hf = hb.HeifFile(files[0], host_only=False)
        first_item = hf.grid_tiles(hf.primary_id)[0] if wl == "c2" else hf.primary_id
        rec0 = hb.parse_picture(hf.coded_stream(first_item))
        rec_bytes_per_px = rec0.upload_bytes / float(rec0.pic.width * rec0.pic.height)
        hf.close()
        m = measure_list(hb, eng, files, args.steps, args.warmup, threads, images, barrier, max_over_ranks, local_rank,
                         dump_dir=args.dump_outputs if rank == 0 else None)
        st = m["stream"]
        # ---- roofline of the dominant reconstruction kernel (algorithmic bytes for 8-bit 4:2:0: SURVEY 8d, DESIGN "kernels") ----
        px = images * file_mp * 1e6
        coded_px = images * (48 * TILE * TILE if wl == "c2" else 1920 * 1088)
        alg = {"k1_transform": rec_bytes_per_px * coded_px + 3.0 * coded_px, "k2_intra": 4.5 * coded_px, "k3_deblock": 2 * 3.0 * coded_px,
               "k4_sao": 1.5 * coded_px + 1.5 * px, "k5_csc": 4.5 * px}
        kernels = {k: m["stage_recon"][k] for k in alg}
        dom = max(kernels, key=kernels.get)
        achieved = alg[dom] / (kernels[dom] * 1e-3) / 1e9 if kernels[dom] > 0 else 0.0
        all_traffic = {}
        for fn in ("r02_traffic.json", "r01_traffic.json"):     # DRAM bytes per launch from the committed ncu captures
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", fn)))
            except (OSError, ValueError):
                continue
            for kname, entries in tj.items():
                for t in (entries if isinstance(entries, list) else [entries]):
                    if isinstance(t, dict) and t.get("workload", "c2") == wl and kname not in all_traffic and t.get("images_per_step"):
                        # a capture at another batch size is scaled by the number of files: the streaming kernels' traffic is
                        # proportional to the pictures of the step (said in the source string)
                        scale = images / float(t["images_per_step"])
                        if scale != 1.0 and fn != "r02_traffic.json":
                            continue
                        all_traffic[kname] = {"dram_bytes": int((t["dram_bytes_read"] + t["dram_bytes_write"]) * scale),
                                              "source": t["source"] + ("" if scale == 1.0 else "; captured at %d files per step, scaled x %.3g to %d" % (t["images_per_step"], scale, images))}
        k0_ms = m["stage"].get("k0_parse", 0.0)
        line.update({
            "value": world * mp_per_step / (m["dev_ms"] * 1e-3), "ms_per_step": m["dev_ms"], "scaling": "weak",
            "value_what": "per step: H2D of the step's inputs + K0 (device CABAC parse) + K1..K5, CUDA events on the streams they run on",
            "value_reconstruction_only": world * mp_per_step / (m["recon_ms"] * 1e-3), "ms_per_step_reconstruction_only": m["recon_ms"],
            "config": {"workload": WORKLOADS[wl].replace("CTB64 WPP", "CTB64 no-WPP (NOT the BASELINE configuration)") if args.no_wpp else WORKLOADS[wl],
                       "images_per_step_per_gpu": images, "distinct_files": len(distinct), "cpu_binding": numa,
                       "coded_pictures_per_step_per_gpu": images * (48 if wl == "c2" else 1),
                       "l2": "working set per step (planes + residuals + RGB, ~%d MB) exceeds the 126 MB L2; no explicit flush" % int(
                           images * file_mp * (1.5 + 1.5 + 3.0 + 3.0)),
                       "host_parse_threads": threads, "parity_vs_oracle": m["parity"]},
            "e2e": {"value": world * mp_per_step / m["e2e_dt"], "unit": UNIT, "h2d_bytes_per_step": int(st["bytes_h2d"] / max(1, st["batches"])),
                    "d2h_bytes_per_step": int(st["bytes_d2h"] / max(1, st["batches"])), "ms_per_step": m["e2e_dt"] * 1e3,
                    "host_parse_ms_per_step": st["seconds_parse"] / st["batches"] * 1e3,
                    "gpu_phase_ms_per_step": st["seconds_gpu_phase"] / st["batches"] * 1e3, "first_batch_ms": m["first_batch_s"] * 1e3,
                    "steps": m["e2e_steps"], "batches_in_flight": st.get("depth"),
                    "excluded": "steady-state period of the engine's second stream call (the first, untimed one pins the output buffers, fills the pools and settles the pipeline depth): deliveries of the first 5 batches (pipeline fill: first_batch_ms) and of the last 5 (drain) are outside the timed window",
                    "value_first_to_last_delivery": world * mp_per_step / m["e2e_first_to_last"],
                    "api": "hc_heic_decode_stream: three batches in flight on the GPU (K0 on a low-priority stream, K1..K5 + copies on "
                           "high-priority ones), header parse (+ host share of the slice data) two batches ahead; pinned host output"},
            "gpu_launches": m["launches"], "clocks": m["clocks"],
            "stage_ms_per_step": {k: round(v, 4) for k, v in m["stage"].items()},
            "record_bytes_per_px": rec_bytes_per_px, "uploaded_bytes_per_px": m["upload_bytes"] / px,
            "parser": "K0 on the device" if args.parser == "device" else "host CABAC parser",
            "roofline": {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": all_traffic.get(dom, {}).get("dram_bytes"), "traffic_unit": "bytes per launch (dram read + write, ncu)",
                         "traffic_source": all_traffic.get(dom, {}).get("source"),
                         "algorithmic_bytes_per_launch": alg[dom], "peak_source": peak_src,
                         "all_kernels": {k: {"ms": round(kernels[k], 4),
                                             "algorithmic_GBps": round(alg[k] / (kernels[k] * 1e-3) / 1e9, 1) if kernels[k] > 0 else None,
                                             "frac": round(alg[k] / (kernels[k] * 1e-3) / 1e9 / peak, 4) if kernels[k] > 0 else None,
                                             "dram_traffic_bytes": all_traffic.get(k, {}).get("dram_bytes")} for k in alg},
                         "k0_parse": {"ms": round(k0_ms, 4), "note": "device CABAC parse: serial per substream, bound by single-thread instruction "
                                      "latency / issue, not by HBM (DESIGN.md); inside `value` and e2e"} if k0_ms > 0 else None,
                         "note": "k2_intra is a dependency-latency-bound CTB wavefront, not a streaming kernel (DESIGN.md)"},
        })
    else:
        c5 = measure_c5(hb, eng, c5_file, args.steps, args.warmup, threads, rank, world, dist, barrier, max_over_ranks,
                        dump_dir=args.dump_outputs)
        rep = c5_report(c5, world)
        line.update({"value": rep["value"], "ms_per_step": rep["ms_per_step"], "scaling": "strong", "value_what": rep["value_what"],
                     "config": {"workload": WORKLOADS["c5"], "tiles": 391, "parity_vs_single_gpu": c5.get("bit_exact_vs_single_gpu")},
                     "e2e": {"value": file_mp / (c5["parse_s"] + c5["first_pass_ms"] * 1e-3 + c5["d2h_s"]), "unit": UNIT,
                             "h2d_bytes_per_step": len(c5_file), "d2h_bytes_per_step": C5_W * C5_H * 3,
                             "what": "one shot: band job creation (container + headers) + upload + K0..K5 with peer writes + D2H of the whole image "
                                     "from rank 0 (pageable destination)"},
                     "gpu_launches": 0, "c5": rep})

    # ---- side measurements of the default run: C4 (short) and C5 on the same box ----
    if extras:
        try:
            n4 = 384      # 1080p pictures are 17 chains each: 96 files fill a third of K0's chain slots (value 1.5 GP/s), 384 fill them (3.2)
            files4 = [c4_files[(i + rank) % len(c4_files)] for i in range(n4)]
            m4 = measure_list(hb, eng, files4, args.steps, args.warmup, threads, n4, barrier, max_over_ranks, local_rank, sample_clocks=False)
            mp4 = n4 * C4_W * C4_H / 1e6
            line["c4"] = {"workload": WORKLOADS["c4"], "images_per_step_per_gpu": n4, "value": world * mp4 / (m4["dev_ms"] * 1e-3),
                          "value_reconstruction_only": world * mp4 / (m4["recon_ms"] * 1e-3), "e2e_value": world * mp4 / m4["e2e_dt"], "unit": UNIT,
                          "stage_ms_per_step": {k: round(v, 4) for k, v in m4["stage"].items()}, "parity_vs_oracle": m4["parity"]}
        except Exception as e:      # a side measurement never takes the main line down
            line["c4"] = {"error": str(e)}
        try:
            line["c5"] = c5_report(measure_c5(hb, eng, c5_file, args.steps, args.warmup, threads, rank, world, dist, barrier, max_over_ranks), world)
        except Exception as e:
            line["c5"] = {"error": str(e)}

    # ---- CPU baseline on the box's cores (rank 0, N = 1 only) ----
    cpu, plugin = None, None
    if rank == 0 and world == 1 and not args.skip_baselines and wl == "c2":
        # the plugin arm runs right behind the GPU measurements (after the CPU arm the GPU has idled for ten seconds and single
        # one-tile batches do not bring its clocks back up: 55 instead of 110 MP/s measured), on an engine of its own
        eng.close()
        eng = None
        plugin = plugin_arm(c2_files, cores)
    if rank == 0 and world == 1 and not args.skip_baselines and wl != "c5":
        r = reference_arm(c2_files if wl == "c2" else c4_files, 2, 1, cores, file_mp)
        cpu = {"value": r["value"] if r else None, "unit": UNIT, "cores": cores, "kind": "reference",
               "sample": r["sample"] if r else "oracle/_ref missing on this box"}
    line["cpu_baseline"] = cpu
    line["plugin_dropin"] = plugin

    if rank == 0:
        print(json.dumps(line))
    if eng is not None:
        eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
