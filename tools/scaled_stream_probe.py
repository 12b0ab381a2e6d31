"""Full-size against scaled delivery (engine option "scale_max_side") on the C2 workload of bench.py: 8 distinct 4032 x 3024
grids of 512 x 512 tiles, RGB24, batches of 64 files, through hc_heic_decode_stream. The settings S = 0 (full size), 1024 and
512 alternate in one process, several rounds each, after a warm-up call of each. One JSON line per setting:

  e2e_gps              steady-state end-to-end GP/s of the stream in SOURCE pixels (bench.py's e2e window; max over ranks of the
                       period), so that the settings compare on the same work
  bytes_d2h_per_src_px hc_stream_stats.bytes_d2h / source pixels (3.0 at full size; 512 x 384 x 3 / 12.2 MP = 0.048 at S = 512)
  k5_ms                K5 device time of one batch (stage_ms[5] of a HeicJob of one batch)
  readback_ms          host clock around reading every image of that job into pinned buffers (hc_host_alloc), after run + sync

plus the device name and power limit read in the same run.
    python tools/scaled_stream_probe.py [--rounds 3] [--steps 10]
    torchrun --nproc-per-node 8 tools/scaled_stream_probe.py"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "heif-decoder-lib_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import bench  # noqa: E402

SETTINGS = (0, 1024, 512)   # scale_max_side
OUT_RGB = 0


def device_info(index):
    out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True).stdout.strip()
    name, _, limit = out.partition(",")
    return name.strip(), float(limit) if limit.strip() else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10, help="batches in the timed window of every stream call")
    ap.add_argument("--images", type=int, default=64, help="files per batch")
    args = ap.parse_args()

    import numpy as np
    import torch
    import heif_b200 as hb
    local_rank, world = int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("scaled_stream_probe.py needs a CUDA device")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist:
            dist.barrier()

    def max_over_ranks(v):
        if not dist:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    cache = os.path.join(tempfile.gettempdir(), "heif_b200_bench_content_%d" % os.getuid())   # shared with bench.py
    if rank == 0:
        bench.make_content(8, cache)
    barrier()
    distinct = bench.make_content(8, cache)
    files = [distinct[i % len(distinct)] for i in range(args.images)]
    threads = max(1, (os.cpu_count() or 1) // world)
    mp_per_batch = args.images * bench.GRID_W * bench.GRID_H / 1e6
    eng = hb.Engine(local_rank)
    skip = bench.STREAM_DEPTH - 1

    def stream(S):
        marks = []

        def on_image(index, desc, rows):
            if index % args.images == args.images - 1:
                marks.append(time.perf_counter())
        barrier()
        eng.set_option("scale_max_side", S)
        n = args.images * (2 * skip + 1 + args.steps)
        st = hb.decode_stream(eng, files * (2 * skip + 1 + args.steps), on_image, threads=threads, files_per_batch=args.images, out_format=OUT_RGB)
        barrier()
        dt = max_over_ranks((marks[-1 - skip] - marks[skip]) / args.steps)
        return world * mp_per_batch / dt / 1e3, st["bytes_d2h"] / (n * bench.GRID_W * bench.GRID_H)

    def one_batch(S, reps=5):
        eng.set_option("scale_max_side", S)
        job = hb.HeicJob(eng, files, threads=threads, out_format=OUT_RGB)
        job.upload()
        job.run()
        job.sync()
        conv = []
        for _ in range(reps):
            job.run()
            conv.append(job.stage_ms()["k5_csc"])
        eng.set_option("scale_max_side", 0)
        L = eng._L
        sizes = [(d.width * d.bytes_per_pixel * d.height, d.width * d.bytes_per_pixel) for d in job.descs]
        bufs = [L.hc_host_alloc(n) for n, _ in sizes]
        reads = []
        for _ in range(reps):
            job.run()
            job.sync()
            t0 = time.perf_counter()
            for i, (n, row) in enumerate(sizes):
                hb.api.check(L, L.hc_heic_job_read_rgb(job._h, i, bufs[i], row), "read")
            reads.append((time.perf_counter() - t0) * 1e3)
        for b in bufs:
            L.hc_host_free(b)
        job.close()
        return float(np.median(conv)), float(np.median(reads))

    res = {S: {"e2e": [], "d2h_px": None} for S in SETTINGS}
    for S in SETTINGS:     # warm-up: pinned output buffers, device pools, the stream depth the engine settles on
        eng.set_option("scale_max_side", S)
        hb.decode_stream(eng, files * (bench.STREAM_DEPTH + 4), None, threads=threads, files_per_batch=args.images, out_format=OUT_RGB)
    for r in range(args.rounds):
        for S in (SETTINGS if r % 2 == 0 else SETTINGS[::-1]):
            gps, d2h_px = stream(S)
            res[S]["e2e"].append(gps)
            res[S]["d2h_px"] = d2h_px
    name, limit = device_info(local_rank)
    for S in SETTINGS:
        k5_ms, read_ms = one_batch(S)
        k5_ms, read_ms = max_over_ranks(k5_ms), max_over_ranks(read_ms)
        if rank == 0:
            e = res[S]["e2e"]
            print(json.dumps({"scale_max_side": S, "n_gpus": world, "e2e_gps": float(np.median(e)), "e2e_gps_rounds": [round(v, 3) for v in e],
                              "bytes_d2h_per_src_px": res[S]["d2h_px"], "files_per_batch": args.images,
                              "k5_ms_per_batch": k5_ms, "readback_ms_per_batch": read_ms,
                              "device": name, "power_limit_w": limit}), flush=True)
    eng.close()
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
