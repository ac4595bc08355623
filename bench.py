#!/usr/bin/env python
"""Contract benchmark: instance-masks/sec of the unmold hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          (N>1: launched under torchrun)
    python bench.py --impl reference ...                   (the reference's CPU algorithm)
    python bench.py ... --dump-outputs DIR                 (also save the last step's outputs)

A step = one pass of the hot path (prologue + class-tile gather, one launch -> fused mask expand)
over one batch of synthetic detections: BASELINE.json configs[1], 32 distinct images of
1024x1024 with 100 instances each, per GPU (weak scaling: every rank processes its own batch;
the path has no exchange step, the final gather to rank 0 is timed separately as `gather`).
`value` is device-timed with inputs resident in HBM; `e2e` goes through the public
NumPy-facing path with pinned host buffers, H2D of the inputs and D2H of the masks inside the
timed region.  Extra blocks on the same JSON line: `roofline`, `cpu_baseline`, `parity`
(image 0 of the timed batch against the oracle), `latency` (the reference's own call pattern:
one image through `api_utils.unmold_detections`), `packed` (extension layout), `gather`
(N > 1) and `config4` (BASELINE.json configs[3], sharded over the N ranks).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "instance-masks/sec"
UNIT = "masks/s"
WORKLOAD = "BASELINE.json configs[1]: batch 32 images 1024x1024, 100 instances each, mask unmold"
BATCH, HW, N_INST, CLASSES = 32, (1024, 1024), 100, 81
SEED = 20260921
C4_BATCH, C4_HW, C4_INST = 128, (2160, 3840), 50     # BASELINE.json configs[3]


def make_bench_images(rank, count=BATCH):
    """The batch rank `rank` times: `count` DISTINCT seeded images (tests import this to check
    image 0 exhaustively against the oracle)."""
    from matterport_maskrcnn_with_tensorflow_serving_b200 import synth

    return synth.make_batch(SEED + rank, count, HW, N_INST, num_classes=CLASSES)


# ----------------------------------------------------------------------------- CPU legs
def _cpu_worker(args):
    """Unmold one synthetic image with the oracle (the reference's NumPy/SciPy algorithm).
    Runs in a spawned process; returns (n_masks, seconds of the unmold call alone)."""
    seed, hw, n_inst, classes = args
    import numpy as np

    import oracle
    from matterport_maskrcnn_with_tensorflow_serving_b200 import synth

    im = synth.make_batch(seed, 1, hw, n_inst, num_classes=classes)[0]
    det = im.detections.astype(np.float64)      # serve.py:131-136 hands float64 arrays over
    msk = im.mrcnn_mask.astype(np.float64)
    t0 = time.perf_counter()
    out = oracle.unmold_detections(det, msk, im.original_image_shape, im.image_shape, im.window)
    dt = time.perf_counter() - t0
    return int(out[0].shape[0]), dt


class CpuPool:
    """Process pool over host cores running the oracle on whole images."""

    def __init__(self, procs):
        import multiprocessing as mp

        self.procs = int(procs)
        self.ctx = mp.get_context("spawn")
        self.pool = self.ctx.Pool(self.procs)
        # spin the workers up (imports) outside any timed region
        self.pool.map(_cpu_worker, [(1, (64, 64), 2, 3)] * self.procs)

    def run(self, n_images, seed0):
        jobs = [(seed0 + i, HW, N_INST, CLASSES) for i in range(n_images)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, jobs, chunksize=1)
        wall = time.perf_counter() - t0
        masks = sum(r[0] for r in res)
        return masks, wall, [r[1] for r in res]

    def close(self):
        self.pool.close()
        self.pool.join()


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def default_procs(cores):
    """Worker processes for the CPU legs.  The reference's path is memory-bound (one fresh
    H x W canvas per instance, then np.stack(axis=-1)).  Measured on this pool's 128-thread
    Xeon 8562Y+ host (masks/s at 16/32/64/128 processes: 1067 / 851 / 604 / 396), more
    processes only make it slower, so the CPU legs use 16."""
    return max(1, min(cores, 16))


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_baseline_block(procs=None, images=None):
    """Bounded sample of the workload on the host: `images` images (100 masks each) over
    `procs` processes, plus one image alone for the single-core figure."""
    cores = host_cores()
    procs = procs or default_procs(cores)
    images = images or procs
    pool = CpuPool(procs)
    try:
        m1, w1, _ = pool.run(1, SEED + 1000)
        masks, wall, per = pool.run(images, SEED + 2000)
    finally:
        pool.close()
    return {
        "value": masks / wall, "unit": UNIT, "cores": procs, "kind": "port",
        "sample": f"{images} of the workload's 1024x1024x100-instance images "
                  f"({masks} masks) over {procs} processes, oracle NumPy/SciPy float64",
        "single_core_value": m1 / w1, "single_image_ms": 1e3 * w1,
        "host_cores": cores, "cpu_model": cpu_model(),
    }


_RESULT_FD = None


def emit_line(line):
    """The one JSON line, on the process's original stdout (see main())."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (oracle port; the reference's
    code for this path is not vendored, SURVEY.md 8c) on all the host threads it can use."""
    if rank != 0:
        return 0
    cores = host_cores()
    procs = args.cpu_procs or default_procs(cores)
    total_steps = args.steps + args.warmup
    images = max(4, min(procs, int(600 / max(total_steps, 1))))
    pool = CpuPool(procs)
    try:
        for w in range(args.warmup):
            pool.run(images, SEED + 10 * w)
        t0 = time.perf_counter()
        masks = 0
        for s in range(args.steps):
            m, _, _ = pool.run(images, SEED + 100 + s)
            masks += m
        wall = time.perf_counter() - t0
    finally:
        pool.close()
    value = masks / wall
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "images_per_step": images, "instances_per_image": N_INST,
                   "num_classes": CLASSES, "layout": "[H,W,N] bool"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port",
                         "sample": f"each step = {images} images x {N_INST} instances over "
                                   f"{procs} processes (host has {cores} logical cores, "
                                   f"{cpu_model()})"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)
    return 0


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.idx), "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "samples": len(sm),
                "reasons": sorted(reasons),
                "window": "identical untimed load (--load-ms) + the timed region, 50 ms period"}


# ----------------------------------------------------------------------------- GPU arm
def load_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu summary."""
    path = os.path.join(ROOT, "profiles", "mask_expand_ncu_summary.json")
    try:
        with open(path) as f:
            j = json.load(f)
        return j.get("dram_bytes_per_launch"), j.get("source")
    except (OSError, ValueError):
        return None, None


class Ctx:
    """What the sections of the GPU arm share."""

    def __init__(self, args, rank, world, local_rank):
        import torch
        import torch.distributed as dist

        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.torch, self.dist = torch, dist
        self.dev = torch.device("cuda", local_rank)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def gather_floats(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(x)]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]


def upload_batch(ctx, ims):
    """Pinned host + device copies of a list of SynthImage."""
    import numpy as np
    torch = ctx.torch
    n = len(ims)
    R = ims[0].detections.shape[0]
    C = ims[0].mrcnn_mask.shape[-1]
    h_det = torch.from_numpy(np.stack([im.detections for im in ims])).pin_memory()
    h_msk = torch.empty((n, R, 28, 28, C), dtype=torch.float32).pin_memory()
    for i, im in enumerate(ims):
        h_msk[i].copy_(torch.from_numpy(im.mrcnn_mask))
    return h_det, h_msk, h_det.to(ctx.dev), h_msk.to(ctx.dev)


def timed_device(ctx, fn, reps):
    """Median and min of `reps` device-timed runs of fn() (CUDA events on the current stream,
    max over ranks per run, barrier before each)."""
    torch = ctx.torch
    ms = []
    for _ in range(reps):
        ctx.barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(ctx.max_over_ranks(e0.elapsed_time(e1)))
    ms.sort()
    return ms[len(ms) // 2], ms[0]


def _bytesum(torch, t, chunk=1 << 28):
    """Sum of a uint8 tensor's bytes (checksum of a gathered buffer), 256 MB at a time: the
    widening reduction materialises an int64 copy of its input."""
    return sum(int(c.sum(dtype=torch.int64).item()) for c in t.split(chunk)) if t.numel() else 0


DUMP_PIXELS_PER_IMAGE = 2048     # canvas positions per image whose mask values --dump-outputs keeps
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, eng, n_images):
    """--dump-outputs: what the last timed step returned, as DIR/<name>.npy, so that two builds
    can be compared output for output on the same seeded inputs.  Per kept instance, in image
    order: boxes, class ids, scores and the mask's pixel count, all complete.  The masks
    themselves (3.4 GB per step) are sampled: the values of every kept mask at
    DUMP_PIXELS_PER_IMAGE positions per image, drawn with a fixed seed from the image's H x W."""
    import numpy as np
    import torch

    counts = eng.d_counts[:n_images].cpu().numpy()
    boxes = eng.d_boxes[:n_images].cpu().numpy()
    class_ids = eng.d_class_ids[:n_images].cpu().numpy()
    scores = eng.d_scores[:n_images].cpu().numpy()
    kept = lambda a: np.concatenate([a[b, :k] for b, k in enumerate(counts)])  # noqa: E731
    rng = np.random.default_rng(SEED)
    areas, samples = [], []
    for b, k in enumerate(counts):
        m = eng.canvas_view(b, int(k))                     # uint8 [H, W, k] on the device
        h, w = m.shape[:2]
        areas.append(m.sum(dim=(0, 1), dtype=torch.int64).cpu().numpy())
        pix = torch.from_numpy(rng.integers(0, h * w, DUMP_PIXELS_PER_IMAGE)).to(m.device)
        samples.append(m.reshape(h * w, int(k))[pix].cpu().numpy().ravel())
    out = {
        "counts": counts.astype(np.float64),
        "boxes": kept(boxes).astype(np.float64),
        "class_ids": kept(class_ids).astype(np.float64),
        "scores": kept(scores).astype(np.float32),
        "mask_pixel_counts": np.concatenate(areas).astype(np.float64),
        "mask_samples": np.concatenate(samples).astype(np.float32),
    }
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def gather_section(ctx, eng, d_det, d_msk, n_images, masks_total, layout_note, chunks=4, reps=3):
    """One step + the gather of every rank's output to rank 0, both layouts, both transports.
    Returns the `gather` dict.  Rank 0's NVLink ingress bounds all of them: (world-1)/world of
    the bytes enter one GPU."""
    import numpy as np

    from matterport_maskrcnn_with_tensorflow_serving_b200 import sharding
    torch, dist, world, rank = ctx.torch, ctx.dist, ctx.world, ctx.rank
    stream = torch.cuda.current_stream()
    res = {"unit": UNIT, "chunks_per_rank": chunks, "reps": reps, "note": layout_note}

    # per-layout geometry of this rank's output (identical on every rank: same image shapes)
    byte_off = eng._offsets
    byte_total = int(byte_off[n_images])
    pk_off, pk_total = eng.packed_layout()
    img_chunks = sharding.chunk_bounds(n_images, chunks)
    k = len(img_chunks)

    # reference content of this rank (local run) -> checksums rank 0 verifies the gathers with
    eng.enqueue(d_det, d_msk)
    d_packed, _ = eng.enqueue_expand_packed()
    sum_bytes = _bytesum(torch, eng.d_canvas[:byte_total])
    sum_packed = _bytesum(torch, d_packed[:pk_total])
    sums = [ctx.gather_floats(sum_bytes), ctx.gather_floats(sum_packed)]

    def verify(slot_fn, which, total):
        if rank != 0:
            return True
        ok = True
        for r in range(world):
            got = _bytesum(torch, slot_fn(r)[:total])
            ok = ok and (got == int(sums[which][r]))
        return ok

    for layout, off, total, which in (("bytes", byte_off, byte_total, 0), ("packed", pk_off, pk_total, 1)):
        sizes = [total] * world
        ranges = [(int(off[a]), int(off[b])) for a, b in img_chunks]
        into_rank0 = total * (world - 1)

        # ---- NCCL send/recv, one chunk of images at a time, overlapped with the next chunk
        g = sharding.RootGather(sizes, ctx.dev)
        local = eng.d_canvas if layout == "bytes" else eng.d_packed

        def run_nccl():
            eng.enqueue(d_det, d_msk, stream, expand=False)
            g.begin(k, [ranges] * world)
            for (a, b), (lo, hi) in zip(img_chunks, ranges):
                ptr = g.slot(0).data_ptr() if rank == 0 else None
                if layout == "bytes":
                    eng.enqueue_expand(stream, canvas_ptr=ptr, images=(a, b))
                else:
                    eng.enqueue_expand_packed(stream, packed_ptr=ptr, images=(a, b))
                g.post(local, lo, hi)
            g.wait()

        run_nccl()                                   # warm-up (NCCL channels, buffers)
        med, best = timed_device(ctx, run_nccl, reps)
        ok = verify(g.slot, which, total)

        def run_transport_only():                    # the same bytes, no kernels: the wire alone
            g.begin(1, [[(0, total)]] * world)
            g.post(local, 0, total)
            g.wait()

        t_med, _ = timed_device(ctx, run_transport_only, reps)
        res[f"{layout}_transport_only"] = {
            "ms": t_med, "ingress_gbs": into_rank0 / (t_med * 1e-3) / 1e9,
            "what": "NCCL send/recv of the finished buffers into rank 0, no compute: the wire time "
                    "the gather variants are compared with"}
        res[f"{layout}_nccl"] = {
            "value": masks_total / (med * 1e-3), "ms": med, "ms_best": best,
            "bytes_into_rank0": into_rank0, "ingress_gbs": into_rank0 / (med * 1e-3) / 1e9,
            "verified": bool(ok)}
        del g
        torch.cuda.empty_cache()

        # ---- fused: the expand kernels store straight into rank 0's buffer over NVLink
        try:
            pg = sharding.PeerGather(sizes, ctx.dev)
        except Exception as e:      # noqa: BLE001  (report, keep the NCCL numbers)
            res[f"{layout}_p2p_fused"] = {"unavailable": f"{type(e).__name__}: {e}"}
            continue

        def run_p2p():
            pg.next_epoch()
            eng.enqueue(d_det, d_msk, stream, expand=False)
            if layout == "bytes":
                eng.enqueue_expand(stream, canvas_ptr=pg.out_ptr())
            else:
                eng.enqueue_expand_packed(stream, packed_ptr=pg.out_ptr())
            pg.signal(stream)
            pg.wait(stream)

        run_p2p()
        med, best = timed_device(ctx, run_p2p, reps)
        ok = verify(pg.slot, which, total)
        res[f"{layout}_p2p_fused"] = {
            "value": masks_total / (med * 1e-3), "ms": med, "ms_best": best,
            "bytes_into_rank0": into_rank0, "ingress_gbs": into_rank0 / (med * 1e-3) / 1e9,
            "verified": bool(ok)}
        pg.close()
        del pg
        torch.cuda.empty_cache()
    res["limiter"] = ("rank 0's NVLink ingress: (world-1)/world of all output bytes enter one GPU; "
                      "see ingress_gbs of each variant against ~900 GB/s per direction")
    return res


def config4_section(ctx, reps=3):
    """BASELINE.json configs[3]: 128 images of 2160x3840 with 50 instances, sharded over the
    ranks (contiguous blocks), kernel-only step time and -- for N > 1 -- the gather."""
    import numpy as np

    from matterport_maskrcnn_with_tensorflow_serving_b200 import sharding, synth
    from matterport_maskrcnn_with_tensorflow_serving_b200.engine import UnmoldEngine, make_geom
    torch, world, rank = ctx.torch, ctx.world, ctx.rank
    lo, hi = sharding.equal_partition(C4_BATCH, world)[rank]
    n = hi - lo
    rng_seed = SEED + 4000 + rank
    ims = synth.make_batch(rng_seed, n, C4_HW, C4_INST, num_classes=CLASSES, max_instances=C4_INST)
    h_det, h_msk, d_det, d_msk = upload_batch(ctx, ims)
    del h_det, h_msk
    eng = UnmoldEngine(n, C4_INST, (28, 28), CLASSES)
    eng.plan([make_geom(im.original_image_shape, im.image_shape, im.window) for im in ims])
    stream = torch.cuda.current_stream()
    for _ in range(3):
        eng.enqueue(d_det, d_msk, stream)
    torch.cuda.synchronize()
    counts = eng.d_counts[:n].cpu().numpy()
    masks_rank = int(counts.sum())
    masks_total = ctx.sum_over_ranks(masks_rank)
    algo = eng.canvas_bytes(counts) + masks_rank * (28 * 28 * 4 + 24)
    med, best = timed_device(ctx, lambda: eng.enqueue(d_det, d_msk, stream), max(reps, 5))
    out = {
        "workload": "BASELINE.json configs[3]: 128 images 2160x3840, 50 instances each, "
                    f"{n} images per GPU over {world} GPU(s)",
        "value": masks_total / (med * 1e-3), "unit": UNIT, "ms_per_step": med, "ms_best": best,
        "images_per_gpu": n, "algorithmic_gbs_per_gpu": algo / (med * 1e-3) / 1e9,
    }
    if world > 1:
        out["gather"] = gather_section(
            ctx, eng, d_det, d_msk, n, masks_total,
            "one step of the shard + gather of all 128 canvases to rank 0", reps=reps)
    eng.release()
    del eng, d_det, d_msk
    torch.cuda.empty_cache()
    return out


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist

    from matterport_maskrcnn_with_tensorflow_serving_b200 import sharding
    from matterport_maskrcnn_with_tensorflow_serving_b200.engine import UnmoldEngine, make_geom

    cpu_block = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_block = cpu_baseline_block(args.cpu_procs or None)   # before CUDA is initialised here

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    ctx = Ctx(args, rank, world, local_rank)
    dev = ctx.dev
    # torchrun does not bind ranks to their GPU's NUMA node; pinned buffers allocated after this
    # are node-local (matters for the e2e figure at N = 8: GPUs 4-7 hang off the second socket)
    numa = sharding.bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"bound": False}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- synthetic inputs (seeded, per rank, 32 DISTINCT images), in HBM and in pinned memory
    ims = make_bench_images(rank, BATCH)
    h_det, h_msk, d_det, d_msk = upload_batch(ctx, ims)
    geoms = [make_geom(im.original_image_shape, im.image_shape, im.window) for im in ims]

    eng = UnmoldEngine(BATCH, N_INST, (28, 28), CLASSES, chunk_bytes=args.chunk_bytes,
                       ctas_per_sm=args.ctas_per_sm)
    eng.plan(geoms)
    stream = torch.cuda.current_stream()
    barrier = ctx.barrier

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        eng.enqueue(d_det, d_msk, stream)
    torch.cuda.synchronize()
    counts = eng.d_counts[:BATCH].cpu().numpy()
    status = eng.d_status[:BATCH].cpu().numpy()
    assert int(status.max()) == 0, "synthetic inputs flagged invalid"
    masks_per_step = int(counts.sum())
    out_bytes = eng.canvas_bytes(counts)
    algo_bytes = out_bytes + masks_per_step * (28 * 28 * 4 + 24)   # SURVEY.md 8d per-instance figure

    # ---- timed region: exactly K steps, device-timed, expand kernel timed per launch
    sampler = ClockSampler(local_rank)
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(args.steps)]
    import ctypes as C

    from matterport_maskrcnn_with_tensorflow_serving_b200 import _native as N
    lib = eng.lib
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    st = N.stream_ptr(stream)
    # clock sampling needs load for longer than a few ms: run the same steps untimed for
    # --load-ms first (clocks settle, nvidia-smi gets samples), keep sampling through the
    # timed region
    sampler.start()
    t_load = time.perf_counter()
    while (time.perf_counter() - t_load) * 1e3 < args.load_ms:
        for _ in range(10):
            eng.enqueue(d_det, d_msk, stream)
        torch.cuda.synchronize()
    barrier()
    ev0.record(stream)
    for s in range(args.steps):
        N.check(lib.mrx_unmold_prepare(P(d_det), N.MRX_F32, P(d_msk), N.MRX_F32, BATCH, N_INST, 28,
                                       28, CLASSES, P(eng.d_geom), P(eng.d_boxes),
                                       P(eng.d_class_ids), P(eng.d_scores), P(eng.d_src_index),
                                       P(eng.d_counts), P(eng.d_status),
                                       P(eng.d_tiles), P(eng.d_sched), st), "prepare")
        kev[s][0].record(stream)
        N.check(lib.mrx_mask_expand(P(eng.d_tiles), P(eng.d_src_index), P(eng.d_boxes),
                                    P(eng.d_counts), P(eng.d_geom),
                                    P(eng.d_canvas_off), P(eng.d_canvas), BATCH, N_INST, 28, 28,
                                    eng.chunk_bytes, eng.ctas_per_sm, P(eng.d_sched), st),
                "expand")
        kev[s][1].record(stream)
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    elapsed_ms = ev0.elapsed_time(ev1)
    expand_ms = [a.elapsed_time(b) for a, b in kev]
    max_ms = ctx.max_over_ranks(elapsed_ms)
    barrier()
    total_masks = ctx.sum_over_ranks(masks_per_step)
    value = total_masks * args.steps / (max_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, BATCH)     # before later sections reuse the buffers

    # ---- parity of the timed step's output: image 0 of this very batch against the oracle
    # (outside timing; rank 0; the same check tests/test_gpu_unmold.py runs exhaustively)
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        import hashlib

        import oracle
        k0 = int(counts[0])
        m0 = eng.canvas_view(0, k0).cpu().numpy()
        digest = hashlib.sha256(m0.tobytes()).hexdigest()[:16]
        im = ims[0]
        t0 = time.perf_counter()
        rb, rc, rs, rm, rz = oracle.unmold_detections(
            im.detections.astype(np.float64), im.mrcnn_mask.astype(np.float64),
            im.original_image_shape, im.image_shape, im.window, return_resized=True)
        oracle_ms = 1e3 * (time.perf_counter() - t0)
        boxes0 = eng.d_boxes[0, :k0].cpu().numpy()
        diff = m0.view(np.bool_) != rm
        flips_out = flips_in = band = 0
        outside = diff.copy()
        for i, (y1, x1, y2, x2) in enumerate(rb):
            near = np.abs(rz[i] - 0.5) <= 1e-6
            band += int(near.sum())
            d = diff[y1:y2, x1:x2, i]
            flips_out += int((d & ~near).sum())
            flips_in += int((d & near).sum())
            outside[y1:y2, x1:x2, i] = False
        flips_out += int(outside.sum())
        parity = {"image": 0, "instances": k0, "boxes_bit_exact": bool(np.array_equal(boxes0, rb)),
                  "mask_pixels": int(m0.size), "flips_outside_1e-6_band": flips_out,
                  "flips_inside_band": flips_in, "band_pixels": band, "canvas_sha256_16": digest,
                  "oracle_ms": oracle_ms, "ok": bool(flips_out == 0 and np.array_equal(boxes0, rb))}
        assert parity["ok"], parity
        del m0, rm, rz, diff, outside

    # ---- e2e: host buffers in, host masks out, every step (public API: StreamingUnmolder,
    # which overlaps the H2D of batch k+1 with the D2H of batch k's masks)
    from matterport_maskrcnn_with_tensorflow_serving_b200.engine import StreamingUnmolder

    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def run_e2e(sm, steps):
        sm.submit(h_det, h_msk)                 # warm-up batch (allocations, first-touch)
        sm.wait(0)
        barrier()
        t0 = time.perf_counter()
        last = None
        for _ in range(steps):
            kk = sm.submit(h_det, h_msk)
            if last is not None:
                sm.wait(last)                   # batch k-1 is consumed while batch k is in flight
            last = kk
        res = sm.wait(last)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        return sec, res

    sm = StreamingUnmolder(eng, geoms)
    e2e_s, (h_counts, h_boxes, h_out) = run_e2e(sm, e2e_steps)
    e2e_value = total_masks * e2e_steps / ctx.max_over_ranks(e2e_s)
    h2d, d2h = sm.h2d_bytes, sm.d2h_bytes
    pcie = {"h2d_gbs_per_rank": [round(v, 2) for v in ctx.gather_floats(h2d * e2e_steps / e2e_s / 1e9)],
            "d2h_gbs_per_rank": [round(v, 2) for v in ctx.gather_floats(d2h * e2e_steps / e2e_s / 1e9)]}
    # sanity: the host copy really holds this step's masks
    assert int(h_counts.sum()) == masks_per_step and int(h_out[: 1 << 20].max()) <= 1
    del sm, h_out
    torch.cuda.empty_cache()

    # ---- extension layout: bit-packed masks written directly by the expand kernel
    packed = None
    if not args.no_packed:
        pk_reps = max(5, min(args.steps, 20))
        pk_med, pk_best = timed_device(ctx, lambda: eng.enqueue_packed(d_det, d_msk, stream), pk_reps)
        # the expand kernel alone (prologue + class-tile gather already done)
        pk_k_med, pk_k_best = timed_device(ctx, lambda: eng.enqueue_expand_packed(stream), pk_reps)
        pk_off, pk_total = eng.packed_layout()
        packed = {
            "layout": "EXTENSION, not the reference's: uint8 [N,H,ceil(W/8)] per image "
                      "(np.packbits of each mask row); bit-exact with packbits of the byte canvas "
                      "(tests/test_gpu_pack.py)",
            "value": total_masks / (pk_med * 1e-3), "unit": UNIT, "ms_per_step": pk_med,
            "kernel": "mask_expand_bits_kernel", "kernel_ms": pk_k_med, "kernel_ms_best": pk_k_best,
            "output_bytes_per_step": int(pk_total),
        }
        for name, kw in (("e2e", {}), ("e2e_zero_copy_masks", {"mask_upload": "zero_copy"})):
            smp = StreamingUnmolder(eng, geoms, packed=True, **kw)
            sec, (pc, pb, po) = run_e2e(smp, e2e_steps)
            assert int(pc.sum()) == masks_per_step
            packed[name] = {
                "value": total_masks * e2e_steps / ctx.max_over_ranks(sec), "unit": UNIT,
                "ms_per_step": 1e3 * sec / e2e_steps,
                "h2d_bytes_per_step": int(smp.h2d_bytes), "d2h_bytes_per_step": int(smp.d2h_bytes),
                "pcie_read_bytes_per_step": int(smp.pcie_read_bytes)}
            del smp, po
            torch.cuda.empty_cache()
        packed["e2e"]["path"] = ("StreamingUnmolder(packed=True): pinned inputs -> H2D -> prologue, "
                                 "class gather, packed expand -> D2H of the packed masks")
        packed["e2e_zero_copy_masks"]["path"] = (
            "same, but mrcnn_mask (99.7 % of the input bytes, 81 classes of which one per instance "
            "is used) is never copied: the class-gather kernel reads the wanted floats from the "
            "pinned host buffer over PCIe")

    # ---- latency of the reference's own call pattern: ONE image through the drop-in call
    latency = None
    if rank == 0 and not args.no_latency:
        from matterport_maskrcnn_with_tensorflow_serving_b200 import api_utils

        im = ims[0]
        det64 = im.detections.astype(np.float64)          # serve.py:131-136: float64 arrays
        msk64 = im.mrcnn_mask.astype(np.float64)
        call = lambda: api_utils.unmold_detections(      # noqa: E731
            det64, msk64, im.original_image_shape, im.image_shape, im.window)
        for _ in range(3):
            out = call()
        ts = []
        for _ in range(10):
            t0 = time.perf_counter()
            out = call()
            ts.append(1e3 * (time.perf_counter() - t0))
        ts.sort()
        latency = {"call": "api_utils.unmold_detections(one 1024x1024 image, 100 instances, "
                           "float64 inputs as serve.py:131-136 builds them) -> NumPy outputs",
                   "ms_median": ts[len(ts) // 2], "ms_min": ts[0], "ms_max": ts[-1], "calls": 10,
                   "input_bytes": int(det64.nbytes + msk64.nbytes),
                   "output_bytes": int(out[3].nbytes),
                   "oracle_ms_one_core": (parity or {}).get("oracle_ms") or
                                         (cpu_block or {}).get("single_image_ms")}
        if latency["oracle_ms_one_core"]:
            latency["speedup_vs_oracle"] = latency["oracle_ms_one_core"] / latency["ms_median"]
        del out, det64, msk64
        api_utils.release()

    # ---- gather-inclusive (N > 1) and BASELINE.json configs[3]
    gather = None
    if world > 1 and not args.no_gather:
        gather = gather_section(ctx, eng, d_det, d_msk, BATCH, total_masks,
                                "one step (32 images per rank) + gather of every rank's output "
                                "to rank 0")
    eng.release()
    del d_det, d_msk, h_det, h_msk
    torch.cuda.empty_cache()
    config4 = None
    if not args.no_config4:
        config4 = config4_section(ctx)

    if rank == 0:
        peak, peak_src = load_peak()
        traffic, traffic_src = load_traffic()
        k_ms = float(np.mean(expand_ms))
        achieved = algo_bytes / (k_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "images_per_gpu": BATCH, "instances_per_image": N_INST,
                       "distinct_images": BATCH,
                       "num_classes": CLASSES, "mask_tile": "28x28 f32", "layout": "[H,W,N] bool",
                       "sharding": f"images over {world} rank(s), no data-path collective",
                       "l2": "per-step working set (813 MB in + 3.36 GB out per GPU) exceeds the "
                             "126 MB L2; no explicit flush",
                       "tile_buffer_bytes": eng.chunk_bytes or "auto", "seed": SEED,
                       "numa": numa},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, **pcie,
                    "path": "engine.StreamingUnmolder: pinned host detections+mrcnn_mask -> H2D "
                            "(own stream, overlaps the previous batch's D2H) -> 2 kernels -> D2H "
                            "of counts, boxes and the [H,W,N] bool canvases; every batch's "
                            "masks are waited for on the host"},
            "gpu_launches": 2 * args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "kernel": "mask_expand_team_kernel",
                         "kernel_ms": k_ms, "kernel_ms_min": float(np.min(expand_ms)),
                         "algorithmic_bytes_per_launch": int(algo_bytes),
                         "peak_source": peak_src, "traffic_source": traffic_src},
            "cpu_baseline": cpu_block,
            "parity": parity,
            "latency": latency,
            "packed": packed,
        }
        if gather is not None:
            line["gather"] = gather
        if config4 is not None:
            line["config4"] = config4
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--load-ms", type=float, default=400.0,
                    help="untimed identical load before the timed region (clock sampling window)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--chunk-bytes", type=int, default=0)
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-packed", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--cpu-procs", type=int, default=0, help="worker processes of the CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write rank 0's outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the device path's outputs; the reference arm has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    # stdout carries ONE line, the JSON result: whatever libraries print there (NCCL's version
    # banner at N > 1) goes to stderr; emit_line() writes to the saved descriptor
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
