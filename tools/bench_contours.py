"""Contour polygons of display_instances (mrx_contours_count / _write) on the BASELINE.json
configs[1] synthetic batch (32 x 1024x1024 x 100 instances), device-timed with CUDA events on
the bit-packed masks the packed expand writes.  Not the contract bench; the numbers go into
profiles/README.md.  Prints one JSON line.

  python tools/bench_contours.py [--iters 20] [--cpu-images 1]

The synthetic tiles are uniform noise, so the masks are far more ragged than real ones (about
7.6 k segments and 38 polygons per instance): a stress case for the contour walk.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from matterport_maskrcnn_with_tensorflow_serving_b200 import _native as N, synth  # noqa: E402
from matterport_maskrcnn_with_tensorflow_serving_b200.engine import UnmoldEngine, make_geom  # noqa: E402


def _p(t):
    return C.c_void_p(t.data_ptr())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--cpu-images", type=int, default=1, help="images the oracle is timed on")
    args = ap.parse_args()
    B, R, hw = args.batch, 100, (1024, 1024)
    ims = synth.make_batch(11, B, hw, R)
    eng = UnmoldEngine(B, R, (28, 28), 81)
    eng.plan([make_geom(im.original_image_shape, im.image_shape, im.window) for im in ims],
             canvas=False)
    d_det = torch.from_numpy(np.stack([im.detections for im in ims]).astype(np.float32)).cuda()
    d_msk = torch.from_numpy(np.stack([im.mrcnn_mask for im in ims]).astype(np.float32)).cuda()
    d_packed, _ = eng.enqueue_packed(d_det, d_msk)
    lib, dev = eng.lib, eng.device
    max_h = max_w = 1024
    d_rows = torch.empty((B * R * (max_h + 1),), dtype=torch.int32, device=dev)
    d_off = torch.empty((B * R + 1,), dtype=torch.int64, device=dev)
    common = (_p(d_packed), _p(eng.d_packed_off), _p(eng.d_boxes), _p(eng.d_counts),
              _p(eng.d_geom), _p(d_rows), _p(d_off))
    st = N.stream_ptr(None)

    def count():
        N.check(lib.mrx_contours_count(*common, B, R, max_h, max_w, st), "mrx_contours_count")

    count()
    off = d_off.cpu().numpy()
    T = int(off[-1])
    d_scratch = torch.empty((2 * T,), dtype=torch.int32, device=dev)
    d_vert = torch.empty((T + T // 4, 2), dtype=torch.float32, device=dev)
    d_len = torch.empty((T // 4,), dtype=torch.int32, device=dev)
    d_ncont = torch.empty((B * R,), dtype=torch.int32, device=dev)

    def write():
        N.check(lib.mrx_contours_write(*common, _p(d_scratch), _p(d_vert), _p(d_len),
                                       _p(d_ncont), C.c_longlong(T), B, R, max_h, max_w, st),
                "mrx_contours_write")

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    count_ms = timed(count)
    write_ms = timed(write)

    # end to end as api_utils runs it: count, one host read, write (host clock, synchronised)
    from matterport_maskrcnn_with_tensorflow_serving_b200.engine import contours_device
    walls = []
    for _ in range(args.iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dc = contours_device(lib, dev, d_packed, eng.d_packed_off, eng.d_boxes, eng.d_counts,
                             eng.d_geom, B, R, max_h, max_w)
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
    n_contours = int(dc.inst_contours.sum().item())
    V = int(dc.contour_len.sum().item())
    out_bytes = V * 8 + n_contours * 4 + B * R * 4

    # the oracle on the same masks (unpacked from the device's packed planes), which must give
    # the same polygons
    from oracle import contours as oracle
    cpu = []
    wb = (hw[1] + 7) // 8
    host = d_packed.cpu().numpy()
    counts = eng.d_counts.cpu().numpy()
    polys = dc.to_host(counts)
    for b in range(args.cpu_images):
        k = int(counts[b])
        o = int(eng.packed_layout()[0][b])
        masks = np.unpackbits(host[o:o + k * hw[0] * wb].reshape(k, hw[0], wb), axis=-1,
                              count=hw[1]).astype(bool)
        t0 = time.perf_counter()
        ref = [oracle.mask_contours(masks[i]) for i in range(k)]
        cpu.append(time.perf_counter() - t0)
        for g, w in zip(polys[b], ref):
            assert len(g) == len(w) and all(np.array_equal(x, y) for x, y in zip(g, w)), \
                "device contours differ from the oracle"

    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        smi = "unknown"
    print(json.dumps({
        "workload": f"contours configs[1]: {B} x {hw[0]}x{hw[1]} x {R} (synthetic noise tiles)",
        "gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi,
        "count_ms": round(count_ms, 4), "write_ms": round(write_ms, 4),
        "count_plus_write_ms": round(count_ms + write_ms, 4),
        "end_to_end_ms_median": round(float(np.median(walls)), 4),
        "segments": T, "segments_per_s": T / ((count_ms + write_ms) * 1e-3),
        "contours": n_contours, "vertices": V, "output_MB": round(out_bytes / 1e6, 3),
        "oracle_cpu_s_per_image": round(float(np.mean(cpu)), 3) if cpu else None,
    }))


if __name__ == "__main__":
    main()
