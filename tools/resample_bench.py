"""Measure the volume resample (pm_resample_affine, SURVEY §8f row 5) on one GPU and print one JSON line.

Workloads (bench.py's 384 x 512 x 512 label volume): int32 labels with order 0 and a uint16 intensity volume with
order 1, each under the identity and under a near-rigid transform (12 degrees about x, scale 1.03, shift (3, -5, 4)
about the volume centre).  Kernel time: CUDA events around one call, 3 warm-up calls, mean of 10, a 160 MB L2 flush
before each.  Algorithmic bytes = source + destination; the reference bandwidth is a plain device-to-device tensor
copy measured in the same process.  The CPU baseline is one scipy.ndimage.affine_transform call per workload on the
same volume, with the near-rigid transform; its output is also compared with the GPU's.

    python tools/resample_bench.py [--no-cpu-baseline]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPE = (384, 512, 512)


def gpu_identity():
    """Name and power limit of GPU 0 (a read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return {"name": name, "power_limit": limit}
    except Exception as e:                        # the measurement stands without it, but says so
        return {"name": None, "power_limit": None, "error": str(e)}


def label_volume():
    """bench.py's label volume (bench_label_row): 6000 nuclei on an ellipsoidal shell, int32."""
    from platymatch_b200.synthetic import make_label_volume
    n = 6000
    rng = np.random.default_rng(1)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    centers = np.array(SHAPE) / 2.0 + d * (np.array(SHAPE) * 0.42) + rng.normal(0, 4.0, size=(n, 3))
    return make_label_volume(SHAPE, radius=(3.0, 5.0), seed=2, centers=centers, dtype=np.int32)


def intensity_volume(labels):
    """A uint16 image: nuclei brighter than the background, plus noise."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 4096, size=SHAPE, dtype=np.uint16)
    img[labels > 0] += np.uint16(20000)
    return img


def near_rigid():
    """Registration transform T (moving zyx -> fixed zyx): 12 degrees about x, scale 1.03, shift (3, -5, 4), about
    the centre of the volume.  The resample takes M = inv(T).  In zyx order a rotation about x mixes z and y, so
    one output plane draws from ~100 source planes."""
    a = np.deg2rad(12.0)
    R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]) * 1.03
    c = (np.array(SHAPE) - 1) / 2.0
    T = np.eye(4)
    T[:3, :3], T[:3, 3] = R, c + np.array([3.0, -5.0, 4.0]) - R @ c
    return T


def to_device(torch, a):
    if a.dtype == np.uint16:
        return torch.from_numpy(a.view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(a).cuda()


def time_ms(torch, fn, flush, warmup=3, reps=10):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        flush.fill_(1)
        flush.fill_(2)             # (~100 us of device work: the host is ahead when the timed region starts)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.mean(ms)), float(np.min(ms)), float(np.max(ms))


def copy_gbs(torch, flush, nbytes=1 << 30):
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    a.fill_(3)
    b = torch.empty_like(a)
    ms, _, _ = time_ms(torch, lambda: b.copy_(a), flush)
    return 2 * nbytes / (ms * 1e-3) / 1e9


def measure(torch, D, vols, flush, peak, transforms=("identity", "near_rigid")):
    rows = []
    for name, vol, order in vols:
        src = to_device(torch, vol)
        out = torch.empty_like(src)
        nbytes = 2 * vol.nbytes
        for tname in transforms:
            M = torch.from_numpy(np.linalg.inv(near_rigid()) if tname == "near_rigid" else np.eye(4)).cuda()
            ms, lo, hi = time_ms(torch, lambda: D.resample_affine(src, M, SHAPE, order, 0.0, out=out), flush)
            gbs = nbytes / (ms * 1e-3) / 1e9
            rows.append({"workload": name, "dtype": str(vol.dtype), "order": order, "transform": tname,
                         "kernel_ms": ms, "kernel_ms_min": lo, "kernel_ms_max": hi, "algorithmic_bytes": nbytes,
                         "achieved_gbs": gbs, "frac_of_copy": gbs / peak, "voxels_per_s": vol.size / (ms * 1e-3)})
        del src, out
    return rows


def cpu_baseline(torch, D, vols, rows):
    import scipy.ndimage as nd
    M = np.linalg.inv(near_rigid())
    for name, vol, order in vols:
        t0 = time.perf_counter()
        ref = nd.affine_transform(vol, M[:3, :3], offset=M[:3, 3], output_shape=SHAPE, order=order, mode="constant",
                                  cval=0.0)
        t = time.perf_counter() - t0
        got = D.resample_affine(to_device(torch, vol), torch.from_numpy(M).cuda(), SHAPE, order, 0.0)
        got = (got.view(torch.int16).cpu().numpy().view(np.uint16) if vol.dtype == np.uint16 else got.cpu().numpy())
        diff = int(np.count_nonzero(got != ref))
        gpu = next(r for r in rows if r["workload"] == name and r["transform"] == "near_rigid")
        gpu["cpu_baseline"] = {"seconds": t, "voxels_per_s": vol.size / t, "cores": 1,
                               "kind": "scipy.ndimage.affine_transform %s" % __import__("scipy").__version__,
                               "speedup": t / (gpu["kernel_ms"] * 1e-3), "voxels_differing_from_gpu": diff}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    args = ap.parse_args()
    import torch
    from platymatch_b200 import device as D
    D._torch()
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    labels = label_volume()
    vols = [("labels_int32_nearest", labels, 0), ("intensity_uint16_linear", intensity_volume(labels), 1)]
    peak = copy_gbs(torch, flush)
    rows = measure(torch, D, vols, flush, peak)
    if not args.no_cpu_baseline:
        cpu_baseline(torch, D, vols, rows)
    print(json.dumps({"gpu": gpu_identity(), "shape": list(SHAPE), "copy_gbs": peak,
                      "copy": "torch d2d copy of 1 GiB, read + write bytes", "l2": "160 MB flush (x2) before each call",
                      "transform_near_rigid": near_rigid().tolist(), "rows": rows}), flush=True)


if __name__ == "__main__":
    main()
