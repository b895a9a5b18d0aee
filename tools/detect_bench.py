"""Measure nuclei detection (find_spheres, SURVEY §2 row 10) on one GPU and write profiles/r5_detect.json.

Workload: a 384 x 512 x 512 float32 image of ~6000 nuclei (Gaussian blobs of radius 3-8 on a jittered lattice,
noise 4), radii 3-8 (6 scales), anisotropy 1 and 2.  After a warm-up call: device-event times of each stage (each
scale's 8-pass LoG, the minima, Otsu, the sort and the suppression), mean of 3; and the end-to-end find_spheres call
(host clock, host array in -> host arrays out), mean of 3.  FP64 work of the passes = (1 + 3 lw) operations per voxel
and pass (the DMUL / DADD count per output of pm_detect_pass_kernel's SASS); the bound assumes 32 FP64 lanes per SM
and clock at the card's maximum SM clock.  Bytes = 4 read + 4 written per voxel and pass, + 8 read by the last pass.
The copy bandwidth is a device-to-device tensor copy of 1 GiB measured in the same process.  The CPU baseline is
scipy.ndimage.gaussian_laplace for all scales and tests/detect_oracle.py::find_spheres on one host core, compared
with the GPU.

    python tools/detect_bench.py [--no-cpu-baseline] [--out profiles/r5_detect.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

SHAPE = (384, 512, 512)
RADII = [3.0, 4.0, 5.0, 6.0, 7.0, 8.0]


def gpu_identity():
    """Name, power limit and maximum SM clock of GPU 0 (a read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit, clk = [s.strip() for s in out.split(",")[:3]]
        return {"name": name, "power_limit": limit, "max_sm_clock": clk}
    except Exception as e:
        return {"name": None, "power_limit": None, "max_sm_clock": None, "error": str(e)}


def image():
    from platymatch_b200.synthetic import make_nuclei_image
    rng = np.random.default_rng(1)
    g = [np.arange(10, s - 10, 17.0) for s in SHAPE]
    c = np.stack(np.meshgrid(*g, indexing="ij"), axis=-1).reshape(-1, 3)
    c = c[rng.permutation(len(c))[:6000]] + rng.uniform(-2, 2, (6000, 3))
    return make_nuclei_image(SHAPE, c, rng.uniform(3.0, 8.0, len(c)), contrast=100.0, noise=4.0, seed=2), c


def stages(img_np, anisotropy, reps=3):
    """Device-event time of every stage, in the order find_spheres enqueues them."""
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.detect_nuclei import ss_log
    a, r, an, tf, ov, weights = ss_log._check(img_np, RADII, anisotropy, 0.2, 0.5)
    img = torch.from_numpy(img_np).cuda()
    wd = [[torch.from_numpy(w).cuda() for w in ws] for ws in weights]
    rdev = torch.from_numpy(r).cuda()
    bufs = [torch.empty_like(img) for _ in range(4)]
    slots = [torch.empty_like(img) for _ in range(3)]
    V, K = img.numel(), len(r)
    cap = max(1 << 16, K * V // 1024)
    times = {}

    def timed(name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        times.setdefault(name, []).append(e0.elapsed_time(e1))
        return out

    for _ in range(reps + 1):
        thr = timed("otsu", lambda: D.detect_otsu(img, 0.2))
        keys = torch.full((cap,), np.iinfo(np.int64).max, dtype=torch.int64, device="cuda")
        values = torch.full((cap,), float("inf"), dtype=torch.float32, device="cuda")
        count = torch.zeros(1, dtype=torch.int64, device="cuda")
        for k in range(K):
            def log(k=k):
                gz, t1, t2, acc = bufs
                wz0, wz2, w0, w2 = wd[k]
                s = r[k] / math.sqrt(3.0)
                D.detect_pass(img, 0, wz0, out=gz)
                D.detect_pass(img, 0, wz2, out=t1)
                D.detect_pass(t1, 1, w0, out=t2)
                D.detect_pass(t2, 2, w0, out=acc)
                D.detect_pass(gz, 1, w2, out=t1)
                D.detect_pass(t1, 2, w0, out=t2)
                D.detect_pass(gz, 1, w0, out=t1)
                D.detect_pass(t1, 2, w2, out=slots[k % 3], t0=acc, t1=t2, scale=float(np.float32(s ** 2)))
            timed("log_r%g" % r[k], log)
            if k >= 1:
                timed("minima", lambda k=k: D.detect_minima(slots[(k - 2) % 3] if k >= 2 else None, slots[(k - 1) % 3],
                                                            slots[k % 3], k - 1, thr, keys, values, count))
        timed("minima", lambda: D.detect_minima(slots[(K - 2) % 3], slots[(K - 1) % 3], None, K - 1, thr, keys,
                                                values, count))

        def srt():
            k1, o1 = torch.sort(keys)
            v2, o2 = torch.sort(values[o1], stable=True)
            return k1[o2]
        ks = timed("sort", srt)
        timed("suppress", lambda: D.detect_suppress(ks, count, SHAPE, rdev, float(r[-1]), an, 0.5))
    n_cand = int(count.item())
    out = {}
    for name, t in times.items():
        per = len(t) // (reps + 1)                 # minima runs K times per repetition
        t = np.array(t[per:]).reshape(reps, per).sum(axis=1)
        out[name] = float(t.mean())
    lw = [[int(4.0 * s + 0.5) for s in (rk / math.sqrt(3.0) / an, rk / math.sqrt(3.0))] for rk in r]
    return out, n_cand, lw


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_detect.json"))
    args = ap.parse_args()
    import torch
    from platymatch_b200.detect_nuclei import find_spheres
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    gpu = gpu_identity()
    img, centres = image()
    V = img.size
    x = torch.empty(256 << 20, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    for _ in range(3):
        y.copy_(x)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        y.copy_(x)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = 10 * 2 * x.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del x, y
    clk = gpu.get("max_sm_clock") or ""
    clk_hz = float(clk.split()[0]) * 1e6 if clk and clk.split()[0].replace(".", "").isdigit() else None
    rows = []
    for an in (1.0, 2.0):
        find_spheres(img, RADII, anisotropy=an)                     # warm-up
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            det, rad, resp = find_spheres(img, RADII, anisotropy=an)
            ts.append(time.perf_counter() - t0)
        st, n_cand, lw = stages(img, an)
        d = np.linalg.norm(det.T[:, None, :].astype(np.float32) - centres[None].astype(np.float32), axis=2) \
            if det.shape[1] * len(centres) < 1e8 else None
        log_ms = sum(v for k, v in st.items() if k.startswith("log_"))
        ops = sum(V * ((1 + 3 * lz) * 2 + (1 + 3 * lxy) * 6) for lz, lxy in lw)   # 2 z passes, 6 y / x passes
        byts = V * 8 * 4 * len(RADII) * 2 + V * 8 * len(RADII)
        row = {"anisotropy": an, "find_spheres_s": float(np.mean(ts)), "find_spheres_s_all": ts,
               "detections": int(det.shape[1]), "candidates_above_threshold": n_cand, "stage_ms": st,
               "log_ms_total": log_ms, "fp64_ops": ops, "fp64_tflops": ops / (log_ms * 1e-3) / 1e12,
               "hbm_bytes_log": byts, "log_gbs": byts / (log_ms * 1e-3) / 1e9, "log_frac_of_copy": byts / (log_ms * 1e-3) / 1e9 / copy_gbs,
               "rendered_nuclei_found_within_1_voxel": float(np.mean(d.min(axis=0) <= 1.0)) if d is not None else None}
        if clk_hz:
            bound_s = ops / (148 * 32 * clk_hz)
            row.update({"fp64_bound_ms": bound_s * 1e3, "frac_of_fp64_bound": bound_s / (log_ms * 1e-3)})
        if not args.no_cpu_baseline:
            import scipy
            import scipy.ndimage as nd
            import detect_oracle as O
            img32 = img.astype(np.float32)
            t0 = time.process_time()
            for rk in RADII:
                s = rk / math.sqrt(3.0)
                nd.gaussian_laplace(img32, (s / an, s, s))
            t_lap = time.process_time() - t0
            t0 = time.process_time()
            ref = O.find_spheres(img, RADII, anisotropy=an)
            t_orc = time.process_time() - t0
            row["cpu_baseline"] = {"kind": "scipy %s gaussian_laplace, 6 scales, one core" % scipy.__version__,
                                   "gaussian_laplace_s": t_lap, "oracle_find_spheres_s": t_orc,
                                   "speedup_vs_oracle": t_orc / float(np.mean(ts)),
                                   "detections_equal": bool(all(np.array_equal(g, e) for g, e in
                                                                zip((det, rad, resp), ref)))}
        rows.append(row)
        print(json.dumps(row), flush=True)
    res = {"gpu": gpu, "shape": list(SHAPE), "radii": RADII, "nuclei_rendered": len(centres), "copy_gbs": copy_gbs,
           "copy": "torch d2d copy of 1 GiB, read + write bytes", "rows": rows}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f)
        f.write("\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
