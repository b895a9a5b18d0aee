"""Measure the thin-plate spline deformation (DESIGN §8 row 8) on one GPU; print one JSON line.

Workload: match_labels' (tools/overlap_bench.py): bench.py's 384 x 512 x 512 label volume of 6000 nuclei is the fixed
specimen.  Its moving counterpart has the fixed centres displaced by six Gaussian bumps (make_deformed_pair's field:
sigma 0.2 x the extent, 3 % of the extent each), mapped through the inverse of the near-rigid transform of
tools/resample_bench.py and jittered (sigma 1); that transform is the affine registration handed to the deformation.
- match_nuclei (host clock, mean of 3 after 1).
- the fit at K = the number of pairs: pm_spline_system and torch.linalg.solve_ex (CUDA events, mean of 5), fit_spline
  end to end from host arrays (host clock, mean of 3 after 1).
- pm_spline_eval on 6000 points (events, mean of 10).
- pm_resample_spline on the full volume through the inverse spline: int32 labels order 0 and float32 intensities
  order 1 (events, 1 warm-up, mean of 3; each call is about 0.65 s of FP64 work, so what the L2
  holds between calls does not matter and there is no flush).
- the FP64 instructions per (voxel, centre) of the warp's inner loop, counted in `cuobjdump -sass` of the built object,
  the FP64 lanes per SM per clock that the measured time implies, and the time that count takes at 32 and at 64 FP64
  lanes per SM per clock (the card's max SM clock).
- CPU baseline (one core): RBFInterpolator at the same K (measured); RBFInterpolator + map_coordinates on an
  8 x 64 x 128 corner of the output (measured, per voxel, compared with the GPU's voxels there); the full volume at
  that rate is reported as extrapolated.

    python tools/deform_bench.py [--no-cpu-baseline]
"""
import os

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):     # the CPU baseline runs on one core
    os.environ.setdefault(_v, "1")

import argparse
import json
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from resample_bench import SHAPE, near_rigid                            # noqa: E402

N = 6000
SUB = (8, 64, 128)


def gpu_identity():
    """Name, power limit and max SM clock of GPU 0 (a read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, limit, clock = [s.strip() for s in out.split(",")[:3]]
        return {"name": name, "power_limit": limit, "max_sm_clock": clock}
    except Exception as e:                        # the measurement stands without it, but says so
        return {"name": None, "power_limit": None, "max_sm_clock": None, "error": str(e)}


def centres_pair():
    """(fixed (3, N), moving (3, N), T): the fixed centres of resample_bench.label_volume and their deformed, moved,
    jittered counterparts (moving nucleus i is fixed nucleus i)."""
    from platymatch_b200.synthetic import deformation_field
    rng = np.random.default_rng(1)
    d = rng.normal(size=(N, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    fixed = (np.array(SHAPE) / 2.0 + d * (np.array(SHAPE) * 0.42) + rng.normal(0, 4.0, size=(N, 3))).T
    r = np.random.default_rng(7)
    extent = float((fixed.max(axis=1) - fixed.min(axis=1)).max())
    v = r.standard_normal((3, 6))
    v /= np.linalg.norm(v, axis=0, keepdims=True)
    field = {"centres": fixed[:, r.choice(N, 6, replace=False)].copy(), "sigma": np.full(6, 0.2 * extent),
             "vectors": v * (0.03 * extent)}
    T = near_rigid()
    Ti = np.linalg.inv(T)
    moving = Ti[:3, :3] @ (fixed + deformation_field(fixed, field)) + Ti[:3, 3:4] + r.normal(0, 1.0, size=(3, N))
    return np.ascontiguousarray(fixed), np.ascontiguousarray(moving), T


def events_ms(torch, fn, warmup=1, reps=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return {"mean": float(np.mean(ms)), "min": float(np.min(ms)), "max": float(np.max(ms))}


def host_s(torch, fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return {"mean": float(np.mean(ts)), "min": float(np.min(ts)), "max": float(np.max(ts))}


def sass_fp64_per_pair(kernel="pm_resample_spline_kernelIiLi0E"):
    """FP64-pipe instructions per (voxel, centre) in the warp kernel's inner loop (int32, order 0): the body of the
    backward branch that contains the shared-memory centre loads, divided by (centres per iteration x 4 voxels)."""
    obj = os.path.join(ROOT, "platymatch_b200", "csrc", "build", "pm_spline.o")
    cuobjdump = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    body = next(f for f in funcs if f.startswith("_Z25" + kernel) or kernel in f.split("\n", 1)[0])
    ins = re.findall(r"/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]+)([^;]*);", body)
    addr = [int(a, 16) for a, _, _ in ins]
    best = None
    for i, (a, op, rest) in enumerate(ins):
        m = re.search(r"0x([0-9a-f]+)", rest)
        if op.startswith("BRA") and m and int(m.group(1), 16) < addr[i]:
            lo = addr.index(int(m.group(1), 16))
            loop = ins[lo:i + 1]
            if sum(op2 == "LDS.128" for _, op2, _ in loop) >= 3 and (best is None or len(loop) > len(best)):
                best = loop
    ops = {}
    for _, op, _ in best:
        key = op.split(".")[0]
        if key in ("DADD", "DMUL", "DFMA", "DSETP", "MUFU"):
            ops[op if key == "MUFU" else key] = ops.get(op if key == "MUFU" else key, 0) + 1
    centres = sum(op == "LDS.128" for _, op, _ in best) // 3
    fp64 = sum(v for k, v in ops.items() if k.startswith("D"))
    return {"loop_instructions": len(best), "centres_per_iteration": centres, "voxels_per_thread": 4, "ops": ops,
            "fp64_per_voxel_centre": fp64 / (centres * 4)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    args = ap.parse_args()
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.estimate_transform import deformable as DF
    from platymatch_b200.synthetic import make_label_volume
    D._torch()
    gpu = gpu_identity()
    fixed, moving, T = centres_pair()
    # the moving specimen's volumes, in the moving frame
    labels = make_label_volume(SHAPE, radius=(3.0, 5.0), seed=2, centers=moving.T, dtype=np.int32)
    rng = np.random.default_rng(3)
    intensity = (rng.uniform(0, 100, size=SHAPE) + 400.0 * (labels > 0)).astype(np.float32)
    out = {"gpu": gpu, "shape": list(SHAPE), "nuclei": N, "transform": T.tolist()}
    t_match = host_s(torch, lambda: DF.match_nuclei(moving, fixed, T))
    mi, fi, dist = DF.match_nuclei(moving, fixed, T)
    k = int(mi.size)
    out["match_nuclei"] = {"s": t_match, "pairs": k, "correct": float(np.mean(mi == fi)),
                           "median_distance": float(np.median(dist))}
    src, dst = fixed[:, fi], moving[:, mi]                       # the inverse spline: fixed -> moving (the pull map)
    lam = DF.DEFAULT_SMOOTHING
    y = np.ascontiguousarray(src.T)
    shift, scale = DF.shift_scale(y)
    yt = torch.from_numpy(y).cuda()
    sst = torch.from_numpy(np.r_[shift, scale]).cuda()
    lhs = D.spline_system(yt, sst, lam)
    rhs = torch.zeros((k + 4, 3), dtype=torch.float64, device="cuda")
    rhs[:k] = torch.from_numpy(np.ascontiguousarray(dst.T)).cuda()
    t_sys = events_ms(torch, lambda: D.spline_system(yt, sst, lam, out=lhs))
    t_solve = events_ms(torch, lambda: torch.linalg.solve_ex(lhs, rhs))
    del lhs
    t_fit = host_s(torch, lambda: DF.fit_spline(src, dst, lam))
    sp = DF.fit_spline(src, dst, lam)
    out["fit"] = {"k": k, "smoothing": lam, "system_kernel_ms": t_sys, "solve_ex_ms": t_solve, "fit_spline_s": t_fit,
                  "matrix_bytes": 8 * (k + 4) ** 2}
    pts = torch.from_numpy(np.ascontiguousarray(fixed.T)).cuda()
    out["eval_6000_ms"] = events_ms(torch, lambda: D.spline_eval(sp.centres, sp.coeffs, sp.shift_scale, pts), reps=10)
    vox = int(np.prod(SHAPE))
    sass = sass_fp64_per_pair()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    try:
        clock_hz = float(gpu["max_sm_clock"].split()[0]) * 1e6
    except Exception:
        clock_hz = None
    warps = {}
    for name, vol, order in (("int32_order0", labels, 0), ("float32_order1", intensity, 1)):
        sv = D.to_device_volume(vol)
        o = torch.empty(SHAPE, dtype=sv.dtype, device="cuda")
        t = events_ms(torch, lambda: D.resample_spline(sv, sp.centres, sp.coeffs, sp.shift_scale, SHAPE, order, 0.0,
                                                       out=o), warmup=1, reps=3)
        row = {"ms": t, "voxel_centre_pairs": vox * k,
               "ns_per_voxel": t["mean"] * 1e6 / vox,
               "pairs_per_s": vox * k / (t["mean"] * 1e-3)}
        if clock_hz:
            lanes = sass["fp64_per_voxel_centre"] * vox * k / (t["mean"] * 1e-3) / (sms * clock_hz)
            row["fp64_lanes_per_sm_clock_achieved"] = lanes
            for n_lanes in (32, 64):
                bound_ms = sass["fp64_per_voxel_centre"] * vox * k / n_lanes / (sms * clock_hz) * 1e3
                row["fp64_bound_ms_%d_lanes" % n_lanes] = bound_ms
                row["frac_of_fp64_bound_%d_lanes" % n_lanes] = bound_ms / t["mean"]
        warps[name] = row
        if name == "int32_order0":
            gpu_corner = o[:SUB[0], :SUB[1], :SUB[2]].cpu().numpy()
        del sv, o
        torch.cuda.empty_cache()
    out["warp"] = warps
    out["sass"] = sass
    out["fp64_bound_model"] = ("SASS FP64 instructions per (voxel, centre) x pairs / (lanes x %d SMs x max SM clock); "
                               "32 lanes = one FP64 warp instruction per SM per clock, 64 lanes = NVIDIA's published "
                               "FP64 rate of the HGX B200 (37 TFLOPS per GPU) at that clock" % sms)
    if not args.no_cpu_baseline:
        import scipy
        import scipy.ndimage as nd
        from scipy.interpolate import RBFInterpolator
        t0 = time.perf_counter()
        ref = RBFInterpolator(src.T, dst.T, kernel="linear", degree=1, smoothing=lam)
        t_cfit = time.perf_counter() - t0
        g = np.stack(np.meshgrid(*(np.arange(n, dtype=np.float64) for n in SUB), indexing="ij"), -1).reshape(-1, 3)
        t0 = time.perf_counter()
        c = ref(g).T
        w = nd.map_coordinates(labels, c, order=0, mode="constant", cval=0).reshape(SUB)
        t_cwarp = time.perf_counter() - t0
        per_voxel = t_cwarp / g.shape[0]
        out["cpu_baseline"] = {
            "cores": 1, "kind": "scipy %s RBFInterpolator(kernel='linear', degree=1) + map_coordinates" % scipy.__version__,
            "fit_s": t_cfit, "fit_speedup_vs_fit_spline": t_cfit / t_fit["mean"],
            "coefficients_max_abs_diff": float(np.abs(sp.coeffs.cpu().numpy() - ref._coeffs).max()),
            "subvolume": list(SUB), "subvolume_warp_s": t_cwarp, "s_per_voxel": per_voxel,
            "subvolume_equal_voxels": int(np.count_nonzero(w == gpu_corner)), "subvolume_voxels": int(w.size),
            "full_volume_s_extrapolated": per_voxel * vox,
            "full_volume_speedup_extrapolated": per_voxel * vox / (warps["int32_order0"]["ms"]["mean"] * 1e-3)}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
