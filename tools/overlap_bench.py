"""Measure the label-overlap table (pm_label_overlap, DESIGN §8 row 7) and `match_labels` on one GPU; print one JSON line.

Workloads: bench.py's 384 x 512 x 512 label volume (6000 nuclei, int32) against itself warped by a near-rigid transform
through `transform_image` (12 degrees about x, scale 1.03, shift (3, -5, 4) about the centre), as int32 / int32 and as
int32 / uint16.  Every volume (403 MB int32, 201 MB uint16) is larger than the B200's 126 MB L2, and each timed call
reads both once, so no flush is needed between calls.
- table pass: CUDA events around one pm_label_overlap call (memsets, stream kernel, compaction) at the capacity
  match_labels picks, 3 warm-up calls, mean of 20; the kernels' own times from torch.profiler in a separate loop.
  Algorithmic bytes = one read of each volume; the reference bandwidth is a 1 GiB device-to-device copy measured in
  the same process.
- sort: torch.sort of the keys plus the gather of the counts (events, mean of 20).
- assignment per threshold (0.1 / 0.5 / 0.9): the matrix build and D.lap_solve (events, mean of 5).
- match_labels end to end from host arrays (host clock, mean of 3).
- CPU baseline: the numpy + scipy oracle (tests/test_gpu_label_overlap.py) on one core, one table and the matching on
  it, with an equality flag.

    python tools/overlap_bench.py [--no-cpu-baseline]
"""
import os

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):     # the CPU baseline runs on one core
    os.environ.setdefault(_v, "1")

import argparse
import json
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from resample_bench import SHAPE, gpu_identity, label_volume, near_rigid       # noqa: E402

THRESHOLDS = (0.1, 0.5, 0.9)


def events_ms(torch, fn, warmup=3, reps=20):
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


def copy_gbs(torch, nbytes=1 << 30):
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    a.fill_(3)
    b = torch.empty_like(a)
    t = events_ms(torch, lambda: b.copy_(a), reps=10)
    return 2 * nbytes / (t["mean"] * 1e-3) / 1e9


def kernel_times(torch, fn, reps=10):
    """Mean device time per call of each kernel named pm_overlap_* (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "pm_overlap" in ev.key or "emset" in ev.key:
            name = "pm_overlap_stream_kernel" if "stream_kernel" in ev.key else \
                   "pm_overlap_compact_kernel" if "compact" in ev.key else "memset"
            dt = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            out[name] = out.get(name, 0.0) + dt / 1e3 / reps            # us -> ms per call
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    args = ap.parse_args()
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200 import evaluate_metrics as E
    from platymatch_b200.utils.images import transform_image
    D._torch()
    fixed = label_volume()
    warped32 = transform_image(fixed, near_rigid(), SHAPE, order=0)
    warped16 = transform_image(fixed.astype(np.uint16), near_rigid(), SHAPE, order=0)
    peak = copy_gbs(torch)
    rows = []
    for name, b in (("int32_int32", warped32), ("int32_uint16", warped16)):
        ta, tb = D.to_device_volume(fixed), D.to_device_volume(b)
        mx = torch.zeros(2, dtype=torch.int32, device="cuda")
        D.label_max_id(ta, mx[0:1])
        D.label_max_id(tb, mx[1:2])
        ma, mb = (int(v) for v in mx.cpu().numpy())
        cap = E._initial_capacity(ma, mb, fixed.size)
        keys, counts, n_out = D.label_overlap(ta, tb, cap)
        n_pairs, dropped = (int(v) for v in n_out.cpu().numpy())
        nbytes = fixed.nbytes + b.nbytes
        t_pass = events_ms(torch, lambda: D.label_overlap(ta, tb, cap))
        kern = kernel_times(torch, lambda: D.label_overlap(ta, tb, cap))
        ks = keys[:n_pairs]

        def sort():
            s, o = torch.sort(ks)
            return counts[:n_pairs][o]
        t_sort = events_ms(torch, sort)
        row = {"workload": name, "algorithmic_bytes": nbytes, "capacity": cap, "pairs": n_pairs, "dropped": dropped,
               "max_ids": [ma, mb], "call_ms": t_pass, "kernels_ms": kern,
               "call_gbs": nbytes / (t_pass["mean"] * 1e-3) / 1e9,
               "call_frac_of_copy": nbytes / (t_pass["mean"] * 1e-3) / 1e9 / peak, "sort_ms": t_sort}
        if "pm_overlap_stream_kernel" in kern:
            gbs = nbytes / (kern["pm_overlap_stream_kernel"] * 1e-3) / 1e9
            row["stream_kernel_gbs"], row["stream_kernel_frac_of_copy"] = gbs, gbs / peak
        # assignment per threshold, on the table match_labels builds
        ia, ib, n = E._contingency(fixed, b)
        sa, sb = E._sizes(ia, n), E._sizes(ib, n)
        fg = (ia > 0) & (ib > 0)
        iou = n[fg] / (sa[fg] + sb[fg] - n[fg]).astype(np.float64)
        row["assignment"] = []
        for t in THRESHOLDS:
            prob = E._matching_problem(ia[fg], ib[fg], iou, t)
            if prob is None:                      # no admissible pair: match_labels makes no solve
                row["assignment"].append({"threshold": t, "admissible": 0, "solve_ms": None})
                continue
            tm = events_ms(torch, lambda: E._solve(torch, prob), warmup=1, reps=5)
            row["assignment"].append({"threshold": t, "rows": int(prob[1].size), "cols": int(prob[2].size),
                                      "admissible": int(prob[3].size), "solve_ms": tm})
        wall = []
        for _ in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = E.match_labels(fixed, b, THRESHOLDS)
            wall.append(time.perf_counter() - t0)
        row["match_labels_s"] = {"mean_of_3_after_1": float(np.mean(wall[1:])), "first": wall[0]}
        row["result"] = {"dice": res["dice"], "jaccard": res["jaccard"], "n_true": res["n_true"], "n_pred": res["n_pred"],
                         "per_threshold": [{k: r[k] for k in ("threshold", "tp", "fp", "fn", "f1", "mean_matched_iou")}
                                           for r in res["per_threshold"]]}
        if not args.no_cpu_baseline:
            import test_gpu_label_overlap as T
            t0 = time.perf_counter()                # one table, then the matching on that same table
            otab = T.oracle_table(fixed, b)
            t_tab = time.perf_counter() - t0
            want = T.oracle_match(fixed, b, THRESHOLDS, table=otab)
            t_all = time.perf_counter() - t0
            table_equal = all(np.array_equal(g, w) for g, w in zip((ia, ib, n), otab))
            match_equal = all(g["tp"] == w["tp"] and abs(g["cost"] - w["cost"]) <= 1e-9 * max(1.0, abs(w["cost"]))
                              for g, w in zip(res["per_threshold"], want["per_threshold"]))
            match_equal &= res["dice"] == want["dice"] and res["n_true"] == want["n_true"]
            row["cpu_baseline"] = {"cores": 1, "kind": "numpy %s np.unique + scipy %s linear_sum_assignment"
                                   % (np.__version__, __import__("scipy").__version__),
                                   "table_s": t_tab, "total_s": t_all,
                                   "speedup_vs_match_labels": t_all / row["match_labels_s"]["mean_of_3_after_1"],
                                   "table_equal": bool(table_equal), "match_equal": bool(match_equal)}
        rows.append(row)
        del ta, tb, keys, counts
        torch.cuda.empty_cache()
    print(json.dumps({"gpu": gpu_identity(), "shape": list(SHAPE), "copy_gbs": peak,
                      "copy": "torch d2d copy of 1 GiB, read + write bytes",
                      "l2": "no flush: each volume (403 MB int32, 201 MB uint16) exceeds the 126 MB L2",
                      "transform_near_rigid": near_rigid().tolist(), "rows": rows}), flush=True)


if __name__ == "__main__":
    main()
