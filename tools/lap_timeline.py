"""Where the assignment's time goes in the headline step (GPU).

Runs bench.py's resident step (the same 4 pairs, seeds, cost buffer and max_bid_rounds = 2048) under
torch.profiler with CUDA activities, one step per pair after a warm-up, and prints

  * for each step, every assignment kernel (pm_lap_* / pm_ls_*) with its stream, start (us from the step's
    first assignment kernel) and duration, then each stream's chain from its first to its last assignment kernel
    and which chain ends last, with the share of pm_lap_sap_sparse_kernel in it;
  * for each matrix (4 pairs x 4 hypotheses), the solver's statistics DIJKSTRA_STEPS, SAP_CYCLES (and their ratio,
    the cost of one Dijkstra step), REFRESH_CYCLES, AUCTION_CYCLES, BIDS and REFRESHES.

The profiler slows the host, so this is a run of its own, never a timing: bench.py measures the step.

    python tools/lap_timeline.py [--warmup 3] > timeline.txt
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the headline workload's constants)

KERNEL = re.compile(r"\b(pm_l(?:ap|s)_\w+?)(?:<(\w+)>)?\(")
STATS = ["DIJKSTRA_STEPS", "SAP_CYCLES", "REFRESH_CYCLES", "AUCTION_CYCLES", "BIDS", "REFRESHES"]


def assignment_kernels(trace_path):
    """-> [(name, stream, start_us, dur_us)] of the assignment kernels in a chrome trace, by start time."""
    out = []
    for e in json.load(open(trace_path))["traceEvents"]:
        if e.get("cat") != "kernel":
            continue
        m = KERNEL.search(e.get("name", ""))
        if m:
            name = m.group(1) + ("<%s>" % m.group(2) if m.group(2) else "")
            out.append((name, int(e["args"].get("stream", -1)), float(e["ts"]), float(e["dur"])))
    return sorted(out, key=lambda k: k[2])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from platymatch_b200 import device as D, pipeline as P
    from platymatch_b200._lib import LAP_STAT
    from platymatch_b200.synthetic import make_pair

    torch.cuda.set_device(0)
    kw = dict(ransac_trials=bench.TRIALS, icp_iterations=bench.ICP_ITERS, max_bid_rounds=2048)
    n_slots = 4
    pairs = [make_pair(bench.N_FIXED, seed=bench.N_FIXED + 97 * s) for s in range(n_slots)]
    n1, n2 = pairs[0]["moving"].shape[1], pairs[0]["fixed"].shape[1]
    dev_pairs = [(D.to_device_points(p["moving"]), D.to_device_points(p["fixed"])) for p in pairs]
    cost_buf = torch.empty((4, n1, (n2 + 3) // 4 * 4), dtype=torch.float32, device="cuda")

    def step_resident(s):
        m, f = dev_pairs[s % n_slots]
        dm, df = P.describe_pair(m, f, 1, 4, transposed=True)
        return P.register_described(dm, df, seed=s, cost_out=cost_buf, **kw)

    for s in range(args.warmup):
        step_resident(s)
    torch.cuda.synchronize()

    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        gpu = "unknown"
    print("lap_timeline: %d x %d, 4 hypotheses, max_bid_rounds 2048; GPU %s (%s)"
          % (n1, n2, torch.cuda.get_device_name(0), gpu))
    per_matrix = []
    with tempfile.TemporaryDirectory() as tmp:
        for s in range(n_slots):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                res = step_resident(s)
                torch.cuda.synchronize()
            path = os.path.join(tmp, "step%d.json" % s)
            prof.export_chrome_trace(path)
            ks = assignment_kernels(path)
            stats = res["lap_stats"].cpu().numpy()
            t0 = ks[0][2] if ks else 0.0
            print("\nstep %d (pair slot %d): %d assignment kernels" % (s, s % n_slots, len(ks)))
            print("  %-34s %7s %10s %10s" % ("kernel", "stream", "start_us", "dur_us"))
            for name, stream, ts, dur in ks:
                print("  %-34s %7d %10.1f %10.1f" % (name, stream, ts - t0, dur))
            chains = {}
            for name, stream, ts, dur in ks:
                c = chains.setdefault(stream, {"start": ts, "end": ts + dur, "sap": 0.0, "busy": 0.0})
                c["end"] = max(c["end"], ts + dur)
                c["busy"] += dur
                if name == "pm_lap_sap_sparse_kernel":
                    c["sap"] += dur
            last = max(chains, key=lambda k: chains[k]["end"]) if chains else None
            for stream, c in sorted(chains.items(), key=lambda kv: kv[1]["end"]):
                span = c["end"] - c["start"]
                print("  chain on stream %d: %.1f -> %.1f us (span %.1f us, kernels %.1f us), sap_sparse %.1f us = %.0f %% "
                      "of the span%s" % (stream, c["start"] - t0, c["end"] - t0, span, c["busy"], c["sap"],
                                        100.0 * c["sap"] / span if span > 0 else 0.0,
                                        "   <- ends last" if stream == last else ""))
            for h, row in enumerate(stats):
                st = {k: int(row[LAP_STAT[k]]) for k in STATS}
                st["cycles_per_step"] = st["SAP_CYCLES"] / st["DIJKSTRA_STEPS"] if st["DIJKSTRA_STEPS"] else 0.0
                per_matrix.append((s % n_slots, h, st))
    print("\nper matrix (pair slot, hypothesis):")
    print("  %4s %3s %9s %11s %10s %14s %14s %8s %9s" % ("pair", "hyp", "dij_steps", "sap_cycles", "cyc/step",
                                                         "refresh_cyc", "auction_cyc", "bids", "refreshes"))
    for slot, h, st in per_matrix:
        print("  %4d %3d %9d %11d %10.0f %14d %14d %8d %9d" % (slot, h, st["DIJKSTRA_STEPS"], st["SAP_CYCLES"],
                                                            st["cycles_per_step"], st["REFRESH_CYCLES"],
                                                            st["AUCTION_CYCLES"], st["BIDS"], st["REFRESHES"]))
    steps = sum(st["DIJKSTRA_STEPS"] for _, _, st in per_matrix)
    cyc = sum(st["SAP_CYCLES"] for _, _, st in per_matrix)
    print("  all 16 matrices: %d Dijkstra steps, %d SAP cycles, %.0f cycles per step" % (steps, cyc, cyc / max(steps, 1)))


if __name__ == "__main__":
    main()
