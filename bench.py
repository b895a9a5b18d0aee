#!/usr/bin/env python
"""bench.py — headline benchmark of the estimate_transform hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this implementation (CUDA, C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # CPU port of the reference's path (oracle/)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy

Workload (config.workload): BASELINE.json configs[1] — synthetic 8k x 8k-nucleus embryo-like pair
(N2 = 8000 fixed, N1 = 7200 moving after 10 % dropout, jitter 2 px), unsupervised
estimate_transform: shape context -> 4 chi^2 cost matrices -> 4 assignments -> 4 affine RANSACs
(8000 trials each, the widget default) -> ICP (50 iterations).
A step = one full registration of one pair.  metric = registrations/sec (whole job, all ranks).
  value   inputs already resident in HBM when the timed region starts
  e2e     the public Python API with HOST (pinned) inputs: H2D of both clouds and D2H of the results
          inside the timed region
Multi-GPU (torchrun, one rank per GPU): independent specimen pairs are sharded across ranks (no
data-path collective) -> weak scaling; timing = max over ranks of the device time.
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "synthetic 8k x 8k-nucleus pair (N1=7200 moving, N2=8000 fixed), unsupervised estimate_transform"
N_FIXED = 8000
TRIALS = 8000
ICP_ITERS = 50
FLOP_PER_PAIR = 1801.0        # SURVEY §8(d): 5 FLOP per bin pair x 360 + 1
METRIC = "registrations/sec"
ALLPAIRS_IN_FLIGHT = 8            # measured on one GPU (tools/allpairs_bench.py): 19.5 / 39 / 50 / 65 / 72 pairs/s with 1 / 3 / 4 / 6 / 8
CHI2_NCU_DRAM_BYTES = 186.9e6     # ncu --set full at the headline size, round 2 (10.7 MB read + 176.2 MB written)
CHI2_NCU_DRAM_BYTES_DENSE = 196.2e6   # the filled-ellipsoid pair (20.2 MB read + 176.0 MB written), profiles/r2_chi2_kernel_dense.txt


def workload_config(n1, n2, trials):
    """`config` of the JSON line: the workload, identical keys and values in both arms (b200 and reference)."""
    return {"workload": WORKLOAD, "n_fixed": int(n2), "n_moving": int(n1), "hypotheses": 4, "ransac_trials": int(trials),
            "icp_iterations": ICP_ITERS,
            "l2": "inputs larger than L2: 4 x %.0f MB cost matrices rewritten every step (> 126 MB L2); 4 input pairs cycled"
                  % (n1 * n2 * 4 / 1e6)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-fixed", type=int, default=N_FIXED, help="override the workload size (not the headline)")
    ap.add_argument("--trials", type=int, default=TRIALS)
    ap.add_argument("--bid-rounds", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stages", action="store_true", help="print a per-stage device-time breakdown to stderr")
    ap.add_argument("--in-flight", type=int, default=6,
                    help="registrations in flight per GPU for the secondary `pipelined` throughput number (0 = skip)")
    ap.add_argument("--no-rows", action="store_true", help="skip the secondary measurements of the widened rows")
    ap.add_argument("--no-square", action="store_true", help="skip the equal-counts (no slack columns) registration row")
    ap.add_argument("--lean", action="store_true",
                    help="profiling aid: warm-up + timed resident steps only (no e2e, stage, roofline or CPU legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ------------------------------------------------------------------------------------------- CPU arm
class CpuArm:
    """The reference's CPU path for this workload, timed on the host cores: the oracle port (oracle/, C + numpy,
    pinned to the unmodified reference by tests/golden), all threads the process may use.

      full_run()      ONE complete, unsampled registration, every stage timed: 6 descriptor sets (the reference
                      builds 2 moving + 4 fixed, shape_context.py:170-185), 4 distinct hypotheses x {full chi^2 matrix,
                      full assignment, full RANSAC}, ICP.  A measured run, no extrapolation.
      sample_step(s)  a bounded sample of the same work: 1/FR of the descriptor query rows, 1/FR of the rows of each of
                      the 4 cost matrices, 1/FR of the RANSAC trials, 1/10 of the ICP iterations, scaled by the sampled
                      fraction (these loops are embarrassingly parallel over the sampled index), and the FULL assignment
                      of ONE hypothesis (s mod 4; the assignment is superlinear and cannot be sampled), the other three
                      taken from their latest measurement (initially the full run).
    Everything the samples need but do not time (full histograms, full matrices, assignments) is built ONCE here."""
    FR = 8
    H = 4

    def __init__(self, pair, trials, icp_iters, threads=None):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        self.O = O
        O.set_num_threads(threads or len(os.sched_getaffinity(0)))      # (torchrun exports OMP_NUM_THREADS=1)
        self.cores = O.num_threads()
        self.m, self.f = pair["moving"], pair["fixed"]
        self.trials, self.icp_iters = trials, icp_iters
        self.n1, self.n2 = self.m.shape[1], self.f.shape[1]
        self.full = None
        self.lap_s = None

    def full_run(self):
        O, m, f, t = self.O, self.m, self.f, {}
        t_all = time.perf_counter()
        t0 = time.perf_counter()
        self.mc, self.fc = O.get_centroid(m, False), O.get_centroid(f, False)
        self.md, self.fd = O.get_mean_distance(m, False), O.get_mean_distance(f, False)
        t["mean_distance"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        self.xm, self.xf = O.pca_first_axis(m.T), O.pca_first_axis(f.T)
        um = [O.normalise_counts(O.shape_context_counts(m.T, self.mc, self.md, self.xm, v)[0]) for v in (1, 2)]
        uf = [O.normalise_counts(O.shape_context_counts(f.T, self.fc, self.fd, self.xf, v)[0]) for v in (1, 2, 3, 4)]
        t["descriptors"] = time.perf_counter() - t0
        self.um, self.uf = um[0], uf
        t["chi2"], t["lap"], t["ransac"] = 0.0, 0.0, 0.0
        self.lap_s, self.assign, inliers, mats = [], [], [], []
        for q in range(self.H):
            t0 = time.perf_counter()
            U = O.unary_distance_matrix(um[0], uf[q])
            t["chi2"] += time.perf_counter() - t0
            t0 = time.perf_counter()
            r, c = O.linear_sum_assignment(U)
            self.lap_s.append(time.perf_counter() - t0)
            t["lap"] += self.lap_s[-1]
            del U
            t0 = time.perf_counter()
            idx = O.ransac_sample_indices(len(r), 4, self.trials, seed=q)
            A, inl = O.do_ransac(m[:, r], f[:, c], 4, self.trials, 16, sample_indices=idx)
            t["ransac"] += time.perf_counter() - t0
            self.assign.append((r, c))
            inliers.append(inl)
            mats.append(A)
        t0 = time.perf_counter()
        self.a_sc = mats[int(np.argmax(inliers))]
        O.perform_icp(O.apply_affine_transform(m, self.a_sc), f, self.icp_iters)
        t["icp"] = time.perf_counter() - t0
        self.full = dict(seconds=time.perf_counter() - t_all, stages=t, inliers=[int(x) for x in inliers])
        self.chi2_gpairs = self.H * self.n1 * self.n2 / t["chi2"] / 1e9
        return self.full

    def sample_step(self, s):
        """-> (extrapolated seconds of one registration, wall seconds actually spent)."""
        O, m, f, FR = self.O, self.m, self.f, self.FR
        n1, n2 = self.n1, self.n2
        w0 = time.perf_counter()
        t0 = time.perf_counter()
        O.get_mean_distance(m, False), O.get_mean_distance(f, False)
        t_md = time.perf_counter() - t0
        t0 = time.perf_counter()
        for v in (1, 2):
            O.shape_context_counts(m.T, self.mc, self.md, self.xm, v, query_range=(0, n1 // FR))
        for v in (1, 2, 3, 4):
            O.shape_context_counts(f.T, self.fc, self.fd, self.xf, v, query_range=(0, n2 // FR))
        t_desc = (time.perf_counter() - t0) * FR
        t0 = time.perf_counter()
        for q in range(self.H):
            O.unary_distance_matrix(self.um[: n1 // FR], self.uf[q])
        t_chi2 = (time.perf_counter() - t0) * FR
        q = s % self.H
        U = O.unary_distance_matrix(self.um, self.uf[q])                 # (not timed: input of the assignment)
        t0 = time.perf_counter()
        O.linear_sum_assignment(U)
        self.lap_s[q] = time.perf_counter() - t0
        del U
        t0 = time.perf_counter()
        nt = max(self.trials // FR, 1)
        for q2 in range(self.H):
            r, c = self.assign[q2]
            O.do_ransac(m[:, r], f[:, c], 4, nt, 16, sample_indices=O.ransac_sample_indices(len(r), 4, nt, seed=q2))
        t_ransac = (time.perf_counter() - t0) * self.trials / nt
        it = max(self.icp_iters // 10, 1)
        t0 = time.perf_counter()
        O.perform_icp(O.apply_affine_transform(m, self.a_sc), f, it)
        t_icp = (time.perf_counter() - t0) * self.icp_iters / it
        return t_md + t_desc + t_chi2 + sum(self.lap_s) + t_ransac + t_icp, time.perf_counter() - w0

    def describe_sample(self):
        return ("oracle (C/numpy port of the reference), %d threads.  full_run_s = one complete unsampled registration "
                "(6 descriptor sets, 4 hypotheses x {full chi2 matrix, full assignment, %d RANSAC trials}, %d ICP iterations), "
                "measured.  Each step: full mean-distance; 1/%d of the query nuclei of the 6 descriptor sets; 1/%d of the rows "
                "of each of the 4 chi2 matrices; the full assignment of one hypothesis (step mod 4; the other three from their "
                "latest measurement); 1/%d of the RANSAC trials of each hypothesis; 1/10 of the ICP iterations; sampled stages "
                "scaled by the sampled fraction" % (self.cores, self.trials, self.icp_iters, self.FR, self.FR, self.FR))

    def baseline_dict(self, value):
        return {"value": value, "unit": "registrations/s", "cores": self.cores, "kind": "port",
                "sample": self.describe_sample(), "full_run_s": self.full["seconds"],
                "full_run_stages_s": self.full["stages"], "full_run_inliers": self.full["inliers"],
                "cost_matrix_gpairs_per_s": self.chi2_gpairs}


def run_reference(args):
    """--impl reference: the reference's CPU path.  The reference is pure Python and does not travel to
    the GPU box (and would need ~27 h per 8k registration), so this arm times the oracle port of it
    (oracle/, pinned to the reference by tests/golden) with all host threads: one complete registration first
    (`cpu_baseline.full_run_s`, measured, not extrapolated), then one bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from platymatch_b200.synthetic import make_pair
    t_start = time.perf_counter()
    arm = CpuArm(make_pair(args.n_fixed), args.trials, ICP_ITERS)
    arm.full_run()
    secs, walls = [], []
    for s in range(args.warmup + args.steps):
        sec, wall = arm.sample_step(s)
        if s >= args.warmup:
            secs.append(sec)
            walls.append(wall)
    sec = float(np.mean(secs))
    val = 1.0 / sec
    cb = arm.baseline_dict(val)
    cb["step_wall_s"] = float(np.mean(walls))
    cb["sample_over_full"] = sec / arm.full["seconds"]
    cb["arm_wall_s"] = time.perf_counter() - t_start
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "registrations/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(arm.n1, arm.n2, args.trials),
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- widened rows
def bench_label_row(torch, D, hbm_peak, with_cpu):
    """SURVEY §8(f) row 2: label volume -> detections (reference _dock_widget.py:497-521).  HBM-bound streaming
    kernel: algorithmic bytes = one read of the volume; roofline against the measured copy bandwidth."""
    from platymatch_b200.synthetic import make_label_volume
    shape, n_nuclei = (384, 512, 512), 6000
    rng = np.random.default_rng(1)
    d = rng.normal(size=(n_nuclei, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    centers = np.array(shape) / 2.0 + d * (np.array(shape) * 0.42) + rng.normal(0, 4.0, size=(n_nuclei, 3))
    vol = make_label_volume(shape, radius=(3.0, 5.0), seed=2, centers=centers, dtype=np.int32)
    dev = torch.from_numpy(vol).cuda()
    nbytes = vol.size * 4
    for _ in range(3):
        ids, cen, sizes = D.label_centroids(dev, 1.0, table_size=n_nuclei + 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    ms = 0.0
    for _ in range(reps):
        flush.fill_(1)
        flush.fill_(2)              # (twice: ~100 us of device work, so that the host is ahead when the timed region starts
        e0.record()                 #  and the region measures the device pass, not Python's launch latency)
        D.label_centroids(dev, 1.0, table_size=n_nuclei + 1, sync=False)          # memset + accumulate + compact
        e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1) / reps
    out = {"workload": "label volume %dx%dx%d int32, %d nuclei (%.0f %% foreground)" %
                       (shape + (int(ids.numel()), 100.0 * float((vol > 0).mean()))),
           "ms": ms, "voxels_per_s": vol.size / (ms * 1e-3),
           "roofline": {"kernel": "pm_label_stream_kernel (+ memset of the table + pm_label_finalize_kernel inside the timed region)", "bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9,
                        "peak": hbm_peak, "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / hbm_peak, "of": "measured",
                        "algorithmic_bytes": nbytes, "l2": "160 MB flush (x2) between repetitions"}}
    if with_cpu:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        k = 4                                          # the reference makes one np.where pass over the volume per id
        sub = vol.copy()
        keep = np.isin(sub, np.unique(sub[sub > 0])[:k])
        sub[~keep] = 0
        t0 = time.perf_counter()
        O.detections_from_labels(sub, 1.0)
        t = (time.perf_counter() - t0) / k * int(ids.numel())
        out["cpu_baseline"] = {"value": vol.size / t, "unit": "voxels/s", "cores": 1, "kind": "port",
                               "sample": "oracle restatement of the per-id np.where loop: %d of %d ids timed, scaled" % (k, int(ids.numel()))}
    return out


# ------------------------------------------------------------------------------------------- GPU arm
DUMP_COST_ENTRIES = 1 << 20      # sampled entries per cost matrix: 4 x 4 MB of the ~25 MB a dump takes


def dump_outputs(out_dir, res, cost, n1, n2):
    """--dump-outputs: the results of one resident step as out_dir/<name>.npy, float64 (integers converted exactly)
    or float32 (cost entries).  They are what a caller of register_described receives, copied to the host as the
    public API copies them, and a fixed, seeded sample of the chi^2 cost matrices the step wrote into the caller's
    buffer (`cost_sample` [hypothesis, k] at the flat row-major positions `cost_sample_index`).  lap_stats is left
    out: it counts the solver's work, which may change between builds that compute the same results."""
    import torch
    from platymatch_b200.pipeline import _to_host
    host = _to_host(res)
    arrays = {k: np.asarray(host[k]) for k in ("transform", "transform_sc", "transform_icp", "ransac_A", "inliers",
                                              "best", "lap_cost", "icp_residuals", "edge_ties")}
    arrays["assignment_moving"] = np.stack([m for m, _ in host["assignments"]])
    arrays["assignment_fixed"] = np.stack([f for _, f in host["assignments"]])
    nr, nc = (n2, n1) if n1 > n2 else (n1, n2)
    flat = np.unique(np.random.default_rng(0).integers(0, nr * nc, size=DUMP_COST_ENTRIES))
    sel = torch.from_numpy(flat).to(cost.device)
    arrays["cost_sample"] = cost[:, sel // nc, sel % nc].cpu().numpy()
    arrays["cost_sample_index"] = flat
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.dtype != np.float32:
            a = a.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for ln in open(self.path):
                p = [x.strip() for x in ln.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); mx.append(float(p[2]))
                except ValueError:
                    continue
                for k, nme in enumerate(names):
                    if p[5 + k].lower().startswith("active"):
                        reasons.add(nme)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def fp32_peaks(torch, lib, D, local):
    """FP32 FMA peak of this GPU, measured now with the library's FFMA probe (burst, kernel alone), and nominal."""
    import ctypes
    sink = torch.zeros(4, dtype=torch.float32, device="cuda")
    flops = ctypes.c_double(0)
    sm = lib.pm_sm_count(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        lib.pm_probe_fp32_fma(sm * 8, 2000, D.ptr(sink), ctypes.byref(flops), D.stream_ptr())
    best = 0.0
    for _ in range(3):                       # best of 3: the denominator is a peak, not an average
        e0.record()
        lib.pm_probe_fp32_fma(sm * 8, 20000, D.ptr(sink), ctypes.byref(flops), D.stream_ptr())
        e1.record()
        torch.cuda.synchronize()
        best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best, 2.0 * 128 * sm * 1.965e9 / 1e12


def chi2_roofline(torch, D, P, pair, out_bufs, fp32_probe, fp32_nominal, hbm_peak, label):
    """The cost-matrix kernel alone on one pair's descriptors: algorithmic FLOP (1801 per pair, SURVEY §8d) / launch
    duration (CUDA events on the launching stream, outputs cycled over > L2 worth of buffers), the lane operations the
    kernel actually executes (it skips bins that are empty on both sides of a 128 x 128 tile: 6 FLOP per evaluated bin
    pair, 1 per one-sided bin), and the populated-bin statistics that explain the difference."""
    dm, df = P.describe_pair(pair["moving"], pair["fixed"], 1, 4)
    a_t, b_t = dm.operand(1), df.operand(2)
    n1, n2 = dm.n, df.n
    for q in range(3):
        D.chi2_cost(a_t, b_t, out=out_bufs[q % len(out_bufs)])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nrep = 8
    e0.record()
    for q in range(nrep):
        D.chi2_cost(a_t, b_t, out=out_bufs[q % len(out_bufs)])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / nrep
    # executed work from the per-128-block non-empty-bin masks (what the kernel itself branches on)
    ma = a_t.mask.cpu().numpy().view(np.uint32)
    mb = b_t.mask.cpu().numpy().view(np.uint32)
    bits = lambda m: np.unpackbits(m.view(np.uint8), axis=1, bitorder="little")[:, :360].astype(np.int64)
    ba, bb = bits(ma), bits(mb)
    both = ba @ bb.T                                   # [row blocks, col blocks] bins populated on both sides
    one = ba.sum(1)[:, None] + bb.sum(1)[None, :] - 2 * both
    exec_flop_per_pair = float((6.0 * both + 1.0 * one).mean())
    ha = (dm.counts[0] > 0).float().mean().item()
    alg = FLOP_PER_PAIR * n1 * n2 / (ms * 1e-3) / 1e12
    chi2_bytes = 4.0 * n1 * n2 + 4.0 * 360 * (n1 + n2)      # algorithmic: write the matrix, read both operands once
    return {"kernel": "pm_chi2_kernel", "bound": "fp32", "achieved": alg, "peak": fp32_probe, "unit": "TFLOP/s",
            "frac": alg / fp32_probe, "peak_nominal": fp32_nominal, "frac_of_nominal": alg / fp32_nominal,
            "peak_source": "`peak` = FFMA probe kernel run in this process, burst (MEASURED_PEAKS.json has no FP32 "
                           "CUDA-core figure); `peak_nominal` = 2*128*SMs*1.965 GHz",
            "input": label, "n_moving": n1, "n_fixed": n2, "flop_per_pair": FLOP_PER_PAIR, "launch_ms": ms,
            "gpairs_per_s": n1 * n2 / (ms * 1e-3) / 1e9,
            "executed": {"flop_per_pair": exec_flop_per_pair, "tflops": exec_flop_per_pair * n1 * n2 / (ms * 1e-3) / 1e12,
                         "frac": exec_flop_per_pair * n1 * n2 / (ms * 1e-3) / 1e12 / fp32_probe,
                         "bins_evaluated_per_tile": float(both.mean()), "one_sided_bins_per_tile": float(one.mean()),
                         "nonzero_bin_fraction_per_histogram": ha,
                         "note": "6 FLOP per bin pair populated on both sides of a tile (2 FADD, 2 FMUL, 1 FFMA; + 0.5 "
                                 "MUFU.RCP), 1 per one-sided bin; derived from the kernel's own block masks"},
            "hbm": {"achieved": chi2_bytes / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": chi2_bytes / (ms * 1e-3) / 1e9 / hbm_peak, "of": "measured", "algorithmic_bytes": chi2_bytes}}


def bench_sharded_20k(torch, dist, world, rank, args):
    """BASELINE config 4: ONE 20k x 20k registration spread over all ranks (descriptor rows and cost rows sharded,
    cost rows stored straight into the owner's matrix over NVLink, LAP + RANSAC on the hypothesis owners)."""
    from platymatch_b200 import distributed as PD
    from platymatch_b200.synthetic import make_pair
    n = 20000 if args.n_fixed == N_FIXED else max(args.n_fixed * 2, 1000)
    big = make_pair(n, seed=2)
    kw = dict(ransac_trials=args.trials, icp_iterations=ICP_ITERS)
    for _ in range(2):
        res = PD.register_pair_sharded(big["moving"], big["fixed"], seed=1, **kw)
    reps, ms, stages = 3, [], {}
    for _ in range(reps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        res = PD.register_pair_sharded(big["moving"], big["fixed"], seed=1, **kw)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms.append((time.perf_counter() - t0) * 1e3)
    tm = {}
    PD.register_pair_sharded(big["moving"], big["fixed"], seed=1, timings=tm, **kw)      # separate, synchronising pass
    t = torch.tensor([float(np.mean(ms)), float(res["exchanged_bytes"])] + [tm.get(k, 0.0) for k in
                     ("describe", "chi2_cost+exchange", "lap+ransac", "reduce+icp")], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t = t.cpu().numpy()
    moved = res["transform"] @ np.vstack([big["moving"], np.ones((1, big["moving"].shape[1]))])
    err = float(np.median(np.linalg.norm(moved[:3] - big["fixed"][:, big["gt_fixed_index"]], axis=0)))
    return {"workload": "one %d x %d registration over %d GPU(s): descriptor rows and cost-matrix rows sharded, rows "
                        "delivered to the matrix owner only" % (big["moving"].shape[1], n, world),
            "ms_per_registration": float(t[0]), "registrations_per_s": 1e3 / float(t[0]),
            "timing": "host clock around the public call with HOST inputs (H2D + D2H inside), barrier + synchronize on both sides, max over ranks, mean of %d" % reps,
            "stage_ms_max_over_ranks": {"describe": float(t[2]), "chi2_cost+exchange": float(t[3]), "lap+ransac": float(t[4]),
                                        "reduce+icp": float(t[5])},
            "bytes_sent_to_other_owners_max_over_ranks": float(t[1]), "peer_stores": bool(res["peer_stores"]),
            "inliers": [int(x) for x in res["inliers"]], "median_error_px": err, "recovered": bool(err < 4.0)}


def bench_allpairs(torch, dist, world, rank, args, vary=0.05, runs=2):
    """BASELINE config 5: 12 specimens (~8k nuclei each; sizes differ by up to 5 %, or EXACTLY equal with vary=0: every
    assignment then is a problem without slack columns), all 66 pairs, pulled from one shared work counter by 3
    in-flight registrations per GPU."""
    from platymatch_b200 import distributed as PD
    from platymatch_b200.synthetic import make_specimens
    n = args.n_fixed
    specs = make_specimens(12, n, seed=0, vary=vary)
    clouds = [sp["points"] for sp in specs]
    kw = dict(ransac_trials=args.trials, icp_iterations=ICP_ITERS)
    PD.register_all_pairs(clouds[:4], in_flight=ALLPAIRS_IN_FLIGHT, **kw)                # warm-up (6 pairs)
    best, st_best = None, None
    for _ in range(runs):
        st = {}
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        pairs, T = PD.register_all_pairs(clouds, in_flight=ALLPAIRS_IN_FLIGHT, stats=st, **kw)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, st_best = dt, st
    t = torch.tensor([best], dtype=torch.float64, device="cuda")
    per_rank = torch.zeros((world, 2), dtype=torch.float64, device="cuda")
    per_rank[rank, 0], per_rank[rank, 1] = st_best["pairs_done"], st_best["busy_s"]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(per_rank)
    dt = float(t.item())
    per_rank = per_rank.cpu().numpy()
    ok = 0
    for (i, j), tr in zip(pairs, T):
        gt = specs[j]["A"] @ np.linalg.inv(specs[i]["A"])
        pts = np.vstack([specs[i]["points"][:, :500], np.ones((1, 500))])
        ok += bool(np.median(np.linalg.norm((tr @ pts)[:3] - (gt @ pts)[:3], axis=0)) < 4.0)
    return {"workload": "12 specimens (%s nuclei), %d pairs, %d GPU(s), %d registrations in flight per GPU, shared work counter"
                        % ("%d-%d" % (min(c.shape[1] for c in clouds), max(c.shape[1] for c in clouds)), len(pairs), world,
                           ALLPAIRS_IN_FLIGHT),
            "seconds": dt, "pairs_per_s": len(pairs) / dt, "recovered": int(ok), "pairs": len(pairs),
            "timing": "host clock around register_all_pairs with HOST inputs (descriptors of the 12 specimens, H2D and the "
                      "result gather inside), barrier + synchronize on both sides, max over ranks, best of %d" % runs,
            "pairs_per_rank": [int(x) for x in per_rank[:, 0]], "busy_s_per_rank": [float(x) for x in per_rank[:, 1]]}


def bench_square(torch, args):
    """One registration of a pair with EXACTLY equal nucleus counts (no slack columns in the assignment: the hard
    case for auctions, DESIGN.md §LAP)."""
    import platymatch_b200 as pm
    from platymatch_b200.synthetic import make_pair
    p = make_pair(args.n_fixed, seed=args.n_fixed + 11, dropout=0.0)
    kw = dict(ransac_trials=args.trials, icp_iterations=ICP_ITERS)
    pm.estimate_transform_unsupervised(p["moving"], p["fixed"], seed=1, **kw)
    ms = []
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = pm.estimate_transform_unsupervised(p["moving"], p["fixed"], seed=1, **kw)
        ms.append((time.perf_counter() - t0) * 1e3)
    moved = res["transform"] @ np.vstack([p["moving"], np.ones((1, p["moving"].shape[1]))])
    err = float(np.median(np.linalg.norm(moved[:3] - p["fixed"][:, p["gt_fixed_index"]], axis=0)))
    st = res["lap_stats"]
    return {"workload": "%d x %d pair (equal counts), unsupervised estimate_transform through the public API" %
                        (p["moving"].shape[1], p["fixed"].shape[1]),
            "ms_per_registration": float(np.mean(ms)), "median_error_px": err, "inliers": [int(x) for x in res["inliers"]],
            "lap_bids": [int(x[5]) for x in st], "lap_augmentations": [int(x[2]) for x in st],
            "lap_dijkstra_steps": [int(x[3]) for x in st]}


def bench_supervised(torch, args, pair, with_cpu):
    """BASELINE config 3: keypoint-supervised mode (reference _dock_widget.py:707-717): affine from 10 keypoint pairs,
    then ICP on the full clouds, through the public numpy API."""
    import platymatch_b200 as pm
    from platymatch_b200.synthetic import make_keypoints
    mk, fk = make_keypoints(pair, 10, seed=0)
    for _ in range(3):
        res = pm.estimate_transform_supervised(pair["moving"], pair["fixed"], mk, fk, icp_iterations=ICP_ITERS)
    reps = 20
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        res = pm.estimate_transform_supervised(pair["moving"], pair["fixed"], mk, fk, icp_iterations=ICP_ITERS)
    ms = (time.perf_counter() - t0) * 1e3 / reps
    moved = res["transform"] @ np.vstack([pair["moving"], np.ones((1, pair["moving"].shape[1]))])
    err = float(np.median(np.linalg.norm(moved[:3] - pair["fixed"][:, pair["gt_fixed_index"]], axis=0)))
    out = {"workload": "%d x %d pair, 10 keypoint pairs (1 px click jitter), affine fit + %d ICP iterations through "
                       "estimate_transform_supervised(numpy...)" % (pair["moving"].shape[1], pair["fixed"].shape[1], ICP_ITERS),
           "ms_per_registration": ms, "registrations_per_s": 1e3 / ms, "median_error_px": err,
           "timing": "host clock around %d calls of the public API with HOST inputs (H2D + D2H inside)" % reps}
    if with_cpu:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        O.set_num_threads(len(os.sched_getaffinity(0)))
        t0 = time.perf_counter()
        O.estimate_transform_supervised(pair["moving"], pair["fixed"], mk, fk, icp_iterations=ICP_ITERS)
        out["cpu_baseline"] = {"value": 1.0 / (time.perf_counter() - t0), "unit": "registrations/s", "cores": O.num_threads(),
                               "kind": "port", "sample": "one complete supervised registration with the oracle port"}
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import platymatch_b200 as pm
    from platymatch_b200 import device as D, pipeline as P
    from platymatch_b200._lib import load
    from platymatch_b200.synthetic import make_pair

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":     # (its banner would go to stdout, next to the JSON line)
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = load()
    bid_rounds = args.bid_rounds if args.bid_rounds is not None else 2048
    kw = dict(ransac_trials=args.trials, icp_iterations=ICP_ITERS, max_bid_rounds=bid_rounds)

    # 4 specimen pairs cycled over the steps; every rank registers the same sequence of pairs, so the per-GPU
    # work is identical at every N and for every K, and the N-GPU value measures scaling, not pair difficulty
    # (the assignment stage of the third pair takes twice as long as that of the others)
    n_slots = 4
    pairs = [make_pair(args.n_fixed, seed=args.n_fixed + 97 * s) for s in range(n_slots)]
    n1, n2 = pairs[0]["moving"].shape[1], pairs[0]["fixed"].shape[1]
    dev_pairs = [(D.to_device_points(p["moving"]), D.to_device_points(p["fixed"])) for p in pairs]
    cost_buf = torch.empty((4, n1, (n2 + 3) // 4 * 4), dtype=torch.float32, device="cuda")

    def step_resident(s, hook=None):
        m, f = dev_pairs[s % n_slots]
        if hook is None:
            dm, df = P.describe_pair(m, f, 1, 4, transposed=True)
        else:
            dm = P.describe_cloud(m, 1, transposed=True)
            hook("describe_moving")
            df = P.describe_cloud(f, 4, transposed=True)
            hook("describe_fixed")
        return P.register_described(dm, df, seed=s, cost_out=cost_buf, stage_hook=hook, **kw)

    e2e_bytes = {}

    def step_e2e(s):
        # the call a user of the reference makes: numpy clouds (3 x N, host) in, numpy results out
        p = pairs[s % n_slots]
        res = pm.estimate_transform_unsupervised(p["moving"], p["fixed"], seed=s, **kw)
        if not e2e_bytes:
            e2e_bytes["h2d"] = (n1 + n2) * 3 * 8
            d2h = 0
            for k, v in res.items():
                if isinstance(v, np.ndarray):
                    d2h += v.nbytes
                elif k == "assignments":
                    d2h += sum(f.size * 4 for _, f in v)          # int32 on the wire (moving indices are implicit)
                elif k == "edge_ties":
                    d2h += 16
                elif k == "best":
                    d2h += 4
            e2e_bytes["d2h"] = d2h
        return res

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (ms, what the last step returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(steps):
            out = fn(s)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    for s in range(args.warmup):
        step_resident(s)
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = lib.pm_launch_count()
    ms, last = timed(step_resident, args.steps)
    launches = lib.pm_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, cost_buf, n1, n2)
    if args.lean:
        if rank == 0:
            print(json.dumps({"lean": True, "ms_per_step": ms / args.steps, "gpu_launches": int(launches)}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    for s in range(max(args.warmup, 3)):
        step_e2e(s)
    ms_e2e, _ = timed(step_e2e, args.steps)

    # ---- per-stage breakdown (CUDA events on the launching stream; stages serialised) ----
    marks = []

    def hook(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        marks.append((name, e))

    stage_ms = {}
    reps = max(2, min(args.steps, 8))
    step_resident(0, lambda name: None)      # untimed: the first batched (non-overlapped) pass pays one-time allocations
    torch.cuda.synchronize()
    lap_ms = []
    for s in range(reps):
        marks.clear()
        hook("start")
        res = step_resident(s, hook)
        torch.cuda.synchronize()
        for (n0, a), (n1_, b) in zip(marks[:-1], marks[1:]):
            stage_ms[n1_] = stage_ms.get(n1_, 0.0) + a.elapsed_time(b) / reps
            if n1_ == "lap":
                lap_ms.append(a.elapsed_time(b))
                if args.stages:
                    print("rep %d (pair slot %d): lap %.2f ms" % (s, s % n_slots, a.elapsed_time(b)), file=sys.stderr)
    lap_stats = res["lap_stats"].cpu().numpy().tolist()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    fp32_probe, fp32_nominal = fp32_peaks(torch, lib, D, local)
    bufs = [cost_buf[q] for q in range(4)]               # 4 x 230 MB outputs cycled: > L2
    roof = chi2_roofline(torch, D, P, pairs[0], bufs, fp32_probe, fp32_nominal, hbm_peak,
                         "shell cloud (the headline workload)")
    roof["traffic"] = CHI2_NCU_DRAM_BYTES if (n1, n2) == (7200, 8000) else None
    roof["traffic_source"] = ("ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch "
                              "(profiles/r2_chi2_kernel_shell.txt: 10.7 MB read + 176.2 MB written; the tail of the matrix is still in L2)")
    roof["dense"] = chi2_roofline(torch, D, P, make_pair(args.n_fixed, filled=True), bufs, fp32_probe, fp32_nominal, hbm_peak,
                                  "filled ellipsoid (late-stage embryo, SURVEY §8d): ~2x more bins populated per histogram")
    roof["dense"]["traffic"] = CHI2_NCU_DRAM_BYTES_DENSE if (n1, n2) == (7200, 8000) else None
    chi2_gpairs = roof["gpairs_per_s"]

    # ---- secondary: independent registrations overlapped on separate streams (one host thread each) ----
    pipelined = None
    if args.in_flight > 1:
        import threading
        nfl = args.in_flight
        bufs = [cost_buf] + [torch.empty_like(cost_buf) for _ in range(nfl - 1)]
        streams = [torch.cuda.Stream() for _ in range(nfl)]

        def worker(k, steps):
            torch.cuda.set_device(local)
            with torch.cuda.stream(streams[k]):
                for s_ in range(k, steps, nfl):
                    m, f = dev_pairs[s_ % n_slots]
                    dmk = P.describe_cloud(m, 1, transposed=True)
                    dfk = P.describe_cloud(f, 4, transposed=True)
                    P.register_described(dmk, dfk, seed=s_, cost_out=bufs[k], overlap_hypotheses=False, **kw)

        def run_all(steps):
            ts = [threading.Thread(target=worker, args=(k, steps)) for k in range(nfl)]
            for t_ in ts: t_.start()
            for t_ in ts: t_.join()

        run_all(2 * nfl)                                   # warm-up
        barrier()
        psteps = max(args.steps, 4 * nfl)                  # (every stream gets at least 4 registrations)
        t0 = time.perf_counter()
        run_all(psteps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        pipelined = {"value": world * psteps / dt, "unit": "registrations/s", "in_flight_per_gpu": nfl,
                     "registrations_per_gpu": psteps, "ms_per_registration": dt / psteps * 1e3,
                     "note": "independent registrations overlapped on %d CUDA streams per GPU (host clock, inputs "
                             "resident); the headline `value` registers one pair at a time" % nfl}
        del bufs

    # ---- BASELINE configs 4 and 5 at this N (collective: every rank takes part) ----
    rows = {}
    if not args.no_rows:
        torch.cuda.empty_cache()
        for name, fn in (("sharded_20k", bench_sharded_20k), ("allpairs_66", bench_allpairs),
                         ("allpairs_66_equal_sizes", lambda *a: bench_allpairs(*a, vary=0.0, runs=1))):
            try:
                rows[name] = fn(torch, dist, world, rank, args)
            except Exception as e:          # a secondary row must not take the headline down with it
                rows[name] = {"error": "%s: %s" % (type(e).__name__, e)}
                if world > 1:
                    raise

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total = world * args.steps
    value = total / (ms * 1e-3)
    e2e_val = total / (ms_e2e * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": "registrations/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 descriptors/duals/transforms, f32 cost matrix", "data": "synthetic",
        "config": workload_config(n1, n2, args.trials),
        "impl_config": {"lap_bid_rounds": bid_rounds, "parallelism": "pairs sharded, 1 rank/GPU",
                        "l2": "4 x %.0f MB cost matrices rewritten every step (> 126 MB L2); 4 input pairs cycled" %
                              (n1 * n2 * 4 / 1e6)},
        "e2e": {"value": e2e_val, "unit": "registrations/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": e2e_bytes.get("h2d"), "d2h_bytes_per_step": e2e_bytes.get("d2h"),
                "api": "platymatch_b200.estimate_transform_unsupervised(numpy 3xN, numpy 3xN) -> dict of numpy arrays: "
                       "host clouds staged through pinned memory, all results (transforms, inliers, 4 assignments, LAP "
                       "statistics, ICP residuals) copied back; one host synchronisation per registration"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "pipelined": pipelined,
        "cost_matrix_gpairs_per_s": chi2_gpairs * world,
        "roofline": roof,
        "stages_ms": stage_ms,
        "lap_ms_per_pair": {"values": lap_ms, "max_over_min": (max(lap_ms) / min(lap_ms)) if lap_ms else None},
        "lap_stats": {"bid_rounds": [s[0] for s in lap_stats], "rows_after_bidding": [s[1] for s in lap_stats],
                      "augmentations": [s[2] for s in lap_stats], "dijkstra_steps": [s[3] for s in lap_stats],
                      "bids": [s[5] for s in lap_stats], "refreshes": [s[6] for s in lap_stats],
                      "retries": [s[7] for s in lap_stats], "parked": [s[8] for s in lap_stats],
                      "refresh_cycles": [s[9] for s in lap_stats], "auction_cycles": [s[10] for s in lap_stats],
                      "bulk_bids": [s[11] for s in lap_stats], "sap_dense_relax": [s[12] for s in lap_stats]},
    }
    # single-GPU secondary measurements and the CPU baseline (rank 0 at N = 1 only)
    if not args.no_rows and world == 1:
        rows["label_centroids"] = bench_label_row(torch, D, hbm_peak, not args.no_cpu_baseline)
        try:
            rows["supervised_8k"] = bench_supervised(torch, args, pairs[0], not args.no_cpu_baseline)
        except Exception as e:
            rows["supervised_8k"] = {"error": "%s: %s" % (type(e).__name__, e)}
        if not args.no_square:
            try:
                rows["square_8k"] = bench_square(torch, args)
            except Exception as e:
                rows["square_8k"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if rows:
        line["rows"] = rows
    if not args.no_cpu_baseline and world == 1:
        arm = CpuArm(pairs[0], args.trials, ICP_ITERS)
        full = arm.full_run()
        cb = arm.baseline_dict(1.0 / full["seconds"])
        cb["sample"] = ("oracle (C/numpy port of the reference), %d threads: ONE complete unsampled registration of the "
                        "bench's first pair (6 descriptor sets, 4 hypotheses x {full chi2 matrix, full assignment, %d RANSAC "
                        "trials}, %d ICP iterations), measured, nothing extrapolated" % (arm.cores, args.trials, ICP_ITERS))
        line["cpu_baseline"] = cb
    if args.stages:
        print(json.dumps(stage_ms, indent=1), file=sys.stderr)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
