#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native ParticleSfM hot paths.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 2..5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one global bundle adjustment (HP2) of the BASELINE.json target workload
— F=200 frames x P=500k trajectories x 12 observations/track, synthetic (SURVEY.md §8d
"target config", seed 5) — from the perturbed start to the reference's termination
criteria (GlobalBundleAdjustment options, controllers/global_mapper.cc:41-71, pass B:
rotations + focal length refined).  `--config N` runs BASELINE.json's configs[N-1] stand-in
(SURVEY.md §8d) instead; the headline (no flag) stays the target config.

`value`  = observations / second of solve = M / t_step, problem resident in HBM
           (observations, structure uploaded once; the state is re-set every step).
`e2e`    = same metric through psfm_ba_solve() on pinned HOST buffers: H2D of
           observations/state, device-side flattening, pair structure, solve, D2H of the
           result — all inside the timed region.
The line also carries the HP1 number (trajectory optimiser, pts/s) under "traj_opt".

`--dump-outputs DIR` writes, after the timed steps, what each timed path returned in its last step:
ba_{qvec,tvec,xyz,cam_params,summary}.npy (resident arm, or the CPU arm with `--impl reference`),
ba_e2e_*.npy (end-to-end arm) and traj_{out,summary}.npy (HP1); summary = [initial cost, final cost,
iterations, termination].  The inputs are seeded, so the same arguments give the same inputs in every
run and two builds can be compared output for output.  HP1 outputs repeat bit for bit; the BA arrays
differ from run to run in the last bits (reduction order; about 1e-13 relative on one B200).

`--impl reference` times the CPU arm — the oracle's restatement of the reference's algorithm
(Ceres LM + SPARSE_SCHUR: block-sparse Schur complement, band Cholesky; OpenMP, the best thread
count of {8,16,32,64} <= min(ncpu, 64) — the reference's cap, sfm/main_sfm.py:144 — found by a
short calibration, see cpu_threads()) — on the SAME workload, full size; the sample
is only shrunk (and said so) when a full-size solve would not fit the driver's time budget.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs / SURVEY.md §8(d) stand-ins.  "target" is the headline.
CONFIGS = {
    "target": dict(name="target: 200 frames x 500k trajectories x 12 obs/track",
                   ba=dict(num_images=200, num_points=500_000, track_len=12, seed=5),
                   traj=dict(num=111_616, height=436, width=1024, seed=1, label="Sintel alley_1 shape 1024x436, sample_ratio 2")),
    "2": dict(name="config 2 stand-in: Sintel alley_1 shape, F=50, P=3e5, track length U{3..50} (dense reduced system)",
              ba=dict(num_images=50, num_points=300_000, track_len=12, track_len_range=(3, 50), seed=1),
              traj=dict(num=111_616, height=436, width=1024, seed=1, label="Sintel alley_1 shape 1024x436, sample_ratio 2")),
    "3": dict(name="config 3 stand-in: DAVIS shape, F=80, P=8e5, L=12, 30% of the observations dynamic and dropped",
              ba=dict(num_images=80, num_points=800_000, track_len=12, dynamic_fraction=0.3, seed=2),
              traj=dict(num=409_920, height=480, width=854, seed=2, label="DAVIS shape 854x480, sample_ratio 1")),
    "4": dict(name="config 4 stand-in: ScanNet shape, F=300, P=2e5, L=15, 1 px noise (4 GPUs in BASELINE.json)",
              ba=dict(num_images=300, num_points=200_000, track_len=15, noise_px=1.0, seed=3),
              traj=dict(num=76_800, height=480, width=640, seed=3, label="ScanNet shape 640x480, sample_ratio 2")),
    "5": dict(name="config 5: 500 frames x 2M trajectories x 12 obs/track (8 GPUs in BASELINE.json)",
              ba=dict(num_images=500, num_points=2_000_000, track_len=12, seed=4),
              traj=None),
}
REFERENCE_BUDGET_S = 240.0       # wall budget of one `--impl reference` run (all its steps)
DUMP_LIMIT_BYTES = 63_000_000    # --dump-outputs: array data of all files together (64 MB with the .npy headers)
SMALL_OUTPUT_BYTES = 1 << 20     # --dump-outputs: arrays up to this size are always written whole


def dump_outputs(path, arrays):
    """--dump-outputs: write each array as <path>/<name>.npy, float32 if it is float32, else float64.
    When the arrays exceed DUMP_LIMIT_BYTES together, every large one is cut to a fixed, seeded sample of
    its rows, the same rows for the same shape, so that two builds can be compared output for output."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    small = sum(a.nbytes for a in arrays.values() if a.nbytes <= SMALL_OUTPUT_BYTES)
    large = sum(a.nbytes for a in arrays.values() if a.nbytes > SMALL_OUTPUT_BYTES)
    keep = min(1.0, (DUMP_LIMIT_BYTES - small) / large) if large else 1.0
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if keep < 1.0 and a.nbytes > SMALL_OUTPUT_BYTES:
            rows = np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * keep), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(path, name + ".npy"), a)


def summary_output(s):
    """The scalars of a BASummary / TrajSummary a comparison of two builds should see."""
    return [s.initial_cost, s.final_cost, s.num_iterations, s.termination]


def ba_outputs(prefix, problem, summary):
    """What a caller of the bundle adjuster receives: the refined model and the solve's summary."""
    model = {name: np.array(getattr(problem, name)) for name in ("qvec", "tvec", "xyz", "cam_params")}
    model["summary"] = summary_output(summary)
    return {prefix + name: a for name, a in model.items()}


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def _lines(self):
        try:
            with open(self.f.name) as g:
                return g.read().splitlines()
        except OSError:
            return []

    def begin(self):
        """Call when the timed region starts: only later samples are reported (the sampler is
        started before the warm-up so that nvidia-smi's start-up is not inside the region)."""
        self.first = len(self._lines())

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        sm, mx, reasons = [], [], set()
        lines = self._lines()
        first = min(getattr(self, "first", 0), max(0, len(lines) - 1))
        for line in lines[first:]:
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        # samples taken under load = upper half of the observed clocks
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def global_pass_b_options(abi, lib, solver):
    o = abi.BAOptions()
    lib.psfm_ba_global_options(C.byref(o))
    o.refine_rotation = 1          # AdjustGlobalBundle(force_update_rotation=true), controllers/global_mapper.cc:219-224
    o.refine_focal_length = 1
    o.minimizer_progress_to_stdout = 0
    o.print_summary = 0
    o.linear_solver = solver
    return o


def workload_text(w, M):
    extra = ""
    if w.get("track_len_range"):
        extra = f", track length U{{{w['track_len_range'][0]}..{w['track_len_range'][1]}}}"
    if w.get("dynamic_fraction"):
        extra += f", {int(100 * w['dynamic_fraction'])}% of the observations dropped as dynamic"
    return (f"global BA pass B (rotation+translation+focal+points), F={w['num_images']} frames x P={w['num_points']} "
            f"trajectories x L={w['track_len']} obs/track{extra}, M={M} observations, seed {w['seed']}")


_CPU_THREADS = None


def cpu_threads(w=None):
    """Threads of the CPU arm.  The reference takes min(cpu_count, 64) (ctx_init, sfm/main_sfm.py:144); on a
    two-socket host the memory-bound sweeps stop scaling well before that (measured on the GPU box, 2 x 32
    cores: 16 threads 3.2 M obs/s, 64 threads 1.9, profiles/r02_cpu_threads.md), so the arm is given the
    BEST count of {8, 16, 32, 64} <= cpu_count, found with a short calibration solve on 1/10 of the
    workload — the CPU arm must not lose to its own thread count."""
    global _CPU_THREADS
    if _CPU_THREADS is not None or w is None:
        return _CPU_THREADS or 0
    import oracle
    from particlesfm_b200 import synthetic as syn, _abi
    cap = min(oracle.num_threads(), 64)
    cands = sorted({c for c in (8, 16, 32, 64) if c <= cap} | {min(cap, 8)})
    if len(cands) > 1:
        ws = dict(w); ws["num_points"] = max(2000, w["num_points"] // 10)
        prob, _ = syn.make_ba_problem(**ws)
        o = oracle.ba_global_options(refine_rotation=True, refine_focal_length=True)
        o.linear_solver = _abi.SOLVER_AUTO
        o.max_num_iterations = 3
        best = None
        for c in cands:
            oracle.ba_solve(prob.copy(), o, num_threads=c)
            t0 = time.perf_counter()
            oracle.ba_solve(prob.copy(), o, num_threads=c)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, c)
        _CPU_THREADS = best[1]
    else:
        _CPU_THREADS = cands[0]
    return _CPU_THREADS


def cpu_solve_once(w):
    """One solve of the CPU arm on workload w; returns (seconds, summary, problem size M, threads)."""
    import oracle
    from particlesfm_b200 import synthetic as syn, _abi
    nt = cpu_threads(w)
    prob, _ = syn.make_ba_problem(**w)
    o = oracle.ba_global_options(refine_rotation=True, refine_focal_length=True)
    o.linear_solver = _abi.SOLVER_AUTO
    t0 = time.perf_counter()
    s = oracle.ba_solve(prob, o, num_threads=nt)
    return time.perf_counter() - t0, s, prob.num_observations, nt


def run_reference(args, rank, cfg):
    """CPU arm: the oracle's restatement of the reference's path (LM + SPARSE_SCHUR for
    50 < F <= 1000, bundle_adjustment.cc:276-286) on the host's best thread count (cpu_threads()), same workload."""
    if rank != 0:
        return
    import oracle
    from particlesfm_b200 import synthetic as syn, _abi
    w = dict(cfg["ba"])
    if args.points:
        w["num_points"] = args.points
    full_points = w["num_points"]
    nt = cpu_threads(w)
    prob, _ = syn.make_ba_problem(**w)
    o = oracle.ba_global_options(refine_rotation=True, refine_focal_length=True)
    o.linear_solver = _abi.SOLVER_AUTO
    # first warm-up solve at full size decides whether the whole run fits the budget
    t0 = time.perf_counter()
    oracle.ba_solve(prob.copy(), o, num_threads=nt)
    t_full = time.perf_counter() - t0
    total_solves = args.warmup + args.steps
    shrunk = False
    if t_full * (total_solves - 1) > REFERENCE_BUDGET_S:
        frac = REFERENCE_BUDGET_S / (t_full * (total_solves - 1))
        w["num_points"] = max(1000, int(full_points * frac))
        prob, _ = syn.make_ba_problem(**w)
        shrunk = True
    M = prob.num_observations
    times, iters = [], 0
    warm_rest = args.warmup if shrunk else max(0, args.warmup - 1)      # the probe solve was the first warm-up
    for k in range(warm_rest + args.steps):
        p = prob.copy()
        t0 = time.perf_counter()
        s = oracle.ba_solve(p, o, num_threads=nt)
        dt = time.perf_counter() - t0
        if k >= warm_rest:
            times.append(dt)
            iters += s.num_iterations
    total = sum(times)
    val = M * len(times) / total
    cores = nt
    sample = ("the full workload" if not shrunk else
              f"P={w['num_points']} of {full_points} points (a full-size solve takes {t_full:.1f} s on this host: "
              f"{total_solves} of them exceed the {REFERENCE_BUDGET_S:.0f} s budget)")
    line = {
        "impl": "reference", "metric": "global_ba_observations_per_sec", "value": val, "unit": "observations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(w, M),
                   "options": "GlobalBundleAdjustment (SoftL1, f_tol 1e-6, g_tol 1, p_tol 1e-8, <=50 LM its)",
                   "linear_solver": "exact step: block-sparse Schur complement + band Cholesky (SPARSE_SCHUR restatement, "
                                    "reference rule for <= 1000 images)",
                   "implementation": "oracle/ba_oracle.c (C + OpenMP, -O3 AVX2/FMA): the reference's algorithm restated — "
                                     "Ceres/COLMAP cannot be built in this image (DESIGN.md §9)"},
        "lm_iterations_per_step": iters / len(times),
        "obs_iterations_per_sec": M * iters / total,
        "cpu_baseline": {"value": val, "unit": "observations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "observations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ba_outputs("ba_", p, s))
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="target", choices=sorted(CONFIGS), help="BASELINE.json configs[N-1] stand-in (SURVEY.md 8d)")
    ap.add_argument("--points", type=int, default=0, help="override the number of trajectories of the BA workload")
    ap.add_argument("--solver", default="auto", choices=["auto", "iterative", "exact"],
                    help="auto = the reference rule (bundle_adjustment.cc:276-286): exact Schur for <= 1000 images")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-traj", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what each timed path returned in its last step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, rank, cfg)
        return

    from particlesfm_b200 import _abi, _lib, ba, synthetic as syn, traj
    lib = _lib.lib()
    if lib.psfm_device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)")
    _lib.check(lib.psfm_set_device(local_rank), "psfm_set_device")
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        uid = (C.c_uint8 * _abi.NCCL_UNIQUE_ID_BYTES)()
        if rank == 0:
            _lib.check(lib.psfm_dist_get_unique_id(uid), "psfm_dist_get_unique_id")
        t = torch.tensor(list(uid), dtype=torch.uint8, device="cuda")
        dist.broadcast(t, 0)
        uid = (C.c_uint8 * _abi.NCCL_UNIQUE_ID_BYTES)(*t.cpu().tolist())
        _lib.check(lib.psfm_dist_init(uid, rank, world), "psfm_dist_init")

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    w = dict(cfg["ba"])
    if args.points:
        w["num_points"] = args.points
    full, truth = syn.make_ba_problem(**w)
    M_total = full.num_observations
    prob = full.shard(rank, world)
    solver_mode = {"auto": _abi.SOLVER_AUTO, "iterative": _abi.SOLVER_ITERATIVE_SCHUR,
                   "exact": _abi.SOLVER_EXACT_SCHUR}[args.solver]
    o = global_pass_b_options(_abi, lib, solver_mode)
    init = (full.qvec.copy(), full.tvec.copy(), full.xyz.copy(), full.cam_params.copy())

    # ---------------- device-resident arm ----------------
    S = ba.ResidentSolver(prob)
    summaries = []

    def step():
        S.set_state(*init)
        return S.run(o)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(args.warmup):
        step()
    barrier()
    if sampler:
        sampler.begin()
    launches0 = lib.psfm_launch_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        summaries.append(step())          # psfm_ba_run synchronises its stream before returning
    t_local = time.perf_counter() - t0
    barrier()
    t_total = max_over_ranks(t_local)
    launches = lib.psfm_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    ms_per_step = 1e3 * t_total / args.steps
    value = M_total * args.steps / t_total
    s_last = summaries[-1]
    iters = sum(s.num_iterations for s in summaries) / len(summaries)
    lin_its = sum(s.num_linear_iterations for s in summaries) / len(summaries)
    S.get_state()
    ate = syn.umeyama_ate(syn.camera_centres(prob.qvec, prob.tvec), truth["centres"])
    outputs = {}

    def collect_ba(prefix, problem, summary):
        if args.dump_outputs:
            if dist is not None:         # each rank refined only its shard of the points
                from particlesfm_b200 import distributed
                distributed.merge_points(problem, dist, world)
            outputs.update(ba_outputs(prefix, problem, summary))
    collect_ba("ba_", prob, s_last)

    # ---------------- rooflines (live CUDA events of this run) ----------------
    # HBM-bound kernels: algorithmic bytes per launch (DESIGN.md §3.4, factored-Jacobian formulation):
    #   Jacobian sweep      read xy 16 + idx 4, write D 24 + r 16; per point X 24 r, E'E/E'r 72 w
    #   implicit S*p        read D 24 + idx 4; per point X 24 + H~ 48
    # fp64-bound kernel: the fused Schur tile kernel does 108 fused multiply-adds per pair entry
    #   (M = Q_i Jp_j' 12, T = M Jc_j 24, Jc_i' T 72) on operands held in shared memory; its HBM traffic
    #   (D 24 + idx 4 per observation, 120 per point, 4 per pair entry) is reported beside it.
    peak, peak_src = read_peaks()
    dfma = C.c_double()
    dlat = C.c_double()
    _lib.check(lib.psfm_measure_dfma(C.byref(dfma), C.byref(dlat)), "psfm_measure_dfma")
    fp64_peak_tflops = 2e-12 * dfma.value
    M_local = prob.num_observations
    Lmean = M_total / max(1, int(np.unique(full.obs_point).size))
    P_local = int(np.unique(prob.obs_point).size)
    n_expl = sum(s.num_explicit_solves for s in summaries)
    fused = bool(s_last.explicit_fused)
    kernels = {
        "k_linearize (Jacobian sweep)": dict(bound="hbm", ms=sum(s.linearize_ms for s in summaries),
                                             n=sum(s.num_linearize for s in summaries), bytes=(20 + 40 + 96.0 / Lmean) * M_local),
        "k_schur_product (implicit S*p, one per PCG iteration)": dict(bound="hbm", ms=sum(s.schur_product_ms for s in summaries),
                                                                      n=sum(s.num_schur_products for s in summaries),
                                                                      bytes=(28 + 72.0 / Lmean) * M_local),
        "k_band_assemble + k_band_chol6 (reduced system: fold, all-reduce, assemble, block-6 factor, solve; two CTAs)": dict(
            bound="latency", ms=sum(s.cholesky_ms for s in summaries), n=n_expl, bytes=None),
    }
    if fused:
        kernels["k_schur_tile (W, W H~ in shared memory + pair products, fused)"] = dict(
            bound="fp64", ms=sum(s.schur_w_ms for s in summaries), n=n_expl,
            flops=2.0 * (108.0 * s_last.num_pair_entries + 60.0 * M_local),
            bytes=28.0 * M_local + 120.0 * P_local + 4.0 * s_last.num_pair_entries + 8.0 * s_last.num_pair_tasks)
    else:
        pairs_local = float(s_last.num_pair_entries)
        kernels["k_schur_w (W = Jc'Jp and W H~ per observation)"] = dict(bound="hbm", ms=sum(s.schur_w_ms for s in summaries), n=n_expl,
                                                                         bytes=(28 + 288 + 120.0 / Lmean) * M_local)
        kernels["k_schur_pairs (image-pair blocks of the Schur complement)"] = dict(bound="hbm", ms=sum(s.schur_pairs_ms for s in summaries), n=n_expl,
                                                                                    bytes=288.0 * M_local + 8.0 * pairs_local)

    # measured DRAM traffic per launch (ncu --set full capture of the headline workload at 1 GPU, this round's kernels)
    traffic = {}
    try:
        if world == 1 and args.config == "target" and not args.points:
            with open(os.path.join(ROOT, "profiles", "traffic_r02b.json")) as f:
                traffic = json.load(f)
    except (OSError, ValueError):
        traffic = {}

    def roof(name):
        k = kernels[name]
        if k["n"] == 0 or k["ms"] <= 0:
            return None
        avg = k["ms"] / k["n"]
        d = {"kernel": name, "bound": k["bound"], "avg_launch_ms": avg, "launches": k["n"], "share_of_step": k["ms"] / (1e3 * t_local),
             "traffic": traffic.get(name.split(" ")[0])}
        if k["bound"] == "fp64":
            d.update({"peak": fp64_peak_tflops, "unit": "TFLOP/s", "peak_source": "measured in this run (psfm_measure_dfma: chip-wide DFMA rate x 2)",
                      "algorithmic_flops_per_launch": k["flops"], "achieved": k["flops"] / (avg * 1e-3) / 1e12})
            d["frac"] = d["achieved"] / fp64_peak_tflops
            d["hbm"] = {"algorithmic_bytes_per_launch": k["bytes"], "achieved_gbs": k["bytes"] / (avg * 1e-3) / 1e9,
                        "frac_of_hbm_peak": k["bytes"] / (avg * 1e-3) / 1e9 / peak}
        elif k["bound"] == "hbm":
            d.update({"peak": peak, "unit": "GB/s", "peak_source": peak_src, "algorithmic_bytes_per_launch": k["bytes"],
                      "achieved": k["bytes"] / (avg * 1e-3) / 1e9})
            d["frac"] = d["achieved"] / peak
        else:
            d.update({"peak": None, "unit": None, "achieved": None, "frac": None,
                      "note": "a chain of F dependent 6 x 6 block pivots per side (two CTAs, top-down and bottom-up): bounded by the latency of one block step (shared-memory wavefronts of the rank-6 window update + the 6-pivot LDL' chain), not by bandwidth or flops"})
        return d
    ranked = sorted((n for n in kernels if kernels[n]["bound"] != "latency" and kernels[n]["n"]), key=lambda n: -kernels[n]["ms"])
    roofline = roof(ranked[0]) if ranked else None
    roofline_lin = roof("k_linearize (Jacobian sweep)")
    if roofline_lin:
        # SURVEY.md 8(d) defines the sweep's algorithmic bytes for the STORED-Jacobian formulation
        # (what Ceres does): 208 B/observation in pass B.  The factored formulation here moves 68.
        # Both are reported; `achieved`/`frac` above use the bytes this implementation really needs.
        b208 = 208.0 * M_local
        roofline_lin["survey_8d_stored_jacobian"] = {
            "bytes_per_observation": 208, "bytes_per_launch": b208,
            "achieved": b208 / (roofline_lin["avg_launch_ms"] * 1e-3) / 1e9,
            "frac": b208 / (roofline_lin["avg_launch_ms"] * 1e-3) / 1e9 / peak}
    roofline_all = [r for r in (roof(n) for n in kernels) if r]
    S.close()

    # ---------------- end to end through the C ABI on host buffers ----------------
    # The caller's buffers are PINNED host memory (torch.Tensor.pin_memory is only the allocator
    # here): the C ABI takes plain pointers and issues the host->device copies itself.
    import torch

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()

    # ONE set of pinned caller buffers, refilled (untimed) before every solve: nothing grows
    p = prob.copy()
    for name in ("qvec", "tvec", "xyz", "cam_params", "obs_image", "obs_point", "obs_xy", "image_camera"):
        setattr(p, name, pin(getattr(p, name)))
    e2e_times = []
    for k in range(0 if args.no_e2e else 1 + args.steps):
        p.qvec[:], p.tvec[:], p.xyz[:], p.cam_params[:] = init
        barrier()
        t0 = time.perf_counter()
        s_e2e = ba.solve_problem(p, o)
        dt = max_over_ranks(time.perf_counter() - t0)
        if k >= 1:
            e2e_times.append(dt)
    if e2e_times:
        collect_ba("ba_e2e_", p, s_e2e)
    e2e_val = M_total * len(e2e_times) / sum(e2e_times) if e2e_times else None
    state_bytes = 8 * (full.qvec.size + full.tvec.size + full.cam_params.size) + 8 * 3 * np.unique(prob.obs_point).size
    h2d = prob.obs_xy.nbytes + prob.obs_image.nbytes + prob.obs_point.nbytes + 2 * prob.num_observations + 4 * prob.num_observations + state_bytes
    d2h = state_bytes

    line = {
        "metric": "global_ba_observations_per_sec", "value": value, "unit": "observations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(w, M_total), "baseline_config": cfg["name"],
                   "options": "GlobalBundleAdjustment (SoftL1, f_tol 1e-6, g_tol 1, p_tol 1e-8, <=50 LM its)",
                   "linear_solver": {2: "PCG on the reduced camera system, Schur-Jacobi, eta=0.1, <=100 its (Ceres ITERATIVE_SCHUR semantics)",
                                     1: "exact step: explicit Schur complement + band Cholesky on the device (reference rule for <= 1000 images)"}
                   [s_last.linear_solver_used],
                   "parallelism": f"points sharded over {world} GPU(s); NCCL all-reduce of the camera-side accumulators / reduced system",
                   "l2": "per-step working set (observations, linearisation, pair entries: ~0.7 GB) is larger than the 126 MB L2; no flush needed"},
        "lm_iterations_per_step": iters, "pcg_iterations_per_step": lin_its,
        "obs_iterations_per_sec": M_total * sum(s.num_iterations for s in summaries) / t_total,
        "device_ms_per_step": sum(s.device_ms for s in summaries) / len(summaries),
        "final_cost": s_last.final_cost, "initial_cost": s_last.initial_cost, "termination": s_last.termination,
        "ate_vs_truth": ate, "pair_entries": int(s_last.num_pair_entries), "pair_units": int(s_last.num_pair_tasks),
        "e2e": {"value": e2e_val, "unit": "observations/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": 1e3 * sum(e2e_times) / len(e2e_times) if e2e_times else None},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "fp64_roof": {"dfma_per_s": dfma.value, "tflops": fp64_peak_tflops, "dependent_dfma_latency_cycles": dlat.value,
                      "how": "psfm_measure_dfma: 8 independent DFMA chains per thread, 8 CTAs x 256 threads per SM, best of 4"},
        "roofline": roofline, "roofline_linearize": roofline_lin, "roofline_all_kernels": roofline_all,
    }

    # ---------------- HP1: trajectory optimiser, pts/s ----------------
    # HP1 does not shard (one Ceres problem = one trust region per frame pair; SURVEY.md 8(e)): "replicas only".
    # Every rank optimises ITS OWN frame pair (same shape, its own seed) on its own GPU, no collective on the data
    # path; the aggregate is (ranks x trajectories) / max over ranks of the mean call time — weak scaling.
    TR = cfg["traj"]
    if not args.no_traj and TR is not None:
        uv12, r1, r2, sc, f12 = syn.make_traj_inputs(TR["num"], TR["height"], TR["width"], seed=TR["seed"] + 1000 * rank)
        n = uv12.shape[0]
        ts, dev_ms = [], []
        for k in range(args.warmup + args.steps):
            if k == args.warmup:
                barrier()
            t0 = time.perf_counter()
            out, ssum = traj.optimize_location(uv12, r1, r2, sc, f12, n, TR["width"], TR["height"], return_summary=True)
            if k >= args.warmup:
                ts.append(time.perf_counter() - t0)
                dev_ms.append(ssum.solve_ms)
        t_call = max_over_ranks(statistics.mean(ts))
        t_dev = max_over_ranks(statistics.mean(dev_ms) * 1e-3)
        traj_bytes = 104.0 * n + 8.0 * TR["height"] * TR["width"]
        line["traj_opt"] = {"metric": "traj_opt_points_per_sec", "value_e2e": world * n / t_call,
                            "value_device": world * n / t_dev, "unit": "trajectories/s", "n": n, "replicas": world,
                            "scaling": "weak (independent replicas, one frame pair per GPU; no collective)",
                            "iterations": ssum.num_iterations, "workload": TR["label"],
                            "roofline": {"bound": "hbm (latency-bound by design)", "achieved": traj_bytes / t_dev / 1e9,
                                         "peak": peak, "unit": "GB/s", "frac": traj_bytes / t_dev / 1e9 / peak}}
        outputs.update(traj_out=out, traj_summary=summary_output(ssum))

    # ---------------- CPU baseline beside it (rank 0, N = 1 only): ONE full-size solve ----------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        dt, sc_, Mc, cores = cpu_solve_once(w)
        line["cpu_baseline"] = {"value": Mc / dt, "unit": "observations/s", "cores": cores,
                                "kind": "port", "lm_iterations": sc_.num_iterations,
                                "sample": f"the full workload (M={Mc}), one solve to the same termination ({dt:.1f} s): oracle restatement of "
                                          "LM + SPARSE_SCHUR (block-sparse Schur complement, band Cholesky), OpenMP"}
        if not args.no_traj and TR is not None:
            t0 = time.perf_counter()
            _, so = oracle.traj_optimize(uv12, r1, r2, sc, f12, num_threads=8)
            line["traj_opt"]["cpu_baseline"] = {"value": n / (time.perf_counter() - t0), "unit": "trajectories/s", "cores": 8,
                                                "kind": "port", "sample": "same call, 8 threads (trajectory_optimize.cpp:79)"}
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if dist is not None:
        lib.psfm_dist_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
