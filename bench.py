#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200: associations/sec of
scorePairwiseConsistency() + solve() (BASELINE.json), measured the way the reference's own
benchmark times the two calls (reference benchmarks/main.cpp:177-188).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

One "step" = one full pass of the hot path over one synthetic association problem:
score the m x m consistency graph, then run the graduated projected-gradient solver.
  value : m*K / device time, inputs (D1, D2, A, u0) already resident in HBM (clp_*_dev entry points)
  e2e   : the same through the host-pointer C-ABI calls (pinned host buffers in, Solution out),
          host<->device copies inside the timed region
  roofline : solver kernel (the dominant launch): passes over the matrix x algorithmic bytes of one pass of the sweep
             in use (compact copy: 6 B per kept entry + item descriptors, clp_sparse_info; dense sweeps: 4 m^2, or
             2 m^2 for the two-sided upper-triangle sweep) / its CUDA-event duration, against MEASURED_PEAKS.json's
             hbm_gbs; the dense-equivalent figure (4 m^2 per pass) is reported beside it
  cpu_baseline / --impl reference : the CPU oracle (Eigen-free restatement of the reference; the
             reference cannot be built offline -- no Eigen) on this box's host cores.
  --dump-outputs DIR : after the timed steps, the Solution of the last timed step (u, selected nodes, F, d_final;
             the same for the config 4 run) as DIR/<name>.npy in float64.  The inputs are seeded, so two builds run
             with the same arguments can be compared output for output.
Prints exactly ONE JSON line on rank 0.  Writes nothing into the source tree (it may be read-only).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the source tree

METRIC = "associations/sec (scorePairwiseConsistency+solve)"
UNIT = "associations/s"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference, all host threads it can use
# ------------------------------------------------------------------------------------------
def oracle_step(prob, nthreads):
    from oracle import clipper_oracle as orc
    cfg = prob["cfg"]
    o = orc.Oracle()
    t0 = time.perf_counter()
    if cfg["kind"] == "euclidean":
        o.score_euclidean(prob["D1"], prob["D2"], prob["A"], sigma=cfg["sigma"], epsilon=cfg["epsilon"], nthreads=nthreads)
    else:
        o.score_pointnormal(prob["D1"], prob["D2"], prob["A"], sigp=cfg["sigp"], epsp=cfg["epsp"], sign=cfg["sign"],
                            epsn=cfg["epsn"], nthreads=nthreads)
    t1 = time.perf_counter()
    s = o.solve(prob["u0"])
    t2 = time.perf_counter()
    return dict(t_score=t1 - t0, t_solve=t2 - t1, evals=int(s.n_evals), nodes=s.nodes.tolist(), score=float(s.score),
                nnz=o.nnz(0))


def workload_name(name, cfg):
    """the SAME string in both arms (the driver compares the two lines' config)"""
    if cfg["kind"] == "euclidean":
        return "%s: synthetic EuclideanDistance m=%d, %d%% outliers, sigma=%g eps=%g" % (
            name, cfg["m"], round(100 * cfg["rho"]), cfg["sigma"], cfg["epsilon"])
    return "%s: synthetic PointNormalDistance m=%d, %d%% outliers" % (name, cfg["m"], round(100 * cfg["rho"]))


def solution_arrays(prefix, sol, u, nodes):
    """what clp_solve_dev hands its caller, as float64 arrays (node indices are exact in float64)"""
    return {prefix + "u": np.asarray(u, dtype=np.float64), prefix + "nodes": nodes[: sol.n_nodes].astype(np.float64),
            prefix + "score": np.array([sol.score]), prefix + "d_final": np.array([sol.d_final])}


def dump_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """--impl reference: the reference's CPU path for the same metric/config, on the host cores.
    The literal reference needs Eigen3 (absent, no network) -> the Eigen-free oracle port is timed:
    scoring with OpenMP on all cores (reference default parallelize_=true, clipper.h:154),
    solver single-threaded (the reference's solver has no threading, clipper.cpp:172-323)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from clipper_b200 import datagen
    cores = cpu_cores()
    # ALWAYS the GPU arm's configuration (same m, same seeded inputs): a ratio across two problem sizes is void.
    # One full c2 step costs ~12 s on the GPU box's cores (scoring OpenMP 0.7 s + single-threaded solver 11.3 s),
    # i.e. K = 20 steps take about 4 minutes; only the untimed warm-up steps run on a small instance.
    prob = datagen.config_problem(args.workload, args.m)
    m_s = prob["cfg"]["m"]
    warm = datagen.config_problem(args.workload, min(2000, m_s))
    for _ in range(args.warmup):
        oracle_step(warm, cores)  # warm-up on a small instance (thread pool, page cache)
    ts = []
    t0 = time.perf_counter()
    info = None
    for _ in range(args.steps):
        info = oracle_step(prob, cores)
        ts.append(info["t_score"] + info["t_solve"])
    total = time.perf_counter() - t0
    value = m_s * args.steps / total
    sample = "full %s problem, m=%d, every step" % (args.workload, m_s)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, prob["cfg"]),
                   "cloud": datagen.cloud_source(),
                   "t_score_s": info["t_score"], "t_solve_s": info["t_solve"], "evals": info["evals"],
                   "F": info["score"], "n_nodes": len(info["nodes"])},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample + "; oracle restatement (Eigen/MKL unavailable offline): scoring OpenMP x%d, "
                                            "solver 1 thread like the reference; untimed warm-up on m=%d" % (cores, min(2000, m_s))},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from clipper_b200 import _capi, datagen
    import clipper_b200 as clipperpy

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs is implemented for one GPU")
        from clipper_b200 import distributed as cdist
        return cdist.run_bench(args, METRIC, UNIT)

    L = _capi.load()
    prob = datagen.config_problem(args.workload, args.m)
    cfg = prob["cfg"]; m = cfg["m"]
    assert cfg["kind"] == "euclidean"
    ip = clipperpy.invariants.EuclideanDistanceParams(); ip.sigma, ip.epsilon = cfg["sigma"], cfg["epsilon"]
    clip = clipperpy.CLIPPER(clipperpy.invariants.EuclideanDistance(ip), clipperpy.Params(), device=local_rank)
    h = clip.handle
    if os.environ.get("CLP_DENSE_MODE"):
        clip.set_dense_mode(int(os.environ["CLP_DENSE_MODE"]))
    if os.environ.get("CLP_CTAS_PER_SM"):
        _capi.check(h, L.clp_set_ctas_per_sm(h, int(os.environ["CLP_CTAS_PER_SM"])))
    # a real (non-default) stream shared by torch and the library: the legacy default stream has handle 0, which
    # clp_set_stream reads as "create your own" -- the CUDA events below must sit on the stream the kernels run on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    clip.set_stream(stream.cuda_stream)

    # ---- inputs resident in HBM
    D1 = torch.from_numpy(np.ascontiguousarray(prob["D1"].T)).to(dev)
    D2 = torch.from_numpy(np.ascontiguousarray(prob["D2"].T)).to(dev)
    A = torch.from_numpy(np.ascontiguousarray(prob["A"].T)).to(dev)
    u0 = torch.from_numpy(prob["u0"]).to(dev)
    u_out = torch.empty_like(u0)
    nodes = np.zeros(m, np.int32)
    sol = _capi.ClpSolution()
    n1, n2 = D1.shape[0], D2.shape[0]

    def step_dev():
        _capi.check(h, L.clp_score_euclidean_dev(h, D1.data_ptr(), 3, n1, D2.data_ptr(), n2, A.data_ptr(), m,
                                                 cfg["sigma"], cfg["epsilon"], 0.0))
        _capi.check(h, L.clp_solve_dev(h, u0.data_ptr(), C.byref(sol), u_out.data_ptr(),
                                       nodes.ctypes.data_as(C.POINTER(C.c_int32))))

    # ---- the same through the host-pointer API (pinned host buffers)
    hD1 = torch.from_numpy(np.ascontiguousarray(prob["D1"].T)).pin_memory()
    hD2 = torch.from_numpy(np.ascontiguousarray(prob["D2"].T)).pin_memory()
    hA = torch.from_numpy(np.ascontiguousarray(prob["A"].T)).pin_memory()
    hu0 = torch.from_numpy(prob["u0"]).pin_memory()
    hu = torch.empty(m, dtype=torch.float64).pin_memory()
    dp = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_double))
    ipt = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_int32))
    sol_h = _capi.ClpSolution()

    def step_host():
        _capi.check(h, L.clp_score_euclidean(h, dp(hD1), 3, n1, dp(hD2), n2, ipt(hA), m, cfg["sigma"], cfg["epsilon"], 0.0))
        _capi.check(h, L.clp_solve(h, dp(hu0), C.byref(sol_h), dp(hu), nodes.ctypes.data_as(C.POINTER(C.c_int32)), None))

    for _ in range(max(args.warmup, 3)):
        step_dev()
    torch.cuda.synchronize()

    # ---- timed region: K steps, CUDA events on the launching stream, clocks sampled meanwhile
    sampler = ClockSampler(local_rank); sampler.start()
    time.sleep(0.3)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms, n_matvec, evals, prof = [], [], [], []
    torch.cuda.synchronize()
    ev0.record(stream)
    for _ in range(args.steps):
        step_dev()
        kernel_ms.append(sol.kernel_ms); n_matvec.append(sol.n_matvec); evals.append(sol.n_evals)
        prof.append((sol.prof_matvec_ms, sol.prof_combine_ms, sol.prof_exchange_ms))
    ev1.record(stream)
    torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    value = m * args.steps / (dev_ms * 1e-3)
    nodes_dev = nodes[: sol.n_nodes].tolist(); F_dev = sol.score
    # copied now: the host-pointer steps below write into the same `nodes` buffer
    outputs = solution_arrays("", sol, u_out.cpu().numpy(), nodes) if args.dump_outputs else None

    # ---- e2e: host buffers in, Solution out, copies inside the timed region (wall clock)
    for _ in range(3):
        step_host()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    e2e_value = m * args.steps / e2e_s
    h2d = hD1.numel() * 8 + hD2.numel() * 8 + hA.numel() * 4 + m * 8
    d2h = m * 8 + 256 + 32 + 32  # u + result header + two status blocks
    assert nodes[: sol_h.n_nodes].tolist() == nodes_dev and sol_h.score == F_dev

    # ---- roofline of the dominant kernel (the persistent solver): algorithmic bytes = n_matvec * 4 m^2
    peak, peak_src = measured_peaks()
    esz = 4
    mode = clip.dense_mode()
    # algorithmic bytes of ONE dense pass: the full dense fp32 matrix (4 m^2) for the full-matrix sweeps, the
    # strict upper triangle only (2 m^2, SURVEY 8d) when every element is applied two-sidedly in-tile (mode 2)
    pass_bytes = (esz * m * m) if mode != 2 else (esz * m * (m - 1) // 2)
    nnz_kept = None
    if mode in (3, 6):  # compact copy: 6 B per kept entry + item descriptors (clp_sparse_info)
        nnz_kept, pass_bytes = clip.sparse_info()
    alg_bytes = float(np.mean(n_matvec)) * pass_bytes
    kms = float(np.mean(kernel_ms))
    achieved = alg_bytes / (kms * 1e-3) / 1e9
    # stand-alone Md.v pass (K2) for the ">= 40 % of HBM roofline on the mat-vec" target
    v = torch.rand(m, dtype=torch.float64, device=dev); y = torch.empty_like(v)
    ms_mv = C.c_double()
    _capi.check(h, L.clp_matvec_dev(h, v.data_ptr(), 1.0, y.data_ptr(), None, None, 5, C.byref(ms_mv)))
    _capi.check(h, L.clp_matvec_dev(h, v.data_ptr(), 1.0, y.data_ptr(), None, None, 50, C.byref(ms_mv)))
    mv_gbs = (pass_bytes + 16 * m) / (ms_mv.value * 1e-3) / 1e9

    # ---- the dense Md.v sweep of the same matrix (north_star: ">= 40 % of the HBM roofline on the Md.u mat-vec"):
    #      switch this handle to the full-matrix dense sweep, time it alone, switch back
    dense_ref = None
    if mode != 0:
        clip.set_dense_mode(0)
        _capi.check(h, L.clp_matvec_dev(h, v.data_ptr(), 1.0, y.data_ptr(), None, None, 5, C.byref(ms_mv0 := C.c_double())))
        _capi.check(h, L.clp_matvec_dev(h, v.data_ptr(), 1.0, y.data_ptr(), None, None, 50, C.byref(ms_mv0)))
        g0 = (esz * m * m + 16 * m) / (ms_mv0.value * 1e-3) / 1e9
        dense_ref = {"sweep": "segments, full dense fp32 matrix, 4 m^2 + 16 m bytes", "ms": ms_mv0.value, "GBps": g0,
                     "frac_of_measured_hbm_peak": g0 / peak}
        clip.set_dense_mode(int(os.environ.get("CLP_DENSE_MODE", "4")))

    # ---- CPU baseline on a bounded sample (rank 0, N=1): one full oracle step (~10-30 s)
    cpu = None
    if not args.no_cpu_baseline:
        cores = cpu_cores()
        info = oracle_step(prob, cores)
        cpu = {"value": m / (info["t_score"] + info["t_solve"]), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "1 full step of the same %s problem (m=%d): oracle restatement, scoring OpenMP x%d %.2f s, "
                         "solver single-threaded %.2f s, %d evaluations; Eigen/MKL reference unbuildable offline"
                         % (args.workload, m, cores, info["t_score"], info["t_solve"], info["evals"]),
               "t_score_s": info["t_score"], "t_solve_s": info["t_solve"],
               "same_inlier_set": sorted(info["nodes"]) == sorted(nodes_dev),
               "rel_dF": abs(info["score"] - F_dev) / abs(info["score"])}

    # ---- BASELINE config 4 (m = 80000) on this one GPU: the N = 1 anchor of the row-sharded scaling runs
    config4 = None
    if not args.no_config4 and args.workload == "c2" and args.m is None:
        config4 = run_config4(clipperpy, _capi, L, dev, stream, max(1, min(3, args.steps)), outputs)

    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if args.m is None:
            traffic = tj[args.workload][str(mode)]["dram_bytes_per_launch"]
    except Exception:
        traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64 (f32 affinity storage, fp64 vectors/accumulators/decisions)", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, cfg), "cloud": datagen.cloud_source(),
                   "l2": "inputs larger than L2 (dense M = %.2f GB vs 126 MB L2)" % (esz * m * m / 1e9),
                   "dense_sweep": {0: "segments, full matrix (4 m^2 B/pass)", 1: "stripes, full matrix (4 m^2 B/pass)",
                                   2: "stripes, upper triangle read once, two-sided in-tile update (2 m^2 B/pass)",
                                   3: "compact sliced-ELL copy, column segments: (fp32 value, 16-bit column offset) per kept entry, 6 B/entry/pass",
                                   6: "compact sliced-ELL copy, whole rows, trial vector resident in shared memory: (fp32 value, 16-bit column index) per kept entry, 6 B/entry/pass"}[mode],
                   "kept_entries": nnz_kept, "dense_equivalent_gbs": float(np.mean(n_matvec)) * esz * m * m / (kms * 1e-3) / 1e9,
                   "algorithmic_bytes_per_pass": pass_bytes,
                   "evals_per_solve": float(np.mean(evals)), "matvec_per_solve": float(np.mean(n_matvec)),
                   "solver_kernel_ms": kms,
                   "solver_phase_ms": dict(zip(("dense_passes", "combine", "exchange"), np.mean(prof, axis=0).tolist())),
                   "matvec_alone_gbs": mv_gbs, "matvec_alone_ms": ms_mv.value,
                   "matvec_alone_frac": mv_gbs / peak, "dense_matvec_alone": dense_ref, "F": F_dev, "n_nodes": len(nodes_dev)},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": 1e3 * e2e_s / args.steps},
        # kernels of this repository launched per step: gather_endpoints + score_tile + solver, plus the kernels that
        # build the compact copy in mode 3 (sort, item lengths, 2 x scan, fill, partition; + the counting pass when
        # the scoring kernel does not produce the counts itself) -- see profiles/r01g_launches_bench_c2.csv
        "gpu_launches": ((9 if FUSED_COUNT else 10) if mode in (3, 6) else 3) * args.steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                     "kernel": "%s (persistent; %d passes over the matrix per launch)"
                               % ("solver_resident_kernel<float>" if mode == 6 else "solver_kernel<float,%d>" % mode,
                                  int(round(np.mean(n_matvec)))), "peak_source": peak_src},
    }
    if cpu:
        line["cpu_baseline"] = cpu
    if config4:
        line["config4"] = config4
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))


def run_config4(clipperpy, _capi, L, dev, stream, steps, outputs=None):
    """m = 80000 (BASELINE config 4) unsharded: device-timed steps with inputs resident in HBM, same metric.
    The last step's Solution goes into `outputs` (names prefixed config4_) when a dict is passed."""
    import torch
    from clipper_b200 import datagen
    prob = datagen.config_problem("c4"); cfg = prob["cfg"]; m = cfg["m"]
    ip = clipperpy.invariants.EuclideanDistanceParams(); ip.sigma, ip.epsilon = cfg["sigma"], cfg["epsilon"]
    clip = clipperpy.CLIPPER(clipperpy.invariants.EuclideanDistance(ip), clipperpy.Params(), device=dev.index)
    h = clip.handle
    clip.set_stream(stream.cuda_stream)
    D1 = torch.from_numpy(np.ascontiguousarray(prob["D1"].T)).to(dev)
    D2 = torch.from_numpy(np.ascontiguousarray(prob["D2"].T)).to(dev)
    A = torch.from_numpy(np.ascontiguousarray(prob["A"].T)).to(dev)
    u0 = torch.from_numpy(prob["u0"]).to(dev)
    u_out = torch.empty_like(u0)
    nodes = np.zeros(m, np.int32)
    sol = _capi.ClpSolution()

    def step():
        _capi.check(h, L.clp_score_euclidean_dev(h, D1.data_ptr(), 3, D1.shape[0], D2.data_ptr(), D2.shape[0], A.data_ptr(), m,
                                                 cfg["sigma"], cfg["epsilon"], 0.0))
        _capi.check(h, L.clp_solve_dev(h, u0.data_ptr(), C.byref(sol), u_out.data_ptr(), nodes.ctypes.data_as(C.POINTER(C.c_int32))))

    step()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    kms = []
    for _ in range(steps):
        step(); kms.append(sol.kernel_ms)
    ev1.record(stream); torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    if outputs is not None:
        outputs.update(solution_arrays("config4_", sol, u_out.cpu().numpy(), nodes))
    mode = clip.dense_mode()
    kept, pass_bytes = clip.sparse_info() if mode in (3, 6) else (None, 4 * m * m)
    return {"workload": workload_name("c4", cfg), "value": m * steps / (ms * 1e-3), "unit": UNIT, "steps": steps,
            "ms_per_step": ms / steps, "solver_kernel_ms": float(np.mean(kms)), "evals": int(sol.n_evals), "sweep_mode": mode,
            "kept_entries": kept, "per_gpu_gbs": sol.n_matvec * pass_bytes / (float(np.mean(kms)) * 1e-3) / 1e9,
            "F": sol.score, "n_nodes": int(sol.n_nodes),
            "note": "unsharded anchor of the N-GPU runs; the CPU oracle at this size (about 5 min, single-threaded solver "
                    "like the reference) is timed by tests/test_gpu_fullsize.py::test_full_size_c4_vs_oracle"}


FUSED_COUNT = os.environ.get("CLP_FUSE_COUNT", "1") != "0" and os.environ.get("CLP_SCORE_FILTER", "1") != "0"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c4"])
    ap.add_argument("--m", type=int, default=None, help="override the workload's m (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the extra m=80000 (BASELINE config 4) measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's Solution arrays as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
