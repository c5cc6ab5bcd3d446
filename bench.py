#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

metric   V-cycle GDOF/s to a 1e-8 relative residual: N^2 / time(phi0 = 0 -> ||r|| < 1e-8 ||r0||)
workload 2-D Poisson, N = 16385 (268M DOF), V(2,2) weighted Jacobi omega = 2/3, fp64, RHS A
         (f = 2 pi^2 sin(pi x) sin(pi y), synthetic), reference-parity prolongation => 39 cycles.
step     one complete solve (reset phi to 0, cycle until converged, residual norm every cycle).

  python bench.py [--gpus N] [--steps K] [--warmup W]          our CUDA path
  python bench.py ... --dump-outputs bench_outputs             also write the last timed solve's results there (.npy)
  python bench.py --impl reference ...                         the reference's CPU path (oracle/_ref)

`value` is measured with f resident in HBM; `e2e` goes through the C ABI with pinned HOST buffers
(H2D of f and phi0, the solve, D2H of phi inside the timed region).  `roofline` is the dominant kernel
(the fused level-0 pass) timed alone with CUDA events on the solver stream against the measured HBM
copy peak.  Only the `cpu_baseline` / `--impl reference` legs touch oracle/ (as the CPU baseline).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "V-cycle GDOF/s to 1e-8 residual"
UNIT = "GDOF/s"
OMEGA = 2.0 / 3.0
REL_TOL = 1e-8
BYTES_PER_DOF_CYCLE = 69.3   # SURVEY.md 8(d): 52 B per level-point * 1.3334 (fused two-pass minimum)
CROSS_BYTES_PER_POINT = 28.0  # cross-cycle pass: read xb, f (16) + e (2), write xb' (8) + coarse f (2)
BYTES_PER_POINT_PASS = 26.0  # one fused pass: read x, read f, write x', + coarse array traffic (2 B)
BYTES_PER_DOF_W2 = 104.0     # SURVEY.md 8(d): W-cycle, gamma = 2: 52 / (1 - 2/4)
BYTES_PER_DOF_FMG = 125.0    # SURVEY.md 8(d): one full-multigrid pass ~ 1.333 * (69.3 + 18 + 24/4)


def goldens():
    """Residual histories of the reference's CPU multigrid (mg_cpu_exec semantics) at the BASELINE sizes:
    tests/golden/golden.json["survey"] (SURVEY.md 8c, N = 16385) and tests/golden/golden_large.json
    (tests/golden/make_golden_large.py over oracle/_ref, N = 4097 and the F-cycle).  Committed fixtures: nothing
    under oracle/ or /root/reference is touched at run time."""
    g = {}
    try:
        with open(os.path.join(ROOT, "tests", "golden", "golden.json")) as fh:
            sv = json.load(fh)["survey"]
        g["V_n16385"] = sv["V_n16385"]
        g["V_n16385_full"] = sv["V_n16385_full_prolong"]
        g["W2_n16385"] = sv["W_alpha2_n16385"]
    except Exception:
        pass
    try:
        with open(os.path.join(ROOT, "tests", "golden", "golden_large.json")) as fh:
            lg = json.load(fh)
        g["V_n4097"] = lg["V_n4097"]["history"][1:]
        g["W2_n4097"] = lg["W_alpha2_n4097"]["history"][1:]
        g["F_n4097"] = lg["F_n4097"]["norms"]
        if "F_n16385" in lg:
            g["F_n16385"] = lg["F_n16385"]["norms"]
    except Exception:
        pass
    return g


def history_check(hist_after_cycles, golden):
    """Parity fields of a bench leg: our per-cycle norms (after cycle 1, 2, ...) against the reference's.  The
    benchmarked configuration sums the norm with the parallel TREE order (pmg_norm_mode), the reference left to
    right: expected deviation <= 1e-10 up to N = 4097 and <= 2e-9 at N = 16385 (the reference's own summation
    drift, DESIGN.md section 2); the cycle count must be identical."""
    if golden is None:
        return {"golden": "missing", "cycles_match": None, "history_max_rel_dev": None}
    ours = [float(v) for v in hist_after_cycles]
    k = min(len(ours), len(golden))
    dev = max(abs(a - b) / abs(b) for a, b in zip(ours[:k], golden[:k])) if k else None
    return {"cycles_match": len(ours) == len(golden), "cycles": len(ours), "golden_cycles": len(golden),
            "history_max_rel_dev": dev}


def config_legs(make_solver, peak, world, reduce_max=None, skip=()):
    """The other BASELINE.json configs as short legs after the headline (extra keys of the JSON line):
      W_gamma2_n16385 / F_n16385   configs[3]: W-cycle and the F-cycle (full multigrid pass) at N = 16385
      V_n4097                      configs[1]: N = 4097 V(2,2) to 1e-8
      V_n32769                     configs[4]: the 1.07 G DOF weak-scaling point, fixed 8 cycles (1e-8 is below
                                   the fp64 rounding floor of the un-scaled residual at this size, DESIGN section 7)
    Each reports cycles, device ms per cycle (max over ranks), GDOF*cycle/s and the fraction of ITS OWN roofline
    (bytes per DOF per cycle from SURVEY 8d times the aggregate measured HBM peak), plus the history parity
    fields where a golden exists.  make_solver(n, **cfg) -> solver on this rank's slab."""
    import pmg_b200 as pmg
    gold = goldens()
    rmax = reduce_max or (lambda v: v)
    legs = {}

    def frac(bytes_per_dof, n, cycles, ms):
        gbs = bytes_per_dof * n * n * cycles / (ms * 1e-3) / 1e9
        return {"effective_gbs": gbs, "bytes_per_dof_cycle": bytes_per_dof, "frac_of_aggregate_peak": gbs / (peak * world)}

    def solve_leg(name, n, kind, gamma, bpd, golden, rel_tol=REL_TOL, max_cycles=100, reps=2):
        try:
            s = make_solver(n, gamma=gamma)
            s.set_rhs_sine()
            best, k, hist = None, 0, None
            for it in range(reps + 1):
                s.zero_guess()
                k, hist = s.solve(kind, rel_tol=rel_tol, max_cycles=max_cycles)
                ms = rmax(s.last_ms)
                if it > 0:
                    best = ms if best is None else min(best, ms)
            s.close()
            leg = {"n": n, "cycles": k, "ms_per_solve": best, "ms_per_cycle": best / max(k, 1),
                   "gdof_per_s_to_tol": (n * n / (best * 1e-3) / 1e9) if rel_tol > 0 else None,
                   "gdof_cycle_per_s": n * n * k / (best * 1e-3) / 1e9,
                   "final_rel_residual": float(hist[-1] / hist[0])}
            leg.update(frac(bpd, n, k, best))
            if golden is not None or rel_tol > 0:
                leg.update(history_check(hist[1:], golden))
            legs[name] = leg
        except Exception as e:  # noqa: BLE001 -- a failing leg must not lose the headline line
            legs[name] = {"error": repr(e)[:300]}

    if "W" not in skip:
        solve_leg("W_gamma2_n16385", 16385, pmg.W, 2, BYTES_PER_DOF_W2, gold.get("W2_n16385"))
    if "F" not in skip:
        try:
            n = 16385
            s = make_solver(n, gamma=1)
            s.set_rhs_sine()
            best, norm = None, None
            for it in range(3):
                s.zero_guess()
                norm = s.cycle(pmg.F)
                ms = rmax(s.last_ms)
                if it > 0:
                    best = ms if best is None else min(best, ms)
            s.close()
            leg = {"n": n, "passes": 1, "ms_per_pass": best, "gdof_per_s": n * n / (best * 1e-3) / 1e9,
                   "residual_norm_after_pass": norm}
            leg.update(frac(BYTES_PER_DOF_FMG, n, 1, best))
            gf = gold.get("F_n16385")
            leg["golden_norm"] = gf[0] if gf else None
            leg["norm_rel_dev"] = abs(norm - gf[0]) / gf[0] if gf else None
            legs["F_n16385"] = leg
        except Exception as e:  # noqa: BLE001
            legs["F_n16385"] = {"error": repr(e)[:300]}
    if "4097" not in skip:
        solve_leg("V_n4097", 4097, pmg.V, 1, BYTES_PER_DOF_CYCLE, gold.get("V_n4097"), reps=3)
    if "32769" not in skip:
        solve_leg("V_n32769", 32769, pmg.V, 1, BYTES_PER_DOF_CYCLE, None, rel_tol=0.0, max_cycles=8, reps=1)
    return legs


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_prefix, n):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` captures (profiles/r1_ncu_full_fused_passes_n16385.json: the two level-0 passes;
    profiles/r2_ncu_full_k_cross_wide_n16385.json: the cross-cycle pass in its default shape, strips of 128 columns), N = 16385."""
    if n != 16385:
        return None
    try:
        recs = []
        for name in ("r1_ncu_full_fused_passes_n16385.json", "r2_ncu_full_k_cross_wide_n16385.json"):
            path = os.path.join(ROOT, "profiles", name)
            if os.path.exists(path):
                with open(path) as fh:
                    recs += json.load(fh)
        unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
        tot = []
        for r in recs:
            if r["kernel"].startswith(kernel_prefix):
                v = 0.0
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    num, u = r[key].split()
                    v += float(num) * unit[u]
                tot.append(v)
        return sum(tot) / len(tot) if tot else None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 9 and r[5 + k].lower() == "active" for r in self.rows)]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "power_w_max": max(pw) if pw else None}


def pinned(pmg, shape):
    """numpy view over pinned host memory obtained through the C ABI."""
    nbytes = int(np.prod(shape)) * 8
    p = ctypes.c_void_p()
    pmg.check(pmg.lib().pmg_host_alloc_pinned(ctypes.byref(p), nbytes))
    buf = (ctypes.c_double * (nbytes // 8)).from_address(p.value)
    return np.frombuffer(buf, dtype=np.float64).reshape(shape), p


DUMP_SAMPLE_POINTS = 1 << 22  # 32 MB of float64: the solution is 2.1 GB at N = 16385


def dump_outputs(out_dir, phi, hist):
    """--dump-outputs: what the last timed solve returned, as float64 .npy files.
      residual_history.npy   ||r|| before cycle 1 and after every cycle (its length is the cycle count + 1)
      solution.npy           the whole N x N solution, when it has at most DUMP_SAMPLE_POINTS points; otherwise
      solution_sample.npy    the solution at DUMP_SAMPLE_POINTS grid points drawn once from a fixed seed, in
                             row-major order -- the same points in every run with the same --n"""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "residual_history.npy"), np.asarray(hist, dtype=np.float64))
    if phi.size <= DUMP_SAMPLE_POINTS:
        np.save(os.path.join(out_dir, "solution.npy"), phi)
        return
    idx = np.sort(np.random.default_rng(0).choice(phi.size, DUMP_SAMPLE_POINTS, replace=False))
    np.save(os.path.join(out_dir, "solution_sample.npy"), phi.reshape(-1)[idx])


def sine_rhs(n, out):
    """DynamicGridUtils::compute_rhs with a = p = q = 1, via its separable form (same rounding order:
    (factor * sin(pi x)) * sin(pi y))."""
    h = 1.0 / (n - 1)
    sx = np.sin(1.0 * np.pi * (np.arange(n) * h) / 1.0)
    factor = (np.pi * np.pi / 1.0) * 2.0
    np.multiply((factor * sx)[None, :], sx[:, None], out=out)


# ------------------------------------------------------------------------------------------------------
def cpu_reference_sample(n_sample, cycles, n_target, cycles_target):
    """Time `cycles` V(2,2) cycles of the reference CPU path at n_sample and scale by DOF*cycles to the
    target workload.  Returns (GDOF/s to solution at n_target, seconds measured, kind)."""
    import cpu_checkers as cc
    lib = cc.load("ref")
    kind = "reference"
    if lib is None:
        lib, kind = cc.load("orc"), "port"
    f = lib.rhs(n_sample)
    phi = np.zeros((n_sample, n_sample))
    t0 = time.perf_counter()
    for _ in range(cycles):
        lib.cycle(phi, f, kind=cc.V, omega=OMEGA, eps=0.0, alpha=1, v1=1, v2=1)
    dt = time.perf_counter() - t0
    dof_cycles_per_s = n_sample * n_sample * cycles / dt
    t_target = n_target * n_target * cycles_target / dof_cycles_per_s
    return n_target * n_target / t_target / 1e9, dt, kind


def reference_cuda_build(sizes=((4097, 3), (16385, 2))):
    """The reference's own CUDA multigrid (3_part_parallel, unmodified, compiled for sm_100a into
    oracle/_ref/ref_gpu_exec) timed on this GPU, ParallelTestRunner::run_v_cycle protocol, data prefetched.
    Time per V-cycle only: it has no convergence test, no omega, a racy in-place smoother, and leaks ~16 N^2
    bytes of managed memory per cycle (hence the small cycle counts)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_gpu_exec")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/ref_gpu_exec not built"}
    out = {}
    for n, cycles in sizes:
        try:
            p = subprocess.run([exe, str(n), str(cycles), "1"], capture_output=True, text=True, timeout=180)
            rec = json.loads(p.stdout.strip().splitlines()[-1])
            out[str(n)] = {"cycle_ms": rec["cycle_ms"], "best_cycle_ms": min(rec["cycle_ms"]),
                           "gdof_cycle_per_s": n * n / (min(rec["cycle_ms"]) * 1e-3) / 1e9}
        except Exception as e:  # noqa: BLE001
            out[str(n)] = {"error": repr(e)[:200]}
    return out


def cpu_same_config_n4097():
    """BASELINE config 2 measured for real on the host: the reference's CPU multigrid from phi0 = 0 to 1e-8 at
    N = 4097 (36 cycles, ~1 min on one core).  bench.py's own arm reports the same solve on the GPU (leg V_n4097)."""
    import cpu_checkers as cc
    lib = cc.load("ref")
    kind = "reference"
    if lib is None:
        lib, kind = cc.load("orc"), "port"
    n = 4097
    f = lib.rhs(n)
    phi = np.zeros((n, n))
    t0 = time.perf_counter()
    k, hist = lib.solve(phi, f, kind=cc.V, omega=OMEGA, eps=0.0, alpha=1, v1=1, v2=1, rel_tol=REL_TOL, max_cycles=100)
    dt = time.perf_counter() - t0
    return {"n": n, "cycles": int(k), "seconds": dt, "gdof_per_s_to_tol": n * n / dt / 1e9, "kind": kind, "cores": 1,
            "final_rel_residual": float(hist[-1] / hist[0])}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (oracle/_ref =
    the unmodified reference headers compiled here).  The named workload (39 cycles at N = 16385) takes the
    reference ~20 min and 13 GB, so each STEP is a bounded sample -- one V(2,2) cycle at N = 4097 -- and `value`
    is that sample scaled by DOF*cycles to the named workload; `ms_per_step` is the time the sample really took
    and `config.workload` says so.  In addition the line carries `measured_same_config`: BASELINE config 2
    (N = 4097 to 1e-8) solved for real, once, which pairs with our arm's `legs.V_n4097`.  The reference is
    single-threaded (no OpenMP / threads anywhere in it): cores = 1."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n_s, cyc_s = 4097, 1
    for _ in range(min(args.warmup, 2)):
        cpu_reference_sample(n_s, cyc_s, args.n, args.cycles_expected)
    vals, secs, kind = [], 0.0, "reference"
    for _ in range(args.steps):
        v, dt, kind = cpu_reference_sample(n_s, cyc_s, args.n, args.cycles_expected)
        vals.append(v)
        secs += dt
    value = len(vals) / sum(1.0 / v for v in vals)  # total work / total time
    same = None if args.no_same_config else cpu_same_config_n4097()
    sample = ("%d V(2,2) cycle(s) at N=%d per step (%.2f s each, 1 core), scaled by DOF*cycles to %d cycles at N=%d"
              % (cyc_s, n_s, secs / max(args.steps, 1), args.cycles_expected, args.n))
    cfg = workload_config(args, 1)
    cfg["workload"] = ("SAMPLE of the named workload: " + sample + " -- the full N=%d solve is NOT run on the CPU "
                       "(~20 min, 13 GB); see measured_same_config for a solve measured end to end" % args.n)
    cfg["sampled"] = True
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(args.steps, 1),
            "ms_per_solve_extrapolated": 1e3 * args.n * args.n / (value * 1e9),
            "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample,
                             "host_cores_available": os.cpu_count(), "measured_seconds": secs},
            "measured_same_config": same,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def workload_config(args, n_gpus):
    return {"workload": "2D Poisson N=%d (%.1fM DOF) V(2,2) weighted-Jacobi omega=2/3 fp64 to rel residual 1e-8, "
                        "RHS 2pi^2 sin(pi x)sin(pi y), phi0=0" % (args.n, args.n * args.n / 1e6),
            "n": args.n, "cycle": "V(2,2)", "omega": OMEGA, "rel_tol": REL_TOL,
            "prolongation": args.prolong, "engine": "fused", "l2": "inputs_exceed_l2 (2.1 GB per array)",
            "norm_mode": "tree (pmg_norm_mode; the reference sums left to right -- see history_max_rel_dev)",
            "parallelism": "1 GPU" if n_gpus == 1 else "row slabs x%d" % n_gpus}


def e2e_measure(pmg, s, n, ny, args, fill_f, max_cycles, fence=None, reduce_max=None):
    """The same solve measured end to end through the C ABI with pinned HOST buffers: every step copies its right-hand
    side host -> device and its solution device -> host inside the timed region (phi0 = 0 is pmg_set_guess(NULL): no
    zeros cross PCIe).  Two figures:
      value / ms_per_step   a stream of problems with the overlapped transfers of include/pmg.h (pmg_stage_rhs /
                            pmg_commit_rhs / pmg_fetch_solution_begin / _wait): the copies of step k+1 and k-1 run on
                            their own streams beside the solve of step k -- every step still moves all its bytes;
      serial                one problem at a time: H2D, solve, D2H strictly one after the other (latency of a single
                            solve including its copies; round 1 reported only this, with 2.1 GB of zeros uploaded too).
    ny: rows of this rank's slab (n on one GPU)."""
    fence = fence or (lambda: pmg.check(pmg.lib().pmg_device_synchronize()))
    rmax = reduce_max or (lambda v: v)
    f_host, pf = pinned(pmg, (ny, n))
    out_host, po = pinned(pmg, (ny, n))
    fill_f(f_host)
    e_steps = max(2, min(args.steps, 8))

    def serial_step():
        s.set_rhs(f_host)
        s.set_guess(None)
        kk, _ = s.solve(pmg.V, rel_tol=REL_TOL, max_cycles=max_cycles)
        s.get_solution(out_host)
        return kk

    serial_step()
    fence()
    t0 = time.perf_counter()
    for _ in range(e_steps):
        ke = serial_step()
    fence()
    serial_wall = rmax((time.perf_counter() - t0) / e_steps)

    def pipelined(steps):
        s.stage_rhs(f_host)
        kk = 0
        for k in range(steps):
            s.commit_rhs()
            if k + 1 < steps:
                s.stage_rhs(f_host)       # H2D of step k+1 beside the solve of step k
            s.set_guess(None)
            kk, _ = s.solve(pmg.V, rel_tol=REL_TOL, max_cycles=max_cycles)
            s.fetch_solution_wait()       # D2H of step k-1 (long done) before its snapshot is re-used
            s.fetch_solution_begin(out_host)
        s.fetch_solution_wait()
        return kk

    pipelined(2)
    fence()
    t0 = time.perf_counter()
    ke = pipelined(e_steps)
    fence()
    pipe_wall = rmax((time.perf_counter() - t0) / e_steps)
    out_ok = bool(np.isfinite(out_host[ny // 2, n // 2]) and out_host[ny // 2, n // 2] != 0.0)
    for p in (pf, po):
        pmg.lib().pmg_host_free_pinned(p)
    return {"value": n * n / pipe_wall / 1e9, "unit": UNIT, "h2d_bytes_per_step": n * n * 8,
            "d2h_bytes_per_step": n * n * 8 + (ke + 1) * 8, "ms_per_step": 1e3 * pipe_wall, "cycles": ke,
            "mode": "overlapped transfers (pmg_stage_rhs / pmg_fetch_solution_begin), %d problems back to back" % e_steps,
            "serial": {"value": n * n / serial_wall / 1e9, "ms_per_step": 1e3 * serial_wall,
                       "what": "H2D f, solve, D2H phi strictly one after the other"},
            "phi0": "zero start via pmg_set_guess(NULL)", "result_read_back": out_ok}


# ------------------------------------------------------------------------------------------------------
def run_single(args):
    import pmg_b200 as pmg
    if pmg.device_count() < 1:
        raise SystemExit("bench.py needs a B200: libpmg.so has no CPU fallback")
    n = args.n
    peak, peak_src = hbm_peak()
    prolong = pmg.PROLONG_FULL if args.prolong == "full" else pmg.PROLONG_REFERENCE
    s = pmg.Solver(n, omega=OMEGA, prolong_mode=prolong, device=0)
    s.set_rhs_sine()
    max_cycles = 100
    cross_cycle = s.cross_cycle

    def step():
        s.zero_guess()
        return s.solve(pmg.V, rel_tol=REL_TOL, max_cycles=max_cycles)

    for _ in range(args.warmup):
        k, hist = step()
    pmg.check(pmg.lib().pmg_device_synchronize())
    clocks = ClockSampler(0)
    clocks.start()
    launches0 = pmg.kernel_launches()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        k, hist = step()
        dev_ms += s.last_ms
    pmg.check(pmg.lib().pmg_device_synchronize())
    wall = time.perf_counter() - t0
    launches = pmg.kernel_launches() - launches0
    clk = clocks.stop()
    ms_per_step = 1e3 * wall / args.steps
    value = n * n / (wall / args.steps) / 1e9
    converged = bool(hist[-1] < REL_TOL * hist[0])
    if args.dump_outputs:  # before the roofline passes below overwrite the iterate
        dump_outputs(args.dump_outputs, s.get_solution(), hist)

    # ---- roofline of the dominant kernel (level-0 fused passes), timed alone with CUDA events ----
    t_down = s.bench_pass(0, 0, 5)
    t_upn = s.bench_pass(1, 0, 5)
    try:
        t_cross = s.bench_pass(4, 0, 5)   # the kernel pmg_solve actually spends its time in (cross-cycle pass)
    except Exception:  # noqa: BLE001
        t_cross = None
    if t_cross is not None:
        # One launch does a whole level visit's streaming work.  SURVEY 8(d) prices that at 52 B per level-point (Pass B +
        # Pass A, 26 B each); the fused pass has to move only 28 (read xb, f: 16, e: 2; write xb': 8, coarse f: 2).  `frac`
        # is taken against the 28 B the kernel must move, so it cannot exceed 1; the 52 B work-equivalent figure (which
        # does exceed the copy peak) is reported beside it.
        alg_bytes = CROSS_BYTES_PER_POINT * n * n
        dom_ms, dom_name = t_cross, "k_cross<nu2=2,nu1=2> (Pass B of cycle k + Pass A of cycle k+1 in one sweep)"
        traffic = ncu_traffic("k_cross", n)
    else:
        alg_bytes = BYTES_PER_POINT_PASS * n * n
        dom_ms, dom_name = (t_upn, "k_up<nu2=2,prolong,norm>") if t_upn >= t_down else (t_down, "k_down<nu1=2,resid>")
        traffic = ncu_traffic("k_up" if t_upn >= t_down else "k_down", n)
    achieved = alg_bytes / (dom_ms * 1e-3) / 1e9
    cycle_gbs = BYTES_PER_DOF_CYCLE * n * n * k / (dev_ms / args.steps * 1e-3) / 1e9
    # Jacobi sweep sub-metric: one HBM pass per sweep, 24 B/point
    s.smooth(3, 1)
    s.smooth(10, 1)
    jac_gbs = 24.0 * n * n * 10 / (s.last_ms * 1e-3) / 1e9
    s.smooth(12, 4)
    jac_blocked_gbs = 24.0 * n * n * 12 / (s.last_ms * 1e-3) / 1e9

    # ---- e2e through the C ABI with pinned HOST buffers ----
    e2e = e2e_measure(pmg, s, n, n, args, lambda out: sine_rhs(n, out), max_cycles)
    s.close()

    # ---- parity of the timed configuration against the reference's CPU history (committed golden) ----
    gold = goldens()
    parity = history_check(hist[1:], gold.get("V_n16385_full" if args.prolong == "full" else "V_n16385")) \
        if n == 16385 else history_check(hist[1:], gold.get("V_n%d" % n))
    # ---- the other BASELINE configs (W, F, N = 4097, N = 32769) as short legs ----
    legs = None
    if not args.no_legs:
        legs = config_legs(lambda nn, **cfg: pmg.Solver(nn, omega=OMEGA, prolong_mode=prolong, device=0, **cfg), peak, 1)

    # ---- CPU baseline (bounded sample of the same workload on the host cores) ----
    cpu = None
    if not args.no_cpu_baseline:
        v, secs, kind = cpu_reference_sample(4097, 4, n, k)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
               "sample": "4 V(2,2) cycles at N=4097 (%.1f s), scaled by DOF*cycles to %d cycles at N=%d; the "
                         "reference is single-threaded" % (secs, k, n),
               "host_cores_available": os.cpu_count()}

    ref_cuda = None
    if not args.no_ref_cuda:
        rc_clocks = ClockSampler(0)
        rc_clocks.start()
        ref_cuda = reference_cuda_build()
        ref_cuda["clocks"] = rc_clocks.stop()
    if ref_cuda and str(n) in ref_cuda and "best_cycle_ms" in ref_cuda[str(n)]:
        ref_cuda["ours_cycle_ms_same_n"] = dev_ms / args.steps / k
        ref_cuda["speedup_per_cycle_same_n"] = ref_cuda[str(n)]["best_cycle_ms"] / (dev_ms / args.steps / k)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args, 1),
            "cycles_to_converge": k, "converged": converged, "final_rel_residual": float(hist[-1] / hist[0]),
            "cycles_match": parity["cycles_match"], "history_max_rel_dev": parity["history_max_rel_dev"],
            "history_parity": parity, "cross_cycle_pass": cross_cycle,
            "gdof_cycle_per_s": n * n * k / (dev_ms / args.steps * 1e-3) / 1e9,
            "device_ms_per_step": dev_ms / args.steps,
            "legs": legs,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": "committed ncu --set full capture (profiles/), not re-measured in this run",
                         "kernel": dom_name,
                         "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": dom_ms, "peak_source": peak_src,
                         "pass_down_ms": t_down, "pass_up_norm_ms": t_upn, "pass_cross_ms": t_cross,
                         "two_pass_frac": BYTES_PER_POINT_PASS * n * n / (max(t_down, t_upn) * 1e-3) / 1e9 / peak,
                         "cross_pass_bytes_moved_per_point": CROSS_BYTES_PER_POINT,
                         "work_equivalent_gbs_at_survey_52B_per_point":
                             (2 * BYTES_PER_POINT_PASS * n * n / (t_cross * 1e-3) / 1e9) if t_cross else None,
                         "frac_vs_two_pass_52B_per_point":
                             (2 * BYTES_PER_POINT_PASS * n * n / (t_cross * 1e-3) / 1e9 / peak) if t_cross else None,
                         "note": "the cross-cycle pass is instruction- and energy-bound, not HBM-bound: it does the work the "
                                 "SURVEY figure prices at 52 B/point while moving 28 (DESIGN.md 4.4); frac is against the 28",
                         "vcycle_effective_gbs_at_69.3B_per_dof": cycle_gbs, "vcycle_frac": cycle_gbs / peak,
                         "vcycle_frac_at_45.3B_per_dof_cross_minimum": cycle_gbs * (45.3 / BYTES_PER_DOF_CYCLE) / peak},
            "jacobi_sweep": {"gbs_24B_per_point": jac_gbs, "frac": jac_gbs / peak,
                             "blocked4_effective_gbs": jac_blocked_gbs},
            "cpu_baseline": cpu, "reference_cuda_build": ref_cuda, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clk}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=16385)
    ap.add_argument("--prolong", default="reference", choices=["reference", "full"])
    ap.add_argument("--cycles-expected", type=int, default=39, dest="cycles_expected")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip timing the reference's own CUDA build")
    ap.add_argument("--no-legs", action="store_true", dest="no_legs",
                    help="skip the W / F / N=4097 / N=32769 legs (the other BASELINE configs)")
    ap.add_argument("--no-same-config", action="store_true", dest="no_same_config",
                    help="--impl reference: skip the N=4097 solve measured end to end (~1 min)")
    ap.add_argument("--agglomerate-below", type=int, default=513, dest="agglomerate_below",
                    help="multi-GPU: levels with n <= this run on rank 0 only")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write what the last timed solve returned to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or world > 1 or args.gpus > 1):
        ap.error("--dump-outputs is implemented for the CUDA path on one GPU")
    if args.impl == "reference":
        return run_reference(args)
    if world > 1 or args.gpus > 1:
        import bench_dist
        return bench_dist.run(args)
    return run_single(args)


if __name__ == "__main__":
    sys.exit(main())
