#!/usr/bin/env python
"""bench.py -- preconditioned Krylov iterations/s and time to solution of the moving-PML sweeping-preconditioner solve.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2]): 2D heterogeneous layered velocity model, 4096^2 grid, 10 points per wavelength,
PML width 12, R = 8 right-hand sides per GPU (the reference's source at R shot positions), GMRES(20).

A "step" is ONE preconditioned GMRES inner iteration of every right-hand side in flight (code.py:516): per right-hand
side one 5-point stencil SpMV, one application of the sweeping preconditioner (algo2_4: front solves + forward and
backward sweeps over all n-b moving-PML strips), the modified Gram-Schmidt orthogonalisation and the host Givens
update.  K steps = restarted GMRES(20) run for exactly K inner iterations (rtol = 0), including the solution update /
true residual at every restart boundary.  `value` counts the inner iterations of all right-hand sides per second.
The preconditioner is applied to the Krylov vector (precond_input='vector'): per iteration this is exactly the work
the reference does (it re-runs algo2_4 on every call, code.py:510-511), but it is NOT the reference's literal data
flow (its LinearOperator ignores its argument); see `time_to_solution` for what converges and what does not.

N > 1: the grid is slab-decomposed over the GPUs (NCCL: halo rows, dot-product all-reduces, sweep hand-over rows), the
8N right-hand sides follow each other through the slabs.  The line also carries `slab_parity` (slab path against one
GPU at n = 1024) and `baseline_configs` (BASELINE.json's single-right-hand-side multi-GPU cases).

One JSON line is printed by rank 0.  See DESIGN.md "Measurement" for the definition of every key.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "precond. Krylov iters/s at 4096^2 2D"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", "--grid-n", dest="n", type=int, default=0, help="interior grid points per side (default: 4096; --grid-n under torchrun, whose parser claims --n)")
    ap.add_argument("--b", type=int, default=12, help="PML width in grid points (reference: 12)")
    ap.add_argument("--ppw", type=float, default=10.0, help="grid points per wavelength")
    ap.add_argument("--const", type=float, default=100.0)
    ap.add_argument("--model", default="layered", choices=["layered", "constant", "c1"])
    ap.add_argument("--rhs", type=int, default=8, help="right-hand sides in flight per GPU")
    ap.add_argument("--cpu-strips", type=int, default=6, help="strips timed for the CPU baseline sample at the bench size")
    ap.add_argument("--cpu-full-n", type=int, default=1024, help="grid size of the fully executed CPU iteration (0 = skip)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-tts", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N > 1: skip slab_parity and the single-right-hand-side BASELINE configs")
    ap.add_argument("--no-baseline-configs", action="store_true", help="N > 1: keep slab_parity, skip the single-right-hand-side BASELINE configs")
    ap.add_argument("--parity-only", action="store_true", help="N > 1: run slab_parity, print it and stop")
    ap.add_argument("--hang-dump", type=int, default=0, help="developer: after this many seconds write the Python stacks of all threads "
                    "to gpurun_out/hang_rank<r>.txt and exit")
    ap.add_argument("--mp-schedule", default="async", choices=["async", "lockstep"],
                    help="N > 1, pipelined mode: groups of right-hand sides as independent pipelines (slab.GroupPipeline) or all in lock step")
    ap.add_argument("--mp-mode", default="pipelined", choices=["pipelined", "weak"],
                    help="N > 1: 'pipelined' (default) = the 4096^2 problem slab-decomposed, --rhs right-hand sides per GPU sent through "
                         "the slabs one behind the other; 'weak' = only the single-right-hand-side weak-scaling case (n = 4096 sqrt(N))")
    ap.add_argument("--dump-outputs", metavar="DIR", help="one GPU: after the timed steps, write what the last timed GMRES batch "
                    "returned as float64 .npy files in DIR: u (right-hand side, sampled point, re/im: every solution at the same "
                    "seeded sample of at most 48 MB in all), residuals (right-hand side, inner iteration) and info")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs: the b200 arm on one GPU only")
    return a


def workload(args, world, n=None):
    n = n or (args.n if args.n else 4096)
    return dict(n=n, b=args.b, wave_num=n / args.ppw, const=args.const, alpha=2.0, model=args.model)


def make_fields(w):
    import helmholtz_preconditioner_b200 as hp
    omega = 2 * np.pi * w["wave_num"] + 1j * w["alpha"]
    n = w["n"]
    if w["model"] == "layered":
        c_mat, f_mat = hp.init_layered_f1(omega, n)
    elif w["model"] == "constant":
        c_mat, f_mat = hp.init_const_f1(omega, n)
    else:
        c_mat, f_mat = hp.init_c1_f1(omega, n)
    return omega, c_mat, np.ascontiguousarray(f_mat.astype(np.complex128))


def shots(f_mat, R):
    """R right-hand sides: the reference's source moved along x1 (one shot position per right-hand side)"""
    n = f_mat.shape[0]
    return [np.ascontiguousarray(np.roll(f_mat, (i * n) // (2 * R), axis=1)) for i in range(R)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower() == "active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path
# ------------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_iteration_sample(w, nstrips, c_mat, f_mat):
    """Time the reference algorithm (oracle port: scipy SuperLU strip solves as in code.py:345-385, CSR matvec) on
    `nstrips` of the n-b strips and extrapolate one preconditioned Krylov iteration linearly in the number of strips
    (every strip costs the same: 3 SuperLU solves of a bn x bn system, code.py:366-380).  EXTRAPOLATED: at 4096^2 the
    4084 strip factorisations need ~160 GB and ~12 min; cpu_iteration_full() is the fully executed counterpart."""
    import scipy.sparse.linalg as spla
    from oracle import helmholtz_oracle as orc
    n, b = w["n"], w["b"]
    omega = 2 * np.pi * w["wave_num"] + 1j * w["alpha"]
    h = 1 / (n + 1)
    eta = b * h
    ms = np.linspace(b + 1, n, nstrips).astype(int)
    t_fac = t_sol = 0.0
    rng = np.random.default_rng(0)
    v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    for m in ms:
        t0 = time.perf_counter()
        Hm = orc.get_Hm(int(m), b, w["const"], eta, omega, h, n, c_mat).tocsc()
        lu = spla.splu(Hm)
        t1 = time.perf_counter()
        t = np.zeros(b * n, dtype=np.complex128)
        for _ in range(3):                        # code.py:370, 375, 380
            t[-n:] = v
            lu.solve(t)[-n:]
        t2 = time.perf_counter()
        t_fac += t1 - t0
        t_sol += t2 - t1
    A = orc.build_A_matrix(b, w["const"], eta, omega, h, n, c_mat)
    x = f_mat.ravel()
    t0 = time.perf_counter()
    A @ x
    t_mv = time.perf_counter() - t0
    # orthogonalisation at the average Krylov index of GMRES(20): ~10 vdot + 10 axpy
    V = np.stack([x, x * 1j])
    t0 = time.perf_counter()
    for _ in range(5):
        hcoef = np.vdot(V[0], V[1])
        V[1] -= hcoef * V[0]
    t_orth = (time.perf_counter() - t0) * 2
    per_strip = t_sol / len(ms)
    t_iter = per_strip * (n - b) + t_mv + t_orth
    return dict(t_iter=t_iter, per_strip_solve=per_strip, per_strip_factor=t_fac / len(ms), t_matvec=t_mv,
                t_setup=t_fac / len(ms) * (n - b), strips=len(ms))


def cpu_iteration_full(args, n):
    """One COMPLETE preconditioned GMRES iteration of the oracle port at grid size n, nothing extrapolated: algo2_3 (all
    n-b SuperLU factorisations), then A x, algo2_4 (all strips, three solves each) and a Gram-Schmidt pass at the
    average Krylov index, timed."""
    from oracle import helmholtz_oracle as orc
    w = workload(args, 1, n=n)
    omega, c_mat, f_mat = make_fields(w)
    b = w["b"]
    h = 1 / (n + 1)
    t0 = time.perf_counter()
    P = orc.SweepingPreconditioner(b, w["const"], b * h, omega, h, n, c_mat)
    A = orc.build_A_matrix(b, w["const"], b * h, omega, h, n, c_mat)
    t_setup = time.perf_counter() - t0
    x = f_mat.ravel()
    t0 = time.perf_counter()
    y = P.apply(A @ x)
    V = np.stack([x, x * 1j])
    for _ in range(10):
        hcoef = np.vdot(V[0], y)
        y -= hcoef * V[0]
    t_iter = time.perf_counter() - t0
    return dict(n=n, b=b, t_iter=t_iter, t_setup=t_setup, strips=n - b)


def cpu_baseline_block(args, w, c_mat, f_mat, nstrips, gpu_full=None):
    c = cpu_iteration_sample(w, nstrips, c_mat, f_mat)
    n, b = w["n"], w["b"]
    out = {"value": 1.0 / c["t_iter"], "unit": "iters/s", "cores": 1, "host_cores": host_cores(), "kind": "port",
           "extrapolated": True, "strips_sampled": c["strips"], "strips_total": n - b,
           "sample": (f"{c['strips']} of {n - b} strips (SuperLU factor + 3 solves each, as code.py:345-380) + 1 CSR matvec on one "
                      f"host core (the reference's scipy/numba path is single-threaded; the box has {host_cores()} cores), "
                      f"extrapolated linearly to all strips"),
           "per_strip_solve_s": c["per_strip_solve"], "per_strip_factor_s": c["per_strip_factor"],
           "setup_s_extrapolated": c["t_setup"]}
    if args.cpu_full_n:
        f = cpu_iteration_full(args, args.cpu_full_n)
        out["full_run"] = {"n": f["n"], "b": f["b"], "extrapolated": False, "iters_per_s": 1.0 / f["t_iter"], "iter_s": f["t_iter"],
                           "setup_s": f["t_setup"], "strips": f["strips"],
                           "what": "one complete oracle iteration (all strips factored and applied) at this grid size"}
        if gpu_full:
            out["full_run"]["gpu_iters_per_s_same_problem"] = gpu_full
    return out, c


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    w = workload(args, world)
    omega, c_mat, f_mat = make_fields(w)
    ns = max(1, args.cpu_strips // 2)
    vals = []
    t_start = time.time()
    for i in range(args.warmup + args.steps):
        r = cpu_iteration_sample(w, ns, c_mat, f_mat)
        if i >= args.warmup:
            vals.append(r["t_iter"])
    t_iter = float(np.mean(vals))
    cb, _ = cpu_baseline_block(args, w, c_mat, f_mat, ns)
    cb["value"] = 1.0 / t_iter
    cb["consistency"] = {"wall_s_of_this_run": time.time() - t_start, "claimed_s_if_fully_executed": t_iter * (args.warmup + args.steps),
                         "fits_in_driver_run": False,
                         "note": "the 4096^2 figure is extrapolated from sampled strips; full_run is executed completely"}
    out = {"impl": "reference", "metric": METRIC, "value": 1.0 / t_iter, "unit": "iters/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_iter,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "complex128 (f64)",
           "data": "synthetic", "config": config_dict(w, world, args.rhs),
           "cpu_baseline": cb,
           "e2e": {"value": 1.0 / t_iter, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def config_dict(w, world, R):
    return {"workload": (f"2D heterogeneous synthetic layered velocity model {w['n']}^2, PML width {w['b']}, "
                         f"{w['n'] / w['wave_num']:.0f} points per wavelength, preconditioned GMRES(20) inner iterations, "
                         f"{R} right-hand sides per GPU"
                         if w["model"] == "layered" else f"2D {w['model']} velocity {w['n']}^2, PML width {w['b']}, {R} right-hand sides per GPU"),
            "n": w["n"], "b": w["b"], "wave_num": w["wave_num"], "const": w["const"], "alpha": w["alpha"],
            "restart": 20, "precond_input": "vector", "diag": "reference", "front": "blockdiag", "rhs_per_gpu": R,
            "l2": "inputs larger than L2: the sweep streams the strip generators (GBs per step) once per sweep",
            "parallelism": f"slab{world}" if world > 1 else "single"}


def peak_hbm():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------
# B200 arm, one GPU
# ------------------------------------------------------------------------------------------------------
def timed_region(torch, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, r


def dump_outputs(torch, out_dir, res):
    """gmres_batch's [(u, info, hist), ...] as float64 .npy files; a larger u is sampled at points fixed by a seed, so that
    two builds run with the same arguments can be compared output for output"""
    N, R = res[0][0].numel(), len(res)
    S = min(N, (48 << 20) // (16 * R))
    idx = np.arange(N) if S == N else np.sort(np.random.default_rng(0).choice(N, S, replace=False))
    idx = torch.from_numpy(idx).to(res[0][0].device)
    hist = np.full((R, max(len(h) for _, _, h in res)), np.nan)
    for i, (_, _, h) in enumerate(res):
        hist[i, :len(h)] = h
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "u.npy"), torch.view_as_real(torch.stack([u[idx] for u, _, _ in res])).cpu().numpy())
    np.save(os.path.join(out_dir, "residuals.npy"), hist)
    np.save(os.path.join(out_dir, "info.npy"), np.array([info for _, info, _ in res], dtype=np.float64))


def true_residual(torch, s, f, u):
    r = s.matvec(u)
    return (torch.linalg.norm(f - r) / torch.linalg.norm(f)).item()


def time_to_solution(torch, hp, s, w, c_mat, f_mat, t_setup, f):
    """Converged solves (rtol 1e-3 on the true residual as scipy checks it): GMRES(20) with the preconditioner applied to
    the Krylov vector and the paper's diagonal solve, (a) with the coupled front block, (b) with the reference's
    block-diagonal front block; next to them the reference call exactly as written, which does not converge."""
    n, b = w["n"], w["b"]
    out = {}

    def solve(diag, pin, cap):
        torch.cuda.synchronize()
        t0 = time.time()
        r = hp.run_solver(n, b, w["wave_num"], w["const"], w["alpha"], c_mat=c_mat, f_mat=f_mat, solver=s, diag=diag,
                          precond_input=pin, maxiter=cap, verbose=False)
        torch.cuda.synchronize()
        return r, time.time() - t0

    t0 = time.time()
    s.set_front("coupled")
    torch.cuda.synchronize()
    t_front = time.time() - t0
    r, dt = solve("paper", "vector", 400)
    out["coupled_front"] = {"mode": "precond_input='vector', diag='paper', front='coupled' (Engquist-Ying as published)", "setup_s": t_setup + t_front,
                            "solve_s": dt, "total_s": t_setup + t_front + dt, "niter": r.niter, "info": r.info,
                            "true_residual": true_residual(torch, s, f, r.u), "front_setup_s": t_front}
    s.set_front("blockdiag")
    r, dt = solve("paper", "vector", 1000)
    out["reference_front"] = {"mode": "precond_input='vector', diag='paper', front='blockdiag' (H_F of code.py:178-183)", "setup_s": t_setup,
                              "solve_s": dt, "total_s": t_setup + dt, "niter": r.niter, "info": r.info,
                              "true_residual": true_residual(torch, s, f, r.u)}
    r, dt = solve("reference", "vector", 100)
    out["reference_diag"] = {"mode": "precond_input='vector', diag='reference' (code.py:372-375 as written), capped at 100 iterations",
                             "solve_s": dt, "niter": r.niter, "info": r.info, "converged": r.info == 0,
                             "true_residual": true_residual(torch, s, f, r.u)}
    r, dt = solve("reference", "rhs", None)
    out["reference_literal"] = {"mode": "the call as written (code.py:510-516: M ignores its argument): NOT a solution", "solve_s": dt,
                                "niter": r.niter, "info": r.info, "converged": r.info == 0,
                                "true_residual": true_residual(torch, s, f, r.u)}
    best = out["coupled_front"] if out["coupled_front"]["info"] == 0 else out["reference_front"]
    out.update({"setup_s": best["setup_s"], "solve_s": best["solve_s"], "total_s": best["total_s"], "niter": best["niter"],
                "info": best["info"], "true_residual": best["true_residual"], "mode": best["mode"],
                "converged": best["info"] == 0 and best["true_residual"] <= 1e-3})
    return out


def run_b200(args):
    import torch
    import ctypes as C
    import helmholtz_preconditioner_b200 as hp
    from helmholtz_preconditioner_b200 import _lib
    from helmholtz_preconditioner_b200.gmres import DeviceVectors, gmres, gmres_batch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        return run_b200_slabs(args)
    torch.cuda.set_device(local)
    lib = _lib.require_device()
    w = workload(args, 1)
    omega, c_mat, f_mat = make_fields(w)
    n, b, R = w["n"], w["b"], args.rhs
    N = n * n
    # process start-up (CUDA context, loading the kernels of the library) is not part of the setup of a problem: a 96^2
    # solve brings both up before the clock starts
    om0 = 2 * np.pi * 9.6 + 2j
    c0, f0 = hp.init_layered_f1(om0, 96)
    s0 = hp.HelmholtzSolver(96, b, om0, w["const"], c0)
    s0.setup_preconditioner(front="coupled")
    s0.precond_apply(torch.from_numpy(f0.ravel().astype(np.complex128)).cuda())
    torch.cuda.synchronize()
    s0.close()
    del s0
    t0 = time.time()
    s = hp.HelmholtzSolver(n, b, omega, w["const"], c_mat)
    s.setup_preconditioner()
    torch.cuda.synchronize()
    t_setup = time.time() - t0
    L = s.layout()
    f_hosts = [torch.from_numpy(x.ravel()).pin_memory() for x in shots(f_mat, R)]
    u_hosts = [torch.empty(N, dtype=torch.complex128).pin_memory() for _ in range(R)]
    fs = [fh.cuda(non_blocking=True) for fh in f_hosts]
    f = fs[0]
    vec = DeviceVectors(N, f.device)
    mv = lambda x, out: s.matvec(x, out)                      # noqa: E731
    ps = lambda x, out: s.precond_apply(x, out=out)           # noqa: E731
    psb = lambda reqs: s.precond_apply_batch(reqs)            # noqa: E731

    def single(k, rhs):
        return gmres(mv, ps, rhs, vec=vec, rtol=0.0, atol=0.0, restart=20, maxiter=k)

    def batch(k, rhss):
        return gmres_batch(mv, psb, rhss, vec=vec, rtol=0.0, atol=0.0, restart=20, maxiter=k)

    # ---- one right-hand side (the round-1 headline): iteration rate and the roofline of the single-vector sweep kernel
    single(args.warmup, f)
    lib.hp_profile_enable(s.handle, 1)
    t_one, (u1, info1, hist1) = timed_region(torch, lambda: single(args.steps, f))
    sw_ms, sw_n, sw_b = C.c_double(), C.c_int(), C.c_int64()
    lib.hp_profile_read(s.handle, C.byref(sw_ms), C.byref(sw_n), C.byref(sw_b))
    lib.hp_profile_enable(s.handle, 0)
    # ---- R right-hand sides in lock step: the headline
    batch(args.warmup, fs)
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    clocks.start()
    lib.hp_profile_enable(s.handle, 1)
    l0 = lib.hp_launch_count()
    t_dev, res = timed_region(torch, lambda: batch(args.steps, fs))
    launches = lib.hp_launch_count() - l0
    bw_ms, bw_n, bw_b = C.c_double(), C.c_int(), C.c_int64()
    lib.hp_profile_read(s.handle, C.byref(bw_ms), C.byref(bw_n), C.byref(bw_b))
    lib.hp_profile_enable(s.handle, 0)
    if args.dump_outputs:
        dump_outputs(torch, args.dump_outputs, res)
    # ---- end to end through the public API with host buffers: pinned f -> device, K iterations, u -> host

    def e2e():
        fs2 = [fh.cuda(non_blocking=True) for fh in f_hosts]
        res2 = batch(args.steps, fs2)
        for uh, (u2, _, _) in zip(u_hosts, res2):
            uh.copy_(u2, non_blocking=True)
    t_e2e, _ = timed_region(torch, e2e)
    clk = clocks.stop()
    s.check_status()
    del res

    # ---- secondary kernels of the path: matrix-free stencil SpMV and CSR assembly, device time per launch
    def timed(fn, reps):
        fn(); torch.cuda.synchronize()
        return timed_region(torch, lambda: [fn() for _ in range(reps)])[0] / reps
    xs = [torch.randn(N, dtype=torch.complex128, device=f.device) for _ in range(3)]   # 3 x 268 MB > L2
    ys = torch.empty_like(f)
    cnt = [0]

    def spmv():
        cnt[0] += 1
        s.matvec(xs[cnt[0] % 3], ys)
    t_spmv = timed(spmv, 30)
    spmv_bytes = N * (16 + 16 + 8)                      # x read, y written, kappa read (DESIGN.md)
    nnz = 5 * N - 4 * n
    A_ = s.assemble_csr()
    t_asm = timed(lambda: lib.hp_assemble_csr(s.handle, A_.indptr.data_ptr(), A_.indices.data_ptr(), A_.data.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream), 5)
    asm_bytes = nnz * (16 + 4) + (N + 1) * 4 + N * 8    # values + column indices + row pointers written, kappa read
    del A_, xs
    peak, peak_src = peak_hbm()
    traffic = None
    try:
        per_strip = json.load(open(os.path.join(ROOT, "profiles", "sweep_traffic.json")))["dram_bytes_per_strip"]
        # ncu figure per strip x the strips of an average timed launch (forward: n-b-1 strips, backward: n-b)
        traffic = per_strip * (n - b - 0.5) if (n, b) == (4096, 12) else None
    except Exception:
        pass

    def roof(ms, nl, by, kernel, rhs_per_launch):
        ach = (by / 1e9) / (ms / 1e3) if ms > 0 else 0.0
        return {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "peak_source": peak_src, "launches_timed": nl, "avg_launch_ms": ms / max(nl, 1),
                "algorithmic_bytes_per_launch": by / max(nl, 1), "rhs_per_launch": rhs_per_launch}
    kern = "hp_sweep4_kernel" if L.get("colN") else "hp_sweep2_kernel"
    roof_b = roof(bw_ms.value, bw_n.value, bw_b.value, s.batch_kernel_name(R), s.batch_group(R))
    roof_b["share_of_step"] = (bw_ms.value / 1e3) / t_dev
    roof_b["note"] = ("algorithmic bytes = generators of the strips once per launch + 3 field rows per strip and right-hand side; a launch "
                      "that carries several right-hand sides re-uses the generators, so GB/s per launch falls while iterations/s rise: "
                      "iters_per_s_at_hbm_floor is the ceiling of this design")
    # one preconditioner application of a group = 2 sweep launches that cannot run faster than their bytes at the HBM peak
    roof_b["iters_per_s_at_hbm_floor"] = (s.batch_group(R) * peak * 1e9 / (2.0 * bw_b.value / bw_n.value)) if bw_n.value else None
    roof_1 = roof(sw_ms.value, sw_n.value, sw_b.value, kern, 1)
    roof_1["share_of_step"] = (sw_ms.value / 1e3) / t_one
    total_steps = args.steps * R
    out = {"metric": METRIC, "value": total_steps / t_dev, "unit": "iters/s", "n_gpus": 1,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_dev / args.steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "complex128 (f64)",
           "data": "synthetic", "config": config_dict(w, 1, R),
           "e2e": {"value": total_steps / t_e2e, "unit": "iters/s", "h2d_bytes_per_step": R * N * 16 / args.steps,
                   "d2h_bytes_per_step": R * (N * 16 / args.steps + 16 * 22),
                   "note": "host f -> device, K GMRES iterations per right-hand side, u -> host; the Hessenberg columns come back every step"},
           "gpu_launches": int(launches),
           "roofline": roof_b,
           "single_rhs": {"value": args.steps / t_one, "unit": "iters/s", "ms_per_step": 1e3 * t_one / args.steps, "roofline": roof_1,
                          "note": "one right-hand side (round-1 headline configuration)"},
           "spmv": {"kernel": "hp_stencil_matvec_kernel", "ms": 1e3 * t_spmv, "GB/s": spmv_bytes / t_spmv / 1e9,
                    "frac_of_hbm_peak": spmv_bytes / t_spmv / 1e9 / peak, "bytes_per_point": 40},
           "assembly": {"kernel": "hp_assemble_csr_kernel", "ms": 1e3 * t_asm, "GB/s": asm_bytes / t_asm / 1e9,
                        "frac_of_hbm_peak": asm_bytes / t_asm / 1e9 / peak, "nnz": nnz},
           "clocks": clk,
           "setup": {"seconds_wall": t_setup, "strip_factor_ms_device": s.setup_ms, "factor_bytes": s.precond_bytes,
                     "note": "wall time of HelmholtzSolver(...) + setup_preconditioner() in a process whose CUDA context and kernels are already loaded",
                     "partition": {k: int(L[k]) for k in ("P", "K", "G", "QP", "CW", "NS", "NR", "PK", "colN", "NRQ", "NXG")}},
           "residual_last": hist1[-1] if hist1 else None}
    if not args.no_tts:
        out["time_to_solution"] = time_to_solution(torch, hp, s, w, c_mat, f_mat, t_setup, f)
    gpu_full = None
    if not args.no_cpu and args.cpu_full_n:
        # the GPU on the problem the CPU executes in full
        s.close()
        del s
        torch.cuda.empty_cache()
        wf = workload(args, 1, n=args.cpu_full_n)
        omf, cf, ff = make_fields(wf)
        sf = hp.HelmholtzSolver(wf["n"], b, omf, wf["const"], cf).setup_preconditioner()
        ffd = torch.from_numpy(ff.ravel()).cuda()
        vf = DeviceVectors(ffd.numel(), ffd.device)
        run = lambda k: gmres(lambda x, o: sf.matvec(x, o), lambda x, o: sf.precond_apply(x, out=o), ffd, vec=vf, rtol=0.0, atol=0.0,  # noqa: E731
                              restart=20, maxiter=k)
        run(3)
        gpu_full = 20 / timed_region(torch, lambda: run(20))[0]
        sf.close()
    if not args.no_cpu:
        out["cpu_baseline"], _ = cpu_baseline_block(args, w, c_mat, f_mat, args.cpu_strips, gpu_full)
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------------
# B200 arm, N GPUs: slab decomposition
# ------------------------------------------------------------------------------------------------------
def slab_parity(torch, dist, hp, args, rank, world, dev):
    """The slab path (CUDA kernels behind the *_buf entry points with row offsets, NCCL hand-over) against one GPU on the
    same inputs at n = 1024: M x, A x, 15 GMRES iterations, and a pipelined batch against one-by-one application."""
    from helmholtz_preconditioner_b200.slab import distributed_gmres_setup
    from helmholtz_preconditioner_b200.gmres import DeviceVectors, gmres
    n, b = 1024, args.b
    omega = 2 * np.pi * n / 10 + 2j
    c_mat, f_mat = hp.init_layered_f1(omega, n)
    S = distributed_gmres_setup(n, b, omega, 100.0, c_mat, rank, world, None, dev)
    rng = np.random.default_rng(11)
    x = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    xl = torch.from_numpy(x[S.j0:S.j1].ravel().copy()).to(dev)
    out = torch.empty_like(xl)
    res = {}
    S.precond_apply(xl, out); res["M"] = out.clone()
    S.matvec(xl, out); res["A"] = out.clone()
    xs = [torch.from_numpy((rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)))[S.j0:S.j1].ravel().copy()).to(dev) for _ in range(5)]
    singles = []
    for xx in xs:
        o = torch.empty_like(xx); S.precond_apply(xx, o); singles.append(o)
    pairs = [(xx, torch.empty_like(xx)) for xx in xs]
    S.precond_apply_batch(pairs)
    eb = max((torch.linalg.norm(o - s1_) / torch.linalg.norm(s1_)).item() for (_, o), s1_ in zip(pairs, singles))
    ebt = torch.tensor([eb], device=dev)
    dist.all_reduce(ebt, op=dist.ReduceOp.MAX)
    vec = DeviceVectors(xl.numel(), dev, group=dist.group.WORLD)
    fl = torch.from_numpy(f_mat[S.j0:S.j1].ravel().astype(np.complex128)).to(dev)
    eg, iters_equal, st_pipe = None, True, 0
    if args.mp_schedule == "async":
        # groups of right-hand sides as independent pipelines (threads, streams, solver contexts, communicators) against the
        # same systems advanced in lock step
        from helmholtz_preconditioner_b200.slab import GroupPipeline
        from helmholtz_preconditioner_b200.gmres import gmres_batch
        fgs = [torch.from_numpy(np.ascontiguousarray(np.roll(f_mat, 31 * i, axis=1)[S.j0:S.j1].ravel().astype(np.complex128))).to(dev) for i in range(6)]
        kwg = dict(rtol=1e-3, restart=20, maxiter=6, nglobal=n * n)
        pipe = GroupPipeline(S, 3)
        rg = pipe.gmres([fgs[0:2], fgs[2:4], fgs[4:6]], lambda nloc, pg: DeviceVectors(nloc, dev, group=pg), diag="paper", **kwg)
        torch.cuda.synchronize()
        st_pipe = pipe.sweep_status()
        pipe.close()
        rl = gmres_batch(lambda a, o: S.matvec(a, o), lambda reqs: S.precond_apply_batch(reqs, diag="paper"), fgs, vec=vec,
                         matvec_batch=lambda reqs: S.matvec_batch(reqs), **kwg)
        num = torch.stack([torch.linalg.norm(a[0] - c[0]) ** 2 for a, c in zip([x for grp in rg for x in grp], rl)])
        den = torch.stack([torch.linalg.norm(c[0]) ** 2 for c in rl])
        dist.all_reduce(num); dist.all_reduce(den)
        eg = float(torch.sqrt(num / den).max().item())
        iters_equal = all(len(a[2]) == len(c[2]) and a[1] == c[1] for a, c in zip([x for grp in rg for x in grp], rl))
    u, info, hist = gmres(lambda a, o: S.matvec(a, o), lambda a, o: S.precond_apply(a, o, diag="paper"), fl, vec=vec,
                          rtol=1e-3, restart=20, maxiter=15, nglobal=n * n)
    res["u"] = u
    # gather the slabs on rank 0 (slabs may differ in size: padded all_gather)
    rows = [S.R[r + 1] - S.R[r] for r in range(world)]
    full = {}
    for k, v in res.items():
        pad = torch.zeros(max(rows) * n, dtype=torch.complex128, device=dev)
        pad[:v.numel()] = v
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad)
        full[k] = torch.cat([p[:rows[r] * n] for r, p in enumerate(parts)])
    st = S.s.sweep_status()
    S.s.close()
    out = None
    if rank == 0:
        s1 = hp.HelmholtzSolver(n, b, omega, 100.0, c_mat, device=dev).setup_preconditioner()
        xf = torch.from_numpy(x.ravel()).to(dev)
        rel = lambda a, c: (torch.linalg.norm(a - c) / torch.linalg.norm(c)).item()      # noqa: E731
        v1 = DeviceVectors(n * n, dev)
        f1 = torch.from_numpy(f_mat.ravel().astype(np.complex128)).to(dev)
        u1, info1, hist1 = gmres(lambda a, o: s1.matvec(a, o), lambda a, o: s1.precond_apply(a, out=o, diag="paper"), f1, vec=v1,
                                 rtol=1e-3, restart=20, maxiter=15)
        out = {"n": n, "M": rel(full["M"], s1.precond_apply(xf)), "A": rel(full["A"], s1.matvec(xf)), "u": rel(full["u"], u1),
               "gmres_iters": [len(hist), len(hist1)], "batch_vs_one_by_one": ebt.item(), "sweep_status": max(st, st_pipe),
               "groups_vs_lock_step": eg, "groups_iters_equal": bool(iters_equal),
               "tolerances": {"M": 1e-11, "A": 1e-13, "u": 1e-8, "batch_vs_one_by_one": 1e-13, "groups_vs_lock_step": 1e-10}}
        out["ok"] = bool(out["M"] < 1e-11 and out["A"] < 1e-13 and out["u"] < 1e-8 and len(hist) == len(hist1) and
                         ebt.item() < 1e-13 and st == 0 and st_pipe == 0 and (eg is None or eg < 1e-10) and iters_equal)
        s1.close()
    torch.cuda.empty_cache()
    return out


def slab_single_rhs(torch, dist, hp, args, n, rank, world, dev, steps=5, warmup=2):
    """BASELINE.json's multi-GPU configurations: ONE right-hand side of an n^2 problem slab-decomposed over the GPUs.  The
    sweeps are a sequential chain over the strips and therefore over the slabs: the GPUs take turns (the decomposition
    buys capacity for the strip factors, ~n^(8/3) bytes, not sweep speed)."""
    from helmholtz_preconditioner_b200.slab import distributed_gmres_setup
    from helmholtz_preconditioner_b200.gmres import CommStats, DeviceVectors, gmres
    w = workload(args, world, n=n)
    omega, c_mat, f_mat = make_fields(w)
    b = w["b"]
    free_b, total_b = torch.cuda.mem_get_info()
    t0 = time.time()
    try:
        S = distributed_gmres_setup(n, b, omega, w["const"], c_mat, rank, world, None, dev)
        err = None
    except Exception as e:                       # capacity: reported, not fatal for the headline
        S, err = None, str(e)
    flag = torch.tensor([0 if S is not None else 1], device=dev)
    dist.all_reduce(flag)
    if flag.item():
        if S is not None:
            S.s.close()
        torch.cuda.empty_cache()
        return {"n": n, "error": err or "another rank could not hold its strips", "free_bytes_rank0": free_b}
    torch.cuda.synchronize()
    t_setup = time.time() - t0
    fl = torch.from_numpy(f_mat[S.j0:S.j1].ravel()).to(dev)
    vec = DeviceVectors(fl.numel(), dev, group=dist.group.WORLD)
    run = lambda k: gmres(lambda a, o: S.matvec(a, o), lambda a, o: S.precond_apply(a, o), fl, vec=vec, rtol=0.0, atol=0.0,   # noqa: E731
                          restart=20, maxiter=k, nglobal=n * n)
    run(warmup)
    torch.cuda.synchronize(); dist.barrier()
    c0 = CommStats.calls
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(steps)
    e1.record()
    torch.cuda.synchronize(); dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1) / 1e3], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    fb = torch.tensor([float(S.s.precond_bytes)], device=dev)
    dist.all_reduce(fb)
    st = S.s.sweep_status()
    S.s.close()
    del S
    torch.cuda.empty_cache()
    return {"n": n, "rhs": 1, "iters_per_s": steps / t.item(), "ms_per_iter": 1e3 * t.item() / steps, "steps": steps, "warmup": warmup,
            "setup_s_wall": t_setup, "factor_bytes_all_ranks": fb.item(), "comm_calls_per_step_rank0": (CommStats.calls - c0) / steps,
            "sweep_status": st}


def run_b200_slabs(args):
    # before CUDA starts: (i) eager module loading - the first launch of a lazily loaded kernel may synchronise the whole
    # context, a deadlock once streams of this process wait for other GPUs (slab.GroupPipeline primes its groups as well);
    # (ii) one hardware queue per stream: a stream that waits for a sequence number of a neighbour (csrc/hp_peer.cu) must not
    # hold back another stream that happens to share its queue (default: 8 queues)
    os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import torch
    import torch.distributed as dist
    import helmholtz_preconditioner_b200 as hp
    from helmholtz_preconditioner_b200 import _lib
    from helmholtz_preconditioner_b200.slab import distributed_gmres_setup
    from helmholtz_preconditioner_b200.gmres import CommStats, DeviceVectors, gmres_batch
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    import faulthandler
    if args.hang_dump:
        os.makedirs("gpurun_out", exist_ok=True)
        faulthandler.dump_traceback_later(args.hang_dump, exit=True, file=open(f"gpurun_out/hang_rank{rank}.txt", "w"))
    else:
        # watchdog: the ranks of a multi-GPU run wait for each other on the device; if that ever stops making progress the
        # process must end (stacks of all threads on stderr, non-zero exit, torchrun takes the other ranks down) instead
        # of holding the box until somebody else's limit
        faulthandler.dump_traceback_later(800, exit=True, file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("nccl", device_id=dev)
    lib = _lib.require_device()
    parity = None
    if not args.no_extras:
        parity = slab_parity(torch, dist, hp, args, rank, world, dev)
        ok = torch.tensor([1 if (rank != 0 or parity["ok"]) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if not ok.item():
            if rank == 0:
                print(json.dumps({"metric": METRIC, "error": "slab_parity failed", "slab_parity": parity, "n_gpus": world}))
            dist.destroy_process_group()
            sys.exit(3)
        if args.parity_only:
            if rank == 0:
                print(json.dumps({"slab_parity": parity}))
            dist.destroy_process_group()
            return
    out = None
    if args.mp_mode == "pipelined":
        w = workload(args, world)
        omega, c_mat, f_mat = make_fields(w)
        n, b = w["n"], w["b"]
        R = args.rhs * world
        t0 = time.time()
        S = distributed_gmres_setup(n, b, omega, w["const"], c_mat, rank, world, None, dev)
        torch.cuda.synchronize()
        t_setup = time.time() - t0
        f_hosts = [torch.from_numpy(np.ascontiguousarray(x[S.j0:S.j1].ravel())).pin_memory() for x in shots(f_mat, R)]
        fs = [fh.to(dev) for fh in f_hosts]
        vec = DeviceVectors(fs[0].numel(), dev, group=dist.group.WORLD)
        mv = lambda x, o: S.matvec(x, o)                          # noqa: E731
        mvb = lambda reqs: S.matvec_batch(reqs)                   # noqa: E731
        psb = lambda reqs: S.precond_apply_batch(reqs)            # noqa: E731

        pipe = None
        if args.mp_schedule == "async":
            from helmholtz_preconditioner_b200.slab import GroupPipeline
            pipe = GroupPipeline(S, world)                        # one group of args.rhs right-hand sides per GPU

        def iterations(k, rhs, host_out=None):
            if pipe is None:
                return gmres_batch(mv, psb, rhs, vec=vec, matvec_batch=mvb, rtol=0.0, atol=0.0, restart=20, maxiter=k, nglobal=n * n)
            cut = lambda xs: [xs[g * args.rhs:(g + 1) * args.rhs] for g in range(world)]      # noqa: E731
            res = pipe.gmres(cut(rhs), lambda nloc, pg: DeviceVectors(nloc, dev, group=pg), rtol=0.0, atol=0.0, restart=20, maxiter=k,
                             nglobal=n * n, host_out=None if host_out is None else cut(host_out))
            return [x for grp in res for x in grp]

        iterations(args.warmup, fs)
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        l0, c0 = lib.hp_launch_count(), CommStats.calls
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); dist.barrier()
        e0.record()
        res = iterations(args.steps, fs)
        e1.record()
        torch.cuda.synchronize(); dist.barrier()
        comm_calls = CommStats.calls - c0
        t_dev = torch.tensor([e0.elapsed_time(e1) / 1e3], device=dev)
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        launches = torch.tensor([lib.hp_launch_count() - l0], device=dev)
        dist.all_reduce(launches)
        # end to end: host slabs of every f -> device, K iterations each, slabs of every u -> host
        u_hosts = [torch.empty(fs[0].numel(), dtype=torch.complex128).pin_memory() for _ in range(R)]
        torch.cuda.synchronize(); dist.barrier()
        e0.record()
        if pipe is None:
            fs2 = [fh.to(dev, non_blocking=True) for fh in f_hosts]
            res2 = iterations(args.steps, fs2)
            for uh, (u2, _, _) in zip(u_hosts, res2):
                uh.copy_(u2, non_blocking=True)
        else:                                                # every group moves its own right-hand sides and solutions
            fs2 = None
            res2 = iterations(args.steps, f_hosts, host_out=u_hosts)
        e1.record()
        torch.cuda.synchronize(); dist.barrier()
        t_e2e = torch.tensor([e0.elapsed_time(e1) / 1e3], device=dev)
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        fb = torch.tensor([float(S.s.precond_bytes)], device=dev)
        dist.all_reduce(fb)
        st = torch.tensor([max(S.s.sweep_status(), pipe.sweep_status() if pipe is not None else 0)], device=dev)
        dist.all_reduce(st, op=dist.ReduceOp.MAX)
        hist_last = res[0][2][-1] if res[0][2] else None
        group = S.batch_group(args.rhs if pipe is not None else len(fs))
        if pipe is not None:
            pipe.close()
        S.s.close()
        del S, res, res2, fs, fs2, vec
        torch.cuda.empty_cache()
        if rank == 0:
            clk = clocks.stop()
            total_steps = args.steps * R
            cfg = config_dict(w, world, args.rhs)
            cfg["parallelism"] = (f"slab{world}, {R} right-hand sides ({args.rhs} per GPU) pipelined through the slabs in groups of {group}, " +
                                  ("every group an independent GMRES (own thread, stream, solver context, communicator)" if args.mp_schedule == "async"
                                   else "all groups in lock step"))
            cfg["schedule"] = args.mp_schedule
            cfg["rhs_in_flight"] = R
            out = {"metric": METRIC, "value": total_steps / t_dev.item(), "unit": "iters/s",
                   "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_dev.item() / args.steps,
                   "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "complex128 (f64)",
                   "data": "synthetic", "config": cfg,
                   "e2e": {"value": total_steps / t_e2e.item(), "unit": "iters/s",
                           "h2d_bytes_per_step": R * n * n * 16 / args.steps, "d2h_bytes_per_step": R * (n * n * 16 / args.steps + 16 * 22)},
                   "gpu_launches": int(launches.item()), "clocks": clk,
                   "comm_calls_per_step_rank0": comm_calls / args.steps, "sweep_status": int(st.item()),
                   "setup": {"seconds_wall": t_setup, "factor_bytes_all_ranks": fb.item()},
                   "note": ("a step = one GMRES(20) inner iteration of every right-hand side in flight; value counts all of them.  "
                            "Per GPU the work is the same at every N (1/N of the strips, 8N right-hand sides): weak scaling in the number "
                            "of right-hand sides on a fixed grid.  The sweeps of the preconditioner are a sequential chain over the "
                            "strips, hence over the slabs, so the right-hand sides follow each other through the slabs (DESIGN.md, "
                            "multi-GPU); baseline_configs holds BASELINE.json's single-right-hand-side cases"),
                   "residual_last": hist_last}
    extras = {}
    guard = None
    if args.mp_mode == "pipelined":
        # The single-right-hand-side BASELINE configurations are extras of the line: if they do not come back (a rank that
        # fails alone leaves the others waiting in a collective), the headline that has been measured is printed without
        # them and every rank ends with exit code 0.
        def give_up():
            if rank == 0 and out is not None:
                out["baseline_configs"] = dict(extras, error="not finished after 300 s; the headline above was measured before")
                out["slab_parity"] = parity
                print(json.dumps(out), flush=True)
            os._exit(0)
        guard = threading.Timer(300.0, give_up)
        guard.daemon = True
        guard.start()
    if (not args.no_extras and not args.no_baseline_configs) or args.mp_mode == "weak":
        nw = int(round(4096 * np.sqrt(world)))

        def single(nn):
            try:
                return slab_single_rhs(torch, dist, hp, args, nn, rank, world, dev)
            except Exception as e:                           # noqa: BLE001 - reported in the line; the same on every rank
                return {"n": nn, "error": f"{type(e).__name__}: {e}"}

        extras["weak_4096sq_per_gpu"] = single(nw)
        if world >= 4 and nw == 8192:                   # N = 4: the weak case IS the 8192^2 problem
            extras["strong_8192sq"] = dict(extras["weak_4096sq_per_gpu"], same_run_as="weak_4096sq_per_gpu")
        elif world >= 4:
            extras["strong_8192sq"] = single(8192)
        else:
            extras["strong_8192sq"] = {"n": 8192, "skipped": "the strip factors of 8192^2 (~320 GB) need at least 4 GPUs of 180 GB"}
    if guard is not None:
        guard.cancel()
    if rank == 0:
        if out is None:                              # --mp-mode weak: the weak case is the line
            e = extras["weak_4096sq_per_gpu"]
            w = workload(args, world, n=e["n"])
            out = {"metric": METRIC, "value": e.get("iters_per_s"), "unit": "iters/s", "n_gpus": world, "steps": e.get("steps"),
                   "warmup": e.get("warmup"), "ms_per_step": e.get("ms_per_iter"), "higher_is_better": True, "scaling": "weak",
                   "vs_baseline": None, "dtype": "complex128 (f64)", "data": "synthetic", "config": config_dict(w, world, 1)}
        out["baseline_configs"] = extras
        out["slab_parity"] = parity
        print(json.dumps(out))
    dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
