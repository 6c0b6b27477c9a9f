"""Several sources per call: what masked slots and run_solver_many cost and save (GPU box).

    python tools/sources_time.py --out DIR [--part launches|solves|all] [--all-active-only] [--reps R]

launches: device time per sweep launch (hp_profile_read, forward + backward sweep over all strips, averaged) at 4096^2
    layered, b = 12: hp_sweep4d with 8, 7, 4 and 1 active slots, hp_sweep4m at 8 (HP_NO_DMMA), 4 and 2 right-hand sides,
    and the single-vector kernel.  The configurations take turns within every repetition, so drifts of the clock hit
    all of them alike.  --all-active-only leaves out the masked launches (a library without masked slots can run it).
solves: wall time of run_solver_many for S = 1, 3, 7, 8 and 12 sources at different shot positions against S calls of
    run_solver and against gmres_batch with the unpadded precond_apply_batch (every source in flight at once), for
    paper/coupled at 4096^2 and paper/blockdiag at 1024^2.  Each timing ends in a device synchronise.

Writes DIR/sources_time_<part>.json and prints it; the GPU's name and power limit are recorded with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import helmholtz_preconditioner_b200 as hp  # noqa: E402
from helmholtz_preconditioner_b200.gmres import DeviceVectors, gmres_batch  # noqa: E402

SHOTS = [(0.5, 0.125), (0.2, 0.3), (0.8, 0.3), (0.35, 0.6), (0.65, 0.6), (0.5, 0.85), (0.15, 0.8), (0.85, 0.8),
         (0.3, 0.45), (0.7, 0.45), (0.25, 0.15), (0.75, 0.15)]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "library": hp.LIB_PATH}
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                    text=True, timeout=30).strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as e:                                   # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return info


def profile_ms(s, fn):
    """device time per sweep launch of fn() and the number of launches"""
    s.lib.hp_profile_enable(s.handle, 1)
    fn()
    ms, cnt, by = C.c_double(), C.c_int(), C.c_int64()
    s.lib.hp_profile_read(s.handle, C.byref(ms), C.byref(cnt), C.byref(by))
    s.lib.hp_profile_enable(s.handle, 0)
    return ms.value / max(cnt.value, 1), cnt.value


def part_launches(a):
    n, b = 4096, 12
    omega = 2 * np.pi * n / 10 + 2j
    c_mat, _ = hp.init_layered_f1(omega, n)
    s = hp.HelmholtzSolver(n, b, omega, 100.0, c_mat).setup_preconditioner()
    assert s.multi_max == 8 and s.multi_kernel(8) == 2, s.layout()
    g = torch.Generator(device="cuda").manual_seed(1)
    xs = [torch.randn(n * n, dtype=torch.complex128, device="cuda", generator=g) for _ in range(8)]

    bufs = [x.clone() for x in xs]                          # every launch starts from the same fields

    def sweeps(slots):
        for u, x in zip(bufs, xs):
            u.copy_(x)
        slots = [None if t is None else bufs[r] for r, t in enumerate(slots)]
        s.sweep_forward_multi_buf(slots, 0, b + 1, n - 1)
        s.sweep_backward_multi_buf(slots, 0, n, b + 1)

    def single():
        bufs[0].copy_(xs[0])
        s.sweep_forward_buf(bufs[0], 0, b + 1, n - 1)
        s.sweep_backward_buf(bufs[0], 0, n, b + 1)

    def masked(k):
        return lambda: sweeps([x if r < k else None for r, x in enumerate(xs)])

    cfgs = {"hp_sweep4d, 8 active": (masked(8), None)}
    if not a.all_active_only:
        cfgs.update({"hp_sweep4d, 7 active": (masked(7), None), "hp_sweep4d, 4 active": (masked(4), None),
                     "hp_sweep4d, 1 active": (masked(1), None)})
    cfgs["hp_sweep4m, RT 8"] = (lambda: sweeps(xs), "no_dmma")
    cfgs["hp_sweep4m, RT 4"] = (lambda: sweeps(xs[:4]), None)
    cfgs["hp_sweep4m, RT 2"] = (lambda: sweeps(xs[:2]), None)
    cfgs["single-vector hp_sweep4"] = (single, None)
    times = {k: [] for k in cfgs}
    for rep in range(a.reps + 1):                            # repetition 0 warms every configuration up
        for name, (fn, env) in cfgs.items():
            if env:
                os.environ["HP_NO_DMMA"] = "1"
            try:
                ms, cnt = profile_ms(s, fn)
            finally:
                os.environ.pop("HP_NO_DMMA", None)
            assert cnt == 2, (name, cnt)
            if rep:
                times[name].append(ms)
    assert s.sweep_status() == 0
    s.close()
    return {"n": n, "b": b, "reps": a.reps, "unit": "ms per sweep launch (mean of forward and backward, all strips)",
            "launches": {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))} for k, v in times.items()}}


def part_solves(a):
    out = []
    for n, front, const in ((4096, "coupled", 100.0), (1024, "blockdiag", 100.0)):
        b = 12
        wave_num, alpha = n / 10, 2.0
        omega = 2 * np.pi * wave_num + 1j * alpha
        c_mat, _ = hp.init_layered_f1(omega, n)
        s = hp.HelmholtzSolver(n, b, omega, const, c_mat).setup_preconditioner(front=front)
        fs = [hp.init_f1_mat(r1, r2, omega, n) for r1, r2 in SHOTS]
        kw = dict(c_mat=c_mat, solver=s, diag="paper", precond_input="vector", rtol=1e-3, verbose=False)
        args = (n, b, wave_num, const, alpha)
        hp.run_solver(*args, f_mat=fs[0], **kw)              # warm-up of every kernel and of the allocator
        hp.run_solver_many(*args, fs[:8], **kw)
        rows = []
        for S in (1, 3, 7, 8, 12):
            torch.cuda.synchronize()
            t = time.perf_counter()
            many = hp.run_solver_many(*args, fs[:S], **kw)
            t_many = time.perf_counter() - t
            t = time.perf_counter()
            singles = [hp.run_solver(*args, f_mat=f, **kw) for f in fs[:S]]
            t_single = time.perf_counter() - t
            vec = DeviceVectors(n * n, s.device, restart=20)
            bs = [torch.from_numpy(np.ascontiguousarray(f, dtype=np.complex128).ravel()).cuda() for f in fs[:S]]
            torch.cuda.synchronize()
            t = time.perf_counter()
            res = gmres_batch(lambda x, o: s.matvec(x, o), lambda reqs: s.precond_apply_batch(reqs, diag="paper"), bs, vec=vec,
                              rtol=1e-3, restart=20, health=s.check_status)
            s.check_status()
            t_batch = time.perf_counter() - t
            rows.append({"S": S, "run_solver_many_s": t_many, "S_x_run_solver_s": t_single, "gmres_batch_unpadded_s": t_batch,
                         "niter": [r.niter for r in many], "niter_run_solver": [r.niter for r in singles],
                         "niter_gmres_batch": [len(h) for _, _, h in res], "info": [r.info for r in many]})
            print(json.dumps({"n": n, "front": front, **rows[-1]}), flush=True)
            del many, singles, res, bs
        s.close()
        torch.cuda.empty_cache()
        out.append({"n": n, "b": b, "front": front, "diag": "paper", "model": "layered", "wave_num": wave_num, "const": const,
                    "rows": rows})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--part", default="all", choices=["launches", "solves", "all"])
    ap.add_argument("--all-active-only", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--tag", default="")
    a = ap.parse_args()
    hp.load()
    if not torch.cuda.is_available():
        raise hp.HelmholtzB200Error("sources_time.py needs a CUDA device")
    res = {"gpu": gpu_info(), "tag": a.tag}
    if a.part in ("launches", "all"):
        res["launches"] = part_launches(a)
        print(json.dumps(res["launches"]), flush=True)
    if a.part in ("solves", "all"):
        res["solves"] = part_solves(a)
    os.makedirs(a.out, exist_ok=True)
    name = f"sources_time_{a.part}{'_' + a.tag if a.tag else ''}.json"
    with open(os.path.join(a.out, name), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
