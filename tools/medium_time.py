"""Real against attenuating (complex) medium at 4096^2, layered, b = 12, on one GPU: whole-grid SpMV time and bandwidth,
preconditioner setup time, and GMRES iterations / solve time of the lossless model and of fields.attenuate(c, q) for
q = 50 and q = 10 (diag='paper', front='coupled', precond_input='vector').  Prints one JSON object and writes it to
--out when given.  Needs a CUDA device; the card name and its power limit are read in the same run.

    python tools/medium_time.py [--n 4096] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import helmholtz_preconditioner_b200 as hp  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def spmv_ms(s, n, reps=60):
    """mean time of one whole-grid SpMV over 3 rotating inputs (268 MB each at 4096^2, larger than the L2)"""
    g = torch.Generator(device="cuda").manual_seed(3)
    xs = [torch.randn(n * n, dtype=torch.complex128, device="cuda", generator=g) for _ in range(3)]
    ys = [torch.empty_like(x) for x in xs]
    for i in range(6):
        s.matvec(xs[i % 3], ys[i % 3])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        s.matvec(xs[i % 3], ys[i % 3])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("medium_time.py needs a CUDA device")
    n, b, const, alpha = args.n, 12, 100.0, 2.0
    wn = n / 10                                           # 10 points per wavelength, as bench.py
    omega = 2 * np.pi * wn + 1j * alpha
    c_real, f_mat = hp.init_layered_f1(omega, n)
    res = {"n": n, "b": b, "card": card(), "spmv": {}, "setup": {}, "gmres": {}}
    models = {"real": c_real, "complex_q50": hp.attenuate(c_real, 50.0), "complex_q10": hp.attenuate(c_real, 10.0),
              "complex_lossless": c_real + 0j}
    for name in ("real", "complex_lossless", "complex_q50", "complex_q10"):
        c = models[name]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s = hp.HelmholtzSolver(n, b, omega, const, c)
        s.setup_preconditioner(front="coupled")
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        assert s.medium_is_complex == (name != "real")
        if name in ("real", "complex_lossless"):
            ms = spmv_ms(s, n)
            nbytes = (40 if name == "real" else 48) * n * n
            res["spmv"][name] = {"ms": ms, "bytes_per_point": nbytes // (n * n), "GB_s": nbytes / ms / 1e6}
            res["setup"][name] = {"setup_ms": s.setup_ms, "create_and_setup_wall_s": wall}
        if name != "complex_lossless":
            r = hp.run_solver(n, b, wn, const, alpha, c_mat=c, f_mat=f_mat, solver=s, diag="paper",
                              precond_input="vector", maxiter=100, verbose=False)
            res["gmres"][name] = {"niter": r.niter, "info": r.info, "solve_s": r.solve_time}
        s.close()
        del s
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
