"""Inversion at 4096^2 on one GPU: the layered model attenuated with q = 50, b = 12, coupled front, paper diagonal, 8 shots
and 256 receivers on a line.  Measures with CUDA events over many launches
- hp_grad_accumulate and hp_born_source at R = 8, as GB/s against their byte models ((2R+2) and (2R+1) x 16 B per point,
  17 and 16 distinct fields of 268 MB, far larger than the L2), and hp_grad_finish;
and the wall time of one misfit_gradient call (rtol 1e-6), split into forward solves, adjoint solves and the rest
(sampling, injection and the gradient kernels).  Prints one JSON object and writes it to --out when given.  Needs a CUDA
device; the card name and its power limit are read in the same run.

    python tools/gradient_time.py [--n 4096] [--reps 40] [--out results.json]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import helmholtz_preconditioner_b200 as hp  # noqa: E402
from helmholtz_preconditioner_b200 import _lib  # noqa: E402
from tools.medium_time import card  # noqa: E402

SHOTS = [(0.5, 0.125), (0.2, 0.3), (0.8, 0.3), (0.35, 0.6), (0.65, 0.6), (0.5, 0.85), (0.15, 0.8), (0.85, 0.8)]
HBM_MEASURED_GB_S = 6537.0          # DESIGN.md: the streaming rate measured on a B200


def event_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gradient_time.py needs a CUDA device")
    n, b, const, alpha = args.n, 12, 100.0, 2.0
    wn = n / 10
    omega = 2 * np.pi * wn + 1j * alpha
    c = hp.attenuate(hp.init_layered_f1(omega, n)[0], 50.0)
    res = {"n": n, "b": b, "card": card(), "kernels": {}}
    t0 = time.perf_counter()
    s = hp.HelmholtzSolver(n, b, omega, const, c).setup_preconditioner(front="coupled")
    torch.cuda.synchronize()
    res["create_and_setup_s"] = time.perf_counter() - t0
    st = torch.cuda.current_stream().cuda_stream
    N, R = n * n, 8
    g = torch.Generator(device="cuda").manual_seed(5)
    xs = [torch.randn(N, dtype=torch.complex128, device="cuda", generator=g) for _ in range(2 * R + 1)]
    us, mus, acc = xs[:R], xs[R:2 * R], xs[2 * R]
    outs = [torch.empty_like(acc) for _ in range(R)]
    dk = torch.randn(n + 2, n + 2, dtype=torch.complex128, device="cuda", generator=g)
    grad = torch.empty(n + 2, n + 2, dtype=torch.complex128, device="cuda")
    pu, pm, po = s._ptr_array(us), s._ptr_array(mus), s._ptr_array(outs)

    def run_acc():
        _lib.check(s.lib.hp_grad_accumulate(s.handle, R, pu, pm, acc.data_ptr(), st), "hp_grad_accumulate")

    def run_born():
        _lib.check(s.lib.hp_born_source(s.handle, R, dk.data_ptr(), pu, po, st), "hp_born_source")

    def run_finish():
        _lib.check(s.lib.hp_grad_finish(s.handle, acc.data_ptr(), 1, grad.data_ptr(), st), "hp_grad_finish")

    for name, fn, bpp in (("hp_grad_accumulate_R8", run_acc, (2 * R + 2) * 16), ("hp_born_source_R8", run_born, (2 * R + 1) * 16),
                          ("hp_grad_finish_velocity", run_finish, 48)):
        ms = event_ms(fn, args.reps)
        gbs = bpp * N / ms / 1e6
        res["kernels"][name] = {"ms": ms, "bytes_per_point": bpp, "GB_s": gbs, "of_measured_stream": gbs / HBM_MEASURED_GB_S}
    del xs, us, mus, outs, pu, pm, po
    torch.cuda.empty_cache()

    fs = np.stack([np.asarray(hp.init_f1_mat(p[0], p[1], omega, n), dtype=np.complex128) for p in SHOTS])
    i = np.linspace(1, n, 256).round().astype(np.int64)
    rec = hp.Receivers(n, i, np.full(256, round(0.2 * (n + 1))))
    d_obs = np.zeros((len(SHOTS), 256), dtype=np.complex128)
    for k in range(2):                      # the first call warms up the allocator and the GMRES buffers
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = hp.misfit_gradient(s, fs, rec, d_obs, wrt="velocity", rtol=1e-6)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    res["misfit_gradient"] = {"wall_s": wall, "split_s": r.times, "forward_niter": r.forward_niter,
                              "adjoint_niter": r.adjoint_niter, "sources": len(SHOTS), "receivers": rec.nrec}
    s.close()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
