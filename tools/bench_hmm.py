#!/usr/bin/env python
"""Bench line of the hidden-Markov row (SURVEY.md §8 f1) — same JSON shape as bench.py, which stays the contract bench.

    python tools/bench_hmm.py [--config h1|h2|h3] [--steps K] [--warmup W] [--impl reference]

One "step" = one VB iteration of `hiddenmarkovnormal.LearnModel.update_posterior` (_hiddenmarkovnormal.py:1104-1113):
M-steps of q(mu, Lambda), q(pi), q(A); emission densities; forward / backward recursions; gamma, xi; statistics; ELBO +
convergence test.  On the device: bgmm_hmm_pass + bgmm_hmm_small (`gpu_launches` / `steps` kernels per step, as counted
by libbgmm).  Synthetic sticky-chain data with Gaussian emissions; the sequence is larger than L2, so every iteration
streams it from HBM.

`value` = N*K element*states per second with x resident in HBM; `e2e` = the same through the public API with a HOST
array; `cpu_baseline` = the numpy oracle port of the reference's sequential recursions on a bounded sample.
The algorithmic flop count is the reference's own: E 2D^2+2D and M 2D^2+2D+1 per (element, state) as for the mixture,
forward 2K^2, backward 2K^2, xi 3K^2 per element.  The parallel scan executes K x more in its basis phase (N K^3);
that overhead is NOT counted as useful work.
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ClockSampler, blas_threads, load_peaks  # noqa: E402
FP64_PEAK_TFLOPS = load_peaks()["fp64_tflops"]

METRIC = "VB iters/sec (N*K elements*states/s) HMM"
UNIT = "element*states/s"
CONFIGS = {"h1": (4_000_000, 8, 8), "h2": (1_000_000, 16, 32), "h3": (4_000_000, 2, 3)}


def alg_flops(n, d, k):
    return n * k * (4 * d * d + 4 * d + 1) + n * 7 * k * k


def synth_host(n, d, k, seed, stay=0.95):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, 4.0, size=(k, d))
    jump = rng.random(n) > stay
    jump[0] = True
    nxt = rng.integers(0, k, size=n)
    last = np.maximum.accumulate(np.where(jump, np.arange(n), 0))
    return mu[nxt[last]] + rng.normal(size=(n, d))


def synth_device(n, d, k, seed, device, stay=0.95):
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    mu = torch.randn(k, d, generator=g, device=device, dtype=torch.float64) * 4.0
    jump = torch.rand(n, generator=g, device=device) > stay
    nxt = torch.randint(0, k, (n,), generator=g, device=device)
    idx = torch.where(jump, torch.arange(n, device=device), torch.zeros(n, dtype=torch.long, device=device))
    z = nxt[torch.cummax(idx, 0).values]
    return mu[z] + torch.randn(n, d, generator=g, device=device, dtype=torch.float64)


def oracle_rate(n_total, d, k, rows, iters=2):
    from oracle.hmm_vb_oracle import OracleHMM
    n = min(n_total, rows)
    x = synth_host(n, d, k, 99)
    m = OracleHMM(k, d, seed=0)
    m.alloc(n)
    m.init_fb_params(); m.reset_hn(); m.init_subsampling(x); m.e_step(x); m.calc_vl()
    t0 = time.perf_counter()
    for _ in range(iters):
        m.iterate(x)
    dt = (time.perf_counter() - t0) / iters
    return n * k / dt, n, dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="h1", choices=sorted(CONFIGS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    args = ap.parse_args()
    n, d, k = CONFIGS[args.config]
    workload = f"{args.config}: HMM (Gaussian emissions) VB, one sequence N={n} D={d} K={k} float64, 1 GPU"

    if args.impl == "reference":
        rate, rows, dt = oracle_rate(n, d, k, 30_000, iters=max(1, min(args.steps, 3)))
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": 1,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt, "higher_is_better": True,
                          "dtype": "f64", "data": "synthetic", "vs_baseline": None,
                          "config": {"workload": workload + f" (timed on a bounded sample of N={rows})"},
                          "cpu_baseline": {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                                           "sample": f"numpy oracle port (oracle/hmm_vb_oracle.py), N={rows}; the "
                                                     "recursions are a Python loop over the sequence, as in the reference"},
                          "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return

    import torch
    from bayesml_b200 import _lib, hiddenmarkovnormal
    from bayesml_b200.engine import HMMEngine
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    x = synth_device(n, d, k, 4321, dev)
    eng = HMMEngine(k, d, device=dev)
    eng.load_data(x)
    eye = np.tile(np.eye(d), (k, 1, 1))
    eng.set_hmm_prior(np.full(k, .5), np.full((k, k), .5), np.zeros((k, d)), np.ones(k), np.full(k, float(d)), eye,
                      np.zeros(k), 0.0, 0.0)
    xh = x[:200_000].cpu().numpy()
    rng = np.random.default_rng(0)
    sub = int(np.sqrt(n))
    m0 = np.stack([xh[rng.choice(len(xh), sub, replace=False)].mean(axis=0) for _ in range(k)])
    cov = np.cov(xh.T).reshape(d, d)
    eng.set_hmm_params(np.full(k, .5), np.full((k, k), .5), m0, np.ones(k), np.full(k, float(d)),
                       np.tile(cov * d + 1e-5 * np.eye(d), (k, 1, 1)))
    total = args.steps + args.warmup
    eng._alloc_state(total + 2)

    def step():
        eng._pass()
        eng._small(_lib.SMALL_ITERATE, 10 ** 6, 0.0)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    launches0 = eng.kernel_launches
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = eng.kernel_launches - launches0
    t_end = time.perf_counter() + 1.0          # keep the GPU busy so the sampler sees clocks under load
    while time.perf_counter() < t_end:
        step()
        torch.cuda.synchronize()
    clocks = sampler.stop()
    hist = eng.state[eng.off["vlhist"]:eng.off["vlhist"] + total].cpu().numpy()
    value = n * k / (ms * 1e-3)
    flops = alg_flops(n, d, k)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "replicas only", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload,
                   "l2": f"per-element arrays {n * (d + 5 * k) * 8 / 2 ** 20:.0f} MB per iteration (> 126 MB L2), no flush needed"},
        "elbo_finite_and_monotone": bool(np.all(np.isfinite(hist)) and np.all(np.diff(hist[1:]) > -1e-6 * np.abs(hist[1:-1]))),
        "gpu_launches": launches, "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                     "frac": flops / (ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS, "traffic": None,
                     "note": "whole iteration against the FP64 pipe peak (DFMA = DMMA rate); algorithmic flops = the "
                             "reference's sequential count, the scan's K-fold basis phase is not counted as useful work"},
    }
    if not args.no_e2e:
        xhost = x.cpu().numpy()
        model = hiddenmarkovnormal.LearnModel(k, d, seed=0)
        iters = 10
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.update_posterior(xhost[: n // 8], max_itr=2, num_init=1, tolerance=0.0)      # warm-up (allocator, JIT-free)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.update_posterior(xhost, max_itr=iters, num_init=1, tolerance=0.0)
            _ = float(model.vl)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        line["e2e"] = {"value": n * k * (iters + 2) / dt, "unit": UNIT, "h2d_bytes_per_step": n * d * 8 // (iters + 2),
                       "d2h_bytes_per_step": 8 * (iters + 1) // (iters + 2), "seconds": dt,
                       "note": f"LearnModel.update_posterior(host x, max_itr={iters}, num_init=1, tolerance=0): "
                               f"{iters + 2} E-steps (post-init, {iters} iterations, final) incl. upload, init, final pass"}
    rate, rows, dt_cpu = oracle_rate(n, d, k, 30_000)
    line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "host_threads_blas": blas_threads(), "kind": "port",
                            "s_per_iter_at_sample": dt_cpu,
                            "sample": f"numpy oracle port (oracle/hmm_vb_oracle.py), N={rows} elements of the same workload; "
                                      "the recursions are a Python loop over the sequence, as in the reference; linear in N"}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
