#!/usr/bin/env python
"""Bench lines of the hidden-Markov row over many independent sequences (`lengths=`), each next to the single-sequence
line it is compared with, timed in the same process with the same method.

    python tools/bench_hmm_seqs.py [--config m1 m2 m3] [--steps K] [--warmup W]

One "step" = one VB iteration with x resident in HBM (bgmm_hmm_pass_seqs + bgmm_hmm_small; the h-lines bgmm_hmm_pass +
bgmm_hmm_small), timed with CUDA events.  The data is tools/bench_hmm.py's sticky-chain generator with a forced jump at
every sequence start, seeded.  For m1 / h1 the Viterbi decode (emission densities + recursion + back-tracking + the
path copied to the host) is timed too.  Every line records the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {  # name: (lengths(seed), D, K, single-sequence config it is compared with)
    "m1": (lambda rng: np.full(4096, 1024), 8, 8, "h1"),
    "m2": (lambda rng: rng.integers(1, 2001, size=1000), 16, 32, "h2"),
    "m3": (lambda rng: np.full(100_000, 40), 2, 3, "h3"),
}
SINGLE = {"h1": (4_000_000, 8, 8), "h2": (1_000_000, 16, 32), "h3": (4_000_000, 2, 3)}


def synth(lengths, d, k, seed, stay=0.95):
    """tools/bench_hmm.py synth_host, with a jump (a fresh state) at every sequence start."""
    n = int(np.sum(lengths))
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, 4.0, size=(k, d))
    jump = rng.random(n) > stay
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    jump[starts] = True
    nxt = rng.integers(0, k, size=n)
    last = np.maximum.accumulate(np.where(jump, np.arange(n), 0))
    return mu[nxt[last]] + rng.normal(size=(n, d)), starts


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001 — the measurement stands; say what is unknown
        return {"name": None, "power_limit": None, "error": str(e)}


def time_fit(x, starts, d, k, steps, warmup, viterbi_reps=0):
    import torch
    from bayesml_b200 import _lib
    from bayesml_b200.engine import HMMEngine
    dev = torch.device("cuda:0")
    eng = HMMEngine(k, d, device=dev)
    eng.load_data(torch.as_tensor(x).to(dev))
    eng.set_sequences(starts)
    eye = np.tile(np.eye(d), (k, 1, 1))
    eng.set_hmm_prior(np.full(k, .5), np.full((k, k), .5), np.zeros((k, d)), np.ones(k), np.full(k, float(d)), eye,
                      np.zeros(k), 0.0, 0.0)
    rng = np.random.default_rng(0)
    xh = x[:200_000]
    sub = int(np.sqrt(x.shape[0]))
    m0 = np.stack([xh[rng.choice(len(xh), sub, replace=False)].mean(axis=0) for _ in range(k)])
    cov = np.cov(xh.T).reshape(d, d)
    eng.set_hmm_params(np.full(k, .5), np.full((k, k), .5), m0, np.ones(k), np.full(k, float(d)),
                       np.tile(cov * d + 1e-5 * np.eye(d), (k, 1, 1)))
    eng._alloc_state(steps + warmup + 2)

    def step():
        eng._pass()
        eng._small(_lib.SMALL_ITERATE, 10 ** 6, 0.0)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    l0 = eng.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    out = {"ms_per_step": e0.elapsed_time(e1) / steps, "gpu_launches": eng.kernel_launches - l0,
           "window": eng.fetch_params()["window"]}
    hist = eng.state[eng.off["vlhist"]:eng.off["vlhist"] + steps + warmup].cpu().numpy()
    out["elbo_finite"] = bool(np.all(np.isfinite(hist)))
    if viterbi_reps:
        p = eng.fetch_params()
        lnpi, lna = p["e_ln_pi"], p["ln_a_tilde"]
        eng.viterbi(lnpi, lna)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(viterbi_reps):
            eng.viterbi(lnpi, lna)
        e1.record()
        torch.cuda.synchronize()
        out["viterbi_ms"] = e0.elapsed_time(e1) / viterbi_reps
        out["viterbi_us_per_element"] = 1e3 * out["viterbi_ms"] / x.shape[0]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", nargs="+", default=sorted(CONFIGS), choices=sorted(CONFIGS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_hmm_seqs.py needs a CUDA device")
    info = card()
    for name in args.config:
        mk, d, k, hname = CONFIGS[name]
        lengths = mk(np.random.default_rng(17))
        x, starts = synth(lengths, d, k, 4321)
        n = x.shape[0]
        vit = 3 if name == "m1" else 0
        r = time_fit(x, starts, d, k, args.steps, args.warmup, viterbi_reps=vit)
        print(json.dumps({"config": name, "workload": f"HMM VB, {len(lengths)} sequences (lengths {int(np.min(lengths))}.."
                          f"{int(np.max(lengths))}), N={n} D={d} K={k} float64, 1 GPU", "n": n, "n_seqs": len(lengths),
                          "value": n * k / (r["ms_per_step"] * 1e-3), "unit": "element*states/s", "steps": args.steps,
                          "warmup": args.warmup, "card": info, **r}), flush=True)
        del x
        hn, hd, hk = SINGLE[hname]
        xh, _ = synth(np.array([hn]), hd, hk, 4321)
        r = time_fit(xh, None, hd, hk, args.steps, args.warmup, viterbi_reps=vit)
        print(json.dumps({"config": hname, "compared_with": name, "workload": f"HMM VB, one sequence N={hn} D={hd} K={hk} "
                          "float64, 1 GPU", "n": hn, "n_seqs": 1, "value": hn * hk / (r["ms_per_step"] * 1e-3),
                          "unit": "element*states/s", "steps": args.steps, "warmup": args.warmup, "card": info, **r}),
              flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
