#!/usr/bin/env python
"""Time `hiddenmarkovnormal.GenModel.gen_sample(..., device=..., as_numpy=False)` (bgmm_hmm_gen_sample) and the host loop.

    python tools/bench_hmm_gen.py [--config h1 h2 h3 m1 m2 m3 host] [--reps R] [--warmup W] [--out DIR]

h1/h2/h3 are single chains at the shapes of tools/bench_hmm.py, m1/m2/m3 the `lengths` mixes of tools/bench_hmm_seqs.py;
the model has a sticky random A and well separated means (seeded).  Each device call is timed with CUDA events after
`warmup` untimed calls of the same shape; the call includes the upload of the K-sized tables, the workspace allocation
and the stream synchronisation that `as_numpy=False` performs.  "host" is the reference's per-element loop
(`gen_sample` without `device`) on 2 000 elements, timed with the host clock.  Every line records the card's name and
power limit; with --out each line is also written to DIR/r04_bench_hmm_gen_<config>.json.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_hmm_seqs import CONFIGS as SEQ_CONFIGS, SINGLE, card  # noqa: E402

HOST_N = 2000


def model(d, k, seed=4321, stay=0.95):
    from bayesml_b200 import hiddenmarkovnormal
    rng = np.random.default_rng(seed)
    a = np.full((k, k), (1.0 - stay) / max(k - 1, 1)) if k > 1 else np.ones((1, 1))
    if k > 1:
        a[np.arange(k), np.arange(k)] = stay
    return hiddenmarkovnormal.GenModel(k, d, seed=seed, pi_vec=rng.dirichlet(np.ones(k)), a_mat=a,
                                       mu_vecs=rng.normal(0.0, 4.0, size=(k, d)))


def time_device(g, n, lengths, reps, warmup):
    import torch
    for _ in range(warmup):
        g.gen_sample(n, lengths=lengths, device="cuda:0", as_numpy=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0.record()
        g.gen_sample(n, lengths=lengths, device="cuda:0", as_numpy=False)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return {"ms_per_call": float(np.median(times)), "ms_min": float(np.min(times)), "ms_max": float(np.max(times))}


def main():
    ap = argparse.ArgumentParser()
    names = sorted(SINGLE) + sorted(SEQ_CONFIGS) + ["host"]
    ap.add_argument("--config", nargs="+", default=names, choices=names)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_hmm_gen.py needs a CUDA device")
    info = card()
    for name in args.config:
        if name == "host":
            g = model(8, 8)
            t0 = time.perf_counter()
            g.gen_sample(HOST_N)
            dt = time.perf_counter() - t0
            line = {"config": "host", "workload": f"host loop, one sequence N={HOST_N} D=8 K=8", "n": HOST_N,
                    "us_per_element": 1e6 * dt / HOST_N, "elements_per_s": HOST_N / dt}
        else:
            if name in SINGLE:
                n, d, k = SINGLE[name]
                lengths = None
            else:
                mk, d, k, _ = SEQ_CONFIGS[name]
                lengths = np.asarray(mk(np.random.default_rng(17)), dtype=np.int64)
                n = int(lengths.sum())
            r = time_device(model(d, k), n, lengths, args.reps, args.warmup)
            line = {"config": name, "workload": f"GenModel.gen_sample on the device, N={n} D={d} K={k}, "
                    f"{1 if lengths is None else len(lengths)} sequence(s)", "n": n,
                    "n_seqs": 1 if lengths is None else len(lengths), "reps": args.reps, "warmup": args.warmup,
                    "elements_per_s": n / (r["ms_per_call"] * 1e-3), **r}
        line["card"] = info
        text = json.dumps(line)
        print(text, flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r04_bench_hmm_gen_{name}.json"), "w") as f:
                f.write(text + "\n")
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
