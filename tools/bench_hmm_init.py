#!/usr/bin/env python
"""End-to-end `hiddenmarkovnormal.LearnModel.update_posterior(x, init_type='random_responsibility')` with the initial
state drawn on the host (the default) and on the device (`device_init=True`), timed in the same process.

    python tools/bench_hmm_init.py [--config h1 h2 h3 m1 m3] [--reps R] [--out DIR]

h1/h2/h3 are the single sequences of tools/bench_hmm.py, m1/m3 the `lengths` mixes of tools/bench_hmm_seqs.py, with that
file's seeded sticky-chain data.  Per config, after one untimed warm-up fit:
  - `e2e_s`: wall time of whole `update_posterior` calls (default max_itr and tolerance), the host clock around work that
    ends in a device synchronise: device_init with num_init 1 and 10, host draw with num_init 1.  Ten host restarts are
    not run (minutes at h2): the per-restart host cost is `host_draw_s`, one `_init_random_responsibility` call timed
    alone with the host clock.
  - `device_draw_ms`: bgmm_hmm_init_random alone (`HMMEngine.draw_random_init`), CUDA events around each of `reps` calls
    after warm-up calls; median, min and max.
Every line records the card's name and power limit; with --out each line is also written to
DIR/r05_bench_hmm_init_<config>.json.
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

from tools.bench_hmm_seqs import CONFIGS as SEQ_CONFIGS, SINGLE, card, synth  # noqa: E402

NAMES = ("h1", "h2", "h3", "m1", "m3")


def shape(name):
    """-> (lengths or None, n, D, K)."""
    if name in SINGLE:
        n, d, k = SINGLE[name]
        return None, n, d, k
    mk, d, k, _ = SEQ_CONFIGS[name]
    lengths = np.asarray(mk(np.random.default_rng(17)), dtype=np.int64)
    return lengths, int(lengths.sum()), d, k


def fit(x, lengths, d, k, device_init, num_init, max_itr=100):
    """-> (seconds, model) of one update_posterior call, synchronised at both ends."""
    import torch
    from bayesml_b200 import hiddenmarkovnormal
    m = hiddenmarkovnormal.LearnModel(k, d, seed=1, device_init=device_init)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.update_posterior(x, max_itr=max_itr, num_init=num_init, init_type="random_responsibility",
                           lengths=None if lengths is None else lengths.tolist())
    torch.cuda.synchronize()
    return time.perf_counter() - t0, m


def time_draw(eng, reps):
    import torch
    for s in range(3):
        eng.draw_random_init(s)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    times = []
    for s in range(reps):
        e0.record()
        eng.draw_random_init(100 + s)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return {"median": float(np.median(times)), "min": float(np.min(times)), "max": float(np.max(times))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", nargs="+", default=list(NAMES), choices=NAMES)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_hmm_init.py needs a CUDA device")
    from bayesml_b200 import hiddenmarkovnormal
    info = card()
    for name in args.config:
        lengths, n, d, k = shape(name)
        x, starts = synth(np.array([n]) if lengths is None else lengths, d, k, 4321)
        starts = None if lengths is None else starts
        fit(x, lengths, d, k, True, 1, max_itr=2)                                     # warm-up
        dev1, m = fit(x, lengths, d, k, True, 1)
        draw = time_draw(m._engine(), args.reps)
        dev10, _ = fit(x, lengths, d, k, True, 10)
        host1, _ = fit(x, lengths, d, k, False, 1)
        t0 = time.perf_counter()
        hiddenmarkovnormal.LearnModel(k, d, seed=2)._init_random_responsibility(n, starts)
        host_draw = time.perf_counter() - t0
        line = {"config": name, "workload": f"HMM update_posterior, init_type='random_responsibility', N={n} D={d} K={k} "
                f"float64, {1 if lengths is None else len(lengths)} sequence(s), max_itr=100, tolerance=1e-8, 1 GPU",
                "n": n, "n_seqs": 1 if lengths is None else len(lengths),
                "e2e_s": {"device_init_num_init_1": dev1, "device_init_num_init_10": dev10, "host_init_num_init_1": host1,
                          "host_init_num_init_10": "not measured: ten host restarts take minutes at h2; the per-restart "
                                                   "host cost is host_draw_s"},
                "host_draw_s": host_draw, "device_draw_ms": draw, "reps": args.reps, "card": info}
        text = json.dumps(line)
        print(text, flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r05_bench_hmm_init_{name}.json"), "w") as f:
                f.write(text + "\n")
        del x
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
