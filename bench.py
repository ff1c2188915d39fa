#!/usr/bin/env python
"""bench.py — VB Gaussian-mixture hot path on B200: VB iterations/s as N*K point*components per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2] [--scaling strong|weak] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one VB iteration of `gaussianmixture.LearnModel.update_posterior` (reference
_gaussianmixture.py:863-869): M-step + q(pi) update + E-step/statistics pass over all rows + ELBO + convergence
test.  On the device that is: bgmm_pass (the fused E/statistics sweep) -> [all-reduce of the statistics when
N > 1] -> bgmm_small (ELBO, convergence flag, M-step).  Workload: BASELINE.json configs[1]
(N=10M, D=16, K=32, fp64) on synthetic mixture data (SURVEY.md §8d); X (1.28 GB) is larger than L2 so every
timed iteration streams it from HBM.

Printed JSON keys follow the driver contract; `value` is whole-job throughput with X resident in HBM, `e2e` is
the same metric through the public API (`LearnModel.update_posterior`) with a HOST array, uploads/downloads
inside the timed region.  `--impl reference` times the UNMODIFIED reference class (`bayesml.gaussianmixture.LearnModel`
from the oracle/_ref archive that oracle/build_ref.py packs from /root/reference; the numpy oracle port only if that
archive is missing) on the host cores, on a bounded sample of the same workload.
"""
import argparse
import atexit
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as the build left it (it may be read-only)

METRIC = "VB iters/sec (N*K points*comps/s) GMM"
UNIT = "point*comps/s"

# name -> (N_total, D, K, precision, config index for the data seed)
CONFIGS = {
    "c1": (1000, 2, 3, "float64", 0),
    "c2": (10_000_000, 16, 32, "float64", 1),
    "c2f32": (10_000_000, 16, 32, "float32", 1),      # the C2 workload in fp32 mode: the tcgen05 kind::tf32 kernels
    "c3": (200_000_000, 2, 8, "float32", 2),
    "c4": (2_000_000, 128, 64, "float64", 3),
    "c5": (4_000_000, 32, 16, "float64", 4),
}
PEAKS_FILE = os.path.join(ROOT, "profiles", "peaks_b200.json")   # tracked: tools/peaks microbenchmarks on this pool's B200


def load_peaks():
    """FP64 / FP32 pipe peaks from the tracked measurement (MEASURED_PEAKS.json, driver-written, has HBM and bf16 only)."""
    with open(PEAKS_FILE) as f:
        p = json.load(f)
    return {"fp64_tflops": float(p["dmma_tflops"]), "fp32_tflops": float(p["ffma2_tflops"]),
            "source": "profiles/peaks_b200.json (tools/peaks on this pool's B200: DMMA %.1f, DFMA %.1f, cuBLAS DGEMM %.1f, "
                      "FFMA2 %.1f TFLOP/s); MEASURED_PEAKS.json has no FP64 / FP32 entry"
                      % (p["dmma_tflops"], p["dfma_tflops"], p["dgemm_cublas_tflops"], p["ffma2_tflops"])}


def alg_flops_per_iter(n, d, k):
    """SURVEY.md §8d: dense forms the reference executes, E: 2D^2+2D, M: 2D^2+2D+1 per (sample, component)."""
    return n * k * (4 * d * d + 4 * d + 1)


def mixture_params(d, k, seed):
    rng = np.random.default_rng(seed)
    mu = rng.normal(0.0, 4.0, size=(k, d))
    a = rng.normal(size=(k, d, d))
    chol = np.linalg.cholesky(a @ a.transpose(0, 2, 1) / d + 0.5 * np.eye(d))
    return mu, chol


def synth_host(n, d, k, seed, sample_seed=0):
    """Seeded mixture sample on the host (numpy) — used by the CPU arms."""
    mu, chol = mixture_params(d, k, seed)
    rng = np.random.default_rng([seed, sample_seed])
    z = rng.integers(0, k, size=n)
    x = np.empty((n, d))
    step = 1 << 18
    for s in range(0, n, step):
        e = min(n, s + step)
        x[s:e] = mu[z[s:e]] + np.einsum("nij,nj->ni", chol[z[s:e]], rng.normal(size=(e - s, d)))
    return x


def synth_device(n, d, k, seed, sample_seed, device, dtype):
    """Same mixture, sampled on the device with torch (plumbing: data generation is not part of the path)."""
    import torch
    mu, chol = mixture_params(d, k, seed)
    mu_t = torch.as_tensor(mu, device=device)
    chol_t = torch.as_tensor(chol, device=device)
    g = torch.Generator(device=device)
    g.manual_seed(seed * 1000 + sample_seed)
    x = torch.empty((n, d), device=device, dtype=dtype)
    step = 1 << 20
    for s in range(0, n, step):
        e = min(n, s + step)
        z = torch.randint(0, k, (e - s,), generator=g, device=device)
        eps = torch.randn(e - s, d, generator=g, device=device, dtype=torch.float64)
        x[s:e] = (mu_t[z] + torch.einsum("nij,nj->ni", chol_t[z], eps)).to(dtype)
    return x


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)     # a run that fails before stop() must not leave the sampler running
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [v.strip() for v in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(names, f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_fit_time(x, k, d, max_itr):
    """(wall seconds, kind) of ONE CPU fit with exactly max_itr VB iterations (tolerance=0.0, num_init=1): the unmodified
    reference class `bayesml.gaussianmixture.LearnModel.update_posterior` when the oracle/_ref archive (or /root/reference)
    is there, else the numpy oracle port."""
    from oracle import ref_loader
    if ref_loader.reference_available():
        gm = ref_loader.load_reference_gaussianmixture()
        m = gm.LearnModel(k, d, seed=0)
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            t0 = time.perf_counter()
            m.update_posterior(x, max_itr=max_itr, num_init=1, tolerance=0.0)
            return time.perf_counter() - t0, "reference"
    from oracle.gmm_vb_oracle import OracleGMM, fit
    m = OracleGMM(k, d, seed=0)
    t0 = time.perf_counter()
    fit(m, x, max_itr=max_itr, num_init=1, tolerance=0.0)
    return time.perf_counter() - t0, "port"


def cpu_iteration_time(x, k, d, t_lo, t_hi):
    """Per-iteration wall time (T(max_itr=t_hi) - T(max_itr=t_lo)) / (t_hi - t_lo): initialisation, the post-init pass and
    the final E-step (:895) cancel."""
    a, kind = cpu_fit_time(x, k, d, t_lo)
    b, _ = cpu_fit_time(x, k, d, t_hi)
    return (b - a) / (t_hi - t_lo), kind


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(cfg, budget_rows=200_000):
    n_total, d, k, _, idx = CONFIGS[cfg]
    n = min(n_total, budget_rows)
    x = synth_host(n, d, k, 1234 + idx)
    per_iter, kind = cpu_iteration_time(x, k, d, 1, 3)
    what = ("the reference class bayesml.gaussianmixture.LearnModel.update_posterior (oracle/_ref archive)" if kind == "reference"
            else "numpy oracle port (oracle/gmm_vb_oracle.py)")
    return {"value": n * k / per_iter, "unit": UNIT, "cores": blas_threads(), "host_cpus": os.cpu_count(),
            "kind": kind, "s_per_iter_at_sample": per_iter,
            "sample": f"{what}, N={n} rows of the {cfg} workload (D={d}, K={k}), "
                      f"(T(max_itr=3)-T(max_itr=1))/2, tolerance=0.0, num_init=1; linear in N"}


def run_reference_arm(args):
    """The UNMODIFIED reference class on the host cores, through its own public API: two calls of
    `LearnModel.update_posterior(x, max_itr=T, num_init=1, tolerance=0.0)` with T = warmup and T = warmup + steps; the
    difference is exactly `steps` VB iterations (:863-869) — initialisation, post-init pass and final E-step cancel.
    Each step is a bounded sample of the workload (N rows of the same synthetic mixture), sized from a short calibration
    so that the whole run stays within a few minutes; the per-row cost of the reference is linear in N."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_total, d, k, _, idx = CONFIGS[args.config]
    t_lo, t_hi = max(args.warmup, 1), max(args.warmup, 1) + args.steps
    # calibration: one short fit on 50k rows -> rows * iterations per second of this host
    n_cal = min(n_total, 50_000)
    x = synth_host(n_cal, d, k, 1234 + idx)
    t_cal, kind = cpu_fit_time(x, k, d, 2)
    rate = n_cal * 4.0 / max(t_cal, 1e-3)                        # 2 iterations + post-init pass + final E-step
    budget_s = float(os.environ.get("BAYESML_B200_REF_BUDGET_S", "200"))
    n = int(min(n_total, max(20_000, budget_s * rate / (t_lo + t_hi + 4))))
    n = int(min(n, 1_000_000)) if n > 1_000_000 else n
    x = synth_host(n, d, k, 1234 + idx)
    per_iter, kind = cpu_iteration_time(x, k, d, t_lo, t_hi)
    value = n * k / per_iter
    what = ("reference class bayesml.gaussianmixture.LearnModel.update_posterior (unmodified, oracle/_ref archive)"
            if kind == "reference" else "numpy oracle port (oracle/gmm_vb_oracle.py; oracle/_ref archive missing)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * per_iter, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.config}: GMM VB N={n_total} D={d} K={k} (timed on a bounded sample of N={n} rows)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": blas_threads(), "host_cpus": os.cpu_count(),
                         "kind": kind,
                         "sample": f"{what}, N={n} rows, (T(max_itr={t_hi}) - T(max_itr={t_lo})) / {args.steps}, "
                                   f"tolerance=0.0, num_init=1"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def engine_outputs(eng, n_hist):
    """What one timed step hands its caller, read back after the step: the posterior hyperparameters the M-step produced
    (under LearnModel's attribute names), the statistics of the pass, the ELBO terms and the ELBO history of the run."""
    p = eng.fetch_params()
    o = eng.off["vlhist"]
    return {"hn_alpha_vec": p["alpha"], "hn_m_vecs": p["m"], "hn_kappas": p["kappa"], "hn_nus": p["nu"],
            "hn_w_mats": p["w"], "hn_w_mats_inv": p["winv"], "e_ln_pi_vec": p["e_ln_pi"],
            "e_ln_lambda_dets": p["e_ln_lambda_dets"], "ln_b_hn_w_nus": p["ln_b"], "ns": p["ns"], "x_bar_vecs": p["x_bar"],
            "s_mats": p["s_mats"], "vl_terms": p["vl_terms"], "vl_history": eng.state[o:o + n_hist].cpu().numpy()}


def dump_plan(eng, n_hist, count):
    """Which of `count` output sets shaped like `eng`'s (one per restart) --dump-outputs writes: all of them, or a fixed,
    seeded sample of them when all would exceed DUMP_LIMIT_BYTES.  Decided from shapes alone, before the timed steps, so
    every rank gets the same answer and an impossible dump fails before any timing."""
    one = sum(np.asarray(a, dtype=np.float64).nbytes for a in engine_outputs(eng, n_hist).values())
    fit = DUMP_LIMIT_BYTES // one
    if fit < 1:
        raise RuntimeError(f"--dump-outputs: one output set takes {one} bytes, over the {DUMP_LIMIT_BYTES}-byte limit")
    if count <= fit:
        return list(range(count))
    return sorted(np.random.default_rng(0).choice(count, size=fit, replace=False).tolist())


def dump_outputs(dirname, arrays):
    """Writes every array as DIR/<name>.npy in float64."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def _rel(a, b):
    """max element-wise relative error, entries below 1e-4 of the array's largest magnitude held to that floor."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    scale = float(np.max(np.abs(b))) if b.size else 0.0
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), max(scale * 1e-4, 1e-300)))) if b.size else 0.0


def parity_multi(world, rank, device, group):
    """Driver-visible multi-GPU parity (world > 1): a small fit with the rows sharded over all ranks — both
    initialisations, deliberately uneven shards — against the same fit on rank 0 alone and against the CPU oracle, plus
    one fit with the restarts spread over the ranks (`restart_group`) against the single-GPU restart loop.
    The oracle is the checker here, exactly as in tests/ (it never feeds the timed path)."""
    import hashlib
    import torch
    import torch.distributed as dist
    from bayesml_b200 import gaussianmixture
    n, d, k = 40_001, 16, 8
    rng = np.random.default_rng(17)
    x = rng.normal(size=(n, d)) + 4.0 * rng.integers(0, k, size=(n, 1)) * rng.normal(size=(1, d))
    cuts = np.linspace(0, n, world + 1).astype(int)
    cuts[1:-1] += (np.arange(1, world) % 2) * 357                # uneven shards
    fields = ("hn_alpha_vec", "hn_m_vecs", "hn_kappas", "hn_nus", "hn_w_mats_inv", "ns", "x_bar_vecs")
    out = {"max_rel": 0.0, "max_rel_vs_single_gpu": 0.0, "ranks_bit_identical": True, "cases": []}

    def quiet_fit(model, data, **kw):
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model.update_posterior(data, **kw)
        return model

    def digest(model):
        h = hashlib.sha256()
        for f in fields + ("hn_w_mats",):
            h.update(np.ascontiguousarray(getattr(model, f)).tobytes())
        h.update(np.float64(model.vl).tobytes())
        return torch.tensor(list(h.digest()[:8]), dtype=torch.int64, device=device)

    def same_on_all_ranks(model):
        dg = digest(model)
        lo, hi = dg.clone(), dg.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
        return bool(torch.equal(lo, hi))

    for init in ("subsampling", "random_responsibility"):
        kw = dict(max_itr=8, num_init=2, tolerance=0.0, init_type=init)
        sharded = quiet_fit(gaussianmixture.LearnModel(k, d, seed=5, device=device, process_group=group),
                            x[cuts[rank]:cuts[rank + 1]], **kw)
        identical = same_on_all_ranks(sharded)
        rec = {"case": f"rows sharded over {world} ranks, init_type={init}", "ranks_bit_identical": identical}
        if rank == 0:
            from oracle.gmm_vb_oracle import OracleGMM, fit
            single = quiet_fit(gaussianmixture.LearnModel(k, d, seed=5, device=device), x, **kw)
            o = OracleGMM(k, d, seed=5)
            fit(o, x, **kw)
            rec["max_rel_vs_oracle"] = max([_rel(getattr(sharded, f), getattr(o, f)) for f in fields] + [_rel(sharded.vl, o.vl)])
            rec["max_rel_vs_single_gpu"] = max([_rel(getattr(sharded, f), getattr(single, f)) for f in fields]
                                               + [_rel(sharded.vl, single.vl)])
            rec["r_rows_vs_oracle"] = _rel(sharded.r_vecs[:256], o.r_vecs[:256])
            out["max_rel"] = max(out["max_rel"], rec["max_rel_vs_oracle"], rec["r_rows_vs_oracle"])
            out["max_rel_vs_single_gpu"] = max(out["max_rel_vs_single_gpu"], rec["max_rel_vs_single_gpu"])
        out["ranks_bit_identical"] = out["ranks_bit_identical"] and identical
        out["cases"].append(rec)
        dist.barrier(group=group)
    # restarts spread over the ranks (x replicated): the selection must equal the sequential rule (:873-883)
    kw = dict(max_itr=25, num_init=2 * world + 1)
    spread = quiet_fit(gaussianmixture.LearnModel(k, d, seed=6, device=device, restart_group=group), x[:6001], **kw)
    identical = same_on_all_ranks(spread)
    rec = {"case": f"{kw['num_init']} restarts spread over {world} ranks (restart_group)", "ranks_bit_identical": identical}
    if rank == 0:
        single = quiet_fit(gaussianmixture.LearnModel(k, d, seed=6, device=device), x[:6001], **kw)
        rec["equal_to_sequential_restart_loop"] = bool(all(np.array_equal(getattr(spread, f), getattr(single, f)) for f in fields)
                                                       and float(spread.vl) == float(single.vl))
        out["restart_group_equals_sequential"] = rec["equal_to_sequential_restart_loop"]
    out["ranks_bit_identical"] = out["ranks_bit_identical"] and identical
    out["cases"].append(rec)
    dist.barrier(group=group)
    return out


def selection_follows_reference_rule(text):
    """The '*' marks of the progress text against the reference's rule (:873-883): restart i is kept iff it is the first
    one or its final VL is STRICTLY larger than the best so far.  -> (ok, index of the kept restart, number of restarts)."""
    import re
    best, kept, ok, n = None, -1, True, 0
    for line in text.split("\n"):
        vals = re.findall(r"VL: (-?[0-9.eE+-]+|nan|inf|-inf)", line)
        if not vals:
            continue
        vl = float(vals[-1])
        should = best is None or vl > best
        if should:
            best, kept = vl, n
        ok = ok and (line.rstrip().endswith("*") == should)
        n += 1
    return ok, kept, n


def bench_restarts(args, world, rank, local_rank, device, group):
    """`--restarts R` (BASELINE configs[4], C5): R restarts of the same fit, X replicated on every GPU, the restarts spread
    over the ranks and advanced `bgmm_batch_capacity` at a time by one shared sweep over X (bgmm_pass_batched).
    One step = one VB iteration (:863-869) of EVERY restart; value = R * N * K / step time.  No data-path collective:
    the only exchange is the all-gather of the finished restarts' records in `update_posterior` (e2e leg)."""
    import torch
    import torch.distributed as dist
    from bayesml_b200 import _lib, gaussianmixture
    from bayesml_b200.engine import RestartBatch, VBEngine
    n_total, d, k, precision, idx = CONFIGS[args.config]
    assert precision == "float64"
    warmup = max(args.warmup, 3)
    r_total = args.restarts
    mine = [i for i in range(r_total) if i % world == rank]
    x_dev = synth_device(n_total, d, k, 1234 + idx, 0, device, torch.float64)      # replicated: same seed on every rank
    lead = VBEngine(k, d, device=device)
    lead.load_data(x_dev)
    del x_dev
    model = gaussianmixture.LearnModel(k, d, seed=0)
    members = [lead] + [VBEngine(k, d, device=device, fused_comm=False).share_data_from(lead) for _ in mine[1:]]
    n_sub = int(np.sqrt(n_total))
    big = 1 << 30
    for i, e in zip(mine, members):
        rng = np.random.default_rng([7, i])                      # a different subsample per restart, as `_init_subsampling`
        m0 = np.empty((k, d)); winv0 = np.empty((k, d, d))
        for c in range(k):
            rows = torch.as_tensor(rng.choice(n_total, size=n_sub, replace=False, shuffle=False), device=device)
            sub = lead.x[rows].cpu().numpy() + lead.center
            m0[c] = sub.sum(axis=0) / n_sub
            cen = sub - m0[c]
            winv0[c] = cen.T @ cen / n_sub * model.hn_nus[c] + np.eye(d) * 1e-5
        e.set_prior(model.h0_alpha_vec, model.h0_m_vecs, model.h0_kappas, model.h0_nus, model.h0_w_mats_inv,
                    model._ln_b_h0_w_nus, model._ln_c_h0_alpha)
        e._alloc_state(args.steps + warmup + 4096)
        e.set_params(model.hn_alpha_vec, m0, model.hn_kappas, model.hn_nus, winv0)
        e._max_itr, e._tol, e._launched = big, 0.0, 0
    cap = int(lead.lib.bgmm_batch_capacity(k, d)) if not args.no_batch else 1
    batches = [members[i:i + cap] for i in range(0, len(members), cap)] if cap >= 2 else [[e] for e in members]
    runner = RestartBatch(lead, cap) if cap >= 2 else None

    def sweep(b, ev=None):
        if ev is not None:
            ev[0].record()
        if len(b) >= 2:
            runner.pass_only(b)
        else:
            b[0].pass_only()
        if ev is not None:
            ev[1].record()
        for e in b:
            e._small(_lib.SMALL_ITERATE, big, 0.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(warmup):
        for b in batches:
            sweep(b)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in batches]
           for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = sum(e.kernel_launches for e in members)
    dumped = dump_plan(lead, warmup + args.steps, r_total) if args.dump_outputs else []
    barrier()
    e0.record()
    for s in range(args.steps):
        for bi, b in enumerate(batches):
            sweep(b, evs[s][bi])
    e1.record()
    launches = sum(e.kernel_launches for e in members) - launches0
    barrier()
    if args.dump_outputs:
        outs = {f"restart{i}_{name}": a for i, e in zip(mine, members) if i in dumped
                for name, a in engine_outputs(e, warmup + args.steps).items()}
        if world > 1:                                   # every rank's restarts: the dump does not depend on the GPU count
            parts = [None] * world if rank == 0 else None
            dist.gather_object(outs, parts, dst=0)
            outs = {k: v for part in parts for k, v in part.items()} if rank == 0 else None
        if rank == 0:
            dump_outputs(args.dump_outputs, outs)
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    pass_ms = torch.tensor([np.mean([sum(a.elapsed_time(b) for a, b in step) for step in evs])], device=device,
                           dtype=torch.float64)                   # all sweeps of one step on this rank
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        dist.all_reduce(pass_ms, op=dist.ReduceOp.MAX)
    n_tail = int(1500.0 / max(float(ms_total.item()) / args.steps, 1e-3)) + 1
    for _ in range(min(n_tail, 2000)):
        for b in batches:
            sweep(b)
    torch.cuda.synchronize(device)
    clocks = sampler.stop() if rank == 0 else None
    ms_total, pass_ms = float(ms_total.item()), float(pass_ms.item())
    ms_per_step = ms_total / args.steps
    value = r_total * n_total * k / (ms_per_step * 1e-3)
    hist_ok = True
    for e in members:
        h = e.state[e.off["vlhist"]: e.off["vlhist"] + warmup + args.steps].cpu().numpy()
        hist_ok = hist_ok and bool(np.all(np.isfinite(h)) and np.all(np.diff(h[1:]) >= -1e-9 * np.abs(h[1:-1])))
    tracked = load_peaks()
    r_max = -(-r_total // world)
    flops = r_max * alg_flops_per_iter(n_total, d, k)            # the busiest rank's restarts
    ach = flops / (pass_ms * 1e-3) / 1e12
    executed = r_max * n_total * 4 * k * (1 + d + d * (d + 1) // 2)      # 2 GEMMs x 2 flops x K x P per sample
    roofline = {"bound": "tensor", "achieved": ach, "peak": tracked["fp64_tflops"], "unit": "TFLOP/s",
                "frac": ach / tracked["fp64_tflops"], "traffic": None,
                "kernel": "bgmm::e_large_kernel + bgmm::m_large_kernel (batched: %d restarts per sweep)" % cap,
                "kernel_ms": pass_ms, "kernel_share_of_step": pass_ms / ms_per_step,
                "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": n_total * d * 8 * len(batches),
                "executed_flops_per_launch": executed,
                "executed_frac_of_pipe": executed / (pass_ms * 1e-3) / 1e12 / tracked["fp64_tflops"],
                "peak_source": "FP64 tensor pipe (DMMA.8x8x4), " + tracked["source"]}

    # e2e: the public API with the restarts spread over the ranks; selection checked against the reference's rule
    e2e = None
    sel = None
    if not args.no_e2e:
        for e in members:
            del e
        del members, batches, runner, lead
        torch.cuda.empty_cache()
        x_host_t = torch.empty((n_total, d), dtype=torch.float64).pin_memory()
        x_host_t.copy_(synth_device(n_total, d, k, 1234 + idx, 0, device, torch.float64))
        x_host = x_host_t.numpy()
        lm = gaussianmixture.LearnModel(k, d, seed=0, device=device, restart_group=group)
        buf = io.StringIO()
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            lm.update_posterior(x_host, max_itr=1, num_init=min(r_total, 2 * world), tolerance=0.0)      # warm-up call
        with contextlib.redirect_stdout(buf), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            barrier()
            t0 = time.perf_counter()
            lm.update_posterior(x_host, max_itr=args.steps, num_init=r_total, tolerance=0.0)
            _ = float(lm.vl)
            torch.cuda.synchronize(device)
            dt = time.perf_counter() - t0
        dt_t = torch.tensor([dt], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt_t, op=dist.ReduceOp.MAX)
        dt = float(dt_t.item())
        ok, kept, n_seen = selection_follows_reference_rule(buf.getvalue())
        sel = {"follows_reference_rule": bool(ok and n_seen == r_total), "kept_restart": kept, "restarts": n_seen}
        e2e = {"value": r_total * n_total * k * args.steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(x_host.nbytes / args.steps), "d2h_bytes_per_step": 0, "seconds": dt,
               "host_buffer": "pinned",
               "api": f"LearnModel(restart_group=...).update_posterior(x_host, max_itr=steps, num_init={r_total}, tolerance=0.0): "
                      "upload + host initialisations + all restarts + all-gather of their records + selection + final E-step"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"{args.config}: GMM VB N={n_total} D={d} K={k} float64, num_init={r_total} restarts spread over "
                                   f"{world} GPU(s) (X replicated), {cap} restarts per shared sweep; one step = one VB iteration "
                                   f"of every restart",
                       "l2": f"X resident in HBM, {n_total * d * 8 / 1e6:.0f} MB per sweep (> 126 MB L2), no flush needed",
                       "init": "subsampling-style, a different subsample per restart; default priors; tolerance=0.0"},
            "restart_iters_per_s": r_total * 1e3 / ms_per_step, "elbo_finite_and_monotone": hist_ok,
            "roofline": roofline, "e2e": e2e, "selection": sel, "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the multi-GPU parity block (world > 1)")
    ap.add_argument("--n", type=int, default=0, help="diagnostics: override the row count of the config (not a bench line)")
    ap.add_argument("--restarts", type=int, default=0,
                    help="restart mode (C5): this many restarts spread over the GPUs, X replicated (default 64 for --config c5)")
    ap.add_argument("--no-batch", action="store_true", help="restart mode: one sweep per restart (no bgmm_pass_batched)")
    ap.add_argument("--variant", default="auto", choices=["auto", "simple", "dmma", "f32", "large", "tf32", "direct"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64); the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the device path; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from bayesml_b200 import _lib, gaussianmixture
    from bayesml_b200.engine import VBEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device(f"cuda:{local_rank}")
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
        group = dist.group.WORLD
    warmup = max(args.warmup, 3)
    if args.restarts == 0 and args.config == "c5":
        args.restarts = 64
    if args.restarts > 1:
        bench_restarts(args, world, rank, local_rank, device, group)
        return

    n_total, d, k, precision, idx = CONFIGS[args.config]
    if args.n > 0:
        n_total = args.n
    if args.scaling == "weak":
        n_total = n_total * world
    n_local = n_total // world + (1 if rank < n_total % world else 0)
    xdtype = torch.float64 if precision == "float64" else torch.float32
    x_dev = synth_device(n_local, d, k, 1234 + idx, rank, device, xdtype)

    variant = {"auto": _lib.PASS_AUTO, "simple": _lib.PASS_SIMPLE, "dmma": _lib.PASS_DMMA, "f32": _lib.PASS_F32,
               "large": _lib.PASS_LARGE, "tf32": _lib.PASS_TF32, "direct": _lib.PASS_DIRECT}[args.variant]
    eng = VBEngine(k, d, device=device, precision=precision, group=group, variant=variant)
    eng.load_data(x_dev)                       # centres into the engine's own buffer
    del x_dev

    # initial parameters in the spirit of `_init_subsampling` (:786-796): rank 0 draws sqrt(N) of its rows per class
    model = gaussianmixture.LearnModel(k, d, seed=0)
    init = torch.empty(k * d + k * d * d, dtype=torch.float64, device=device)
    if rank == 0:
        n_sub = int(np.sqrt(n_total))
        rng = np.random.default_rng(0)
        m0 = np.empty((k, d)); winv0 = np.empty((k, d, d))
        for c in range(k):
            rows = torch.as_tensor(rng.choice(n_local, size=n_sub, replace=False, shuffle=False), device=device)
            sub = eng.x[rows].double().cpu().numpy() + eng.center
            m0[c] = sub.sum(axis=0) / n_sub
            cen = sub - m0[c]
            winv0[c] = cen.T @ cen / n_sub * model.hn_nus[c] + np.eye(d) * 1e-5
        init.copy_(torch.as_tensor(np.concatenate([m0.ravel(), winv0.ravel()])))
    if world > 1:
        dist.broadcast(init, src=0)
    init_h = init.cpu().numpy()
    eng.set_prior(model.h0_alpha_vec, model.h0_m_vecs, model.h0_kappas, model.h0_nus, model.h0_w_mats_inv,
                  model._ln_b_h0_w_nus, model._ln_c_h0_alpha)
    eng._alloc_state(args.steps + warmup + 4096)
    eng.set_params(model.hn_alpha_vec, init_h[:k * d].reshape(k, d), model.hn_kappas, model.hn_nus,
                   init_h[k * d:].reshape(k, d, d))
    big = 1 << 30
    eng_comm = eng.comm_desc is not None

    def vb_iteration():
        eng._pass()
        eng._small(_lib.SMALL_ITERATE, big, 0.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(warmup):
        vb_iteration()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    pass_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = eng.kernel_launches
    if args.dump_outputs:
        dump_plan(eng, warmup + args.steps, 1)
    barrier()
    e0.record()
    for i in range(args.steps):
        pass_ev[i][0].record()
        eng.pass_only()
        pass_ev[i][1].record()
        eng.exchange()
        eng._small(_lib.SMALL_ITERATE, big, 0.0)
    e1.record()
    launches = eng.kernel_launches - launches0
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engine_outputs(eng, warmup + args.steps))
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    pass_ms = torch.tensor([np.mean([a.elapsed_time(b) for a, b in pass_ev])], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        dist.all_reduce(pass_ms, op=dist.ReduceOp.MAX)
    # nvidia-smi cannot sample faster than ~100 ms and the timed region may be shorter than that: keep the SAME iteration
    # running (untimed) for another ~1.5 s so that the clock / throttle record is taken under this load.  The number of
    # tail iterations is derived from the max-reduced time, so every rank runs the same count (the exchange needs that).
    n_tail = int(1500.0 / max(float(ms_total.item()) / args.steps, 1e-3)) + 1
    for _ in range(min(n_tail, 4000)):
        vb_iteration()
    torch.cuda.synchronize(device)
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["sampled"] = "timed region + ~1.5 s of the identical, untimed iteration (nvidia-smi -lms 100)"
    ms_total, pass_ms = float(ms_total.item()), float(pass_ms.item())
    ms_per_step = ms_total / args.steps
    value = n_total * k / (ms_per_step * 1e-3)
    # sanity: the loop really ran (ELBO history is finite and non-decreasing after the first step)
    hist = eng.state[eng.off["vlhist"]: eng.off["vlhist"] + warmup + args.steps].cpu().numpy()
    ok = bool(np.all(np.isfinite(hist)) and np.all(np.diff(hist[1:]) >= -1e-9 * np.abs(hist[1:-1])))

    # roofline of the dominant kernel (the pass): algorithmic flops of this rank's rows / its average duration
    flops = alg_flops_per_iter(n_local, d, k)
    ach_tflops = flops / (pass_ms * 1e-3) / 1e12
    x_bytes = n_local * d * (8 if precision == "float64" else 4)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tracked = load_peaks()
    fp64_peak = tracked["fp64_tflops"]
    traffic, pipe_active = None, None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tr.get(f"{args.config}_n{world}")
        pipe_active = tr.get("tensor_pipe_active_pct", {}).get(f"{args.config}_n{world}")
    except Exception:
        pass
    kname = {_lib.PASS_DMMA: "bgmm::pass_dmma_kernel", _lib.PASS_F32: "bgmm::pass_f32_kernel",
             _lib.PASS_TF32: "bgmm::pass_tf32_e_kernel + bgmm::pass_tf32_m_kernel (tcgen05 kind::tf32)",
             _lib.PASS_DIRECT: "bgmm::pass_simple_kernel<DIRECT>",
             _lib.PASS_LARGE: "bgmm::e_large_kernel + bgmm::m_large_kernel", _lib.PASS_SIMPLE: "bgmm::pass_simple_kernel"}[
        eng.lib.bgmm_pass_resolve(k, d, eng.x_code, eng.variant, 0)]
    roofline = {
        "bound": "tensor", "achieved": ach_tflops, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": ach_tflops / fp64_peak, "traffic": traffic,
        "kernel": kname,
        "kernel_ms": pass_ms, "kernel_share_of_step": pass_ms / ms_per_step,
        "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": x_bytes,
        # frac can exceed 1: SURVEY §8d's algorithmic count charges the full D x D quadratic form, the kernels contract the
        # packed symmetric feature map (about half the flops); the ncu capture of the same kernel gives the pipe's duty cycle
        "tensor_pipe_active_pct_ncu": pipe_active,
        "peak_source": "FP64 tensor pipe (DMMA.8x8x4), " + tracked["source"],
        "hbm": {"achieved_gbs": x_bytes / (pass_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                "frac": x_bytes / (pass_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s"},
    }

    resolved = eng.lib.bgmm_pass_resolve(k, d, eng.x_code, eng.variant, 0)
    if precision == "float32" and resolved == _lib.PASS_TF32:
        # fp32 mode on the tensor cores: roofline = the tf32 tensor pipe.  MEASURED_PEAKS.json has dense bf16 only; kind::tf32
        # runs at half the bf16 rate (B200_PROFILING.md: 1.1 vs 2.25 PFLOP/s nominal), so peak = measured bf16 / 2.
        # `achieved` counts the ALGORITHMIC flops (SURVEY §8d); the kernels execute 3 split products on padded tiles.
        tf32_peak = float(peaks.get("bf16_tflops", 1640.0)) / 2.0
        kd, dp, kp = (d + 1 + 7) // 8 * 8, (4 if d <= 4 else 8 if d <= 8 else 16 if d <= 16 else 32), (k + 3) // 4 * 4
        p_feat = 1 + d + d * (d + 1) // 2
        # executed: E = 3 split products of [128 x kd] . [kd x kp dp]; statistics = 128-row (component) tiles against
        # nf features, 2 products when the lo parts ride in spare tensor-memory lanes (K <= 32), else 3
        nf = (p_feat + 15) // 16 * 16
        executed = n_local * 2.0 * (3.0 * kd * kp * dp + (2.0 if k <= 32 else 3.0) * 128 * nf)
        roofline.update({"bound": "tensor", "achieved": ach_tflops, "peak": tf32_peak, "unit": "TFLOP/s",
                         "frac": ach_tflops / tf32_peak,
                         "peak_source": "kind::tf32 dense = MEASURED_PEAKS.json bf16_tflops / 2 (no measured tf32 entry)",
                         "executed_flops_per_launch": executed,
                         "executed_frac_of_pipe": executed / (pass_ms * 1e-3) / 1e12 / tf32_peak})
    elif precision == "float32":
        # fp32 mode (C3): BASELINE labels it HBM-streaming; the kernel is in fact FP32-issue bound (SURVEY.md §8d caveat),
        # so the HBM fraction is the headline roofline and the FP32 FMA-pipe fraction is reported beside it
        roofline.update({"bound": "hbm", "achieved": roofline["hbm"]["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                         "frac": roofline["hbm"]["frac"], "peak_source": roofline["hbm"]["peak_source"],
                         "fp32": {"achieved_tflops": ach_tflops, "peak_tflops": tracked["fp32_tflops"],
                                  "frac": ach_tflops / tracked["fp32_tflops"], "peak_source": tracked["source"]}})

    # ---- e2e: the public API with a HOST array (pinned), upload + init + steps iterations + final E-step + readback ----
    e2e = None
    if not args.no_e2e:
        del eng
        torch.cuda.empty_cache()
        x_host_t = torch.empty((n_local, d), dtype=xdtype).pin_memory()
        x_host_t.copy_(synth_device(n_local, d, k, 1234 + idx, rank, device, xdtype))
        x_host = x_host_t.numpy()
        lm = gaussianmixture.LearnModel(k, d, seed=0, device=device, precision=precision, process_group=group)
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            # warm-up: one short full-size call (allocator, pinned staging, kernel modules) so that the timed call is
            # the steady state of a second fit on data of the same shape
            lm.update_posterior(x_host, max_itr=1, num_init=1, tolerance=0.0)
            barrier()
            t0 = time.perf_counter()
            lm.update_posterior(x_host, max_itr=args.steps, num_init=1, tolerance=0.0)
            _ = float(lm.vl); _ = lm.hn_alpha_vec.sum()
            torch.cuda.synchronize(device)
            dt = time.perf_counter() - t0
        dt_t = torch.tensor([dt], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt_t, op=dist.ReduceOp.MAX)
        dt = float(dt_t.item())
        state_bytes = int(lm._engine().state.numel() * 8)
        e2e = {"value": n_total * k * args.steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(x_host.nbytes / args.steps), "d2h_bytes_per_step": int(2 * state_bytes / args.steps),
               "seconds": dt, "host_buffer": "pinned",
               "api": "bayesml_b200.gaussianmixture.LearnModel.update_posterior(x_host, max_itr=steps, "
                      "num_init=1, tolerance=0.0): upload + centring + host init + steps iterations + final E-step"}
        # the same call on an ordinary (pageable) numpy array, as a user of the reference would pass it
        x_page = np.array(x_host)
        del x_host, x_host_t
        with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            barrier()
            t0 = time.perf_counter()
            lm.update_posterior(x_page, max_itr=args.steps, num_init=1, tolerance=0.0)
            _ = float(lm.vl); _ = lm.hn_alpha_vec.sum()
            torch.cuda.synchronize(device)
            dtp = time.perf_counter() - t0
        dtp_t = torch.tensor([dtp], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dtp_t, op=dist.ReduceOp.MAX)
        dtp = float(dtp_t.item())
        e2e["pageable"] = {"value": n_total * k * args.steps / dtp, "unit": UNIT, "seconds": dtp,
                           "host_buffer": "pageable numpy array (cudaMemcpy from unpinned memory)"}
        del x_page

    pm = None
    if world > 1 and not args.no_parity:
        pm = parity_multi(world, rank, device, group)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64" if precision == "float64" else "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: GMM VB N={n_total} D={d} K={k} {precision}, rows sharded over {world} GPU(s), "
                                   f"one exchange of K*PITCH+8 doubles per iteration ({'peer-memory, fused into bgmm_small' if eng_comm else 'ncclAllReduce'})" if world > 1 else
                                   f"{args.config}: GMM VB N={n_total} D={d} K={k} {precision}, 1 GPU",
                       "l2": f"X resident in HBM, {x_bytes / 1e6:.0f} MB per GPU per iteration (> 126 MB L2), no flush needed"
                             if x_bytes > 130e6 else "X fits in L2: cold-L2 not enforced",
                       "init": "subsampling-style (sqrt(N) rows per class), default priors, tolerance=0.0"},
            "iters_per_s": 1e3 / ms_per_step, "elbo_finite_and_monotone": ok,
            "roofline": roofline, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
        }
        if e2e is not None:
            line["e2e_pageable"] = e2e.pop("pageable")
        if pm is not None:
            line["parity_multi"] = pm
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.config)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
