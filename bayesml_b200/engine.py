"""Device engine of the VB Gaussian-mixture hot path.

Owns the device buffers (torch tensors: plumbing only) and drives the kernels of libbgmm.so through the C ABI
(include/bgmm.h).  One engine lives on one GPU; with a torch.distributed process group every rank holds a
shard of the rows of X and the only exchange per VB iteration is one all-reduce of the packed statistics
buffer [K*PITCH raw moments | sum r ln r | rows]  (SURVEY.md §8e).

Reference call sites replaced (bayesml/gaussianmixture/_gaussianmixture.py): the VB loop :862-872 runs on the
device; the host only syncs once per chunk of iterations to read the ELBO history and the done flag.
"""
from __future__ import annotations

import ctypes
import os
import time
import warnings

import numpy as np
import torch

from . import _lib

_DTYPES = {"float64": (_lib.F64, torch.float64), "float32": (_lib.F32, torch.float32)}


class _Phase:
    """Wall-clock phase timer (device-synchronised), active only with BAYESML_B200_TIMING=1."""

    def __init__(self, eng, name):
        self.eng, self.name = eng, name

    def __enter__(self):
        if self.eng.timing is not None:
            torch.cuda.synchronize(self.eng.device)
            self.t0 = time.perf_counter()

    def __exit__(self, *exc):
        if self.eng.timing is not None:
            torch.cuda.synchronize(self.eng.device)
            self.eng.timing[self.name] = self.eng.timing.get(self.name, 0.0) + time.perf_counter() - self.t0


class VBEngine:
    def __init__(self, K, D, device=None, precision="float64", group=None, variant=_lib.PASS_AUTO, fused_comm=True):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("bayesml_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.K, self.D = int(K), int(D)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if precision not in _DTYPES:
            raise ValueError(f"precision must be 'float64' or 'float32', got {precision!r}")
        self.precision = precision
        self.x_code, self.x_torch_dtype = _DTYPES[precision]
        if precision == "float32" and not (self.lib.bgmm_pass_supported(self.K, self.D, _lib.F32, _lib.PASS_F32)
                                           or self.lib.bgmm_pass_supported(self.K, self.D, _lib.F32, _lib.PASS_TF32)):
            # fp32 mode has two kernels: the streaming FFMA kernel (D <= 3, K <= 8) and the tcgen05 kind::tf32 kernels
            # (D <= 31, K <= 64); any other shape keeps X in fp64 on the device and runs the fp64 kernels
            self.x_code, self.x_torch_dtype = _DTYPES["float64"]
        self.group = group
        env = os.environ.get("BAYESML_B200_PASS_VARIANT", "").lower()     # debugging / tests: force a kernel variant
        if env:
            variant = {"auto": _lib.PASS_AUTO, "simple": _lib.PASS_SIMPLE, "dmma": _lib.PASS_DMMA, "f32": _lib.PASS_F32, "large": _lib.PASS_LARGE, "direct": _lib.PASS_DIRECT, "tf32": _lib.PASS_TF32}[env]
        self.variant = variant
        self.hist_len = 0
        self.state = None
        self.x = None
        self.n_local = 0
        self.n_global = 0
        self.center = np.zeros(self.D)
        self.timing = {} if os.environ.get("BAYESML_B200_TIMING") else None
        self.kernel_launches = 0              # kernels libbgmm launched for this engine's calls (_call)
        self._pending = None
        self.failed = False
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(int(self.lib.bgmm_workspace_doubles(self.K, self.D)), dtype=torch.float64,
                                         device=self.device)
        self._alloc_state(2)
        self.r_dev = self.lnrho_dev = self.argmax_dev = None
        self._r_scratch = None
        # multi-GPU exchange: peer memory (fused into bgmm_small) when the ranks share a box, else ncclAllReduce
        self.comm_desc = None
        self._comm_base, self._comm_peers = None, []
        if group is not None and fused_comm and os.environ.get("BAYESML_B200_COMM", "peer").lower() != "nccl":
            self._setup_peer_comm()

    def _setup_peer_comm(self):
        import torch.distributed as dist
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if dist.get_backend(self.group) != "nccl" or world > _lib.MAX_RANKS or world < 2:
            return
        lib = self.lib
        ok = 1
        base, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            try:
                self._call(lib.bgmm_comm_alloc, lib.bgmm_comm_block_doubles(self.K, self.D), ctypes.byref(base), handle)
            except RuntimeError:
                ok = 0
            handles = [None] * world
            dist.all_gather_object(handles, (handle.raw, ok), group=self.group)
            ptrs = [0] * world
            if all(h[1] for h in handles):
                for r in range(world):
                    if r == rank:
                        ptrs[r] = base.value
                        continue
                    p = ctypes.c_void_p()
                    if lib.bgmm_comm_open(handles[r][0], ctypes.byref(p)) != 0:
                        ok = 0
                        break
                    ptrs[r] = p.value
                    self._comm_peers.append(p.value)
            else:
                ok = 0
            flag = torch.tensor([ok], device=self.device, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
            if int(flag.item()) == 0:
                warnings.warn("bayesml_b200: peer-memory exchange unavailable (CUDA IPC); using ncclAllReduce")
                return
            self._comm_base = base.value
            desc = np.zeros(2 + _lib.MAX_RANKS, dtype=np.int64)
            desc[0] = world | (rank << 32)                       # int32 world, int32 rank (little endian)
            desc[2:2 + world] = ptrs
            self.comm_desc = torch.as_tensor(desc).to(self.device)
            self._write_comm_ptr()
            dist.barrier(group=self.group)

    def _write_comm_ptr(self):
        """ctrl.comm <- device address of the exchange descriptor: every bgmm_pass then publishes its statistics from the
        last CTA of its reduction."""
        if self.comm_desc is not None:
            p = self.comm_desc.data_ptr()
            c = self.ctrl
            c[_lib.CTRL_COMM_LO] = (p & 0xFFFFFFFF) - (1 << 32 if (p & 0x80000000) else 0)     # int32 bit pattern
            c[_lib.CTRL_COMM_HI] = ((p >> 32) & 0xFFFFFFFF) - (1 << 32 if ((p >> 32) & 0x80000000) else 0)

    def close(self):
        """Release the peer-memory mappings (optional; process exit does it too)."""
        for p in self._comm_peers:
            self.lib.bgmm_comm_close(p)
        if self._comm_base:
            self.lib.bgmm_comm_free(self._comm_base)
        self._comm_peers, self._comm_base, self.comm_desc = [], None, None
        if self.state is not None:
            self.ctrl[_lib.CTRL_COMM_LO:_lib.CTRL_COMM_HI + 1].zero_()

    def phase(self, name):
        return _Phase(self, name)

    def _call(self, fn, *args):
        """One libbgmm call that returns a status code: raise RuntimeError on failure, and add the kernels the library
        launched for it to kernel_launches."""
        n0 = self.lib.bgmm_launch_count()
        rc = fn(*args)
        self.kernel_launches += self.lib.bgmm_launch_count() - n0
        _lib.check(rc, fn.__name__)

    # ------------------------------------------------------------------ buffers
    def _alloc_state(self, hist_len):
        if self.state is not None and hist_len <= self.hist_len:
            return
        old = None
        if self.state is not None:
            old = (self.state, self.off)
        self.hist_len = int(hist_len)
        self.off, self.poff = _lib.layout(self.K, self.D, self.hist_len)
        self.state = torch.zeros(self.off["total"], dtype=torch.float64, device=self.device)
        if old is not None:  # keep everything in front of the (variable-length, last) ELBO history: no offset there depends on it
            n_keep = old[1]["vlhist"]
            assert n_keep == self.off["vlhist"]
            self.state[:n_keep].copy_(old[0][:n_keep])
        self._host_ctrl = torch.empty(_lib.N_CTRL, dtype=torch.int32).pin_memory()
        self._host_hist = torch.empty(self.hist_len, dtype=torch.float64).pin_memory()

    def _view(self, name, length):
        o = self.off[name]
        return self.state[o:o + length]

    def _pview(self, which, name, length):
        o = self.off[f"params{which}"] + self.poff[name]
        return self.state[o:o + length]

    @property
    def ctrl(self):
        o = self.off["ctrl"]
        return self.state[o:o + _lib.N_CTRL // 2].view(torch.int32)

    @property
    def stats(self):
        o = self.off["stats"]
        return self.state[o:o + self.off["stats_len"]]

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _put(self, view, arr):
        view.copy_(torch.as_tensor(np.ascontiguousarray(arr, dtype=np.float64).reshape(-1)), non_blocking=False)

    # ------------------------------------------------------------------ data
    def load_data(self, x):
        """Upload the local rows of X ((n, D) numpy array or torch tensor), centre them about the global column mean."""
        self.load_data_begin(x)
        return self.load_data_finish()

    def load_data_begin(self, x):
        """Asynchronous part: host->device copy (truly async from pinned memory) and the column sums; the caller may do
        host work (e.g. draw the initial states) before load_data_finish()."""
        D = self.D
        with torch.cuda.device(self.device):
            own = not isinstance(x, torch.Tensor)
            if not own:
                xt = x.reshape(-1, D)
                if xt.device != self.device:
                    xt = xt.to(self.device, non_blocking=True)
                raw = xt if xt.dtype in (torch.float64, torch.float32) else xt.to(torch.float64)
                raw = raw.contiguous()
            else:
                xa = np.ascontiguousarray(x).reshape(-1, D)
                if xa.dtype not in (np.float64, np.float32):
                    xa = xa.astype(np.float64)
                raw = torch.from_numpy(xa).to(self.device, non_blocking=True)
            raw_code = _lib.F64 if raw.dtype == torch.float64 else _lib.F32
            n = raw.shape[0]
            self.n_local = int(n)
            colsum = torch.zeros(D + 1, dtype=torch.float64, device=self.device)
            self._call(self.lib.bgmm_colsum, raw.data_ptr(), n, D, raw_code, colsum.data_ptr(), self.workspace.data_ptr(),
                       self._stream())
            colsum[D] = float(n)
            if self.group is not None:
                torch.distributed.all_reduce(colsum, group=self.group)
            host = torch.empty(D + 1, dtype=torch.float64).pin_memory()
            host.copy_(colsum, non_blocking=True)
            self._pending = (raw, raw_code, own, host)
        return self

    def load_data_finish(self):
        raw, raw_code, own, host = self._pending
        self._pending = None
        D, n = self.D, self.n_local
        with torch.cuda.device(self.device):
            torch.cuda.current_stream(self.device).synchronize()
            tot = host.numpy()
            self.n_global = int(round(tot[D]))
            self.center = tot[:D] / max(self.n_global, 1)
            cview = self._view("center", D)
            self._put(cview, self.center)
            if raw.dtype == self.x_torch_dtype and own:
                out = raw          # our own upload buffer: centre in place
            else:
                out = torch.empty((n, D), dtype=self.x_torch_dtype, device=self.device)
            self._call(self.lib.bgmm_center, raw.data_ptr(), raw_code, out.data_ptr(), self.x_code, n, D, cview.data_ptr(),
                       self._stream())
            self.x = out
            self.r_dev = self.lnrho_dev = self.argmax_dev = None
            # the tcgen05 fp32-mode kernels keep r (float32, [n][K]) and their operand image in the workspace
            need = int(self.lib.bgmm_tf32_workspace_doubles(self.K, self.D, n)) if self.x_code == _lib.F32 else 0
            if need > self.workspace.numel():
                self.workspace = torch.empty(need, dtype=torch.float64, device=self.device)
        return self

    # ------------------------------------------------------------------ prior / parameters
    def set_prior(self, alpha0, m0, kappa0, nu0, w0inv, ln_b_h0, ln_c_h0_alpha):
        K, D = self.K, self.D
        self._put(self._view("alpha0", K), alpha0)
        self._put(self._view("kappa0", K), kappa0)
        self._put(self._view("nu0", K), nu0)
        self._put(self._view("m0", K * D), np.asarray(m0) - self.center)
        self._put(self._view("w0inv", K * D * D), w0inv)
        self._put(self._view("lnb0", K), ln_b_h0)
        self._put(self._view("lnc0", 1), [ln_c_h0_alpha])

    def set_params(self, alpha, m, kappa, nu, winv):
        """Load (alpha, m, kappa, nu, W^-1) as parameter set 0, reset the control words, compute W/features/coef."""
        K, D = self.K, self.D
        self._put(self._pview(0, "alpha", K), alpha)
        self._put(self._pview(0, "kappa", K), kappa)
        self._put(self._pview(0, "nu", K), nu)
        self._put(self._pview(0, "m", K * D), np.asarray(m) - self.center)
        self._put(self._pview(0, "winv", K * D * D), winv)
        c = self.ctrl                          # reset everything but the exchange sequence number and descriptor address
        c[:_lib.CTRL_SEQ].zero_()
        c[_lib.CTRL_SEQ + 1:_lib.CTRL_COMM_LO].zero_()
        self._small(_lib.SMALL_FEATURES, 0, 0.0)

    def _small(self, mode, max_itr, tol):
        comm = self.comm_desc.data_ptr() if (self.comm_desc is not None and mode != _lib.SMALL_FEATURES) else 0
        self._call(self.lib.bgmm_small, self.K, self.D, self.state.data_ptr(), mode, int(max_itr), float(tol), self.hist_len,
                   comm, self._stream())

    def _pass(self, r_out=None, lnrho_out=None, argmax_out=None, r_in=None, force=0, r_in_variant=_lib.PASS_SIMPLE):
        self.pass_only(r_out, lnrho_out, argmax_out, r_in, force, r_in_variant)
        self.exchange(force)

    def pass_only(self, r_out=None, lnrho_out=None, argmax_out=None, r_in=None, force=0, r_in_variant=_lib.PASS_SIMPLE):
        """One bgmm_pass launch (E-step + local statistics) without the cross-rank exchange."""
        ptr = lambda t: 0 if t is None else t.data_ptr()  # noqa: E731
        if r_out is None and r_in is None and self.lib.bgmm_pass_resolve(
                self.K, self.D, self.x_code, self.variant, 0) == _lib.PASS_LARGE:
            # large K*P regime: r is the hand-over between the E and the M kernel and lives in HBM ([n][K] fp64)
            if self._r_scratch is None or self._r_scratch.shape[0] != self.n_local:
                self._r_scratch = torch.empty((self.n_local, self.K), dtype=torch.float64, device=self.device)
            r_out = self._r_scratch
        self._call(self.lib.bgmm_pass, ptr(self.x), self.n_local, self.K, self.D, self.x_code, self.state.data_ptr(),
                   self.workspace.data_ptr(), ptr(r_out), ptr(lnrho_out), ptr(argmax_out), ptr(r_in),
                   self.variant if r_in is None else r_in_variant, force, self._stream())

    def exchange(self, force=0):
        """The per-iteration exchange of the statistics between row shards.  Peer memory: nothing to launch — bgmm_pass has
        published the statistics from its reduction's last CTA (ctrl.comm) and the next bgmm_small sums the peers' blocks.
        Without peer access: ncclAllReduce."""
        if self.comm_desc is None and self.group is not None:
            torch.distributed.all_reduce(self.stats, group=self.group)

    # ------------------------------------------------------------------ the VB loop (:860-872)
    # begin / enqueue / poll / finish let a caller interleave several engines (concurrent restarts on CUDA streams);
    # run() is the single-engine driver.
    def begin(self, max_itr, tol, r_init=None):
        """Post-init pass + ELBO (:852/:854, :860) and the first M-step; nothing is synchronised."""
        self._max_itr, self._tol, self._launched = int(max_itr), float(tol), 0
        with torch.cuda.device(self.device):
            self._alloc_state(self._max_itr + 1)
            if r_init is not None:
                if isinstance(r_init, torch.Tensor):
                    r_dev = r_init.to(self.device, dtype=torch.float64).contiguous()
                else:
                    r_dev = torch.as_tensor(np.ascontiguousarray(r_init, dtype=np.float64)).to(self.device)
                self._pass(r_in=r_dev, force=1)
            else:
                self._pass()
            self._small(_lib.SMALL_ITERATE, self._max_itr, self._tol)

    def enqueue(self, n_iters):
        """Queue up to n_iters VB iterations (no-ops on the device once ctrl.done is set), then an async read of ctrl."""
        todo = max(0, min(int(n_iters), self._max_itr - self._launched))
        with torch.cuda.device(self.device):
            for _ in range(todo):
                self._pass()
                self._small(_lib.SMALL_ITERATE, self._max_itr, self._tol)
            self._launched += todo
            self._host_ctrl.copy_(self.ctrl, non_blocking=True)
        return todo

    def finished(self):
        """After the stream has been synchronised: did the device stop (converged / max_itr) or is the budget queued?"""
        return bool(self._host_ctrl[_lib.CTRL_DONE]) or self._launched >= self._max_itr

    def finish(self):
        """-> (vl_history [1 + n_iter], converged)."""
        with torch.cuda.device(self.device):
            self._host_ctrl.copy_(self.ctrl, non_blocking=True)
            o = self.off["vlhist"]
            self._host_hist.copy_(self.state[o:o + self.hist_len], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        hc = self._host_ctrl
        self.failed = bool(int(hc[_lib.CTRL_ERROR]))     # a W^-1 lost positive definiteness: the loop stopped there
        n_eval = int(hc[_lib.CTRL_ITER])
        return self._host_hist[:n_eval].numpy().copy(), bool(hc[_lib.CTRL_CONVERGED])

    def run(self, max_itr, tol, r_init=None, chunk=None):
        """Post-init ELBO + up to max_itr VB iterations on the device.

        Returns (vl_history [1 + n_iter], converged).  `r_init`: (n_local, K) responsibilities for the
        'random_responsibility' initialisation (:734-736); otherwise the first pass is an E-step with the
        parameters loaded by set_params (:852)."""
        self.begin(max_itr, tol, r_init)
        step = 4 if chunk is None else int(chunk)
        done = self._max_itr == 0
        while not done:
            t0 = time.perf_counter()
            todo = self.enqueue(step)
            torch.cuda.current_stream(self.device).synchronize()
            done = self.finished()
            if chunk is None:      # aim for ~30 ms between host syncs, at most 64 queued iterations
                per = (time.perf_counter() - t0) / max(todo, 1)
                step = int(min(64, max(1, 0.03 / max(per, 1e-6))))
        return self.finish()

    def share_data_from(self, other):
        """Use another engine's resident X (read-only) — concurrent restarts on one GPU."""
        self.x, self.n_local, self.n_global, self.center = other.x, other.n_local, other.n_global, other.center
        self._put(self._view("center", self.D), self.center)
        self.r_dev = self.lnrho_dev = self.argmax_dev = None
        return self

    # ------------------------------------------------------------------ results
    def fetch_params(self):
        """Current parameter set as numpy arrays (m back in the original frame)."""
        K, D = self.K, self.D
        host = self.state.cpu().numpy()
        cur = int(host[self.off["ctrl"]:self.off["ctrl"] + _lib.N_CTRL // 2].view(np.int32)[_lib.CTRL_CUR])
        base = self.off[f"params{cur}"]
        g = lambda name, n: host[base + self.poff[name]: base + self.poff[name] + n].copy()  # noqa: E731
        out = {
            "alpha": g("alpha", K), "kappa": g("kappa", K), "nu": g("nu", K),
            "m": g("m", K * D).reshape(K, D) + self.center,
            "winv": g("winv", K * D * D).reshape(K, D, D), "w": g("w", K * D * D).reshape(K, D, D),
            "e_ln_pi": g("elnpi", K), "e_ln_lambda_dets": g("elndet", K), "ln_b": g("lnb", K),
            "coef": g("coef", K * self.off["pitch"]).reshape(K, self.off["pitch"]),
            "vl_terms": host[self.off["vlterms"]:self.off["vlterms"] + 8].copy(),
        }
        out.update(self._stats_from_host(host))
        return out

    def _stats_from_host(self, host):
        K, D = self.K, self.D
        ns = host[self.off["ns"]:self.off["ns"] + K].copy()
        xbar = host[self.off["xbar"]:self.off["xbar"] + K * D].reshape(K, D) + self.center
        smats = host[self.off["smats"]:self.off["smats"] + K * D * D].reshape(K, D, D).copy()
        return {"ns": ns, "x_bar": xbar, "s_mats": smats}

    def final_pass(self, want_r=True, want_lnrho=True, want_argmax=True):
        """E-step with the current parameters that materialises r / ln rho / argmax (:895, :1186)."""
        K, n = self.K, self.n_local
        with torch.cuda.device(self.device):
            self.r_dev = torch.empty((n, K), dtype=torch.float64, device=self.device) if want_r else None
            self.lnrho_dev = torch.empty((n, K), dtype=torch.float64, device=self.device) if want_lnrho else None
            self.argmax_dev = torch.empty(n, dtype=torch.int32, device=self.device) if want_argmax else None
            self._pass(r_out=self.r_dev, lnrho_out=self.lnrho_dev, argmax_out=self.argmax_dev, force=1)
            self._small(_lib.SMALL_STATS, 0, 0.0)
            host = self.state.cpu().numpy()
        out = self._stats_from_host(host)
        # False: moments about the global centre (feature-map kernels), s_mats carries an absolute error of
        # ~ eps * |x_bar_k - c|^2 (far below what the E-step's own rounding does to r, measured in tests/cond_sweep.py);
        # refine_smats() recomputes it in the two-pass centred form from the materialised r if that is ever wanted
        out["centred"] = bool(host[self.off["stats"] + self.K * self.off["pitch"] + _lib.STATS_FORMAT] > 0.5)
        return out

    def pred_log_density(self, ck, hk, nuk):
        """ln of the predictive mixture-of-Student-t density of every resident row (bgmm_pred_logdensity): the quadratic
        forms come from one bgmm_pass with the parameter set loaded by set_params (Lambda_k = p_lambda_mats[k]).
        -> numpy array [n_local]."""
        K, n = self.K, self.n_local
        with torch.cuda.device(self.device):
            lnrho = torch.empty((n, K), dtype=torch.float64, device=self.device)
            self.pass_only(lnrho_out=lnrho, force=_lib.FORCE | _lib.FORCE_NO_PUBLISH)    # rows are independent: no exchange
            cur = int(self.ctrl[_lib.CTRL_CUR].item())
            acst = self._pview(cur, "acst", K)
            consts = torch.as_tensor(np.ascontiguousarray(np.stack([ck, hk, nuk]), dtype=np.float64)).to(self.device)
            out = torch.empty(n, dtype=torch.float64, device=self.device)
            self._call(self.lib.bgmm_pred_logdensity, lnrho.data_ptr(), n, K, acst.data_ptr(), consts[0].data_ptr(),
                       consts[1].data_ptr(), consts[2].data_ptr(), out.data_ptr(), self._stream())
            return out.cpu().numpy()

    def draw_dirichlet1(self, seed, row_offset=0):
        """(n_local, K) responsibilities ~ Dirichlet(1_K) drawn on the device (bgmm_dirichlet1; Philox, keyed by the
        global row index) -> device tensor."""
        with torch.cuda.device(self.device):
            r = torch.empty((self.n_local, self.K), dtype=torch.float64, device=self.device)
            self._call(self.lib.bgmm_dirichlet1, r.data_ptr(), self.n_local, self.K, int(seed) & (2 ** 64 - 1), int(row_offset),
                       self._stream())
        return r

    def refine_smats(self):
        """s_mats of the last final_pass in the reference's two-pass centred form (:730-732): one more sweep over X with
        the materialised responsibilities, moments about x_bar_k (bgmm_pass DIRECT with r_in).  -> s_mats [K][D][D]."""
        if self.r_dev is None or self.x is None:
            raise RuntimeError("refine_smats needs the responsibilities of a preceding final_pass on the resident X")
        with torch.cuda.device(self.device):
            self._pass(r_in=self.r_dev, force=1, r_in_variant=_lib.PASS_DIRECT)
            self._small(_lib.SMALL_STATS, 0, 0.0)
            o = self.off["smats"]
            return self.state[o:o + self.K * self.D * self.D].cpu().numpy().reshape(self.K, self.D, self.D)


class RestartBatch:
    """Several restarts of the same fit advanced by ONE sweep over X per VB iteration (north_star (4); the restart loop
    `update_posterior` :847-883 run concurrently instead of one after another).

    Members are VBEngines that share the resident X (`share_data_from`); bgmm_pass_batched stacks their coefficient rows
    into one E-GEMM / M-GEMM of R * Kp components with one softmax per member, then every member runs its own bgmm_small
    (ELBO, convergence flag, M-step).  Members that are done are carried along as no-ops until the caller swaps them out."""

    def __init__(self, lead, capacity):
        self.lead, self.lib = lead, lead.lib
        K, D = lead.K, lead.D
        self.Kp = (K + 7) // 8 * 8
        self.capacity = int(capacity)
        ke = self.capacity * self.Kp
        with torch.cuda.device(lead.device):
            off, _ = _lib.layout(ke, D, 1)
            self.super_state = torch.zeros(off["total"], dtype=torch.float64, device=lead.device)
            self.workspace = torch.empty(int(self.lib.bgmm_workspace_doubles(ke, D)), dtype=torch.float64, device=lead.device)
            self.r_scratch = torch.empty((lead.n_local, ke), dtype=torch.float64, device=lead.device)

    def pass_only(self, members):
        """The shared E-step / statistics sweep of every engine in `members` (2 <= len <= capacity)."""
        lead = self.lead
        R = len(members)
        ptrs = (ctypes.c_void_p * R)(*[m.state.data_ptr() for m in members])
        with torch.cuda.device(lead.device):
            lead._call(self.lib.bgmm_pass_batched, lead.x.data_ptr(), lead.n_local, lead.K, lead.D, R, ptrs,
                       self.super_state.data_ptr(), self.workspace.data_ptr(), self.r_scratch.data_ptr(), lead._stream())

    def step(self, members, max_itr=None, tol=None):
        """One VB iteration (:863-869) of every engine in `members`."""
        self.pass_only(members)
        with torch.cuda.device(self.lead.device):
            for m in members:
                m._small(_lib.SMALL_ITERATE, m._max_itr if max_itr is None else max_itr, m._tol if tol is None else tol)
                m._launched += 1


class HMMEngine(VBEngine):
    """Device engine of the VB hidden-Markov (Gaussian emission) fit: the mixture engine's state block (alpha plays eta)
    plus the transition-matrix block `hst` and the per-element buffers of the forward-backward scan.

    Reference call sites replaced (bayesml/hiddenmarkovnormal/_hiddenmarkovnormal.py): the VB loop :1102-1113 —
    `_update_q_mu_lambda`/`_update_q_pi`/`_update_q_a` -> bgmm_hmm_small, `_update_q_z` -> bgmm_hmm_pass, `_calc_vl`
    and the convergence test -> bgmm_hmm_small; on one GPU (the recursions couple all elements of a sequence).

    The loaded rows are one sequence, or (`set_sequences`) several independent sequences, concatenated, that share the
    posterior: then the E-step and the Viterbi decode run through bgmm_hmm_pass_seqs / bgmm_hmm_viterbi_seqs."""

    def __init__(self, K, D, device=None):
        super().__init__(K, D, device=device, precision="float64", group=None, variant=_lib.PASS_LARGE)
        if not self.lib.bgmm_hmm_supported(self.K, self.D):
            raise RuntimeError(f"bayesml_b200 hidden-Markov path: unsupported shape K={K}, D={D} "
                               "(float64, K <= 32, D <= 128); there is no CPU fallback")
        self.hoff = _lib.hmm_layout(self.K)
        self.hst = torch.zeros(self.hoff["total"], dtype=torch.float64, device=self.device)
        self.lnrho_buf = self.alpha_buf = self.gamma_buf = self.cs_buf = self.beta_buf = self.scan_ws = None
        self.seq_starts = self.plan = self.plan_dev = None

    def _hview(self, name, length, which=None):
        o = self.hoff[name] if which is None else self.hoff[f"set{which}"] + self.hoff[name]
        return self.hst[o:o + length]

    def load_data_finish(self):
        super().load_data_finish()
        n, K = self.n_local, self.K
        with torch.cuda.device(self.device):
            if self.lnrho_buf is None or self.lnrho_buf.shape[0] != n:
                mk = lambda *shape: torch.empty(shape, dtype=torch.float64, device=self.device)  # noqa: E731
                self.lnrho_buf, self.alpha_buf, self.gamma_buf, self.cs_buf = mk(n, K), mk(n, K), mk(n, K), mk(n)
                self.scan_ws = mk(int(self.lib.bgmm_hmm_scan_workspace_doubles(K, n)))
            self.beta_buf = None
        self.seq_starts = self.plan = self.plan_dev = None
        return self

    def set_sequences(self, seq_starts):
        """The loaded rows are the sequences starting at rows `seq_starts` (sorted, first 0), concatenated; None: one
        sequence.  Builds the chunk table (bgmm_hmm_seq_plan) on the host and keeps a device copy for the E-steps."""
        self.seq_starts = self.plan = self.plan_dev = None
        if seq_starts is None:
            return self
        n, K = self.n_local, self.K
        starts = np.ascontiguousarray(seq_starts, dtype=np.int64)
        size = int(self.lib.bgmm_hmm_seq_plan(n, starts.size, starts.ctypes.data, None, 0))
        if size < 0:
            _lib.check(size, "bgmm_hmm_seq_plan")
        plan = np.zeros(size, dtype=np.int64)
        _lib.check(int(self.lib.bgmm_hmm_seq_plan(n, starts.size, starts.ctypes.data, plan.ctypes.data, size)) - size,
                   "bgmm_hmm_seq_plan")
        with torch.cuda.device(self.device):
            self.plan_dev = torch.from_numpy(plan).to(self.device)
            need = int(self.lib.bgmm_hmm_seq_workspace_doubles(K, n, starts.size))
            if self.scan_ws.numel() < need:
                self.scan_ws = torch.empty(need, dtype=torch.float64, device=self.device)
        self.seq_starts, self.plan = starts, plan
        return self

    def _seq_starts_dev(self):
        nch, nseg = int(self.plan[3]), int(self.plan[4] + self.plan[5])
        return self.plan_dev[8 + 3 * nch + 1 + 2 * nseg:]

    def set_hmm_prior(self, eta0, zeta0, m0, kappa0, nu0, w0inv, ln_b_h0, ln_c_h0_eta, ln_c_h0_zeta_sum):
        self.set_prior(eta0, m0, kappa0, nu0, w0inv, ln_b_h0, ln_c_h0_eta)
        self._put(self._hview("zeta0", self.K * self.K), zeta0)
        self._put(self._hview("lncz0", 1), [ln_c_h0_zeta_sum])

    def set_hmm_params(self, eta, zeta, m, kappa, nu, winv):
        """Load (eta, zeta, m, kappa, nu, W^-1) as parameter set 0, reset the control words, compute all features."""
        self._put(self._hview("set_zeta", self.K * self.K, which=0), zeta)
        self.set_params(eta, m, kappa, nu, winv)

    def _small(self, mode, max_itr, tol):
        self._call(self.lib.bgmm_hmm_small, self.K, self.D, self.state.data_ptr(), self.hst.data_ptr(), mode, int(max_itr),
                   float(tol), self.hist_len, self._stream())

    def _pass(self, mode=_lib.HMM_FULL, force=0, beta_out=None):
        ptr = lambda t: 0 if t is None else t.data_ptr()  # noqa: E731
        if self.plan is not None:
            self._call(self.lib.bgmm_hmm_pass_seqs, self.x.data_ptr(), self.n_local, self.K, self.D, self.state.data_ptr(),
                       self.hst.data_ptr(), self.workspace.data_ptr(), ptr(self.scan_ws), ptr(self.lnrho_buf),
                       ptr(self.alpha_buf), ptr(self.gamma_buf), ptr(self.cs_buf), ptr(beta_out), mode, force,
                       self.plan.ctypes.data, self.plan_dev.data_ptr(), self._stream())
            return
        self._call(self.lib.bgmm_hmm_pass, self.x.data_ptr(), self.n_local, self.K, self.D, self.state.data_ptr(),
                   self.hst.data_ptr(), self.workspace.data_ptr(), ptr(self.scan_ws), ptr(self.lnrho_buf), ptr(self.alpha_buf),
                   ptr(self.gamma_buf), ptr(self.cs_buf), ptr(beta_out), mode, force, self._stream())

    def draw_random_init(self, seed):
        """The 'random_responsibility' initial state drawn on the device (bgmm_hmm_init_random, Philox keyed by `seed`
        and the element index): gamma into gamma_buf, sum xi into hst.MS, gamma summed over the sequence starts into
        hst.G0, hst.SC zeroed.  Over the sequences of set_sequences when it was given some."""
        n, K = self.n_local, self.K
        with torch.cuda.device(self.device):
            ws = torch.empty(int(self.lib.bgmm_hmm_init_random_workspace_doubles(K, n)), dtype=torch.float64,
                             device=self.device)
            starts_host = starts_dev = None
            n_seqs = 1
            if self.plan is not None:
                starts_host, starts_dev = self.seq_starts.ctypes.data, self._seq_starts_dev().data_ptr()
                n_seqs = self.seq_starts.size
            self._call(self.lib.bgmm_hmm_init_random, n, K, int(seed) & (2 ** 64 - 1), starts_host, starts_dev, n_seqs,
                       self.gamma_buf.data_ptr(), self.hst.data_ptr(), ws.data_ptr(), self._stream())

    def begin(self, max_itr, tol, init=None):
        """Post-init E-step + ELBO (:1092-1101) and the first M-step.  `init` for the 'random_responsibility'
        initialisation (:944-952): (gamma [n][K], ms [K][K]) drawn on the host, or an int, the seed of the device draw
        (draw_random_init); then the statistics of that gamma / xi, with ln rho = 0 and c = 1 as `_init_fb_params`
        (:934-942) leaves them."""
        self._max_itr, self._tol, self._launched = int(max_itr), float(tol), 0
        with torch.cuda.device(self.device):
            self._alloc_state(self._max_itr + 1)
            if init is not None:
                if isinstance(init, int):
                    self.draw_random_init(init)
                else:
                    gamma, ms = init
                    self.gamma_buf.copy_(torch.as_tensor(np.ascontiguousarray(gamma, dtype=np.float64)))
                    self._put(self._hview("ms", self.K * self.K), ms)
                    g0 = gamma[0] if self.seq_starts is None else gamma[self.seq_starts].sum(axis=0)
                    self._put(self._hview("g0", self.K), g0)
                    self._hview("sc", 8).zero_()
                self._pass(mode=_lib.HMM_STATS_FROM_GAMMA, force=1)
            else:
                self._pass()
            self._small(_lib.SMALL_ITERATE, self._max_itr, self._tol)

    def run(self, max_itr, tol, init=None, chunk=None):
        self.begin(max_itr, tol, init)
        step = 4 if chunk is None else int(chunk)
        done = self._max_itr == 0
        while not done:
            t0 = time.perf_counter()
            todo = self.enqueue(step)
            torch.cuda.current_stream(self.device).synchronize()
            done = self.finished()
            if chunk is None:
                per = (time.perf_counter() - t0) / max(todo, 1)
                step = int(min(64, max(1, 0.03 / max(per, 1e-6))))
        return self.finish()

    def fetch_params(self):
        out = super().fetch_params()
        K = self.K
        h = self.hst.cpu().numpy()
        cur = int(self.ctrl.cpu().numpy()[_lib.CTRL_CUR])
        base = self.hoff[f"set{cur}"]
        g = lambda name: h[base + self.hoff[name]: base + self.hoff[name] + K * K].reshape(K, K).copy()  # noqa: E731
        out.update({"zeta": g("set_zeta"), "ln_a_tilde": g("set_lna"), "a_tilde": g("set_at"),
                    "ln_c_zeta_sum": float(h[base + self.hoff["set_misc"] + 1]),
                    "ms": h[self.hoff["ms"]:self.hoff["ms"] + K * K].reshape(K, K).copy(),
                    "gamma0": h[self.hoff["g0"]:self.hoff["g0"] + K].copy(),
                    "sc": h[self.hoff["sc"]:self.hoff["sc"] + 2].copy(),
                    "window": int(h[self.hoff["sc"] + 2]),      # warm-up window of the last E-step (0 = basis + sweep path)
                    "vlx": h[self.hoff["vlx"]:self.hoff["vlx"] + 4].copy()})
        return out

    def viterbi(self, ln_pi_tilde, ln_a_tilde):
        """Most probable state path of the loaded sequence under the current parameter set (:1466-1480): the emission log
        densities (bgmm_hmm_pass, emission-only mode), then the max-plus recursion and the back-tracking on the device
        (bgmm_hmm_viterbi; bgmm_hmm_viterbi_seqs per sequence, in parallel, after set_sequences).
        -> (path [n] int64 numpy, omega [n][K] device tensor, phi [n][K] int32 device tensor)."""
        n, K = self.n_local, self.K
        with torch.cuda.device(self.device):
            self._call(self.lib.bgmm_hmm_pass, self.x.data_ptr(), n, K, self.D, self.state.data_ptr(), self.hst.data_ptr(),
                       self.workspace.data_ptr(), 0, self.lnrho_buf.data_ptr(), 0, 0, 0, 0, _lib.HMM_EMISSION_ONLY, 1,
                       self._stream())
            lnpi = torch.as_tensor(np.ascontiguousarray(ln_pi_tilde, dtype=np.float64)).to(self.device)
            lna = torch.as_tensor(np.ascontiguousarray(ln_a_tilde, dtype=np.float64)).to(self.device)
            omega = torch.empty((n, K), dtype=torch.float64, device=self.device)
            phi = torch.empty((n, K), dtype=torch.int32, device=self.device)
            path = torch.empty(n, dtype=torch.int32, device=self.device)
            if self.plan is not None:
                self._call(self.lib.bgmm_hmm_viterbi_seqs, n, K, self.lnrho_buf.data_ptr(), lnpi.data_ptr(), lna.data_ptr(),
                           omega.data_ptr(), phi.data_ptr(), path.data_ptr(), self._seq_starts_dev().data_ptr(),
                           self.seq_starts.size, self._stream())
                return path.cpu().numpy().astype(np.int64), omega, phi
            self._call(self.lib.bgmm_hmm_viterbi, n, K, self.lnrho_buf.data_ptr(), lnpi.data_ptr(), lna.data_ptr(),
                       omega.data_ptr(), phi.data_ptr(), path.data_ptr(), self._stream())
            return path.cpu().numpy().astype(np.int64), omega, phi

    def final_pass(self):
        """`_update_q_z` with the current parameters (:1133, :1490) keeping ln rho, alpha, beta, gamma, c on the device."""
        with torch.cuda.device(self.device):
            self.beta_buf = torch.empty((self.n_local, self.K), dtype=torch.float64, device=self.device)
            self._pass(force=1, beta_out=self.beta_buf)
            self._small(_lib.SMALL_STATS, 0, 0.0)
            host = self.state.cpu().numpy()
            h = self.hst.cpu().numpy()
        out = self._stats_from_host(host)
        K = self.K
        out["ms"] = h[self.hoff["ms"]:self.hoff["ms"] + K * K].reshape(K, K).copy()
        return out
