"""
CUDA engine: device memory / streams / collectives (torch) around the C ABI of
libevcplm.so.  This is the only execution path of the package -- there is no
CPU implementation behind it; construction raises EngineUnavailableError when
the library or a CUDA device is missing.

Multi-GPU (one process per GPU, torch.distributed / NCCL): sequences are
sharded in contiguous blocks over ranks, parameters are replicated, and every
objective evaluation does ONE all-reduce of the gradient (+ one 8-byte
all-reduce of -loglk); the regulariser and the whole L-BFGS update then run
identically (bit-for-bit, deterministic reductions) on every rank.  The Hamming
pass shards the upper-triangular pair tiles and all-reduces the int32 counters.
"""
import ctypes
import os
import time

import numpy as np

from . import _lib
from . import lbfgs as _lbfgs


# backward implementation of the data term: "gather" (shared-memory bucket kernel) or "tc" (tcgen05 GEMM)
DEFAULT_BACKWARD = "tc"
DEFAULT_FORWARD = "tc"
# arithmetic of the tensor-core products: "fp32" (bf16 hi+lo pairs, fp32-equivalent; default), "bf16" (one bf16
# product, BASELINE configs[4] "bf16 tiles / fp32 parameters"), "auto" (fit only: bf16 until close to convergence,
# then fp32 to the end)
DEFAULT_PRECISION = "fp32"
PRECISIONS = ("fp32", "bf16", "auto")


def _torch():
    import torch
    return torch


from .dist import Collective, shard_bounds   # noqa: E402,F401


class CudaEngine(object):
    def __init__(self, device=None, group=None, standalone=False):
        """``standalone=True``: ignore an initialised torch.distributed group (this process works alone on its
        GPU, e.g. rank 0 checking a sharded result against a single-GPU evaluation)."""
        self.lib = _lib.load()
        _lib.require_device()
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.EngineUnavailableError("torch sees no CUDA device; the PLM engine has no CPU fallback")
        self.coll = Collective(group, standalone=standalone)
        self.rank, self.world = self.coll.rank, self.coll.world
        if device is None:
            device = torch.cuda.current_device()
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        torch.cuda.set_device(self.device)
        self.kernel_launches = 0

    # -- helpers ---------------------------------------------------------------------------
    def stream(self):
        return ctypes.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def all_reduce(self, tensor):
        self.coll.all_reduce_sum(tensor)

    def agree_any(self, flag):
        """True on every rank if ``flag`` is true on any rank (doubles as the barrier after rank 0 wrote files)."""
        if self.world == 1:
            return bool(flag)
        t = _torch().tensor([1 if flag else 0], dtype=_torch().int32, device=self.device)
        self.coll.all_reduce_max(t)
        return bool(int(t.item()))

    @staticmethod
    def ptr(t):
        return ctypes.c_void_p(t.data_ptr())

    # -- (b) Hamming reweighting -----------------------------------------------------------
    def hamming_counts(self, codes, min_identical):
        """codes: (N, L) uint8 numpy (replicated on every rank).  Returns int32 numpy counts."""
        torch = _torch()
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        N, L = codes.shape
        if int(codes.max(initial=0)) >= 32:
            raise ValueError("sequence codes must be < 32")
        d_codes = torch.from_numpy(codes).to(self.device)
        d_counts = self.hamming_counts_device(d_codes, N, L, min_identical)
        return d_counts.cpu().numpy()

    def hamming_counts_device(self, d_codes, N, L, min_identical):
        torch = _torch()
        lib = self.lib
        words = lib.evc_hamming_plane_words(N, L)
        d_planes = torch.empty(words, dtype=torch.int32, device=self.device)
        d_counts = torch.zeros(N, dtype=torch.int32, device=self.device)
        _lib.check(lib.evc_hamming_pack(self.ptr(d_codes), N, L, self.ptr(d_planes), self.stream()),
                   "evc_hamming_pack")
        ntiles = lib.evc_hamming_num_tiles(N)
        lo, hi = shard_bounds(ntiles, self.world, self.rank)
        _lib.check(lib.evc_hamming_count_tiles(self.ptr(d_planes), N, L, int(min_identical), lo, hi,
                                               self.ptr(d_counts), self.stream()), "evc_hamming_count_tiles")
        self.kernel_launches += 2
        self.all_reduce(d_counts)
        return d_counts

    # -- mean-field DCA (fp64, csrc/mean_field.cu) ------------------------------------------------
    def mean_field(self, codes, weights, q, pseudo_count, timings=None):
        """Mean-field DCA of (N, L) codes (alphabet order, last state = reference state) with fp64 sequence
        weights, on device-resident buffers.  Returns float64 numpy arrays: fi, rfi (L, q), h (L, q), fij_tri and
        J_tri (pairs i<j, q, q), di, fn (zero-sum gauge), mi (pairs i<j) and di_iters.  ``timings``: a dict that
        receives the milliseconds of each stage (CUDA events on the engine's stream)."""
        torch = _torch()
        lib, vp = self.lib, self.ptr
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        N, L = codes.shape
        n, Lq, npairs = L * (q - 1), L * q, L * (L - 1) // 2
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        n_eff = float(weights.sum())
        dev, f64, st = self.device, torch.float64, self.stream()
        events = []

        def mark(name):
            if timings is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream(dev))
                events.append((name, ev))

        d_codes = torch.from_numpy(codes).to(dev)
        d_w = torch.from_numpy(weights).to(dev)
        mark("start")
        F = torch.empty((Lq, Lq), dtype=f64, device=dev)
        _lib.check(lib.evc_mf_weighted_counts_f64(vp(d_codes), vp(d_w), N, L, q, n_eff, vp(F), st),
                   "evc_mf_weighted_counts_f64")
        mark("counts")
        C = torch.empty((n, n), dtype=f64, device=dev)
        fi = torch.empty((L, q), dtype=f64, device=dev)
        rfi = torch.empty((L, q), dtype=f64, device=dev)
        fij = torch.empty((npairs, q, q), dtype=f64, device=dev)
        _lib.check(lib.evc_mf_covariance(vp(F), L, q, float(pseudo_count), vp(C), vp(fi), vp(rfi), vp(fij), st),
                   "evc_mf_covariance")
        mark("covariance")
        del F
        work = torch.empty((n, n), dtype=f64, device=dev)
        info = ctypes.c_int32(0)
        _lib.check(lib.evc_spd_inverse_f64(vp(C), n, vp(work), ctypes.byref(info), st), "evc_spd_inverse_f64")
        mark("inverse")
        del work
        J = torch.empty((npairs, q, q), dtype=f64, device=dev)
        h = torch.empty((L, q), dtype=f64, device=dev)
        _lib.check(lib.evc_mf_couplings_fields(vp(C), vp(rfi), L, q, vp(J), vp(h), st), "evc_mf_couplings_fields")
        mark("fields")
        del C
        di = torch.empty(npairs, dtype=f64, device=dev)
        iters = torch.empty(npairs, dtype=torch.int32, device=dev)
        _lib.check(lib.evc_mf_di_scores(vp(J), vp(rfi), L, q, vp(di), vp(iters), st), "evc_mf_di_scores")
        mark("di")
        scores = torch.empty((2, npairs), dtype=f64, device=dev)
        _lib.check(lib.evc_ec_scores_f64(vp(J), vp(fij), vp(fi), L, q, None, vp(scores[0]), vp(scores[1]), st),
                   "evc_ec_scores_f64")
        mark("scores")
        torch.cuda.synchronize(dev)
        if timings is not None:
            for (_, a), (name, b) in zip(events, events[1:]):
                timings[name] = a.elapsed_time(b)
        s = scores.cpu().numpy()
        return dict(fi=fi.cpu().numpy(), rfi=rfi.cpu().numpy(), h=h.cpu().numpy(), fij_tri=fij.cpu().numpy(),
                    J_tri=J.cpu().numpy(), di=di.cpu().numpy(), fn=s[0], mi=s[1], di_iters=iters.cpu().numpy())

    # -- (a) PLM ---------------------------------------------------------------------------
    def plm_problem(self, codes, weights, q, gap_code, lambda_h, lambda_J, m=6, backward=None, forward=None,
                    precision=None):
        return CudaPlmProblem(self, codes, weights, q, gap_code, lambda_h, lambda_J, m, backward, forward, precision)


class _DevicePointer(object):
    """Zero-copy torch view of library-owned device memory (CUDA array interface)."""

    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": "<f4", "data": (int(ptr), False),
                                         "version": 2}


class CudaPlmProblem(object):
    """PLM objective on this rank's sequence shard + the L-BFGS vector space
    (see lbfgs.py for the protocol).  All n-vectors are torch CUDA tensors."""

    def __init__(self, engine, codes, weights, q, gap_code, lambda_h, lambda_J, m=6, backward=None,
                 forward=None, precision=None):
        torch = _torch()
        if precision is None:
            precision = os.environ.get("EVC_PRECISION", DEFAULT_PRECISION)
        if precision not in PRECISIONS:
            raise ValueError("precision must be one of %s" % (PRECISIONS,))
        self.precision = precision
        if forward is None:
            forward = os.environ.get("EVC_FORWARD", DEFAULT_FORWARD)
        if forward not in ("gather", "tc", "tcfused"):
            raise ValueError("forward must be 'gather', 'tc' or 'tcfused'")
        if forward in ("tc", "tcfused"):
            backward = "tc"
        self.forward = forward
        if backward is None:
            backward = os.environ.get("EVC_BACKWARD", DEFAULT_BACKWARD)
        if backward not in ("gather", "tc"):
            raise ValueError("backward must be 'gather' or 'tc'")
        self.backward = backward
        self.engine = engine
        self.lib = engine.lib
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        weights = np.ascontiguousarray(weights, dtype=np.float32)
        N, L = codes.shape
        if weights.shape != (N,):
            raise ValueError("weights must have one entry per sequence")
        n_states = int(q) + (1 if int(gap_code) >= 0 else 0)
        if N and int(codes.max()) >= n_states:
            raise ValueError("sequence codes must be < %d (q%s)" % (n_states, " + ignored gap" if gap_code >= 0 else ""))
        self.N_total, self.L, self.q, self.gap_code = N, L, int(q), int(gap_code)
        self.lambda_h, self.lambda_J = float(lambda_h), float(lambda_J)
        lo, hi = shard_bounds(N, engine.world, engine.rank)
        if hi <= lo:
            raise ValueError("fewer sequences than ranks")
        self.shard = (lo, hi)
        c_shard = np.ascontiguousarray(codes[lo:hi])
        w_shard = np.ascontiguousarray(weights[lo:hi])
        self.handle = ctypes.c_void_p()
        _lib.check(self.lib.evc_plm_create(ctypes.byref(self.handle), c_shard.ctypes.data_as(ctypes.c_void_p),
                                           hi - lo, L, self.q, self.gap_code,
                                           w_shard.ctypes.data_as(ctypes.c_void_p), engine.device_index),
                   "evc_plm_create")
        if backward == "tc":
            _lib.check(self.lib.evc_plm_set_backward(self.handle, 1), "evc_plm_set_backward")
        if forward in ("tc", "tcfused"):
            _lib.check(self.lib.evc_plm_set_forward(self.handle, 2 if forward == "tcfused" else 1),
                       "evc_plm_set_forward")
        if precision == "bf16":
            _lib.check(self.lib.evc_plm_set_precision(self.handle, 1), "evc_plm_set_precision")
        self.n = int(self.lib.evc_plm_num_params(self.handle))
        dev = engine.device
        self.m = m
        f32 = dict(dtype=torch.float32, device=dev)
        self.x = torch.zeros(self.n, **f32)
        # gradient + 4 trailing floats: -loglk rides behind g as exact fixed-point limbs => ONE all-reduce
        self.g_packed = torch.zeros(self.n + 4, **f32)
        self.g = self.g_packed[:self.n]
        self._python_space = False          # vectors of the Python L-BFGS driver are allocated on demand
        self.fxbuf = torch.zeros(2, dtype=torch.float64, device=dev)
        self.dotbuf = torch.zeros(1, dtype=torch.float64, device=dev)
        self.last_negloglk = float("nan")
        self.evaluations = 0
        # own kernels per evaluate(): expand, fwd, bwd, finalize pairs + fields, add_reg x2
        self.launches_per_eval = {"tc": 8, "tcfused": 7, "gather": 7}[forward]

    def close(self):
        if self.handle:
            self.lib.evc_plm_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- objective ----------------------------------------------------------------------------
    def evaluate_async(self, x):
        """Launch data term + all-reduce + regulariser on the current stream; results in self.g / self.fxbuf."""
        e, p = self.engine, self.engine.ptr
        _lib.check(self.lib.evc_plm_eval_data(self.handle, p(x), p(self.g), p(self.fxbuf), e.stream()),
                   "evc_plm_eval_data")
        if e.world > 1:
            limbs = self.g_packed[self.n:]
            _lib.check(self.lib.evc_plm_pack_fx(p(self.fxbuf), p(limbs), e.stream()), "evc_plm_pack_fx")
            timed = getattr(self, "time_collective", False)
            if timed:
                torch = _torch()
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                ev[0].record()
            e.all_reduce(self.g_packed)                     # ONE collective: [g, -loglk]
            if timed:
                ev[1].record()
                self.collective_events.append(ev)
            _lib.check(self.lib.evc_plm_unpack_fx(p(limbs), p(self.fxbuf), e.stream()), "evc_plm_unpack_fx")
            e.kernel_launches += 2
        _lib.check(self.lib.evc_plm_add_regulariser(self.handle, p(x), p(self.g), p(self.fxbuf),
                                                    self.lambda_h, self.lambda_J, e.stream()),
                   "evc_plm_add_regulariser")
        self.evaluations += 1
        e.kernel_launches += self.launches_per_eval

    def evaluate(self, x):
        self.evaluate_async(x)
        nll, fx = self.fxbuf.tolist()
        self.last_negloglk = nll
        return fx

    def evaluate_host(self, x_host, g_host):
        """Public host-buffer entry: x_host / g_host are CPU float32 torch tensors (pinned for speed).
        H2D of x, evaluation (incl. the all-reduce), D2H of the gradient and of fx, then synchronise."""
        self.x.copy_(x_host, non_blocking=True)
        self.evaluate_async(self.x)
        g_host.copy_(self.g, non_blocking=True)
        nll, fx = self.fxbuf.tolist()          # D2H of the result scalars; synchronises the stream
        self.last_negloglk = nll
        return fx

    # -- vector space protocol (Python L-BFGS driver, kept for comparison / tests) -------------------
    def _ensure_python_space(self):
        if self._python_space:
            return
        torch = _torch()
        f32 = dict(dtype=torch.float32, device=self.engine.device)
        m = self.m
        self.xp = torch.zeros(self.n, **f32)
        self.gp = torch.zeros(self.n, **f32)
        self.d = torch.zeros(self.n, **f32)
        self.S = torch.zeros((m, self.n), **f32)
        self.Y = torch.zeros((m, self.n), **f32)
        self.ys = torch.zeros(m, dtype=torch.float64, device=self.engine.device)
        self.scratch = torch.zeros(m + 2, dtype=torch.float64, device=self.engine.device)
        self._python_space = True

    def dot(self, a, b):
        e = self.engine
        _lib.check(self.lib.evc_vec_dot(e.ptr(a), e.ptr(b), self.n, e.ptr(self.dotbuf), e.stream()), "evc_vec_dot")
        e.kernel_launches += 2
        return float(self.dotbuf.item())

    def copy(self, dst, src):
        e = self.engine
        _lib.check(self.lib.evc_vec_copy(e.ptr(dst), e.ptr(src), self.n, e.stream()), "evc_vec_copy")

    def axpby(self, y, x, a, b):
        e = self.engine
        _lib.check(self.lib.evc_vec_axpby(e.ptr(y), e.ptr(x), float(a), float(b), self.n, e.stream()),
                   "evc_vec_axpby")
        e.kernel_launches += 1

    def update_pair(self, slot, xp, gp):
        e, p = self.engine, self.engine.ptr
        _lib.check(self.lib.evc_lbfgs_update_pair(p(self.S[slot]), p(self.Y[slot]), p(self.x), p(xp), p(self.g),
                                                  p(gp), p(self.ys[slot:slot + 1]), p(self.scratch[0:1]),
                                                  self.n, e.stream()), "evc_lbfgs_update_pair")
        e.kernel_launches += 3

    def direction(self, d, bound, end):
        e, p = self.engine, self.engine.ptr
        _lib.check(self.lib.evc_lbfgs_direction(p(d), p(self.g), p(self.S), p(self.Y), p(self.ys), p(self.scratch),
                                                self.n, self.m, int(bound), int(end), e.stream()),
                   "evc_lbfgs_direction")
        e.kernel_launches += 2 + 6 * int(bound)

    # -- a6 / a10 ---------------------------------------------------------------------------------
    def weighted_counts(self):
        """Returns (fi_counts (L,q), fij_counts (npairs,q,q)) float64 numpy, summed over all ranks."""
        torch = _torch()
        e = self.engine
        L, q = self.L, self.q
        buf = torch.zeros(self.n, dtype=torch.float32, device=e.device)
        _lib.check(self.lib.evc_plm_weighted_counts(self.handle, e.ptr(buf), e.ptr(buf[L * q:]), e.stream()),
                   "evc_plm_weighted_counts")
        e.kernel_launches += 5
        e.all_reduce(buf)
        host = buf.cpu().numpy().astype(np.float64)
        return host[:L * q].reshape(L, q), host[L * q:].reshape(L * (L - 1) // 2, q, q)

    def fn_scores(self, x=None):
        torch = _torch()
        e = self.engine
        x = self.x if x is None else x
        L, q = self.L, self.q
        out = torch.zeros(L * (L - 1) // 2, dtype=torch.float32, device=e.device)
        _lib.check(self.lib.evc_fn_scores(e.ptr(x[L * q:]), L, q, e.ptr(out), e.stream()), "evc_fn_scores")
        e.kernel_launches += 1
        return out.cpu().numpy()

    def set_x(self, x_host):
        torch = _torch()
        self.x.copy_(torch.from_numpy(np.ascontiguousarray(x_host, dtype=np.float32)))

    def get_x(self):
        return self.x.cpu().numpy()

    def norms(self):
        """(|h|, |J|) of the current parameters (for the iteration table)."""
        import math
        cached = getattr(self, "_cached_norms", None)
        if cached is not None:                  # evc_plm_fit reports them with every iteration
            return cached
        e = self.engine
        nh = self.L * self.q
        out = []
        for lo, n in ((0, nh), (nh, self.n - nh)):
            v = self.x[lo:lo + n]
            _lib.check(self.lib.evc_vec_dot(e.ptr(v), e.ptr(v), n, e.ptr(self.dotbuf), e.stream()), "evc_vec_dot")
            e.kernel_launches += 2
            out.append(math.sqrt(float(self.dotbuf.item())))
        return out[0], out[1]

    def fit(self, x0, params, progress=None, driver="device"):
        """Minimise from x0.  driver "device": the whole L-BFGS loop runs inside libevcplm (evc_plm_fit);
        "python": the same algorithm with host-side control (lbfgs.py), kept for comparison.
        ``progress(k, fx, xnorm, gnorm, step, n_ls)``; returns lbfgs.LbfgsResult."""
        self.set_x(x0)
        if driver == "python":
            self._ensure_python_space()
            self._cached_norms = None
            return _lbfgs.minimize(self, params, progress)
        return self._fit_device(params, progress)

    def _fit_device(self, params, progress):
        e, lib = self.engine, self.lib
        torch = _torch()
        fp = _lib.FitParams()
        lib.evc_fit_default_params(ctypes.byref(fp))
        fp.max_iterations, fp.m, fp.epsilon = int(params.max_iterations), int(params.m), float(params.epsilon)
        fp.lambda_h, fp.lambda_J = self.lambda_h, self.lambda_J
        fp.max_linesearch = int(params.max_linesearch)
        fp.min_step, fp.max_step = float(params.min_step), float(params.max_step)
        fp.ftol, fp.gtol, fp.xtol = float(params.ftol), float(params.gtol), float(params.xtol)
        fp.precision_schedule = 1 if self.precision == "auto" else 0
        errors = []
        views = {}

        stats = {"allreduce_calls": 0, "allreduce_callback_s": 0.0}

        def allreduce(user, d_buf, count, stream):
            try:
                t_cb = time.perf_counter()
                key = (d_buf, count)
                if key not in views:
                    views[key] = torch.as_tensor(_DevicePointer(d_buf, count), device=e.device)
                e.all_reduce(views[key])
                stats["allreduce_calls"] += 1
                stats["allreduce_callback_s"] += time.perf_counter() - t_cb      # host time only (the collective is async)
                return 0
            except BaseException as exc:          # never let an exception cross the C boundary
                errors.append(exc)
                return 1

        def on_iteration(user, k, fx, xnorm, gnorm, step, n_ls, nll, hnorm, enorm):
            try:
                self.last_negloglk = nll
                self._cached_norms = (hnorm, enorm)
                if progress is not None and progress(k, fx, xnorm, gnorm, step, n_ls):
                    return 1
                return 0
            except BaseException as exc:
                errors.append(exc)
                return 1

        ar_cb = _lib.ALLREDUCE_CB(allreduce) if e.world > 1 else None
        pr_cb = _lib.PROGRESS_CB(on_iteration)
        res = _lib.FitResult()
        rc = lib.evc_plm_fit(self.handle, e.ptr(self.x), ctypes.byref(fp),
                             ctypes.cast(ar_cb, ctypes.c_void_p) if ar_cb is not None else None, None,
                             ctypes.cast(pr_cb, ctypes.c_void_p), None, ctypes.byref(res), e.stream())
        self._cached_norms = None
        if errors:
            raise errors[0]
        _lib.check(rc, "evc_plm_fit")
        self.last_negloglk = res.negloglk
        self.evaluations += res.evaluations
        e.kernel_launches += res.evaluations * (self.launches_per_eval + 2)
        self.fit_seconds = res.seconds
        self.switched_at = res.switched_at
        self.fit_stats = dict(stats, fit_s=res.seconds, evaluations=res.evaluations, iterations=res.iterations)
        return _lbfgs.LbfgsResult(_lib.LBFGS_STATUS.get(res.status, "LBFGSERR_UNKNOWNERROR"), res.iterations,
                                  res.fx, res.evaluations)
