"""CasADi-shaped facade over the C ABI: the one line a reference script swaps.

Reference (Python/NMPC_TT.py:250-267, :358-367):
    solver = ca.nlpsol('solver', 'ipopt', nlp_prob, opts)
    sol = solver(x0=args['x0'], lbx=args['lbx'], ubx=args['ubx'], lbg=args['lbg'], ubg=args['ubg'], p=args['p'])
    u = ca.reshape(sol['x'], n_controls, N)
Here:
    solver = b200nmpc.nlpsol('solver', 'ipm', scenario_or_dict, opts)       # nlp_prob -> problem constants
    sol = solver(x0=..., lbx=..., ubx=..., lbg=..., ubg=..., p=...)          # same keywords, same layouts
    u = sol['x'].reshape(N, 6).T

Every argument may be a single instance ((n,), (n,1), list) or a batch (B, n); host containers (numpy, lists)
go through nmpc_solve_host (copies inside), torch CUDA float64 tensors are used in place on torch's current
stream.  Like CasADi's nlpsol the call never raises on a non-converged instance: the outcome is in
solver.stats() ('return_status', 'success', 'iter_count'), which the reference never reads (:358-367).
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import Any, Dict, Optional

import numpy as np

from . import _ffi
from .scenarios import NP, NU, Scenario

try:  # torch is plumbing for device memory / streams only
    import torch
except Exception:  # pragma: no cover
    torch = None


def _is_cuda_tensor(a) -> bool:
    return torch is not None and isinstance(a, torch.Tensor) and a.is_cuda


def _spec_from(problem, opts: Optional[dict]) -> Dict[str, Any]:
    if isinstance(problem, Scenario):
        d = dict(T=problem.T, N=problem.N, obstacles=problem.obstacle_table(), w1=problem.w1, w2=problem.w2,
                 vfov=problem.vfov, hfov=problem.hfov, model=problem.model)
    else:
        d = dict(problem)
        if "obstacles" in d:
            o = np.asarray(d["obstacles"], dtype=np.float64).reshape(-1, 3).copy()
            o[:, 2] += float(d.get("uav_r", 5.0))
            d["obstacles"] = o
        else:
            d["obstacles"] = np.zeros((int(d.get("n_obs", 0)), 3))
    ip = dict((opts or {}).get("ipopt", {}))
    d["max_iter"] = int(ip.get("max_iter", 100))          # NMPC_TT.py:259
    d["tol"] = float(ip.get("tol", 1e-8))
    d["scaling"] = 0 if ip.get("nlp_scaling_method", "gradient-based") == "none" else int(ip.get("_scaling_debug_mode", 1))
    # NON-REFERENCE mode (no script sets it): IPOPT's warm_start_init_point and its pushes; lam_x0 / lam_g0 are ignored without it
    d["warm"] = str(ip.get("warm_start_init_point", "no")).lower() == "yes"
    d["warm_opts"] = (float(ip.get("mu_init", 0.0)) if d["warm"] else 0.0, float(ip.get("warm_start_bound_push", 0.0)),
                      float(ip.get("warm_start_bound_frac", 0.0)), float(ip.get("warm_start_slack_bound_push", 0.0)),
                      float(ip.get("warm_start_slack_bound_frac", 0.0)), float(ip.get("warm_start_mult_bound_push", 0.0)))
    return d


class _Sol(dict):
    """Result dict of a solve.  The keys in `lazy` are computed on first access instead of on every call: sol['lam_p'] -- the
    sixth key of CasADi's result dict, which no reference script reads -- (one small launch, nmpc_lam_p), and with want_jac
    sol['jac_x_p'] / sol['jac_x_w'] (nmpc_sensitivity)."""

    def __init__(self, items, lam_p_fn=None, lazy=None):
        super().__init__(items)
        self._lazy = dict(lazy or {})
        if lam_p_fn is not None:
            self._lazy["lam_p"] = lam_p_fn
        for k in self._lazy:
            super().__setitem__(k, None)

    def __getitem__(self, k):
        fn = self._lazy.pop(k, None)
        if fn is not None:
            super().__setitem__(k, fn())
        return super().__getitem__(k)

    def get(self, k, default=None):
        return self[k] if k in self else default

    def items(self):
        return [(k, self[k]) for k in self.keys()]

    def values(self):
        return [self[k] for k in self.keys()]


class Solver:
    """Callable returned by nlpsol(); owns one nmpc_handle."""

    def __init__(self, name: str, problem, opts: Optional[dict] = None, device: int = 0, max_batch: int = 1, fill: int = 1):
        self.name = name
        self.fill = int(fill)
        d = _spec_from(problem, opts)
        self.T, self.N = float(d["T"]), int(d["N"])
        self.obstacles = np.ascontiguousarray(d["obstacles"], dtype=np.float64)
        self.n_obs = self.obstacles.shape[0]
        self.model = int(d.get("model", 0))     # 0: the scripts' 8-state UAV + camera; 1: the gimbal-less 5-state tracker (nmpc_b200.h)
        self.n_p = 8 if self.model else NP
        self.n_w, self.n_g = (3 if self.model else NU) * self.N, ((2 if self.model else 5) + self.n_obs) * (self.N + 1)
        self.device = device
        self._d = d
        self._h = C.c_void_p()
        self._max_batch = 0
        self._dev_cache: Dict[str, Any] = {}
        self._stats: Dict[str, Any] = {}
        self._warm = None
        self._sched = None
        self._held: Dict[str, Any] = {}      # tensors of the last call's per-call settings (_setting)
        self._solves = 0                     # solve calls so far: the handle's kept barrier data belongs to the last one
        self._create(max_batch)

    # -- handle management ---------------------------------------------------------------------
    def _create(self, max_batch: int):
        L = _ffi.lib()
        if self._h:
            L.nmpc_destroy(self._h)
            self._h = C.c_void_p()
        d = self._d
        spec = _ffi.NmpcSpec(self.T, self.N, self.n_obs, float(d.get("w1", 1.0)), float(d.get("w2", 2.0)),
                             float(d.get("vfov", 1.0)), float(d.get("hfov", 1.0)),
                             d["max_iter"], d["scaling"], d["tol"], int(max_batch), self.fill, self.model)
        _ffi.check(L.nmpc_create(C.byref(spec), self.device, C.byref(self._h)), "nmpc_create")
        self._max_batch = max_batch
        self.spec = spec

    def close(self):
        if self._h:
            _ffi.lib().nmpc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers ---------------------------------------------------------------------------------
    def _dev_const(self, key: str, arr) -> "torch.Tensor":
        """Device copy of a batch-shared vector (bounds, obstacle table), cached by content."""
        if _is_cuda_tensor(arr):
            return arr.to(torch.float64).contiguous().view(-1)
        a = np.ascontiguousarray(np.asarray(arr, dtype=np.float64).reshape(-1))
        hit = self._dev_cache.get(key)
        if hit is not None and hit[0].shape == a.shape and np.array_equal(hit[0], a):
            return hit[1]
        t = torch.from_numpy(a.copy()).to(f"cuda:{self.device}")
        self._dev_cache[key] = (a.copy(), t)
        return t

    @staticmethod
    def _host(a, n: int, what: str = "argument", shared: bool = False) -> np.ndarray:
        """Host container -> contiguous float64 [rows, n].  Raises ValueError on a wrong length (the C ABI takes plain
        pointers: a short vector would be read past its end).  shared: a batch-shared vector (bounds), exactly n entries."""
        if torch is not None and isinstance(a, torch.Tensor):
            a = a.detach().cpu().numpy()
        a = np.asarray(a, dtype=np.float64)
        if a.ndim == 2 and a.shape[1] == 1 and a.shape[0] == n:   # CasADi column vector
            a = a.reshape(1, n)
        if a.ndim == 2 and a.shape[1] != n:
            raise ValueError(f"solver: {what} has {a.shape[1]} columns, expected {n}")
        if a.ndim != 2:
            if a.size % n != 0 or a.size == 0:
                raise ValueError(f"solver: {what} has {a.size} entries, expected a multiple of {n}")
            a = a.reshape(-1, n)
        if shared and a.shape[0] != 1:
            raise ValueError(f"solver: {what} must have exactly {n} entries (it is shared by the batch), got {a.size}")
        return np.ascontiguousarray(a)

    # -- the call --------------------------------------------------------------------------------
    def __call__(self, x0=None, p=None, lbx=None, ubx=None, lbg=None, ubg=None, obstacles=None,
                 want_g: bool = True, want_lam: bool = True, order=None, weights=None, target_traj=None,
                 blocking: bool = True, lam_x0=None, lam_g0=None, want_jac: bool = False):
        """lam_x0 [B, n_w], lam_g0 [B, n_g]: CasADi's multiplier guesses.  Like IPOPT they are ignored unless the solver was
        built with opts = {'ipopt': {'warm_start_init_point': 'yes', ...}} (no reference script does: non-reference fast mode,
        nmpc_set_warm_start); a NaN in lam_x0[b, 0] cold-starts instance b.
        weights: optional [B, 2] per-instance cost weights (w1, w2) for this call (numpy or CUDA tensor); the
        reference edits them in source (NMPC_TT.py:204-205) and its MATLAB outer loop sweeps them (MPC.m:90).
        target_traj: optional [B, N, 2] predicted target positions per stage (default: p[8:10] for every stage, as
        in the reference).
        blocking=False (host buffers only): enqueue the copies and the solve and return at once; the outputs are
        page-locked arrays owned by this solver that become valid after `solver.wait()` and are reused by the next
        call.  Pass page-locked inputs (torch pin_memory) for the copies to overlap.
        want_jac (blocking calls): the result also has sol['jac_x_p'] [B, n_w, n_p] = dx*/dp (CasADi's jac:x:p) and, for model 0,
        sol['jac_x_w'] [B, n_w, 2] = dx*/d(w1, w2), computed on first access (nmpc_sensitivity; the solve keeps its barrier data,
        NMPC_KEEP_BARRIER, and its results do not change).  With obstacle rows there is also sol['jac_x_obst'] [B, n_w, n_obs, 3]
        = dx*/d(cx, cy, r_uav + r_obs) of each obstacle of the call's table (shared or per instance), computed by its own launch on
        first access (nmpc_sensitivity_obstacles).  They must be read before the next solve on this solver.  Rows of
        instances that did not converge, or whose reduced Hessian is not positive definite (no sensitivity exists), are NaN.
        The theta_t column is 0, and so are the target columns with target_traj.  want_jac implies want_lam."""
        if p is None:
            raise ValueError("solver: p is required")
        if any(v is None for v in (lbx, ubx, lbg, ubg)):
            raise ValueError("solver: lbx, ubx, lbg, ubg are required (the reference passes all four)")
        warm = self._d["warm"] and lam_x0 is not None and lam_g0 is not None
        if warm and not _is_cuda_tensor(p):       # the multiplier guesses live on the device: take the device path, hand numpy back
            dev = f"cuda:{self.device}"
            t = lambda a, n: None if a is None else torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev).reshape(-1, n)
            out = self(x0=t(x0, self.n_w), p=t(p, self.n_p), lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg, obstacles=obstacles, want_g=want_g,
                       want_lam=want_lam, order=order, weights=weights, target_traj=target_traj, lam_x0=lam_x0, lam_g0=lam_g0,
                       want_jac=want_jac)
            torch.cuda.synchronize()
            self._stats = {k: v.cpu().numpy() for k, v in self._stats.items()}
            return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}
        B = self._batch_of(p)
        if B > self._max_batch and not _is_cuda_tensor(p):     # spec.max_batch sizes the staging buffers of the host path only
            self._create(max(B, 2 * self._max_batch))
        with self._settings(B, weights, target_traj) as stack:
            if warm:
                self.set_warm_start(torch.as_tensor(lam_x0, dtype=torch.float64, device=p.device).reshape(B, self.n_w),
                                    torch.as_tensor(lam_g0, dtype=torch.float64, device=p.device).reshape(B, self.n_g))
                stack.callback(self.set_warm_start, None, None)
            jac = (weights, target_traj) if want_jac else None
            if _is_cuda_tensor(p):
                return self._call_device(x0, p, lbx, ubx, lbg, ubg, obstacles, want_g, want_lam, order, jac)
            if jac is not None and not blocking:
                raise ValueError("solver: want_jac needs a blocking call")
            return self._call_host(x0, p, lbx, ubx, lbg, ubg, obstacles, want_g, want_lam, blocking, jac)

    def wait(self):
        """Complete a blocking=False call (nmpc_synchronize)."""
        _ffi.check(_ffi.lib().nmpc_synchronize(self._h), "nmpc_synchronize")

    def done(self) -> bool:
        """True when no blocking=False call is in flight any more (nmpc_query; never blocks)."""
        busy = C.c_int32(0)
        _ffi.check(_ffi.lib().nmpc_query(self._h, C.byref(busy)), "nmpc_query")
        return busy.value == 0

    def _pinned(self, key: str, shape, dtype=np.float64):
        """Page-locked output buffer, cached per (name, shape)."""
        k = ("pin", key, tuple(shape), np.dtype(dtype).str)
        buf = self._dev_cache.get(k)
        if buf is None:
            t = torch.empty(tuple(shape), dtype=torch.float64 if dtype == np.float64 else torch.int32).pin_memory()
            buf = (t, t.numpy())
            self._dev_cache[k] = buf
        return buf[1]

    def _batch_of(self, p) -> int:
        """Batch size of a parameter argument in any of the accepted containers (list, numpy, torch; (11,), (11,1), (B,11))."""
        if _is_cuda_tensor(p):
            return int(p.numel() // self.n_p)
        return int(np.asarray(p, dtype=np.float64).size // self.n_p)

    @contextlib.contextmanager
    def _setting(self, setter: str, *tensors):
        """One per-call handle setting (nmpc_set_weights, nmpc_set_target_trajectory, nmpc_set_obstacle_motion) for the duration
        of a call.  The tensors stay referenced afterwards: the kernel may read them later (device call, or blocking=False)."""
        fn = getattr(_ffi.lib(), setter)
        _ffi.check(fn(self._h, *(t.data_ptr() for t in tensors)), setter)
        try:
            yield
        finally:
            self._held[setter] = tensors
            fn(self._h, *(None for _ in tensors))

    def _settings(self, B, weights=None, target_traj=None, obstacles=None, obstacle_vel=None) -> contextlib.ExitStack:
        """The per-call settings of a call of B instances as one context, all validated before the first is applied.
        obstacle_vel: the kernel moves `obstacles` in place after the solve (fused calls only)."""
        rows = lambda a, *shape: torch.as_tensor(a if _is_cuda_tensor(a) else np.asarray(a, dtype=np.float64), dtype=torch.float64,
                                                 device=f"cuda:{self.device}").reshape(-1, *shape).contiguous()
        todo = []
        if weights is not None:
            w = rows(weights, 2)
            if w.shape[0] != B:
                raise ValueError("solver: weights must be [B, 2]")
            todo.append(("nmpc_set_weights", w))
        if target_traj is not None:
            t = rows(target_traj, self.N, 2)
            if t.shape[0] != B:
                raise ValueError("solver: target_traj must be [B, N, 2]")
            todo.append(("nmpc_set_target_trajectory", t))
        if obstacle_vel is not None:
            if self.n_obs == 0:
                raise ValueError("solver: obstacle_vel given, but this solver has no obstacle rows")
            if not (_is_cuda_tensor(obstacles) and obstacles.dtype == torch.float64 and obstacles.is_contiguous()
                    and tuple(obstacles.shape) == (B, self.n_obs, 3)):
                raise ValueError(f"solver: moving obstacles (obstacle_vel) need obstacles as a contiguous CUDA float64 [B, n_obs, 3] = "
                                 f"[{B}, {self.n_obs}, 3] tensor, which is moved in place")
            if not (_is_cuda_tensor(obstacle_vel) and obstacle_vel.dtype == torch.float64 and tuple(obstacle_vel.shape) == (B, self.n_obs, 2)):
                raise ValueError(f"solver: obstacle_vel must be a CUDA float64 [B, n_obs, 2] = [{B}, {self.n_obs}, 2] tensor")
            if obstacle_vel.device != obstacles.device:
                raise ValueError("solver: obstacles and obstacle_vel must be on the same device")
            todo.append(("nmpc_set_obstacle_motion", obstacles, obstacle_vel.contiguous()))
        with contextlib.ExitStack() as stack:
            for setter, *tensors in todo:
                stack.enter_context(self._setting(setter, *tensors))
            return stack.pop_all()

    def _obs_flag(self, size: int, B: int) -> int:
        """The obstacle shape rule: 3 n_obs entries are one table shared by the batch, 3 n_obs B entries one table per instance."""
        if size == 3 * self.n_obs:
            return 0
        if size == 3 * self.n_obs * B:
            return _ffi.NMPC_OBS_PER_INSTANCE
        raise ValueError("solver: obstacles must be [n_obs,3] or [B,n_obs,3] of (cx, cy, r_uav + r_obs)")

    def _obst(self, obstacles, B):
        if obstacles is None:
            return self.obstacles, 0
        o = obstacles.detach().cpu().numpy() if (torch is not None and isinstance(obstacles, torch.Tensor)) else obstacles
        o = np.ascontiguousarray(np.asarray(o, dtype=np.float64))
        return o, self._obs_flag(o.size, B)

    def _dev_inputs(self, B: int, obstacles, bounds=()):
        """The batch-shared inputs of a device call of B instances: the bounds (lbx, ubx, lbg, ubg) as cached device copies,
        length-checked, and the obstacle table with its flag.  A contiguous CUDA float64 obstacle tensor is used as it is
        (nmpc_set_obstacle_motion registers it and the kernel moves it in place)."""
        dev_bounds = []
        for key, a, n in zip(("lbx", "ubx", "lbg", "ubg"), bounds, (self.n_w, self.n_w, self.n_g, self.n_g)):
            dev_bounds.append(self._dev_const(key, a))
            if dev_bounds[-1].numel() != n:
                raise ValueError("solver: bound vector has the wrong length")
        if obstacles is None:
            return dev_bounds, self._dev_const("obs", self.obstacles), 0
        if _is_cuda_tensor(obstacles):
            obs = obstacles.to(torch.float64).contiguous()
            return dev_bounds, obs, self._obs_flag(obs.numel(), B)
        o, flags = self._obst(obstacles, B)
        return dev_bounds, torch.from_numpy(o).to(f"cuda:{self.device}"), flags

    def _call_host(self, x0, p, lbx, ubx, lbg, ubg, obstacles, want_g, want_lam, blocking=True, jac=None):
        L = _ffi.lib()
        want_lam = want_lam or jac is not None
        single = np.asarray(p).ndim == 1 or (np.asarray(p).ndim == 2 and np.asarray(p).shape[1] == 1)
        p = self._host(p, self.n_p, "p")
        B = p.shape[0]
        x0 = np.zeros((B, self.n_w)) if x0 is None else self._host(x0, self.n_w, "x0")
        if x0.shape[0] != B:
            raise ValueError("solver: x0 and p disagree on the batch size")
        lbx, ubx = self._host(lbx, self.n_w, "lbx", True), self._host(ubx, self.n_w, "ubx", True)
        lbg, ubg = self._host(lbg, self.n_g, "lbg", True), self._host(ubg, self.n_g, "ubg", True)
        obs, flags = self._obst(obstacles, B)
        new = (lambda k, shape, dt=np.float64: np.empty(shape, dtype=dt)) if blocking else self._pinned
        x = new("x", (B, self.n_w)); f = new("f", (B,))
        g = new("g", (B, self.n_g)) if want_g else None
        lam_x = new("lam_x", (B, self.n_w)) if want_lam else None
        lam_g = new("lam_g", (B, self.n_g)) if want_lam else None
        status = new("status", (B,), np.int32); iters = new("iters", (B,), np.int32)
        ptr = lambda a: None if a is None else a.ctypes.data
        fn = L.nmpc_solve_host if blocking else L.nmpc_solve_host_async
        if not blocking:
            self._keep = (p, x0, lbx, ubx, lbg, ubg, obs)      # inputs stay alive until wait()
        self._solves += 1
        _ffi.check(fn(self._h, B, ptr(p), ptr(x0), ptr(lbx), ptr(ubx), ptr(lbg), ptr(ubg), ptr(obs), flags | (_ffi.NMPC_KEEP_BARRIER if jac else 0),
                      ptr(x), ptr(f), ptr(g), ptr(lam_x), ptr(lam_g), ptr(status), ptr(iters)),
                   "nmpc_solve_host")
        self._stats = dict(return_status=status, iter_count=iters)      # success is derived in stats(): valid after wait()
        def lam_p_host():      # CasADi's result dict also carries lam_p (nobody in the reference reads it): on first access
            dev = f"cuda:{self.device}"
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
            xd, pd, ld, od = up(x), up(p), up(lam_g), up(obs)
            lp = torch.empty((B, self.n_p), dtype=torch.float64, device=dev)
            _ffi.check(L.nmpc_lam_p(self._h, B, xd.data_ptr(), pd.data_ptr(), od.data_ptr() if od.numel() else None, flags, ld.data_ptr(),
                                    lp.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), "nmpc_lam_p")
            r = lp.cpu().numpy()
            return r[0] if single else r
        out = dict(x=x, f=f, g=g, lam_x=lam_x, lam_g=lam_g)
        if single:
            out = {k: (v[0] if v is not None else None) for k, v in out.items()}
        lazy = self._jac_keys(B, single, True, x, p, lam_g, obs, flags, status, *jac) if jac is not None else None
        return _Sol(out, lam_p_host if (want_lam and blocking) else None, lazy)

    def _call_device(self, x0, p, lbx, ubx, lbg, ubg, obstacles, want_g, want_lam, order=None, jac=None):
        L = _ffi.lib()
        want_lam = want_lam or jac is not None
        dev = p.device
        single = p.dim() == 1
        p = p.to(torch.float64).reshape(-1, self.n_p).contiguous()
        B = p.shape[0]
        x0 = torch.zeros((B, self.n_w), dtype=torch.float64, device=dev) if x0 is None else x0.to(torch.float64).reshape(B, self.n_w).contiguous()
        (lbx, ubx, lbg, ubg), obs, flags = self._dev_inputs(B, obstacles, (lbx, ubx, lbg, ubg))
        x = torch.empty((B, self.n_w), dtype=torch.float64, device=dev)
        f = torch.empty(B, dtype=torch.float64, device=dev)
        g = torch.empty((B, self.n_g), dtype=torch.float64, device=dev) if want_g else None
        lam_x = torch.empty((B, self.n_w), dtype=torch.float64, device=dev) if want_lam else None
        lam_g = torch.empty((B, self.n_g), dtype=torch.float64, device=dev) if want_lam else None
        status = torch.empty(B, dtype=torch.int32, device=dev)
        iters = torch.empty(B, dtype=torch.int32, device=dev)
        ptr = lambda t: None if t is None else t.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        if order is not None:      # scheduling hint only: longest-first fetch order of the persistent kernel
            order = order.to(torch.int32).contiguous()
            if order.numel() != B:
                raise ValueError("solver: order must be a permutation of range(B)")
            _ffi.check(L.nmpc_set_order(self._h, order.data_ptr()), "nmpc_set_order")
        self._solves += 1
        _ffi.check(L.nmpc_solve(self._h, B, ptr(p), ptr(x0), ptr(lbx), ptr(ubx), ptr(lbg), ptr(ubg), ptr(obs), flags | (_ffi.NMPC_KEEP_BARRIER if jac else 0),
                                ptr(x), ptr(f), ptr(g), ptr(lam_x), ptr(lam_g), ptr(status), ptr(iters), stream),
                   "nmpc_solve")
        def lam_p_dev():      # CasADi's result dict also carries lam_p (nobody in the reference reads it): on first access
            lp = torch.empty((B, self.n_p), dtype=torch.float64, device=dev)
            with torch.cuda.device(dev):
                _ffi.check(L.nmpc_lam_p(self._h, B, ptr(x), ptr(p), ptr(obs), flags, ptr(lam_g), ptr(lp),
                                        torch.cuda.current_stream(dev).cuda_stream), "nmpc_lam_p")
            return lp[0] if single else lp
        self._keep = (p, x0, obs, order)   # keep inputs alive until the stream has consumed them
        self._stats = dict(return_status=status, iter_count=iters)      # success is derived lazily in stats()
        out = dict(x=x, f=f, g=g, lam_x=lam_x, lam_g=lam_g)
        if single:
            out = {k: (v[0] if v is not None else None) for k, v in out.items()}
        lazy = self._jac_keys(B, single, False, x, p, lam_g, obs, flags, status, *jac) if jac is not None else None
        return _Sol(out, lam_p_dev if want_lam else None, lazy)

    def _jac_keys(self, B, single, host, x, p, lam_g, obs, flags, status, weights, target_traj):
        """The lazy result keys of the solve just launched, with the solve's own weights / target trajectory / obstacles: jac_x_p
        (and jac_x_w for model 0) from one nmpc_sensitivity launch on first access of either, and with obstacle rows jac_x_obst
        from its own nmpc_sensitivity_obstacles launch.  NaN rows where the solve did not converge or no sensitivity exists
        (sens_status 1).  host: numpy inputs, numpy results."""
        L = _ffi.lib()
        solve_no = self._solves

        def family(fn, shapes):
            """shapes: key -> shape of each output pointer of `fn`, in order (None: pass NULL, no key)."""
            memo = {}

            def compute():
                if not memo:
                    if self._solves != solve_no:
                        raise RuntimeError(f"solver: {' / '.join(k for k, s in shapes.items() if s)} must be read before the next "
                                           "solve on this solver (the sensitivity needs that solve's barrier data, which the next "
                                           "solve replaces)")
                    dev = torch.device(f"cuda:{self.device}")
                    up = lambda a: a if _is_cuda_tensor(a) else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
                    xd, pd, ld, od, sd = up(x), up(p), up(lam_g), up(obs), up(status)
                    outs = {k: None if s is None else torch.empty(s, dtype=torch.float64, device=dev) for k, s in shapes.items()}
                    ss = torch.empty(B, dtype=torch.int32, device=dev)
                    ptr = lambda t: None if t is None else t.data_ptr()
                    with torch.cuda.device(dev), self._settings(B, weights, target_traj):
                        _ffi.check(getattr(L, fn)(self._h, B, ptr(xd), ptr(pd), ptr(ld), ptr(od) if od.numel() else None, flags,
                                                  *(ptr(t) for t in outs.values()), ptr(ss), torch.cuda.current_stream(dev).cuda_stream),
                                   fn)
                    bad = (sd != 0) | (ss != 0)
                    for k, t in outs.items():
                        if t is None:
                            continue
                        t[bad] = float("nan")
                        if host:
                            t = t.cpu().numpy()
                        memo[k] = t[0] if single else t
                return memo
            return {k: (lambda k=k: compute()[k]) for k, s in shapes.items() if s}

        keys = family("nmpc_sensitivity", {"jac_x_p": (B, self.n_w, self.n_p), "jac_x_w": None if self.model else (B, self.n_w, 2)})
        if self.n_obs:
            keys.update(family("nmpc_sensitivity_obstacles", {"jac_x_obst": (B, self.n_w, self.n_obs, 3)}))
        return keys

    def stats(self) -> Dict[str, Any]:
        """Per-instance outcome of the last call (CasADi: solver.stats()); after a blocking=False call, valid once
        wait() has returned."""
        d = dict(self._stats)
        if d and "success" not in d:
            d["success"] = d["return_status"] == 0
        return d

    def work_counters(self) -> Dict[str, int]:
        st = _ffi.NmpcStats()
        _ffi.check(_ffi.lib().nmpc_get_stats(self._h, C.byref(st)), "nmpc_get_stats")
        return {name: int(getattr(st, name)) for name, _ in _ffi.NmpcStats._fields_}

    # -- function-level evaluation (nlp_f / nlp_g / nlp_grad_f / nlp_hess_l of the reference's nlpsol) ----
    def evaluate(self, w, p, lam=None, v=None, sigma: float = 1.0, obstacles=None, weights=None, target_traj=None):
        L = _ffi.lib()
        dev = f"cuda:{self.device}"
        to = lambda a, n: torch.as_tensor(np.asarray(a, dtype=np.float64) if not _is_cuda_tensor(a) else a,
                                          dtype=torch.float64, device=dev).reshape(-1, n).contiguous()
        w, p = to(w, self.n_w), to(p, self.n_p)
        B = w.shape[0]
        lam_t = to(lam, self.n_g) if lam is not None else None
        v_t = to(v, self.n_w) if v is not None else None
        _, obs, flags = self._dev_inputs(B, obstacles)
        z = lambda *s: torch.empty(s, dtype=torch.float64, device=dev)
        f, g, grad = z(B), z(B, self.n_g), z(B, self.n_w)
        jtv = z(B, self.n_w) if lam_t is not None else None
        hv = z(B, self.n_w) if v_t is not None else None
        ptr = lambda t: None if t is None else t.data_ptr()
        stream = torch.cuda.current_stream(torch.device(dev)).cuda_stream
        with self._settings(B, weights, target_traj):
            _ffi.check(L.nmpc_eval(self._h, B, ptr(w), ptr(p), ptr(obs), flags, float(sigma), ptr(lam_t), ptr(v_t),
                                   ptr(f), ptr(g), ptr(grad), ptr(jtv), ptr(hv), stream), "nmpc_eval")
        torch.cuda.synchronize()
        return dict(f=f, g=g, grad=grad, jtv=jtv, hv=hv)

    # -- shift_timestep (NMPC_TT.py:13-30) on device --------------------------------------------
    def solve_and_step(self, p, u_warm, lbx, ubx, lbg, ubg, target_vw, fov_centre=None, err_accum=None, obstacles=None,
                       want_x: bool = False, weights=None, target_traj=None, predict_target: bool = False, obstacle_vel=None):
        """One closed-loop step of B instances in ONE kernel launch (nmpc_solve_and_step): solves from the warm start
        u_warm with parameters p, then shifts p / u_warm in place (torch CUDA float64 tensors).  Returns dict(x, f)
        with x None unless want_x; status / iterations through stats().
        predict_target: every solve uses the target's own Euler prediction over the horizon, made in the kernel from p's
        target block and this step's target input (NMPC_PREDICT_TARGET; the arithmetic of ClosedLoop.target_prediction()).
        obstacle_vel [B, n_obs, 2] (CUDA float64): obstacles, then a CUDA float64 [B, n_obs, 3] tensor, is moved in place by
        T * obstacle_vel after the solve (nmpc_set_obstacle_motion); this step's constraint rows use the positions before."""
        if predict_target and target_traj is not None:
            raise ValueError("solver: predict_target and target_traj exclude each other (the prediction replaces the trajectory)")
        status = torch.empty(p.shape[0], dtype=torch.int32, device=p.device)
        iters = torch.empty(p.shape[0], dtype=torch.int32, device=p.device)
        x, f = self._fused("nmpc_solve_and_step", (), (status, iters), p, u_warm, (lbx, ubx, lbg, ubg), target_vw, fov_centre,
                           err_accum, obstacles, want_x, predict_target, obstacle_vel, weights, target_traj)
        self._stats = dict(return_status=status, iter_count=iters)
        return dict(x=x, f=f, g=None, lam_x=None, lam_g=None)

    def run_closed_loop(self, steps: int, p, u_warm, lbx, ubx, lbg, ubg, target_vw, fov_centre=None, err_accum=None,
                        obstacles=None, want_x: bool = False, log: bool = True, predict_target: bool = False, obstacle_vel=None):
        """`steps` closed-loop steps of every instance in ONE launch, without a batch-wide barrier between the steps
        (nmpc_run_closed_loop; the scripts' `while mpc_iter < sim_time / T` loop, NMPC_TT.py:346-402).  p / u_warm are advanced in
        place.  Returns dict(x, f of the last step, status_log / iters_log [steps, B] when log, converged [B] = number of
        converged solves per instance); stats() reports the last step.  Bit-identical to `steps` solve_and_step calls, also
        with predict_target / obstacle_vel (as in solve_and_step: the prediction is made every step, the obstacles move every step)."""
        B = p.shape[0]
        slog = torch.empty((steps, B), dtype=torch.int32, device=p.device) if log else None
        ilog = torch.empty((steps, B), dtype=torch.int32, device=p.device) if log else None
        conv = torch.zeros(B, dtype=torch.int32, device=p.device)
        x, f = self._fused("nmpc_run_closed_loop", (int(steps),), (slog, ilog, conv), p, u_warm, (lbx, ubx, lbg, ubg), target_vw,
                           fov_centre, err_accum, obstacles, want_x, predict_target, obstacle_vel)
        self._stats = dict(return_status=slog[-1], iter_count=ilog[-1]) if log else {}
        return dict(x=x, f=f, status_log=slog, iters_log=ilog, converged=conv)

    def _fused(self, entry, lead, logs, p, u_warm, bounds, target_vw, fov_centre, err_accum, obstacles, want_x, predict_target,
               obstacle_vel, weights=None, target_traj=None):
        """One call of the fused closed-loop entry point `entry`: `lead` are its arguments between B and p, `logs` its outputs
        after err_accum.  Returns (x, f)."""
        B = p.shape[0]
        bounds, obs, flags = self._dev_inputs(B, obstacles, bounds)
        if predict_target:
            flags |= _ffi.NMPC_PREDICT_TARGET
        if target_vw is None and self._sched is None:
            raise ValueError("solver: target_vw is None and no schedule is set (set_schedule)")
        x = torch.empty((B, self.n_w), dtype=torch.float64, device=p.device) if want_x else None
        f = torch.empty(B, dtype=torch.float64, device=p.device)
        ptr = lambda t: None if t is None else t.data_ptr()
        self._solves += 1
        with self._settings(B, weights, target_traj, obstacles, obstacle_vel):
            _ffi.check(getattr(_ffi.lib(), entry)(self._h, B, *lead, ptr(p), ptr(u_warm), *map(ptr, bounds), ptr(obs), flags,
                                                  ptr(target_vw), ptr(x), ptr(f), ptr(fov_centre), ptr(err_accum), *map(ptr, logs),
                                                  torch.cuda.current_stream(p.device).cuda_stream), entry)
        self._keep = (obs,)
        return x, f

    def set_warm_start(self, lam_x0, lam_g0):
        """nmpc_set_warm_start: CUDA float64 tensors lam_x0 [B, n_w], lam_g0 [B, n_g] read by the following solves (and
        overwritten with the shifted multipliers by solve_and_step); None, None restores IPOPT's cold multiplier start.
        NON-REFERENCE mode; the pushes / mu_init come from the solver's 'ipopt' options."""
        L = _ffi.lib()
        if lam_x0 is None:
            self._warm = None
            _ffi.check(L.nmpc_set_warm_start(self._h, None, None, None), "nmpc_set_warm_start")
            return
        if not (_is_cuda_tensor(lam_x0) and _is_cuda_tensor(lam_g0)) or lam_x0.dtype != torch.float64 or lam_g0.dtype != torch.float64:
            raise ValueError("solver: lam_x0 / lam_g0 must be CUDA float64 tensors")
        lam_x0, lam_g0 = lam_x0.contiguous(), lam_g0.contiguous()
        if lam_x0.numel() % self.n_w or lam_g0.numel() % self.n_g or lam_x0.numel() // self.n_w != lam_g0.numel() // self.n_g:
            raise ValueError("solver: lam_x0 must be [B, n_w] and lam_g0 [B, n_g]")
        self._warm = (lam_x0, lam_g0)        # owned here: the handle keeps raw pointers
        o = _ffi.NmpcWarmOpts(*self._d["warm_opts"])
        _ffi.check(L.nmpc_set_warm_start(self._h, lam_x0.data_ptr(), lam_g0.data_ptr(), C.byref(o)), "nmpc_set_warm_start")

    def set_schedule(self, table, row_of_instance=None, phase=None, mpc_iter: int = 0):
        """Device-side target schedule (nmpc_set_schedule): table [n_rows, len, 2] of (v, omega) per closed-loop step;
        instance b follows row row_of_instance[b] starting at step phase[b].  solve_and_step(target_vw=None) then looks
        the pair up in the kernel's epilogue and advances the step counter.  table=None removes the schedule."""
        L = _ffi.lib()
        if table is None:
            self._sched = None
            _ffi.check(L.nmpc_set_schedule(self._h, None, 0, 0, None, None, 0), "nmpc_set_schedule")
            return
        dev = f"cuda:{self.device}"
        t = torch.as_tensor(np.asarray(table, dtype=np.float64) if not torch.is_tensor(table) else table, dtype=torch.float64, device=dev).contiguous()
        if t.dim() != 3 or t.shape[2] != 2:
            raise ValueError("solver: schedule table must be [n_rows, len, 2]")
        i32 = lambda a: None if a is None else torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a, device=dev).to(torch.int32).contiguous()
        rows, ph = i32(row_of_instance), i32(phase)
        if rows is not None and (int(rows.min()) < 0 or int(rows.max()) >= t.shape[0]):
            raise ValueError("solver: schedule row index out of range")
        if ph is not None and int(ph.min()) < 0:
            raise ValueError("solver: schedule phases must be >= 0")
        self._sched = (t, rows, ph)          # owned here: the handle keeps raw pointers
        ptr = lambda a: None if a is None else a.data_ptr()
        _ffi.check(L.nmpc_set_schedule(self._h, t.data_ptr(), int(t.shape[0]), int(t.shape[1]), ptr(rows), ptr(ph), int(mpc_iter)),
                   "nmpc_set_schedule")

    def step(self, x_sol, p, u_warm, target_vw, fov_centre=None, err_accum=None):
        """In-place closed-loop shift of B instances (torch CUDA float64 tensors): p [B,11], u_warm [B,6N];
        err_accum [B] += ||new FOV centre - this step's target|| (NMPC_TT.py:435)."""
        L = _ffi.lib()
        B = p.shape[0]
        stream = torch.cuda.current_stream(p.device).cuda_stream
        _ffi.check(L.nmpc_step(self._h, B, x_sol.data_ptr(), p.data_ptr(), u_warm.data_ptr(),
                               target_vw.data_ptr(), None if fov_centre is None else fov_centre.data_ptr(),
                               None if err_accum is None else err_accum.data_ptr(), stream),
                   "nmpc_step")


if torch is not None:
    class SolveFunction(torch.autograd.Function):
        """x* = solver(p=p, weights=weights, **kw)['x'] as a differentiable torch operation: SolveFunction.apply(solver, p, weights, kw)
        with p [B, n_p] and weights [B, 2] (or None: the solver's own) CUDA float64 tensors and kw the other keywords of the call.
        backward returns grad_p = jac_x_p^T grad_x and grad_weights = jac_x_w^T grad_x (want_jac; computed in the forward pass when
        a gradient is needed).  Instances that did not converge, or have no sensitivity, have NaN rows and so NaN gradients.

        SolveFunction.apply(solver, p, weights, kw, obstacles) also differentiates with respect to the obstacle table, a CUDA
        float64 tensor of (cx, cy, r_uav + r_obs) rows (then not in kw): grad_obstacles = jac_x_obst^T grad_x.
          [B, n_obs, 3], one table per instance: per instance, NaN rows for instances without a sensitivity, as for p.
          [n_obs, 3], shared by the batch: the sum over the instances of their contributions, where an instance whose grad_x row is
            exactly zero contributes exactly zero, even with NaN columns -- so a non-converged instance left out of the loss does
            not make the shared gradient NaN.  One that enters the loss with NaN columns still does."""

        @staticmethod
        def forward(ctx, solver, p, weights, kw, obstacles=None):
            if obstacles is not None:
                if "obstacles" in kw:
                    raise ValueError("SolveFunction: obstacles given both as an argument and in kw")
                if not (_is_cuda_tensor(obstacles) and obstacles.dtype == torch.float64):
                    raise ValueError("SolveFunction: obstacles must be a CUDA float64 tensor, [n_obs, 3] or [B, n_obs, 3]")
                kw = dict(kw, obstacles=obstacles)
            need_po = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
            need_o = len(ctx.needs_input_grad) > 4 and ctx.needs_input_grad[4]
            sol = solver(p=p, weights=weights, want_jac=need_po or need_o, **kw)
            ctx.jac = (sol["jac_x_p"], sol.get("jac_x_w") if weights is not None else None) if need_po else (None, None)
            ctx.jac_o = sol["jac_x_obst"] if need_o else None
            # the solver's shape rule: 3 n_obs entries are one table shared by the batch
            ctx.shared = need_o and solver._obs_flag(obstacles.numel(), sol["x"].numel() // solver.n_w) == 0
            ctx.obs_shape = None if obstacles is None else obstacles.shape
            return sol["x"]

        @staticmethod
        def backward(ctx, grad_x):
            jp, jw = ctx.jac
            gp = torch.einsum("...wp,...w->...p", jp, grad_x) if ctx.needs_input_grad[1] else None
            gw = torch.einsum("...wk,...w->...k", jw, grad_x) if (ctx.needs_input_grad[2] and jw is not None) else None
            go = None
            if ctx.jac_o is not None:
                if ctx.shared:
                    jo = ctx.jac_o.reshape(-1, *ctx.jac_o.shape[-3:])
                    gx = grad_x.reshape(jo.shape[0], -1)
                    used = (gx != 0).any(dim=1)      # instances outside the loss contribute exactly zero, NaN columns or not
                    go = torch.einsum("bwoc,bw->oc", jo[used], gx[used])
                else:
                    go = torch.einsum("...woc,...w->...oc", ctx.jac_o, grad_x)
                go = go.reshape(ctx.obs_shape)
            return (None, gp, gw, None, go)[:len(ctx.needs_input_grad)]


def nlpsol(name: str, plugin: str, problem, opts: Optional[dict] = None, device: int = 0, max_batch: int = 1,
           fill: int = 1) -> Solver:
    """Mirror of ca.nlpsol(name, 'ipopt', nlp_prob, opts) (NMPC_TT.py:267).

    plugin: 'ipm' (or 'ipopt' for drop-in spelling) -- the in-kernel interior-point method.
    problem: a scenarios.Scenario or a dict(T=, N=, obstacles=[(cx,cy,r_obs)...], uav_r=5, w1=1, w2=2).
    opts: {'ipopt': {'max_iter': 100, ...}} as in the reference; unknown keys are ignored like print_level.
    fill: scheduling hint for solvers that run next to others (PipelinedClosedLoop): instances per resident warp."""
    if plugin not in ("ipm", "ipopt"):
        raise ValueError(f"nlpsol: unknown plugin '{plugin}' (only the in-kernel 'ipm' exists)")
    return Solver(name, problem, opts, device=device, max_batch=max_batch, fill=fill)
