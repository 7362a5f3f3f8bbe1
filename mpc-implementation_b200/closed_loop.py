"""Batched shift-and-apply-first-input closed loop (Python/NMPC_TT.py:346-402) with all state on the GPU.

Per step and per instance the reference does
    p  = vertcat(x0, xs);  x0_nlp = reshape(u0, 6N, 1)                     :350-356
    sol = solver(x0=..., lbx, ubx, lbg, ubg, p)                             :358-365
    u   = reshape(sol['x'], 6, N)                                           :367
    t0, x0, u0, xs = shift_timestep(T, t0, x0, u, f_u, xs)                  :382  (schedule keyed on mpc_iter)
    x_e_1, y_e_1 = FOV centre of the new x0                                 :399-402
Here B such loops advance together: one nmpc_solve launch + one nmpc_step launch per batch step, no host
round trip.  The final metric of the scripts, sum_i ||FOVcentre_{i+1} - target_i|| (:433-440), is
accumulated per instance.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch

from .nlpsol import Solver
from .scenarios import NP, Scenario


class ClosedLoop:
    def __init__(self, solver: Solver, scenario: Scenario, p0, target_vw=None, device: Optional[str] = None,
                 phase=None, predict_target: bool = False, obstacles=None, obstacle_vel=None, schedules=None, schedule_of=None,
                 warm_duals: bool = False):
        """warm_duals (NON-REFERENCE mode, off by default; needs a solver built with ipopt.warm_start_init_point = 'yes'): the
        multipliers of every solve, shifted by one stage in the fused epilogue, start the next one (nmpc_set_warm_start).
        p0 [B,11] initial [state; target]; target_vw [B,2] constant per-instance target (v, omega) or None to
        follow scenario.schedule(mpc_iter + phase[b]).  schedules: optional list of schedule functions (mpc_iter ->
        (v, omega)) with schedule_of[b] the one instance b follows (BASELINE config 3 mixes the T and the Plus
        trajectory in one batch); default: the scenario's own.  The schedule lives on the device as a table
        (nmpc_set_schedule), so that a step costs no host work whatever the batch size.  predict_target: hand the solver the target's own Euler
        prediction over the horizon (same model as the target step of shift_timestep, NMPC_TT.py:24-27) instead of
        the frozen target the reference uses.  obstacles [B, n_obs, 3] = (cx, cy, r_uav + r_obs) per instance and
        obstacle_vel [B, n_obs, 2]: obstacle fields as data, moved by T * velocity after every step (the moving
        obstacles of MATLAB/Dynamic Obstacles/Dynamic Obstacle avoidance.m:128-133, whose positions are parameters; a shared
        [n_obs, 3] field with [n_obs, 2] velocities is given every instance as its own copy).  The fused step and run_free
        make the prediction and move the obstacles inside the kernel (NMPC_PREDICT_TARGET, nmpc_set_obstacle_motion), bit-identical
        to target_prediction() and _move_obstacles(), which the unfused step (want_g / want_lam) still uses."""
        self.predict_target = predict_target
        dev0 = device or f"cuda:{solver.device}"
        t64 = lambda a: None if a is None else torch.as_tensor(np.asarray(a, dtype=np.float64) if not torch.is_tensor(a) else a,
                                                               dtype=torch.float64, device=dev0).contiguous().clone()
        self.obstacles, self.obstacle_vel = t64(obstacles), t64(obstacle_vel)
        self.solver, self.sc = solver, scenario
        dev = device or f"cuda:{solver.device}"
        self.p = torch.as_tensor(np.asarray(p0, dtype=np.float64), device=dev).reshape(-1, scenario.n_p).contiguous().clone()
        self.B = self.p.shape[0]
        if self.obstacles is not None and self.obstacle_vel is not None:      # per-instance fields: the kernel moves them in place
            n_obs = self.obstacles.shape[-2]
            self.obstacles = self.obstacles.reshape(-1, n_obs, 3).expand(self.B, n_obs, 3).contiguous()
            self.obstacle_vel = self.obstacle_vel.reshape(-1, n_obs, 2).expand(self.B, n_obs, 2).contiguous()
        self.u_warm = torch.zeros((self.B, scenario.n_w), dtype=torch.float64, device=dev)     # u0 = 0  (:329)
        lbx, ubx, lbg, ubg = scenario.bounds()
        to = lambda a: torch.as_tensor(a, dtype=torch.float64, device=dev)
        self.lbx, self.ubx, self.lbg, self.ubg = to(lbx), to(ubx), to(lbg), to(ubg)
        self.fov = torch.zeros((self.B, 2), dtype=torch.float64, device=dev)
        self.err_sum = torch.zeros(self.B, dtype=torch.float64, device=dev)
        self.mpc_iter = 0
        self.phase = None if phase is None else np.asarray(phase, dtype=np.int64)
        self.sched_fns = list(schedules) if schedules is not None else [scenario.schedule]
        self.sched_of = None if schedule_of is None else np.asarray(schedule_of, dtype=np.int64)
        if target_vw is not None:
            self.vw = to(np.asarray(target_vw, dtype=np.float64)).reshape(self.B, 2).contiguous()
            self._const_vw = True
        else:
            self.vw = torch.zeros((self.B, 2), dtype=torch.float64, device=dev)
            self._const_vw = False
            # breakpoint schedules as a dense table [n_sched][len][2]: every script's schedule is constant after its
            # last breakpoint (< scenario.steps), so len = steps + max phase covers any run; later steps use the last entry
            L = int(scenario.steps + (int(self.phase.max()) if self.phase is not None else 0) + 1)
            self.sched_table = torch.as_tensor(np.array([[fn(i) for i in range(L)] for fn in self.sched_fns], dtype=np.float64),
                                               device=dev).contiguous()
            self._phase_dev = None if self.phase is None else torch.as_tensor(self.phase, device=dev)
            self._sched_dev = None if self.sched_of is None else torch.as_tensor(self.sched_of, device=dev)
            solver.set_schedule(self.sched_table, self._sched_dev, self._phase_dev, mpc_iter=0)
        self.last = None
        self.warm_duals = bool(warm_duals)
        if self.warm_duals:
            self.lam_x0 = torch.zeros((self.B, scenario.n_w), dtype=torch.float64, device=dev)
            self.lam_g0 = torch.zeros((self.B, scenario.n_g), dtype=torch.float64, device=dev)
            self.lam_x0[:, 0] = float("nan")             # no guess yet: the first solve is a cold start
            solver.set_warm_start(self.lam_x0, self.lam_g0)

    def _schedule_vw(self):
        """(v, omega) of this step into self.vw -- one gather on the device (only the unfused path and the target
        prediction read it; the fused step looks the schedule up inside the kernel)."""
        if self._const_vw:
            return
        L = self.sched_table.shape[1]
        at = torch.full((self.B,), self.mpc_iter, dtype=torch.int64, device=self.vw.device)
        if self._phase_dev is not None:
            at = at + self._phase_dev
        at = at.clamp(max=L - 1)
        rows = self._sched_dev if self._sched_dev is not None else torch.zeros_like(at)
        self.vw.copy_(self.sched_table[rows, at])

    def _moving_vel(self):
        return self.obstacle_vel if self.obstacles is not None else None

    def _move_obstacles(self):
        if self.obstacles is not None and self.obstacle_vel is not None:
            self.obstacles[:, :, :2] += self.sc.T * self.obstacle_vel

    def target_prediction(self):
        """[B, N, 2]: x_t, y_t of stages 0..N-1 under theta_{k+1} = theta_k + T w, (x, y)_{k+1} = (x, y)_k + T v (cos, sin)(theta_k)."""
        N, T = self.sc.N, self.sc.T
        k = torch.arange(N, dtype=torch.float64, device=self.p.device)
        nt = self.sc.n_p - 3                                                       # target block of p
        th = self.p[:, nt + 2:nt + 3] + T * self.vw[:, 1:2] * k[None, :]                        # theta at stage k
        step = T * self.vw[:, 0:1, None] * torch.stack([torch.cos(th), torch.sin(th)], dim=2)
        excl = torch.cat([torch.zeros_like(step[:, :1]), torch.cumsum(step[:, :-1], dim=1)], dim=1)   # exclusive prefix sum
        pos = self.p[:, None, nt:nt + 2] + excl
        return pos.contiguous()

    def next_order(self):
        """Explicit longest-first fetch order (previous iteration counts, descending) for `solver(order=)`.  The
        library does the same by itself for consecutive calls with equal B (include/nmpc_b200.h, "Scheduling"), so
        the loop below does not pass one; kept for callers that permute their instances between steps."""
        st = self.solver.stats()
        it = st.get("iter_count") if st else None
        if it is None or not torch.is_tensor(it) or it.numel() != self.B:
            return None
        return torch.argsort(it, descending=True)

    def step(self, want_g: bool = False, want_lam: bool = False, want_x: bool = True):
        """One closed-loop batch step; returns the solver output dict (device tensors).  Without g / multipliers
        the solve and the shift -- with the target prediction and the obstacle motion -- are one launch (nmpc_solve_and_step)
        and the step costs no host work."""
        if self.warm_duals and (want_g or want_lam):
            raise ValueError("ClosedLoop: warm_duals needs the fused step (want_g = want_lam = False)")
        if not (want_g or want_lam):
            sol = self.solver.solve_and_step(self.p, self.u_warm, self.lbx, self.ubx, self.lbg, self.ubg,
                                             self.vw if self._const_vw else None, self.fov,
                                             self.err_sum, obstacles=self.obstacles, want_x=want_x,
                                             predict_target=self.predict_target, obstacle_vel=self._moving_vel())
            self.mpc_iter += 1
            self.last = sol
            return sol
        self._schedule_vw()
        sol = self.solver(x0=self.u_warm, p=self.p, lbx=self.lbx, ubx=self.ubx, lbg=self.lbg, ubg=self.ubg, obstacles=self.obstacles,
                          want_g=want_g, want_lam=want_lam,
                          target_traj=self.target_prediction() if self.predict_target else None)
        # shift + error[i] = || FOVcentre_{i+1} - target_i ||   (NMPC_TT.py:435), one kernel
        self.solver.step(sol["x"], self.p, self.u_warm, self.vw, self.fov, self.err_sum)
        if not self._const_vw:      # keep the device-side step counter of the fused path in line with this loop's
            self.solver.set_schedule(self.sched_table, self._sched_dev, self._phase_dev, mpc_iter=self.mpc_iter + 1)
        self._move_obstacles()
        self.mpc_iter += 1
        self.last = sol
        return sol

    def run_free(self, steps: int, log: bool = True, want_x: bool = False):
        """`steps` closed-loop steps of every instance in one launch with no batch-wide barrier between the steps
        (Solver.run_closed_loop): the fast way through a Monte-Carlo study; per instance bit-identical to step() x steps, also with
        the target prediction and moving obstacles."""
        out = self.solver.run_closed_loop(steps, self.p, self.u_warm, self.lbx, self.ubx, self.lbg, self.ubg,
                                          self.vw if self._const_vw else None, self.fov, self.err_sum, obstacles=self.obstacles,
                                          want_x=want_x, log=log, predict_target=self.predict_target, obstacle_vel=self._moving_vel())
        self.mpc_iter += steps
        self.last = out
        return out

    def run(self, steps: int):
        conv = 0
        for _ in range(steps):
            self.step()
            conv += int(self.solver.stats()["success"].sum().item())
        return conv


class PipelinedClosedLoop:
    """The same batch of independent closed loops, advanced as `pipelines` sub-batches, each with its own solver
    handle and CUDA stream (include/nmpc_b200.h: one handle per (device, stream)).

    Why: a batch step ends when its slowest instance does (iteration counts 15...100), and while those stragglers
    run most SMs are idle -- 43 % of a 4096-instance step.  Sub-batches are independent, so sub-batch B's step k can
    fill the SMs that sub-batch A's stragglers of step k leave idle, and A's step k+1 follows A's step k on its own
    stream.  Per-instance results are identical to the single-batch loop; only the schedule changes (+39 % converged
    solves/s at 4096 instances per GPU, DESIGN.md section 2)."""

    def __init__(self, make_solver: Callable[[int], Solver], scenario: Scenario, p0, target_vw=None,
                 pipelines: Optional[int] = None, device: Optional[str] = None, phase=None, predict_target: bool = False,
                 obstacles=None, obstacle_vel=None, schedules=None, schedule_of=None):
        """make_solver(n) -> Solver for a sub-batch of n instances (give it `fill=2`: a sub-batch then leaves SMs to
        the others).  pipelines: number of sub-batches; None = about 32768 / B, at least 2, at most 8 (measured best: 8 at
        B = 4096, 2 at B = 16384 ... 131072 on a B200)."""
        p0 = np.asarray(p0, dtype=np.float64).reshape(-1, scenario.n_p)
        B = p0.shape[0]
        if pipelines is None:
            pipelines = max(2, min(8, 32768 // max(B, 1)))
        S = max(1, min(int(pipelines), B))
        self.index = np.array_split(np.arange(B), S)
        self.B, self.sc = B, scenario
        self.loops, self.streams = [], []
        for idx in self.index:
            sol = make_solver(len(idx))
            dev = device or f"cuda:{sol.device}"
            st = torch.cuda.Stream(device=dev)
            with torch.cuda.stream(st):
                sub = lambda a: None if a is None else (a[torch.as_tensor(idx, device=a.device)] if torch.is_tensor(a) else np.asarray(a)[idx])
                lp = ClosedLoop(sol, scenario, p0[idx], None if target_vw is None else np.asarray(target_vw)[idx], device=dev,
                                phase=None if phase is None else np.asarray(phase)[idx], predict_target=predict_target,
                                obstacles=sub(obstacles), obstacle_vel=sub(obstacle_vel), schedules=schedules,
                                schedule_of=None if schedule_of is None else np.asarray(schedule_of)[idx])
            self.loops.append(lp); self.streams.append(st)
        self.synchronize()

    def step(self, want_g: bool = False, want_lam: bool = False):
        """Enqueue one closed-loop step of every sub-batch (asynchronous); returns the list of solver outputs."""
        out = []
        for lp, st in zip(self.loops, self.streams):
            with torch.cuda.stream(st):
                out.append(lp.step(want_g=want_g, want_lam=want_lam))
        return out

    def synchronize(self):
        for st in self.streams:
            st.synchronize()

    def join(self, stream=None):
        """Make `stream` (default: the current stream) wait for everything enqueued so far."""
        cur = stream or torch.cuda.current_stream(self.loops[0].p.device)
        for st in self.streams:
            cur.wait_stream(st)

    def stats(self):
        """Solver stats of the last step of every sub-batch, concatenated in instance order (synchronises)."""
        self.synchronize()
        parts = [lp.solver.stats() for lp in self.loops]
        return {k: torch.cat([q[k] for q in parts]) for k in parts[0]}

    @property
    def p(self):
        self.synchronize()
        return torch.cat([lp.p for lp in self.loops])

    @property
    def u_warm(self):
        self.synchronize()
        return torch.cat([lp.u_warm for lp in self.loops])

    @property
    def err_sum(self):
        self.synchronize()
        return torch.cat([lp.err_sum for lp in self.loops])
