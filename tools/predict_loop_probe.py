"""Converged solves/s of the closed loops with a predicted target and with moving obstacles, three arms each, alternated:
  host     the per-step loop with the work on the host side: the target prediction built by torch every step and handed over
           as target_traj (nmpc_set_target_trajectory), or the obstacle field moved by a torch update after every step
  fused    ClosedLoop.step() with the prediction / the motion inside the kernel (NMPC_PREDICT_TARGET, nmpc_set_obstacle_motion)
  free     ClosedLoop.run_free(K): K steps of every instance in one launch
Loops: t_trajectory with the device schedule and random phases (B = 65 536); 10_obstacles with per-instance moving fields
(B = 32 768).
   python tools/predict_loop_probe.py [--steps K] [--reps R] [--json PATH]"""
import argparse, json, subprocess, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np, torch
import b200nmpc, bench
from mpc_implementation_b200.closed_loop import ClosedLoop

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10, help="closed-loop steps per timed window")
ap.add_argument("--reps", type=int, default=3, help="timed windows per arm (the arms alternate)")
ap.add_argument("--json", default=None)
args = ap.parse_args()
K = args.steps


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return q.strip().splitlines()[0] if q.strip() else torch.cuda.get_device_name(0)


def timed(fn):
    torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); conv = fn(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1), int(conv.item())


def per_step(cl, one_step):
    def run():
        c = torch.zeros((), dtype=torch.int64, device="cuda")
        for _ in range(K):
            one_step(); c += cl.solver.stats()["success"].sum()
        return c
    return run


def free(cl):
    return lambda: cl.run_free(K, log=False)["converged"].sum()


def predicted_target():
    sc = b200nmpc.SCENARIOS["t_trajectory"]; B = 65536
    p, _ = b200nmpc.random_instances(sc, B, seed=1000)
    kw = dict(phase=np.random.default_rng(7).integers(0, sc.steps, B))
    host = ClosedLoop(b200nmpc.nlpsol("h", "ipm", sc, max_batch=B), sc, p, **kw)

    def host_step():      # what the fused step did before the prediction moved into the kernel
        host._schedule_vw()
        host.solver.solve_and_step(host.p, host.u_warm, host.lbx, host.ubx, host.lbg, host.ubg, None, host.fov, host.err_sum,
                                   target_traj=host.target_prediction())
        host.mpc_iter += 1
    fused = ClosedLoop(b200nmpc.nlpsol("f", "ipm", sc, max_batch=B), sc, p, predict_target=True, **kw)
    fr = ClosedLoop(b200nmpc.nlpsol("r", "ipm", sc, max_batch=B), sc, p, predict_target=True, **kw)
    return f"t_trajectory B={B}, predicted target", B, dict(host=per_step(host, host_step), fused=per_step(fused, fused.step), free=free(fr))


def moving_obstacles():
    cfg = bench.CONFIGS[4]; B = 32768
    sc, p, vw, obs, _ = bench.make_workload(b200nmpc, cfg, B, seed=1000)
    vel = np.random.default_rng(11).uniform(-3.0, 3.0, (B, sc.n_obs, 2))
    host = ClosedLoop(b200nmpc.nlpsol("h", "ipm", sc, max_batch=B), sc, p, target_vw=vw, obstacles=obs)
    vel_t = torch.as_tensor(vel, device=host.obstacles.device)

    def host_step():      # the fused solve, then the torch update of the field
        host.step(); host.obstacles[:, :, :2] += sc.T * vel_t
    fused = ClosedLoop(b200nmpc.nlpsol("f", "ipm", sc, max_batch=B), sc, p, target_vw=vw, obstacles=obs, obstacle_vel=vel)
    fr = ClosedLoop(b200nmpc.nlpsol("r", "ipm", sc, max_batch=B), sc, p, target_vw=vw, obstacles=obs, obstacle_vel=vel)
    return f"10_obstacles B={B}, moving obstacles", B, dict(host=per_step(host, host_step), fused=per_step(fused, fused.step), free=free(fr))


result = dict(card=card(), steps_per_window=K, reps=args.reps, loops={})
print("card:", result["card"], flush=True)
for make in (predicted_target, moving_obstacles):
    name, B, arms = make()
    for fn in arms.values():      # warm-up window of every arm (module load, first solves from a cold start)
        timed(fn)
    rates = {a: [] for a in arms}
    for _ in range(args.reps):
        for a, fn in arms.items():
            ms, conv = timed(fn)
            rates[a].append(conv / ms * 1e3)
    result["loops"][name] = {a: dict(median=float(np.median(r)), runs=[float(x) for x in r]) for a, r in rates.items()}
    for a, r in rates.items():
        print(f"{name}: {a:6s} {np.median(r):12.0f} converged solves/s (median of {len(r)}; runs {', '.join(f'{x:.0f}' for x in r)})", flush=True)
    del arms
    torch.cuda.empty_cache()
if args.json:
    Path(args.json).parent.mkdir(parents=True, exist_ok=True)
    Path(args.json).write_text(json.dumps(result, indent=1))
