"""Time of nmpc_sensitivity next to one solve (CUDA events): python tools/sens_probe.py [B] [reps] [--obstacles]
Solves B seeded instances of the t_trajectory scenario (N = 15, 3 obstacle rows) with NMPC_KEEP_BARRIER, then times the solve
and the sensitivity launch (dx/dp and dx/d(w1, w2) of every instance) over `reps` repetitions each.  --obstacles: the
race_track_2 scenario (N = 15, 10 obstacle rows) instead, and also the launch of the obstacle columns
(nmpc_sensitivity_obstacles, dx/d(cx, cy, r) of every obstacle).  Prints one JSON line with the card and its power limit."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import b200nmpc  # noqa: E402
from mpc_implementation_b200 import _ffi  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
obstacles = "--obstacles" in sys.argv[1:]
B = int(args[0]) if len(args) > 0 else 4096
reps = int(args[1]) if len(args) > 1 else 20
sc = b200nmpc.SCENARIOS["race_track_2" if obstacles else "t_trajectory"]
dev = "cuda:0"
p = torch.as_tensor(b200nmpc.random_instances(sc, B, seed=1)[0], device=dev)
x0 = torch.zeros((B, sc.n_w), dtype=torch.float64, device=dev)
lbx, ubx, lbg, ubg = sc.bounds()
s = b200nmpc.nlpsol("s", "ipm", sc, {"ipopt": {"max_iter": 100}}, device=0, max_batch=B)
solve = lambda: s(x0=x0, p=p, lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg, want_jac=True)
sol = solve()
L = _ffi.lib()
obs = s._dev_const("obs", s.obstacles)
jp = torch.empty((B, sc.n_w, sc.n_p), dtype=torch.float64, device=dev)
jw = torch.empty((B, sc.n_w, 2), dtype=torch.float64, device=dev)
jo = torch.empty((B, sc.n_w, sc.n_obs, 3), dtype=torch.float64, device=dev)
st = torch.empty(B, dtype=torch.int32, device=dev)
st_o = torch.empty(B, dtype=torch.int32, device=dev)
stream = torch.cuda.current_stream().cuda_stream


def sens():
    _ffi.check(L.nmpc_sensitivity(s._h, B, sol["x"].data_ptr(), p.data_ptr(), sol["lam_g"].data_ptr(), obs.data_ptr(), 0,
                                  jp.data_ptr(), jw.data_ptr(), st.data_ptr(), stream), "nmpc_sensitivity")


def sens_obst():
    _ffi.check(L.nmpc_sensitivity_obstacles(s._h, B, sol["x"].data_ptr(), p.data_ptr(), sol["lam_g"].data_ptr(), obs.data_ptr(), 0,
                                            jo.data_ptr(), st_o.data_ptr(), stream), "nmpc_sensitivity_obstacles")


def timed(fn):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return q.strip().splitlines()[0] if q.strip() else torch.cuda.get_device_name(0)


t_solve = timed(solve)
sol = solve()
t_sens = timed(sens)
conv = int((s.stats()["return_status"] == 0).sum())
out = dict(device=card(), scenario=sc.name, N=sc.N, n_obs=sc.n_obs, B=B, reps=reps, solve_ms=t_solve, sensitivity_ms=t_sens,
           sensitivity_us_per_instance=1e3 * t_sens / B, converged=conv, sens_status_nonzero=int((st != 0).sum()))
if obstacles:
    t_obst = timed(sens_obst)
    out.update(obstacle_columns=3 * sc.n_obs, sensitivity_obstacles_ms=t_obst, sensitivity_obstacles_us_per_instance=1e3 * t_obst / B,
               sensitivity_obstacles_over_solve=t_obst / t_solve, sens_status_equal=bool(torch.equal(st, st_o)))
print(json.dumps(out))
