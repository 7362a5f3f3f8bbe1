"""Time of nmpc_sensitivity next to one solve (CUDA events): python tools/sens_probe.py [B] [reps]
Solves B seeded instances of the t_trajectory scenario (N = 15, 3 obstacle rows) with NMPC_KEEP_BARRIER, then times the solve
and the sensitivity launch (dx/dp and dx/d(w1, w2) of every instance) over `reps` repetitions each.  Prints one JSON line."""
import json
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import b200nmpc  # noqa: E402
from mpc_implementation_b200 import _ffi  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
sc = b200nmpc.SCENARIOS["t_trajectory"]
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
st = torch.empty(B, dtype=torch.int32, device=dev)
stream = torch.cuda.current_stream().cuda_stream


def sens():
    _ffi.check(L.nmpc_sensitivity(s._h, B, sol["x"].data_ptr(), p.data_ptr(), sol["lam_g"].data_ptr(), obs.data_ptr(), 0,
                                  jp.data_ptr(), jw.data_ptr(), st.data_ptr(), stream), "nmpc_sensitivity")


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


t_solve = timed(solve)
sol = solve()
t_sens = timed(sens)
conv = int((s.stats()["return_status"] == 0).sum())
print(json.dumps(dict(device=torch.cuda.get_device_name(0), B=B, reps=reps, solve_ms=t_solve, sensitivity_ms=t_sens,
                      sensitivity_us_per_instance=1e3 * t_sens / B, converged=conv, sens_status_nonzero=int((st != 0).sum()))))
