"""GPU (-m gpu): the paired backtracking trial pass (NMPC_B200_PAIR_TRIALS, N <= 15 layouts) evaluates the next trial
point on the idle half of the warp.  Results must be bit-identical with pairing on and off, the line search must see
the same trials, and the reused trials must show in the work counters."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

KNOB = "NMPC_B200_PAIR_TRIALS"


def _solver(pkg, sc, B, pair):
    """The knob is read when the handle is created."""
    old = os.environ.get(KNOB)
    os.environ[KNOB] = "1" if pair else "0"
    try:
        return pkg.nlpsol("solver", "ipm", sc, max_batch=B)
    finally:
        if old is None:
            del os.environ[KNOB]
        else:
            os.environ[KNOB] = old


def _run_loop(pkg, sc, p, vw, pair, steps):
    from mpc_implementation_b200.closed_loop import ClosedLoop
    cl = ClosedLoop(_solver(pkg, sc, len(p), pair), sc, p, target_vw=vw)
    outs, counters = [], {}
    for _ in range(steps):
        sol = cl.step()
        st = cl.solver.stats()
        outs.append((sol["f"].clone(), st["return_status"].clone(), st["iter_count"].clone()))
        for k, v in cl.solver.work_counters().items():
            counters[k] = counters.get(k, 0) + v
    torch.cuda.synchronize()
    return cl, outs, counters


def _check_counters(on, off):
    assert on["factorizations"] == off["factorizations"] and on["ls_trials"] == off["ls_trials"], (on, off)
    assert off["trial_passes"] == off["ls_trials"], off
    assert on["trial_passes"] < on["ls_trials"], on


@pytest.mark.parametrize("name,N,B,scheduled", [("nmpc_tt", None, 2000, False), ("10_obstacles", None, 2000, False),
                                                ("t_trajectory", None, 2000, True), ("nmpc_tt", 5, 2000, False)])
def test_paired_trials_are_bit_identical(pkg, name, N, B, scheduled):
    sc = pkg.SCENARIOS[name]
    if N:
        sc = sc.with_horizon(N)
    p, vw = pkg.random_instances(sc, B, seed=2024 + B)
    if scheduled:
        vw = None          # the scenario's target schedule, looked up on the device
    on, outs_on, wc_on = _run_loop(pkg, sc, p, vw, True, 8)
    off, outs_off, wc_off = _run_loop(pkg, sc, p, vw, False, 8)
    for a, b in zip(outs_on, outs_off):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    for k in ("p", "u_warm", "fov", "err_sum"):
        assert torch.equal(getattr(on, k), getattr(off, k)), k
    _check_counters(wc_on, wc_off)


def test_paired_trials_in_the_restoration_phase(pkg):
    """The infeasible-by-construction batch of test_gpu_parity.py::test_restoration_outcomes: the restoration problem's
    line search (ph_trial<RS = true>) is paired too."""
    sc = pkg.SCENARIOS["nmpc_tt"]
    lbx, ubx, lbg, ubg = sc.bounds()
    B = 32
    p, _ = pkg.random_instances(sc, B, seed=99)
    ob = sc.obstacle_table()
    p[:16, 0] = ob[1, 0] + 10.0; p[:16, 1] = ob[1, 1] - 5.0
    p[16:, 2] = 150.0 + 10.0 ** np.linspace(-5.5, -2, 16)
    x0 = np.tile(np.array([16.0, 0, 0, 0, 0, 0]), (B, sc.N))
    res = {}
    for pair in (True, False):
        s = _solver(pkg, sc, B, pair)
        sol = s(x0=x0, p=p, lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg)
        res[pair] = (sol, {k: np.asarray(v.cpu() if torch.is_tensor(v) else v) for k, v in s.stats().items()}, s.work_counters())
    (son, ston, wcon), (soff, stoff, wcoff) = res[True], res[False]
    assert wcon["resto_calls"] >= B // 2 and wcon["resto_iters"] == wcoff["resto_iters"] > 0
    for k in ("return_status", "iter_count"):
        assert np.array_equal(ston[k], stoff[k]), k
    for k in ("x", "f", "g", "lam_x", "lam_g"):
        a, b = son[k], soff[k]
        a = a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
        b = b.cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
        assert a.tobytes() == b.tobytes(), k
    _check_counters(wcon, wcoff)
