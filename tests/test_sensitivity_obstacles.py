"""Obstacle sensitivities dx*/d(cx, cy, r) of converged solves (nmpc_sensitivity_obstacles, csrc/nmpc_sens.cuh).

The references are those of test_sensitivity.py with the obstacle table as the parameter: M = grad2_{w o} L and J_o = dg/do by
autograd of oracle/nlp_ref.py with respect to the table entries.  Random instances leave the obstacle rows inactive, and then the
obstacle columns are near zero and prove little; so every check here first solves, then moves obstacle 0 beside the returned
path at one stage, its boundary a little inside the path, and solves again: that row ends active.
"""
import dataclasses

import numpy as np
import pytest
import torch

from oracle import nlp_ref
from test_sensitivity import FD_TOL, LAYOUTS, _scenario, _sigmas, _solve, active_sens, active_set, refine_solve

BIG = 1e-3          # a row with |lam_g| above this is active (active_set's threshold)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def dense_parts_obst(sc, w, p, lam_g, obst):
    """W [n_w, n_w], M [n_w, 3 n_obs], J [n_g, n_w], J_o [n_g, 3 n_obs] at (w, p) with multipliers lam_g; o = the obstacle table
    [n_obs][3] = (cx, cy, r_uav + r_obs) flattened, column 3 j + (0, 1, 2) = (cx_j, cy_j, r_j).  Model 0."""
    n_w = sc.n_w
    obst = np.asarray(obst, dtype=np.float64).reshape(-1, 3)
    n_o = obst.size
    spec0 = nlp_ref.RefSpec(T=sc.T, N=sc.N, obstacles=[tuple(o) for o in obst], uav_r=0.0, vfov=sc.vfov, hfov=sc.hfov,
                            w1=sc.w1, w2=sc.w2)
    pt = torch.tensor(np.asarray(p, dtype=np.float64))
    lam = torch.tensor(np.asarray(lam_g, dtype=np.float64))

    def g_fn(z):
        o = z[n_w:]
        spec = dataclasses.replace(spec0, obstacles=[(o[3 * j], o[3 * j + 1], o[3 * j + 2]) for j in range(n_o // 3)])
        return nlp_ref.constraints(spec, z[:n_w], pt)

    def lag(z):
        return nlp_ref.objective(spec0, z[:n_w], pt, None) + (lam * g_fn(z)).sum()
    z0 = torch.tensor(np.concatenate([w, obst.reshape(-1)]), dtype=torch.float64)
    H = torch.autograd.functional.hessian(lag, z0).numpy()
    Jz = torch.autograd.functional.jacobian(g_fn, z0).numpy()
    return H[:n_w, :n_w], H[:n_w, n_w:], Jz[:, :n_w], Jz[:, n_w:]


def path_xy(sc, w, p):
    """(x, y) of stages 0..N of the solution w."""
    X = nlp_ref.rollout(nlp_ref.RefSpec(T=sc.T, N=sc.N), torch.as_tensor(np.asarray(w, dtype=np.float64)),
                        torch.as_tensor(np.asarray(p, dtype=np.float64)))
    return np.array([[float(s[0]), float(s[1])] for s in X])


def active_tables(sc, x, p, delta=2.0):
    """Per-instance tables [B, n_obs, 3]: the spec's table with obstacle 0 moved beside the path of solution x[b] at stage k (one
    of three late stages, the terminal one included), its boundary `delta` inside the path, on the inner side of the turn there (the
    paths turn at the rate bound towards the target, so only a turn less sharp gets around an obstacle).  The re-solve has to go
    around it: the row ends active."""
    obst = np.repeat(sc.obstacle_table()[None], len(p), axis=0)
    N = sc.N
    ks = sorted({max(2, N - 5), max(2, N - 3), N})
    for b in range(len(p)):
        xy = path_xy(sc, x[b], p[b])
        k = ks[b % len(ks)]
        t = xy[min(k + 1, N)] - xy[k - 1]
        t = t / np.linalg.norm(t)
        r = obst[b, 0, 2]
        a, c = xy[k] - xy[k - 1], xy[min(k + 1, N)] - xy[k]
        side = 1.0 if a[0] * c[1] - a[1] * c[0] >= 0 else -1.0       # the inner side of the turn
        obst[b, 0, :2] = xy[k] + (r - delta) * side * np.array([-t[1], t[0]])
    return obst


def obstacle_rows(sc, lam_g):
    """Multipliers of the obstacle rows [B, N + 1, n_obs]."""
    return np.asarray(lam_g).reshape(len(lam_g), sc.N + 1, -1)[:, :, sc.n_box:]


def has_active_obstacle(sc, lam_g):
    """[B]: some obstacle row of a stage 1..N is active."""
    return (np.abs(obstacle_rows(sc, lam_g)[:, 1:]) > BIG).any(axis=(1, 2))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the limit reference against central differences of oracle re-solves with perturbed tables
# ---------------------------------------------------------------------------------------------------------------------
def test_active_set_reference_matches_oracle_finite_differences(oracle_mod, pkg):
    sc = pkg.SCENARIOS["t_trajectory"]
    lbx, ubx, lbg, ubg = sc.bounds()
    sp = oracle_mod.make_spec(sc.T, sc.N, sc.n_obs, sc.w1, sc.w2, sc.vfov, sc.hfov)
    p, _ = pkg.random_instances(sc, 48, seed=5)
    base = oracle_mod.solve(sp, sc.obstacle_table(), p, np.zeros((len(p), sc.n_w)), lbx, ubx, lbg, ubg, tol=1e-10)
    obst = active_tables(sc, base["x"], p)
    ref = oracle_mod.solve(sp, obst, p, base["x"], lbx, ubx, lbg, ubg, obs_per_instance=True, tol=1e-10)
    act_obs = has_active_obstacle(sc, ref["lam_g"])
    checked, worst, n_o = 0, 0.0, 3 * sc.n_obs
    for b in np.flatnonzero((ref["status"] == 0) & act_obs):
        act = active_set(ref["x"][b], ref["lam_x"][b], ref["g"][b], ref["lam_g"][b], lbx, ubx, lbg, ubg)
        if act is None or checked == 4:
            continue
        W, M, J, Jo = dense_parts_obst(sc, ref["x"][b], p[b], ref["lam_g"][b], obst[b])
        D, det, _, _ = active_sens(W, M, J, Jo, *act)
        assert np.abs(D[det]).max() > 1e-3          # the active obstacle moves the solution
        # the step rule and tolerance of the CPU test of dx*/dp: h = 1e-4 max(1, |o_j|)
        hs = [1e-4 * max(1.0, abs(obst[b].reshape(-1)[j])) for j in range(n_o)]
        oo = np.repeat(obst[b].reshape(1, -1), 2 * n_o, axis=0)
        for j, h in enumerate(hs):
            oo[2 * j, j] += h
            oo[2 * j + 1, j] -= h
        r = oracle_mod.solve(sp, oo, np.repeat(p[b:b + 1], 2 * n_o, axis=0), np.repeat(ref["x"][b:b + 1], 2 * n_o, axis=0),
                             lbx, ubx, lbg, ubg, obs_per_instance=True, tol=1e-10)
        assert np.all(r["status"] == 0)
        for j, h in enumerate(hs):
            fd = (r["x"][2 * j] - r["x"][2 * j + 1]) / (2 * h)
            e = np.abs(fd - D[:, j])[det].max() / max(np.abs(D[det, j]).max(), 1e-3)
            worst = max(worst, e)
            assert e <= 1e-3, (b, j, e)
        checked += 1
    print("obstacle columns, limit reference vs oracle central differences: %d instances, max rel err %.1e" % (checked, worst))
    assert checked >= 3, checked


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
OBS_LAYOUTS = [l for l in LAYOUTS if l[1] > 0]
DEV = "cuda:0"


def _warm_solve(s, sc, p, x0, obst, want_jac=True):
    """Solve from the start point x0 (the solution without the moved obstacle: from zero many instances end infeasible)."""
    lbx, ubx, lbg, ubg = sc.bounds()
    return s(x0=torch.as_tensor(x0, device=DEV), p=torch.as_tensor(p, device=DEV), lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg,
             obstacles=obst, want_jac=want_jac)


def _active_batch(pkg, sc, B, seed, tol=1e-8, shared=False):
    """(solver, p, obstacles, x0): per instance, obstacle 0 placed on each instance's path (active_tables); with shared=True, one
    table -- that of the first instance where it ends active -- for a batch of small perturbations of that instance (start and
    target within 1 m).  x0: the solutions without the moved obstacle, the start point of the solves."""
    p, _ = pkg.random_instances(sc, B, seed=seed)
    s, sol = _solve(pkg, sc, p, want_jac=False, tol=tol)
    x0 = sol["x"].cpu().numpy()
    obst = active_tables(sc, x0, p)
    if not shared:
        return s, p, obst, x0
    r = _warm_solve(s, sc, p, x0, obst, want_jac=False)
    good = np.flatnonzero((s.stats()["return_status"].cpu().numpy() == 0) & has_active_obstacle(sc, r["lam_g"].cpu().numpy()))
    assert len(good), "no instance with an active obstacle row"
    b = good[0]
    p = np.repeat(p[b:b + 1], B, axis=0)
    p[1:, [0, 1, 8, 9]] += np.random.default_rng(seed).uniform(-1.0, 1.0, (B - 1, 4))
    _, sol = _solve(pkg, sc, p, want_jac=False, solver=s)
    return s, p, obst[b], sol["x"].cpu().numpy()


def _barrier_check_obst(sc, x, p, lam_g, sx, sg, obst, jac):
    """GPU obstacle columns against the dense barrier solve of the same data, self-calibrated as test_sensitivity._barrier_check."""
    W, M, J, Jo = dense_parts_obst(sc, x, p, lam_g, obst)
    K = W + np.diag(sx) + J.T @ (sg[:, None] * J)
    X64, Xr = refine_solve(K, M + J.T @ (sg[:, None] * Jo))
    scale = np.maximum(np.abs(Xr).max(axis=0), 1e-300)
    eg = (np.abs(jac - Xr) / scale).max(axis=0)
    ed = (np.abs(X64 - Xr) / scale).max()
    return eg, ed, max(32 * ed, 1e-11)


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("N,n_obs,model", OBS_LAYOUTS)
def test_kernel_matches_dense_barrier_solve(pkg, N, n_obs, model, shared):
    sc = _scenario(pkg, N, n_obs, model)
    B = 48
    s, p, obst, x0 = _active_batch(pkg, sc, B, seed=11, shared=shared)
    sol = _warm_solve(s, sc, p, x0, obst)
    st = s.stats()["return_status"].cpu().numpy()
    jo = sol["jac_x_obst"].cpu().numpy()
    assert jo.shape == (B, sc.n_w, sc.n_obs, 3)
    sx, sg = _sigmas(s, B)
    x, lg = sol["x"].cpu().numpy(), sol["lam_g"].cpu().numpy()
    assert np.all(np.isnan(jo[st != 0]))
    picked = np.flatnonzero((st == 0) & has_active_obstacle(sc, lg))
    assert len(picked) >= 3, (st, has_active_obstacle(sc, lg))
    for b in picked[:3]:
        jac = jo[b].reshape(sc.n_w, -1)
        assert np.abs(jac).max() > 1e-3
        eg, ed, bound = _barrier_check_obst(sc, x[b], p[b], lg[b], sx[b], sg[b], obst if shared else obst[b], jac)
        print(f"({N},{n_obs}) {'shared' if shared else 'per-instance'} b={b}: gpu rel err {eg.max():.2e}, float64 dense rel err {ed:.2e}")
        assert np.all(eg <= bound), (b, eg, bound)


@pytest.mark.gpu
def test_finite_differences_of_re_solves(pkg):
    """Central differences of GPU re-solves with perturbed tables, all 2 * 3 n_obs of one instance in one per-instance batch, on
    strictly complementary instances with an active obstacle row; the components the limit system determines."""
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 48
    lbx, ubx, lbg, ubg = sc.bounds()
    s, p, obst, x0 = _active_batch(pkg, sc, B, seed=5, tol=1e-10)     # 1e-10: the re-solves end closer to their solutions
    sol = _warm_solve(s, sc, p, x0, obst)
    st = s.stats()["return_status"].cpu().numpy()
    jo = sol["jac_x_obst"].cpu().numpy().reshape(B, sc.n_w, -1)
    x, lx, g, lg = (sol[k].cpu().numpy() for k in ("x", "lam_x", "g", "lam_g"))
    act_obs = has_active_obstacle(sc, lg)
    picked = [b for b in np.flatnonzero((st == 0) & act_obs) if active_set(x[b], lx[b], g[b], lg[b], lbx, ubx, lbg, ubg) is not None]
    assert len(picked) >= 3, (len(picked), st, act_obs)
    n_o = 3 * sc.n_obs
    s2 = pkg.nlpsol("fd", "ipm", sc, {"ipopt": {"max_iter": 100, "tol": 1e-10}}, device=0, max_batch=2 * n_o)
    fd_err = []
    for b in picked[:4]:
        assert np.abs(jo[b]).max() > 1e-3
        W, M, J, Jo = dense_parts_obst(sc, x[b], p[b], lg[b], obst[b])
        _, det, _, _ = active_sens(W, M, J, Jo, *active_set(x[b], lx[b], g[b], lg[b], lbx, ubx, lbg, ubg))
        # the step rule of test_sensitivity: h = 1e-4 max(1, |o_j|)
        hs = [1e-4 * max(1.0, abs(obst[b].reshape(-1)[j])) for j in range(n_o)]
        oo = np.repeat(obst[b].reshape(1, -1), 2 * n_o, axis=0)
        for j, h in enumerate(hs):
            oo[2 * j, j] += h
            oo[2 * j + 1, j] -= h
        r = _warm_solve(s2, sc, np.repeat(p[b:b + 1], 2 * n_o, axis=0), np.repeat(x[b:b + 1], 2 * n_o, axis=0),
                        oo.reshape(2 * n_o, sc.n_obs, 3), want_jac=False)
        assert np.all(s2.stats()["return_status"].cpu().numpy() == 0)
        xr = r["x"].cpu().numpy()
        for j, h in enumerate(hs):
            fd = (xr[2 * j] - xr[2 * j + 1]) / (2 * h)
            fd_err.append(np.abs(fd - jo[b][:, j])[det].max() / max(np.abs(jo[b][det, j]).max(), 1e-3))
    # measured on a B200: 5.7e-4 of a column (the CPU test's limit reference against oracle re-solves: 5.7e-4 as well, the h^2
    # term of the positions |c| ~ 150); the tolerance is test_sensitivity's for the same step
    print("obstacle columns vs central differences of re-solves: %d instances, max rel err %.2e" % (min(len(picked), 4), max(fd_err)))
    assert max(fd_err) <= FD_TOL, fd_err


def _same_bits(a, b):
    """Bit-for-bit equality, NaN rows included (rows of instances that did not converge)."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int64), b.contiguous().view(torch.int64))


@pytest.mark.gpu
def test_existing_columns_and_solve_unchanged(pkg):
    """Reading jac_x_obst changes neither jac_x_p / jac_x_w of the same solve nor the solve itself, bit for bit."""
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 16
    s, p, obst, x0 = _active_batch(pkg, sc, B, seed=13)
    a = _warm_solve(s, sc, p, x0, obst, want_jac=False)
    sa = {k: v.clone() for k, v in s.stats().items()}
    b1 = _warm_solve(s, sc, p, x0, obst)
    for k in ("x", "f", "g", "lam_x", "lam_g"):
        assert _same_bits(a[k], b1[k]), k
    for k in ("return_status", "iter_count"):
        assert torch.equal(sa[k], s.stats()[k]), k
    assert int((sa["return_status"] == 0).sum()) >= 3
    jp1, jw1 = b1["jac_x_p"].clone(), b1["jac_x_w"].clone()
    jo1 = b1["jac_x_obst"]
    assert _same_bits(b1["jac_x_p"], jp1) and _same_bits(b1["jac_x_w"], jw1)
    b2 = _warm_solve(s, sc, p, x0, obst)           # the obstacle columns first, then the others
    jo2 = b2["jac_x_obst"]
    assert _same_bits(b2["jac_x_p"], jp1) and _same_bits(b2["jac_x_w"], jw1) and _same_bits(jo1, jo2)


@pytest.mark.gpu
def test_autograd_backward(pkg):
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 8
    lbx, ubx, lbg, ubg = sc.bounds()
    # per instance: grad_obstacles = jac_x_obst^T grad_x, bit for bit on converged rows
    s, p0, obst0, x0 = _active_batch(pkg, sc, B, seed=9)
    kw = dict(x0=torch.as_tensor(x0, device=DEV), lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg)
    p = torch.as_tensor(p0, device=DEV)
    obst = torch.as_tensor(obst0, device=DEV).requires_grad_(True)
    x = pkg.SolveFunction.apply(s, p, None, kw, obst)
    ok = s.stats()["return_status"] == 0
    assert int(ok.sum()) >= 3
    v = torch.randn_like(x)
    (x * v)[ok].sum().backward()
    sol = s(p=p, obstacles=obst.detach(), want_jac=True, **kw)
    ref = torch.einsum("...woc,...w->...oc", sol["jac_x_obst"], v)
    assert torch.equal(obst.grad[ok], ref[ok])
    assert torch.equal(x.detach(), sol["x"])
    with pytest.raises(ValueError, match="both"):
        pkg.SolveFunction.apply(s, p, None, dict(kw, obstacles=obst.detach()), obst)
    # shared table: the sum over the instances in the loss; the last instance starts inside obstacle 0 and does not converge
    s, p0, tab, x0 = _active_batch(pkg, sc, B, seed=9, shared=True)
    kw["x0"] = torch.as_tensor(x0, device=DEV)
    p0[-1, :2] = tab[0, :2] + 1.0
    p = torch.as_tensor(p0, device=DEV)
    tab_t = torch.as_tensor(tab, device=DEV).requires_grad_(True)
    x = pkg.SolveFunction.apply(s, p, None, kw, tab_t)
    ok = s.stats()["return_status"] == 0
    assert not bool(ok[-1]) and int(ok.sum()) >= 3, ok
    v = torch.randn_like(x)
    (x * v)[ok].sum().backward()
    sol = s(p=p, obstacles=tab, want_jac=True, **kw)
    jo = sol["jac_x_obst"]
    assert torch.isnan(jo[-1]).all() and int(has_active_obstacle(sc, sol["lam_g"].cpu().numpy()).sum()) >= 3
    ref = torch.einsum("bwoc,bw->oc", jo[ok], v[ok])
    assert torch.isfinite(tab_t.grad).all()
    assert torch.allclose(tab_t.grad, ref, rtol=1e-12, atol=1e-12 * float(ref.abs().max())), (tab_t.grad, ref)
    tab_t.grad = None
    x = pkg.SolveFunction.apply(s, p, None, kw, tab_t)
    (x * v).sum().backward()                       # the non-converged instance in the loss: NaN
    assert torch.isnan(tab_t.grad).any()
    # end to end: d/dr_0 of the sum of x^2 over the converged instances against a central difference -- a check of the plumbing
    # (sign, magnitude), with the step and the bound of test_sensitivity.test_autograd_backward
    tab_t = torch.as_tensor(tab, device=DEV).requires_grad_(True)
    x = pkg.SolveFunction.apply(s, p, None, kw, tab_t)
    okm = s.stats()["return_status"] == 0
    x[okm].square().sum().backward()
    h = 1e-2

    def L(dr):
        t = tab.copy()
        t[0, 2] += dr
        return s(p=p, obstacles=t, **kw)["x"][okm].square().sum().item()
    fd = (L(h) - L(-h)) / (2 * h)
    g = tab_t.grad[0, 2].item()
    print("d loss / d r_0: autograd %.6e, central difference %.6e" % (g, fd))
    assert abs(g) > 1e-3
    assert abs(g - fd) <= 5e-2 * max(1.0, abs(fd)), (g, fd)


@pytest.mark.gpu
def test_refusals(pkg):
    from mpc_implementation_b200 import _ffi
    L = _ffi.lib()
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 4
    p, _ = pkg.random_instances(sc, B, seed=2)
    s, sol = _solve(pkg, sc, p, want_jac=False)
    out = torch.empty((B, sc.n_w, sc.n_obs, 3), dtype=torch.float64, device=DEV)
    pt = torch.as_tensor(p, device=DEV)
    obs = s._dev_const("obs", s.obstacles)
    fn = b"nmpc_sensitivity_obstacles: "

    def call(BB=B, o=obs, flags=0, dst=out):
        return L.nmpc_sensitivity_obstacles(s._h, BB, sol["x"].data_ptr(), pt.data_ptr(), sol["lam_g"].data_ptr(),
                                            None if o is None else o.data_ptr(), flags, None if dst is None else dst.data_ptr(),
                                            None, None)

    def refused(rc, what):
        err = L.nmpc_last_error()
        return rc != 0 and err.startswith(fn) and what in err
    assert refused(L.nmpc_sensitivity_obstacles(None, B, None, None, None, None, 0, None, None, None), b"null handle")
    assert refused(call(), b"did not keep")
    s, sol = _solve(pkg, sc, p, want_jac=True, solver=s)
    assert call() == 0
    assert refused(call(B - 1), b"differs")
    assert refused(call(flags=_ffi.NMPC_PREDICT_TARGET), b"NMPC_PREDICT_TARGET")
    assert refused(call(o=None), b"obstacle table required")
    assert refused(call(dst=None), b"null required pointer")
    # a problem without obstacle rows (the gimbal-less layout): refused, and the facade has no jac_x_obst key
    g1 = pkg.SCENARIOS["gimbal_less"]
    p1, _ = pkg.random_instances(g1, B, seed=2)
    s1, sol1 = _solve(pkg, g1, p1, want_jac=True)
    assert "jac_x_obst" not in sol1 and "jac_x_p" in sol1
    rc = L.nmpc_sensitivity_obstacles(s1._h, B, sol1["x"].data_ptr(), torch.as_tensor(p1, device=DEV).data_ptr(),
                                      sol1["lam_g"].data_ptr(), None, 0, out.data_ptr(), None, None)
    assert refused(rc, b"no obstacle rows")
    # the facade: a stale key after the next solve
    _, sol = _solve(pkg, sc, p, want_jac=True, solver=s)
    _solve(pkg, sc, p, want_jac=False, solver=s)
    with pytest.raises(RuntimeError, match="jac_x_obst must be read before the next solve"):
        sol["jac_x_obst"]
    # the host path: numpy results, NaN rows exactly where the solve did not converge (instance 0 starts inside obstacle 0)
    obst = np.repeat(sc.obstacle_table()[None], B, axis=0)
    obst[0, 0, :2] = p[0, :2] + 1.0
    lb = sc.bounds()
    hs = s(x0=np.zeros((B, sc.n_w)), p=p, lbx=lb[0], ubx=lb[1], lbg=lb[2], ubg=lb[3], obstacles=obst, want_jac=True)
    hst = s.stats()["return_status"].copy()
    ho = hs["jac_x_obst"]
    assert isinstance(ho, np.ndarray) and ho.shape == (B, sc.n_w, sc.n_obs, 3)
    assert hst[0] != 0 and (hst == 0).sum() >= 2
    assert np.array_equal(np.isnan(ho).all(axis=(1, 2, 3)), hst != 0) and not np.isnan(ho[hst == 0]).any()
    # a single instance: the [n_w, n_obs, 3] form
    h1 = s(x0=np.zeros(sc.n_w), p=p[1], lbx=lb[0], ubx=lb[1], lbg=lb[2], ubg=lb[3], want_jac=True)
    assert h1["jac_x_obst"].shape == (sc.n_w, sc.n_obs, 3)
