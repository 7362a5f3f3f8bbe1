"""Solution sensitivities dx*/dp and dx*/d(w1, w2) of converged solves (nmpc_sensitivity, csrc/nmpc_sens.cuh).

W = grad2_ww L, M = grad2_{w th} L, J and J_th come from oracle/nlp_ref.py by autograd at a solution.  Two references use them:
  barrier   K dw/dth = -(M + J^T Sigma_g J_th), K = W + Sigma_x + J^T Sigma_g J, with the Sigmas the solve kept: the system the
            kernel solves, so it judges the kernel's LQ assembly and sweeps to rounding (self-calibrated as in
            test_riccati_kernel.py).  It takes the Sigmas from the kernel, so it cannot judge them.
  active    the mu -> 0 limit: the active bounds and rows of a strictly complementary solution become equalities, the inactive
            ones drop out.  It uses no Sigma.  On the CPU it is checked against central differences of oracle re-solves; on the
            GPU the kernel's columns are checked against it and against central differences of GPU re-solves, which is what
            judges the kept Sigmas (their unscaling and the relaxed-bound distances).
The limit system is singular in the controls that move only uncosted, inactive quantities (those of the last stages, whose effect
reaches only the terminal state or the states after the last costed stage): there neither the limit nor a difference quotient
across re-solves (which end at different mu) is determined, so the comparisons with the limit and with re-solves use the other
components -- those orthogonal to the null space of the limit system.
"""
import dataclasses

import mpmath
import numpy as np
import pytest
import scipy.linalg
import torch

from oracle import nlp_ref

LD = np.longdouble


# ---------------------------------------------------------------------------------------------------------------------
# dense references
# ---------------------------------------------------------------------------------------------------------------------
def dense_parts(sc, w, p, lam_g, obst, weights=None, target_traj=None):
    """W [n_w, n_w], M [n_w, n_th], J [n_g, n_w], J_th [n_g, n_th] at (w, p) with multipliers lam_g; th = p (+ (w1, w2) for
    model 0).  obst [n_obs][3] = (cx, cy, r_uav + r_obs)."""
    n_w, n_p = sc.n_w, sc.n_p
    if sc.model:
        spec = nlp_ref.RefSpec5(T=sc.T, N=sc.N)
        f_fn = lambda ww, pp, th: nlp_ref.objective5(spec, ww, pp)
        g_fn = lambda ww, pp: nlp_ref.constraints5(spec, ww, pp)
        n_th = n_p
    else:
        wt = (sc.w1, sc.w2) if weights is None else tuple(weights)
        spec0 = nlp_ref.RefSpec(T=sc.T, N=sc.N, obstacles=[tuple(o) for o in np.asarray(obst).reshape(-1, 3)], uav_r=0.0,
                                vfov=sc.vfov, hfov=sc.hfov)
        tt = None if target_traj is None else torch.tensor(np.asarray(target_traj, dtype=np.float64))

        def f_fn(ww, pp, th):
            s = dataclasses.replace(spec0, w1=th[0], w2=th[1])
            return nlp_ref.objective(s, ww, pp, tt)
        g_fn = lambda ww, pp: nlp_ref.constraints(spec0, ww, pp)
        n_th = n_p + 2
    lam = torch.tensor(np.asarray(lam_g, dtype=np.float64))
    th0 = np.concatenate([p, wt]) if not sc.model else np.asarray(p, dtype=np.float64)
    z0 = torch.tensor(np.concatenate([w, th0]), dtype=torch.float64)

    def lag(z):
        ww, pp = z[:n_w], z[n_w:n_w + n_p]
        return f_fn(ww, pp, z[n_w + n_p:]) + (lam * g_fn(ww, pp)).sum()
    H = torch.autograd.functional.hessian(lag, z0).numpy()
    Jz = torch.autograd.functional.jacobian(lambda z: g_fn(z[:n_w], z[n_w:n_w + n_p]), z0).numpy()
    return H[:n_w, :n_w], H[:n_w, n_w:n_w + n_th], Jz[:, :n_w], Jz[:, n_w:n_w + n_th]


def refine_solve(K, R):
    """X = -K^-1 R in float64 (X64) and refined in longdouble (Xr)."""
    X64 = np.linalg.solve(K, -R)
    X = X64.copy()
    for _ in range(4):
        res = K.astype(LD) @ X.astype(LD) + R.astype(LD)
        X = X - np.linalg.solve(K, res.astype(np.float64))
    return X64, X


def fov_grad_mp(sc, w, p, dps=50):
    """grad_w of the FOV term sum_k ((A (x_t - X_E)^2 + B (y_t - Y_E)(x_t - X_E) + C (y_t - Y_E)^2) - 1) -- the literal form of
    nlp_ref.objective, i.e. the right-hand side of the w2 column -- in mpmath at `dps` digits by central differences with
    h = 1e-25 (truncation ~h^2, rounding ~10^-dps / h: both far below float64)."""
    mp = mpmath.mp
    with mpmath.workdps(dps):
        V2, H2 = mp.mpf(sc.vfov) / 2, mp.mpf(sc.hfov) / 2
        T = mp.mpf(sc.T)
        pm = [mp.mpf(float(v)) for v in p]

        def fov(u):
            X = pm[0:8]
            tot = mp.mpf(0)
            for k in range(sc.N):
                st = X
                a = (st[2] * mp.tan(st[6] + V2) - st[2] * mp.tan(st[6] - V2)) / 2
                b = (st[2] * mp.tan(st[5] + H2) - st[2] * mp.tan(st[5] - H2)) / 2
                c7, s7 = mp.cos(st[7]), mp.sin(st[7])
                A = c7 ** 2 / a ** 2 + s7 ** 2 / b ** 2
                B = 2 * c7 * s7 * (1 / a ** 2 - 1 / b ** 2)
                C = s7 ** 2 / a ** 2 + c7 ** 2 / b ** 2
                XE = st[0] + a + st[2] * mp.tan(st[6] - V2)
                YE = st[1] + b + st[2] * mp.tan(st[5] - H2)
                xt, yt = pm[8], pm[9]
                tot += (A * (xt - XE) ** 2 + B * (yt - YE) * (xt - XE) + C * (yt - YE) ** 2) - 1
                v, o2, o3, o1g, o2g, o3g = u[6 * k: 6 * k + 6]
                th, ps = st[3], st[4]
                X = [st[0] + T * v * mp.cos(ps) * mp.cos(th), st[1] + T * v * mp.sin(ps) * mp.cos(th), st[2] + T * v * mp.sin(th),
                     st[3] + T * o2, st[4] + T * o3, st[5] + T * o1g, st[6] + T * o2g, st[7] + T * o3g]
            return tot
        u0 = [mp.mpf(float(v)) for v in w]
        h = mp.mpf("1e-25")
        g = np.empty(len(u0))
        for i in range(len(u0)):
            up, dn = list(u0), list(u0)
            up[i] += h
            dn[i] -= h
            g[i] = float((fov(up) - fov(dn)) / (2 * h))
    return g


def active_set(w, lam_x, g, lam_g, lbx, ubx, lbg, ubg, big=1e-3, small=1e-6, gap=1e-6):
    """(active control bounds, active rows) of a strictly complementary solution, or None when it is not one: every multiplier
    is either clearly nonzero (|lam| > big) with its constraint at the bound (relative distance <= gap), or clearly zero
    (|lam| < small) with its constraint clearly away from the bound (distance >= 1e3 gap)."""
    def pick(lam, v, lo, hi):
        act, ina = np.abs(lam) > big, np.abs(lam) < small
        d = np.minimum(np.abs(v - lo), np.abs(hi - v))
        if not np.all(act | ina) or np.any(act & (d > gap * np.maximum(1.0, np.abs(v)))) or np.any(ina & (d < 1e3 * gap)):
            return None
        return np.flatnonzero(act)
    ax, ag = pick(lam_x, w, lbx, ubx), pick(lam_g, g, lbg, ubg)
    return None if ax is None or ag is None else (ax, ag)


def active_sens(W, M, J, Jth, ax, ag):
    """dw/dth of the mu -> 0 limit, [W A^T; A 0] [dw; dnu] = -[M; A_th] with A the active bounds and rows (stage-0 rows are
    constant in w and drop out), and the mask of the components it determines (orthogonal to the null space of the system).
    Also returns the system, for the tolerance of the barrier comparison."""
    n_w = W.shape[0]
    ag = [r for r in ag if np.any(J[r] != 0.0)]
    A = np.concatenate([np.eye(n_w)[ax], J[ag]], axis=0)
    Ath = np.concatenate([np.zeros((len(ax), M.shape[1])), Jth[ag]], axis=0)
    m = A.shape[0]
    KKT = np.block([[W, A.T], [A, np.zeros((m, m))]])
    D = np.linalg.lstsq(KKT, -np.concatenate([M, Ath], axis=0), rcond=1e-12)[0][:n_w]
    null = scipy.linalg.null_space(KKT, rcond=1e-12)[:n_w]
    return D, np.abs(null).max(axis=1, initial=0.0) < 1e-8, KKT, ag


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the limit reference against central differences of oracle re-solves
# ---------------------------------------------------------------------------------------------------------------------
def test_active_set_reference_matches_oracle_finite_differences(oracle_mod, pkg):
    sc = pkg.SCENARIOS["t_trajectory"]
    lbx, ubx, lbg, ubg = sc.bounds()
    obst = sc.obstacle_table()
    sp = oracle_mod.make_spec(sc.T, sc.N, sc.n_obs, sc.w1, sc.w2, sc.vfov, sc.hfov)
    p, _ = pkg.random_instances(sc, 12, seed=5)
    ref = oracle_mod.solve(sp, obst, p, np.zeros((len(p), sc.n_w)), lbx, ubx, lbg, ubg, tol=1e-10)
    checked, worst = 0, 0.0
    for b in np.flatnonzero(ref["status"] == 0):
        act = active_set(ref["x"][b], ref["lam_x"][b], ref["g"][b], ref["lam_g"][b], lbx, ubx, lbg, ubg)
        if act is None:
            continue
        W, M, J, Jth = dense_parts(sc, ref["x"][b], p[b], ref["lam_g"][b], obst)
        D, det, _, _ = active_sens(W, M, J, Jth, *act)
        # h = 1e-4 max(1, |p_j|): the oracle solves to 1e-10, so re-solve noise is ~1e-10 / h <= 1e-6 of a column, and the h^2
        # term of the central difference is ~1e-8 |p_j|^2 x (third derivative) -- measured up to 2e-4 of a column for the
        # positions (|p_j| ~ 150).  The tolerance is 1e-3 of the column.
        for j in range(10):
            h = 1e-4 * max(1.0, abs(p[b, j]))
            pp = np.repeat(p[b:b + 1], 2, axis=0)
            pp[0, j] += h
            pp[1, j] -= h
            r = oracle_mod.solve(sp, obst, pp, np.repeat(ref["x"][b:b + 1], 2, axis=0), lbx, ubx, lbg, ubg, tol=1e-10)
            assert np.all(r["status"] == 0)
            fd = (r["x"][0] - r["x"][1]) / (2 * h)
            e = np.abs(fd - D[:, j])[det].max() / max(np.abs(D[det, j]).max(), 1e-3)
            worst = max(worst, e)
            assert e <= 1e-3, (b, j, e)
        checked += 1
    print("limit reference vs oracle central differences: %d instances, max rel err %.1e" % (checked, worst))
    assert checked >= 3, checked


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _scenario(pkg, N, n_obs, model):
    S = pkg.SCENARIOS
    if model:
        return S["gimbal_less"]
    base = S["t_trajectory"] if n_obs == 3 else S["race_track_2"]
    if n_obs == 7:
        base = dataclasses.replace(base, obstacles=base.obstacles[:7], name="race_track_2_7")
    return base if N == 15 else base.with_horizon(N)


LAYOUTS = [(15, 3, 0), (15, 10, 0), (30, 10, 0), (30, 3, 0), (5, 3, 0), (15, 7, 0), (15, 0, 1)]


def _solve(pkg, sc, p, B=None, weights=None, target_traj=None, obstacles=None, want_jac=True, solver=None, tol=1e-8):
    dev = "cuda:0"
    lbx, ubx, lbg, ubg = sc.bounds()
    s = solver or pkg.nlpsol("s", "ipm", sc, {"ipopt": {"max_iter": 100, "tol": tol}}, device=0, max_batch=len(p))
    pt = torch.as_tensor(p, device=dev)
    sol = s(x0=torch.zeros((len(p), sc.n_w), dtype=torch.float64, device=dev), p=pt, lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg,
            weights=weights, target_traj=target_traj, obstacles=obstacles, want_jac=want_jac)
    return s, sol


def _sigmas(s, B):
    sx = torch.empty((B, s.n_w), dtype=torch.float64, device="cuda:0")
    sg = torch.empty((B, s.n_g), dtype=torch.float64, device="cuda:0")
    from mpc_implementation_b200 import _ffi
    _ffi.check(_ffi.lib().nmpc_barrier_data(s._h, sx.data_ptr(), sg.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "nmpc_barrier_data")
    torch.cuda.synchronize()
    return sx.cpu().numpy(), sg.cpu().numpy()


def _barrier_check(sc, x, p, lam_g, sx, sg, obst, jac, weights=None, target_traj=None):
    """GPU columns against the dense barrier solve of the same data: per-column relative errors of the GPU and of the float64
    dense solve (the self-calibration).
    The w2 column's right-hand side is grad_w of the FOV term, which loses digits to cancellation in float64 on some instances
    (the target far outside the field of view): the kernel evaluates it in float64 (stage_cost_d2, the compact form the solve
    uses), and so does float64 autograd of the literal ellipse form.  The reference takes it at 50 digits (fov_grad_mp), and the
    calibration of that column includes what a float64 evaluation of the right-hand side costs: the solve of K with the
    difference between the float64 autograd value and the 50-digit one."""
    W, M, J, Jth = dense_parts(sc, x, p, lam_g, obst, weights, target_traj)
    K = W + np.diag(sx) + J.T @ (sg[:, None] * J)
    rhs_err = None
    if not sc.model:
        M = M.copy()
        g_mp = fov_grad_mp(sc, x, p)
        rhs_err = np.linalg.solve(K, M[:, -1] - g_mp)
        M[:, -1] = g_mp
    R = M + J.T @ (sg[:, None] * Jth)
    X64, Xr = refine_solve(K, R)
    scale = np.maximum(np.abs(Xr).max(axis=0), 1e-300)
    eg = (np.abs(jac - Xr) / scale).max(axis=0)
    ed = (np.abs(X64 - Xr) / scale).max()
    bound = np.full(eg.shape, max(32 * ed, 1e-11))
    if rhs_err is not None:
        bound[-1] = max(bound[-1], 32 * np.abs(rhs_err).max() / scale[-1])
    return eg, ed, bound


@pytest.mark.gpu
@pytest.mark.parametrize("N,n_obs,model", LAYOUTS)
def test_kernel_matches_dense_barrier_solve(pkg, N, n_obs, model):
    sc = _scenario(pkg, N, n_obs, model)
    B = 8
    p, _ = pkg.random_instances(sc, B, seed=11)
    s, sol = _solve(pkg, sc, p)
    st = s.stats()["return_status"].cpu().numpy()
    jp = sol["jac_x_p"].cpu().numpy()
    jw = None if model else sol["jac_x_w"].cpu().numpy()
    sx, sg = _sigmas(s, B)
    x, lg = sol["x"].cpu().numpy(), sol["lam_g"].cpu().numpy()
    ok = np.flatnonzero(st == 0)
    assert len(ok) >= B // 2, st
    assert np.all(np.isnan(jp[st != 0]))
    for b in ok:
        jac = jp[b] if model else np.concatenate([jp[b], jw[b]], axis=1)
        eg, ed, bound = _barrier_check(sc, x[b], p[b], lg[b], sx[b], sg[b], sc.obstacle_table(), jac)
        print(f"({N},{n_obs},{model}) b={b}: gpu rel err {eg.max():.2e}, float64 dense rel err {ed:.2e}, last column {eg[-1]:.2e} <= {bound[-1]:.2e}")
        assert np.all(eg <= bound), (b, eg, bound)


@pytest.mark.gpu
@pytest.mark.parametrize("N,n_obs,model", LAYOUTS)
def test_keep_barrier_changes_nothing(pkg, N, n_obs, model):
    """NMPC_KEEP_BARRIER runs a separately compiled kernel (ptxas schedules its copy of the phases differently): same results."""
    sc = _scenario(pkg, N, n_obs, model)
    p, _ = pkg.random_instances(sc, 64, seed=3)
    s, a = _solve(pkg, sc, p, want_jac=False)
    sa = {k: v.clone() for k, v in s.stats().items()}
    _, b = _solve(pkg, sc, p, want_jac=True, solver=s)
    sb = s.stats()
    for k in ("x", "f", "g", "lam_x", "lam_g"):
        assert torch.equal(a[k], b[k]), k
    for k in ("return_status", "iter_count"):
        assert torch.equal(sa[k], sb[k]), k


@pytest.mark.gpu
def test_zero_columns_and_per_instance_data(pkg):
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 6
    p, _ = pkg.random_instances(sc, B, seed=21)
    rng = np.random.default_rng(4)
    weights = np.stack([rng.uniform(0.5, 2.0, B), rng.uniform(1.0, 3.0, B)], axis=1)
    obst = np.repeat(sc.obstacle_table()[None], B, axis=0)
    obst[:, :, :2] = p[:, None, :2] + rng.uniform(100, 200, (B, sc.n_obs, 2))      # each instance its own obstacles
    s, sol = _solve(pkg, sc, p, weights=weights, obstacles=obst)
    st = s.stats()["return_status"].cpu().numpy()
    jp, jw = sol["jac_x_p"].cpu().numpy(), sol["jac_x_w"].cpu().numpy()
    ok = st == 0
    assert ok.sum() >= 3
    assert np.all(jp[ok][:, :, 10] == 0.0)                                             # theta_t
    sx, sg = _sigmas(s, B)
    x, lg = sol["x"].cpu().numpy(), sol["lam_g"].cpu().numpy()
    for b in np.flatnonzero(ok):
        eg, ed, bound = _barrier_check(sc, x[b], p[b], lg[b], sx[b], sg[b], obst[b], np.concatenate([jp[b], jw[b]], axis=1), weights[b])
        print(f"per-instance weights and obstacles b={b}: gpu rel err {eg.max():.2e}, float64 dense rel err {ed:.2e}")
        assert np.all(eg <= bound), (b, eg, bound)
    # a per-stage target trajectory: the target columns are exactly 0
    tt = np.repeat(p[:, None, 8:10], sc.N, axis=1) + np.linspace(0, 5, sc.N)[None, :, None]
    s2, sol2 = _solve(pkg, sc, p, target_traj=tt)
    ok2 = s2.stats()["return_status"].cpu().numpy() == 0
    assert np.all(sol2["jac_x_p"].cpu().numpy()[ok2][:, :, 8:11] == 0.0)


@pytest.mark.gpu
def test_finite_differences_and_active_set_limit(pkg):
    """(b) central differences of GPU re-solves and (a') the mu -> 0 limit, on strictly complementary instances.  Neither uses the
    kept Sigmas: both judge them."""
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 24
    p, _ = pkg.random_instances(sc, B, seed=7)
    lbx, ubx, lbg, ubg = sc.bounds()
    s, sol = _solve(pkg, sc, p, tol=1e-10)          # 1e-10: the re-solves below end closer to their solutions
    st = s.stats()["return_status"].cpu().numpy()
    jp, jw = sol["jac_x_p"].cpu().numpy(), sol["jac_x_w"].cpu().numpy()
    sx, sg = _sigmas(s, B)
    x, lx, g, lg = (sol[k].cpu().numpy() for k in ("x", "lam_x", "g", "lam_g"))
    picked = [b for b in np.flatnonzero(st == 0) if active_set(x[b], lx[b], g[b], lg[b], lbx, ubx, lbg, ubg) is not None]
    assert len(picked) >= 3, len(picked)
    cols = list(range(10))
    s2 = pkg.nlpsol("fd", "ipm", sc, {"ipopt": {"max_iter": 100, "tol": 1e-10}}, device=0, max_batch=2 * len(cols) + 4)
    fd_err, lim_err = [], []
    for b in picked[:4]:
        ax, ag = active_set(x[b], lx[b], g[b], lg[b], lbx, ubx, lbg, ubg)
        W, M, J, Jth = dense_parts(sc, x[b], p[b], lg[b], sc.obstacle_table())
        D, det, KKT, agj = active_sens(W, M, J, Jth, ax, ag)
        jac = np.concatenate([jp[b], jw[b]], axis=1)
        # (a') The barrier system is the limit system with the active constraints weighted by Sigma_act ~ z^2 / mu instead of
        # being exact, and the inactive ones weighted by Sigma_in ~ mu / d^2 instead of dropped.  First-order perturbation of the
        # limit solution: relative change <= ||KKT^+|| (||KKT||^2 / Sigma_act,min + Sigma_in,max), both of order the final mu.
        # The Sigmas here only size that bound; the tolerance is 10x it.
        sxb, sgb = sx[b], sg[b]
        act_w = np.concatenate([sxb[ax], sgb[agj] * np.sum(J[agj] ** 2, axis=1)])
        ina = np.setdiff1d(np.arange(sc.n_w), ax)
        inr = np.array([r for r in range(sc.n_g) if r not in set(ag) and np.any(J[r] != 0.0)], dtype=int)
        in_w = np.concatenate([sxb[ina], sgb[inr] * np.sum(J[inr] ** 2, axis=1)])
        sv = np.linalg.svd(KKT, compute_uv=False)
        nk, nki = sv[0], 1.0 / sv[sv > 1e-12 * sv[0]][-1]
        bound = nki * (nk ** 2 / act_w.min() + in_w.max())
        scale = np.maximum(np.abs(D[det]).max(axis=0), 1e-3)
        e = (np.abs(jac - D)[det] / scale).max()
        lim_err.append(e)
        print(f"b={b}: barrier vs limit rel err {e:.2e}, bound {bound:.2e}")
        assert e <= 10 * bound, (b, e, bound)
        # (b) h = 1e-4 max(1, |p_j|) and 1e-4 for the weights: the re-solves stop at tol 1e-10, so their noise is ~1e-10 / h, and
        # the h^2 term is ~1e-8 |p_j|^2 x (third derivative), as in the CPU test
        hs = [1e-4 * max(1.0, abs(p[b, j])) for j in cols]
        pp = np.repeat(p[b:b + 1], 2 * len(cols), axis=0)
        for i, (j, h) in enumerate(zip(cols, hs)):
            pp[2 * i, j] += h
            pp[2 * i + 1, j] -= h
        _, r = _solve(pkg, sc, pp, want_jac=False, solver=s2)
        assert np.all(s2.stats()["return_status"].cpu().numpy() == 0)
        xr = r["x"].cpu().numpy()
        for i, (j, h) in enumerate(zip(cols, hs)):
            fd = (xr[2 * i] - xr[2 * i + 1]) / (2 * h)
            fd_err.append(np.abs(fd - jp[b][:, j])[det].max() / max(np.abs(jp[b][det, j]).max(), 1e-3))
        h = 1e-4
        wts = np.array([[sc.w1 + h, sc.w2], [sc.w1 - h, sc.w2], [sc.w1, sc.w2 + h], [sc.w1, sc.w2 - h]])
        _, r = _solve(pkg, sc, np.repeat(p[b:b + 1], 4, axis=0), weights=wts, want_jac=False, solver=s2)
        assert np.all(s2.stats()["return_status"].cpu().numpy() == 0)
        xr = r["x"].cpu().numpy()
        for k in range(2):
            fd = (xr[2 * k] - xr[2 * k + 1]) / (2 * h)
            fd_err.append(np.abs(fd - jw[b][:, k])[det].max() / max(np.abs(jw[b][det, k]).max(), 1e-3))
    print("central differences of re-solves: max rel err %.2e;  limit: max rel err %.2e" % (max(fd_err), max(lim_err)))
    assert max(fd_err) <= FD_TOL, fd_err


# Central differences of the re-solves agreed with the kernel's columns to 5.3e-5 of a column on the determined components
# (measured on a B200); the tolerance is the CPU test's for the same step, 1e-3, about 20x that.
FD_TOL = 1e-3


@pytest.mark.gpu
def test_autograd_backward(pkg):
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 8
    p0, _ = pkg.random_instances(sc, B, seed=9)
    lbx, ubx, lbg, ubg = sc.bounds()
    s = pkg.nlpsol("s", "ipm", sc, {"ipopt": {"max_iter": 100}}, device=0, max_batch=B)
    kw = dict(x0=torch.zeros((B, sc.n_w), dtype=torch.float64, device="cuda:0"), lbx=lbx, ubx=ubx, lbg=lbg, ubg=ubg)
    p = torch.as_tensor(p0, device="cuda:0").requires_grad_(True)
    w = torch.tensor([[sc.w1, sc.w2]] * B, dtype=torch.float64, device="cuda:0", requires_grad=True)
    x = pkg.SolveFunction.apply(s, p, w, kw)
    ok = s.stats()["return_status"] == 0
    v = torch.randn_like(x)
    (x * v)[ok].sum().backward()
    sol = s(p=p.detach(), weights=w.detach(), want_jac=True, **kw)
    ref_p = torch.einsum("bwp,bw->bp", sol["jac_x_p"], v)
    ref_w = torch.einsum("bwk,bw->bk", sol["jac_x_w"], v)
    assert torch.equal(p.grad[ok], ref_p[ok]) and torch.equal(w.grad[ok], ref_w[ok])
    # tiny end-to-end use: d/dw1 of sum x^2 against a central difference
    w1 = torch.tensor(1.0, dtype=torch.float64, device="cuda:0", requires_grad=True)
    wb = torch.stack([w1.expand(B), torch.full((B,), sc.w2, dtype=torch.float64, device="cuda:0")], dim=1)
    x = pkg.SolveFunction.apply(s, torch.as_tensor(p0, device="cuda:0"), wb, kw)
    okm = (s.stats()["return_status"] == 0)
    loss = x[okm].square().sum()
    loss.backward()
    # h = 1e-2: the solves stop at tol 1e-8, and x enters the loss with |x| up to 30 over 90 entries, so a smaller step drowns
    # the difference in re-solve noise (h = 1e-5 gave a difference quotient off by 40 %).  At h = 1e-2 the two differ by 3 %
    # (measured on a B200): the barrier sensitivity is the derivative at the final mu, the difference quotient also sees
    # bounds that become active or inactive between w1 - h and w1 + h.  The bound is 5 %: a check of the end-to-end use
    # (sign, magnitude, the plumbing of the weights through autograd), not of the sensitivity's accuracy, which the dense
    # comparisons above pin to rounding.
    h = 1e-2

    def L(w1v):
        wv = torch.tensor([[w1v, sc.w2]] * B, dtype=torch.float64, device="cuda:0")
        return s(p=torch.as_tensor(p0, device="cuda:0"), weights=wv, **kw)["x"][okm].square().sum().item()
    fd = (L(1.0 + h) - L(1.0 - h)) / (2 * h)
    print("d loss / d w1: autograd %.6e, central difference %.6e" % (w1.grad.item(), fd))
    assert abs(w1.grad.item() - fd) <= 5e-2 * max(1.0, abs(fd)), (w1.grad.item(), fd)


@pytest.mark.gpu
def test_refusals(pkg):
    from mpc_implementation_b200 import _ffi
    L = _ffi.lib()
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 4
    p, vw = pkg.random_instances(sc, B, seed=2)
    s, sol = _solve(pkg, sc, p, want_jac=False)
    dev = "cuda:0"
    out = torch.empty((B, sc.n_w, sc.n_p), dtype=torch.float64, device=dev)
    pt = torch.as_tensor(p, device=dev)
    obs = s._dev_const("obs", s.obstacles)
    call = lambda BB, dw=None, h=s._h: L.nmpc_sensitivity(h, BB, sol["x"].data_ptr(), pt.data_ptr(), sol["lam_g"].data_ptr(), obs.data_ptr(), 0,
                                                            out.data_ptr(), dw, None, None)
    assert call(B) != 0 and b"nmpc_sensitivity" in L.nmpc_last_error() and b"did not keep" in L.nmpc_last_error()
    s, sol = _solve(pkg, sc, p, want_jac=True, solver=s)
    assert call(B) == 0
    assert call(B - 1) != 0 and b"differs" in L.nmpc_last_error()
    # the fused and free-running calls refuse the flag
    lbx, ubx, lbg, ubg = (s._dev_const(k, a) for k, a in zip(("lbx", "ubx", "lbg", "ubg"), sc.bounds()))
    u = torch.zeros((B, sc.n_w), dtype=torch.float64, device=dev)
    vwt = torch.as_tensor(vw, device=dev)
    f = torch.empty(B, dtype=torch.float64, device=dev)
    rc = L.nmpc_solve_and_step(s._h, B, pt.data_ptr(), u.data_ptr(), lbx.data_ptr(), ubx.data_ptr(), lbg.data_ptr(), ubg.data_ptr(),
                               obs.data_ptr(), _ffi.NMPC_KEEP_BARRIER, vwt.data_ptr(), None, f.data_ptr(), None, None, None, None, None)
    assert rc != 0 and b"nmpc_solve_and_step: NMPC_KEEP_BARRIER" in L.nmpc_last_error()
    rc = L.nmpc_run_closed_loop(s._h, B, 2, pt.data_ptr(), u.data_ptr(), lbx.data_ptr(), ubx.data_ptr(), lbg.data_ptr(), ubg.data_ptr(),
                                obs.data_ptr(), _ffi.NMPC_KEEP_BARRIER, vwt.data_ptr(), None, f.data_ptr(), None, None, None, None, None, None)
    assert rc != 0 and b"nmpc_run_closed_loop: NMPC_KEEP_BARRIER" in L.nmpc_last_error()
    # dx_dw for model 1
    g1 = pkg.SCENARIOS["gimbal_less"]
    p1, _ = pkg.random_instances(g1, B, seed=2)
    s1, sol1 = _solve(pkg, g1, p1, want_jac=True)
    dw = torch.empty((B, g1.n_w, 2), dtype=torch.float64, device=dev)
    out1 = torch.empty((B, g1.n_w, g1.n_p), dtype=torch.float64, device=dev)
    rc = L.nmpc_sensitivity(s1._h, B, sol1["x"].data_ptr(), torch.as_tensor(p1, device=dev).data_ptr(), sol1["lam_g"].data_ptr(), None, 0,
                            out1.data_ptr(), dw.data_ptr(), None, None)
    assert rc != 0 and b"nmpc_sensitivity: dx_dw is for model 0 only" in L.nmpc_last_error()
    # the facade: a stale jacobian after the next solve
    _, sol = _solve(pkg, sc, p, want_jac=True, solver=s)
    _solve(pkg, sc, p, want_jac=False, solver=s)
    with pytest.raises(RuntimeError, match="before the next solve"):
        sol["jac_x_p"]
    # the host path: numpy results of the right shape, NaN rows exactly where the solve did not converge
    lb = sc.bounds()
    hs = s(x0=np.zeros((B, sc.n_w)), p=p, lbx=lb[0], ubx=lb[1], lbg=lb[2], ubg=lb[3], want_jac=True)
    hst = s.stats()["return_status"].copy()
    hj, hw = hs["jac_x_p"], hs["jac_x_w"]
    assert isinstance(hj, np.ndarray) and hj.shape == (B, sc.n_w, sc.n_p) and hw.shape == (B, sc.n_w, 2)
    assert np.array_equal(np.isnan(hj).all(axis=(1, 2)), hst != 0) and not np.isnan(hj[hst == 0]).any()
