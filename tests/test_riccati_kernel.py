"""The Riccati factorisation and sweeps (csrc/nmpc_riccati.cuh) against a high-precision reference of the stage LQ problem.

The kernel runs through its own harness (csrc/ric_harness.cu -> libnmpc_ric_harness.so) on generated LQ data, one warp per
instance, for the seven production layouts and five forced edge layouts.  The reference is written from the data
contract between ph_derivs and the factorisation (DESIGN.md section 2.1), not from the kernel's ownership maps:

  stages k = 0..N-1, terminal stage N, entry e of stage k at LQ0 + e S + k
  dx_0 = 0,  dx_{k+1} = A_k dx_k + B_k du_k,   A_k = I + EE at (0,3) (1,3) (2,3) (0,4) (1,4)  (EE holds T already),
                                               B_k[0:3, 0] = T DD,  B_k[i+2, i] = T (i = 1..5)
  Q_k: LQ_Q[0..20] packed lower over states (0,1,2,5,6,7), LQ_Q[21..23] = (3,3) (4,3) (4,4); without FOLD + dw NN on
       (0,0) (0,1) (1,1) and dw DG on the diagonal of states 2, 3, 5, 6, 7
  R_k = diag(RD + dw),  S_k (state, control): (3,0) = SV0, (4,0) = SV1,  r_k = mu RB,
  q_k = QA + mu QB + dw QD (without FOLD) or QA (FOLD: mu and dw are folded in),  LQ_ZERO = 0
  du_k = -K_k dx_k - kappa_k;  the SOC re-solve uses the same factors with q replaced by q' and the same r.

It is solved two ways: (a) a textbook Riccati recursion in np.longdouble and (b) a dense condensed solve (dx eliminated)
factored in float64 with iterative refinement in longdouble.  The CPU tests show (a) and (b) agree, inertia verdicts
included, before (a) judges the kernel in the GPU tests.
"""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "mpc-implementation_b200" / "csrc"
HARNESS = Path(os.environ.get("NMPC_RIC_HARNESS_LIB", CSRC / "libnmpc_ric_harness.so"))   # override: a rebuilt harness

LD = np.longdouble
EPS = np.finfo(np.float64).eps

# the order of ric_consts in ric_harness.cu
RIC_CONSTS = ["N", "S", "MODEL", "FOLD", "TOTAL", "LV0", "RW0", "LQ0", "LQ_NE", "SOCX0", "STG0", "OBS0", "ALG0", "RES0",
              "PAR0", "SOC_DUS", "SOC_Q2", "STG_N", "RIC_N", "RIC_K", "RIC_L", "RIC_K2", "RIC_MAP_WORDS", "LV_DX", "LV_DU",
              "LV_N", "LQ_Q", "LQ_DEAD", "LQ_QA", "LQ_SV", "LQ_RD", "LQ_RB", "LQ_DD", "LQ_EE", "LQ_ZERO", "LQ_DG", "LQ_NN",
              "LQ_QD", "LQ_QB"]
# harness tag -> (N, n_obs, model, FOLD or None for the production choice)
LAYOUTS = {"p15_3": (15, 3, 0, None), "p15_10": (15, 10, 0, None), "p30_10": (30, 10, 0, None), "p30_3": (30, 3, 0, None),
           "p5_3": (5, 3, 0, None), "p15_7": (15, 7, 0, None), "p15_0_1": (15, 0, 1, None),
           "f15_3": (15, 3, 0, True), "n30_10": (30, 10, 0, False), "n1_3": (1, 3, 0, False), "n2_3": (2, 3, 0, False),
           "n31_16": (31, 16, 0, False)}
TS = (0.2, 1.0, 0.37)
# sizes of the logical LQ entries (generator / reference); packed at the layout's offsets by pack_lq
ENT = {"Q": 24, "QA": 8, "SV": 2, "RD": 6, "RB": 6, "DD": 3, "EE": 5, "DG": 5, "NN": 3, "QD": 8, "QB": 8}
CS = (0, 1, 2, 5, 6, 7)       # states of the packed 6 x 6 block of LQ_Q


def tri(r, c):
    return r * (r + 1) // 2 + c if r >= c else c * (c + 1) // 2 + r


# ---------------------------------------------------------------------------------------------------------------------
# input generator
# ---------------------------------------------------------------------------------------------------------------------
def gen_lq(rng, B, N, model=0, neg=1.0, rd=None):
    """B instances of stage LQ data with the solver's structure and magnitudes.  Returns the logical entries {name: [B, n, S]}.
    Q_k is indefinite (an obstacle-like negative curvature in the x-y plane, scaled by `neg`), RD spans 1e-8 .. 1e10
    (or is `rd` for every present control)."""
    S = N + 1
    d = {}
    M = rng.standard_normal((B, S, 6, 6)) * np.exp(rng.uniform(-1.0, 1.0, (B, S, 1, 1)))
    Qc = M @ np.swapaxes(M, -1, -2) / 6.0
    v = np.zeros((B, S, 6))
    ang = rng.uniform(0.0, 2 * np.pi, (B, S))
    v[..., 0], v[..., 1] = np.cos(ang), np.sin(ang)
    # Qc - c v v' is singular at c = 1 / v' Qc^-1 v and has one negative eigenvalue beyond: so on about a third of the
    # stages (those near an obstacle) the x-y block gets a negative curvature that grows with `neg`
    w = 1.0 / np.einsum("bsi,bsi->bs", v, np.linalg.solve(Qc, v[..., None])[..., 0])
    c = w * (1.0 + 0.5 * neg) * (rng.uniform(0.0, 1.0, (B, S)) < 0.35)
    Qc = Qc - c[..., None, None] * v[..., :, None] * v[..., None, :]
    M2 = rng.standard_normal((B, S, 2, 2))
    Qa = M2 @ np.swapaxes(M2, -1, -2) / 2.0 + 0.05 * np.eye(2)
    q = np.zeros((B, 24, S))
    for a in range(6):
        for b in range(a + 1):
            q[:, tri(a, b)] = Qc[:, :, a, b]
    q[:, 21], q[:, 22], q[:, 23] = Qa[:, :, 0, 0], Qa[:, :, 1, 0], Qa[:, :, 1, 1]
    d["Q"] = q
    d["QA"] = rng.standard_normal((B, 8, S))
    d["QB"] = rng.standard_normal((B, 8, S))
    d["QD"] = rng.standard_normal((B, 8, S))
    d["RD"] = 10.0 ** rng.uniform(-8.0, 10.0, (B, 6, S)) if rd is None else np.full((B, 6, S), rd)
    # v-theta / v-psi couplings, small enough to keep [R S; S^T Q] from being indefinite on their own
    d["SV"] = 0.3 * rng.standard_normal((B, 2, S)) * np.sqrt(d["RD"][:, :1] * Qa[:, :, [0, 1], [0, 1]].transpose(0, 2, 1))
    d["RB"] = rng.standard_normal((B, 6, S))
    th, ps = rng.uniform(-0.6, 0.6, (B, S)), rng.uniform(-np.pi, np.pi, (B, S))
    d["DD"] = np.stack([np.cos(ps) * np.cos(th), np.sin(ps) * np.cos(th), np.sin(th)], axis=1)
    tv = rng.uniform(0.5, 5.0, (B, S)) * rng.choice(TS, (B, 1))     # T v (EE holds T already)
    d["EE"] = np.stack([-tv * np.cos(ps) * np.sin(th), -tv * np.sin(ps) * np.sin(th), tv * np.cos(th),
                        -tv * np.sin(ps) * np.cos(th), tv * np.cos(ps) * np.cos(th)], axis=1)
    d["DG"] = 10.0 ** rng.uniform(-2.0, 2.0, (B, 5, S))
    nn = rng.standard_normal((B, 2, S))
    d["NN"] = np.stack([nn[:, 0] ** 2 + 0.1, nn[:, 0] * nn[:, 1], nn[:, 1] ** 2 + 0.1], axis=1)
    if model == 1:      # the absent camera controls / states, as ph_derivs sets them
        d["RD"][:, 3:] = 1.0
        d["RB"][:, 3:] = 0.0
        for a in range(6):
            for b in range(a + 1):
                if a >= 3:
                    d["Q"][:, tri(a, b)] = 0.0
        for e in ("QA", "QB", "QD"):
            d[e][:, 5:] = 0.0
        d["DG"][:, 2:] = 0.0
    return d


def take(d, idx):
    return {k: v[idx] for k, v in d.items()}


def join(*ds):
    return {k: np.concatenate([d[k] for d in ds]) for k in ds[0]}


# ---------------------------------------------------------------------------------------------------------------------
# reference (a): the stage problem from the data contract, and the textbook Riccati recursion in any dtype
# ---------------------------------------------------------------------------------------------------------------------
def stage_problem(d, T, mu, dw, fold, dtype=LD):
    """A [B,N,8,8], Bu [B,N,8,6], Q [B,S,8,8], R [B,N,6,6], Sx [B,N,8,6] (state, control), q [B,S,8], r [B,N,6]"""
    g = {k: np.asarray(v, np.float64).astype(dtype) for k, v in d.items()}
    T, mu, dw = (np.asarray(x, np.float64).astype(dtype) for x in (T, mu, dw))
    Bn, _, S = g["QA"].shape
    N = S - 1
    A = np.zeros((Bn, N, 8, 8), dtype) + np.eye(8, dtype=dtype)
    for e, (i, j) in enumerate(((0, 3), (1, 3), (2, 3), (0, 4), (1, 4))):
        A[:, :, i, j] = g["EE"][:, e, :N]
    Bu = np.zeros((Bn, N, 8, 6), dtype)
    Bu[:, :, 0:3, 0] = T[:, None, None] * np.swapaxes(g["DD"][:, :, :N], 1, 2)
    for i in range(1, 6):
        Bu[:, :, i + 2, i] = T[:, None]
    Q = np.zeros((Bn, S, 8, 8), dtype)
    for a in range(6):
        for b in range(a + 1):
            Q[:, :, CS[a], CS[b]] = Q[:, :, CS[b], CS[a]] = g["Q"][:, tri(a, b)]
    Q[:, :, 3, 3] = g["Q"][:, 21]
    Q[:, :, 3, 4] = Q[:, :, 4, 3] = g["Q"][:, 22]
    Q[:, :, 4, 4] = g["Q"][:, 23]
    q = np.swapaxes(g["QA"], 1, 2).copy()
    if not fold:
        w = dw[:, None]
        Q[:, :, 0, 0] += w * g["NN"][:, 0]
        Q[:, :, 0, 1] += w * g["NN"][:, 1]
        Q[:, :, 1, 0] += w * g["NN"][:, 1]
        Q[:, :, 1, 1] += w * g["NN"][:, 2]
        for e, s in enumerate((2, 3, 5, 6, 7)):
            Q[:, :, s, s] += w * g["DG"][:, e]
        q += mu[:, None, None] * np.swapaxes(g["QB"], 1, 2) + dw[:, None, None] * np.swapaxes(g["QD"], 1, 2)
    R = np.zeros((Bn, N, 6, 6), dtype)
    for i in range(6):
        R[:, :, i, i] = g["RD"][:, i, :N] + dw[:, None]
    Sx = np.zeros((Bn, N, 8, 6), dtype)
    Sx[:, :, 3, 0] = g["SV"][:, 0, :N]
    Sx[:, :, 4, 0] = g["SV"][:, 1, :N]
    r = mu[:, None, None] * np.swapaxes(g["RB"][:, :, :N], 1, 2)
    return dict(A=A, Bu=Bu, Q=Q, R=R, Sx=Sx, q=q, r=r, N=N, dtype=dtype)


def chol6(Lam):
    """Batched Cholesky of [B,6,6]; returns L (lower, with NaN past a non-positive pivot) and the pivots d_j."""
    L = np.zeros_like(Lam)
    piv = np.zeros(Lam.shape[:-1], Lam.dtype)
    with np.errstate(invalid="ignore", divide="ignore"):
        for j in range(6):
            dj = Lam[:, j, j] - np.sum(L[:, j, :j] ** 2, axis=-1)
            piv[:, j] = dj
            L[:, j, j] = np.sqrt(np.where(dj > 0, dj, np.nan))
            for i in range(j + 1, 6):
                L[:, i, j] = (Lam[:, i, j] - np.sum(L[:, i, :j] * L[:, j, :j], axis=-1)) / L[:, j, j]
    return L, piv


def chol_solve(L, b):
    """L L^T x = b for b [B,6,m]"""
    y = np.zeros_like(b)
    with np.errstate(invalid="ignore"):
        for i in range(6):
            y[:, i] = (b[:, i] - np.einsum("bk,bkm->bm", L[:, i, :i], y[:, :i])) / L[:, i, i, None]
        x = np.zeros_like(b)
        for i in range(5, -1, -1):
            x[:, i] = (y[:, i] - np.einsum("bk,bkm->bm", L[:, i + 1:, i], x[:, i + 1:])) / L[:, i, i, None]
    return x


def riccati(pb, q2=None):
    """Textbook Riccati recursion + forward sweeps on the stage problem pb (any dtype).  q2 [B,8,S]: SOC right-hand side."""
    A, Bu, Q, R, Sx, q, r, N = (pb[k] for k in ("A", "Bu", "Q", "R", "Sx", "q", "r", "N"))
    Bn, dt = A.shape[0], pb["dtype"]
    out = {k: np.full((Bn, N) + s, np.nan, dt) for k, s in
           (("K", (6, 8)), ("kap", (6,)), ("Lc", (6, 6)), ("piv", (6,)), ("lamd", (6,)), ("G", (6, 8)), ("kap2", (6,)))}
    ok = np.ones(Bn, bool)
    fail = np.full(Bn, -1)
    P, p = Q[:, N].copy(), q[:, N].copy()
    with np.errstate(invalid="ignore", over="ignore"):
        for k in range(N - 1, -1, -1):
            PB = P @ Bu[:, k]
            Lam = R[:, k] + np.swapaxes(Bu[:, k], 1, 2) @ PB
            G = np.swapaxes(Sx[:, k], 1, 2) + np.swapaxes(PB, 1, 2) @ A[:, k]
            g = r[:, k] + np.einsum("bij,bi->bj", Bu[:, k], p)
            Lc, piv = chol6(Lam)
            out["piv"][:, k], out["lamd"][:, k] = piv, np.diagonal(Lam, axis1=1, axis2=2)
            bad = ok & ~(piv > 0).all(-1)
            fail[bad] = k
            ok &= ~bad
            X = chol_solve(Lc, np.concatenate([G, g[:, :, None]], axis=2))
            K, kap = X[:, :, :8], X[:, :, 8]
            out["K"][:, k], out["kap"][:, k], out["Lc"][:, k], out["G"][:, k] = K, kap, Lc, G
            At = np.swapaxes(A[:, k], 1, 2)
            P = Q[:, k] + At @ P @ A[:, k] - np.swapaxes(G, 1, 2) @ K
            P = 0.5 * (P + np.swapaxes(P, 1, 2))
            p = q[:, k] + np.einsum("bij,bj->bi", At, p) - np.einsum("bri,br->bi", G, kap)
    out["ok"], out["fail"] = ok, fail
    out["dx"], out["du"] = forward(pb, out["K"], out["kap"])
    if q2 is not None:
        q2 = np.asarray(q2, np.float64).astype(dt)
        p = q2[:, :, N].copy()
        with np.errstate(invalid="ignore", over="ignore"):
            for k in range(N - 1, -1, -1):
                g = r[:, k] + np.einsum("bij,bi->bj", Bu[:, k], p)
                kap2 = chol_solve(out["Lc"][:, k], g[:, :, None])[:, :, 0]
                out["kap2"][:, k] = kap2
                p = q2[:, :, k] + np.einsum("bji,bj->bi", A[:, k], p) - np.einsum("bri,br->bi", out["G"][:, k], kap2)
        out["dx2"], out["du2"] = forward(pb, out["K"], out["kap2"])
    return out


def forward(pb, K, kap):
    A, Bu, N = pb["A"], pb["Bu"], pb["N"]
    Bn, dt = A.shape[0], pb["dtype"]
    dx = np.zeros((Bn, N + 1, 8), dt)
    du = np.zeros((Bn, N, 6), dt)
    with np.errstate(invalid="ignore", over="ignore"):
        for k in range(N):
            du[:, k] = -np.einsum("bij,bj->bi", K[:, k], dx[:, k]) - kap[:, k]
            dx[:, k + 1] = np.einsum("bij,bj->bi", A[:, k], dx[:, k]) + np.einsum("bij,bj->bi", Bu[:, k], du[:, k])
    return dx, du


# ---------------------------------------------------------------------------------------------------------------------
# reference (b): dense condensed solve
# ---------------------------------------------------------------------------------------------------------------------
def condensed(pb, q2=None, solve_step=True):
    """Eliminate dx (dx = G du), form the 6N x 6N reduced Hessian H and gradient g, solve H du = -g in float64 with two
    steps of iterative refinement whose residuals are longdouble.  Also the smallest eigenvalue of the Jacobi-scaled H
    relative to its largest (its sign is the sign of H's smallest eigenvalue: congruence)."""
    A, Bu, Q, R, Sx, q, r, N = (pb[k] for k in ("A", "Bu", "Q", "R", "Sx", "q", "r", "N"))
    Bn, S = A.shape[0], N + 1
    Gm = np.zeros((Bn, S, 8, N, 6), LD)
    for k in range(N):
        Gm[:, k + 1] = np.einsum("bij,bjnc->binc", A[:, k], Gm[:, k])
        Gm[:, k + 1, :, k, :] += Bu[:, k]
    Gf = Gm.reshape(Bn, S, 8, 6 * N)

    def hv(u):          # H u in longdouble, without forming H
        x = np.einsum("bsim,bm->bsi", Gf, u)
        uk = u.reshape(Bn, N, 6)
        y = np.einsum("bsij,bsj->bsi", Q, x)
        y[:, :N] += np.einsum("bkic,bkc->bki", Sx, uk)
        out = np.einsum("bsim,bsi->bm", Gf, y)
        out += (np.einsum("bkij,bkj->bki", R, uk) + np.einsum("bkic,bki->bkc", Sx, x[:, :N])).reshape(Bn, 6 * N)
        return out

    g = r.reshape(Bn, 6 * N) + np.einsum("bsim,bsi->bm", Gf, q)
    Gd = Gf.astype(np.float64)
    H = (np.einsum("bsim,bsij,bsjn->bmn", Gd, Q.astype(np.float64), Gd))
    Rd = np.zeros((Bn, 6 * N, 6 * N))
    for k in range(N):
        Rd[:, 6 * k:6 * k + 6, 6 * k:6 * k + 6] = R[:, k].astype(np.float64)
    SG = np.einsum("bkic,bkim->bkcm", Sx.astype(np.float64), Gd[:, :N]).reshape(Bn, 6 * N, 6 * N)
    H = H + Rd + SG + np.swapaxes(SG, 1, 2)
    H = 0.5 * (H + np.swapaxes(H, 1, 2))
    hd = np.abs(np.diagonal(H, axis1=1, axis2=2))
    dsc = 1.0 / np.sqrt(np.where(hd > 0, hd, 1.0))
    Hs = H * dsc[:, :, None] * dsc[:, None, :]
    ev = np.linalg.eigvalsh(Hs)
    lam_rel = ev[:, 0] / np.abs(ev).max(-1)

    def solve(rhs):
        u = (dsc * np.linalg.solve(Hs, (dsc * rhs.astype(np.float64))[..., None])[..., 0]).astype(LD)
        for _ in range(2):
            res = rhs - hv(u)
            u = u + (dsc * np.linalg.solve(Hs, (dsc * res.astype(np.float64))[..., None])[..., 0]).astype(LD)
        return u

    out = {"lam_rel": lam_rel}
    if not solve_step:
        return out
    du = solve(-g)
    out["du"] = du.reshape(Bn, N, 6)
    out["dx"] = np.einsum("bsim,bm->bsi", Gf, du)
    if q2 is not None:
        q2 = np.swapaxes(np.asarray(q2, np.float64).astype(LD), 1, 2)
        du2 = solve(-(r.reshape(Bn, 6 * N) + np.einsum("bsim,bsi->bm", Gf, q2)))
        out["du2"], out["dx2"] = du2.reshape(Bn, N, 6), np.einsum("bsim,bm->bsi", Gf, du2)
    return out


def relerr(x, ref):
    """normwise relative error per instance (all stages)"""
    x, ref = np.asarray(x, LD).reshape(len(ref), -1), np.asarray(ref, LD).reshape(len(ref), -1)
    return (np.linalg.norm((x - ref).astype(np.float64), axis=1) / np.maximum(np.linalg.norm(ref.astype(np.float64), axis=1), 1e-300))


# ---------------------------------------------------------------------------------------------------------------------
# generated cases
# ---------------------------------------------------------------------------------------------------------------------
MARGIN = 1e-6      # a Lambda_k counts as clearly PD when every pivot d_j > MARGIN * |Lambda_k[j][j]|


def rel_pivot(ref):
    """smallest pivot relative to its diagonal entry, per instance (NaN-free: a failed stage gives -inf)"""
    with np.errstate(invalid="ignore", divide="ignore"):
        x = (ref["piv"] / np.abs(ref["lamd"])).astype(np.float64)
    return np.where(ref["ok"], np.nanmin(np.where(np.isnan(x), np.inf, x), axis=(-1, -2)), -np.inf)


def well_posed(seed, B, N, model, fold, neg=1.0, rd=None):
    """B instances whose every Lambda_k is PD with margin (redrawn until so); T cycles through TS, mu != dw, both nonzero."""
    rng = np.random.default_rng(seed)
    T = np.array([TS[i % 3] for i in range(B)])
    mu = rng.uniform(0.05, 0.5, B)
    dw = 10.0 ** rng.uniform(-4.0, -1.0, B)
    d = gen_lq(rng, B, N, model, neg, rd)
    for attempt in range(40):
        good = rel_pivot(riccati(stage_problem(d, T, mu, dw, fold))) > MARGIN
        if good.all():
            break
        nb = int((~good).sum())
        dn = gen_lq(rng, nb, N, model, neg * 0.6 ** (attempt + 1), rd)
        for k in d:
            d[k][~good] = dn[k]
    assert good.all(), "generator: no well-posed draw"
    q2 = rng.standard_normal((B, 8, N + 1))
    if model == 1:
        q2[:, 5:] = 0.0
    return dict(d=d, T=T, mu=mu, dw=dw, q2=q2)


def inertia_cases(seed, N, model, fold, mag=1e3):
    """Instances whose first non-PD Lambda_k is at k = N-1, a middle stage and k = 0, at control pivot 0 (v: the special
    column) or 5 (the last camera rate; the last gimbal rate of model 1 is pivot 2), and two with an exactly zero pivot.  Each gets a negative curvature placed in Q_{k+1}; expected: first failing stage, failing pivot."""
    base = well_posed(seed, 8, N, model, fold, rd=1e-3)
    d, exp = base["d"], []
    pv_last = 2 if model == 1 else 5
    q_last = 23 if model == 1 else 20      # LQ_Q entry of its state: (psi, psi) for model 1, (X7, X7) otherwise
    stages = sorted({N - 1, N // 2, 0})
    i = 0
    for k in stages:
        for pv in (0, pv_last):
            if i >= 7:
                break
            if pv == 0:         # Q_{k+1} strongly negative along d_k in (x, y, z)
                dd = d["DD"][i, :, k]
                for a in range(3):
                    for b in range(a + 1):
                        d["Q"][i, tri(a, b), k + 1] -= mag * dd[a] * dd[b]
            else:
                d["Q"][i, q_last, k + 1] -= mag
            exp.append((k, pv))
            i += 1
    # exactly zero pivots, d = 0.0 in every operation order: pivot 0 at k = N-1 (P_N zero in rows 0..2, RD_0 + dw = 0),
    # and pivot 5 at k = 0 (state 7 has no curvature at any stage, so Lambda_k is diagonal in it; RD_5 + dw = 0).  A zero
    # pivot that is not the last one is caught by the NaN it leaves in the next pivot, so only the second case tells
    # "d > 0" from "d >= 0".
    j = i
    for a in range(6):
        for b in range(a + 1):
            if a < 3 or b < 3:
                d["Q"][j, tri(a, b), N] = 0.0
    d["NN"][j, :, N] = 0.0
    d["DG"][j, 0, N] = 0.0
    base["dw"][j] = 0.5
    d["RD"][j, 0, N - 1] = -0.5
    exp.append((N - 1, 0))
    j += 1
    for b in range(6):
        d["Q"][j, tri(5, b)] = 0.0
    d["DG"][j, 4] = 0.0
    base["dw"][j] = 0.5
    d["RD"][j, 5, 0] = -0.5
    exp.append((0, 5))
    B = j + 1
    sub = {k: v[:B] for k, v in base.items() if k != "d"}
    sub["d"] = take(d, slice(0, B))
    return sub, exp


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference agrees with itself
# ---------------------------------------------------------------------------------------------------------------------
REF_CASES = [(1, 0, False), (2, 0, True), (5, 0, False), (15, 0, False), (15, 0, True), (15, 1, False), (30, 0, True),
             (31, 0, False)]


@pytest.mark.parametrize("N,model,fold", REF_CASES)
def test_reference_riccati_matches_condensed(N, model, fold):
    assert np.finfo(LD).nmant > 52, "np.longdouble must be wider than float64"
    c = well_posed(100 + N, 12, N, model, fold)
    pb = stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold)
    a = riccati(pb, c["q2"])
    b = condensed(pb, c["q2"])
    assert a["ok"].all() and (b["lam_rel"] > 0).all()
    for key in ("du", "dx", "du2", "dx2"):
        e = relerr(a[key], b[key])
        assert e.max() <= 1e-13, (key, e.max())
    # and the float64 recursion is a fair but imperfect baseline: close to (a), not equal
    f = riccati(stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold, np.float64), c["q2"])
    e64 = relerr(f["du"], a["du"])
    assert 0 < e64.max() <= 1e-6


@pytest.mark.parametrize("N,model,fold", REF_CASES)
def test_reference_inertia_matches_condensed_eigenvalue(N, model, fold):
    c, exp = inertia_cases(200 + N, N, model, fold)
    pb = stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold)
    a = riccati(pb)
    b = condensed(pb, solve_step=False)
    for i, (k, pv) in enumerate(exp):
        assert not a["ok"][i] and a["fail"][i] == k, (i, k, a["fail"][i])
        assert np.argmax(~(a["piv"][i, k] > 0)) == pv            # the first non-positive pivot
        if i >= len(exp) - 2:
            assert a["piv"][i, k, pv] == 0.0                          # the exactly singular cases
    # the verdict is the sign of the condensed Hessian's smallest eigenvalue wherever that is away from zero
    w = well_posed(300 + N, 12, N, model, fold)
    pw = stage_problem(w["d"], w["T"], w["mu"], w["dw"], fold)
    okw = riccati(pw)["ok"]
    lam = np.concatenate([b["lam_rel"], condensed(pw, solve_step=False)["lam_rel"]])
    ok = np.concatenate([a["ok"], okw])
    decided = np.abs(lam) > 1e-10
    assert decided.sum() >= len(lam) - 2          # only the exactly singular cases may sit at zero
    assert np.array_equal(ok[decided], lam[decided] > 0)


# ---------------------------------------------------------------------------------------------------------------------
# the harness
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def harness():
    if not HARNESS.exists():        # a tree that was never built: compile (nvcc cross-compiles without a GPU)
        subprocess.check_call(["make", "-C", str(CSRC), "-s", "libnmpc_ric_harness.so"])
    return C.CDLL(str(HARNESS))


def consts(lib, tag):
    buf = (C.c_longlong * 64)()
    n = getattr(lib, "ric_consts_" + tag)(buf)
    assert n == len(RIC_CONSTS)
    return dict(zip(RIC_CONSTS, buf[:n]))


def test_harness_builds_and_layouts(harness):
    """Every layout is in the harness with the shape the tests expect (no GPU needed)."""
    for tag, (N, nobs, model, fold) in LAYOUTS.items():
        c = consts(harness, tag)
        assert (c["N"], c["S"], c["MODEL"]) == (N, N + 1, model)
        if fold is not None:
            assert bool(c["FOLD"]) == fold
        assert c["LQ_NE"] == (c["LQ_DG"] if c["FOLD"] else c["LQ_QB"] + 8)
        assert c["LV0"] < c["RW0"] <= c["LQ0"] < c["STG0"] < c["OBS0"] < c["ALG0"] < c["RES0"] < c["PAR0"] < c["TOTAL"]
        assert c["SOC_Q2"] + 8 * c["S"] <= c["LQ0"] + c["LQ_DEAD"] * c["S"]
    # the production FOLD choice at the default tuning: the long horizons fold
    assert [consts(harness, t)["FOLD"] for t in ("p15_3", "p5_3", "p30_10")] == [0, 0, 1]


def pack_lq(c, d):
    Bn, S = d["QA"].shape[0], c["S"]
    lq = np.zeros((Bn, c["LQ_NE"], S))
    for e, n in ENT.items():
        off = c["LQ_" + e]
        if off + n <= c["LQ_NE"]:
            lq[:, off:off + n] = d[e]
    lq[:, c["LQ_ZERO"]] = 0.0
    return lq


def poison(c):
    """shared slice: NaN over the staging area, LV_DX / LV_DU and the dead LQ entries, distinct finite values elsewhere"""
    S = c["S"]
    p = -1.0e6 - np.arange(c["TOTAL"], dtype=np.float64)
    p[c["STG0"]:c["STG0"] + c["STG_N"]] = np.nan
    p[c["LV0"] + c["LV_DX"] * S:c["LV0"] + (c["LV_DU"] + 6) * S] = np.nan
    p[c["LQ0"]:c["LQ0"] + c["LQ_DEAD"] * S] = np.nan
    return p


class Run:
    pass


def run(lib, tag, case, seq=None, soc=True):
    """One launch.  seq [B, n, 2] of (mu, dw) (default: the case's one pair)."""
    import torch
    c = consts(lib, tag)
    S, dev = c["S"], torch.device("cuda", 0)
    d = case["d"]
    Bn = d["QA"].shape[0]
    if seq is None:
        seq = np.stack([case["mu"], case["dw"]], axis=1)[:, None, :]
    t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
    T, lq, sq = t(case["T"]), t(pack_lq(c, d)), t(seq)
    q2 = t(case["q2"]) if soc else None
    pz, rpz = t(poison(c)), t(np.full(c["RIC_N"], np.nan))
    mp = torch.zeros(c["RIC_MAP_WORDS"] * 32, dtype=torch.int32, device=dev)
    ok = torch.full((Bn, seq.shape[1]), -1, dtype=torch.int32, device=dev)
    sl = torch.zeros((Bn, 2, c["TOTAL"]), dtype=torch.float64, device=dev)
    ric = torch.zeros((Bn, S, c["RIC_N"]), dtype=torch.float64, device=dev)
    vp = C.c_void_p
    fn = getattr(lib, "ric_run_" + tag)
    fn.argtypes = [C.c_int, vp, vp, vp, C.c_int, vp] + [vp] * 7
    rc = fn(Bn, T.data_ptr(), lq.data_ptr(), sq.data_ptr(), seq.shape[1], q2.data_ptr() if soc else None, pz.data_ptr(),
            rpz.data_ptr(), mp.data_ptr(), ok.data_ptr(), sl.data_ptr(), ric.data_ptr(), vp(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    r = Run()
    r.c, r.ok, r.sl, r.ric = c, ok.cpu().numpy(), sl.cpu().numpy(), ric.cpu().numpy()
    r.lq, r.poison = pack_lq(c, d), poison(c)
    lv = lambda s, e, n: s[:, c["LV0"] + e * S:c["LV0"] + (e + n) * S].reshape(Bn, n, S).transpose(0, 2, 1)
    r.dx, r.du = lv(r.sl[:, 0], c["LV_DX"], 8), lv(r.sl[:, 0], c["LV_DU"], 6)
    r.dx2 = lv(r.sl[:, 1], c["LV_DX"], 8)
    r.du2 = r.sl[:, 1, c["SOC_DUS"]:c["SOC_DUS"] + 6 * S].reshape(Bn, 6, S).transpose(0, 2, 1)
    N = c["N"]
    kk = r.ric[:, :N, c["RIC_K"]:c["RIC_K"] + 54].reshape(Bn, N, 6, 9)
    r.K, r.kap = kk[..., :8], kk[..., 8]
    r.Lp, r.idg = r.ric[:, :N, c["RIC_L"]:c["RIC_L"] + 21], r.ric[:, :N, c["RIC_L"] + 21:c["RIC_L"] + 27]
    r.kap2 = r.ric[:, :N, c["RIC_K2"]:c["RIC_K2"] + 6]
    return r


def bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def case_for(lib, tag, seed, B=48, **kw):
    N, _, model, _ = LAYOUTS[tag]
    return well_posed(seed, B, N, model, fold_of(lib, tag), **kw)


def fold_of(lib, tag):
    return bool(consts(lib, tag)["FOLD"])


def packed(Lc):
    idx = [(i, j) for i in range(6) for j in range(i + 1)]
    return np.stack([Lc[..., i, j] for i, j in idx], axis=-1)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
TAGS = list(LAYOUTS)
# kernel error <= C_CAL x (error of the float64 textbook recursion) + FLOOR, per instance.  Measured on a B200: the
# kernel's error is at most 2.7x the float64 recursion's (or the floor) on every layout.
C_CAL = 32.0
FLOOR = 64.0 * EPS


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_step_accuracy(harness, tag):
    """du, dx and the SOC du, dx against the longdouble reference, relative to what a float64 recursion achieves"""
    c = case_for(harness, tag, 1000 + TAGS.index(tag))
    fold = fold_of(harness, tag)
    r = run(harness, tag, c)
    assert (r.ok == 1).all()
    ref = riccati(stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold), c["q2"])
    f64 = riccati(stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold, np.float64), c["q2"])
    for key in ("du", "dx", "du2", "dx2"):
        ek, e64 = relerr(getattr(r, key)[:, :ref[key].shape[1]], ref[key]), relerr(f64[key], ref[key])
        ratio = ek / np.maximum(e64, FLOOR)
        print(f"\n[{tag}] {key}: max err kernel {ek.max():.3g}, float64 recursion {e64.max():.3g}; "
              f"max kernel / max(float64, floor) {ratio.max():.3g}")
        assert (ek <= C_CAL * e64 + FLOOR).all(), (key, ek.max(), e64.max(), ratio.max())


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_step_accuracy_well_conditioned(harness, tag):
    """an absolute bound where the problem is well conditioned (RD = 1, mild curvature); measured on a B200: <= 4e-15"""
    c = case_for(harness, tag, 2000 + TAGS.index(tag), neg=0.2, rd=1.0)
    fold = fold_of(harness, tag)
    r = run(harness, tag, c)
    assert (r.ok == 1).all()
    ref = riccati(stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold), c["q2"])
    for key in ("du", "dx", "du2", "dx2"):
        e = relerr(getattr(r, key)[:, :ref[key].shape[1]], ref[key])
        print(f"\n[{tag}] {key}: max rel err {e.max():.3g}")
        assert e.max() <= 1e-13, (key, e.max())


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_factors(harness, tag):
    """K, kappa, chol Lambda, 1/diag and kappa_soc at every stage"""
    c = case_for(harness, tag, 3000 + TAGS.index(tag), neg=0.2, rd=1.0)
    fold = fold_of(harness, tag)
    r = run(harness, tag, c)
    assert (r.ok == 1).all()
    ref = riccati(stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold), c["q2"])
    N = r.c["N"]
    Lref = packed(ref["Lc"])
    idg_ref = 1.0 / np.diagonal(ref["Lc"], axis1=-2, axis2=-1)
    for name, x, xr in (("K", r.K, ref["K"]), ("kappa", r.kap, ref["kap"]), ("L", r.Lp, Lref), ("1/diag", r.idg, idg_ref),
                        ("kappa_soc", r.kap2, ref["kap2"])):
        for k in range(N):
            e = relerr(x[:, k], xr[:, k])
            assert e.max() <= 1e-12, (name, k, e.max())
    dg = r.Lp[..., [tri(j, j) for j in range(6)]]
    assert np.abs(dg * r.idg - 1.0).max() <= 4 * EPS


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_inertia_verdict(harness, tag):
    """first non-PD Lambda_k at k = N-1, a middle stage and k = 0, at pivot 0 and the last pivot, and exactly zero pivots"""
    N, _, model, _ = LAYOUTS[tag]
    fold = fold_of(harness, tag)
    c, exp = inertia_cases(4000 + TAGS.index(tag), N, model, fold)
    ref = riccati(stage_problem(c["d"], c["T"], c["mu"], c["dw"], fold))
    assert [int(f) for f in ref["fail"]] == [k for k, _ in exp]
    good = well_posed(4100 + TAGS.index(tag), 4, N, model, fold)
    allc = {k: np.concatenate([c[k], good[k]]) for k in ("T", "mu", "dw", "q2")}
    allc["d"] = join(c["d"], good["d"])
    r = run(harness, tag, allc, soc=False)
    assert r.ok[:, 0].tolist() == [0] * len(exp) + [1] * 4


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_retry_hygiene(harness, tag):
    """(mu, 0) fails, then (mu, dw) on the same shared memory: bit-identical to a fresh (mu, dw)"""
    N, _, model, _ = LAYOUTS[tag]
    fold = fold_of(harness, tag)
    c, exp = inertia_cases(5000 + TAGS.index(tag), N, model, fold, mag=10.0)
    n = len(exp) - 2           # not the singular cases: a moderate negative curvature that dw = 1e3 repairs
    c = {k: (v[:n] if k != "d" else take(v, slice(0, n))) for k, v in c.items()}
    dw = np.full(n, 1e3)
    ref0 = riccati(stage_problem(c["d"], c["T"], c["mu"], np.zeros(n), fold))
    ref1 = riccati(stage_problem(c["d"], c["T"], c["mu"], dw, fold))
    assert not ref0["ok"].any() and ref1["ok"].all()
    seq2 = np.stack([np.stack([c["mu"], np.zeros(n)], 1), np.stack([c["mu"], dw], 1)], 1)
    seq1 = seq2[:, 1:]
    a = run(harness, tag, c, seq=seq2)
    b = run(harness, tag, c, seq=seq1)
    assert a.ok.tolist() == [[0, 1]] * n and b.ok.tolist() == [[1]] * n
    assert np.array_equal(bits(a.sl), bits(b.sl)) and np.array_equal(bits(a.ric), bits(b.ric))


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_no_stale_reads_no_stray_writes(harness, tag):
    """no poison reaches an output; outside the staging area, LV_DX / LV_DU and the dead LQ entries nothing changes;
    the ric rows past the last stage and the unused last slot of every row keep their poison"""
    c = case_for(harness, tag, 6000 + TAGS.index(tag), B=16)
    r = run(harness, tag, c)
    assert (r.ok == 1).all()
    N, S, k = r.c["N"], r.c["S"], r.c
    for name in ("dx", "du", "dx2", "du2", "K", "kap", "Lp", "idg", "kap2"):
        assert np.isfinite(getattr(r, name)).all(), name
    init = r.poison.copy()[None].repeat(len(r.lq), 0)
    init[:, k["LQ0"]:k["LQ0"] + k["LQ_NE"] * S] = r.lq.reshape(len(r.lq), -1)
    free = np.zeros(k["TOTAL"], bool)
    free[k["STG0"]:k["STG0"] + k["STG_N"]] = True
    free[k["LV0"] + k["LV_DX"] * S:k["LV0"] + (k["LV_DU"] + 6) * S] = True
    free[k["LQ0"]:k["LQ0"] + k["LQ_DEAD"] * S] = True
    for snap in range(2):
        same = bits(r.sl[:, snap]) == bits(init)
        assert same[:, ~free].all(), np.nonzero(~same[:, ~free].all(0))[0][:10]
    rp = bits(np.full(k["RIC_N"], np.nan))
    assert (bits(r.ric[:, N:]) == rp).all()
    used = k["RIC_K2"] + 6
    assert (bits(r.ric[:, :N, used:]) == rp[used:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("tag", TAGS)
def test_instances_independent(harness, tag):
    """the same instance at different rows of a batch gives bit-identical outputs"""
    c = case_for(harness, tag, 7000 + TAGS.index(tag), B=12)
    rows = [0, 5, 11]
    for i in rows[1:]:
        for key in ("T", "mu", "dw", "q2"):
            c[key][i] = c[key][0]
        for e in c["d"]:
            c["d"][e][i] = c["d"][e][0]
    r = run(harness, tag, c)
    for i in rows[1:]:
        assert np.array_equal(bits(r.sl[i]), bits(r.sl[0])) and np.array_equal(bits(r.ric[i]), bits(r.ric[0]))


@pytest.mark.gpu
def test_model1_absent_controls(harness):
    tag = "p15_0_1"
    c = case_for(harness, tag, 8000)
    r = run(harness, tag, c)
    assert (r.ok == 1).all()
    for x in (r.du, r.du2):
        assert (x[:, :, 3:] == 0.0).all()
    assert (r.K[:, :, 3:] == 0.0).all() and (r.kap[:, :, 3:] == 0.0).all() and (r.kap2[:, :, 3:] == 0.0).all()
