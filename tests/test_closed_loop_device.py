"""GPU: the target prediction (NMPC_PREDICT_TARGET) and the obstacle motion (nmpc_set_obstacle_motion) inside the fused closed-loop
step -- bit-identical to the host computations they replace (ClosedLoop.target_prediction(), the torch obstacle update), the
same in the free-running loop, and refused where they cannot apply."""
import numpy as np
import pytest
import torch


def _scenario(pkg, name, N):
    sc = pkg.SCENARIOS[name]
    return sc if N == sc.N else sc.with_horizon(N)


def _target_kw(B, sched, vw):
    return dict(phase=np.random.default_rng(3).integers(0, 400, B)) if sched else dict(target_vw=vw)


def _moving_field(sc, B, seed):
    """Per-instance obstacle fields [B, n_obs, 3] near the scenario's table and their velocities [B, n_obs, 2]."""
    rng = np.random.default_rng(seed)
    obs = np.tile(sc.obstacle_table(), (B, 1, 1))
    obs[:, :, :2] += rng.uniform(-2.0, 2.0, (B, sc.n_obs, 2))
    return obs, rng.uniform(-3.0, 3.0, (B, sc.n_obs, 2))


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,sched", [("nmpc_tt", 15, False), ("t_trajectory", 15, True), ("gimbal_less", 15, False),
                                          ("race_track_2", 30, False)])
def test_device_prediction_is_the_host_prediction(pkg, name, N, sched):
    """A fused step with NMPC_PREDICT_TARGET against solve_and_step(target_traj=ClosedLoop.target_prediction()) on the same batch:
    the same bits everywhere (p, warm start, FOV centre, error sum, solution, objective, status, iterations), step after step."""
    from mpc_implementation_b200.closed_loop import ClosedLoop
    sc = _scenario(pkg, name, N)
    B = 257
    p0, vw = pkg.random_instances(sc, B, seed=23)
    kw = _target_kw(B, sched, vw)
    dev = ClosedLoop(pkg.nlpsol("d", "ipm", sc, max_batch=B), sc, p0, predict_target=True, **kw)
    host = ClosedLoop(pkg.nlpsol("h", "ipm", sc, max_batch=B), sc, p0, **kw)
    for k in range(3):
        a = dev.step(want_x=True)
        sa = dev.solver.stats()
        host._schedule_vw()
        traj = host.target_prediction()
        b = host.solver.solve_and_step(host.p, host.u_warm, host.lbx, host.ubx, host.lbg, host.ubg,
                                       host.vw if host._const_vw else None, host.fov, host.err_sum, want_x=True, target_traj=traj)
        host.mpc_iter += 1
        sb = host.solver.stats()
        torch.cuda.synchronize()
        assert torch.equal(a["x"], b["x"]) and torch.equal(a["f"], b["f"]), k
        assert torch.equal(sa["return_status"], sb["return_status"]) and torch.equal(sa["iter_count"], sb["iter_count"]), k
        assert torch.equal(dev.p, host.p) and torch.equal(dev.u_warm, host.u_warm), k
        assert torch.equal(dev.fov, host.fov) and torch.equal(dev.err_sum, host.err_sum), k
    assert int((sa["return_status"] == 0).sum()) >= B // 2
    # the prediction is not the frozen target: the problem changed
    frozen = ClosedLoop(pkg.nlpsol("f", "ipm", sc, max_batch=B), sc, p0, **kw)
    c = frozen.step(want_x=True)
    first = ClosedLoop(pkg.nlpsol("g", "ipm", sc, max_batch=B), sc, p0, predict_target=True, **kw).step(want_x=True)
    assert not torch.equal(c["f"], first["f"])


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,B,K,sched,moving", [("t_trajectory", 15, 200, 6, True, True), ("10_obstacles", 15, 96, 5, False, True),
                                                     ("race_track_2", 30, 64, 4, False, True), ("gimbal_less", 15, 150, 6, False, False)])
def test_free_running_loop_predicts_and_moves(pkg, name, N, B, K, sched, moving):
    """ClosedLoop(predict_target=True, obstacles=, obstacle_vel=): K step() calls and run_free(K) give the same bits -- states, warm
    starts, error sums, FOV centres, the obstacle fields and the status / iteration count of every solve."""
    from mpc_implementation_b200.closed_loop import ClosedLoop
    sc = _scenario(pkg, name, N)
    p0, vw = pkg.random_instances(sc, B, seed=31)
    kw = _target_kw(B, sched, vw)
    if moving:
        obs, vel = _moving_field(sc, B, seed=5)
        kw.update(obstacles=obs, obstacle_vel=vel)
    a = ClosedLoop(pkg.nlpsol("a", "ipm", sc, max_batch=B), sc, p0, predict_target=True, **kw)
    b = ClosedLoop(pkg.nlpsol("b", "ipm", sc, max_batch=B), sc, p0, predict_target=True, **kw)
    st, it = [], []
    for _ in range(K):
        a.step(); s = a.solver.stats()
        st.append(s["return_status"].clone()); it.append(s["iter_count"].clone())
    out = b.run_free(K)
    torch.cuda.synchronize()
    assert torch.equal(a.p, b.p) and torch.equal(a.u_warm, b.u_warm) and torch.equal(a.err_sum, b.err_sum) and torch.equal(a.fov, b.fov)
    assert torch.equal(torch.stack(st), out["status_log"]) and torch.equal(torch.stack(it), out["iters_log"])
    if moving:
        assert torch.equal(a.obstacles, b.obstacles)
        moved = torch.as_tensor(obs, device=a.obstacles.device)
        for _ in range(K):
            moved[:, :, :2] += sc.T * torch.as_tensor(vel, device=moved.device)
        assert torch.equal(a.obstacles, moved)          # the torch update of the same field, K times
    assert int((torch.stack(st) == 0).sum()) >= K * B // 2
    a.step(); b.step(); torch.cuda.synchronize()        # and the two loops stay interchangeable afterwards
    assert torch.equal(a.p, b.p) and torch.equal(a.u_warm, b.u_warm)
    if moving:
        assert torch.equal(a.obstacles, b.obstacles)


@pytest.mark.gpu
@pytest.mark.parametrize("name,predict", [("10_obstacles", False), ("t_trajectory", True)])
def test_fused_motion_is_the_unfused_loop(pkg, name, predict):
    """Moving obstacles in the fused step against the unfused path (solve with g, nmpc_step, the torch update of the field) over
    K steps: obstacle fields and states are the same bits."""
    from mpc_implementation_b200.closed_loop import ClosedLoop
    sc = pkg.SCENARIOS[name]
    B, K = 128, 8
    p0, vw = pkg.random_instances(sc, B, seed=47)
    obs, vel = _moving_field(sc, B, seed=9)
    kw = dict(target_vw=vw, obstacles=obs, obstacle_vel=vel, predict_target=predict)
    fused = ClosedLoop(pkg.nlpsol("a", "ipm", sc, max_batch=B), sc, p0, **kw)
    unfused = ClosedLoop(pkg.nlpsol("b", "ipm", sc, max_batch=B), sc, p0, **kw)
    for k in range(K):
        fused.step()
        unfused.step(want_g=True)
        torch.cuda.synchronize()
        assert torch.equal(fused.obstacles, unfused.obstacles), k
        assert torch.equal(fused.p, unfused.p) and torch.equal(fused.u_warm, unfused.u_warm) and torch.equal(fused.err_sum, unfused.err_sum), k


@pytest.mark.gpu
def test_refusals(pkg):
    """The C ABI refuses what it cannot do, with a message; nlpsol refuses the same with ValueError before any launch."""
    sc = pkg.SCENARIOS["nmpc_tt"]
    B = 4
    s = pkg.nlpsol("s", "ipm", sc, max_batch=B)
    L, ffi = pkg._ffi.lib(), pkg._ffi
    dev = "cuda:0"
    p0, vw = pkg.random_instances(sc, B, seed=2)
    t = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev).contiguous()
    p, u, vwt = t(p0), torch.zeros((B, sc.n_w), dtype=torch.float64, device=dev), t(vw)
    lbx, ubx, lbg, ubg = (t(a) for a in sc.bounds())
    obs, vel = (t(a) for a in _moving_field(sc, B, seed=1))
    other = obs.clone()
    shared = t(sc.obstacle_table())
    x, f = torch.empty((B, sc.n_w), dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.float64, device=dev)
    st, it = torch.empty(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    P = lambda a: a.data_ptr()
    per, pred = ffi.NMPC_OBS_PER_INSTANCE, ffi.NMPC_PREDICT_TARGET

    def solve(flags, ob=obs):
        return L.nmpc_solve(s._h, B, P(p), P(u), P(lbx), P(ubx), P(lbg), P(ubg), P(ob), flags, P(x), P(f), None, None, None, P(st), P(it), stream)

    def solve_and_step(flags, ob=obs):
        return L.nmpc_solve_and_step(s._h, B, P(p), P(u), P(lbx), P(ubx), P(lbg), P(ubg), P(ob), flags, P(vwt), None, P(f), None, None,
                                     P(st), P(it), stream)

    def err():
        return L.nmpc_last_error().decode()

    # the flag on a call that has no (v, omega)
    assert solve(per | pred) != 0 and "NMPC_PREDICT_TARGET" in err()
    assert L.nmpc_eval(s._h, B, P(x), P(p), P(obs), per | pred, 1.0, None, None, P(f), None, None, None, None, stream) != 0
    assert "NMPC_PREDICT_TARGET" in err()
    # the flag together with a caller-given trajectory
    traj = torch.zeros((B, sc.N, 2), dtype=torch.float64, device=dev)
    ffi.check(L.nmpc_set_target_trajectory(s._h, P(traj)), "nmpc_set_target_trajectory")
    assert solve_and_step(per | pred) != 0 and "nmpc_set_target_trajectory" in err()
    ffi.check(L.nmpc_set_target_trajectory(s._h, None), "nmpc_set_target_trajectory")
    # motion with another obstacle field than the registered one, and with a shared table while B > 1
    ffi.check(L.nmpc_set_obstacle_motion(s._h, P(obs), P(vel)), "nmpc_set_obstacle_motion")
    assert solve_and_step(per, other) != 0 and "registered" in err()
    ffi.check(L.nmpc_set_obstacle_motion(s._h, P(shared), P(vel)), "nmpc_set_obstacle_motion")
    assert solve_and_step(0, shared) != 0 and "per-instance" in err()
    assert L.nmpc_set_obstacle_motion(s._h, P(obs), None) != 0 and "neither" in err()
    ffi.check(L.nmpc_set_obstacle_motion(s._h, None, None), "nmpc_set_obstacle_motion")
    # nothing of the refused calls ran: a plain call still works and leaves the field where it was
    before = obs.clone()
    ffi.check(solve_and_step(per | pred), "nmpc_solve_and_step")
    torch.cuda.synchronize()
    assert torch.equal(obs, before) and bool((st >= 0).all())

    # the Python layer
    p, u = t(p0), torch.zeros((B, sc.n_w), dtype=torch.float64, device=dev)
    with pytest.raises(ValueError, match="exclude"):
        s.solve_and_step(p, u, *sc.bounds(), vwt, predict_target=True, target_traj=traj)
    with pytest.raises(ValueError, match="obstacle_vel"):
        s.solve_and_step(p, u, *sc.bounds(), vwt, obstacles=obs, obstacle_vel=vel[:, :, :1].contiguous())
    with pytest.raises(ValueError, match="CUDA float64"):
        s.run_closed_loop(2, p, u, *sc.bounds(), vwt, obstacles=shared, obstacle_vel=vel)
    gl = pkg.SCENARIOS["gimbal_less"]
    with pytest.raises(ValueError, match="no obstacle rows"):
        pkg.nlpsol("g", "ipm", gl, max_batch=B).solve_and_step(t(pkg.random_instances(gl, B, 1)[0]), torch.zeros((B, gl.n_w), dtype=torch.float64, device=dev),
                                                                *gl.bounds(), vwt, obstacle_vel=vel)
    # a bound vector with extra entries, an obstacle tensor with three entries more than [B, n_obs, 3]: every device path
    bounds = list(sc.bounds())
    too_long = [np.concatenate([bounds[0], bounds[0][:2]])] + bounds[1:]
    big = torch.cat([obs.reshape(-1), obs.reshape(-1)[:3]])
    for bnd, ob in ((too_long, None), (bounds, big)):
        with pytest.raises(ValueError, match="bound vector|obstacles must be"):
            s.solve_and_step(p, u, *bnd, vwt, obstacles=ob)
        with pytest.raises(ValueError, match="bound vector|obstacles must be"):
            s.run_closed_loop(2, p, u, *bnd, vwt, obstacles=ob)
        with pytest.raises(ValueError, match="bound vector|obstacles must be"):
            s(x0=u, p=p, lbx=bnd[0], ubx=bnd[1], lbg=bnd[2], ubg=bnd[3], obstacles=ob)
    torch.cuda.synchronize()
    assert torch.equal(p, t(p0))          # none of them launched


@pytest.mark.gpu
def test_device_call_keeps_the_handle(pkg):
    """max_batch sizes the staging buffers of the host path only: a device-tensor call with more instances and weights= keeps the
    handle, and with it the schedule set before."""
    sc = pkg.SCENARIOS["t_trajectory"]
    B = 4
    s = pkg.nlpsol("s", "ipm", sc, max_batch=1)
    s.set_schedule(np.array([[sc.schedule(k) for k in range(sc.steps)]]))
    p = torch.as_tensor(pkg.random_instances(sc, B, seed=6)[0], dtype=torch.float64, device="cuda:0").contiguous()
    u = torch.zeros((B, sc.n_w), dtype=torch.float64, device="cuda:0")
    s(x0=u, p=p, lbx=sc.bounds()[0], ubx=sc.bounds()[1], lbg=sc.bounds()[2], ubg=sc.bounds()[3], weights=np.tile([sc.w1, sc.w2], (B, 1)))
    s.solve_and_step(p, u, *sc.bounds(), None)
    torch.cuda.synchronize()
    assert bool((s.stats()["return_status"] >= 0).all())
