"""The differentiable solve on the B200: the VJP kernel against the dense restatement (tests/vjp_oracle.py)
at every lane width in modes 3, 6, 7 and 8, the forward of plan_batch_differentiable against plan_batch,
torch.autograd.gradcheck, recovery of w_pos and w_vel from demonstrated plans, and the refusals on the
device."""
import ctypes as C

import numpy as np
import pytest

import vjp_oracle
from test_rollout_mode import _inputs
from test_vjp import MARGIN, W, _params, _rel, check_refusals

pytestmark = pytest.mark.gpu

B_KERNEL = 4096


def _spheres(p0):
    """spheres on the paths of the first starts (contacts with h > 0) and one out of reach"""
    return np.array([[*(p0[0] + [0.5, 0.0, 0.3]), 1.0], [*(p0[1] - [0.2, 0.4, 0.0]), 1.5],
                     [*(p0[2] + [0.0, 0.0, -0.5]), 2.0], [50.0, 50.0, 50.0, 1.0]])


def _case(mode, N, seed):
    """B_KERNEL problems of the benchmark's start distribution; every sixteenth has a far goal (or a far
    reference), which pins T_z at max_thrust and the lateral thrust at tilt_thrust"""
    rng = np.random.default_rng(seed)
    p0, v0, goal, hg = _inputs(B_KERNEL, seed)
    goal[5::16] = p0[5::16] + [80.0, -60.0, 120.0]
    r = u = s = None
    if mode in (7, 8):
        r = goal[:, None] + rng.normal(0, 0.6, (B_KERNEL, N, 3)).cumsum(1)
        u = rng.normal(0, 2, (B_KERNEL, N, 3))
    if mode in (6, 8):
        s = _spheres(p0)
    return p0, v0, goal, hg, r, u, s


def run_vjp(params, x, p0, v0, goal, hg, r, u, s, gx, gc):
    """dart_se3mpc_solve_vjp_batch on device copies of batch-first host arrays; returns host arrays"""
    import torch
    from dart_planner_b200 import _cabi
    B, N = len(p0), int(params.horizon)
    d = lambda a: torch.as_tensor(np.ascontiguousarray(np.asarray(a, np.float64).reshape(B, -1).T)).cuda()  # noqa: E731
    ins = [d(p0), d(v0), d(goal), d(x), d(gx), torch.as_tensor(gc, dtype=torch.float64).cuda()]
    hgd = torch.as_tensor(np.asarray(hg, np.uint8)).cuda()
    ref = rows = sph = lst = None
    if r is not None:
        rows = torch.cat([d(r), d(u)])
        ref = _cabi.TrackRef(N, 0, rows.data_ptr())
    if s is not None:
        lst = torch.as_tensor(np.ascontiguousarray(s, np.float64)).cuda()
        sph = _cabi.Spheres(len(s), 0, lst.data_ptr(), MARGIN)
    out = {k: torch.full((n, B), 7.0, dtype=torch.float64, device="cuda")
           for k, n in (("gp0", 3), ("gv0", 3), ("ggoal", 3), ("gref", 6 * N), ("gw", 4))}
    st = torch.full((B,), -9, dtype=torch.int32, device="cuda")
    rc = _cabi.lib().dart_se3mpc_solve_vjp_batch(
        C.byref(params), B, B, *(t.data_ptr() for t in ins[:3]), hgd.data_ptr(), ins[3].data_ptr(),
        None if ref is None else C.byref(ref), None if sph is None else C.byref(sph), ins[4].data_ptr(),
        ins[5].data_ptr(), *(out[k].data_ptr() for k in ("gp0", "gv0", "ggoal", "gref", "gw")), st.data_ptr(), None)
    _cabi.check(rc, "dart_se3mpc_solve_vjp_batch")
    torch.cuda.synchronize()
    res = {k: v.cpu().numpy().T for k, v in out.items()}
    res["status"] = st.cpu().numpy()
    return res


@pytest.mark.parametrize("N", [1, 4, 6, 8, 13, 16])
@pytest.mark.parametrize("mode", [3, 6, 7, 8])
def test_kernel_matches_restatement(mode, N):
    import dart_planner_b200 as dp
    from dart_planner_b200.config import SE3MPCConfig
    p0, v0, goal, hg, r, u, s = _case(mode, N, 17 * N + mode)
    cfg = SE3MPCConfig(prediction_horizon=N, dt=0.1, obstacle_weight=W)
    sol = dp.plan_batch(p0, v0, None if r is not None else goal, cfg, dynamics_consistent=True, has_goal=hg,
                        reference=None if r is None else (r, u), spheres=None if s is None else (s[:, :3], s[:, 3]),
                        sphere_margin=MARGIN, to_host=True)
    x = sol.x
    params = _params(mode, N)
    T = x[:, 6 * N:]
    pr0 = vjp_oracle.Problems(params, p0, v0, goal)
    if N > 1:                                                        # at N = 1, T_0 enters no state
        assert pr0.active(T)[5::16].sum() >= 2 * len(T[5::16])      # the saturated cases reach the bounds
    rng = np.random.default_rng(N + mode)
    gx, gc = rng.normal(size=(B_KERNEL, 9 * N)), rng.normal(size=B_KERNEL)
    got = run_vjp(params, x, p0, v0, goal, hg, None if r is None else r.reshape(B_KERNEL, -1),
                  None if u is None else u.reshape(B_KERNEL, -1), s, gx, gc)
    want = {}
    for lo in range(0, B_KERNEL, 512):
        sl = slice(lo, lo + 512)
        pr = vjp_oracle.Problems(params, p0[sl], v0[sl], goal=None if r is not None else goal[sl],
                                 r=None if r is None else r[sl].reshape(-1, 3 * N),
                                 u=None if u is None else u[sl].reshape(-1, 3 * N), has_goal=hg[sl], spheres=s,
                                 weight=W, margin=MARGIN)
        for k, v in pr.vjp(T[sl], gx[sl], gc[sl]).items():
            want.setdefault(k, []).append(v)
    want = {k: np.concatenate(v) for k, v in want.items()}
    assert (got["status"] == want["status"]).all()
    ok = want["status"] == 0
    assert ok.mean() > 0.95, np.bincount(want["status"])            # sphere contacts can make H_FF indefinite
    keys = ("gp0", "gv0", "gw") + (("gref",) if r is not None else ("ggoal",))
    for k in keys:
        assert _rel(got[k][ok], want[k][ok]) <= 1e-10, k
        assert np.isnan(got[k][~ok]).all(), k
    untouched = "ggoal" if r is not None else "gref"
    assert (got[untouched] == 7.0).all()                                # the other target's output is not written


@pytest.mark.parametrize("mode", [3, 6, 7, 8])
def test_forward_is_plan_batch(mode):
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.config import SE3MPCConfig
    N = 8
    p0, v0, goal, hg, r, u, s = _case(mode, N, 3)
    cfg = SE3MPCConfig(prediction_horizon=N, dt=0.1, obstacle_weight=W, position_weight=80.0, velocity_weight=12.0)
    kw = dict(has_goal=hg, reference=None if r is None else (r, u),
              spheres=None if s is None else (s[:, :3], s[:, 3]), sphere_margin=MARGIN)
    g = None if r is not None else goal
    sol = dp.plan_batch(p0, v0, g, cfg, dynamics_consistent=True, **kw)
    w = torch.tensor([80.0, 12.0, 1.0, 0.1], dtype=torch.float64, requires_grad=True)
    x, cost = dp.plan_batch_differentiable(torch.as_tensor(p0).requires_grad_(), v0, g,
                                           SE3MPCConfig(prediction_horizon=N, dt=0.1, obstacle_weight=W),
                                           weights=w, **kw)
    assert torch.equal(x, sol.x) and torch.equal(cost, sol.cost)
    (x.square().sum() + cost.sum()).backward()
    assert w.grad is not None
    if mode in (3, 7):                     # with spheres, a problem whose H_FF is indefinite gives NaN
        assert torch.isfinite(w.grad).all()


@pytest.mark.parametrize("mode", [7, 8])
def test_goals_beside_a_reference_get_a_zero_gradient(mode):
    """With a reference the goals are not read, so their gradient is exactly zero -- not whatever the
    allocator last held."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.config import SE3MPCConfig
    N = 8
    p0, v0, goal, hg, r, u, s = _case(mode, N, 5)
    cfg = SE3MPCConfig(prediction_horizon=N, dt=0.1, obstacle_weight=W)
    junk = torch.full((4 * B_KERNEL * 3,), 3.5e7, dtype=torch.float64, device="cuda")   # recycled memory
    del junk
    g = torch.tensor(goal, dtype=torch.float64, device="cuda", requires_grad=True)
    P = torch.tensor(r, dtype=torch.float64, device="cuda", requires_grad=True)
    x, cost = dp.plan_batch_differentiable(p0, v0, g, cfg, reference=(P, u), has_goal=hg,
                                           spheres=None if s is None else (s[:, :3], s[:, 3]), sphere_margin=MARGIN)
    (x.sum() + cost.sum()).backward()
    assert g.grad is not None and (g.grad == 0).all()
    assert P.grad is not None and (torch.isfinite(P.grad).all(1).all(1).sum() > 0.95 * B_KERNEL)


def _grad_problems(N, B=8, seed=4):
    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-2, 2, (B, 3))
    v0 = rng.uniform(-0.5, 0.5, (B, 3))
    goal = p0 + rng.uniform(-1.0, 1.0, (B, 3))
    return p0, v0, goal


@pytest.mark.parametrize("mode", [3, 7])
def test_gradcheck(mode):
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.config import SE3MPCConfig
    N = 8
    # tolerance 0: the solve runs until its line search can no longer reduce f, about 3e-5 from the exact
    # plan on these problems (the oracle's driver), so differences of 1e-2 are accurate to about 1e-4
    cfg = SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=0.0, max_iterations=200)
    p0, v0, goal = _grad_problems(N)
    t = lambda a: torch.tensor(a, dtype=torch.float64, device="cuda", requires_grad=True)  # noqa: E731
    wp, wv = t(100.0), t(10.0)
    const = torch.tensor([1.0, 0.1], dtype=torch.float64, device="cuda")
    if mode == 3:
        def fn(p, v, g, a, b):
            return dp.plan_batch_differentiable(p, v, g, cfg, weights=torch.cat([a[None], b[None], const]))
        inputs = (t(p0), t(v0), t(goal), wp, wv)
    else:
        rng = np.random.default_rng(9)
        P = goal[:, None] + rng.normal(0, 0.3, (8, N, 3))
        V = rng.normal(0, 0.5, (8, N, 3))

        def fn(p, v, rp, rv, a, b):
            return dp.plan_batch_differentiable(p, v, None, cfg, reference=(rp, rv),
                                                weights=torch.cat([a[None], b[None], const]))
        inputs = (t(p0), t(v0), t(P), t(V), wp, wv)
    # p0, v0, goal and reference enter linearly on a fixed active set: central differences are exact up to
    # the solve's own accuracy
    assert torch.autograd.gradcheck(fn, inputs, eps=1e-2, atol=1e-4, rtol=1e-3)


def test_weight_recovery():
    """w_pos and w_vel from demonstrated plans (w_acc, w_thrust fixed: a = (T - m g e3)/m, so only
    w_acc/m^2 + w_thrust is identifiable)."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.config import SE3MPCConfig
    N = 8
    cfg = SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=1e-10, max_iterations=2000)
    p0, v0, goal = _grad_problems(N, B=64, seed=11)
    truth = torch.tensor([100.0, 10.0, 1.0, 0.1], dtype=torch.float64)
    x_demo, _ = dp.plan_batch_differentiable(p0, v0, goal, cfg, weights=truth)
    logw = torch.tensor([np.log(60.0), np.log(20.0)], dtype=torch.float64, requires_grad=True)
    opt = torch.optim.LBFGS([logw], lr=1.0, max_iter=200, tolerance_grad=1e-14, tolerance_change=1e-16,
                            line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        w = torch.cat([logw.exp(), truth[2:]])
        x, _ = dp.plan_batch_differentiable(p0, v0, goal, cfg, weights=w)
        loss = (x - x_demo).square().sum()
        loss.backward()
        return loss

    for _ in range(3):
        opt.step(closure)
    got = logw.detach().exp().numpy()
    assert np.abs(got / np.array([100.0, 10.0]) - 1).max() <= 1e-3, got


def test_vjp_entry_refuses_bad_arguments_on_the_device():
    import torch
    from dart_planner_b200 import _cabi
    L = _cabi.lib()
    check_refusals(L)
    # a launch that is refused writes nothing
    N, B = 8, 64
    p = _params(3, N)
    buf = torch.zeros((9 * N, B), dtype=torch.float64, device="cuda")
    st = torch.full((B,), -9, dtype=torch.int32, device="cuda")
    bp = buf.data_ptr()
    args = lambda q, s: (C.byref(q), B, B, bp, bp, bp, None, bp, None, None, None, None,  # noqa: E731
                         None, None, None, None, None, s, None)
    q = _params(3, 17)
    assert L.dart_se3mpc_solve_vjp_batch(*args(q, st.data_ptr())) == _cabi.DART_E_UNSUPPORTED
    q = _params(2, N)
    assert L.dart_se3mpc_solve_vjp_batch(*args(q, st.data_ptr())) == _cabi.DART_E_BADARG
    torch.cuda.synchronize()
    assert (st == -9).all()
    assert L.dart_se3mpc_solve_vjp_batch(*args(p, st.data_ptr())) == _cabi.DART_OK
    torch.cuda.synchronize()
    assert (st == 0).all()
