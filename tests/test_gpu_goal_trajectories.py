"""Per-step cost goals (x_goal [B, N+1, DA], u_goal [B, N, nu]): reference-trajectory tracking in batched solves and
receding-horizon MPC.

Every kernel only changes where it loads the goal from, so a per-step goal that is constant in time gives what the
per-problem goal gives, problem b of a batch gives what a batch of one gives with that problem's trajectory, and a
change to row t of the goal only changes the cost terms of step t.  Covered on every cost path (known pendulum family
in both layouts, known rendezvous, BNN on the CUDA-core and the tcgen05 MLP, BNN rendezvous), then the oracle, whole
fits, the single-problem API, MPC windowing, argument errors and a sharded fit."""
import ctypes as C
import os
import warnings

import pytest
import torch

import pddp_oracle as O
from test_gpu_goals import (GEOS, OUT_NAMES, bounds, close, consts, cost_spec, dynamics, fit_case, inputs,
                            problem_goals, qr_cost, rel, run, with_goal)

pytestmark = pytest.mark.gpu


def goal_trajectories(name, B, N, seed=5):
    """Time-varying goals: x [B, N+1, DA], u [B, N, nu] (a smooth drift plus noise, so every row differs)."""
    _, D, nu, ang, _, _, _ = GEOS[name]
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    tx = torch.linspace(0, 1, N + 1, dtype=torch.float64).reshape(1, N + 1, 1)
    tu = torch.linspace(0, 1, N, dtype=torch.float64).reshape(1, N, 1)
    xg = 0.4 * r(B, 1, D + len(ang)) + 0.5 * tx * r(B, 1, D + len(ang)) + 0.05 * r(B, N + 1, D + len(ang))
    ug = 0.2 * r(B, 1, nu) + 0.2 * tu * r(B, 1, nu) + 0.02 * r(B, N, nu)
    return xg, ug


def solver(name, enc, layout, dtype, bnn, B, N):
    from pddp_b200.solver import BatchedSolver
    dyn, _ = dynamics(name, bnn)
    spec = cost_spec(name)
    return BatchedSolver(dyn, consts(spec), enc, B, N, dtype=dtype, layout=layout), spec


def dev(g, dtype):
    return None if g is None else g.to(dtype).cuda()


# ------------------------------------------------------------------------ 1. constant in time == per problem
CONST_CASES = ([("pendulum", enc, layout, torch.float64, None) for enc in range(5) for layout in (0, 1)]
               + [(g, enc, layout, torch.float64, None) for g in ("cartpole", "double_cartpole")
                  for enc in range(5) for layout in (0, 1)]
               + [("rendezvous", enc, 0, torch.float64, None) for enc in range(5)] + [("rendezvous", 4, 1, torch.float64, None)]
               + [("pendulum", 4, 1, torch.float32, None), ("cartpole", 1, 0, torch.float32, None),
                  ("rendezvous", 4, 1, torch.float32, None)]
               + [("cartpole", 1, 0, torch.float64, "small"), ("cartpole", 4, 0, torch.float64, "small"),
                  ("cartpole", 1, 0, torch.float32, "tc"), ("rendezvous", 4, 0, torch.float64, "small"),
                  ("rendezvous", 1, 0, torch.float64, "small")])


@pytest.mark.parametrize("name,enc,layout,dtype,bnn", CONST_CASES)
def test_constant_in_time_equals_per_problem(name, enc, layout, dtype, bnn):
    B, N = 8, 6
    s, _ = solver(name, enc, layout, dtype, bnn, B, N)
    xg, ug = problem_goals(name, B)
    z0, U = inputs(name, enc, B, N)
    lo, hi = bounds(name, True)
    want = run(s, z0, U, lo, hi, dev(xg, dtype), dev(ug, dtype))
    xt = xg.unsqueeze(1).expand(B, N + 1, -1).contiguous()
    ut = ug.unsqueeze(1).expand(B, N, -1).contiguous()
    for kw in (dict(x_goal=xt, u_goal=ut), dict(x_goal=xt, u_goal=ug), dict(x_goal=xg, u_goal=ut)):
        got = run(s, z0, U, lo, hi, dev(kw["x_goal"], dtype), dev(kw["u_goal"], dtype),
                  gains=(want["k"], want["K"]))
        for n, v in want.items():
            assert close(got[n], v, dtype), (n, [tuple(g.shape) for g in kw.values()])


# ------------------------------------------------------------------------ 2. indexing
IDX_CASES = [("pendulum", 4, 1, None), ("pendulum", 1, 0, None), ("cartpole", 2, 1, None),
             ("rendezvous", 4, 0, None), ("rendezvous", 0, 1, None),
             ("cartpole", 1, 0, "small"), ("rendezvous", 4, 0, "small")]


@pytest.mark.parametrize("name,enc,layout,bnn", IDX_CASES)
def test_perturbing_one_row_changes_only_that_step(name, enc, layout, bnn):
    B, N = 4, 6
    s, _ = solver(name, enc, layout, torch.float64, bnn, B, N)
    xg, ug = goal_trajectories(name, B, N)
    z0, U = inputs(name, enc, B, N)
    lo, hi = bounds(name, False)
    base = run(s, z0, U, lo, hi, dev(xg, torch.float64), dev(ug, torch.float64))
    cases = [("x", t) for t in (0, N // 2, N)] + [("u", N - 1)]
    for which, t in cases:
        x2, u2 = xg.clone(), ug.clone()
        (x2 if which == "x" else u2)[:, t] += 0.3
        got = run(s, z0, U, lo, hi, dev(x2, torch.float64), dev(u2, torch.float64), gains=(base["k"], base["K"]))
        may = ("L", "L_z", "L_zz") if which == "x" else ("L", "L_u")
        must = ("L", "L_z") if which == "x" else ("L", "L_u")
        for n in OUT_NAMES:
            for step in range(got[n].shape[1]):
                same = torch.equal(got[n][:, step], base[n][:, step])
                if step == t and n in must:
                    assert not same, (which, t, n)
                elif not (step == t and n in may):
                    assert same, (which, t, n, step)


# ------------------------------------------------------------------------ 3. against the oracle
def oracle_cost_terms(spec, xg, ug, Z, U, enc):
    """Per-step loop over O.cost_derivatives, step t with the goal rows xg[t], ug[t]."""
    N = U.shape[0]
    sites = [O.cost_derivatives(with_goal(spec, xg[t], ug[t]), Z[t], U[t], False, enc) for t in range(N)]
    term = O.cost_derivatives(with_goal(spec, xg[N], None), Z[N], None, True, enc)
    return dict(L=torch.stack([c[0] for c in sites] + [term[0]]),
                L_z=torch.stack([c[1] for c in sites] + [term[1]]), L_u=torch.stack([c[2] for c in sites]),
                L_zz=torch.stack([c[3] for c in sites] + [term[3]]), L_uu=torch.stack([c[5] for c in sites]))


def oracle_trajectory_cost(spec, xg, ug, Z, U, enc):
    """J[a] with step t's goal: Z [N+1, A, nz], U [N, A, nu]."""
    N = U.shape[0]
    J = sum(O.cost_value(with_goal(spec, xg[t], ug[t]), Z[t], U[t], False, enc) for t in range(N))
    return J + O.cost_value(with_goal(spec, xg[N], None), Z[N], None, True, enc)


@pytest.mark.parametrize("name,enc,dtype,bnn,bounded", [
    ("pendulum", 0, torch.float64, None, False), ("pendulum", 4, torch.float64, None, True),
    ("pendulum", 4, torch.float32, None, True), ("cartpole", 1, torch.float64, None, True),
    ("double_cartpole", 3, torch.float64, None, False),
    ("rendezvous", 4, torch.float64, None, True), ("rendezvous", 1, torch.float64, None, False),
    ("cartpole", 1, torch.float64, "small", True), ("rendezvous", 4, torch.float64, "small", True),
])
def test_matches_oracle_per_step(name, enc, dtype, bnn, bounded):
    B, N = 6, 6
    s, spec = solver(name, enc, None, dtype, bnn, B, N)
    _, odyn = dynamics(name, bnn)
    xg, ug = goal_trajectories(name, B, N)
    z0, U = inputs(name, enc, B, N)
    lo, hi = bounds(name, bounded)
    got = run(s, z0, U, lo, hi, dev(xg, dtype), dev(ug, dtype))
    tol = 1e-5 if dtype == torch.float64 else 1e-3
    alphas = O.fit_alphas(torch.float64)
    for b in range(B):
        lin = O.linearize(z0[b], U[b], odyn, spec, enc, lo, hi)        # Z, F: the goal does not enter the dynamics
        Uc = U[b] if lo is None else O.clamp(U[b], lo, hi)
        want = oracle_cost_terms(spec, xg[b], ug[b], lin[0], Uc, enc)
        want["Z"] = lin[0]
        for n in OUT_NAMES:
            assert rel(got[n][b].reshape(want[n].shape), want[n]) <= tol, (n, b)
        assert rel(got["J_opt"][b], want["L"].sum()) <= tol, b
        cost_want = oracle_cost_terms(spec, xg[b], ug[b], lin[0], U[b], enc)   # the cost pass sees the stored U
        for n, w in cost_want.items():
            assert rel(got["cost_" + n][b].reshape(w.shape), w) <= tol, ("cost_" + n, b)
        Zr, Ur = O.rollout(odyn, lin[0], U[b], got["k"][b].double().cpu(), got["K"][b].double().cpu(), alphas, enc,
                           lo, hi)
        assert rel(got["J_all"][b], oracle_trajectory_cost(spec, xg[b], ug[b], Zr, Ur, enc)) <= tol, b


# ------------------------------------------------------------------------ 4. batch == singles
@pytest.mark.parametrize("name,enc,bnn", [("cartpole", 1, None), ("rendezvous", 4, "small")])
def test_batch_equals_singles_one_step(name, enc, bnn):
    B, N = 6, 6
    s, _ = solver(name, enc, 0, torch.float64, bnn, B, N)
    one, _ = solver(name, enc, 0, torch.float64, bnn, 1, N)
    xg, ug = goal_trajectories(name, B, N)
    z0, U = inputs(name, enc, B, N)
    lo, hi = bounds(name, True)
    got = run(s, z0, U, lo, hi, dev(xg, torch.float64), dev(ug, torch.float64))
    for b in range(B):
        w = run(one, z0[b:b + 1], U[b:b + 1], lo, hi, dev(xg[b:b + 1], torch.float64),
                dev(ug[b:b + 1], torch.float64), gains=(got["k"][b:b + 1], got["K"][b:b + 1]))
        for n, v in w.items():
            assert close(got[n][b:b + 1], v, torch.float64), (n, b)


@pytest.mark.parametrize("name", ["cartpole", "rendezvous"])
def test_whole_fit_equals_single_fits(name):
    import pddp_b200 as P
    model, spec, enc, z0, U = fit_case(name)
    B, N = z0.shape[0], U.shape[1]
    xg, ug = goal_trajectories(name, B, N)
    lo, hi = bounds(name, True)
    kw = dict(encoding=enc, n_iterations=5, u_min=lo.cuda(), u_max=hi.cuda())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ctrl = P.iLQRController(None, model, qr_cost(spec))
        Z, Uo, state = ctrl.fit(U, z0=z0, x_goal=xg.cuda(), u_goal=ug.cuda(), **kw)
        K = ctrl._K.clone()
        for b in range(B):
            one = P.iLQRController(None, model, qr_cost(spec))
            Z1, U1, s1 = one.fit(U[b:b + 1], z0=z0[b:b + 1], x_goal=xg[b:b + 1].cuda(), u_goal=ug[b:b + 1].cuda(), **kw)
            assert int(s1[0]) == int(state[b]), b
            for a, w in ((Z[b:b + 1], Z1), (Uo[b:b + 1], U1), (K[b:b + 1], one._K)):
                assert close(a, w, torch.float64), b
    assert not close(Z, P.iLQRController(None, model, qr_cost(spec)).fit(U, z0=z0, **kw)[0], torch.float64)


# ------------------------------------------------------------------------ 5. single-problem API
def test_single_problem_api_equals_batch_of_one():
    import pddp_b200 as P
    from pddp_b200.controllers.ilqr import _trajectory_cost
    model, spec, enc, z0, U = fit_case("cartpole")
    N = U.shape[1]
    xg, ug = goal_trajectories("cartpole", 1, N)
    xg, ug = xg.cuda(), ug.cuda()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a, b = P.iLQRController(None, model, qr_cost(spec)), P.iLQRController(None, model, qr_cost(spec))
        Z1, U1, s1 = a.fit(U[0], encoding=enc, n_iterations=4, z0=z0[0], x_goal=xg[0], u_goal=ug[0])
        Zb, Ub, sb = b.fit(U[:1], encoding=enc, n_iterations=4, z0=z0[:1], x_goal=xg, u_goal=ug)
        assert torch.equal(Z1, Zb[0]) and torch.equal(U1, Ub[0]) and int(s1) == int(sb[0])
        st1 = a.step(z0[0], U[0], encoding=enc, x_goal=xg[0], u_goal=ug[0])
        stb = b.step(z0[:1], U[:1], encoding=enc, x_goal=xg, u_goal=ug)
        assert int(st1) == int(stb[0]) and torch.equal(a._U_nominal, b._U_nominal[0])
    J1 = _trajectory_cost(qr_cost(spec), Z1, U1, enc, {"x_goal": xg[0], "u_goal": ug[0]})
    Jb = _trajectory_cost(qr_cost(spec), Z1.unsqueeze(1), U1.unsqueeze(1), enc, {"x_goal": xg, "u_goal": ug})
    assert torch.equal(J1.reshape(1), Jb)


# ------------------------------------------------------------------------ 6. MPC windowing
def test_mpc_forward_equals_step_on_the_clamped_window():
    import pddp_b200 as P
    from pddp_b200.controllers.ilqr import reference_window
    model, spec, enc, z0, U = fit_case("cartpole")
    B, N = z0.shape[0], U.shape[1]
    T = N + 4                                                   # the trial runs past the reference's end
    xref, uref = goal_trajectories("cartpole", B, T, seed=9)
    xref, uref = xref.cuda(), uref[:, :T].cuda()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a, b = P.iLQRController(None, model, qr_cost(spec)), P.iLQRController(None, model, qr_cost(spec))
        a.fit(U, encoding=enc, n_iterations=3, z0=z0)
        b.fit(U, encoding=enc, n_iterations=3, z0=z0)
        z = z0.clone()
        for i in range(T + 3):
            ua = a.forward(z, i, enc, mpc=True, x_goal=xref, u_goal=uref)
            rows = torch.arange(i, i + N + 1).clamp(max=xref.shape[1] - 1)
            xw, uw = xref[:, rows], uref[:, rows[:N].clamp(max=uref.shape[1] - 1)]
            assert torch.equal(reference_window(xref, i, N + 1, True), xw)
            b.step(z, i=i, encoding=enc, _keep_reg=False, x_goal=xw, u_goal=uw)
            ub = b._U_nominal[:, 0].clone()
            b._U_nominal = torch.cat([b._U_nominal[:, 1:], b._U_nominal[:, -1:]], 1)
            assert torch.equal(ua, ub), i
            z = z + 0.01 * torch.randn_like(z)


def test_closed_loop_mpc_follows_a_moving_reference():
    import pddp_b200 as P
    from pddp_b200.controllers import _apply_controller
    from pddp_b200.controllers.ilqr import _trajectory_cost
    torch.set_default_dtype(torch.float64)
    try:
        model = P.examples.pendulum.PendulumDynamicsModel(0.1)
        Q = torch.diag(torch.tensor([0.1, 10.0, 10.0]))
        cost = P.costs.QRCost(Q, 0.01 * torch.eye(1), Q, [0.0, 0.0, 1.0], state_size=2, angular_indices=(0,)).double()
        envs = [P.examples.pendulum.PendulumEnv.from_model(model, batch_size=4, dtype=torch.float64) for _ in range(2)]
    finally:
        torch.set_default_dtype(torch.float32)
    enc, N, H = 4, 15, 30
    # every pendulum swings from hanging down to its own angle along a ramp
    final = torch.tensor([-0.9, -0.4, 0.4, 0.9], dtype=torch.float64)
    theta = final.unsqueeze(1) * torch.linspace(0, 1, H + 1, dtype=torch.float64).clamp(max=0.7).unsqueeze(0) / 0.7
    ref = torch.stack([torch.zeros_like(theta), theta.sin(), theta.cos()], 2).cuda()        # [4, H+1, DA]
    ends = []
    for env, goal in zip(envs, (ref, ref[:, :1].expand(-1, H + 1, -1).contiguous())):
        torch.manual_seed(0)
        env.set_state(torch.zeros(4, 2, dtype=torch.float64))
        ctrl = P.iLQRController(env, model, cost)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ctrl.fit(torch.zeros(4, N, 1, dtype=torch.float64, device="cuda"), encoding=enc, n_iterations=10,
                     z0=env.get_state().encode(enc), x_goal=goal[:, :N + 1])
            (X, Um, dX), J = _apply_controller(env, cost, ctrl, H, enc, True, True, {"x_goal": goal}, x_goal=goal)
        ends.append((env.get_state().mean()[:, 0].cpu() - final).abs())
        assert J.shape == (4,) and bool(torch.isfinite(J).all())
    assert bool((ends[0] < ends[1]).all()), ends


# ------------------------------------------------------------------------ 7. errors and no carry-over
def test_errors_and_no_carry_over():
    import pddp_b200 as P
    from pddp_b200.controllers.ilqr import _trajectory_cost
    model, spec, enc, z0, U = fit_case("cartpole")
    B, N = z0.shape[0], U.shape[1]
    xg, ug = goal_trajectories("cartpole", B, N)
    ctrl = P.iLQRController(None, model, qr_cost(spec))
    fit = lambda **kw: ctrl.fit(U, encoding=enc, n_iterations=3, z0=z0, **kw)
    for bad in (dict(x_goal=xg[:, :N].cuda()), dict(x_goal=xg[:, :, :4].cuda()), dict(u_goal=ug[:, :N - 1].cuda()),
                dict(u_goal=torch.zeros(B, N + 1, 1, dtype=torch.float64, device="cuda")),
                dict(x_goal=xg[:-1].cuda())):
        with pytest.raises(ValueError):
            fit(**bad)
    with pytest.raises(RuntimeError):
        fit(x_goal=xg)                                          # CPU tensor
    with pytest.raises(ValueError):
        ctrl.fit(U[0], encoding=enc, n_iterations=3, z0=z0[0], x_goal=xg[0, :N].cuda())
    with pytest.raises(RuntimeError):
        ctrl.step(z0[0], U[0], encoding=enc, u_goal=ug[0])
    with pytest.raises(ValueError):
        _trajectory_cost(qr_cost(spec), torch.zeros(N + 1, 14, dtype=torch.float64, device="cuda"),
                         torch.zeros(N, 1, dtype=torch.float64, device="cuda"), enc, {"x_goal": xg[0, :N].cuda()})
    assert ctrl._solver is None or ctrl._solver.goals == {}        # nothing was copied before the errors
    Zg, _, _ = fit(x_goal=xg.cuda(), u_goal=ug.cuda())
    Z0, U0, s0 = fit()                                          # same cached solver, no goals
    fresh = P.iLQRController(None, model, qr_cost(spec))
    Zf, Uf, sf = fresh.fit(U, encoding=enc, n_iterations=3, z0=z0)
    assert not torch.equal(Zg, Z0)
    assert torch.equal(Z0, Zf) and torch.equal(U0, Uf) and torch.equal(s0, sf)


@pytest.mark.parametrize("name,bnn", [("cartpole", None), ("rendezvous", None), ("cartpole", "small")])
def test_c_abi_rejects_per_problem_and_per_step_together(name, bnn):
    from pddp_b200 import _lib
    B, N = 4, 5
    s, _ = solver(name, 1, 0, torch.float64, bnn, B, N)
    xg, ug = problem_goals(name, B)
    xt, ut = goal_trajectories(name, B, N)
    z0, U = inputs(name, 1, B, N)
    s.set_problem(z0.cuda(), U.cuda())
    keep = [t.cuda() for t in (xg, ug, xt, ut)]
    p = [t.data_ptr() for t in keep]
    for ptrs in ((p[0], None, p[2], None), (None, p[1], None, p[3])):
        s._goal_ptrs = ptrs
        before = s.view("L").clone()
        with pytest.raises(RuntimeError, match="exclusive"):
            s.linearize()
        with pytest.raises(RuntimeError, match="exclusive"):
            s.cost_only()
        torch.cuda.synchronize()
        assert torch.equal(s.view("L"), before)                # nothing was launched
        b = s.buf
        code = _lib.load().pddp_cost_derivatives(C.byref(s.shape), s._cost(), _lib.ptr(b["Z"]), _lib.ptr(b["U"]), None,
                                                 *[_lib.ptr(b[n]) for n in ("L", "L_z", "L_u", "L_zz", "L_uz", "L_uu")],
                                                 None, _lib.stream_ptr())
        assert code == -1                                   # PDDP_E_BADARG
    s.set_goals()


# ------------------------------------------------------------------------ 8. two ranks
def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    import pddp_b200 as P
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    B, N = 37, 12                                              # uneven shards (19 + 18)
    model = P.examples.cartpole.CartpoleDynamicsModel(0.1)
    spec = cost_spec("cartpole")
    z0, U = inputs("cartpole", 1, B, N)
    xg, ug = goal_trajectories("cartpole", B, N)
    kw = dict(encoding=1, n_iterations=6, z0=z0.float().to(d), x_goal=xg.to(d), u_goal=ug.to(d))
    ctrl = P.iLQRController(None, model, qr_cost(spec).float())
    Zs, Us, ss = ctrl.fit(U.float().to(d), **kw)
    single = P.iLQRController(None, model, qr_cost(spec).float())
    Z1, U1, s1 = single.fit(U.float().to(d), shard=False, **kw)
    ok = (torch.equal(Zs, Z1) and torch.equal(Us, U1) and torch.equal(ss, s1) and torch.equal(ctrl._K, single._K))
    torch.save(bool(ok), os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_fit_with_goal_trajectories_equals_single_gpu_fit(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_sharded_worker, args=(2, 29757, str(tmp_path)), nprocs=2, join=True)
    for rank in range(2):
        assert torch.load(os.path.join(str(tmp_path), "rank%d.pt" % rank)), rank
