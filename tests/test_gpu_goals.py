"""Per-problem cost goals (x_goal [B, DA], u_goal [B, nu]) in batched solves.

A batch in which every problem has its own goal must give, problem for problem, what a batch of one gives with a
QRCost whose x_goal / u_goal is that problem's goal: the arithmetic is the same, only the goal is loaded per problem.
Every cost path is covered (known pendulum family in both layouts, known rendezvous, BNN on the tcgen05 and the
CUDA-core MLP, BNN rendezvous), then the oracle, whole fits, closed-loop MPC, argument errors and a sharded fit."""
import os
import warnings

import pytest
import torch

import pddp_oracle as O

pytestmark = pytest.mark.gpu

# name -> (geo, D, nu, angular, non-angular, known parameters in the C ABI order, oracle spec)
GEOS = {
    "pendulum": (0, 2, 1, (0,), (1,), [0.1, 1.0, 1.0, 0.1, 9.80665], O.pendulum_spec(0.1)),
    "cartpole": (1, 4, 1, (2,), (0, 1, 3), [0.1, 0.5, 0.5, 0.5, 0.1, 9.82], O.cartpole_spec(0.1)),
    "double_cartpole": (2, 6, 1, (2, 4), (0, 1, 3, 5), [0.1, 0.5, 0.5, 0.5, 0.6, 0.6, 0.1, 9.80665],
                        O.double_cartpole_spec(0.1)),
    "rendezvous": (3, 8, 4, (), tuple(range(8)), [0.1, 1.0, 0.1], O.rendezvous_spec(0.1)),
}
OUT_NAMES = ("Z", "L", "L_z", "L_u", "L_zz", "L_uu")


def close(a, b, dtype):
    """Equal up to the last bits: max |a - b| relative to the scale of b."""
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    a, b = a.double().cpu(), b.double().cpu()
    return (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item())


def spd(n, g, scale=1.0):
    A = torch.randn(n, n, generator=g, dtype=torch.float64)
    return scale * (A @ A.T / n + 0.5 * torch.eye(n, dtype=torch.float64))


def cost_spec(name, seed=0):
    """A shared QR cost: random SPD weights, shared goals that differ from every problem's own goal."""
    _, D, nu, ang, nonang, _, _ = GEOS[name]
    DA = D + len(ang)
    g = torch.Generator().manual_seed(seed)
    return O.QRCostSpec(spd(DA, g), spd(nu, g, 0.1), spd(DA, g, 4.0), 0.3 * torch.randn(DA, generator=g,
                        dtype=torch.float64), 0.1 * torch.randn(nu, generator=g, dtype=torch.float64), D, ang, nonang)


def problem_goals(name, B, seed=1):
    _, D, nu, ang, _, _, _ = GEOS[name]
    g = torch.Generator().manual_seed(seed)
    return (0.5 * torch.randn(B, D + len(ang), generator=g, dtype=torch.float64),
            0.2 * torch.randn(B, nu, generator=g, dtype=torch.float64))


def with_goal(spec, xg=None, ug=None):
    return O.QRCostSpec(spec.Q, spec.R, spec.Q_term, spec.x_goal if xg is None else xg,
                        spec.u_goal if ug is None else ug, spec.D, spec.ang, spec.nonang)


def consts(spec):
    from pddp_b200.solver import QRCostConstants
    return QRCostConstants(spec.Q, spec.R, spec.Q_term, spec.x_goal, spec.u_goal)


def synth_bnn(name, P, H, seed):
    """Two hidden layers of H, P particles (weights scaled so the rollouts stay bounded)."""
    _, D, nu, ang, nonang, _, _ = GEOS[name]
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    W = [r(H, D + len(ang) + nu) * 0.5, r(H, H) * (1.0 / H ** 0.5), r(2 * D, H) * 0.02]
    bias = [0.1 * r(H), 0.1 * r(H), 0.01 * r(2 * D)]
    masks = [torch.rand(P, H, generator=g, dtype=torch.float64), torch.rand(P, H, generator=g, dtype=torch.float64)]
    eps0 = r(P, D)
    eps0 = (eps0 - eps0.mean(0)) / eps0.std(0)
    return W, bias, masks, eps0


def dynamics(name, bnn):
    """(solver dynamics, oracle dynamics); bnn = None | "small" (CUDA-core MLP) | "tc" (2 x 200, 50 particles)."""
    from pddp_b200.solver import BNNDynamics, KnownDynamics
    geo, D, nu, ang, nonang, params, spec = GEOS[name]
    if bnn is None:
        return KnownDynamics(geo, params), spec
    if bnn == "tc":
        import bench
        W, bias, masks, eps0 = [[t.double() for t in x] if isinstance(x, list) else x.double()
                                for x in bench.synth_bnn(name, 50, 200, seed=0)]
    else:
        W, bias, masks, eps0 = synth_bnn(name, 12, 32, seed=3)
    return BNNDynamics(geo, W, bias, masks, eps0), O.BNNSpec(list(zip(W, bias)), masks, eps0, D, nu, ang, nonang)


def inputs(name, enc, B, N, seed=2):
    _, D, nu, _, _, _, _ = GEOS[name]
    g = torch.Generator().manual_seed(seed)
    mean = 0.1 * torch.randn(B, D, generator=g, dtype=torch.float64)
    V = 1e-2 * (1 + torch.rand(B, D, generator=g, dtype=torch.float64))
    z0 = torch.stack([O.encode(m, V=v, enc=enc) for m, v in zip(mean, V)])
    return z0, 0.3 * torch.randn(B, N, nu, generator=g, dtype=torch.float64)


def bounds(name, bounded):
    nu = GEOS[name][2]
    return ((None, None) if not bounded else
            (torch.full((nu,), -0.4, dtype=torch.float64), torch.full((nu,), 0.4, dtype=torch.float64)))


def run(solver, z0, U, lo, hi, x_goal=None, u_goal=None, gains=None):
    """Linearise, backward (or the given gains), rollout and the stand-alone cost pass on the solver's own Z / U."""
    dt = solver.dtype
    solver.set_problem(z0.to(dt).cuda(), U.to(dt).cuda(), lo, hi, x_goal=x_goal, u_goal=u_goal)
    solver.linearize()
    out = {n: solver.matrices(n).clone() for n in OUT_NAMES}
    out["J_opt"] = solver.J_opt.clone()
    if gains is None:
        solver.mu.fill_(1.0)
        solver.backward()
    else:
        solver.store("k", gains[0])
        solver.store("K", gains[1].reshape(gains[1].shape[0], gains[1].shape[1], -1))
    out["k"], out["K"] = solver.matrices("k").clone(), solver.matrices("K").clone()
    solver.rollout(use_bw_status=False)
    for n in ("Z_new", "U_new"):
        out[n] = solver.view(n).clone()
    out["J_all"], out["amin"] = solver.J_all.clone(), solver.amin.clone()
    solver.cost_only()
    for n in ("L", "L_z", "L_u", "L_zz", "L_uu"):
        out["cost_" + n] = solver.matrices(n).clone()
    out["cost_J"] = solver.J_opt.clone()
    torch.cuda.synchronize()
    return out


def batched_and_single(name, enc, layout, dtype, bnn, bounded, B, N, goals="both"):
    from pddp_b200.solver import BatchedSolver
    dyn, _ = dynamics(name, bnn)
    spec = cost_spec(name)
    xg, ug = problem_goals(name, B)
    xg, ug = (xg if goals != "u" else None), (ug if goals != "x" else None)
    z0, U = inputs(name, enc, B, N)
    lo, hi = bounds(name, bounded)
    s = BatchedSolver(dyn, consts(spec), enc, B, N, dtype=dtype, layout=layout)
    got = run(s, z0, U, lo, hi, None if xg is None else xg.to(dtype).cuda(), None if ug is None else ug.to(dtype).cuda())
    one = BatchedSolver(dyn, consts(spec), enc, 1, N, dtype=dtype, layout=layout)
    singles = []
    for b in range(B):
        one.c_cost = consts(with_goal(spec, None if xg is None else xg[b], None if ug is None else ug[b])).c_struct()
        singles.append(run(one, z0[b:b + 1], U[b:b + 1], lo, hi, gains=(got["k"][b:b + 1], got["K"][b:b + 1])))
    return got, singles, spec, (xg, ug), (z0, U, lo, hi)


def assert_batched_equals_single(got, singles, dtype):
    for b, one in enumerate(singles):
        for n, v in one.items():
            if n in ("k", "K"):
                continue
            assert close(got[n][b:b + 1], v, dtype), (n, b)
    assert len(set(round(float(v), 6) for v in got["J_opt"].cpu())) == len(singles)     # the goals do differ


KNOWN_CASES = ([("pendulum", enc, 1, bounded) for enc in range(5) for bounded in (False, True)]
               + [(g, enc, layout, True) for g, encs in (("cartpole", (1, 4)), ("double_cartpole", (0, 4)))
                  for enc in encs for layout in (0, 1)]
               + [("rendezvous", enc, 0, enc % 2 == 0) for enc in range(5)] + [("rendezvous", 4, 1, True)])


@pytest.mark.parametrize("name,enc,layout,bounded", KNOWN_CASES)
def test_known_batched_equals_per_problem(name, enc, layout, bounded):
    got, singles, *_ = batched_and_single(name, enc, layout, torch.float64, None, bounded, B=12, N=8)
    assert_batched_equals_single(got, singles, torch.float64)


@pytest.mark.parametrize("name", ["pendulum", "rendezvous"])
def test_known_fp32_batched_equals_per_problem(name):
    got, singles, *_ = batched_and_single(name, 4, 1, torch.float32, None, True, B=16, N=8)
    assert_batched_equals_single(got, singles, torch.float32)


@pytest.mark.parametrize("name,enc,dtype,bnn,bounded", [
    ("cartpole", 1, torch.float32, "tc", True),                 # tcgen05 particle MLP
    ("cartpole", 1, torch.float64, "small", False),             # CUDA-core MLP
    ("cartpole", 4, torch.float64, "small", True),
    ("rendezvous", 4, torch.float64, "small", True),
    ("rendezvous", 1, torch.float64, "small", False),
])
def test_bnn_batched_equals_per_problem(name, enc, dtype, bnn, bounded):
    got, singles, *_ = batched_and_single(name, enc, 0, dtype, bnn, bounded, B=8, N=6)
    assert_batched_equals_single(got, singles, dtype)


@pytest.mark.parametrize("name,goals", [("pendulum", "x"), ("pendulum", "u"), ("rendezvous", "x"),
                                        ("rendezvous", "u"), ("cartpole", "u")])
def test_each_goal_on_its_own(name, goals):
    got, singles, *_ = batched_and_single(name, 4 if name != "cartpole" else 1, 0, torch.float64, None, True, B=10,
                                          N=8, goals=goals)
    assert_batched_equals_single(got, singles, torch.float64)


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return (a - b).abs().max().item() / max(1.0, b.abs().max().item())


@pytest.mark.parametrize("name,enc,dtype,bnn,bounded", [
    ("pendulum", 0, torch.float64, None, False), ("pendulum", 1, torch.float64, None, True),
    ("pendulum", 2, torch.float64, None, False), ("pendulum", 3, torch.float64, None, True),
    ("pendulum", 4, torch.float32, None, True), ("cartpole", 1, torch.float64, None, True),
    ("rendezvous", 4, torch.float64, None, True), ("rendezvous", 1, torch.float64, None, False),
    ("cartpole", 1, torch.float64, "small", True), ("rendezvous", 4, torch.float64, "small", True),
])
def test_matches_oracle_per_problem(name, enc, dtype, bnn, bounded):
    got, _, spec, (xg, ug), (z0, U, lo, hi) = batched_and_single(name, enc, 0, dtype, bnn, bounded, B=8, N=6)
    _, odyn = dynamics(name, bnn)
    tol = 1e-5 if dtype == torch.float64 else 1e-3
    alphas = O.fit_alphas(torch.float64)
    for b in range(z0.shape[0]):
        ocost = with_goal(spec, xg[b], ug[b])
        lin = O.linearize(z0[b], U[b], odyn, ocost, enc, lo, hi)
        want = dict(zip(("Z", "F_z", "F_u", "L", "L_z", "L_u", "L_zz", "L_uz", "L_uu"), lin))
        for n in OUT_NAMES:
            assert rel(got[n][b].reshape(want[n].shape), want[n]) <= tol, (n, b)
        # the stand-alone cost pass ran on the solver's Z and the stored (unclamped) U
        N = U.shape[1]
        sites = [O.cost_derivatives(ocost, lin[0][t], U[b][t], False, enc) for t in range(N)]
        term = O.cost_derivatives(ocost, lin[0][N], None, True, enc)
        cost_want = dict(L=torch.stack([c[0] for c in sites] + [term[0]]),
                         L_z=torch.stack([c[1] for c in sites] + [term[1]]), L_u=torch.stack([c[2] for c in sites]),
                         L_zz=torch.stack([c[3] for c in sites] + [term[3]]), L_uu=torch.stack([c[5] for c in sites]))
        for n, w in cost_want.items():
            assert rel(got["cost_" + n][b].reshape(w.shape), w) <= tol, ("cost_" + n, b)
        Zr, Ur = O.rollout(odyn, lin[0], U[b], got["k"][b].double().cpu(), got["K"][b].double().cpu(), alphas, enc, lo,
                           hi)
        assert rel(got["J_all"][b], O.trajectory_cost(ocost, Zr, Ur, enc)) <= tol, b


# ---------------------------------------------------------------------------------------------- whole fits
def qr_cost(spec, xg=None):
    import pddp_b200 as P
    return P.costs.QRCost(spec.Q, spec.R, spec.Q_term, spec.x_goal if xg is None else xg, spec.u_goal,
                          state_size=spec.D, angular_indices=tuple(spec.ang))


def fit_case(name):
    """(model, cost spec, encoding, z0, U): known cartpole, or a BNN model on the rendezvous problem."""
    import pddp_b200 as P
    if name == "cartpole":
        model, enc = P.examples.cartpole.CartpoleDynamicsModel(0.1).double(), 1
    else:
        torch.manual_seed(0)
        mc = P.examples.rendezvous.RendezvousDynamicsModel
        model = P.models.bnn.bnn_dynamics_model_factory(8, 4, [32, 32], mc.angular_indices, mc.non_angular_indices)(
            n_particles=12)
        model.eval()
        enc = 4
    z0, U = inputs(name, enc, 6, 10)
    return model, cost_spec(name), enc, z0.cuda(), U.cuda()


@pytest.mark.parametrize("name", ["cartpole", "rendezvous"])
def test_whole_fit_equals_per_problem_fits(name):
    import pddp_b200 as P
    model, spec, enc, z0, U = fit_case(name)
    B = z0.shape[0]
    xg, ug = problem_goals(name, B)
    lo, hi = bounds(name, True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ctrl = P.iLQRController(None, model, qr_cost(spec))
        Z, Uo, state = ctrl.fit(U, encoding=enc, n_iterations=5, z0=z0, u_min=lo.cuda(), u_max=hi.cuda(),
                                x_goal=xg.cuda(), u_goal=ug.cuda())
        K = ctrl._K.clone()
        for b in range(B):
            c = qr_cost(spec, xg[b])
            c.u_goal.data.copy_(ug[b])
            one = P.iLQRController(None, model, c)
            Z1, U1, s1 = one.fit(U[b:b + 1], encoding=enc, n_iterations=5, z0=z0[b:b + 1], u_min=lo.cuda(),
                                 u_max=hi.cuda())
            assert int(s1[0]) == int(state[b]), b
            for a, w in ((Z[b:b + 1], Z1), (Uo[b:b + 1], U1), (K[b:b + 1], one._K)):
                assert close(a, w, torch.float64), b


def test_errors_and_no_carry_over():
    import pddp_b200 as P
    from pddp_b200.controllers.ilqr import _trajectory_cost
    model, spec, enc, z0, U = fit_case("cartpole")
    B = z0.shape[0]
    xg, ug = problem_goals("cartpole", B)
    ctrl = P.iLQRController(None, model, qr_cost(spec))
    fit = lambda **kw: ctrl.fit(U, encoding=enc, n_iterations=3, z0=z0, **kw)
    with pytest.raises(ValueError):
        fit(x_goal=xg[:, :4].cuda())                             # [B, D] instead of [B, DA]
    with pytest.raises(ValueError):
        fit(x_goal=xg[:-1].cuda())
    with pytest.raises(ValueError):
        fit(u_goal=ug.reshape(-1).cuda())
    with pytest.raises(RuntimeError):
        fit(x_goal=xg)                                          # CPU tensor
    with pytest.raises(ValueError):                             # goals with one (unbatched) problem
        ctrl.fit(U[0], encoding=enc, n_iterations=3, z0=z0[0], x_goal=xg[:1].cuda())
    with pytest.raises(ValueError):
        ctrl.step(z0[0], U[0], encoding=enc, u_goal=ug[:1].cuda())
    with pytest.raises(ValueError):
        _trajectory_cost(qr_cost(spec), torch.zeros(11, 14, dtype=torch.float64, device="cuda"),
                         torch.zeros(10, 1, dtype=torch.float64, device="cuda"), enc, {"x_goal": xg[:1].cuda()})
    assert ctrl._solver is None or ctrl._solver.goals == {}        # nothing was copied before the errors
    Zg, _, _ = fit(x_goal=xg.cuda(), u_goal=ug.cuda())
    Z0, U0, s0 = fit()                                          # same cached solver, no goals
    fresh = P.iLQRController(None, model, qr_cost(spec))
    Zf, Uf, sf = fresh.fit(U, encoding=enc, n_iterations=3, z0=z0)
    assert not torch.equal(Zg, Z0)
    assert torch.equal(Z0, Zf) and torch.equal(U0, Uf) and torch.equal(s0, sf)


def test_closed_loop_mpc_tracks_each_target():
    import pddp_b200 as P
    from pddp_b200.controllers import _apply_controller
    from pddp_b200.controllers.ilqr import _trajectory_cost
    torch.set_default_dtype(torch.float64)
    try:
        model = P.examples.pendulum.PendulumDynamicsModel(0.1)
        Q = torch.diag(torch.tensor([0.1, 10.0, 10.0]))
        cost = P.costs.QRCost(Q, 0.01 * torch.eye(1), Q, [0.0, 0.0, 1.0], state_size=2, angular_indices=(0,)).double()
        env = P.examples.pendulum.PendulumEnv.from_model(model, batch_size=4, dtype=torch.float64)
    finally:
        torch.set_default_dtype(torch.float32)
    targets = torch.tensor([-0.9, -0.3, 0.3, 0.9], dtype=torch.float64)
    xg = torch.stack([torch.zeros(4, dtype=torch.float64), targets.sin(), targets.cos()], 1).cuda()
    enc, N, H = 4, 15, 25
    env.set_state(torch.zeros(4, 2, dtype=torch.float64))
    ctrl = P.iLQRController(env, model, cost)
    U0 = torch.zeros(4, N, 1, dtype=torch.float64, device="cuda")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ctrl.fit(U0, encoding=enc, n_iterations=10, z0=env.get_state().encode(enc), x_goal=xg)
        # x_goal reaches every MPC step through **kwargs; cost_opts carries it to the trial's cost J
        (X, Um, dX), J = _apply_controller(env, cost, ctrl, H, enc, True, True, {"x_goal": xg}, x_goal=xg)
    theta = env.get_state().mean()[:, 0].cpu()
    dist = (theta.unsqueeze(1) - targets.unsqueeze(0)).abs()
    assert torch.equal(dist.argmin(1), torch.arange(4)), dist
    Z = X.reshape(4, H, 2)                                          # instance-major rows -> [H+1, B, nz] below
    Zall = torch.cat([Z, (Z[:, -1] + dX.reshape(4, H, 2)[:, -1]).unsqueeze(1)], 1).transpose(0, 1).contiguous().cuda()
    Uall = Um.reshape(4, H, 1).transpose(0, 1).contiguous().cuda()
    for b in range(4):
        cb = P.costs.QRCost(Q.double(), 0.01 * torch.eye(1, dtype=torch.float64), Q.double(), xg[b].cpu(), state_size=2,
                            angular_indices=(0,))
        assert close(J[b:b + 1], _trajectory_cost(cb, Zall[:, b], Uall[:, b], enc).reshape(1), torch.float64), b
    J_shared = torch.stack([_trajectory_cost(cost, Zall[:, b], Uall[:, b], enc) for b in range(4)])
    assert close(_trajectory_cost(cost, Zall, Uall, enc), J_shared, torch.float64)   # no goals carried over
    assert not close(J, J_shared, torch.float64)


def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    import pddp_b200 as P
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    B, N = 37, 12                                              # uneven shards (19 + 18)
    model = P.examples.cartpole.CartpoleDynamicsModel(0.1)
    spec = cost_spec("cartpole")
    z0, U = inputs("cartpole", 1, B, N)
    xg, ug = problem_goals("cartpole", B)
    kw = dict(encoding=1, n_iterations=6, z0=z0.float().to(dev), x_goal=xg.to(dev), u_goal=ug.to(dev))
    ctrl = P.iLQRController(None, model, qr_cost(spec).float())
    Zs, Us, ss = ctrl.fit(U.float().to(dev), **kw)
    single = P.iLQRController(None, model, qr_cost(spec).float())
    Z1, U1, s1 = single.fit(U.float().to(dev), shard=False, **kw)
    ok = (torch.equal(Zs, Z1) and torch.equal(Us, U1) and torch.equal(ss, s1) and torch.equal(ctrl._K, single._K))
    torch.save(bool(ok), os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_fit_with_goals_equals_single_gpu_fit(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_sharded_worker, args=(2, 29753, str(tmp_path)), nprocs=2, join=True)
    for rank in range(2):
        assert torch.load(os.path.join(str(tmp_path), "rank%d.pt" % rank)), rank
