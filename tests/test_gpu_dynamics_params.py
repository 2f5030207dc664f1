"""Per-problem dynamics parameters (pddp_known_dynamics.p_b [B, 8]) in batched solves, MPC and the simulators.

A batch of B distinct systems must give, problem for problem, what a batch of one gives with that problem's system
as the shared parameters: the step arithmetic is the same, only where the parameters are loaded from changes.
Every known geometry is covered (pendulum, cartpole, double cartpole, rendezvous), with IGNORE_UNCERTAINTY and the
uncertain encodings, both layouts and both dtypes; then the oracle, isolation, per-step goals, the environment step,
closed loops, the public API with its errors, and a sharded fit."""
import os
import warnings

import pytest
import torch

import pddp_oracle as O
from test_gpu_goals import GEOS, bounds, close, consts, cost_spec, inputs, qr_cost, rel, run

pytestmark = pytest.mark.gpu

SPECS = {"pendulum": O.pendulum_spec, "cartpole": O.cartpole_spec, "double_cartpole": O.double_cartpole_spec,
         "rendezvous": O.rendezvous_spec}
LIN = ("Z", "F_z", "F_u", "L", "L_z", "L_u", "L_zz", "L_uz", "L_uu")


def shared_params(name):
    return GEOS[name][5]


def rows(name, B, seed=5, spread=0.2):
    """B parameter sets: the shared ones, each value scaled by a factor in [1 - spread, 1 + spread]."""
    p = torch.tensor(shared_params(name), dtype=torch.float64)
    g = torch.Generator().manual_seed(seed)
    r = torch.zeros(B, 8, dtype=torch.float64)
    r[:, :p.numel()] = p * (1 + spread * (2 * torch.rand(B, p.numel(), generator=g, dtype=torch.float64) - 1))
    return r


def known(name, params_b=None, params=None):
    from pddp_b200.solver import KnownDynamics
    return KnownDynamics(GEOS[name][0], shared_params(name) if params is None else params, params_b)


def solve(name, enc, layout, dtype, dyn, bounded, B, N, gains=None, x_goal=None, u_goal=None, z0U=None):
    from pddp_b200.solver import BatchedSolver
    z0, U = inputs(name, enc, B, N) if z0U is None else z0U
    lo, hi = bounds(name, bounded)
    s = BatchedSolver(dyn, consts(cost_spec(name)), enc, B, N, dtype=dtype, layout=layout)
    out = run(s, z0, U, lo, hi, x_goal, u_goal, gains)
    for n in ("F_z", "F_u", "L_uz"):
        out[n] = s.matrices(n).clone()
    return out


def row_list(name, r):
    return r[:len(shared_params(name))].tolist()


CASES = ([("pendulum", enc, layout) for enc in range(5) for layout in (0, 1)]
         + [(g, enc, layout) for g, encs in (("cartpole", (1, 4)), ("double_cartpole", (0, 4))) for enc in encs
            for layout in (0, 1)]
         + [("rendezvous", enc, 0) for enc in range(5)] + [("rendezvous", 4, 1)])
DTYPES = (torch.float64, torch.float32)


def is_step_output(n):
    return n not in ("k", "K")


# ----------------------------------------------------------------------------------------------- 1. equal rows
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name,enc,layout", CASES)
def test_rows_equal_to_shared_reproduce_shared_path(name, enc, layout, dtype):
    B, N = 9, 8
    r = torch.tensor(shared_params(name) + [0.0] * (8 - len(shared_params(name))), dtype=torch.float64).repeat(B, 1)
    want = solve(name, enc, layout, dtype, known(name), True, B, N)
    got = solve(name, enc, layout, dtype, known(name, r), True, B, N)
    for n in LIN + ("J_opt", "J_all", "amin", "Z_new", "U_new"):
        assert close(got[n], want[n], dtype), n
    same = all(torch.equal(got[n], want[n]) for n in want)
    print("bit-identical %s enc=%d layout=%d %s: %s" % (name, enc, layout, dtype, same))


# ------------------------------------------------------------------------- 2. distinct systems = batches of one
def batched_and_singles(name, enc, layout, dtype, bounded, B=6, N=8, x_goal=None, u_goal=None):
    r = rows(name, B)
    z0U = inputs(name, enc, B, N)
    got = solve(name, enc, layout, dtype, known(name, r), bounded, B, N, x_goal=x_goal, u_goal=u_goal, z0U=z0U)
    singles = []
    for b in range(B):
        xg = None if x_goal is None else x_goal[b:b + 1]
        ug = None if u_goal is None else u_goal[b:b + 1]
        singles.append(solve(name, enc, layout, dtype, known(name, params=row_list(name, r[b])), bounded, 1, N,
                             gains=(got["k"][b:b + 1], got["K"][b:b + 1]), x_goal=xg, u_goal=ug,
                             z0U=(z0U[0][b:b + 1], z0U[1][b:b + 1])))
    return got, singles, r, z0U


def assert_equals_singles(got, singles, dtype):
    for b, one in enumerate(singles):
        for n, v in one.items():
            if is_step_output(n):
                assert close(got[n][b:b + 1], v, dtype), (n, b)
    assert len(set(round(float(v), 6) for v in got["J_opt"].cpu())) == len(singles)      # the systems do differ


@pytest.mark.parametrize("bounded", (False, True))
@pytest.mark.parametrize("name,enc,layout", CASES)
def test_distinct_systems_equal_batches_of_one(name, enc, layout, bounded):
    got, singles, *_ = batched_and_singles(name, enc, layout, torch.float64, bounded)
    assert_equals_singles(got, singles, torch.float64)


@pytest.mark.parametrize("name,enc", [("pendulum", 4), ("pendulum", 1), ("cartpole", 4), ("double_cartpole", 4),
                                      ("rendezvous", 4), ("rendezvous", 1)])
def test_distinct_systems_equal_batches_of_one_fp32(name, enc):
    got, singles, *_ = batched_and_singles(name, enc, 1, torch.float32, True)
    assert_equals_singles(got, singles, torch.float32)


def family_model(name, r):
    import pddp_b200 as P
    cls = {"pendulum": P.examples.pendulum.PendulumDynamicsModel, "cartpole": P.examples.cartpole.CartpoleDynamicsModel,
           "double_cartpole": P.examples.double_cartpole.DoubleCartpoleDynamicsModel,
           "rendezvous": P.examples.rendezvous.RendezvousDynamicsModel}[name]
    k = len(shared_params(name))
    cols = r[:, :k] if r.dim() == 2 else r[:k]
    return cls(*[cols[..., j].clone() for j in range(k)]).double()


@pytest.mark.parametrize("name,enc", [("pendulum", 4), ("cartpole", 1), ("double_cartpole", 4), ("rendezvous", 4)])
def test_whole_fit_equals_per_problem_fits(name, enc):
    import pddp_b200 as P
    B, N = 5, 10
    r = rows(name, B)
    z0, U = inputs(name, enc, B, N)
    z0, U = z0.cuda(), U.cuda()
    lo, hi = (t.cuda() for t in bounds(name, True))
    spec = cost_spec(name)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ctrl = P.iLQRController(None, family_model(name, r), qr_cost(spec))
        Z, Uo, state = ctrl.fit(U, encoding=enc, n_iterations=5, z0=z0, u_min=lo, u_max=hi)
        K = ctrl._K.clone()
        for b in range(B):
            one = P.iLQRController(None, family_model(name, r[b]), qr_cost(spec))
            Z1, U1, s1 = one.fit(U[b:b + 1], encoding=enc, n_iterations=5, z0=z0[b:b + 1], u_min=lo, u_max=hi)
            assert int(s1[0]) == int(state[b]), b
            for a, w in ((Z[b:b + 1], Z1), (Uo[b:b + 1], U1), (K[b:b + 1], one._K)):
                assert close(a, w, torch.float64), b


# ------------------------------------------------------------------------------------------------ 3. the oracle
@pytest.mark.parametrize("name,enc,dtype,bounded", [
    ("pendulum", 0, torch.float64, False), ("pendulum", 1, torch.float64, True), ("pendulum", 2, torch.float64, False),
    ("pendulum", 3, torch.float64, True), ("pendulum", 4, torch.float64, True), ("pendulum", 4, torch.float32, True),
    ("cartpole", 1, torch.float64, True), ("cartpole", 4, torch.float32, False),
    ("double_cartpole", 0, torch.float64, True), ("double_cartpole", 4, torch.float64, False),
    ("rendezvous", 4, torch.float64, True), ("rendezvous", 1, torch.float64, False),
    ("rendezvous", 4, torch.float32, True),
])
def test_matches_oracle_per_problem(name, enc, dtype, bounded):
    got, _, r, (z0, U) = batched_and_singles(name, enc, 0, dtype, bounded, B=5, N=6)
    spec = cost_spec(name)
    lo, hi = bounds(name, bounded)
    tol = 1e-5 if dtype == torch.float64 else 1e-3
    alphas = O.fit_alphas(torch.float64)
    for b in range(z0.shape[0]):
        odyn = SPECS[name](*row_list(name, r[b]))
        lin = O.linearize(z0[b], U[b], odyn, spec, enc, lo, hi)
        want = dict(zip(LIN, lin))
        for n in ("Z", "F_z", "F_u", "L", "L_z", "L_u", "L_zz", "L_uu"):
            assert rel(got[n][b].reshape(want[n].shape), want[n]) <= tol, (n, b)
        Zr, Ur = O.rollout(odyn, lin[0], U[b], got["k"][b].double().cpu(), got["K"][b].double().cpu(), alphas, enc,
                           lo, hi)
        assert rel(got["J_all"][b], O.trajectory_cost(spec, Zr, Ur, enc)) <= tol, b


# --------------------------------------------------------------------------------------------------- 4. isolation
@pytest.mark.parametrize("name,enc,dtype", [("pendulum", 4, torch.float32), ("cartpole", 1, torch.float64),
                                            ("double_cartpole", 4, torch.float64), ("rendezvous", 4, torch.float32)])
def test_changing_one_row_changes_only_that_problem(name, enc, dtype):
    B, N, hit = 6, 8, 2
    r = rows(name, B)
    z0U = inputs(name, enc, B, N)
    base = solve(name, enc, 0, dtype, known(name, r), True, B, N, z0U=z0U)
    r2 = r.clone()
    r2[hit, 1] *= 1.3                                           # a mass
    got = solve(name, enc, 0, dtype, known(name, r2), True, B, N, z0U=z0U, gains=(base["k"], base["K"]))
    others = [b for b in range(B) if b != hit]
    for n in LIN + ("J_opt", "J_all", "Z_new", "U_new"):
        assert torch.equal(got[n][others], base[n][others]), n
    assert not torch.equal(got["Z"][hit], base["Z"][hit]) and not torch.equal(got["F_u"][hit], base["F_u"][hit])


# -------------------------------------------------------------------------------------------- 5. per-step goals
@pytest.mark.parametrize("name,enc,dtype", [("pendulum", 4, torch.float64), ("pendulum", 1, torch.float64),
                                            ("cartpole", 4, torch.float32), ("double_cartpole", 3, torch.float64),
                                            ("rendezvous", 4, torch.float64), ("rendezvous", 1, torch.float64)])
def test_with_per_step_goals_equals_batches_of_one(name, enc, dtype):
    _, D, nu, ang, _, _, _ = GEOS[name]
    B, N = 5, 8
    g = torch.Generator().manual_seed(11)
    xg = (0.5 * torch.randn(B, N + 1, D + len(ang), generator=g, dtype=torch.float64)).to(dtype).cuda()
    ug = (0.2 * torch.randn(B, N, nu, generator=g, dtype=torch.float64)).to(dtype).cuda()
    got, singles, *_ = batched_and_singles(name, enc, 0, dtype, True, B=B, N=N, x_goal=xg, u_goal=ug)
    assert_equals_singles(got, singles, dtype)


# ------------------------------------------------------------------------------------------------- 6. env step
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", list(SPECS))
def test_env_step_per_instance_matches_oracle(name, dtype):
    import pddp_b200 as P
    env_class = P.examples.problems.SampleProblems[name.upper()].get_env_class()
    _, D, nu, _, _, _, _ = GEOS[name]
    B = 7
    r = rows(name, B)
    env = env_class.from_model(family_model(name, r), batch_size=B, dtype=dtype)
    g = torch.Generator().manual_seed(4)
    x = 0.3 * torch.randn(B, D, generator=g, dtype=torch.float64)
    u = 0.5 * torch.randn(B, nu, generator=g, dtype=torch.float64)
    env.set_state(x)
    env.apply(u.cuda())
    got = env.get_state().mean().double().cpu()
    tol = 1e-5 if dtype == torch.float64 else 1e-3
    x_in = x.to(dtype).float().double()              # the simulator keeps its state in float32 (gym_env.py)
    for b in range(B):
        want = O._KNOWN[name](SPECS[name](*row_list(name, r[b])).params, x_in[b], u[b].to(dtype).double())
        assert rel(got[b], want) <= tol, b
    shared = env_class.from_model(family_model(name, r[0]), batch_size=B, dtype=dtype)
    shared.set_state(x)
    shared.apply(u.cuda())
    assert torch.equal(shared.get_state().mean()[0], env.get_state().mean()[0])     # row 0 = the shared system 0


# ------------------------------------------------------------------------------------------------ 7. closed loop
def _pendulum_mpc(model, env, cost, z0, N, H, enc=4):
    import pddp_b200 as P
    from pddp_b200.controllers import _apply_controller
    B = z0.shape[0]
    ctrl = P.iLQRController(env, model, cost)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ctrl.fit(torch.zeros(B, N, 1, dtype=torch.float64, device="cuda"), encoding=enc, n_iterations=10, z0=z0,
                 u_min=torch.tensor([-3.0], device="cuda", dtype=torch.float64),
                 u_max=torch.tensor([3.0], device="cuda", dtype=torch.float64))
        return _apply_controller(env, cost, ctrl, H, enc, True, True)


def test_closed_loop_per_instance_equals_single_instance_loops():
    import pddp_b200 as P
    B, N, H = 4, 12, 15
    masses = torch.tensor([0.6, 0.9, 1.2, 1.6], dtype=torch.float64)
    cost = P.examples.pendulum.PendulumCost().double()
    x0 = 0.1 * torch.randn(B, 2, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    mk = lambda m: P.examples.pendulum.PendulumDynamicsModel(0.1, m=m).double()
    env = P.examples.pendulum.PendulumEnv.from_model(mk(masses), batch_size=B, dtype=torch.float64)
    env.set_state(x0)
    (X, U, dX), J = _pendulum_mpc(mk(masses), env, cost, env.get_state().encode(4), N, H)
    for b in range(B):
        env1 = P.examples.pendulum.PendulumEnv.from_model(mk(masses[b]), batch_size=1, dtype=torch.float64)
        env1.set_state(x0[b:b + 1])
        (X1, U1, dX1), J1 = _pendulum_mpc(mk(masses[b]), env1, cost, env1.get_state().encode(4), N, H)
        for a, w in ((X.reshape(B, H, 2)[b], X1), (U.reshape(B, H, 1)[b], U1), (J[b:b + 1], J1)):
            assert close(a, w, torch.float64), b


def test_matching_model_beats_nominal_model_under_mismatch():
    import pddp_b200 as P
    B, N, H = 16, 20, 40
    g = torch.Generator().manual_seed(7)
    masses = 0.3 * torch.exp(torch.rand(B, generator=g, dtype=torch.float64) * torch.log(torch.tensor(10.0)))
    cost = P.examples.pendulum.PendulumCost().double()
    x0 = 0.05 * torch.randn(B, 2, generator=g, dtype=torch.float64)
    Js = []
    for model in (P.examples.pendulum.PendulumDynamicsModel(0.1, m=masses).double(),
                  P.examples.pendulum.PendulumDynamicsModel(0.1).double()):
        env = P.examples.pendulum.PendulumEnv.from_model(P.examples.pendulum.PendulumDynamicsModel(0.1, m=masses),
                                                         batch_size=B, dtype=torch.float64)
        env.set_state(x0)
        _, J = _pendulum_mpc(model, env, cost, env.get_state().encode(4), N, H)
        Js.append(J)
    assert Js[0].mean() < Js[1].mean(), (Js[0].mean().item(), Js[1].mean().item())


def test_sample_problems_setup_with_a_mass_per_instance():
    import pddp_b200 as P
    env, cost, model = P.examples.problems.SampleProblems.PENDULUM.setup(0.1, m=torch.tensor([0.5, 1.0, 2.0]))
    assert model.n_sets == 3 and env.batch_size == 3
    env.set_state(torch.tensor([[0.5, 0.0]] * 3))
    env.apply(torch.zeros(3, 1, device="cuda"))
    thd = env.get_state().mean()[:, 1].cpu()
    assert torch.allclose(thd, thd[0].expand(3))                # gravity alone: the mass cancels in the pendulum


# -------------------------------------------------------------------------------------- 8. public API and errors
def test_single_problem_api_equals_batch_of_one():
    import pddp_b200 as P
    r = rows("pendulum", 3)
    cost = P.examples.pendulum.PendulumCost().double()
    z0, U = inputs("pendulum", 4, 3, 10)
    z0, U = z0.cuda(), U.cuda()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fam = P.iLQRController(None, family_model("pendulum", r), cost)
        Zb, Ub, sb = fam.fit(U, encoding=4, n_iterations=5, z0=z0)
        one = family_model("pendulum", r[1])
        ctrl = P.iLQRController(None, one, cost)
        Z1, U1, s1 = ctrl.fit(U[1], encoding=4, n_iterations=5, z0=z0[1])
    assert int(s1) == int(sb[1])
    assert close(Z1.unsqueeze(0), Zb[1:2], torch.float64) and close(U1.unsqueeze(0), Ub[1:2], torch.float64)


@pytest.mark.parametrize("name,enc", [("pendulum", 4), ("pendulum", 1), ("double_cartpole", 4), ("rendezvous", 1)])
def test_model_forward_with_one_set_per_row(name, enc):
    B = 5
    r = rows(name, B)
    z0, U = inputs(name, enc, B, 1)
    z, u = z0.cuda(), U[:, 0].cuda()
    got = family_model(name, r)(z, u, 0, encoding=enc)
    for b in range(B):
        want = family_model(name, r[b])(z[b], u[b], 0, encoding=enc)
        assert close(got[b], want, torch.float64), b
        assert rel(got[b], O.known_step(SPECS[name](*row_list(name, r[b])), z0[b], U[b, 0], enc)[0]) <= 1e-5, b


def test_argument_errors_launch_nothing():
    import pddp_b200 as P
    from pddp_b200 import _lib
    from pddp_b200.controllers.ilqr import _control_law, forward
    from pddp_b200.solver import BatchedSolver
    from pddp_b200.utils.evaluation import eval_dynamics
    lib = _lib.load()
    fam = family_model("pendulum", rows("pendulum", 3))
    cost = P.examples.pendulum.PendulumCost().double()
    z0, U = inputs("pendulum", 4, 4, 6)
    z0, U = z0.cuda(), U.cuda()
    torch.cuda.synchronize()
    before = lib.pddp_launch_count()
    ctrl = P.iLQRController(None, fam, cost)
    with pytest.raises(ValueError):
        ctrl.fit(U, encoding=4, n_iterations=2, z0=z0)                 # 3 sets, 4 problems
    with pytest.raises(ValueError):
        ctrl.fit(U[0], encoding=4, n_iterations=2, z0=z0[0])           # one problem, 3 sets
    with pytest.raises(ValueError):
        ctrl.step(z0[:2], U[:2], encoding=4)
    with pytest.raises(ValueError):
        fam(z0[:2], U[:2, 0], 0, encoding=4)
    with pytest.raises(ValueError):
        forward(z0[0], U[0], fam, cost, encoding=4)
    with pytest.raises(ValueError):
        _control_law(fam, torch.zeros(7, 2, dtype=torch.float64, device="cuda"), U[0], U[0], U[0].unsqueeze(-1), 1.0)
    with pytest.raises(ValueError):
        eval_dynamics(fam, z0[0], U[0, 0], 0, encoding=4)
    with pytest.raises(ValueError):
        P.examples.pendulum.PendulumEnv(model=fam)
    with pytest.raises(ValueError):
        P.examples.pendulum.PendulumEnv(model=fam, batch_size=4)
    with pytest.raises(ValueError):
        BatchedSolver(known("pendulum", rows("pendulum", 3)), consts(cost_spec("pendulum")), 4, 4, 6)
    assert lib.pddp_launch_count() == before


# --------------------------------------------------------------------------------------------- 9. sharded fit
def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    import pddp_b200 as P
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    B, N = 37, 12                                              # uneven shards (19 + 18)
    model = family_model("cartpole", rows("cartpole", B)).float()
    spec = cost_spec("cartpole")
    z0, U = inputs("cartpole", 1, B, N)
    kw = dict(encoding=1, n_iterations=6, z0=z0.float().to(dev))
    ctrl = P.iLQRController(None, model, qr_cost(spec).float())
    Zs, Us, ss = ctrl.fit(U.float().to(dev), **kw)
    single = P.iLQRController(None, model, qr_cost(spec).float())
    Z1, U1, s1 = single.fit(U.float().to(dev), shard=False, **kw)
    ok = (torch.equal(Zs, Z1) and torch.equal(Us, U1) and torch.equal(ss, s1) and torch.equal(ctrl._K, single._K))
    torch.save(bool(ok), os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_fit_with_per_problem_parameters_equals_single_gpu_fit(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_sharded_worker, args=(2, 29771, str(tmp_path)), nprocs=2, join=True)
    for rank in range(2):
        assert torch.load(os.path.join(str(tmp_path), "rank%d.pt" % rank)), rank
