"""Learned (MC-dropout BNN) dynamics on the rendezvous geometry: D = 8, action_size 4, no angles -- the one shipped
problem with more than one control.  Every kernel of the BNN path (particle MLP with 4 control inputs and 4 control
tangents, moment-matching linearisation with F_u of width 4, the line-search rollout with a 4 x nz gain, the
rendezvous QR cost, training with input width 12) is compared with the CPU oracle evaluated at test time.  The oracle
is pinned to the reference on each ingredient (the bnn_* fixtures: BNN forward under every model option; the
known_rendezvous_* fixtures: the rendezvous cost and the nu = 4 backward pass with box QP), and nu enters the BNN
forward only as the width of cat([x, u]).

Every batch has several problems with different z0 and U, so a wrong per-problem stride of the controls shows up.
Tolerances: fp64 1e-5 relative; fp32 1e-3, with the ReLU-kink allowance of test_gpu_bench_shape.py on
derivative-like outputs (max(1e-3, 4 x the oracle's own fp32-vs-fp64 spread of that problem))."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

D, NU = 8, 4
START = torch.tensor([-10.0, -10.0, 10.0, 10.0, 0.0, -5.0, 5.0, 0.0])     # ref: examples/rendezvous/env.py:106-108
U_MIN = torch.tensor([-0.5, -0.3, -0.4, -0.2])
U_MAX = torch.tensor([0.4, 0.5, 0.3, 0.2])
LIN = ("Z", "F_z", "F_u", "L", "L_z", "L_u", "L_zz", "L_uz", "L_uu")
VALUES = ("Z", "L", "L_z", "L_u", "L_zz", "L_uz", "L_uu")


def rel_err(a, b):
    a, b = torch.as_tensor(a).double().reshape(-1).cpu(), torch.as_tensor(b).double().reshape(-1).cpu()
    if not torch.isfinite(a).all():
        return float("inf")
    return ((a - b).abs().max() / max(1.0, b.abs().max().item())).item()


def synth(P, H, seed):
    """Network initialised like the reference's bayesian_model (Xavier-normal, ReLU gain; modules.py:797-849) with
    input width D + nu = 12, concrete-dropout eval masks and standardised eps0 -- fp64."""
    g = torch.Generator().manual_seed(seed)
    dims = [D + NU, H, H, 2 * D]
    W, b = [], []
    for din, dout in zip(dims[:-1], dims[1:]):
        W.append(torch.randn(dout, din, generator=g, dtype=torch.float64) * math.sqrt(2.0) * math.sqrt(2.0 / (din + dout)))
        b.append(torch.rand(dout, generator=g, dtype=torch.float64) * 0.2 - 0.1)
    W[-1] *= 0.02
    b[-1] *= 0.02
    masks = []
    for _ in range(2):
        r = torch.rand(P, H, generator=g, dtype=torch.float64).clamp(1e-6, 1 - 1e-6)
        masks.append(torch.sigmoid((r.log() - (1 - r).log()) / 0.1))
    eps = torch.randn(P, D, generator=g, dtype=torch.float64)
    return W, b, masks, (eps - eps.mean(0)) / eps.std(0)


def inputs(B, N, enc, seed):
    """Different start state, covariance and controls for every problem."""
    import pddp_oracle as O
    g = torch.Generator().manual_seed(seed)
    M = START.double() + 0.5 * torch.randn(B, D, generator=g, dtype=torch.float64)
    A = 0.1 * torch.randn(B, D, D, generator=g, dtype=torch.float64)
    C = A @ A.mT + 1e-2 * torch.eye(D, dtype=torch.float64)
    if enc == O.IGNORE_UNCERTAINTY:
        z0 = M
    elif enc in (O.FULL_COVARIANCE_MATRIX, O.UPPER_TRIANGULAR_CHOLESKY):
        z0 = torch.stack([O.encode(M[i], C=C[i], enc=enc) for i in range(B)])
    else:
        z0 = torch.stack([O.encode(M[i], V=C[i].diagonal(), enc=enc) for i in range(B)])
    U = 0.4 * torch.randn(B, N, NU, generator=g, dtype=torch.float64)
    return z0, U


def cost_spec(dtype=torch.float64):
    import bench
    import pddp_oracle as O
    Q, R, Qt, goal = bench.cost_constants("rendezvous", dtype)
    return O.QRCostSpec(Q, R, Qt, goal, torch.zeros(NU, dtype=dtype), D, (), tuple(range(D)))


def cost_constants():
    import bench
    from pddp_b200.solver import QRCostConstants
    return QRCostConstants(*bench.cost_constants("rendezvous"))


def solver(net, enc, B, N, dtype, **dyn_kw):
    from pddp_b200 import _lib
    from pddp_b200.solver import BatchedSolver, BNNDynamics
    W, b, masks, eps0 = net
    return BatchedSolver(BNNDynamics(_lib.GEO_RENDEZVOUS, W, b, masks, eps0, **dyn_kw), cost_constants(), enc, B, N,
                         dtype=dtype)


def oracle_dyn(net, dtype=torch.float64, **kw):
    import pddp_oracle as O
    W, b, masks, eps0 = net
    return O.BNNSpec(list(zip(W, b)), masks, eps0, D, NU, (), tuple(range(D)), **kw).to(dtype)


def bounds(bounded, dtype):
    return (U_MIN.to(dtype), U_MAX.to(dtype)) if bounded else (None, None)


# ---------------------------------------------------------------------------------------------------------------
# 1. linearisation: all five encodings, bounded / unbounded, SIMT (H = 32) and H = 200, P = 13 / 50, fp64 and fp32
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("P,H", [(13, 32), (50, 200)])
@pytest.mark.parametrize("bounded", [False, True])
@pytest.mark.parametrize("enc", [0, 1, 2, 3, 4])
def test_linearize_matches_oracle(enc, bounded, P, H, dtype):
    import pddp_oracle as O
    B, N = 3, 4
    net = synth(P, H, seed=10 + enc)
    z0, U = inputs(B, N, enc, seed=20 + enc)
    lo, hi = bounds(bounded, torch.float64)
    s = solver(net, enc, B, N, dtype)
    s.set_problem(z0.to(dtype).cuda(), U.to(dtype).cuda(), *(bounds(bounded, dtype) if bounded else (None, None)))
    s.linearize()
    torch.cuda.synchronize()
    assert int(s.lin_status.abs().sum()) == 0
    got = {n: s.matrices(n).cpu() for n in LIN}
    cost64, dyn64 = cost_spec(), oracle_dyn(net)
    for i in range(B):
        o64 = dict(zip(LIN, O.linearize(z0[i], U[i], dyn64, cost64, enc, lo, hi)))
        if dtype == torch.float64:
            for n in LIN:
                assert rel_err(got[n][i], o64[n]) <= 1e-5, (n, i, rel_err(got[n][i], o64[n]))
            continue
        lo32, hi32 = bounds(bounded, torch.float32)
        o32 = dict(zip(LIN, O.linearize(z0[i].float(), U[i].float(), oracle_dyn(net, torch.float32),
                                        cost_spec(torch.float32), enc, lo32, hi32)))
        for n in VALUES:
            assert rel_err(got[n][i], o64[n]) <= 1e-3, (n, i, rel_err(got[n][i], o64[n]))
        for n in ("F_z", "F_u"):
            allow = max(1e-3, 4.0 * rel_err(o32[n], o64[n]))
            assert rel_err(got[n][i], o64[n]) <= allow, (n, i, rel_err(got[n][i], o64[n]), allow)


def test_bnn_shape_with_wrong_nu_is_rejected():
    """The C ABI takes nu from pddp_shape: a rendezvous BNN call with nu != 4 fails loudly."""
    import ctypes as C
    from pddp_b200 import _lib
    s = solver(synth(13, 32, 0), 1, 2, 3, torch.float64)
    shape = _lib.Shape(*[getattr(s.shape, f) for f, _ in _lib.Shape._fields_])
    shape.nu = 1
    assert s.lib.pddp_bnn_workspace_bytes(C.byref(shape), C.byref(s.c_bnn), 1) < 0


# ---------------------------------------------------------------------------------------------------------------
# 2. backward pass + line-search rollout
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P,H", [(13, 32), (50, 200)])
@pytest.mark.parametrize("bounded", [False, True])
@pytest.mark.parametrize("enc", [0, 1, 4])
def test_backward_and_rollout_match_oracle(enc, bounded, P, H):
    import pddp_oracle as O
    B, N, mu = 3, 5, 1.0
    net = synth(P, H, seed=30 + enc)
    z0, U = inputs(B, N, enc, seed=40 + enc)
    lo, hi = bounds(bounded, torch.float64)
    s = solver(net, enc, B, N, torch.float64)
    s.set_problem(z0.cuda(), U.cuda(), lo, hi)
    s.mu.fill_(mu)
    s.linearize(); s.backward(); s.rollout()
    torch.cuda.synchronize()
    assert int(s.lin_status.abs().sum()) == 0 and int(s.bw_status.abs().sum()) == 0
    cost, dyn = cost_spec(), oracle_dyn(net)
    alphas = O.fit_alphas(torch.float64)
    for i in range(B):
        lin = O.linearize(z0[i], U[i], dyn, cost, enc, lo, hi)
        k, K = O.backward_pass(*lin, reg=mu, u_min=lo, u_max=hi, U=U[i], symmetric_eig=True)
        Zb, Ub = O.rollout(dyn, lin[0], U[i], k, K, alphas, enc, lo, hi)
        J = O.trajectory_cost(cost, Zb, Ub, enc)
        a = int(J.argmin())
        assert rel_err(s.matrices("k").cpu()[i], k) <= 1e-5
        assert rel_err(s.matrices("K").cpu()[i], K) <= 1e-5
        assert rel_err(s.J_all.cpu()[i], J) <= 1e-5
        assert int(s.amin.cpu()[i]) == a
        assert rel_err(s.view("Z_new").cpu()[i], Zb[:, a]) <= 1e-5
        assert rel_err(s.view("U_new").cpu()[i], Ub[:, a]) <= 1e-5
        if bounded:
            Un = s.view("U_new").cpu()[i]
            assert bool((Un >= U_MIN.double()).all()) and bool((Un <= U_MAX.double()).all())


# ---------------------------------------------------------------------------------------------------------------
# 3. fit: state sequence, mu, J, Z and U against the oracle's fit, fp64
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bounded", [False, True])
def test_fit_trace_matches_oracle(bounded):
    import pddp_oracle as O
    B, N, iters, enc = 3, 6, 4, 1
    net = synth(13, 32, seed=50)
    z0, U = inputs(B, N, enc, seed=51)
    lo, hi = bounds(bounded, torch.float64)
    s = solver(net, enc, B, N, torch.float64)
    trace = []
    Z, Uo, _ = s.fit(z0.cuda(), U.cuda(), n_iterations=iters, u_min=lo, u_max=hi,
                     on_pass=lambda p, sv: trace.append((sv.state.cpu().clone(), sv.J_opt.cpu().clone(),
                                                         sv.mu.cpu().clone())))
    torch.cuda.synchronize()
    for i in range(B):
        ilqr = O.ILQR(oracle_dyn(net), cost_spec(), enc)
        want = []
        oZ, oU, _ = ilqr.fit(z0[i], U[i], n_iterations=iters, u_min=lo, u_max=hi, trace=want)
        assert len(want) >= 2 and len(trace) >= len(want)
        for p, (st, J, mu) in enumerate(want):
            assert int(trace[p][0][i]) == st, (i, p)
            assert abs(float(trace[p][1][i]) - J) <= 1e-5 * max(1.0, abs(J)), (i, p)
            assert abs(float(trace[p][2][i]) - mu) <= 1e-9 * max(1.0, mu), (i, p)
        assert rel_err(Z.cpu()[i], oZ) <= 1e-5 and rel_err(Uo.cpu()[i], oU) <= 1e-5


# ---------------------------------------------------------------------------------------------------------------
# 4. model options on this geometry
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("option", ["resample_inputs", "mean_inputs", "predicted_std", "predicted_std_independent"])
def test_model_options_match_oracle(option):
    import pddp_oracle as O
    from pddp_b200 import _lib
    B, N, P, enc = 3, 4, 13, 1
    net = synth(P, 32, seed=60)
    g = torch.Generator().manual_seed(61)
    eps = torch.randn(N, P, D, generator=g, dtype=torch.float64)
    eps = (eps - eps.mean(1, keepdim=True)) / eps.std(1, keepdim=True)
    dyn_kw, o_kw = {}, {}
    if option == "resample_inputs":                      # infer_noise_variables=False
        eps[0] = net[3]
        dyn_kw, o_kw = dict(input_mode=_lib.BNN_INPUT_RESAMPLE, eps_in=eps), dict(input_mode="resample", eps_in=eps)
    elif option == "mean_inputs":                        # sample_input_distribution=False
        dyn_kw, o_kw = dict(input_mode=_lib.BNN_INPUT_MEAN), dict(input_mode="mean")
    else:                                                # use_predicted_std=True (+ independent_noise)
        ind = option.endswith("independent")
        dyn_kw, o_kw = dict(eps_out=eps, independent_noise=ind), dict(eps_out=eps, independent_noise=ind)
    z0, U = inputs(B, N, enc, seed=62)
    lo, hi = bounds(True, torch.float64)
    s = solver(net, enc, B, N, torch.float64, **dyn_kw)
    s.set_problem(z0.cuda(), U.cuda(), lo, hi)
    s.mu.fill_(1.0)
    s.linearize(); s.backward(); s.rollout()
    torch.cuda.synchronize()
    assert int(s.lin_status.abs().sum()) == 0 and int(s.bw_status.abs().sum()) == 0
    cost, dyn = cost_spec(), oracle_dyn(net, **o_kw)
    for i in range(B):
        lin = O.linearize(z0[i], U[i], dyn, cost, enc, lo, hi)
        for n, want in zip(LIN, lin):
            assert rel_err(s.matrices(n).cpu()[i], want) <= 1e-5, (n, i)
        k, K = O.backward_pass(*lin, reg=1.0, u_min=lo, u_max=hi, U=U[i], symmetric_eig=True)
        Zb, Ub = O.rollout(dyn, lin[0], U[i], k, K, O.fit_alphas(torch.float64), enc, lo, hi)
        J = O.trajectory_cost(cost, Zb, Ub, enc)
        assert rel_err(s.J_all.cpu()[i], J) <= 1e-5
        a = int(J.argmin())
        assert int(s.amin.cpu()[i]) == a and rel_err(s.view("U_new").cpu()[i], Ub[:, a]) <= 1e-5


# ---------------------------------------------------------------------------------------------------------------
# 5. tcgen05 MLP (fp32) against the fp64 SIMT path at a large batch
# ---------------------------------------------------------------------------------------------------------------
def test_tc_matches_fp64_at_large_batch():
    B, N, enc = 1024, 8, 1
    net = synth(50, 200, seed=70)
    z0, U = inputs(B, N, enc, seed=71)
    lo, hi = U_MIN.double(), U_MAX.double()
    out = {}
    for dtype in (torch.float64, torch.float32):
        s = solver(net, enc, B, N, dtype)
        s.set_problem(z0.to(dtype).cuda(), U.to(dtype).cuda(), lo.to(dtype), hi.to(dtype))
        s.mu.fill_(1.0)
        s.linearize(); s.backward(); s.rollout()
        torch.cuda.synchronize()
        assert int(s.lin_status.abs().sum()) == 0 and int(s.bw_status.abs().sum()) == 0
        out[dtype] = {n: s.matrices(n).clone() for n in ("Z", "F_z", "F_u", "L", "L_z", "L_zz", "k", "K", "Z_new", "U_new")}
        out[dtype]["J"] = s.J_all.clone()

    def scale_err(a, b, per_problem=False):            # as test_gpu_bnn_tc.py
        a, b = a.double().cpu(), b.double().cpu()
        e = (a - b).abs() / b.abs().max().clamp_min(1e-30)
        return e.reshape(e.shape[0], -1).max(1).values if per_problem else e.max().item()

    errs = {n: scale_err(out[torch.float32][n], out[torch.float64][n]) for n in out[torch.float64]}
    print("rendezvous tcgen05 vs fp64", {k: "%.1e" % v for k, v in errs.items()})
    for n in ("Z", "L", "L_z", "L_zz", "Z_new", "J"):
        assert errs[n] < 1e-3, (n, errs[n])
    for n in ("F_z", "F_u", "k", "K", "U_new"):
        per = scale_err(out[torch.float32][n], out[torch.float64][n], per_problem=True)
        assert per.median() < 1e-4, (n, per.median())
        assert (per < 1e-3).float().mean() >= 0.85, (n, per)
        assert errs[n] < 5e-2, (n, errs[n])


# ---------------------------------------------------------------------------------------------------------------
# 6. dropout masks are per-particle rows
# ---------------------------------------------------------------------------------------------------------------
def test_mask_rows_are_per_particle():
    """Permuting (mask0, mask1, eps0) together leaves Z unchanged; permuting only the masks changes it."""
    B, N, P, enc = 3, 4, 13, 1
    W, b, masks, eps0 = synth(P, 32, seed=80)
    z0, U = inputs(B, N, enc, seed=81)
    perm = torch.randperm(P, generator=torch.Generator().manual_seed(0))
    outs = []
    for net in ((W, b, masks, eps0), (W, b, [m[perm] for m in masks], eps0[perm]), (W, b, [m[perm] for m in masks], eps0)):
        s = solver(net, enc, B, N, torch.float64)
        s.set_problem(z0.cuda(), U.cuda())
        s.linearize()
        outs.append(s.view("Z").cpu().clone())
    assert rel_err(outs[1], outs[0]) <= 1e-12
    assert rel_err(outs[2], outs[0]) > 1e-8


# ---------------------------------------------------------------------------------------------------------------
# 7. training with input width 12
# ---------------------------------------------------------------------------------------------------------------
def test_training_matches_oracle():
    import pddp_oracle as O
    from pddp_b200.models.bnn import bnn_dynamics_model_factory
    g = torch.Generator().manual_seed(90)
    n, bs, iters, hidden = 96, 32, 5, [24, 20]
    X = START.double() + torch.randn(n, D, generator=g, dtype=torch.float64)
    U = torch.randn(n, NU, generator=g, dtype=torch.float64)
    dX = 0.1 * torch.randn(n, D, generator=g, dtype=torch.float64) + 0.05 * X.roll(1, -1) + 0.1 * U.repeat(1, 2)
    batch = torch.stack([torch.randperm(n, generator=g)[:bs] for _ in range(iters)])
    batch[:, -3:] = -1                                                # empty slots
    noise = torch.rand(iters, bs, sum(hidden), generator=g, dtype=torch.float64).clamp(1e-6, 1 - 1e-6)
    default = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        Model = bnn_dynamics_model_factory(D, NU, hidden, [], list(range(D)))
        model = Model(n_particles=10)
    finally:
        torch.set_default_dtype(default)
    p0 = model.flat_parameters().clone()
    args = dict(batch_size=bs, reg_scale=1.0, learning_rate=1e-3, quiet=True, return_diagnostics=True)
    loss, grads = model.fit(X, U, dX, n_iter=1, batch_indices=batch[:1], noise=noise[:1], **args)
    X_ = torch.cat([X, U], -1)
    Xm, Xs, dXm, dXs = X_.mean(0), X_.std(0), dX.mean(0), dX.std(0)
    common = dict(reg=1.0, rate=0.5, X_mean=Xm, X_std_inv=Xs.reciprocal(), dX_mean=dXm, dX_std=dXs)
    _, g0, l0 = O.bnn_train(p0, X_, dX, batch[:1], noise[:1], hidden, D, 0, 1e-3, 1.0, **common)
    assert abs(float(loss[0]) - float(l0[0])) <= 1e-9 * max(1.0, abs(float(l0[0])))
    assert float((grads.cpu() - g0).abs().max()) <= 1e-9 * max(1.0, float(g0.abs().max()))
    model._store_flat(p0)
    model.fit(X, U, dX, n_iter=iters, batch_indices=batch, noise=noise, **args)
    pf, _, _ = O.bnn_train(p0, X_, dX, batch, noise, hidden, D, 0, 1e-3, 1.0, **common)
    p = model.flat_parameters().cpu()
    assert float((p - pf).abs().max()) <= 1e-7
    assert float((p - p0).abs().max()) > 1e-4


# ---------------------------------------------------------------------------------------------------------------
# 8. the public API end to end
# ---------------------------------------------------------------------------------------------------------------
def test_pddp_controller_end_to_end():
    """RendezvousEnv -> bnn_dynamics_model_factory(8, 4, ...) -> PDDPController.train() -> fit -> an MPC trial, all on
    the device (the flow of INTEGRATION.md, with the rendezvous problem's four controls)."""
    import warnings
    import pddp_b200 as P
    torch.manual_seed(0)
    torch.set_default_device("cuda")
    try:
        N, DT = 20, 0.1
        enc = P.StateEncoding.DEFAULT
        UMIN, UMAX = -torch.ones(NU), torch.ones(NU)
        cost = P.examples.rendezvous.RendezvousCost()
        env = P.examples.rendezvous.RendezvousEnv(dt=DT, render=False)
        mc = P.examples.rendezvous.RendezvousDynamicsModel
        model = P.models.bnn.bnn_dynamics_model_factory(env.state_size, env.action_size, [200, 200],
                                                        mc.angular_indices, mc.non_angular_indices)(n_particles=50)
        assert model.action_size == 4 and model.model.fc_0.in_features == 12
        controller = P.controllers.PDDPController(env, model, cost, training_opts={"n_iter": 200, "learning_rate": 1e-3})
        controller.train()
        J_hist, trials = [], []
        U0 = (UMAX - UMIN) * torch.rand(N, NU) + UMIN
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            Z, U, state = controller.fit(U0, encoding=enc, n_iterations=4, max_trials=3, u_min=UMIN, u_max=UMAX,
                                         quiet=True, on_iteration=lambda it, st, Z, U, J: J_hist.append((it, float(J))),
                                         on_trial=lambda t, X, U: trials.append((tuple(X.shape), tuple(U.shape))))
        assert Z.shape == (N + 1, 44) and U.shape == (N, NU)
        assert Z.is_cuda and bool(torch.isfinite(Z).all()) and bool(torch.isfinite(U).all())
        assert bool((U >= UMIN).all()) and bool((U <= UMAX).all())
        assert len(trials) == 3 and trials[-1] == ((2 * N, D), (2 * N, NU))   # 2 initial trials + 1 MPC trial
        assert all(math.isfinite(j) for _, j in J_hist)
        # the passes of the fit on the trained model come first (iteration numbers never decrease: a retried pass
        # repeats its number); the MPC trial's re-plans from other states follow, numbered by time step from 0 again
        fit = [J_hist[0][1]]
        for (i0, _), (i1, j) in zip(J_hist, J_hist[1:]):
            if i1 < i0:
                break
            fit.append(j)
        assert len(fit) >= 2 and fit[-1] <= fit[0]
        env.close()
    finally:
        torch.set_default_device(None)
