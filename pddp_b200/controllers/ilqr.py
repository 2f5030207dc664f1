"""iLQR controller: the reference's controller API on top of the batched GPU solver.

Same class name, constructor / `fit` / `step` / `forward` signatures, callbacks, return values and `iLQRState`
enum as pddp/controllers/ilqr.py, so a script written against the reference keeps working; additionally `U` may
carry a leading problem dimension ([B, N, nu] with z0 [B, nz]) and then B independent problems are optimised
together, each with its own regularisation state -- and, under `torchrun`, split across the GPUs of the job.

The module-level functions `forward`, `Q`, `backward`, `_control_law`, `_trajectory_cost` keep the reference
signatures (single problem, time-major tensors) and call the same kernels with B = 1 on cached buffers.
"""
import warnings
from enum import IntEnum

import torch

from .. import _lib, sharding
from ..models.bnn.modules import check_model_opts
from ..solver import (LIN_NAMES, cached_solver, check_dynamics_rows, check_goals, expand_bound, fit_alphas,
                      require_single_system, step_alphas)
from ..utils.encoding import StateEncoding, decode_mean
from .base import Controller


class iLQRState(IntEnum):
    """ref: pddp/controllers/ilqr.py:35-64"""
    UNDEFINED = 0
    ACCEPTED = 1
    REJECTED = 2
    NOT_PD = 3
    MAX_REG = 4
    CONVERGED = 5

    def should_retry(self):
        return self in (iLQRState.UNDEFINED, iLQRState.NOT_PD, iLQRState.REJECTED)

    def is_terminal(self):
        return self in (iLQRState.CONVERGED, iLQRState.MAX_REG)


def batch_goals(batched, N, x_goal, u_goal):
    """The goals of a call in the batched solver's form.  A batched call passes them through: x_goal [B, DA] or
    [B, N+1, DA], u_goal [B, nu] or [B, N, nu].  A single problem (U [N, nu]) takes only the per-step forms
    x_goal [N+1, DA] / u_goal [N, nu], returned as a batch of one; its fixed goal is its cost's x_goal / u_goal.
    Raises ValueError on a row count that fits neither rule (widths are checked by solver.check_goals)."""
    if batched:
        return x_goal, u_goal
    out = []
    for name, g, Nt in (("x_goal", x_goal, N + 1), ("u_goal", u_goal, N)):
        if g is None:
            out.append(None)
        elif isinstance(g, torch.Tensor) and g.dim() == 2 and g.shape[0] == Nt:
            out.append(g.unsqueeze(0))
        else:
            raise ValueError("a single problem (U [N, nu]) takes a per-step %s of %d rows ([%d, E]), got %s; "
                             "per-problem goals need a batched call (U [B, N, nu])"
                             % (name, Nt, Nt, list(g.shape) if isinstance(g, torch.Tensor) else type(g).__name__))
    return out


def reference_window(ref, i, n, batched):
    """Rows min(i + t, T - 1), t = 0 .. n-1, of a reference with a time axis of length T >= 1 (ref [B, T, E]
    batched, [T, E] unbatched): the goals that MPC step i optimises against, held at the reference's last row past
    its end.  A goal without a time axis ([B, E] batched) and None pass through."""
    if ref is None or ref.dim() != (3 if batched else 2):
        return ref
    T = ref.shape[-2]
    if T < 1:
        raise ValueError("a reference needs at least one row")
    rows = torch.arange(i, i + n, device=ref.device).clamp(max=T - 1)
    return ref.index_select(ref.dim() - 2, rows)


def _bounds(u_min, u_max):
    if (u_min is None) != (u_max is None):
        return None, None       # ref: ilqr.py:461,636 -- bounds apply only when both are given
    return u_min, u_max


class iLQRController(Controller):
    """ref: pddp/controllers/ilqr.py:67-390"""

    def __init__(self, env, model, cost, model_opts={}, cost_opts={}, **kwargs):
        super().__init__()
        self.env, self.model, self.cost = env, model, cost
        self._model_opts, self._cost_opts = model_opts, cost_opts
        check_model_opts(model, model_opts)
        self._Z_nominal = self._U_nominal = self._K = None
        self._solver = None
        self._batched = False

    # regularisation state of problem 0 (the reference keeps python floats, ilqr.py:93-97)
    @property
    def _mu(self):
        return 0.0 if self._solver is None else float(self._solver.mu[0])

    @property
    def _delta(self):
        return 2.0 if self._solver is None else float(self._solver.delta[0])

    def invalidate(self):
        """Drops the device buffers (and the device copies of the model they captured)."""
        self._solver = None

    def _get_solver(self, B, N, encoding, dtype, device, n_alphas, problems=None):
        """Buffers for this problem shape.  The cache is keyed on the model's `_version` (bumped by
        resample / fit / load_reference), and the cost / closed-form model constants are re-read on every call,
        so an edited model or cost is never served from stale device copies.  problems = (lo, hi): the rows of a
        closed-form model's per-problem parameters that this shard solves."""
        if not self._batched:
            require_single_system(self.model, "a single-problem call (U [N, nu])")
        s = cached_solver(self.model, self.cost, encoding, B, N, dtype, device, max_alphas=max(16, n_alphas),
                          model_opts=self._model_opts, problems=problems)
        if s is not self._solver:
            s.view("K_nominal").zero_()
        self._solver = s
        return s

    def _results(self, s):
        """Nominal trajectory, controls and the gains of the last ACCEPTED step (ref: ilqr.py:166-171: `_K` is
        only stored on acceptance; K_nominal is written by pddp_accept_update where accepted[b] is set)."""
        Z, U, K = s.view("Z").clone(), s.view("U").clone(), s.matrices("K_nominal").clone()
        if self._batched:
            self._Z_nominal, self._U_nominal, self._K = Z, U, K
            return Z, U, s.state.clone()
        self._Z_nominal, self._U_nominal, self._K = Z[0], U[0], K[0]
        return Z[0], U[0], iLQRState(int(s.state[0]))

    def step(self, z0, U=None, i=0, encoding=StateEncoding.DEFAULT, batch_rollout=True, alphas=None, u_min=None,
             u_max=None, on_iteration=None, tol=5e-6, max_reg=1e10, _keep_reg=True, x_goal=None, u_goal=None,
             **kwargs):
        """One optimisation step: linearise once, then retry backward + rollout with a larger
        regularisation while the state is NOT_PD / REJECTED (ref: ilqr.py:183-235).  `batch_rollout` is accepted
        for signature compatibility: the kernels always evaluate every alpha and every tangent in parallel.
        x_goal / u_goal give every problem its own goal, fixed or per step (see `fit`)."""
        if U is None:
            U = self._U_nominal
        _lib.require_cuda(U, "U")
        x_goal, u_goal = batch_goals(U.dim() == 3, U.shape[-2], x_goal, u_goal)
        self._batched = U.dim() == 3
        Ub = U if self._batched else U.unsqueeze(0)
        zb = z0.reshape(Ub.shape[0], -1)
        alphas = step_alphas(U.dtype) if alphas is None else alphas
        u_min, u_max = _bounds(u_min, u_max)
        s = self._get_solver(Ub.shape[0], Ub.shape[1], encoding, U.dtype, U.device, int(alphas.numel()))
        mu, delta = s.mu.clone(), s.delta.clone()
        s.set_problem(zb.to(device=U.device, dtype=U.dtype), Ub, u_min, u_max, alphas=alphas, iterations=1,
                      x_goal=x_goal, u_goal=u_goal)
        if _keep_reg:            # regularisation persists across steps of one fit (ilqr.py:277 resets per fit)
            s.mu.copy_(mu)
            s.delta.copy_(delta)
        for _ in range(256):
            s.iterate(tol, max_reg)
            if on_iteration is not None and not self._batched:
                on_iteration(i, iLQRState(int(s.state[0])), s.view("Z")[0].clone(), s.view("U")[0].clone(),
                             s.J_opt[0].clone())
            if int(s.n_active.item()) == 0:
                break
        if bool((s.state == int(iLQRState.MAX_REG)).any()):
            warnings.warn("exceeded max regularization term")
        self._results(s)
        return s.state.clone() if self._batched else iLQRState(int(s.state[0]))

    def fit(self, U, encoding=StateEncoding.DEFAULT, n_iterations=50, tol=5e-6, max_reg=1e10, batch_rollout=True,
            quiet=False, on_iteration=None, u_min=None, u_max=None, z0=None, shard=None, max_passes=None, x_goal=None,
            u_goal=None, **kwargs):
        """ref: pddp/controllers/ilqr.py:237-316.  U: [N, nu] (z0 read from env.get_state() unless
        given) or [B, N, nu] with z0 [B, nz].  Returns (Z, U, state).

        Multi-GPU (SURVEY 8e): with torch.distributed initialised (one process per GPU under torchrun) and a
        batched call, every rank passes the SAME full batch; each optimises its contiguous share of the problems
        -- no collective inside the iteration -- and ONE all-gather at the end gives every rank the full
        (Z, U, K, state).  shard=False keeps the whole batch on this rank.  max_passes bounds the number of
        whole-batch passes (a pass = linearise / backward / rollout / accept for every problem still in play).

        Per-problem goals (batched calls): x_goal [B, DA] in the cost's coordinates -- the angle-augmented state
        for the pendulum family (cartpole: [x, xdot, thetadot, sin theta, cos theta]), the state for rendezvous -- and
        u_goal [B, nu], CUDA tensors.  Per-step goals track a reference: x_goal [B, N+1, DA] (row t = the goal of the
        state at step t, row N with Q_term), u_goal [B, N, nu]; a single problem (U [N, nu]) takes them as
        [N+1, DA] / [N, nu].  x and u choose their form independently; a goal not given is the cost's x_goal /
        u_goal.  A sharded fit splits them like z0.

        Per-problem dynamics (batched calls): a closed-form model whose parameters are 1-D tensors of length B solves
        problem b with parameter set b (KnownDynamicsModel); a sharded fit splits the sets like z0.  A single
        problem needs a model with one set."""
        _lib.require_cuda(U, "U")
        x_goal, u_goal = batch_goals(U.dim() == 3, U.shape[-2], x_goal, u_goal)
        self._batched = U.dim() == 3
        Ub = (U if self._batched else U.unsqueeze(0)).detach()
        if z0 is None:
            z0 = self.env.get_state().encode(encoding).detach()
        zb = z0.to(device=U.device, dtype=U.dtype).reshape(Ub.shape[0], -1)
        u_min, u_max = _bounds(u_min, u_max)
        world, rank = sharding.world_and_rank()
        sharded = self._batched and world > 1 and shard is not False and Ub.shape[0] >= world
        B_total = Ub.shape[0]
        x_goal, u_goal = check_goals(x_goal, u_goal, B_total, self.cost.geometry(), U.dtype, Ub.shape[1])
        problems = None
        if sharded:
            Ub, zb = sharding.shard(Ub, world, rank).contiguous(), sharding.shard(zb, world, rank).contiguous()
            x_goal, u_goal = (None if g is None else sharding.shard(g, world, rank).contiguous() for g in (x_goal, u_goal))
            if not getattr(self.model, "is_bnn", False):
                check_dynamics_rows(self.model.descriptor(), B_total)
                problems = sharding.shard_bounds(B_total, world, rank)      # per-problem parameters split like z0
        s = self._get_solver(Ub.shape[0], Ub.shape[1], encoding, U.dtype, U.device, 10, problems)
        it = [0]

        def on_pass(p, sv):
            if on_iteration is None:
                return
            if self._batched:
                on_iteration(p - 1, sv.state.clone(), sv.view("Z"), sv.view("U"), sv.J_opt)
            else:
                st = iLQRState(int(sv.state[0]))
                on_iteration(it[0], st, sv.view("Z")[0].clone(), sv.view("U")[0].clone(), sv.J_opt[0].clone())
                if not st.should_retry():
                    it[0] += 1

        s.fit(zb, Ub, n_iterations=n_iterations, tol=tol, max_reg=max_reg, u_min=u_min, u_max=u_max,
              alphas=fit_alphas(U.dtype), on_pass=on_pass, max_passes=max_passes, x_goal=x_goal, u_goal=u_goal)
        if bool((s.state == int(iLQRState.MAX_REG)).any()):
            warnings.warn("exceeded max regularization term")
        if not sharded:
            return self._results(s)
        Z, Uo, K, state = sharding.all_gather_problems(
            [s.view("Z").contiguous(), s.view("U").contiguous(), s.matrices("K_nominal").contiguous(), s.state], B_total)
        self._Z_nominal, self._U_nominal, self._K = Z, Uo, K
        return Z, Uo, state

    def forward(self, z, i, encoding=StateEncoding.DEFAULT, mpc=False, ignore_uncertainty=True, u_min=None,
                u_max=None, **kwargs):
        """ref: pddp/controllers/ilqr.py:318-362 -- time-varying feedback law, or one MPC iteration
        from the measured state followed by a left shift of the nominal controls.

        Receding-horizon tracking: under mpc, an x_goal with a time axis ([B, T, DA] batched, [T, DA] for one
        problem) is a reference for the whole trial, of any length T >= 1; MPC step i optimises against its rows
        min(i + t, T - 1), t = 0 .. N (reference_window).  A u_goal with a time axis likewise, t = 0 .. N-1.  Goals
        without one ([B, DA] / [B, nu]) pass through to `step` as they are."""
        if self._U_nominal is None:
            raise RuntimeError("You need to either call fit or initialize _U_nominal")
        if not mpc:
            Un = self._U_nominal[:, i] if self._batched else self._U_nominal[i]
            if self._Z_nominal is None:
                return Un
            Zn = self._Z_nominal[:, i] if self._batched else self._Z_nominal[i]
            Kn = self._K[:, i] if self._batched else self._K[i]
            z = z.to(Zn.device)
            if ignore_uncertainty:
                D = self.model.state_size
                dx = decode_mean(z, encoding, D) - decode_mean(Zn, encoding, D)
                return Un + (Kn[..., :D] @ dx.unsqueeze(-1)).squeeze(-1)
            return Un + (Kn @ (z - Zn).unsqueeze(-1)).squeeze(-1)
        batched, N = self._U_nominal.dim() == 3, self._U_nominal.shape[-2]
        for name, n in (("x_goal", N + 1), ("u_goal", N)):
            if kwargs.get(name) is not None:
                kwargs[name] = reference_window(kwargs[name], i, n, batched)
        self.step(z, i=i, encoding=encoding, u_min=u_min, u_max=u_max, _keep_reg=False, **kwargs)
        if self._batched:
            u = self._U_nominal[:, 0].clone()
            self._U_nominal = torch.cat([self._U_nominal[:, 1:], self._U_nominal[:, -1:]], 1)
        else:
            u = self._U_nominal[0].clone()
            self._U_nominal = torch.cat([self._U_nominal[1:], self._U_nominal[-1:]], 0)
        return u


# ---------------------------------------------------------------------------------------------
# module-level functions with the reference signatures (single problem, B = 1)
# ---------------------------------------------------------------------------------------------
def forward(z0, U, model, cost, encoding=StateEncoding.DEFAULT, batch_rollout=True, model_opts={}, cost_opts={},
            u_min=None, u_max=None):
    """ref: pddp/controllers/ilqr.py:393-486 -> (Z, F_z, F_u, L, L_z, L_u, L_zz, L_uz, L_uu).  One problem, so one
    system: a model with several parameter sets raises ValueError."""
    check_model_opts(model, model_opts)
    require_single_system(model, "pddp_b200.controllers.ilqr.forward")
    _lib.require_cuda(U, "U")
    u_min, u_max = _bounds(u_min, u_max)
    s = cached_solver(model, cost, encoding, 1, U.shape[0], U.dtype, U.device, model_opts=model_opts)
    s.set_problem(z0.reshape(1, -1).to(device=U.device, dtype=U.dtype), U.unsqueeze(0), u_min, u_max)
    s.linearize(use_active=False)
    return tuple(s.matrices(n)[0].clone() for n in LIN_NAMES)


@torch.no_grad()
def Q(F_z, F_u, L_z, L_u, L_zz, L_uz, L_uu, V_z, V_zz):
    """ref: pddp/controllers/ilqr.py:489-526 (host-side helper; the kernels fuse this)."""
    Q_z = L_z + F_z.t().matmul(V_z)
    Q_u = L_u + F_u.t().matmul(V_z)
    Q_zz = L_zz + F_z.t().mm(V_zz).mm(F_z)
    Q_uz = L_uz + F_u.t().mm(V_zz).mm(F_z)
    Q_uu = L_uu + F_u.t().mm(V_zz).mm(F_u)
    return Q_z, Q_u, 0.5 * (Q_zz + Q_zz.t()), Q_uz, 0.5 * (Q_uu + Q_uu.t())


@torch.no_grad()
def backward(Z, F_z, F_u, L, L_z, L_u, L_zz, L_uz, L_uu, reg=0.0, V_zz_reg=False, u_min=None, u_max=None, U=None,
             quiet=False, model=None, cost=None, encoding=None):
    """ref: pddp/controllers/ilqr.py:529-674 -> (k, K); raises RuntimeError where the reference does
    (Q_uu not positive definite / NaN gains / BoxQP failure)."""
    if V_zz_reg:
        raise NotImplementedError("pddp_b200: the V_zz_reg=True branch is never enabled by the reference's callers")
    _lib.require_cuda(Z, "Z")
    N, nu = L_u.shape
    nz = Z.shape[1]
    u_min, u_max = _bounds(u_min, u_max)
    s = _RawBackward(nz, nu, N, Z.dtype, Z.device)
    k, K, status = s.run(F_z, F_u, L_z, L_u, L_zz, L_uz, L_uu, reg, U, u_min, u_max)
    if status != 0:
        raise RuntimeError("non-positive definite matrix")
    return k, K


class _RawBackward:
    """pddp_backward on caller tensors (B = 1): only shapes matter, not the model."""

    def __init__(self, nz, nu, N, dtype, device):
        if not 1 <= nu <= _lib.MAX_NU:
            raise NotImplementedError("pddp_b200.backward: action_size must be in [1, %d], got %d" % (_lib.MAX_NU, nu))
        # pddp_backward ignores geo / enc: the derivative tensors carry everything it needs
        self.shape = _lib.Shape(_lib.dtype_code(dtype), _lib.PROBLEM_MAJOR, 0, 0, 1, N, nz, nu)
        self.N, self.nz, self.nu, self.dtype, self.device = N, nz, nu, dtype, device

    def run(self, F_z, F_u, L_z, L_u, L_zz, L_uz, L_uu, reg, U, u_min, u_max):
        import ctypes as C
        lib, p = _lib.load(), _lib.ptr
        c = lambda t: t.detach().to(self.dtype).contiguous()
        o = dict(dtype=self.dtype, device=self.device)
        k, K = torch.zeros(self.N, self.nu, **o), torch.zeros(self.N, self.nu, self.nz, **o)
        mu = torch.full((1,), float(reg), dtype=torch.float64, device=self.device)
        status = torch.zeros(1, dtype=torch.int32, device=self.device)
        args = [c(t) for t in (F_z, F_u, L_z, L_u, L_zz, L_uz, L_uu)]
        Uc = None if U is None else c(U)
        lo = expand_bound(u_min, self.nu, self.dtype, self.device)     # the reference broadcasts a 1-element bound
        hi = expand_bound(u_max, self.nu, self.dtype, self.device)
        with torch.cuda.device(self.device):
            _lib.check(lib.pddp_backward(C.byref(self.shape), *[p(t) for t in args], p(mu), p(Uc), p(lo), p(hi), None,
                                         p(k), p(K), p(status), _lib.stream_ptr()), "backward")
        return k, K, int(status.item())


@torch.no_grad()
def _control_law(model, Z, U, k, K, alpha, encoding=StateEncoding.DEFAULT, model_opts={}, u_min=None, u_max=None,
                 cost=None):
    """ref: pddp/controllers/ilqr.py:677-723 -> (Z_new [N+1, A, nz], U_new [N, A, nu]) for every
    alpha (the fused kernel only keeps the winner's trajectory, so this reference-shaped wrapper rolls the A
    candidates as A problems of a batch with one alpha each).  One trajectory, so one system: a model with several
    parameter sets raises ValueError (the candidates are rolled as a batch, whose rows are not systems)."""
    check_model_opts(model, model_opts)
    require_single_system(model, "_control_law (its line-search candidates are rolled as the problems of one batch)")
    u_min, u_max = _bounds(u_min, u_max)
    alpha = torch.as_tensor(alpha).reshape(-1)
    s = cached_solver(model, cost, encoding, 1, U.shape[0], U.dtype, U.device, model_opts=model_opts)
    Zs, Us = [], []
    s.set_problem(Z[0].reshape(1, -1), U.unsqueeze(0), u_min, u_max, alphas=alpha[:1])
    s.store("Z", Z.detach().unsqueeze(0))
    s.store("k", k.detach().unsqueeze(0))
    s.store("K", K.detach().reshape(1, K.shape[0], -1))
    for a in alpha:
        s.alphas.copy_(a.reshape(1))
        s.rollout(use_active=False, use_bw_status=False)
        Zs.append(s.view("Z_new")[0].clone())
        Us.append(s.view("U_new")[0].clone())
    if alpha.numel() == 1:
        return Zs[0], Us[0]
    return torch.stack(Zs, 1), torch.stack(Us, 1)


@torch.no_grad()
def _trajectory_cost(cost, Z, U, encoding=StateEncoding.DEFAULT, cost_opts={}):
    """ref: pddp/controllers/ilqr.py:764-791 -> J (scalar, or [A] for Z [N+1, A, nz]).  The reference hands cost_opts
    to the cost; here they may carry per-trajectory goals: for Z [N+1, B, nz], cost_opts["x_goal"] [B, DA] /
    cost_opts["u_goal"] [B, nu] give trajectory b its own goal, and x_goal [B, N+1, DA] / u_goal [B, N, nu] (problem
    major, as in iLQRController.fit) a goal per step; for an unbatched Z [N+1, nz], [N+1, DA] / [N, nu]."""
    batched = Z.dim() == 3
    x_goal, u_goal = batch_goals(batched, U.shape[0], cost_opts.get("x_goal"), cost_opts.get("u_goal"))
    Zb = Z.permute(1, 0, 2) if batched else Z.unsqueeze(0)
    Ub = U.permute(1, 0, 2) if batched else U.unsqueeze(0)
    s = cached_solver(None, cost, encoding, Zb.shape[0], Ub.shape[1], Z.dtype, Z.device, layout=_lib.PROBLEM_MAJOR)
    s.set_goals(x_goal, u_goal)
    s.store("Z", Zb.detach())
    s.store("U", Ub.detach())
    try:
        s.cost_only()
    finally:
        s.set_goals()           # the solver is cached and shared with cost-only entry points that take no goals
    J = s.J_opt.clone()
    return J if batched else J[0]


__all__ = ["iLQRController", "iLQRState", "StateEncoding", "forward", "Q", "backward", "_control_law",
           "_trajectory_cost"]
