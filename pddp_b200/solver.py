"""Batched iLQR / PDDP iteration on the GPU: B independent problems advance together, one pass =
linearise -> backward Riccati -> rollout with parallel line search -> per-problem accept/reject.

This is the host side of the hot path: it owns the device buffers (laid out once, reused by every
pass), marshals pointers into the C ABI and never touches the data itself.  There is no CPU path.

ref: pddp/controllers/ilqr.py:102-316 (what one problem's `step`/`fit` do; here vectorised over B
with per-problem mu/delta/state, SURVEY.md section 5 "failure detection" row).
"""
import collections
import ctypes as C
import functools
import weakref

import torch

from . import _lib
from .utils.encoding import StateEncoding, infer_encoded_state_size

LIN_NAMES = ("Z", "F_z", "F_u", "L", "L_z", "L_u", "L_zz", "L_uz", "L_uu")


def on_own_device(method):
    """Runs a method with the object's device current: the C ABI launches on the CURRENT device and
    torch.cuda.current_stream() is per device, so a solver on cuda:1 must not launch on cuda:0."""
    @functools.wraps(method)
    def wrapped(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return method(self, *args, **kwargs)
    return wrapped


def expand_bound(u, nu, dtype, device):
    """u_min / u_max as the kernels read them: a contiguous [nu] vector.  The reference broadcasts a
    scalar or 1-element bound in clamp() and in `u_min - U[i]` (ilqr.py:461-462, 649-651)."""
    if u is None:
        return None
    u = torch.as_tensor(u, dtype=dtype).reshape(-1)
    if u.numel() not in (1, nu):
        raise ValueError("control bounds must have 1 or action_size=%d elements, got %d" % (nu, u.numel()))
    return u.expand(nu).to(device).contiguous()


def fit_alphas(dtype=torch.float32, device=None, n=10):
    """Line-search candidates of `fit`: 1.025 ** -(j^2), j < n.  ref: pddp/controllers/ilqr.py:282"""
    return (1.025 ** (-torch.arange(float(n), dtype=torch.float64) ** 2)).to(dtype=dtype,
                                                                             device=device)


def step_alphas(dtype=torch.float32, device=None):
    """Default candidates of `step` / MPC: 10 ** linspace(0,-3,11).  ref: ilqr.py:189"""
    return (10.0 ** torch.linspace(0, -3, 11, dtype=torch.float64)).to(dtype=dtype, device=device)


class KnownDynamics:
    """Closed-form dynamics constants (ref: pddp/examples/<problem>/model.py constructors).  `params` is the one
    system every problem integrates; `params_b` [B, 8], if given, gives problem b its own system instead: row b holds
    its parameters in the order of `params` (trailing entries unused)."""

    def __init__(self, geo, params, params_b=None):
        self.geo = geo
        self.params = [float(p) for p in params]
        self.is_bnn = False
        if params_b is not None:
            params_b = (params_b if isinstance(params_b, torch.Tensor) else torch.as_tensor(params_b)).detach()
            if params_b.dim() != 2 or params_b.shape[1] != 8 or params_b.shape[0] < 1:
                raise ValueError("per-problem dynamics parameters must have shape [B, 8], got %s"
                                 % list(params_b.shape))
        self.params_b = params_b

    @property
    def n_sets(self):
        """Number of parameter sets: 1 (shared by every problem) or the B rows of params_b."""
        return 1 if self.params_b is None else int(self.params_b.shape[0])

    def rows(self, lo, hi):
        """The dynamics of problems [lo, hi) (a shard of the batch)."""
        return self if self.params_b is None else KnownDynamics(self.geo, self.params, self.params_b[lo:hi])

    def c_struct(self, p_b=None):
        """pddp_known_dynamics; p_b = the device copy of params_b the kernels read (BatchedSolver keeps it)."""
        s = _lib.KnownDynamicsBatch()
        for i, p in enumerate(self.params):
            s.p[i] = p
        s.p_b = None if p_b is None else p_b.data_ptr()
        return s


def require_single_system(model, what):
    """Raises ValueError when a closed-form model carries more than one parameter set: `what` evaluates one system."""
    n = 1 if model is None or getattr(model, "is_bnn", False) else model.n_sets
    if n != 1:
        raise ValueError("%s evaluates one system, but the model carries %d parameter sets; per-problem dynamics run in "
                         "batched calls (iLQRController.fit / step with U [B, N, nu], model(z [B, nz], u, i), "
                         "KnownDynamicsEnv(model, batch_size=B))" % (what, n))


def check_dynamics_rows(dyn, B):
    """Raises ValueError unless a closed-form model's parameter sets fit a batch of B problems: one set (shared) or
    B sets (one per problem)."""
    n = dyn.n_sets
    if n != 1 and n != B:
        raise ValueError("the dynamics carry %d parameter sets, the batch has %d problem%s: per-problem parameters need "
                         "one row per problem" % (n, B, "" if B == 1 else "s"))


class BNNDynamics:
    """Eval-mode MC-dropout BNN: weights, persistent dropout masks [P,H] and eps_in[0] [P,D]
    (ref: pddp/models/bnn/modules.py:287-386; SURVEY quirks 8-12).  Two hidden layers."""

    def __init__(self, geo, weights, biases, masks, eps0, X_mean=None, X_std_inv=None,
                 dX_mean=None, dX_std=None, input_mode=_lib.BNN_INPUT_INFER, eps_in=None, eps_out=None,
                 independent_noise=False):
        if len(weights) != 3 or len(biases) != 3 or len(masks) != 2:
            raise NotImplementedError("pddp_b200: the BNN path supports exactly two hidden layers")
        self.geo = geo
        self.is_bnn = True
        self.tensors = dict(W0=weights[0], W1=weights[1], W2=weights[2], b0=biases[0], b1=biases[1],
                            b2=biases[2], mask0=masks[0], mask1=masks[1], eps0=eps0, X_mean=X_mean,
                            X_std_inv=X_std_inv, dX_mean=dX_mean, dX_std=dX_std, eps_in=eps_in, eps_out=eps_out)
        # eps_out [N,P,D] given = use_predicted_std=True (ref: modules.py:242-262)
        self.independent_noise = bool(independent_noise)
        # input particles of step i (ref: modules.py:320-358): INFER (default), RESAMPLE = eps_in[i] [N,P,D]
        # at every step (infer_noise_variables=False), MEAN (sample_input_distribution=False)
        self.input_mode = int(input_mode)
        self.P = int(eps0.shape[0])
        self.H0, self.H1 = int(weights[0].shape[0]), int(weights[1].shape[0])
        D, nu, ang, _ = _lib.GEO_INFO[geo]
        DA = D + len(ang)
        if tuple(weights[0].shape) != (self.H0, DA + nu) or tuple(weights[1].shape) != (self.H1, self.H0) \
                or tuple(weights[2].shape) != (2 * D, self.H1):
            raise ValueError("BNN weight shapes do not match the geometry")
        if tuple(masks[0].shape) != (self.P, self.H0) or tuple(masks[1].shape) != (self.P, self.H1) \
                or tuple(eps0.shape) != (self.P, D):
            raise ValueError("BNN mask / eps0 shapes must be [P,H] / [P,D]")
        if self.input_mode == _lib.BNN_INPUT_RESAMPLE and (
                eps_in is None or eps_in.dim() != 3 or tuple(eps_in.shape[1:]) != (self.P, D)):
            raise ValueError("BNN_INPUT_RESAMPLE needs eps_in [N,P,D]")
        if eps_out is not None and (eps_out.dim() != 3 or tuple(eps_out.shape[1:]) != (self.P, D)):
            raise ValueError("eps_out must be [N,P,D]")
        self._device_copies = {}

    def c_struct(self, dtype, device):
        key = (dtype, str(device))
        if key not in self._device_copies:
            self._device_copies[key] = {
                k: None if v is None else torch.as_tensor(v).detach().to(dtype=dtype, device=device).contiguous()
                for k, v in self.tensors.items()}
        t = self._device_copies[key]
        s = _lib.BNN()
        s.P, s.H0, s.H1 = self.P, self.H0, self.H1
        s.input_mode = self.input_mode
        s.independent_noise = int(self.independent_noise)
        for k, v in t.items():
            setattr(s, k, None if v is None else v.data_ptr())
        return s


def check_goal_shapes(x_goal, u_goal, B, geo, N=None):
    """The shape rules of per-problem and per-step goals; raises ValueError on any other shape.  x_goal is [B, DA] on
    the angle-augmented state, or with N given also [B, N+1, DA] (row t = the goal of the state at step t, row N the
    terminal one); u_goal is [B, nu], or with N given [B, N, nu].  Returns, for x and u, whether the goal is per step
    (None where no goal is given)."""
    D, nu, ang, _ = _lib.GEO_INFO[geo]
    out = []
    for name, g, E, Nt in (("x_goal", x_goal, D + len(ang), None if N is None else N + 1),
                           ("u_goal", u_goal, nu, N)):
        if g is None:
            out.append(None)
        elif tuple(g.shape) == (B, E):
            out.append(False)
        elif Nt is not None and tuple(g.shape) == (B, Nt, E):
            out.append(True)
        elif Nt is None:
            raise ValueError("per-problem %s must have shape [B, %d] = [%d, %d], got %s" % (name, E, B, E, list(g.shape)))
        else:
            raise ValueError("%s must have shape [B, %d] = [%d, %d] (per problem) or [B, %d, %d] = [%d, %d, %d] (per "
                             "step), got %s" % (name, E, B, E, Nt, E, B, Nt, E, list(g.shape)))
    return out


def check_goals(x_goal, u_goal, B, geo, dtype, N=None):
    """Per-problem (and, with N given, per-step) goals as the kernels read them -- shapes as in check_goal_shapes --
    CUDA tensors, cast to the solver dtype (None stays None).  Raises before anything is launched."""
    for name, g in (("x_goal", x_goal), ("u_goal", u_goal)):
        if g is not None and (not isinstance(g, torch.Tensor) or not g.is_cuda):
            raise RuntimeError("pddp_b200: per-problem %s must be a CUDA tensor (no CPU fallback)" % name)
    check_goal_shapes(x_goal, u_goal, B, geo, N)
    return [None if g is None else g.detach().to(dtype) for g in (x_goal, u_goal)]


class QRCostConstants:
    """Q, R, Q_term, x_goal, u_goal of a QRCost on the augmented state (ref: costs/quadratic.py)."""

    def __init__(self, Q, R, Q_term, x_goal, u_goal=None):
        self.Q = torch.as_tensor(Q, dtype=torch.float64).cpu()
        self.Q_term = torch.as_tensor(Q_term, dtype=torch.float64).cpu()
        self.R = torch.as_tensor(R, dtype=torch.float64).cpu().reshape(-1)
        self.x_goal = torch.as_tensor(x_goal, dtype=torch.float64).cpu().reshape(-1)
        ug = torch.zeros(1, dtype=torch.float64) if u_goal is None else torch.as_tensor(
            u_goal, dtype=torch.float64).cpu().reshape(-1)
        self.u_goal = ug

    def c_struct(self):
        DA = self.Q.shape[0]
        if DA > _lib.MAX_DA or self.Q.shape != (DA, DA) or self.Q_term.shape != (DA, DA):
            raise ValueError("Q / Q_term must be square, at most %dx%d" % (_lib.MAX_DA, _lib.MAX_DA))
        nu = int(round(self.R.numel() ** 0.5))
        if nu * nu != self.R.numel() or nu > _lib.MAX_NU or self.u_goal.numel() not in (1, nu):
            raise ValueError("R must be nu x nu with nu <= %d, u_goal a scalar or [nu]" % _lib.MAX_NU)
        s = _lib.CostGoals()
        for i, v in enumerate(self.Q.reshape(-1).tolist()):
            s.Q[i] = v
        for i, v in enumerate(self.Q_term.reshape(-1).tolist()):
            s.Q_term[i] = v
        for i, v in enumerate(self.x_goal.tolist()):
            s.x_goal[i] = v
        for i, v in enumerate(self.R.tolist()):          # row-major nu x nu
            s.R[i] = v
        for i, v in enumerate(self.u_goal.reshape(-1).expand(nu).tolist()):
            s.u_goal[i] = v
        return s


class BatchedSolver:
    """Device buffers + pass sequencing for B problems of one (dynamics, cost, encoding, N)."""

    def __init__(self, dynamics, cost, encoding, B, N, dtype=torch.float32, device="cuda",
                 layout=None, max_alphas=16):
        self.lib = _lib.load()
        self.dyn, self.cost = dynamics, cost
        self.enc = StateEncoding(int(encoding))
        self.geo = dynamics.geo
        self.D, self.nu, _, _ = _lib.GEO_INFO[self.geo]
        self.nz = infer_encoded_state_size(self.D, self.enc)
        self.B, self.N, self.dtype = int(B), int(N), dtype
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("pddp_b200 runs on CUDA devices only (no CPU fallback)")
        if layout is None:   # SoA for thread-per-problem kernels, records for warp-per-problem
            layout = _lib.BATCH_INNER if (not dynamics.is_bnn and self.nz <= 8) else _lib.PROBLEM_MAJOR
        self.layout = layout
        self.shape = _lib.Shape(_lib.dtype_code(dtype), layout, self.geo, int(self.enc), self.B,
                                self.N, self.nz, self.nu)
        self.c_cost = cost.c_struct()
        self.p_b = None            # device copy [B, 8] of per-problem dynamics parameters (set_dynamics)
        self.c_dyn = None
        if not dynamics.is_bnn:
            self.set_dynamics(dynamics)
        nz, nu, N = self.nz, self.nu, self.N
        dims = dict(Z=(N + 1, nz), F_z=(N, nz * nz), F_u=(N, nz * nu), L=(N + 1, 1), L_z=(N + 1, nz),
                    L_u=(N, nu), L_zz=(N + 1, nz * nz), L_uz=(N, nu * nz), L_uu=(N, nu * nu),
                    U=(N, nu), k=(N, nu), K=(N, nu * nz), K_nominal=(N, nu * nz), Z_new=(N + 1, nz), U_new=(N, nu))
        self.buf = {n: self._alloc(nt, e) for n, (nt, e) in dims.items()}
        o = dict(device=self.device)
        self.z0 = torch.zeros(self.B, nz, dtype=dtype, **o)
        self.J_opt = torch.zeros(self.B, dtype=dtype, **o)
        self.J_new = torch.zeros(self.B, dtype=dtype, **o)
        self.max_alphas = int(max_alphas)
        self.J_all = torch.zeros(self.B, 10, dtype=dtype, **o)
        self.amin = torch.zeros(self.B, dtype=torch.int32, **o)
        self.mu = torch.zeros(self.B, dtype=torch.float64, **o)
        self.delta = torch.full((self.B,), 2.0, dtype=torch.float64, **o)
        self.state = torch.zeros(self.B, dtype=torch.int32, **o)
        self.iters_left = torch.zeros(self.B, dtype=torch.int32, **o)
        self.active = torch.ones(self.B, dtype=torch.int32, **o)
        self.accepted = torch.zeros(self.B, dtype=torch.int32, **o)
        self.lin_status = torch.zeros(self.B, dtype=torch.int32, **o)
        self.bw_status = torch.zeros(self.B, dtype=torch.int32, **o)
        self.roll_status = torch.zeros(self.B, dtype=torch.int32, **o)
        self.n_active = torch.zeros(1, dtype=torch.int32, **o)
        self.u_min = self.u_max = None
        # goal buffers, made on first use: per problem "x_goal" [B, DA], "u_goal" [B, nu]; per step "x_goal_t"
        # [B, N+1, DA], "u_goal_t" [B, N, nu] in the solver's layout (view / store like the buffers above)
        self.goals = {}
        self._goal_ptrs = (None, None, None, None)       # x_goal_b, u_goal_b, x_goal_bt, u_goal_bt
        self.alphas = fit_alphas(dtype, self.device)
        self.launches = 0          # CUDA kernels enqueued by this solver (bench.py reports it)
        self.workspace = None
        if dynamics.is_bnn:
            if dynamics.input_mode == _lib.BNN_INPUT_RESAMPLE and dynamics.tensors["eps_in"].shape[0] < self.N:
                raise ValueError("BNN_INPUT_RESAMPLE: eps_in holds %d steps, the horizon is %d"
                                 % (dynamics.tensors["eps_in"].shape[0], self.N))
            if dynamics.tensors["eps_out"] is not None and dynamics.tensors["eps_out"].shape[0] < self.N:
                raise ValueError("use_predicted_std: eps_out holds %d steps, the horizon is %d"
                                 % (dynamics.tensors["eps_out"].shape[0], self.N))
            self.c_bnn = dynamics.c_struct(dtype, self.device)
            nbytes = self.lib.pddp_bnn_workspace_bytes(C.byref(self.shape), C.byref(self.c_bnn),
                                                       max_alphas)
            if nbytes < 0:
                _lib.check(int(nbytes), "bnn_workspace_bytes")
            self.workspace = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)

    # ---------------------------------------------------------------- buffers
    def _alloc(self, nt, e):
        shape = (nt, e, self.B) if self.layout == _lib.BATCH_INNER else (self.B, nt, e)
        return torch.zeros(shape, dtype=self.dtype, device=self.device)

    def view(self, name):
        """[B, Nt, E] view of a buffer whatever the internal layout."""
        t = self.buf[name] if name in self.buf else self.goals[name]
        return t.permute(2, 0, 1) if self.layout == _lib.BATCH_INNER else t

    def store(self, name, value):
        """Copies a [B, Nt, E]-shaped tensor into the named buffer."""
        self.view(name).copy_(value.reshape(self.view(name).shape))

    def matrices(self, name):
        """Reference-shaped view: F_z [B,N,nz,nz], K [B,N,nu,nz], L [B,N+1] ..."""
        v = self.view(name)
        nz, nu = self.nz, self.nu
        shapes = dict(F_z=(nz, nz), F_u=(nz, nu), L_zz=(nz, nz), L_uz=(nu, nz), L_uu=(nu, nu),
                      K=(nu, nz), K_nominal=(nu, nz))
        if name in shapes:
            return v.reshape(v.shape[0], v.shape[1], *shapes[name])
        if name == "L":
            return v.reshape(v.shape[0], v.shape[1])
        return v

    # ---------------------------------------------------------------- setup
    def set_dynamics(self, dynamics):
        """Closed-form dynamics constants: shared by every problem, or params_b [B, 8] with one row per problem,
        copied to the device in the solver dtype.  Raises ValueError (before anything is launched) unless the rows
        number B."""
        if dynamics.is_bnn or dynamics.geo != self.geo:
            raise ValueError("set_dynamics takes closed-form dynamics of the solver's geometry")
        check_dynamics_rows(dynamics, self.B)
        if dynamics.params_b is None:
            self.p_b = None
        else:
            if self.p_b is None:
                self.p_b = torch.empty(self.B, 8, dtype=self.dtype, device=self.device)
            self.p_b.copy_(dynamics.params_b)
        self.dyn = dynamics
        self.c_dyn = dynamics.c_struct(self.p_b)

    def set_goals(self, x_goal=None, u_goal=None):
        """Gives every problem its own goal: x_goal [B, DA] in the cost's coordinates (the angle-augmented state,
        like QRCost.x_goal), u_goal [B, nu]; or a goal per problem and step, to track a reference: x_goal
        [B, N+1, DA] (row N goes with Q_term), u_goal [B, N, nu].  x and u choose their form independently.  A goal
        left None is the cost's own, shared by every problem; setting goals clears the ones set before."""
        goals = check_goals(x_goal, u_goal, self.B, self.geo, self.dtype, self.N)
        ptrs = [None] * 4
        for i, (name, g) in enumerate(zip(("x_goal", "u_goal"), goals)):
            if g is None:
                continue
            if g.dim() == 3:
                name, i = name + "_t", i + 2
                if name not in self.goals:
                    self.goals[name] = self._alloc(g.shape[1], g.shape[2])
                self.store(name, g)
            else:
                if name not in self.goals:
                    self.goals[name] = torch.empty(g.shape, dtype=self.dtype, device=self.device)
                self.goals[name].copy_(g)
            ptrs[i] = self.goals[name].data_ptr()
        self._goal_ptrs = tuple(ptrs)

    def _cost(self):
        """The cost argument of a C ABI call, carrying this solver's per-problem / per-step goals (or NULL)."""
        (self.c_cost.x_goal_b, self.c_cost.u_goal_b, self.c_cost.x_goal_bt,
         self.c_cost.u_goal_bt) = self._goal_ptrs
        return C.byref(self.c_cost)

    def set_problem(self, z0, U, u_min=None, u_max=None, alphas=None, iterations=1, x_goal=None, u_goal=None):
        """Initial states z0 [B, nz], controls U [B, N, nu], bounds, line-search candidates and the per-problem
        goals of set_goals; goals not given are cleared."""
        self.set_goals(x_goal, u_goal)
        # (no torch.as_tensor on tensors: under torch.set_default_device it would MOVE them to the default device)
        z0 = (z0 if isinstance(z0, torch.Tensor) else torch.as_tensor(z0)).detach()
        _lib.require_cuda(z0, "z0")
        self.z0.copy_(z0.reshape(self.B, self.nz))
        self.store("U", (U if isinstance(U, torch.Tensor) else torch.as_tensor(U)).detach())
        if (u_min is None) != (u_max is None):
            raise ValueError("u_min and u_max must be given together")
        self.u_min = expand_bound(u_min, self.nu, self.dtype, self.device)
        self.u_max = expand_bound(u_max, self.nu, self.dtype, self.device)
        if alphas is not None:
            self.alphas = torch.as_tensor(alphas).to(dtype=self.dtype, device=self.device).contiguous()
        if self.alphas.numel() > self.max_alphas:
            raise ValueError("more line-search candidates than max_alphas=%d" % self.max_alphas)
        if self.alphas.numel() != self.J_all.shape[1]:     # the C ABI writes J_all as [B, A]
            self.J_all = torch.zeros(self.B, self.alphas.numel(), dtype=self.dtype, device=self.device)
        self.reset(iterations)

    def reset(self, iterations=1):
        """ref: ilqr.py:364-367 (_reset_reg) per problem + bookkeeping for `iterations` steps."""
        self.mu.zero_()
        self.delta.fill_(2.0)
        self.state.zero_()
        self.iters_left.fill_(int(iterations))
        self.active.fill_(1)

    # ---------------------------------------------------------------- the four stages
    @on_own_device
    def linearize(self, use_active=True):
        b, p = self.buf, _lib.ptr
        act = p(self.active) if use_active else None
        self.lin_status.zero_()
        if self.dyn.is_bnn:
            code = self.lib.pddp_linearize_bnn(
                C.byref(self.shape), C.byref(self.c_bnn), self._cost(), p(self.z0), p(b["U"]),
                p(self.u_min), p(self.u_max), act, *[p(b[n]) for n in LIN_NAMES], p(self.J_opt),
                p(self.lin_status), p(self.workspace), self.workspace.numel(), _lib.stream_ptr())
            _lib.check(code, "linearize_bnn")
        else:
            code = self.lib.pddp_linearize_known(
                C.byref(self.shape), C.byref(self.c_dyn), self._cost(), p(self.z0), p(b["U"]),
                p(self.u_min), p(self.u_max), act, *[p(b[n]) for n in LIN_NAMES], p(self.J_opt),
                p(self.lin_status), _lib.stream_ptr())
            _lib.check(code, "linearize_known")

    @on_own_device
    def cost_only(self):
        """Cost value / gradient / Hessian of whatever is stored in Z, U (no rollout)."""
        b, p = self.buf, _lib.ptr
        code = self.lib.pddp_cost_derivatives(
            C.byref(self.shape), self._cost(), p(b["Z"]), p(b["U"]), None, p(b["L"]), p(b["L_z"]),
            p(b["L_u"]), p(b["L_zz"]), p(b["L_uz"]), p(b["L_uu"]), p(self.J_opt), _lib.stream_ptr())
        _lib.check(code, "cost_derivatives")

    @on_own_device
    def backward(self, use_active=True):
        b, p = self.buf, _lib.ptr
        code = self.lib.pddp_backward(
            C.byref(self.shape), p(b["F_z"]), p(b["F_u"]), p(b["L_z"]), p(b["L_u"]), p(b["L_zz"]),
            p(b["L_uz"]), p(b["L_uu"]), p(self.mu), p(b["U"]), p(self.u_min), p(self.u_max),
            p(self.active) if use_active else None, p(b["k"]), p(b["K"]), p(self.bw_status),
            _lib.stream_ptr())
        _lib.check(code, "backward")

    @on_own_device
    def rollout(self, use_active=True, use_bw_status=True):
        b, p = self.buf, _lib.ptr
        A = int(self.alphas.numel())
        common = (p(b["Z"]), p(b["U"]), p(b["k"]), p(b["K"]), p(self.alphas), A, p(self.u_min),
                  p(self.u_max), p(self.active) if use_active else None,
                  p(self.bw_status) if use_bw_status else None, p(self.J_all), p(self.amin),
                  p(self.J_new), p(b["Z_new"]), p(b["U_new"]))
        if self.dyn.is_bnn:
            code = self.lib.pddp_rollout_bnn(
                C.byref(self.shape), C.byref(self.c_bnn), self._cost(), *common,
                p(self.roll_status), p(self.workspace), self.workspace.numel(), _lib.stream_ptr())
            _lib.check(code, "rollout_bnn")
        else:
            code = self.lib.pddp_rollout_known(C.byref(self.shape), C.byref(self.c_dyn),
                                               self._cost(), *common, _lib.stream_ptr())
            _lib.check(code, "rollout_known")

    @on_own_device
    def accept(self, tol=5e-6, max_reg=1e10):
        b, p = self.buf, _lib.ptr
        self.n_active.zero_()
        code = self.lib.pddp_accept_update(
            C.byref(self.shape), p(self.J_new), p(self.bw_status), p(b["Z_new"]), p(b["U_new"]),
            float(tol), float(max_reg), p(self.mu), p(self.delta), p(self.J_opt), p(self.state),
            p(self.iters_left), p(self.active), p(b["Z"]), p(b["U"]), p(self.accepted),
            p(self.n_active), p(b["K"]), p(b["K_nominal"]), _lib.stream_ptr())
        _lib.check(code, "accept_update")

    def iterate(self, tol=5e-6, max_reg=1e10):
        """One pass of the hot path over the whole batch (no host synchronisation)."""
        self.linearize()
        self.backward()
        self.rollout()
        self.accept(tol, max_reg)

    # ---------------------------------------------------------------- driver
    def fit(self, z0, U, n_iterations=50, tol=5e-6, max_reg=1e10, u_min=None, u_max=None,
            alphas=None, max_passes=None, on_pass=None, x_goal=None, u_goal=None):
        """Runs every problem until it has done `n_iterations` accepted steps or reached a
        terminal state (CONVERGED / MAX_REG), exactly like B sequential reference `fit` calls
        (ref: ilqr.py:237-316); rejected / not-PD attempts retry with a larger mu and do not
        consume iterations (ref: ilqr.py:213).  x_goal [B, DA] or [B, N+1, DA] / u_goal [B, nu] or [B, N, nu]:
        per-problem or per-step goals (set_goals)."""
        self.set_problem(z0, U, u_min, u_max, alphas, iterations=n_iterations, x_goal=x_goal, u_goal=u_goal)
        passes = 0
        limit = max_passes if max_passes is not None else n_iterations * 64
        while passes < limit:
            self.iterate(tol, max_reg)
            passes += 1
            if on_pass is not None:
                on_pass(passes, self)
            if int(self.n_active.item()) == 0:     # one 4-byte D2H read per pass
                break
        return self.view("Z"), self.view("U"), self.state


# ---------------------------------------------------------------------------------------------
# Solver cache for the reference-shaped entry points (module-level forward / _control_law /
# _trajectory_cost, model(z, u, i), cost(z, u, i), utils.evaluation.*): the reference calls these once
# per time step or per iteration, so buffers, BNN device copies and tensor-core weight images must not
# be rebuilt per call.  Small LRU keyed on the objects and shapes; cheap host constants (cost matrices,
# closed-form model parameters) are re-read on every hit, BNN weights are tracked by `model._version`.
# ---------------------------------------------------------------------------------------------
_SOLVER_CACHE = collections.OrderedDict()
_SOLVER_CACHE_SIZE = 6


def _zero_cost(geo):
    D, nu, ang, _ = _lib.GEO_INFO[geo]
    DA = D + len(ang)
    return QRCostConstants(torch.zeros(DA, DA), torch.zeros(nu, nu), torch.zeros(DA, DA), torch.zeros(DA))


def cached_solver(model, cost, encoding, B, N, dtype, device, max_alphas=16, model_opts=None, layout=None,
                  problems=None):
    """BatchedSolver for (model, cost) -- either may be None: a cost-only solver (pddp_cost_derivatives) or a
    model-only one with a zero cost (model forward / eval_dynamics).  problems = (lo, hi): the solver holds problems
    [lo, hi) of a larger batch (a shard), and takes those rows of a closed-form model's per-problem parameters."""
    if model is None and cost is None:
        raise ValueError("cached_solver needs a model or a cost")
    opts = tuple(sorted((model_opts or {}).items()))
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    key = (id(model), getattr(model, "_version", 0), id(cost), int(encoding), int(B), int(N), dtype, str(device),
           layout, opts)
    hit = _SOLVER_CACHE.get(key)
    if hit is not None and hit[0]() is model and hit[1]() is cost and hit[2].max_alphas >= max_alphas:
        _SOLVER_CACHE.move_to_end(key)
        s = hit[2]
    else:
        is_bnn = getattr(model, "is_bnn", False)
        if model is None:
            desc = KnownDynamics(cost.geometry(), [0.0] * 8)
        else:
            desc = model.descriptor(dict(opts), N) if is_bnn else model.descriptor()
            if not is_bnn and problems is not None:
                desc = desc.rows(*problems)
        if cost is not None and model is not None and cost.geometry() != desc.geo:
            raise ValueError("model and cost disagree on the state geometry")
        consts = cost.constants() if cost is not None else _zero_cost(desc.geo)
        s = BatchedSolver(desc, consts, encoding, B, N, dtype=dtype, device=device, layout=layout,
                          max_alphas=max(16, max_alphas))
        ref = lambda o: (lambda: None) if o is None else weakref.ref(o)
        _SOLVER_CACHE[key] = (ref(model), ref(cost), s)
        while len(_SOLVER_CACHE) > _SOLVER_CACHE_SIZE:
            _SOLVER_CACHE.popitem(last=False)
        return s
    if cost is not None:                                  # live constants, like the reference's live objects
        s.c_cost = cost.constants().c_struct()
    if model is not None and not s.dyn.is_bnn:
        desc = model.descriptor()
        s.set_dynamics(desc if problems is None else desc.rows(*problems))
    return s


def clear_solver_cache():
    _SOLVER_CACHE.clear()
