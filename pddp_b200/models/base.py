"""Dynamics-model interface (mirror of pddp/models/base.py).

A model object is a plain torch.nn.Module holding constants / weights exactly like the reference's;
what the CUDA kernels consume is its `descriptor()` (flat constants for the closed-form models,
weights + persistent dropout masks + eps_in[0] for the BNN).  Nothing here computes dynamics on the
CPU: `forward()` runs one step of the device rollout kernel.
"""
import torch

from .. import _lib
from ..solver import KnownDynamics, cached_solver
from ..utils.encoding import StateEncoding


def geometry_of(state_size, angular_indices):
    """Maps (D, angular dims) to a kernel geometry id; unsupported geometries raise."""
    ang = tuple(int(i) for i in angular_indices)
    for geo, (D, _, a, _) in _lib.GEO_INFO.items():
        if D == state_size and a == ang:
            return geo
    raise NotImplementedError("pddp_b200 has kernels for the pendulum (D=2, angle 0), cartpole (D=4, angle 2), "
                              "double-cartpole (D=6, angles 2,4) and rendezvous (D=8, no angles) state geometries; "
                              "got D=%d angles=%s" % (state_size, ang))


class DynamicsModel(torch.nn.Module):
    """ref: pddp/models/base.py:23-83 (same members; class-level sizes are plain class attributes)."""
    action_size = None
    state_size = None
    angular_indices = torch.tensor([]).long()
    non_angular_indices = torch.tensor([]).long()

    def fit(self, X, U, dX, quiet=False, **kwargs):
        raise NotImplementedError

    def descriptor(self):
        """KnownDynamics / BNNDynamics consumed by pddp_b200.solver.BatchedSolver."""
        raise NotImplementedError

    def reset_parameters(self, initializer=torch.nn.init.normal_):
        """ref: pddp/models/base.py:27-40"""
        for p in self.parameters():
            if p.requires_grad:
                initializer(p)
        return self

    def forward(self, z, u, i, encoding=StateEncoding.DEFAULT, identical_inputs=False, **kwargs):
        """Next encoded state distribution(s) z' for z:[..., nz], u:[..., nu] (on the GPU).

        One step of the device rollout kernel with zero gains (k = K = 0, alpha = 1)."""
        squeeze = z.dim() == 1
        zz = z.reshape(-1, z.shape[-1])
        uu = u.reshape(-1, u.shape[-1]).expand(zz.shape[0], -1)
        _lib.require_cuda(zz, "z")
        if getattr(self, "is_bnn", False) and int(i) != 0:
            raise NotImplementedError("pddp_b200: a stand-alone BNN forward is only defined for step 0 (particles "
                                      "drawn from eps_in[0]); later steps depend on the particle cache that the "
                                      "controller's rollout carries on the device")
        kwargs.pop("resample", None)
        s = cached_solver(self, None, encoding, zz.shape[0], 1, zz.dtype, zz.device, model_opts=kwargs)
        s.set_problem(zz, uu.unsqueeze(1), alphas=torch.ones(1))
        s.view("Z")[:, 0] = zz.detach()
        s.view("k").zero_()
        s.view("K").zero_()
        s.rollout(use_active=False, use_bw_status=False)
        out = s.view("Z_new")[:, 1].clone()
        return out[0] if squeeze else out.reshape(*z.shape[:-1], -1)


def _DA(model):
    return model.state_size + len(model.angular_indices)


def _param_tensor(v):
    """A closed-form model's parameter value: a scalar, or a 1-D tensor with one value per problem of a batch."""
    t = v.detach().clone() if isinstance(v, torch.Tensor) else torch.tensor(v)
    if not t.is_floating_point():
        t = t.to(torch.get_default_dtype())
    if t.dim() > 1:
        raise ValueError("a dynamics parameter is a scalar or a 1-D tensor of one value per problem, got shape %s"
                         % list(t.shape))
    return t


class KnownDynamicsModel(DynamicsModel):
    """Closed-form example dynamics (pddp/examples/<problem>/model.py): constants are Parameters like the
    reference's; the step itself is a device function (csrc/core.cuh, csrc/known_lq.cu).

    Every parameter, dt included, is a scalar or a 1-D tensor of length B: the model is then a family of B systems,
    and like the reference's element-wise dynamics, row b of a [B, nz] batch integrates system b.  Scalars are shared
    by all B.  Batched solves (iLQRController.fit / step with U [B, N, nu]), model(z [B, nz], u, i) and
    KnownDynamicsEnv(model, batch_size=B) take such a model; entry points that evaluate one system need one set."""
    _param_order = ()
    action_size = 1

    def _init_params(self, dt, **params):
        """dt (a constant, like the reference's) and the named parameters (trainable), in _param_order."""
        self.dt = torch.nn.Parameter(_param_tensor(dt), requires_grad=False)
        for n, v in params.items():
            setattr(self, n, torch.nn.Parameter(_param_tensor(v), requires_grad=True))
        _ = self.n_sets                 # raises on 1-D parameters of different lengths

    @property
    def n_sets(self):
        """Number of parameter sets: B when some parameter is a 1-D tensor of length B, else 1.  Raises ValueError
        when 1-D parameters differ in length."""
        lengths = {}
        for n in self._param_order:
            p = getattr(self, n)
            if p.dim() > 1:
                raise ValueError("dynamics parameter %s must be a scalar or 1-D, got shape %s" % (n, list(p.shape)))
            if p.dim() == 1:
                lengths[n] = int(p.shape[0])
        if len(set(lengths.values())) > 1:
            raise ValueError("per-problem dynamics parameters must have one length, got %s"
                             % ", ".join("%s: %d" % kv for kv in lengths.items()))
        n = next(iter(lengths.values()), 1)
        if n < 1:
            raise ValueError("per-problem dynamics parameters must not be empty")
        return n

    def fit(self, X, U, dX, quiet=False, **kwargs):
        pass            # ref: examples/*/model.py -- known models have nothing to fit

    def descriptor(self):
        """KnownDynamics: one shared parameter set, or with B sets the rows params_b [B, 8] (scalars repeated, in
        _param_order, zero padded to 8)."""
        geo = geometry_of(self.state_size, self.angular_indices.tolist())
        n = self.n_sets
        values = [getattr(self, k).detach() for k in self._param_order]
        if n == 1:
            return KnownDynamics(geo, [float(v.reshape(-1)[0]) for v in values])
        dev = values[0].device
        rows = torch.zeros(n, 8, dtype=torch.float64, device=dev)
        for j, v in enumerate(values):
            rows[:, j] = v.to(dtype=torch.float64, device=dev).expand(n)
        return KnownDynamics(geo, [0.0] * len(values), rows)
