"""Dynamics-model and cost evaluation with derivatives, the reference's `pddp.utils.evaluation` entry points.

The reference obtains the Jacobian / Hessian by autograd, row by row (`eval_*`, autodiff.jacobian) or with the
"replicate the input and back-propagate an identity" trick (`batch_eval_*`, pddp/utils/evaluation.py:134-288).
Here both spellings run the same kernels: one step of `pddp_linearize_known` / `pddp_linearize_bnn` (forward-mode
tangents through the dynamics) and `pddp_cost_derivatives` (hyper-dual value + gradient + Hessian of the expected
cost), with B = 1, N = 1.  There is no CPU path.
"""
import torch

from .. import _lib
from ..solver import LIN_NAMES, cached_solver, require_single_system
from .encoding import StateEncoding


def eval_cost(cost, z, u, i, terminal=False, encoding=StateEncoding.DEFAULT, approximate=False, **kwargs):
    """-> (l, l_z, l_u, l_zz, l_uz, l_uu); l_u / l_uz / l_uu are None for a terminal cost.
    ref: pddp/utils/evaluation.py:23-94.  approximate=True returns the Gauss-Newton outer products
    l_z l_z^T, l_u l_z^T, l_u l_u^T (evaluation.py:72-78, 176-199)."""
    _lib.require_cuda(z, "z")
    s = cached_solver(None, cost, encoding, 1, 1, z.dtype, z.device, layout=_lib.PROBLEM_MAJOR)
    zd = z.detach().reshape(1, 1, -1)
    s.store("Z", zd.expand(1, 2, -1))                     # row 0: running cost, row 1 (= N): terminal cost
    if not terminal:
        s.store("U", u.detach().reshape(1, 1, -1))
    else:
        s.view("U").zero_()
    s.cost_only()
    t = 1 if terminal else 0
    l = s.matrices("L")[0, t].clone()
    l_z = s.matrices("L_z")[0, t].clone()
    l_zz = s.matrices("L_zz")[0, t].clone()
    if approximate:
        l_zz = l_z.view(-1, 1).mm(l_z.view(1, -1))
    if terminal:
        return l, l_z, None, l_zz, None, None
    l_u = s.matrices("L_u")[0, 0].clone()
    if approximate:
        return l, l_z, l_u, l_zz, l_u.view(-1, 1).mm(l_z.view(1, -1)), l_u.view(-1, 1).mm(l_u.view(1, -1))
    return l, l_z, l_u, l_zz, s.matrices("L_uz")[0, 0].clone(), s.matrices("L_uu")[0, 0].clone()


def eval_dynamics(model, z, u, i, encoding=StateEncoding.DEFAULT, **kwargs):
    """-> (z_next [nz], dz'/dz [nz, nz], dz'/du [nz, nu]).  ref: pddp/utils/evaluation.py:97-131.
    `kwargs` are the model options (use_predicted_std, infer_noise_variables, ...)."""
    require_single_system(model, "eval_dynamics")
    _lib.require_cuda(z, "z")
    if getattr(model, "is_bnn", False) and int(i) != 0:
        raise NotImplementedError("pddp_b200: a stand-alone BNN evaluation is only defined for step 0 (particles drawn "
                                  "from eps_in[0]); later steps depend on the particle cache the controller's passes "
                                  "carry on the device")
    kwargs.pop("identical_inputs", None)
    s = cached_solver(model, None, encoding, 1, 1, z.dtype, z.device, model_opts=kwargs)
    s.set_problem(z.detach().reshape(1, -1), u.detach().reshape(1, 1, -1))
    s.linearize(use_active=False)
    return s.matrices("Z")[0, 1].clone(), s.matrices("F_z")[0, 0].clone(), s.matrices("F_u")[0, 0].clone()


# the "batch" variants differ from the row-wise ones only in how autograd is driven (evaluation.py:134-288)
batch_eval_cost = eval_cost
batch_eval_dynamics = eval_dynamics

__all__ = ["eval_cost", "eval_dynamics", "batch_eval_cost", "batch_eval_dynamics", "StateEncoding", "LIN_NAMES"]
