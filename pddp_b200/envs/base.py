"""Environments (mirror of pddp/envs/base.py + pddp/envs/gym_env.py), batched and
device resident: B independent instances of a problem whose ground truth is one of the closed-form
dynamics models, stepped by `pddp_env_step_known` so that a closed-loop MPC run or a data-collection
trial (pddp/controllers/pddp.py:209-247, `_apply_controller`) never leaves the GPU.

There is no rendering and no gym dependency; `apply / get_state / reset / state_size / action_size`
are the members the controllers use (ref: pddp/envs/base.py:24-68)."""
import ctypes as C

import torch

from .. import _lib
from ..solver import check_dynamics_rows, require_single_system
from ..utils.gaussian_variable import GaussianVariable


class Env(object):
    """ref: pddp/envs/base.py:21-75"""

    def __enter__(self):
        return self

    def __exit__(self, type, value, traceback):
        self.close()

    @property
    def action_size(self):
        raise NotImplementedError

    @property
    def state_size(self):
        raise NotImplementedError

    def apply(self, u):
        raise NotImplementedError

    def get_state(self):
        raise NotImplementedError

    def reset(self):
        raise NotImplementedError

    def close(self):
        pass


class KnownDynamicsEnv(Env):
    """`batch_size` instances of an environment whose step is `model(x, u, 0, IGNORE_UNCERTAINTY)`
    (ref: pddp/examples/*/env.py step()).  batch_size=None mirrors the reference exactly (state [D],
    actions [nu]); with batch_size=B states are [B, D] and actions [B, nu].  A model with B parameter sets
    (KnownDynamicsModel) simulates instance b with set b, a fleet of different plants; batch_size=None needs one set.
    The parameters are read when the environment is built."""

    initial_state = None      # mean of reset()
    reset_noise = 1e-2        # ref: examples/*/env.py reset(): state += 1e-2 * randn

    def __init__(self, model, batch_size=None, dtype=torch.float32, device="cuda", generator=None, render=False):
        if render:
            raise NotImplementedError("pddp_b200 environments are device-resident simulators without rendering")
        self.model = model
        self.batch_size = batch_size
        self.dtype, self.device = dtype, torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("pddp_b200 environments live on CUDA devices only (no CPU fallback)")
        self._generator = generator
        self._desc = model.descriptor()
        B = 1 if batch_size is None else int(batch_size)
        if batch_size is None:
            require_single_system(model, "KnownDynamicsEnv(batch_size=None)")
        check_dynamics_rows(self._desc, B)
        self._p_b = None                # device copy [B, 8] of per-instance parameters
        if self._desc.params_b is not None:
            self._p_b = torch.empty(B, 8, dtype=dtype, device=self.device).copy_(self._desc.params_b)
        self._c_dyn = self._desc.c_struct(self._p_b)
        D, nu, _, _ = _lib.GEO_INFO[self._desc.geo]
        self._shape = _lib.Shape(_lib.dtype_code(dtype), _lib.PROBLEM_MAJOR, self._desc.geo, 4, B, 1, D, nu)
        self._state = torch.zeros(B, D, dtype=dtype, device=self.device)
        self.reset()

    @classmethod
    def from_model(cls, model, **kwargs):
        """An environment of this class simulated by a given model object (its constants, its dtype)."""
        env = cls.__new__(cls)
        KnownDynamicsEnv.__init__(env, model, **kwargs)
        return env

    @property
    def action_size(self):
        return int(self.model.action_size)

    @property
    def state_size(self):
        return int(self.model.state_size)

    def _view(self, t):
        return t[0] if self.batch_size is None else t

    def set_state(self, x):
        """Places the instances at x ([D] or [B, D])."""
        self._state.copy_(torch.as_tensor(x).to(device=self.device, dtype=self.dtype).reshape(self._state.shape))

    def apply(self, u):
        """ref: pddp/envs/gym_env.py:63-73 -> examples/*/env.py step().  The reference keeps the simulator
        state in float32 whatever the default dtype (`x = self.state.astype(np.float32)`); so does this."""
        u = torch.as_tensor(u).detach().to(device=self.device, dtype=self.dtype).reshape(self._state.shape[0], -1).contiguous()
        x = self._state.float().to(self.dtype)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().pddp_env_step_known(C.byref(self._shape), C.byref(self._c_dyn), _lib.ptr(x),
                                                       _lib.ptr(u), _lib.ptr(self._state), _lib.stream_ptr()),
                       "env_step_known")

    def get_state(self, var=1e-2):
        """ref: pddp/envs/gym_env.py:75-85"""
        mean = self._view(self._state).clone()
        return GaussianVariable(mean, var=var * torch.ones_like(mean))

    def reset(self):
        x0 = torch.tensor(self.initial_state, dtype=torch.float64, device="cpu")
        noise = torch.randn(self._state.shape, dtype=torch.float64, generator=self._generator, device="cpu")
        self._state.copy_((x0 + self.reset_noise * noise).to(self.dtype))
