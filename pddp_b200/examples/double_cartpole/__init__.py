"""Double cartpole example problem, namespaced like pddp.examples.double_cartpole: closed-form dynamics constants
(the step is a device function: csrc/core.cuh), the QRCost constants on the angle-augmented state, and the
device-resident environment whose ground truth is that model."""
import math

import torch

from ...costs.quadratic import QRCost
from ...envs.base import KnownDynamicsEnv
from ...models.base import KnownDynamicsModel
from ...utils.angular import augment_state


def _goal(x, ang):
    non = [i for i in range(len(x)) if i not in ang]
    return augment_state(torch.as_tensor(x, dtype=torch.float32), list(ang), non)


class DoubleCartpoleDynamicsModel(KnownDynamicsModel):
    """ref: pddp/examples/double_cartpole/model.py:33-195."""
    state_size = 6
    angular_indices = torch.tensor([2, 4]).long()
    non_angular_indices = torch.tensor([0, 1, 3, 5]).long()
    _param_order = ("dt", "mc", "mp1", "mp2", "l1", "l2", "mu", "g")

    def __init__(self, dt, mc=0.5, mp1=0.5, mp2=0.5, l1=0.6, l2=0.6, mu=0.1, g=9.80665):
        super().__init__()
        self._init_params(dt, mc=mc, mp1=mp1, mp2=mp2, l1=l1, l2=l2, mu=mu, g=g)


class DoubleCartpoleCost(QRCost):
    """ref: pddp/examples/double_cartpole/cost.py:32-96"""

    def __init__(self, pole1_length=0.6, pole2_length=0.6):
        C = torch.tensor([[1, -pole1_length, 0, -pole2_length, 0], [0, 0, pole1_length, 0, pole2_length]])
        Q = torch.zeros(8, 8)
        dims = torch.tensor([0, 4, 5, 6, 7])
        Q[dims[:, None], dims[None, :]] = C.t().mm(C)
        super().__init__(Q, 0.1 * torch.eye(1), 100 * torch.eye(8), _goal(torch.zeros(6), (2, 4)),
                         state_size=6, angular_indices=(2, 4))


class DoubleCartpoleEnv(KnownDynamicsEnv):
    """ref: pddp/examples/double_cartpole/env.py (constructor signature (model=None, dt, render); reset() mean and noise)"""
    initial_state = [0.0, 0.0, math.pi, 0.0, math.pi, 0.0]

    def __init__(self, model=None, dt=0.1, render=False, **kwargs):
        self.dt = dt
        super().__init__(DoubleCartpoleDynamicsModel(dt) if model is None else model, render=render, **kwargs)


__all__ = ["DoubleCartpoleCost", "DoubleCartpoleDynamicsModel", "DoubleCartpoleEnv"]
