"""Cartpole example problem, namespaced like pddp.examples.cartpole: closed-form dynamics constants
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


class CartpoleDynamicsModel(KnownDynamicsModel):
    """ref: pddp/examples/cartpole/model.py:30-141 (state [x, x', theta, theta'], action [F])."""
    state_size = 4
    angular_indices = torch.tensor([2]).long()
    non_angular_indices = torch.tensor([0, 1, 3]).long()
    _param_order = ("dt", "mc", "mp", "l", "mu", "g")

    def __init__(self, dt, mc=0.5, mp=0.5, l=0.5, mu=0.1, g=9.82):
        super().__init__()
        self._init_params(dt, mc=mc, mp=mp, l=l, mu=mu, g=g)


class CartpoleCost(QRCost):
    """ref: pddp/examples/cartpole/cost.py:32-87"""

    def __init__(self, pole_length=0.5):
        l = pole_length
        Q = torch.zeros(5, 5)
        Q[0, 0] = 1.0
        Q[0, 3] = Q[3, 0] = l
        Q[3, 3] = Q[4, 4] = l ** 2
        super().__init__(Q, 0.1 * torch.eye(1), torch.eye(5), _goal([0.0, 0.0, math.pi, 0.0], (2,)),
                         state_size=4, angular_indices=(2,))


class CartpoleEnv(KnownDynamicsEnv):
    """ref: pddp/examples/cartpole/env.py (constructor signature (model=None, dt, render); reset() mean and noise)"""
    initial_state = [0.0, 0.0, 0.0, 0.0]

    def __init__(self, model=None, dt=0.1, render=False, **kwargs):
        self.dt = dt
        super().__init__(CartpoleDynamicsModel(dt) if model is None else model, render=render, **kwargs)


__all__ = ["CartpoleCost", "CartpoleDynamicsModel", "CartpoleEnv"]
