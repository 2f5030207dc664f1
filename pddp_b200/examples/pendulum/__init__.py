"""Pendulum example problem, namespaced like pddp.examples.pendulum: closed-form dynamics constants
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


class PendulumDynamicsModel(KnownDynamicsModel):
    """ref: pddp/examples/pendulum/model.py:33-119 (state [theta, theta'], action [torque])."""
    state_size = 2
    angular_indices = torch.tensor([0]).long()
    non_angular_indices = torch.tensor([1]).long()
    _param_order = ("dt", "m", "l", "mu", "g")

    def __init__(self, dt, m=1.0, l=1.0, mu=0.1, g=9.80665):
        super().__init__()
        self._init_params(dt, m=m, l=l, mu=mu, g=g)


class PendulumCost(QRCost):
    """ref: pddp/examples/pendulum/cost.py:32-88"""

    def __init__(self, pendulum_length=0.5):
        l = pendulum_length
        Q = torch.zeros(3, 3)
        Q[0, 0] = 1.0
        Q[0, 1] = Q[1, 0] = l
        Q[1, 1] = Q[2, 2] = l ** 2
        super().__init__(Q, 0.1 * torch.eye(1), 100 * torch.eye(3), _goal([math.pi, 0.0], (0,)),
                         state_size=2, angular_indices=(0,))


class PendulumEnv(KnownDynamicsEnv):
    """ref: pddp/examples/pendulum/env.py (constructor signature (model=None, dt, render); reset() mean and noise)"""
    initial_state = [0.0, 0.0]

    def __init__(self, model=None, dt=0.1, render=False, **kwargs):
        self.dt = dt
        super().__init__(PendulumDynamicsModel(dt) if model is None else model, render=render, **kwargs)


__all__ = ["PendulumCost", "PendulumDynamicsModel", "PendulumEnv"]
