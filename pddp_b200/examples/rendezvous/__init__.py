"""Rendezvous example problem, namespaced like pddp.examples.rendezvous: closed-form dynamics constants
(the step is a device function: csrc/known_lq.cu), the QRCost constants on the angle-augmented state, and the
device-resident environment whose ground truth is that model."""
import math

import torch

from ...costs.quadratic import QRCost
from ...envs.base import KnownDynamicsEnv
from ...models.base import KnownDynamicsModel
from ...utils.angular import augment_state


class RendezvousDynamicsModel(KnownDynamicsModel):
    """ref: pddp/examples/rendezvous/model.py:25-115 (state [x0, y0, x1, y1, and their velocities],
    action [Fx0, Fy0, Fx1, Fy1]; linear dynamics, the whole covariance is passed through)."""
    state_size = 8
    action_size = 4
    angular_indices = torch.tensor([]).long()
    non_angular_indices = torch.arange(8).long()
    _param_order = ("dt", "m", "alpha")

    def __init__(self, dt, m=1.0, alpha=0.1):
        super().__init__()
        self._init_params(dt, m=m, alpha=alpha)


class RendezvousCost(QRCost):
    """ref: pddp/examples/rendezvous/cost.py:29-43 (||x_0 - x_1||^2 + velocities, R = 0.1 I, Q_term = Q)"""

    def __init__(self):
        Q = torch.eye(8)
        Q[0, 2] = Q[2, 0] = -1
        Q[1, 3] = Q[3, 1] = -1
        super().__init__(Q, 0.1 * torch.eye(4), state_size=8, angular_indices=())


class RendezvousEnv(KnownDynamicsEnv):
    """ref: pddp/examples/rendezvous/env.py (constructor signature (model=None, dt, render); reset() mean and noise)"""
    initial_state = [-10.0, -10.0, 10.0, 10.0, 0.0, -5.0, 5.0, 0.0]

    def __init__(self, model=None, dt=0.05, render=False, **kwargs):
        self.dt = dt
        super().__init__(RendezvousDynamicsModel(dt) if model is None else model, render=render, **kwargs)


__all__ = ["RendezvousCost", "RendezvousDynamicsModel", "RendezvousEnv"]
