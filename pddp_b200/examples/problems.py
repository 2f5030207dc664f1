"""ref: pddp/examples/problems.py:21-90"""
from enum import IntEnum

from . import cartpole, double_cartpole, pendulum, rendezvous


class SampleProblems(IntEnum):
    CARTPOLE = 1
    DOUBLE_CARTPOLE = 2
    PENDULUM = 3
    RENDEZVOUS = 4

    def _classes(self):
        return {SampleProblems.CARTPOLE: (cartpole.CartpoleEnv, cartpole.CartpoleCost, cartpole.CartpoleDynamicsModel),
                SampleProblems.DOUBLE_CARTPOLE: (double_cartpole.DoubleCartpoleEnv, double_cartpole.DoubleCartpoleCost,
                                                 double_cartpole.DoubleCartpoleDynamicsModel),
                SampleProblems.PENDULUM: (pendulum.PendulumEnv, pendulum.PendulumCost, pendulum.PendulumDynamicsModel),
                SampleProblems.RENDEZVOUS: (rendezvous.RendezvousEnv, rendezvous.RendezvousCost,
                                            rendezvous.RendezvousDynamicsModel)}[self]

    def setup(self, dt, render=False, **kwargs):
        """-> (env, cost, model).  Model parameters may be 1-D tensors of length B (e.g. m=masses): the model is then a
        family of B systems and the environment simulates B instances, instance b with system b."""
        env_class, cost_class, model_class = self._classes()
        model = model_class(dt, **kwargs)
        env_opts = {"batch_size": model.n_sets} if model.n_sets > 1 else {}
        return env_class(dt=dt, model=model_class(dt, **kwargs), render=render, **env_opts), cost_class(), model

    def get_env_class(self):
        return self._classes()[0]

    def get_cost_class(self):
        return self._classes()[1]

    def get_model_class(self):
        return self._classes()[2]
