"""Host side of the BNN model on the rendezvous geometry (D = 8, action_size 4): the factory sizes the network and the
trainer's input for the four controls, and refuses an action size the kernels do not have."""
import pytest
import torch

from pddp_b200 import _lib, models


def test_factory_builds_the_rendezvous_bnn():
    Model = models.bnn.bnn_dynamics_model_factory(8, 4, [200, 200], [], range(8))
    model = Model(n_particles=10)
    assert Model.action_size == 4 and model.action_size == 4
    assert model.model.fc_0.in_features == 12 and model.model.fc_out.out_features == 16
    assert model.train_config(torch.float64, 100, 32, 10, 1e-3, 1.0, seed=0).K0 == 12
    assert _lib.GEO_INFO[_lib.GEO_RENDEZVOUS][1] == 4


def test_factory_rejects_other_action_sizes():
    with pytest.raises(NotImplementedError):
        models.bnn.bnn_dynamics_model_factory(8, 2, [200, 200], [], range(8))
    with pytest.raises(NotImplementedError):
        models.bnn.bnn_dynamics_model_factory(8, 4, [200, 200, 200], [], range(8))


def test_single_control_geometries_keep_their_input_width():
    model = models.bnn.bnn_dynamics_model_factory(4, 1, [32, 32], [2], [0, 1, 3])(n_particles=8)
    assert model.action_size == 1 and model.model.fc_0.in_features == 6
    assert model.train_config(torch.float32, 100, 32, 10, 1e-3, 1.0, seed=0).K0 == 6
