"""Per-problem dynamics parameters on the CPU: how a closed-form model with B parameter sets packs its rows, the
shape and length rules, the entry points that evaluate one system, and the split of the rows across two ranks."""
import ctypes
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import pddp_b200 as P
from pddp_b200 import _lib
from pddp_b200.solver import KnownDynamics, check_dynamics_rows

EX = P.examples


def test_struct_carries_the_row_pointer():
    assert ctypes.sizeof(_lib.KnownDynamics) == 64
    assert ctypes.sizeof(_lib.KnownDynamicsBatch) == 72
    assert _lib.KnownDynamicsBatch.p_b.offset == 64
    s = KnownDynamics(_lib.GEO_PENDULUM, [0.1, 1.0, 1.0, 0.1, 9.8]).c_struct()
    assert isinstance(s, _lib.KnownDynamicsBatch) and s.p_b is None and list(s.p)[:5] == [0.1, 1.0, 1.0, 0.1, 9.8]


def test_scalar_parameters_are_one_shared_set():
    m = EX.pendulum.PendulumDynamicsModel(0.1, m=1.5)
    assert m.n_sets == 1
    d = m.descriptor()
    assert d.params_b is None and d.n_sets == 1
    assert d.params == pytest.approx([0.1, 1.5, 1.0, 0.1, 9.80665])
    one = EX.pendulum.PendulumDynamicsModel(0.1, m=torch.tensor([1.5]))      # one set given as a 1-element tensor
    assert one.n_sets == 1 and one.descriptor().params_b is None
    assert one.descriptor().params == pytest.approx(d.params)


@pytest.mark.parametrize("cls,kwargs,order", [
    (EX.pendulum.PendulumDynamicsModel, dict(m=[1.0, 2.0, 3.0]), ("dt", "m", "l", "mu", "g")),
    (EX.cartpole.CartpoleDynamicsModel, dict(mp=[0.4, 0.5, 0.6], l=torch.tensor([0.5, 0.6, 0.7], dtype=torch.float64)),
     ("dt", "mc", "mp", "l", "mu", "g")),
    (EX.double_cartpole.DoubleCartpoleDynamicsModel, dict(l2=[0.5, 0.6, 0.7], g=[9.0, 9.5, 10.0]),
     ("dt", "mc", "mp1", "mp2", "l1", "l2", "mu", "g")),
    (EX.rendezvous.RendezvousDynamicsModel, dict(alpha=[0.1, 0.2, 0.3]), ("dt", "m", "alpha")),
])
def test_descriptor_packs_rows_in_geometry_order(cls, kwargs, order):
    dt = torch.tensor([0.05, 0.1, 0.2])                         # dt may vary per problem too
    model = cls(dt, **kwargs)
    assert model.n_sets == 3
    d = model.descriptor()
    assert d.n_sets == 3 and tuple(d.params_b.shape) == (3, 8) and d.params_b.dtype == torch.float64
    for j, name in enumerate(order):
        want = getattr(model, name).detach().double().expand(3)
        assert torch.equal(d.params_b[:, j], want), name
    assert torch.equal(d.params_b[:, len(order):], torch.zeros(3, 8 - len(order), dtype=torch.float64))
    # a scalar broadcasts: the defaults repeat in every row
    ref = cls(0.1).descriptor().params
    for j, name in enumerate(order):
        if name not in kwargs and name != "dt":
            assert torch.all(d.params_b[:, j] == ref[j]), name


def test_setup_accepts_tensors():
    model = EX.problems.SampleProblems.PENDULUM.get_model_class()(0.1, m=torch.tensor([0.5, 1.0]))
    assert model.n_sets == 2 and tuple(model.m.shape) == (2,) and model.m.requires_grad
    assert not model.dt.requires_grad


def test_shape_and_length_errors():
    with pytest.raises(ValueError, match="one length"):
        EX.pendulum.PendulumDynamicsModel(0.1, m=[1.0, 2.0, 3.0], l=[1.0, 2.0])
    with pytest.raises(ValueError, match="one length"):
        EX.pendulum.PendulumDynamicsModel(torch.tensor([0.1, 0.2]), m=[1.0, 2.0, 3.0])
    with pytest.raises(ValueError, match="one length"):                      # a 1-element tensor is not a scalar
        EX.rendezvous.RendezvousDynamicsModel(0.1, m=torch.tensor([1.0]), alpha=[0.1, 0.2])
    with pytest.raises(ValueError):
        EX.cartpole.CartpoleDynamicsModel(0.1, mc=torch.ones(2, 2))
    m = EX.pendulum.PendulumDynamicsModel(0.1)
    m.l = torch.nn.Parameter(torch.ones(3))
    m.m = torch.nn.Parameter(torch.ones(4))                   # edited after construction: caught when read
    with pytest.raises(ValueError, match="one length"):
        m.descriptor()
    with pytest.raises(ValueError, match=r"\[B, 8\]"):
        KnownDynamics(_lib.GEO_PENDULUM, [0.1, 1, 1, 0.1, 9.8], torch.zeros(3, 7))
    with pytest.raises(ValueError, match=r"\[B, 8\]"):
        KnownDynamics(_lib.GEO_PENDULUM, [0.1, 1, 1, 0.1, 9.8], torch.zeros(8))
    d = KnownDynamics(_lib.GEO_PENDULUM, [0.1, 1, 1, 0.1, 9.8], torch.zeros(3, 8))
    check_dynamics_rows(d, 3)
    check_dynamics_rows(KnownDynamics(_lib.GEO_PENDULUM, [0.1, 1, 1, 0.1, 9.8]), 5)    # one shared set fits any B
    for B in (1, 2, 4):
        with pytest.raises(ValueError, match="3 parameter sets"):
            check_dynamics_rows(d, B)


def test_single_problem_entry_points_reject_several_sets():
    from pddp_b200.controllers.ilqr import _control_law, forward
    from pddp_b200.utils.evaluation import eval_dynamics
    model = EX.pendulum.PendulumDynamicsModel(0.1, m=[1.0, 2.0, 3.0])
    cost = EX.pendulum.PendulumCost()
    z, U = torch.zeros(2), torch.zeros(5, 1)
    with pytest.raises(ValueError, match="one system.*3 parameter sets"):
        forward(z, U, model, cost)
    with pytest.raises(ValueError, match="_control_law.*3 parameter sets"):
        _control_law(model, torch.zeros(6, 2), U, torch.zeros(5, 1), torch.zeros(5, 1, 2), 1.0)
    with pytest.raises(ValueError, match="eval_dynamics.*3 parameter sets"):
        eval_dynamics(model, z, torch.zeros(1), 0)
    with pytest.raises(ValueError, match="batch_size=None.*3 parameter sets"):
        EX.pendulum.PendulumEnv(model=model)
    with pytest.raises(ValueError, match="batch_size=None.*3 parameter sets"):
        EX.problems.SampleProblems.PENDULUM.get_env_class()(model=model, dt=0.1)


def test_rows_of_a_shard():
    rows = torch.arange(7 * 8, dtype=torch.float64).reshape(7, 8)
    d = KnownDynamics(_lib.GEO_CARTPOLE, [0.0] * 6, rows)
    assert torch.equal(d.rows(2, 5).params_b, rows[2:5]) and d.rows(2, 5).geo == _lib.GEO_CARTPOLE
    shared = KnownDynamics(_lib.GEO_CARTPOLE, [0.1] * 6)
    assert shared.rows(2, 5) is shared


def _worker(rank, world, port, out_path):
    from pddp_b200.sharding import all_gather_problems, shard, shard_bounds
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    B = 7
    model = EX.cartpole.CartpoleDynamicsModel(0.1, mp=torch.linspace(0.3, 0.9, B), l=torch.linspace(0.4, 0.7, B))
    desc = model.descriptor()
    lo, hi = shard_bounds(B, world, rank)
    mine = desc.rows(lo, hi)                     # what iLQRController.fit hands this rank's solver
    z0 = torch.arange(B * 4, dtype=torch.float64).reshape(B, 4)
    assert mine.n_sets == shard(z0, world, rank).shape[0] == hi - lo
    # each row stays with its problem: gathering rank by rank restores the full table next to z0
    rows, z = all_gather_problems([mine.params_b.contiguous(), shard(z0, world, rank).contiguous()], B)
    ok = torch.equal(rows, desc.params_b) and torch.equal(z, z0)
    if rank == 0:
        torch.save(bool(ok), out_path)
    dist.destroy_process_group()


def test_two_rank_gloo_split_of_the_rows(tmp_path):
    out = str(tmp_path / "ok.pt")
    mp.spawn(_worker, args=(2, 29767, out), nprocs=2, join=True)
    assert torch.load(out)
