"""Host-side rules of per-step goals: the MPC reference window and the goal shapes (CPU tensors, no GPU)."""
import pytest
import torch

from pddp_b200 import _lib
from pddp_b200.controllers.ilqr import batch_goals, reference_window
from pddp_b200.solver import check_goal_shapes, check_goals


def ref(B, T, E):
    return torch.arange(B * T * E, dtype=torch.float64).reshape(B, T, E)


def test_window_inside_the_reference():
    r = ref(3, 20, 5)
    w = reference_window(r, 4, 7, True)
    assert torch.equal(w, r[:, 4:11])


def test_window_clamps_past_the_end():
    r = ref(2, 6, 3)
    w = reference_window(r, 4, 5, True)
    assert torch.equal(w, r[:, [4, 5, 5, 5, 5]])
    assert torch.equal(reference_window(r, 40, 3, True), r[:, [5, 5, 5]])


def test_window_of_a_single_row_reference():
    r = ref(2, 1, 3)
    for i in (0, 3):
        assert torch.equal(reference_window(r, i, 4, True), r.expand(2, 4, 3))


def test_window_of_a_reference_longer_than_the_trial():
    r = ref(2, 100, 3)
    assert torch.equal(reference_window(r, 9, 11, True), r[:, 9:20])


def test_window_unbatched_and_pass_through():
    r = ref(1, 6, 3)[0]                                         # [T, E]: one problem
    assert torch.equal(reference_window(r, 3, 5, False), r[[3, 4, 5, 5, 5]])
    g = torch.zeros(4, 5)                                       # [B, DA]: no time axis
    assert reference_window(g, 3, 7, True) is g
    assert reference_window(None, 3, 7, True) is None


@pytest.mark.parametrize("geo,DA,nu", [(_lib.GEO_PENDULUM, 3, 1), (_lib.GEO_CARTPOLE, 5, 1),
                                       (_lib.GEO_DOUBLE_CARTPOLE, 8, 1), (_lib.GEO_RENDEZVOUS, 8, 4)])
def test_shape_rules(geo, DA, nu):
    B, N = 4, 7
    z = torch.zeros
    assert check_goal_shapes(z(B, DA), z(B, nu), B, geo, N) == [False, False]
    assert check_goal_shapes(z(B, N + 1, DA), z(B, N, nu), B, geo, N) == [True, True]
    assert check_goal_shapes(z(B, N + 1, DA), None, B, geo, N) == [True, None]
    assert check_goal_shapes(None, z(B, N, nu), B, geo, N) == [None, True]
    assert check_goal_shapes(z(B, DA), z(B, N, nu), B, geo, N) == [False, True]
    for bad in (dict(x_goal=z(B, N, DA)), dict(x_goal=z(B, N + 2, DA)), dict(x_goal=z(B, N + 1, DA + 1)),
                dict(x_goal=z(B + 1, N + 1, DA)), dict(u_goal=z(B, N + 1, nu)), dict(u_goal=z(B, N, nu + 1)),
                dict(x_goal=z(B, DA - 1)), dict(u_goal=z(B)), dict(x_goal=z(N + 1, DA))):
        with pytest.raises(ValueError):
            check_goal_shapes(bad.get("x_goal"), bad.get("u_goal"), B, geo, N)
    with pytest.raises(ValueError):                             # without N only the per-problem form
        check_goal_shapes(z(B, N + 1, DA), None, B, geo)
    with pytest.raises(RuntimeError):                           # CPU tensors never reach the kernels
        check_goals(z(B, N + 1, DA), None, B, geo, torch.float64, N)


def test_single_problem_takes_only_per_step_goals():
    N = 6
    x, u = torch.zeros(N + 1, 5), torch.zeros(N, 1)
    xb, ub = batch_goals(False, N, x, u)
    assert xb.shape == (1, N + 1, 5) and ub.shape == (1, N, 1)
    assert batch_goals(False, N, None, None) == [None, None]
    for bad in (dict(x_goal=torch.zeros(1, 5)), dict(u_goal=torch.zeros(1, 1)), dict(x_goal=torch.zeros(N, 5)),
                dict(x_goal=torch.zeros(5)), dict(u_goal=torch.zeros(1, N, 1))):
        with pytest.raises(ValueError):
            batch_goals(False, N, bad.get("x_goal"), bad.get("u_goal"))
    g = torch.zeros(3, 5)
    assert batch_goals(True, N, g, None)[0] is g                # batched calls pass through
