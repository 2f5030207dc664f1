"""Multi-GPU entry of the PRODUCT (SURVEY 8e): `iLQRController.fit(U[B,N,nu], z0=[B,nz])` under torch.distributed
splits the batch contiguously across the ranks (one process per GPU, no collective inside the iteration) and
all-gathers (Z, U, K, state) once at the end.  The gathered 2-rank result must equal the single-GPU result of
the same call BIT FOR BIT (every problem runs the same kernels on the same inputs, wherever it lives).
Needs two GPUs: skipped on a one-GPU machine (`python -m pytest tests/test_gpu_multi.py -m gpu` on two or more)."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    import pddp_b200 as P
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    g = torch.Generator().manual_seed(0)                       # the SAME full batch on every rank
    B, N = 37, 12                                              # 37: the shards are uneven (19 + 18)
    results = {}
    for name, model, cost, enc, nz, nu in (
            ("pendulum", P.examples.pendulum.PendulumDynamicsModel(0.1), P.examples.pendulum.PendulumCost(), 4, 2, 1),
            ("cartpole_ut", P.examples.cartpole.CartpoleDynamicsModel(0.1), P.examples.cartpole.CartpoleCost(), 1, 14, 1)):
        mean = 0.05 * torch.randn(B, model.state_size, generator=g)
        z0 = torch.stack([P.GaussianVariable(m, var=1e-2 * torch.ones_like(m)).encode(P.StateEncoding(enc)) for m in mean])
        U = 0.1 * torch.randn(B, N, nu, generator=g)
        lo, hi = torch.tensor([-2.0]).to(dev), torch.tensor([2.0]).to(dev)
        ctrl = P.iLQRController(None, model, cost)
        Zs, Us, ss = ctrl.fit(U.to(dev), encoding=P.StateEncoding(enc), n_iterations=6, z0=z0.to(dev), u_min=lo, u_max=hi)
        Ks = ctrl._K.clone()
        assert Zs.shape == (B, N + 1, nz) and ss.shape == (B,)
        single = P.iLQRController(None, model, cost)
        Z1, U1, s1 = single.fit(U.to(dev), encoding=P.StateEncoding(enc), n_iterations=6, z0=z0.to(dev), u_min=lo,
                                u_max=hi, shard=False)
        results[name] = bool(torch.equal(Zs, Z1) and torch.equal(Us, U1) and torch.equal(ss, s1)
                             and torch.equal(Ks, single._K))
        # the feedback law of the sharded controller works on the full batch on every rank
        u = ctrl(Zs[:, 2], 2, P.StateEncoding(enc))
        results[name + "_feedback"] = bool(torch.allclose(u, Us[:, 2]))
    torch.save(results, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_fit_equals_single_gpu_fit(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_worker, args=(world, 29741, str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        res = torch.load(os.path.join(str(tmp_path), "rank%d.pt" % rank))
        assert all(res.values()), (rank, res)
