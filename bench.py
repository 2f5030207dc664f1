#!/usr/bin/env python
"""Benchmark of the PDDP/iLQR iteration hot path (BASELINE.json metric: trajectory-steps/s).

A "step" is ONE pass of the hot path over the whole batch of problems:
    linearise (dynamics + cost derivatives) -> backward Riccati -> rollout of all line-search
    alphas + trajectory cost -> per-problem accept/reject.
One trajectory-step = one time step of one problem through one such pass, so
    value = n_gpus * B * N * steps / seconds.

Workload (N=1 and per rank for N>1, weak scaling): BASELINE.json configs[1] --
"Cartpole PDDP with BNN dynamics (MC-dropout, 50 particles), horizon 100, batch 4096 initial
states": UT-Cholesky encoding (nz=14), MLP 6->200->200->8, 10 line-search alphas, u in [-10, 10].
Synthetic data: random-init BNN weights (reference initialiser, fc_out x0.02 so 100-step rollouts
stay finite -- SURVEY.md 6), CDropout eval masks and standardised eps_in[0] drawn once.

The JSON line also carries (rank 0): `roofline` (dominant kernel + per-kernel HBM / tensor fractions from CUDA
events on the launch stream), `e2e` (the same metric through `iLQRController.fit` with HOST buffers),
`cpu_baseline` (the CPU port of the reference on this box's host cores), `other_workloads` (BASELINE configs
1, 3, 4, 5 and config 2 in fp64, a few steps each) and, for N > 1, `strong` (config 2's 4096 problems split over
the ranks) and the timed final NCCL all-gather.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...          (one rank per GPU, no collective in
                                                                 the iteration, final NCCL gather)

--dump-outputs DIR writes what the last timed pass left for a caller as DIR/<name>.npy, so that two builds can
be compared output for output on the same seeded inputs (see dump_outputs).
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (geo name, encoding, B, N, P, A, hidden, u bound)
    "cartpole_bnn_b4096": dict(problem="cartpole", enc=1, B=4096, N=100, P=50, A=10, hidden=200, umax=10.0),
    "double_cartpole_bnn_fullcov_b1024": dict(problem="double_cartpole", enc=0, B=1024, N=100, P=50, A=10,
                                              hidden=200, umax=20.0),
    "cartpole_bnn_mpc_b8192": dict(problem="cartpole", enc=1, B=8192, N=50, P=50, A=16, hidden=200, umax=10.0),
    "pendulum_known_b1m": dict(problem="pendulum", enc=4, B=1 << 20, N=100, P=0, A=10, hidden=0, umax=2.5),
    # BASELINE configs[0]: one pendulum problem (launch-latency bound on any GPU; reported for completeness)
    "pendulum_known_single": dict(problem="pendulum", enc=4, B=1, N=100, P=0, A=10, hidden=0, umax=2.5),
    "cartpole_bnn_small": dict(problem="cartpole", enc=1, B=64, N=10, P=50, A=10, hidden=200, umax=10.0),
    # SURVEY 8f rank 1: action_size 4 (Jacobi eigen-clipping + 4-dimensional box QP in the backward pass)
    "rendezvous_known_b64k": dict(problem="rendezvous", enc=4, B=1 << 16, N=100, P=0, A=10, hidden=0, umax=1.0),
}
OTHER_WORKLOADS = (("pendulum_known_single", "f32"), ("double_cartpole_bnn_fullcov_b1024", "f32"),
                   ("pendulum_known_b1m", "f32"), ("cartpole_bnn_mpc_b8192", "f32"), ("cartpole_bnn_b4096", "f64"),
                   ("pendulum_known_b1m", "f64"), ("rendezvous_known_b64k", "f32"))
GEOMETRY = {"pendulum": (0, 2, (0,), (1,)), "cartpole": (1, 4, (2,), (0, 1, 3)),
            "double_cartpole": (2, 6, (2, 4), (0, 1, 3, 5)), "rendezvous": (3, 8, (), tuple(range(8)))}
KNOWN_PARAMS = {"pendulum": [0.1, 1.0, 1.0, 0.1, 9.80665], "rendezvous": [0.1, 1.0, 0.1]}
ACTION_SIZE = {"rendezvous": 4}
PROFILE_KINDS = ("mlp_linearise", "mlp_rollout", "moment_linearise", "rollout_step", "backward", "cost",
                 "linearize_known", "rollout_known", "accept")


def cost_constants(problem, dtype=torch.float64):
    """Q, R, Q_term, x_goal of the reference's example costs (pddp/examples/*/cost.py)."""
    if problem == "pendulum":
        Q = torch.tensor([[1, .5, 0], [.5, .25, 0], [0, 0, .25]], dtype=dtype)
        return Q, 0.1 * torch.eye(1, dtype=dtype), 100 * torch.eye(3, dtype=dtype), torch.tensor(
            [0.0, math.sin(math.pi), math.cos(math.pi)], dtype=dtype)
    if problem == "cartpole":
        Q = torch.zeros(5, 5, dtype=dtype)
        Q[0, 0] = 1
        Q[0, 3] = Q[3, 0] = .5
        Q[3, 3] = Q[4, 4] = .25
        return Q, 0.1 * torch.eye(1, dtype=dtype), torch.eye(5, dtype=dtype), torch.tensor(
            [0, 0, 0, math.sin(math.pi), math.cos(math.pi)], dtype=dtype)
    if problem == "rendezvous":            # pddp/examples/rendezvous/cost.py:29-43
        Q = torch.eye(8, dtype=dtype)
        Q[0, 2] = Q[2, 0] = Q[1, 3] = Q[3, 1] = -1
        return Q, 0.1 * torch.eye(4, dtype=dtype), Q.clone(), torch.zeros(8, dtype=dtype)
    C_ = torch.tensor([[1, -.6, 0, -.6, 0], [0, 0, .6, 0, .6]], dtype=dtype)
    Q = torch.zeros(8, 8, dtype=dtype)
    dims = [0, 4, 5, 6, 7]
    Q[torch.tensor(dims)[:, None], torch.tensor(dims)[None, :]] = C_.T @ C_
    goal = torch.tensor([0, 0, 0, 0, 0, 1, 0, 1.0], dtype=dtype)
    return Q, 0.1 * torch.eye(1, dtype=dtype), 100 * torch.eye(8, dtype=dtype), goal


def synth_bnn(problem, P, H, seed):
    """Random-init network exactly as pddp/models/bnn/modules.py:797-801,838-849 builds it
    (Xavier-normal with ReLU gain, biases U(-0.1,0.1)); CDropout eval masks (modules.py:540-548)
    and standardised eps_in[0] (modules.py:321-329)."""
    g = torch.Generator().manual_seed(seed)
    _, D, ang, _ = GEOMETRY[problem]
    dims = [D + len(ang) + 1, H, H, 2 * D]
    W, b = [], []
    for din, dout in zip(dims[:-1], dims[1:]):
        std = math.sqrt(2.0) * math.sqrt(2.0 / (din + dout))
        W.append(torch.randn(dout, din, generator=g) * std)
        b.append(torch.rand(dout, generator=g) * 0.2 - 0.1)
    W[-1] *= 0.02
    b[-1] *= 0.02
    masks = []
    for _ in range(2):
        r = torch.rand(P, H, generator=g).clamp(1e-6, 1 - 1e-6)
        masks.append(torch.sigmoid((r.log() - (1 - r).log()) / 0.1))
    eps = torch.randn(P, D, generator=g)
    eps0 = (eps - eps.mean(0)) / eps.std(0)
    return W, b, masks, eps0


def synth_inputs(w, seed, dtype):
    """z0: env reset distribution (mean 1e-2 randn around the start state, variance 1e-2 per dim,
    gym_env.py:75-85) in the workload's encoding; U = 0.1 randn (examples/animation.py:27)."""
    g = torch.Generator().manual_seed(seed)
    _, D, _, _ = GEOMETRY[w["problem"]]
    start = torch.zeros(D)
    if w["problem"] == "double_cartpole":
        start[2] = start[4] = math.pi
    if w["problem"] == "rendezvous":       # pddp/examples/rendezvous/env.py:106-108
        start = torch.tensor([-10.0, -10.0, 10.0, 10.0, 0.0, -5.0, 5.0, 0.0])
    mean = start + 1e-2 * torch.randn(w["B"], D, generator=g)
    if w["enc"] == 4:
        z0 = mean
    elif w["enc"] == 1:
        iu = torch.triu_indices(D, D)
        z0 = torch.cat([mean, (0.1 * torch.eye(D))[iu[0], iu[1]].expand(w["B"], -1)], -1)
    else:
        z0 = torch.cat([mean, (1e-2 * torch.eye(D)).reshape(-1).expand(w["B"], -1)], -1)
    U = 0.1 * torch.randn(w["B"], w["N"], ACTION_SIZE.get(w["problem"], 1), generator=g)
    return z0.to(dtype).contiguous(), U.to(dtype).contiguous()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], None, set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx = float(c[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v == "Active":
                    reasons.add(name)
        os.unlink(self.f.name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get("hbm_gbs", 6650.0), p.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


def committed_traffic(workload, kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel from the committed
    `ncu --set full` export profiles/kernel_traffic.json (written by tools/ncu_summary.py --traffic); None when
    the kernel has no committed capture."""
    path = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        table = json.load(f)
    row = table.get(workload, {}).get(kernel)
    if not row:
        return None, None
    return float(row["dram_bytes_per_launch"]), row.get("source")


# ---------------------------------------------------------------------------------------------
def oracle_problem(w, dtype, n_problems, seed):
    """The same synthetic workload expressed for the CPU oracle (checker / cpu baseline only)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pddp_oracle as O
    geo, D, ang, nonang = GEOMETRY[w["problem"]]
    Q, R, Qt, goal = cost_constants(w["problem"], dtype)
    cost = O.QRCostSpec(Q, R, Qt, goal, torch.zeros(ACTION_SIZE.get(w["problem"], 1), dtype=dtype), D, ang, nonang)
    if w["P"]:
        W, b, masks, eps0 = synth_bnn(w["problem"], w["P"], w["hidden"], seed)
        dyn = O.BNNSpec(list(zip(W, b)), masks, eps0, D, 1, ang, nonang).to(dtype)
    else:
        dyn = {"pendulum": O.pendulum_spec, "rendezvous": O.rendezvous_spec}[w["problem"]](*KNOWN_PARAMS[w["problem"]])
    z0, U = synth_inputs(dict(w, B=max(n_problems, 1)), seed + 1, dtype)
    return O, dyn, cost, z0, U


def oracle_iteration(O, dyn, cost, z0, U, w, dtype):
    """One problem-iteration of the reference algorithm: linearise, backward, rollout of every alpha, cost, argmin
    (pddp/controllers/ilqr.py:183-235 with mu = 1, as in the GPU step)."""
    nu = ACTION_SIZE.get(w["problem"], 1)
    lo, hi = torch.full((nu,), -w["umax"], dtype=dtype), torch.full((nu,), w["umax"], dtype=dtype)
    alphas = O.fit_alphas(dtype, w["A"])
    lin = O.linearize(z0, U, dyn, cost, w["enc"], lo, hi)
    try:
        k, K = O.backward_pass(*lin, reg=1.0, u_min=lo, u_max=hi, U=U)
        Zb, Ub = O.rollout(dyn, lin[0], U, k, K, alphas, w["enc"], lo, hi)
        O.trajectory_cost(cost, Zb, Ub, w["enc"]).argmin()
    except RuntimeError:
        pass


def time_oracle(w, dtype, n_problems, passes, budget_s, seed=0):
    """Warm-up, then `passes` timed sweeps over `n_problems` problems, sequentially (the reference optimises one
    problem at a time, SURVEY.md section 2 note).  Stops early once the budget is spent and at least 3
    problem-iterations are timed.  Returns the list of seconds per problem-iteration."""
    O, dyn, cost, z0, U = oracle_problem(w, dtype, n_problems, seed)
    warm = dict(w, N=min(w["N"], 5))
    oracle_iteration(O, dyn, cost, z0[0], U[0, :warm["N"]], warm, dtype)          # warm-up (autograd / thread pools)
    times, t_start = [], time.perf_counter()
    for _ in range(passes):
        for i in range(n_problems):
            t0 = time.perf_counter()
            oracle_iteration(O, dyn, cost, z0[i], U[i], w, dtype)
            times.append(time.perf_counter() - t0)
            if len(times) >= 3 and time.perf_counter() - t_start > budget_s:
                return times
    return times


def cpu_baseline_record(w, budget_s=30.0):
    """BASELINE.md section 3: warm-up + >= 3 timed problem-iterations over min(B, 8) problems, all host cores."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = min(w["B"], 8)
    times = time_oracle(w, torch.float32, n, passes=3, budget_s=budget_s)
    mean = sum(times) / len(times)
    return {"value": w["N"] / mean, "unit": "trajectory-steps/s", "cores": cores, "kind": "port",
            "sample": "warm-up + %d timed problem-iterations over %d problem(s) of the same workload, %.2f s each "
                      "(min %.2f, max %.2f); the reference handles one problem at a time, so the batch figure is "
                      "extrapolated from these" % (len(times), min(n, len(times)), mean, min(times), max(times))}


def run_reference(args, w, rank):
    """--impl reference: the reference's algorithm on the host CPU (oracle port; the reference is
    pure Python and cannot travel to the GPU box, see DESIGN.md)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dtype = torch.float32
    O, dyn, cost, z0, U = oracle_problem(w, dtype, min(w["B"], 8), 0)
    warm = dict(w, N=min(w["N"], 5))
    for _ in range(max(1, min(args.warmup, 2))):
        oracle_iteration(O, dyn, cost, z0[0], U[0, :warm["N"]], warm, dtype)
    t0 = time.perf_counter()
    for i in range(args.steps):                      # one step = one problem-iteration (problems cycle)
        oracle_iteration(O, dyn, cost, z0[i % z0.shape[0]], U[i % z0.shape[0]], w, dtype)
    sec = time.perf_counter() - t0
    value = w["N"] * args.steps / sec
    line = {"impl": "reference", "metric": "trajectory-steps/s", "value": value, "unit": "trajectory-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, w),
            "cpu_baseline": {"value": value, "unit": "trajectory-steps/s", "cores": cores, "kind": "port",
                             "sample": "1 problem x 1 iteration per step over %d distinct problems (the reference "
                                       "handles one problem at a time; whole-batch time = B x this)" % min(w["B"], 8)},
            "e2e": {"value": value, "unit": "trajectory-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def enc_size(w):
    D = GEOMETRY[w["problem"]][1]
    return {4: D, 1: (3 * D + D * D) // 2, 0: D * (1 + D)}[w["enc"]]


def workload_config(name, w):
    return {"workload": name, "problems_per_gpu": w["B"], "horizon": w["N"], "particles": w["P"],
            "alphas": w["A"], "nz": enc_size(w), "hidden": [w["hidden"]] * 2 if w["hidden"] else None,
            "encoding": {0: "FULL_COVARIANCE_MATRIX", 1: "UPPER_TRIANGULAR_CHOLESKY", 4: "IGNORE_UNCERTAINTY"}[w["enc"]],
            "bounded": True, "mu": 1.0, "l2": "inputs_exceed_l2 (per-step working set >> 126 MB)" if w["B"] > 64 else
            "working set fits L2 (single problem; launch-latency bound)",
            "parallelism": "independent problems sharded per GPU, no collective in the iteration"}


# ---------------------------------------------------------------------------------------------
# Algorithmic work per trajectory-step (SURVEY.md 8d): elements moved through HBM by each stage, MLP flops
# ---------------------------------------------------------------------------------------------
def stage_elements(nz, nu):
    E_lw = 2 * nz * nz + 2 * nz * nu + 2 * nz + nu + nu * nu + 1          # linearise writes Z,F_z,F_u,L,L_z,L_u,L_zz,L_uz,L_uu
    E_br = 2 * nz * nz + 2 * nz * nu + nz + nu + nu * nu                  # backward reads
    cost_w = 1 + nz + nu + nz * nz + nu * nz + nu * nu
    return {
        "linearize_known": E_lw + nu,
        "moment_linearise": nz * nz + nz * nu + nz,                       # F_z, F_u, Z[t+1] written by the BNN linearise step
        "cost": cost_w + nz + nu,
        "backward": E_br + nu + nu * nz,
        "rollout_known": (nz + 2 * nu + nu * nz) + (nz + nu),
        "rollout_step": (nz + 2 * nu + nu * nz) + (nz + nu),
        "accept": 2 * (nz + nu) + 2 * nu * nz,
        "whole_pass": (E_lw + nu) + (E_br + nu + nu * nz) + (nz + 2 * nu + nu * nz) + (nz + nu),
    }


def mlp_tile_flops(w):
    """Tensor FLOPs the tcgen05 kernel EXECUTES per 128-row tile, averaged over the particles (bnn_mlp_tc.cuh): for
    particle p layer 1 = 3 split-FP16 passes of M128 x N(p) x K16 per K-block, with K(p) = kept layer-0 units + the
    bias unit and N(p) = kept layer-1 units, both rounded up to 16 (units whose dropout mask is below 2^-24 are
    compacted away); layer 0 = 2 (3 when the input needs 16 columns) MMAs of M128 x N32 x K16 per 32-unit chunk.
    Compare with the algorithmic 2 * MACs per row."""
    _, D, ang, _ = GEOMETRY[w["problem"]]
    _, _, masks, _ = synth_bnn(w["problem"], w["P"], w["hidden"], seed=0)
    compact = os.environ.get("PDDP_MLP_COMPACT", "1") != "0"
    keep = [(m >= 2.0 ** -24) if compact else torch.ones_like(m, dtype=torch.bool) for m in masks]
    nkb = (keep[0].sum(1) + 1 + 15) // 16
    ncol = ((keep[1].sum(1) + 15) // 16 * 16).clamp_min(16)
    l0_mmas = 2 if D + len(ang) + 2 <= 8 else 3
    per_particle = 2.0 * 128 * (3 * nkb * ncol * 16 + l0_mmas * ((nkb + 1) // 2) * 32 * 16)
    return float(per_particle.double().mean())


def build_solver(name, dtype, dev, rank, B=None):
    from pddp_b200.solver import BatchedSolver, BNNDynamics, KnownDynamics, QRCostConstants
    w = dict(WORKLOADS[name])
    if B is not None:
        w["B"] = B
    geo, D, ang, nonang = GEOMETRY[w["problem"]]
    cost = QRCostConstants(*cost_constants(w["problem"]))
    if w["P"]:
        dyn = BNNDynamics(geo, *synth_bnn(w["problem"], w["P"], w["hidden"], seed=0))
    else:
        dyn = KnownDynamics(geo, KNOWN_PARAMS[w["problem"]])
    solver = BatchedSolver(dyn, cost, w["enc"], w["B"], w["N"], dtype=dtype, device=dev, max_alphas=w["A"])
    z0_h, U_h = synth_inputs(w, seed=1 + rank, dtype=dtype)
    nu = ACTION_SIZE.get(w["problem"], 1)
    lo, hi = [-w["umax"]] * nu, [w["umax"]] * nu
    alphas = (1.025 ** (-torch.arange(float(w["A"]), dtype=torch.float64) ** 2)).to(dtype)
    solver.set_problem(z0_h.to(dev), U_h.to(dev), lo, hi, alphas=alphas, iterations=1 << 30)
    return w, solver, z0_h, U_h, lo, hi, alphas


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(solver, out_dir, limit=DUMP_LIMIT_BYTES, seed=0):
    """Writes what `iLQRController.fit` hands its caller after the last pass -- trajectories Z [B,N+1,nz], controls
    U [B,N,nu], the gains of the last accepted step K [B,N,nu,nz], the accepted costs J_opt [B] and the per-problem
    iLQRState [B] -- as <out_dir>/<name>.npy in the solver's dtype (state as float32), with problem_index.npy
    (float64) naming the problems written.  When the whole batch would pass `limit` bytes, a fixed seeded sample
    of problems is written instead."""
    arrays = {"Z": solver.view("Z"), "U": solver.view("U"), "K": solver.matrices("K_nominal"), "J_opt": solver.J_opt,
              "state": solver.state.float()}
    per_problem = 8 + sum(t[0].numel() * t.element_size() for t in arrays.values())
    room = limit - 128 * (len(arrays) + 1)                    # less one .npy header per file
    idx = torch.arange(solver.B)
    if per_problem * solver.B > room:
        idx = torch.randperm(solver.B, generator=torch.Generator().manual_seed(seed))[:room // per_problem].sort().values
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "problem_index.npy"), idx.double().numpy())
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[idx.to(t.device)].cpu().numpy())


def measure(name, dtype, steps, warmup, dev, rank, world, dist, B=None, profile=True, dump_dir=None):
    """Device-timed passes of one workload + per-kernel times from CUDA events on the launch stream.  With
    `dump_dir`, rank 0 writes the outputs of the last timed pass there (dump_outputs), before the profiled pass."""
    from pddp_b200 import _lib
    lib = _lib.load()
    w, solver, z0_h, U_h, lo, hi, alphas = build_solver(name, dtype, dev, rank, B)

    def step():
        # every problem stays in play with a fixed regularisation so the work per step is constant
        solver.active.fill_(1)
        solver.mu.fill_(1.0)
        solver.iterate()

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(warmup):
        step()
    sync_all()
    not_pd = int((solver.bw_status != 0).sum().item())
    launches0 = int(lib.pddp_launch_count())
    sampler = ClockSampler(dev.index) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    launches = int(lib.pddp_launch_count()) - launches0
    clocks = sampler.stop() if sampler else None
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    not_pd = max(not_pd, int((solver.bw_status != 0).sum().item()))
    if dump_dir is not None and rank == 0:
        dump_outputs(solver, dump_dir)
    rec = {"w": w, "solver": solver, "ms_per_step": ms / steps, "value": world * w["B"] * w["N"] * steps / (ms * 1e-3),
           "launches": launches, "clocks": clocks, "not_pd": not_pd, "step": step, "sync_all": sync_all,
           "host": (z0_h, U_h, lo, hi, alphas), "kernels": None}
    if profile:
        n = len(PROFILE_KINDS)
        lib.pddp_profile_enable(1)
        step()
        pms, pcnt = (C.c_double * n)(), (C.c_int64 * n)()
        _lib.check(lib.pddp_profile_read(pms, pcnt), "profile_read")
        lib.pddp_profile_enable(0)
        rec["kernels"] = {k: (pms[i], int(pcnt[i])) for i, k in enumerate(PROFILE_KINDS) if pcnt[i]}
    return rec


def roofline_record(name, rec, dtype, peaks):
    """`roofline` of a workload: the dominant kernel against its bound, plus every profiled kernel with its own
    fraction (HBM kernels: algorithmic bytes / event time / measured copy bandwidth; MLP: algorithmic and executed
    tensor FLOP/s against the measured sustained bf16 rate)."""
    hbm_peak, tensor_peak, peak_src = peaks
    w, solver = rec["w"], rec["solver"]
    s = 4 if dtype == torch.float32 else 8
    nz, nu, BN = solver.nz, solver.nu, w["B"] * w["N"]
    elems = stage_elements(nz, nu)
    ms_step = rec["ms_per_step"]
    kernels = {}
    tc_path = bool(w["P"]) and dtype == torch.float32 and 64 < w["hidden"] <= 207
    rows = {}
    if w["P"]:
        geo, D, ang, _ = GEOMETRY[w["problem"]]
        macs = sum(a * b_ for a, b_ in zip([D + len(ang) + 1, w["hidden"], w["hidden"]], [w["hidden"], w["hidden"], 2 * D]))
        rows = {"mlp_linearise": w["B"] * w["P"] * (1 + D + 1), "mlp_rollout": w["B"] * w["A"] * w["P"]}
    for kind, (ms, cnt) in (rec["kernels"] or {}).items():
        k = {"launches_per_step": cnt, "avg_ms": ms / cnt, "ms_per_step": ms, "share_of_step": ms / ms_step}
        if kind in rows:
            flops = 2.0 * macs * rows[kind]                       # per launch (one time step of the whole batch)
            k.update(bound="tensor", algorithmic_flops_per_launch=flops,
                     achieved_tflops=flops / (ms / cnt * 1e-3) / 1e12,
                     frac=flops / (ms / cnt * 1e-3) / 1e12 / tensor_peak)
            if tc_path:
                tiles = w["P"] * math.ceil(rows[kind] / w["P"] / 128)
                ex = tiles * mlp_tile_flops(w)
                k.update(executed_tflops=ex / (ms / cnt * 1e-3) / 1e12, executed_per_algorithmic=ex / flops,
                         executed_frac_of_peak=ex / (ms / cnt * 1e-3) / 1e12 / tensor_peak)
        elif kind in elems:
            nbytes = elems[kind] * s * BN                         # per step (all launches of the kind together)
            k.update(bound="hbm", algorithmic_bytes_per_step=nbytes, achieved_gbs=nbytes / (ms * 1e-3) / 1e9,
                     frac=nbytes / (ms * 1e-3) / 1e9 / hbm_peak)
        kernels[kind] = k
    if w["P"] and kernels:
        dom = max(("mlp_linearise", "mlp_rollout"), key=lambda k_: kernels.get(k_, {}).get("ms_per_step", 0.0))
        d = kernels[dom]
        traffic, tsrc = committed_traffic(name, dom)
        return {"bound": "tensor", "kernel": "bnn_mlp (%s rows)" % dom.split("_")[1], "achieved": d["achieved_tflops"],
                "peak": tensor_peak, "unit": "TFLOP/s", "frac": d["frac"], "traffic": traffic, "traffic_source": tsrc,
                "peak_source": "bf16 dense sustained, " + peak_src,
                "executed_tflops": d.get("executed_tflops"), "executed_per_algorithmic": d.get("executed_per_algorithmic"),
                "tensor_passes_per_product": 3 if tc_path else None,
                "note": "achieved = ALGORITHMIC flops (2 x MACs per row) / mean launch time; executed_tflops = tensor "
                        "FLOPs the kernel issues (3 split-FP16 passes per fp32-accurate product + tile padding)",
                "flops_per_launch": d["algorithmic_flops_per_launch"], "avg_launch_ms": d["avg_ms"],
                "mlp_share_of_step": sum(kernels[k_]["ms_per_step"] for k_ in rows if k_ in kernels) / ms_step,
                "kernels": kernels}
    nbytes = elems["whole_pass"] * s * BN
    achieved = nbytes / (ms_step * 1e-3) / 1e9
    dom = max(kernels, key=lambda k_: kernels[k_]["ms_per_step"]) if kernels else None
    traffic, tsrc = committed_traffic(name, dom) if dom else (None, None)
    return {"bound": "hbm", "kernel": "whole pass (linearise+backward+rollout+accept); slowest kernel: %s" % dom,
            "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
            "traffic_source": tsrc, "peak_source": "copy bandwidth, " + peak_src, "kernels": kernels}


def controller_for(name, w, dtype):
    """The synthetic workload as the objects a user of the reference API holds (model, cost, controller)."""
    import pddp_b200 as P
    from pddp_b200.costs import QRCost
    geo, D, ang, nonang = GEOMETRY[w["problem"]]
    Q, R, Qt, goal = cost_constants(w["problem"], dtype)
    cost = QRCost(Q, R, Qt, goal, state_size=D, angular_indices=ang)
    if w["P"]:
        W, b, masks, eps0 = synth_bnn(w["problem"], w["P"], w["hidden"], seed=0)
        model = P.models.bnn.bnn_dynamics_model_factory(D, 1, [w["hidden"]] * 2, list(ang), list(nonang))(
            n_particles=w["P"]).to(dtype)
        model._store_flat(torch.cat([t.reshape(-1) for pair in zip(W, b) for t in pair] + [torch.zeros(2)]).to(dtype))
        model.model.drop_0.mask, model.model.drop_1.mask = masks[0].to(dtype), masks[1].to(dtype)
        model.eps_in = {0: eps0.to(dtype)}
        opts = {"use_predicted_std": False, "infer_noise_variables": True}
    else:
        cls = {"pendulum": P.examples.pendulum.PendulumDynamicsModel,
               "rendezvous": P.examples.rendezvous.RendezvousDynamicsModel}[w["problem"]]
        model, opts = cls(*KNOWN_PARAMS[w["problem"]]).to(dtype), {}
    return P.controllers.iLQRController(None, model, cost, model_opts=opts)


def measure_e2e(name, rec, dtype, steps, dev, world, dist):
    """The same metric through the public API -- `iLQRController.fit(U, z0=..., n_iterations=1, max_passes=1)` --
    with HOST buffers: every step copies z0 / U from pinned host memory and reads Z, U, state (and J) back."""
    w = rec["w"]
    z0_h, U_h, lo, hi, _ = rec["host"]
    z0_h, U_h = z0_h.pin_memory(), U_h.pin_memory()
    ctrl = controller_for(name, w, dtype)
    nz, nu = enc_size(w), ACTION_SIZE.get(w["problem"], 1)
    Z_h = torch.empty(w["B"], w["N"] + 1, nz, dtype=dtype).pin_memory()
    Uo_h = torch.empty(w["B"], w["N"], nu, dtype=dtype).pin_memory()
    st_h = torch.empty(w["B"], dtype=torch.int32).pin_memory()
    lo_d, hi_d = torch.tensor(lo, dtype=dtype, device=dev), torch.tensor(hi, dtype=dtype, device=dev)
    h2d = z0_h.numel() * z0_h.element_size() + U_h.numel() * U_h.element_size()
    d2h = sum(t.numel() * t.element_size() for t in (Z_h, Uo_h, st_h))

    def e2e_step():
        Z, U, state = ctrl.fit(U_h.to(dev, non_blocking=True), encoding=w["enc"], n_iterations=1, max_passes=1,
                               u_min=lo_d, u_max=hi_d, z0=z0_h.to(dev, non_blocking=True), shard=False, quiet=True)
        Z_h.copy_(Z, non_blocking=True)
        Uo_h.copy_(U, non_blocking=True)
        st_h.copy_(state, non_blocking=True)
        torch.cuda.synchronize(dev)

    e2e_step()
    e2e_step()
    rec["sync_all"]()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        e2e_step()
    e1.record()
    rec["sync_all"]()
    ms = torch.tensor([max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    states = torch.bincount(st_h.long(), minlength=6).tolist()
    return {"value": world * w["B"] * w["N"] * steps / (float(ms.item()) * 1e-3), "unit": "trajectory-steps/s",
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "api": "iLQRController.fit(U[B,N,nu], z0=[B,nz], n_iterations=1, max_passes=1) from pinned host buffers",
            "states_after_one_pass": dict(zip(("undefined", "accepted", "rejected", "not_pd", "max_reg", "converged"), states))}


def measure_api_latency(dev, reps=20):
    """Level-2 drop-in (INTEGRATION.md): the reference's module-level functions called the way its own `step()` calls
    them, ONE problem at a time (pendulum, known dynamics, N = 100, 10 alphas) -- wall-clock milliseconds per call with
    cached device buffers, including every host-side marshalling step and a device synchronisation."""
    import pddp_b200 as P
    from pddp_b200.controllers.ilqr import _control_law, _trajectory_cost, backward, forward
    model, cost = P.examples.pendulum.PendulumDynamicsModel(0.1), P.examples.pendulum.PendulumCost()
    enc = P.StateEncoding.IGNORE_UNCERTAINTY
    g = torch.Generator().manual_seed(0)
    z0 = (1e-2 * torch.randn(2, generator=g)).to(dev)
    U = (0.1 * torch.randn(100, 1, generator=g)).to(dev)
    alphas = (1.025 ** (-torch.arange(10.0) ** 2)).to(dev)
    out = {}

    def timed(name, fn):
        fn()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        torch.cuda.synchronize(dev)
        out[name + "_ms"] = (time.perf_counter() - t0) * 1e3 / reps
        return r

    lin = timed("forward", lambda: forward(z0, U, model, cost, enc))
    k, K = timed("backward", lambda: backward(*lin, reg=1.0))
    Zb, Ub = timed("control_law_10_alphas", lambda: _control_law(model, lin[0], U, k, K, alphas, enc))
    timed("trajectory_cost", lambda: _trajectory_cost(cost, Zb, Ub, enc))
    ctrl = P.controllers.iLQRController(None, model, cost)
    timed("controller_fit_1_iteration", lambda: ctrl.fit(U, encoding=enc, n_iterations=1, z0=z0, quiet=True))
    out["iteration_ms"] = out["forward_ms"] + out["backward_ms"] + out["control_law_10_alphas_ms"] + out["trajectory_cost_ms"]
    out["trajectory_steps_per_s"] = 100 / (out["iteration_ms"] * 1e-3)
    out["what"] = ("pendulum known dynamics, one problem, N = 100: forward / backward / _control_law / _trajectory_cost "
                   "(reference signatures) and iLQRController.fit(n_iterations=1); launch-latency bound by construction")
    return out


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cartpole_bnn_b4096", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the other_workloads / strong sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed pass (rank 0's "
                    "problems) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, w, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch.distributed as dist
    from pddp_b200 import sharding

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float32 if args.dtype == "f32" else torch.float64
    peaks = measured_peaks()

    rec = measure(args.workload, dtype, args.steps, args.warmup, dev, rank, world, dist, dump_dir=args.dump_outputs)
    roofline = roofline_record(args.workload, rec, dtype, peaks)
    e2e = measure_e2e(args.workload, rec, dtype, args.steps, dev, world, dist)

    # ---- final exchange of the results over NCCL (outside the timed iteration): Z, U, J, state in one all-gather,
    #      timed with CUDA events AFTER a first call has set the channels up -----------------------------------
    gather = None
    if world > 1:
        s = rec["solver"]
        parts = [s.view("Z").contiguous(), s.view("U").contiguous(), s.J_opt, s.state]
        sharding.all_gather_problems(parts, world * w["B"])
        torch.cuda.synchronize(dev)
        dist.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        full = sharding.all_gather_problems(parts, world * w["B"])
        g1.record()
        torch.cuda.synchronize(dev)
        gms = torch.tensor([g0.elapsed_time(g1)], device=dev, dtype=torch.float64)
        dist.all_reduce(gms, op=dist.ReduceOp.MAX)
        nbytes = sum(t.numel() * t.element_size() for t in parts)
        gather = {"ms": float(gms.item()), "bytes_per_rank": nbytes, "tensors": "Z, U, J, state",
                  "gbs_per_rank_received": (world - 1) * nbytes / (float(gms.item()) * 1e-3) / 1e9,
                  "rows_gathered": int(full[0].shape[0])}
        del full
    del rec["solver"], rec["step"]
    torch.cuda.empty_cache()

    # ---- strong scaling: configs[1]'s 4096 problems split over the ranks -----------------------------------------
    strong = None
    if world > 1 and not args.no_others:
        total_B = WORKLOADS[args.workload]["B"]
        lo_, hi_ = sharding.shard_bounds(total_B, world, rank)
        r2 = measure(args.workload, dtype, max(3, args.steps // 2), 3, dev, rank, world, dist, B=hi_ - lo_, profile=False)
        strong = {"problems_total": total_B, "problems_per_gpu": hi_ - lo_, "ms_per_step": r2["ms_per_step"],
                  "value": total_B * w["N"] / (r2["ms_per_step"] * 1e-3), "unit": "trajectory-steps/s", "scaling": "strong"}
        del r2
        torch.cuda.empty_cache()

    # ---- the other BASELINE configurations, a few steps each (single GPU only) -----------------------------------
    others = None
    if world == 1 and not args.no_others:
        others = []
        for name, dt in OTHER_WORKLOADS:
            if name == args.workload and dt == args.dtype:
                continue
            d = torch.float32 if dt == "f32" else torch.float64
            try:
                r = measure(name, d, 3, 3, dev, 0, 1, dist)
                rf = roofline_record(name, r, d, peaks)
                others.append({"workload": name, "dtype": dt, "config": workload_config(name, r["w"]),
                               "ms_per_step": r["ms_per_step"], "value": r["value"], "unit": "trajectory-steps/s",
                               "steps": 3, "warmup": 3, "gpu_launches": r["launches"], "not_pd_problems": r["not_pd"],
                               "roofline": {k: v for k, v in rf.items() if k != "note"}})
                del r
            except Exception as exc:                          # a sub-record must never take the headline line down
                others.append({"workload": name, "dtype": dt, "error": "%s: %s" % (type(exc).__name__, exc)})
            torch.cuda.empty_cache()

    api = None
    if world == 1 and not args.no_others:
        try:
            api = measure_api_latency(dev)
        except Exception as exc:
            api = {"error": "%s: %s" % (type(exc).__name__, exc)}
    cpu = cpu_baseline_record(w) if rank == 0 and not args.no_cpu_baseline else None
    if rank == 0:
        line = {"metric": "trajectory-steps/s", "value": rec["value"], "unit": "trajectory-steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                "config": workload_config(args.workload, w), "clocks": rec["clocks"], "e2e": e2e,
                "gpu_launches": rec["launches"], "roofline": roofline, "cpu_baseline": cpu,
                "not_pd_problems": rec["not_pd"], "final_gather": gather, "strong": strong, "other_workloads": others,
                "api_latency": api}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True          # the tree may be read-only; nothing of a run is written into it
    main()
