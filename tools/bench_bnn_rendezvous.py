"""Learned-model PDDP on the rendezvous problem (D = 8, action_size 4, UPPER_TRIANGULAR_CHOLESKY): device-timed passes
(linearise + backward + line search + accept) of B problems with a BNN of two hidden layers of H units, in fp32
(tcgen05 particle MLP) and fp64 (CUDA-core particle MLP).  Prints one JSON line.

bench.py's synth_bnn builds networks with one control input, so the network is built here with input width
D + nu = 12 and the same initialisation; inputs, cost constants, peaks, the clock sampler and the per-stage profiling
events are bench.py's.

MLP work per trajectory-step (algorithmic, 2 FLOP per multiply-add): 2 W P (1 + T + A) with
W = 12 x 200 + 200 x 200 + 200 x 16 = 45 600 weights, T = D + nu = 12 tangent rows per particle in the
linearisation and A line-search candidates in the rollout: 104.9 MFLOP at P = 50, A = 10.

    python tools/bench_bnn_rendezvous.py [--steps 10 --warmup 3 --steps-f64 2 --dtypes f32,f64 --out FILE]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

D, NU = 8, 4


def synth_bnn(P, H, seed):
    """bench.synth_bnn with input width D + nu (Xavier-normal with ReLU gain, biases U(-0.1, 0.1), concrete-dropout
    eval masks, standardised eps0)."""
    g = torch.Generator().manual_seed(seed)
    dims = [D + NU, H, H, 2 * D]
    W, b = [], []
    for din, dout in zip(dims[:-1], dims[1:]):
        W.append(torch.randn(dout, din, generator=g) * math.sqrt(2.0) * math.sqrt(2.0 / (din + dout)))
        b.append(torch.rand(dout, generator=g) * 0.2 - 0.1)
    W[-1] *= 0.02
    b[-1] *= 0.02
    masks = []
    for _ in range(2):
        r = torch.rand(P, H, generator=g).clamp(1e-6, 1 - 1e-6)
        masks.append(torch.sigmoid((r.log() - (1 - r).log()) / 0.1))
    eps = torch.randn(P, D, generator=g)
    return W, b, masks, (eps - eps.mean(0)) / eps.std(0)


def card():
    """Name and power limit of GPU 0, read with the measurement."""
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, mx = [x.strip() for x in out.strip().split(",")[:2]]
        return {"name": name, "power_limit_w": float(pl), "sm_max_mhz": float(mx)}
    except Exception as e:                                   # the numbers are reported without it
        return {"name": name, "power_limit_w": None, "error": repr(e)}


def mlp_kernel(dtype, H):
    """The particle-MLP kernel bnn_mlp.cu dispatches to (use_tensor_cores: fp32 and 64 < H, H + 1 <= 208)."""
    tc = dtype == torch.float32 and 64 < H and H + 1 <= 208 and os.environ.get("PDDP_FORCE_SIMT", "0") != "1"
    return "bnn_mlp_tc_kernel (tcgen05)" if tc else "bnn_mlp_simt_kernel (CUDA cores)"


def run(w, dtype, steps, warmup):
    from pddp_b200 import _lib
    from pddp_b200.solver import BatchedSolver, BNNDynamics, QRCostConstants
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    W, b, masks, eps0 = synth_bnn(w["P"], w["hidden"], seed=0)
    solver = BatchedSolver(BNNDynamics(_lib.GEO_RENDEZVOUS, W, b, masks, eps0),
                           QRCostConstants(*bench.cost_constants("rendezvous")), w["enc"], w["B"], w["N"],
                           dtype=dtype, device=dev, max_alphas=w["A"])
    z0, U = bench.synth_inputs(w, seed=1, dtype=dtype)
    alphas = (1.025 ** (-torch.arange(float(w["A"]), dtype=torch.float64) ** 2)).to(dtype)
    solver.set_problem(z0.to(dev), U.to(dev), [-w["umax"]] * NU, [w["umax"]] * NU, alphas=alphas, iterations=1 << 30)

    def step():                     # as bench.py: every problem stays in play at a fixed regularisation
        solver.active.fill_(1)
        solver.mu.fill_(1.0)
        solver.iterate()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    sampler = bench.ClockSampler(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    clocks = sampler.stop()
    not_pd = int((solver.bw_status != 0).sum().item())
    finite = bool(torch.isfinite(solver.view("Z")).all().item() and torch.isfinite(solver.J_opt).all().item())
    # one more pass with the library's per-stage CUDA events (a separate pass: the events serialise the stream)
    n = len(bench.PROFILE_KINDS)
    lib.pddp_profile_enable(1)
    step()
    pms, pcnt = (C.c_double * n)(), (C.c_int64 * n)()
    _lib.check(lib.pddp_profile_read(pms, pcnt), "profile_read")
    lib.pddp_profile_enable(0)
    stages = {k: round(pms[i], 4) for i, k in enumerate(bench.PROFILE_KINDS) if pcnt[i]}
    H, P, A, T = w["hidden"], w["P"], w["A"], D + NU
    weights = (D + NU) * H + H * H + H * 2 * D
    steps_per_pass = w["B"] * w["N"]
    f_lin, f_roll = 2.0 * weights * P * (1 + T) * steps_per_pass, 2.0 * weights * P * A * steps_per_pass
    mlp_ms = stages.get("mlp_linearise", 0.0) + stages.get("mlp_rollout", 0.0)
    return {
        "dtype": "f32" if dtype == torch.float32 else "f64",
        "ms_per_pass": round(ms, 4),
        "trajectory_steps_per_s": steps_per_pass / (ms * 1e-3),
        "stage_ms": stages,
        "mlp_kernel": mlp_kernel(dtype, H),
        "mlp_mflop_per_trajectory_step": round((f_lin + f_roll) / steps_per_pass / 1e6, 2),
        "mlp_tflops": {"linearise": f_lin / (stages["mlp_linearise"] * 1e-3) / 1e12 if stages.get("mlp_linearise") else None,
                       "rollout": f_roll / (stages["mlp_rollout"] * 1e-3) / 1e12 if stages.get("mlp_rollout") else None,
                       "both": (f_lin + f_roll) / (mlp_ms * 1e-3) / 1e12 if mlp_ms else None},
        "steps_timed": steps, "warmup": warmup, "not_pd": not_pd, "finite": finite, "clocks": clocks,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--N", type=int, default=100)
    ap.add_argument("--P", type=int, default=50)
    ap.add_argument("--A", type=int, default=10)
    ap.add_argument("--H", type=int, default=200)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps-f64", type=int, default=2)
    ap.add_argument("--dtypes", default="f32,f64")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_bnn_rendezvous: needs a CUDA device")
    w = dict(problem="rendezvous", enc=1, B=args.B, N=args.N, P=args.P, A=args.A, hidden=args.H, umax=1.0)
    rec = {"workload": "rendezvous_bnn_b%d" % args.B, "card": card(), "problems": args.B, "horizon": args.N,
           "particles": args.P, "alphas": args.A, "hidden": [args.H, args.H], "encoding": "UPPER_TRIANGULAR_CHOLESKY",
           "nz": 44, "nu": NU, "u_bounds": [-1.0, 1.0], "peaks": dict(zip(("hbm_gbs", "fp16_dense_tflops", "source"),
                                                                         bench.measured_peaks())), "runs": []}
    for name in args.dtypes.split(","):
        dtype = {"f32": torch.float32, "f64": torch.float64}[name]
        steps = args.steps if dtype == torch.float32 else args.steps_f64
        rec["runs"].append(run(w, dtype, steps, 1 if dtype == torch.float64 else args.warmup))
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
