"""Cost of per-step goals: device-timed passes (linearise + backward + line search + accept) of bench.py's workloads
with the cost's shared goal, with x_goal [B, DA] / u_goal [B, nu] per problem, and with x_goal [B, N+1, DA] /
u_goal [B, N, nu] per problem and step.  The three settings alternate, run after run, in one process.  Prints one
JSON line, with the card's name, power limit and clocks read in the same call.

Per launch that reads the cost, a per-step goal adds (DA + nu) * sizeof(T) bytes per problem and step: 16 B for the
fp32 pendulum (B = 2^20, N = 100: 1.7 GB per pass over linearise and the rollout's cost), 48 B for fp32 rendezvous.

    python tools/bench_goal_trajectories.py [--steps 10 --warmup 3 --runs 5
        --workloads pendulum_known_b1m,rendezvous_known_b64k,cartpole_bnn_b4096]
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

SETTINGS = ("shared", "per_problem", "per_step")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return out or None
    except OSError:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--workloads", default="pendulum_known_b1m,rendezvous_known_b64k,cartpole_bnn_b4096")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_goal_trajectories.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    dtype = torch.float32
    rec = {"card": card(), "dtype": "f32", "steps": args.steps, "runs": args.runs}
    for name in args.workloads.split(","):
        w, solver, *_ = bench.build_solver(name, dtype, dev, 0)
        c = solver.cost
        B, N, DA, nu = solver.B, solver.N, c.Q.shape[0], solver.nu
        g = torch.Generator().manual_seed(3)
        x_goal = c.x_goal.reshape(1, DA) + 0.05 * torch.randn(B, DA, generator=g, dtype=torch.float64)
        u_goal = c.u_goal.reshape(-1).expand(nu).reshape(1, nu) + 0.05 * torch.randn(B, nu, generator=g,
                                                                                   dtype=torch.float64)
        x_goal, u_goal = x_goal.to(dtype=dtype, device=dev), u_goal.to(dtype=dtype, device=dev)
        # a drifting reference around each problem's goal
        ramp = torch.linspace(0, 0.1, N + 1, dtype=dtype, device=dev).reshape(1, N + 1, 1)
        x_goal_t = x_goal.unsqueeze(1) + ramp
        u_goal_t = u_goal.unsqueeze(1) + ramp[:, :N]
        goals = {"shared": (None, None), "per_problem": (x_goal, u_goal), "per_step": (x_goal_t, u_goal_t)}

        def step():
            # every problem stays in play with a fixed regularisation, as in bench.py: constant work per pass
            solver.active.fill_(1)
            solver.mu.fill_(1.0)
            solver.iterate()

        def timed(setting):
            solver.set_goals(*goals[setting])
            for _ in range(args.warmup):
                step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / args.steps

        ms = {k: [] for k in SETTINGS}
        for _ in range(args.runs):
            for k in SETTINGS:
                ms[k].append(round(timed(k), 4))
        med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
        rec[name] = {"B": w["B"], "N": w["N"], **{"ms_per_pass_" + k: v for k, v in ms.items()},
                     "median_ratio_per_problem": round(med["per_problem"] / med["shared"], 4),
                     "median_ratio_per_step": round(med["per_step"] / med["shared"], 4)}
        del solver
        torch.cuda.empty_cache()
    rec["card_after"] = card()
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
