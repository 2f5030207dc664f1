"""Cost of per-problem goals: device-timed passes (linearise + backward + line search + accept) of bench.py's
workloads with the cost's shared goal against the same passes with x_goal [B, DA] / u_goal [B, nu] given per problem.
The two settings alternate, run after run, in one process.  Prints one JSON line.

Per launch that reads the cost, a problem's goal adds (DA + nu) * sizeof(T) bytes of reads: 16 B for the fp32
pendulum (B = 2^20: 16 MB per launch), 24 B for the fp32 cartpole.

    python tools/bench_goals.py [--steps 10 --warmup 3 --runs 5 --workloads pendulum_known_b1m,cartpole_bnn_b4096]
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


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return out or None
    except OSError:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--workloads", default="pendulum_known_b1m,cartpole_bnn_b4096")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_goals.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    dtype = torch.float32
    rec = {"card": card(), "dtype": "f32", "steps": args.steps, "runs": args.runs}
    for name in args.workloads.split(","):
        w, solver, *_ = bench.build_solver(name, dtype, dev, 0)
        c = solver.cost
        DA, nu = c.Q.shape[0], solver.nu
        g = torch.Generator().manual_seed(3)
        x_goal = (c.x_goal.reshape(1, DA) + 0.05 * torch.randn(solver.B, DA, generator=g, dtype=torch.float64))
        u_goal = c.u_goal.reshape(-1).expand(nu).reshape(1, nu) + 0.05 * torch.randn(solver.B, nu, generator=g,
                                                                                   dtype=torch.float64)
        x_goal, u_goal = x_goal.to(dtype=dtype, device=dev), u_goal.to(dtype=dtype, device=dev)

        def step():
            # every problem stays in play with a fixed regularisation, as in bench.py: constant work per pass
            solver.active.fill_(1)
            solver.mu.fill_(1.0)
            solver.iterate()

        def timed(per_problem):
            solver.set_goals(x_goal, u_goal) if per_problem else solver.set_goals()
            for _ in range(args.warmup):
                step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / args.steps

        shared, per = [], []
        for _ in range(args.runs):
            shared.append(round(timed(False), 4))
            per.append(round(timed(True), 4))
        rec[name] = {"B": w["B"], "N": w["N"], "ms_per_pass_shared_goal": shared, "ms_per_pass_per_problem_goal": per,
                     "median_ratio": round(sorted(per)[len(per) // 2] / sorted(shared)[len(shared) // 2], 4)}
        del solver
        torch.cuda.empty_cache()
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
