"""Cost of per-problem dynamics parameters: device-timed passes (linearise + backward + line search + accept) of
bench.py's known-dynamics workloads with the shared parameters, with per-problem rows p_b [B, 8] equal to the shared
values (the same work, read per problem), and with rows perturbed by up to +-20 %.  The three settings alternate, run
after run, in one process.  Prints one JSON line with the card, its power limit and clocks.

Per launch that integrates the dynamics, a problem's row adds nparams * sizeof(T) bytes of reads: 20 B for the fp32
pendulum (B = 2^20: 20 MB per launch, one 32-byte sector per problem), 12 B for the fp32 rendezvous.

    python tools/bench_dynamics_params.py [--steps 10 --warmup 3 --runs 5 --workloads pendulum_known_b1m,...]
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
from pddp_b200.solver import KnownDynamics  # noqa: E402


def query(fields):
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + fields, "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or None
    except OSError:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--workloads", default="pendulum_known_b1m,rendezvous_known_b64k")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dynamics_params.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    dtype = torch.float32
    rec = {"card": query("name,power.limit,clocks.max.sm"), "dtype": "f32", "steps": args.steps, "runs": args.runs}
    for name in args.workloads.split(","):
        w, solver, *_ = bench.build_solver(name, dtype, dev, 0)
        shared = solver.dyn
        k = len(shared.params)
        equal = torch.zeros(solver.B, 8, dtype=torch.float64)
        equal[:, :k] = torch.tensor(shared.params, dtype=torch.float64)
        g = torch.Generator().manual_seed(3)
        perturbed = equal * (1 + 0.2 * (2 * torch.rand(solver.B, 8, generator=g, dtype=torch.float64) - 1))
        settings = {"shared": shared, "per_problem_equal": KnownDynamics(shared.geo, shared.params, equal),
                    "per_problem_perturbed": KnownDynamics(shared.geo, shared.params, perturbed)}

        def step():
            # every problem stays in play with a fixed regularisation, as in bench.py: constant work per pass
            solver.active.fill_(1)
            solver.mu.fill_(1.0)
            solver.iterate()

        def timed(dyn):
            solver.set_dynamics(dyn)
            for _ in range(args.warmup):
                step()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / args.steps

        ms = {s: [] for s in settings}
        for _ in range(args.runs):
            for s, dyn in settings.items():
                ms[s].append(round(timed(dyn), 4))
        med = {s: sorted(v)[len(v) // 2] for s, v in ms.items()}
        rec[name] = {"B": w["B"], "N": w["N"], **{"ms_per_pass_" + s: v for s, v in ms.items()},
                     "median_ratio_equal": round(med["per_problem_equal"] / med["shared"], 4),
                     "median_ratio_perturbed": round(med["per_problem_perturbed"] / med["shared"], 4)}
        solver.set_dynamics(shared)
        del solver
        torch.cuda.empty_cache()
    rec["clocks_after"] = query("clocks.sm,power.draw,clocks_throttle_reasons.active")
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
