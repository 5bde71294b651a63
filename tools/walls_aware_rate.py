#!/usr/bin/env python
"""What walls-aware humans (`[sim] orca_obstacles = true`) cost on the reference's seeded scenes: BatchedEnv.reset_batch
(the scene replay, plus the obstacle build with the key on) and one decision plus committed step (ORCA, lookahead,
value network, selection, step; with the key on ORCA adds the obstacle half-planes), key off against key on, each
timed over a run that ends in a device synchronise.

    python tools/walls_aware_rate.py [--config env_ebcadrl.config] [--episodes 256 4096] [--repeat 20] [--out FILE]

Prints one JSON object with the card's name and power limit next to the times.
"""
import argparse
import configparser
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "eb-cadrl_b200"))
sys.path.insert(0, os.path.join(REPO, "tests"))

import torch  # noqa: E402

import oracle_backend as ob  # noqa: E402
from ebc.actions import build_action_space  # noqa: E402
from ebc.batched_env import BatchedEnv  # noqa: E402


def timed(fn, repeat):
    """Per-call seconds of `repeat` back-to-back calls, between two device synchronises."""
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(repeat):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) / repeat


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--config", default="env_ebcadrl.config", help="a config of tests/golden/configs")
    ap.add_argument("--phase", default="test")
    ap.add_argument("--episodes", type=int, nargs="+", default=[256, 4096])
    ap.add_argument("--repeat", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("walls_aware_rate: needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    weights = ob.load_weights("weights_sarl_baseline.npz")
    result = {"config": args.config, "phase": args.phase, "device": torch.cuda.get_device_name(0), "nvidia_smi": smi,
              "runs": []}
    for n in args.episodes:
        seeds = np.arange(1000, 1000 + n)
        for key in ("false", "true"):
            cp = configparser.RawConfigParser()
            assert cp.read(os.path.join(REPO, "tests", "golden", "configs", args.config))
            cp.set("sim", "orca_obstacles", key)
            env = BatchedEnv(cp, None, n, "cuda:0")
            sim = env.sim
            sim.set_actions(build_action_space(env.robot.v_pref))
            sim.set_weights(weights)
            sim.fused_input = sim.value_mode().startswith("tc")     # as BatchedEnv.sync_weights sets it
            env.reset_batch(args.phase, seeds)                      # warm-up: module load, configs, allocations
            reset = timed(lambda: env.reset_batch(args.phase, seeds), args.repeat)

            def decide_step():
                sim.step(action_idx=sim.decide())

            decide_step()                                           # warm-up of the decision's kernels
            env.reset_batch(args.phase, seeds)
            step = timed(decide_step, args.repeat)
            result["runs"].append({"episodes": n, "orca_obstacles": key == "true", "omax": sim.Omax,
                                   "reset_batch_ms": reset * 1e3, "decide_step_ms": step * 1e3})
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
