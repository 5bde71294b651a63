#!/usr/bin/env python
"""Episode resets of the reference's seeded scenes: the per-episode host work BatchedEnv.reset_batch used to do
(SceneGenerator.generate_random_scene + rects_from_zero_cells + padded arrays + the upload) against the device replay
it does now (one ebc_replay_scenes launch + reading the counts back), both ending in a device synchronise.

    python tools/scene_replay_rate.py [--config env_ebcadrl.config] [--episodes 256 4096] [--repeat 3] [--out FILE]

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

from ebc.batched_env import BatchedEnv  # noqa: E402
from host_scenes import host_batch  # noqa: E402


def host_reset(env, phase, seeds):
    """The per-episode host loop reset_batch ran before the device replay, with its upload."""
    z = host_batch(env, phase, seeds, restore_counter=False)
    n, rad = len(seeds), env.scene.circle_radius
    poly_xy = torch.as_tensor(z["poly_xy"]).to(env.device)
    rob_pv = np.tile(np.array([0, -rad, 0, 0], np.float32), (n, 1))
    rob_gr = np.tile(np.array([0, rad, env.robot.v_pref, env.robot.radius], np.float32), (n, 1))
    env.sim.load_episodes(0, z["hum_pv"], z["hum_gr"], z["hum_type"], z["hum_count"], z["stat"], z["stat_count"],
                          z["rect"], z["rect_count"], rob_pv, rob_gr, np.full(n, np.pi / 2, np.float32), np.zeros(n))
    return poly_xy


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--config", default="env_ebcadrl.config", help="a config of tests/golden/configs")
    ap.add_argument("--phase", default="test")
    ap.add_argument("--episodes", type=int, nargs="+", default=[256, 4096])
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("scene_replay_rate: needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    cp = configparser.RawConfigParser()
    assert cp.read(os.path.join(REPO, "tests", "golden", "configs", args.config))
    result = {"config": args.config, "phase": args.phase, "device": torch.cuda.get_device_name(0), "nvidia_smi": smi,
              "runs": []}
    for n in args.episodes:
        env = BatchedEnv(cp, None, n, "cuda:0")
        seeds = np.arange(1000000, 1000000 + n)
        torch.cuda.synchronize()
        free_before = torch.cuda.mem_get_info(0)[0]
        env.reset_batch(args.phase, seeds)                       # warm-up: module load, config, allocations
        torch.cuda.synchronize()
        # device memory the first launch took beyond the call's own outputs: mostly the local-memory (stack) reservation
        # the driver makes for the kernel's per-thread stack at the device's full resident-thread capacity
        first_launch = free_before - torch.cuda.mem_get_info(0)[0]
        host = [timed(lambda: host_reset(env, args.phase, seeds)) for _ in range(args.repeat)]
        dev = [timed(lambda: env.reset_batch(args.phase, seeds)) for _ in range(max(args.repeat, 10))]
        result["runs"].append({"episodes": n, "first_launch_device_bytes": int(first_launch), "host_loop_s": min(host),
                               "host_loop_ms_per_scene": min(host) / n * 1e3,
                               "reset_batch_s": min(dev), "reset_batch_median_s": float(np.median(dev)),
                               "ratio": min(host) / min(dev)})
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
