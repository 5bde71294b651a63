#!/usr/bin/env python
"""bench.py — throughput of the EB-CADRL hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] — EB-CADRL entity-typed agents + static
obstacles, 10 humans (4 adults + 3 bicycles + 3 children), 3 walls (6 static discs, n = 16 rows,
D = 17), 81 holonomic actions, 4096 parallel episodes PER GPU (weak scaling), synthetic scenes
(ebc/synth.py, counter-based RNG keyed by the global episode id), EB-CADRL value network
(379,202 parameters; the shipped rl_model_val weights fixture, else seeded random init).

One "step" = what the reference does per env step with the policy in the loop
(rl/utils/explorer.py:41-46): robot decision by one-step lookahead over all 81 actions
(ORCA for the humans, lookahead expansion, value network, argmax) + the committed env.step
+ re-initialisation of finished episodes.  Reported:
    value                 agent-steps/s  = episodes * (H + 1) / step time      (whole job, all GPUs)
    lookahead_evals_per_sec              = episodes * 81 / step time
    sim_only              the policy-free path (ORCA + step in one launch), its own timing
    roofline              the dominant kernel pair (K4 value network)
    e2e                   the same step through the host-facing API: pinned host state -> device,
                          decide + step, observation / reward / done / event -> pinned host
    cpu_baseline          the CPU oracle (port of the reference path) on this box's cores
    sustained             the same step back to back for >= 2 s (the board reaches its power cap there): its own
                          ms per step, clocks, K4 TFLOP/s -- `value` / `ms_per_step` are the driver's --steps region
`value` is the POLICY-IN-THE-LOOP metric (every agent-step pays a full 81-action lookahead through the value
network); `sim_only` is SURVEY 8d(i)'s committed-step path, the one north_star's 1e8 agent-steps/s target is
stated on.  `--workload cfg5` times the training loop instead (rl/train.py semantics, see run_cfg5).

`--dump-outputs DIR` writes what the last of the K timed steps handed back (DUMPED: values and action values of the
decision, the chosen action, reward / done / event, the state after the step and the re-initialisation) as
DIR/<name>.npy, so that two builds can be compared output for output: scenes and weights are fixed, so the same
arguments give the same inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "eb-cadrl_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch, from the committed
# `ncu --set full` capture (profiles/); None until a capture of that mode exists
ROOFLINE_TRAFFIC = {"fp32": 492.2e6, "tc_fp32": 490.3e6, "tc_fp16x2": 502.0e6, "tc_bf16": None}       # materialised input
ROOFLINE_TRAFFIC_FUSED = {"tc_fp16x2": 115.8e6}                                                            # fused input path
EPISODES_PER_GPU = 4096
N_ACTIONS = 81
METRIC = "agent_steps_per_sec"
UNIT = "agent-steps/s"
DUMPED = ("values", "action_values", "argmax", "reward", "done", "event", "hum_pv", "rob_pv")   # BatchedSim, [N, ...]
DUMP_BYTES = 64_000_000


WORKLOADS = {   # name -> (synth shape, robot kinematics, entity-typed rows, weights fixture, episodes per GPU)
    "cfg2": ("CFG2", "holonomic", True, "weights_ebcadrl.npz", 4096),          # BASELINE configs[1]: the bench line
    "cfg3": ("CFG3", "unicycle", False, "weights_sarl_baseline.npz", 16384),   # configs[2] (side measurement)
    "cfg4": ("CFG4", "holonomic", True, "weights_ebcadrl.npz", 8192),          # configs[3], one GPU's shard
}


def workload(name="cfg2"):
    from ebc import synth
    from ebc.config import SimConfig
    shape = getattr(synth, WORKLOADS[name][0])
    c = SimConfig()   # reward block of data/eb-cadrl/adults_8_..._fix_static.config:26-44
    c.time_step, c.time_limit = 0.25, 35.0
    c.new_reward, c.time_max, c.time_good, c.max_goal_distance = True, 35.0, 10.0, 10.0
    c.success_reward = 1.0
    c.collision_penalty_adult, c.collision_penalty_bicycle = -1.0, -1.5
    c.collision_penalty_child, c.collision_penalty_obstacle = -2.0, -0.5
    c.discomfort_dist = c.discomfort_dist_adult = 0.1
    c.discomfort_dist_bicycle = c.discomfort_dist_child = 0.2
    c.discomfort_penalty_factor_adult = 0.5
    c.discomfort_penalty_factor_bicycle = c.discomfort_penalty_factor_child = 1.0
    c.map_size_m, c.map_resolution = shape.map_size_m, shape.map_resolution
    c.robot_kinematics, c.with_agent_type, c.gamma = WORKLOADS[name][1], WORKLOADS[name][2], 0.9
    return shape, c


def value_net_weights(D=17, seed=0, fixture="weights_ebcadrl.npz"):
    path = os.path.join(ROOT, "tests", "golden", fixture)
    if os.path.exists(path):
        z = np.load(path)
        return {k: z[k] for k in z.files}, ("rl_model_val fixture" if fixture == "weights_ebcadrl.npz" else fixture)
    rng = np.random.default_rng(seed)
    dims = {"mlp1": [D, 300, 200], "mlp2": [200, 200, 100], "attention": [400, 200, 200, 1],
            "mlp3": [106, 300, 200, 200, 1]}
    sd = {}
    for name, ds in dims.items():
        for i in range(len(ds) - 1):
            b = 1.0 / np.sqrt(ds[i])
            sd["%s.%d.weight" % (name, 2 * i)] = rng.uniform(-b, b, (ds[i + 1], ds[i])).astype(np.float32)
            sd["%s.%d.bias" % (name, 2 * i)] = rng.uniform(-b, b, ds[i + 1]).astype(np.float32)
    return sd, "seeded random init"


def dump_outputs(path, arrays, budget=DUMP_BYTES):
    """Write each [N, ...] array of `arrays` as path/<name>.npy, float32 / float64 kept, integers and flags as float64,
    plus episode_index.npy (the rows written).  Above `budget` bytes in all, every array keeps the same rows: a
    fixed-seed sample of the episodes, so that two runs of the same arguments write the same files."""
    out = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    n = len(next(iter(out.values())))
    room = budget - 256 * (len(out) + 1)                          # .npy headers
    row_bytes = sum(v.nbytes for v in out.values()) // n + 8      # + its episode_index entry
    idx = np.arange(n)
    if n * row_bytes > room:
        idx = np.sort(np.random.default_rng(0).choice(n, room // row_bytes, replace=False))
        out = {k: v[idx] for k, v in out.items()}
    out["episode_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)


def flops_per_eval(sd, n):
    """2 * (n * M_e + M_s) of SURVEY §8d from the actual layer shapes."""
    me = sum(int(np.prod(sd[k].shape)) for k in sd if k.endswith("weight") and not k.startswith("mlp3"))
    ms = sum(int(np.prod(sd[k].shape)) for k in sd if k.endswith("weight") and k.startswith("mlp3"))
    return 2 * (n * me + ms)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / power / throttle reasons every 20 ms; `stop(t0, t1)` keeps the samples whose own timestamp
    lies inside the timed region [t0, t1] (wall clock), so that idle samples before it do not dilute the median."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    @staticmethod
    def _epoch(stamp):
        import datetime
        try:
            return datetime.datetime.strptime(stamp, "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0=None, t1=None):
        if self.proc is not None:
            time.sleep(0.05)
            self.proc.terminate()
            self.join(timeout=2.0)
        rows = [r for r in self.rows if len(r) == 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        if t0 is not None and t1 is not None:
            inside = [r for r in rows if (self._epoch(r[0]) or 0.0) >= t0 and (self._epoch(r[0]) or 0.0) <= t1 + 0.02]
            if inside:
                rows = inside
        sm = sorted(float(r[1]) for r in rows if r[1].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[4 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows), "samples": len(rows),
                "reasons": reasons}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tensor_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tensor_tflops_burst": d.get("bf16_tflops"),
                "source": "MEASURED_PEAKS.json (bf16 sustained, copy bandwidth)"}
    return {"hbm_gbs": 6650.0, "tensor_tflops": 1400.0, "tensor_tflops_burst": None, "source": "fallback (B200_PROFILING.md)"}


def cpu_oracle_rate(shape, cfg, weights, episodes, steps, threads, full_loop=True, kin="holonomic", min_seconds=None):
    """agent-steps/s of the CPU oracle on `episodes` episodes of the same workload; with `min_seconds`, `steps` is the
    upper bound and the loop ends after the first step that passes that much wall time.  Returns (rate, seconds, steps)."""
    import oracle_backend as ob
    from ebc import synth
    from ebc.actions import build_action_space
    from ebc.engine import BatchedSim
    be = ob.OracleBackend()
    be.set_threads(threads)
    sim = BatchedSim(cfg, episodes, shape.H, shape.Smax, shape.Rmax, N_ACTIONS, device="cpu", backend=be)
    sim.set_actions(build_action_space(shape.robot_v_pref, kin))
    sim.set_weights(weights)
    synth.load(sim, synth.generate(shape, np.arange(episodes)))
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        if full_loop:
            sim.decide()
            sim.step(action_idx=sim.argmax)
        else:
            sim.step(action_idx=torch.zeros(episodes, dtype=torch.int32), fused_orca=True)
        done += 1
        if min_seconds is not None and time.perf_counter() - t0 >= min_seconds:
            break
    dt = time.perf_counter() - t0
    return episodes * (shape.H + 1) * done / dt, dt, done


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path.  The reference is pure
    Python + the un-vendored rvo2 and cannot travel to the GPU box, so this is the oracle port
    (oracle/ebc_oracle.c, the restatement pinned against the reference's golden vectors) with all
    host threads, each step a bounded sample of the workload."""
    if rank != 0:
        return
    shape, cfg = workload()
    weights, wsrc = value_net_weights()
    threads = os.cpu_count() or 1
    sample = max(2 * threads, 16)
    steps = max(1, args.steps)
    for _ in range(min(args.warmup, 1)):
        cpu_oracle_rate(shape, cfg, weights, sample, 1, threads)
    rate, dt, _ = cpu_oracle_rate(shape, cfg, weights, sample, steps, threads)
    desc = "%d episodes x %d full steps (decision over 81 actions + env.step) of %s" % (sample, steps, shape.name)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": shape.name, "episodes_per_step": sample, "humans": shape.H, "actions": N_ACTIONS,
                   "weights": wsrc},
        "lookahead_evals_per_sec": rate / (shape.H + 1) * N_ACTIONS,
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_cfg5(args, rank, world, local_rank):
    """BASELINE configs[4]: the EB-CADRL reinforcement-learning loop at N GPUs (one process per GPU).

    One "step" = one training iteration of rl/train.py:212-273 with data/eb-cadrl/train_50k_8x.config semantics:
    k = --episodes-per-iter episodes per GPU (the reference's PROCESSES_NUM = 8) run to their end with epsilon-greedy
    exploration on the shipped 24-human + 3-wall scene (decisions on K1 + K3 + K4 + K5, statistics in the step kernel),
    TD targets from the target network (K4, second handle), replay push, then `train_batches` SGD steps of batch 100
    with ONE NCCL all-reduce of the flat 379,202-float gradient per optimizer step.  Weights start from the shipped
    rl_model_val fixture (the imitation-learning warm-up is not part of the timed loop)."""
    import configparser
    import torch.distributed as dist
    from ebc.batched_env import BatchedEnv
    from rl.policy.policy_factory import policy_factory
    from rl.utils.explorer import Explorer
    from rl.utils.memory import ReplayMemory
    from rl.utils.trainer import Trainer
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    cfgdir = os.path.join(ROOT, "tests", "golden", "configs")

    def ini(name):
        cp = configparser.RawConfigParser()
        assert cp.read(os.path.join(cfgdir, name)), name
        return cp

    ec, pc, tc = ini("env_ebcadrl.config"), ini("policy_ebcadrl.config"), ini("train_50k_8x.config")
    policy = policy_factory["sarl"]()
    policy.configure(pc)
    weights, wsrc = value_net_weights(fixture="weights_ebcadrl.npz")
    policy.get_model().load_state_dict({k: torch.as_tensor(v) for k, v in weights.items()})
    policy.set_device(dev)
    policy.set_phase("train")
    model = policy.get_model().to(dev)
    k = args.episodes_per_iter
    batch_size = tc.getint("trainer", "batch_size")
    train_batches = args.train_batches or tc.getint("train", "train_batches")
    env = BatchedEnv(ec, policy, k, dev)
    memory = ReplayMemory(tc.getint("train", "capacity"), device=dev)
    trainer = Trainer(model, memory, dev, batch_size, policy=policy)
    trainer.set_optimizer(tc.getfloat("train", "rl_learning_rate"), tc.get("train", "optimizer_algorithm", fallback="sgd"))
    explorer = Explorer(env, None, dev, memory, policy.gamma, target_policy=policy)
    explorer.update_target_model(model)
    env.seed_exploration(20261018, rank)
    epsilon = tc.getfloat("train", "epsilon_start")
    policy.set_epsilon(epsilon)
    episode = [0]
    acc = {"explore_s": 0.0, "sgd_s": 0.0, "steps": 0, "decisions": 0}

    def iteration(timed):
        seeds = [episode[0] + rank * k + i for i in range(k)]     # scene_number = episode (parallel_explorer.py:43-52)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stats, traj = env.run_episodes("train", seeds, epsilon=epsilon, record=True)
        explorer.update_memory(traj, stats, False, True)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        trainer.optimize_batch(train_batches)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        episode[0] += k * world
        if timed:
            acc["explore_s"] += t1 - t0
            acc["sgd_s"] += t2 - t1
            acc["steps"] += int(stats.steps.sum())
            acc["decisions"] += int(stats.steps.sum())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 1)):
        iteration(False)
    if args.profile and rank == 0:      # where the host time of one iteration goes (cProfile, top of the cumulative list)
        import cProfile
        import pstats
        pr = cProfile.Profile()
        pr.enable()
        iteration(False)
        pr.disable()
        pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(45)
    launches0 = env.sim.launch_count()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    wall0 = time.time()
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin.record()
    for _ in range(args.steps):
        iteration(True)
    t_end.record()
    barrier()
    wall1 = time.time()
    elapsed_ms = t_begin.elapsed_time(t_end)
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    launches = env.sim.launch_count() - launches0
    # the collective alone: the flat gradient bucket, 200 all-reduces, CUDA events
    n_params = sum(p.numel() for p in model.parameters())
    ar_us = None
    if world > 1:
        flat = torch.zeros(n_params + 1, device=dev)
        for _ in range(20):
            dist.all_reduce(flat)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for _ in range(200):
            dist.all_reduce(flat)
        b.record()
        torch.cuda.synchronize()
        ar_us = a.elapsed_time(b) / 200 * 1e3
    t = torch.tensor([elapsed_ms, acc["explore_s"], acc["sgd_s"], ar_us or 0.0], dtype=torch.float64, device=dev)
    cnt = torch.tensor([acc["steps"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    if rank == 0:
        sec = float(t[0]) / 1e3
        H = env.sim.Hmax
        line = {
            "metric": "training_episodes_per_sec", "value": args.steps * k * world / sec, "unit": "episodes/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": sec / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg5_rl_training_loop", "env": "env_ebcadrl.config (24 humans, 3 walls, D = 17)",
                       "episodes_per_iter_per_gpu": k, "train_batches": train_batches, "batch_size": batch_size,
                       "global_batch": batch_size * world, "weights": wsrc, "epsilon": epsilon,
                       "parallelism": "dp%d: episodes and replay shards per rank, one flat gradient all-reduce per optimizer step" % world},
            "decisions_per_sec": float(cnt[0]) / sec, "agent_steps_per_sec": float(cnt[0]) * (H + 1) / sec,
            "optimizer_steps_per_sec": args.steps * train_batches / sec,
            "phase_s_per_iteration": {"explore_and_td_targets": float(t[1]) / args.steps, "sgd": float(t[2]) / args.steps},
            "sgd_ms_per_optimizer_step": float(t[2]) / args.steps / train_batches * 1e3,
            "allreduce": {"bytes": (n_params + 1) * 4, "us_per_call": float(t[3]) if world > 1 else None,
                          "calls_per_iteration": train_batches},
            "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--episodes", type=int, default=None, help="episodes per GPU (default: the workload's)")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + ["cfg5"],
                    help="cfg2 = BASELINE configs[1], the bench line; cfg3 / cfg4 are side measurements; cfg5 = the RL "
                         "training loop (configs[4]), its own metric")
    ap.add_argument("--episodes-per-iter", type=int, default=8, help="cfg5: episodes per iteration and GPU (reference: 8)")
    ap.add_argument("--train-batches", type=int, default=None, help="cfg5: SGD steps per iteration (default: the config's 800)")
    ap.add_argument("--profile", action="store_true", help="cfg5: cProfile of one untimed iteration to stderr")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--materialize-input", action="store_true",
                    help="write the value-network input to HBM (K3) and read it back (K4) instead of the fused input path")
    ap.add_argument("--sustained-seconds", type=float, default=2.0,
                    help="length of the extra back-to-back region reported under `sustained` (0 = skip)")
    ap.add_argument("--value-mode", default="tc_fp16x2", choices=["fp32", "tc_fp32", "tc_fp16x2", "tc_bf16"],
                    help="K4 arithmetic; tc_fp16x2 (tcgen05, fp32-accurate operand splitting) is the parity mode")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (at most 64 MB; rank 0's episodes)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload == "cfg5"):
        ap.error("--dump-outputs covers the --impl b200 step workloads (%s)" % ", ".join(sorted(WORKLOADS)))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "cfg5":
        run_cfg5(args, rank, world, local_rank)
        return
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    if args.warmup < 3:
        args.warmup = 3
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist = None

    from ebc.actions import build_action_space
    from ebc.batched_env import BatchedEnv
    shape, cfg = workload(args.workload)
    weights, wsrc = value_net_weights(fixture=WORKLOADS[args.workload][3])
    N = args.episodes or WORKLOADS[args.workload][4]
    # episodes shard trivially: rank r owns global episode ids [r N, (r + 1) N) and, as episodes finish, the ids
    # r N + e + k N W (fresh scenes from the device generator, keyed by the global id): no data-path collective
    env = BatchedEnv.synthetic(cfg, shape, N, dev, build_action_space(shape.robot_v_pref, cfg.robot_kinematics), weights,
                               value_mode=args.value_mode, first_episode_id=rank * N, id_stride=N * world)
    sim = env.sim
    n_rows = shape.H + shape.Smax
    H = shape.H
    fused = sim.fused_input and not args.materialize_input
    jd_pad = (6 + int(np.asarray(weights["mlp2.2.weight"]).shape[0]) + 7) // 8 * 8
    joint_mb = (N * N_ACTIONS + 127) // 128 * 128 * jd_pad * 4 / 1e6

    def one_step(marks=None):
        def mark():
            if marks is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append(e)
        mark(); sim.orca()
        if fused:       # K3 leaves 48 B per (episode, action), K4 builds the rotated rows itself: no N*A*n*D buffer
            mark(); sim.lookahead(build_inputs=False)
            mark(); sim.value(fused=True)
        else:
            mark(); sim.lookahead()
            mark(); sim.value()
        mark(); sim.select()
        mark(); sim.step(action_idx=sim.argmax)
        mark(); env.reset_done()
        mark()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = sim.launch_count()
    marks = []
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.time()
    t_begin.record()
    for _ in range(args.steps):
        one_step(marks)
    t_end.record()
    barrier()
    wall1 = time.time()
    launches = sim.launch_count() - launches0
    elapsed_ms = t_begin.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: getattr(sim, k).cpu().numpy() for k in DUMPED})
    phase_names = ["orca", "lookahead", "value", "select", "step", "reset"]
    phase_ms = dict.fromkeys(phase_names, 0.0)
    for s in range(args.steps):
        m = marks[s * 7:(s + 1) * 7]
        for i, nm in enumerate(phase_names):
            phase_ms[nm] += m[i].elapsed_time(m[i + 1])
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None

    # ---- sustained regime: the same step back to back for >= --sustained-seconds (power cap, settled clocks) ----
    sustained = None
    if args.sustained_seconds > 0:
        est = max(elapsed_ms / 1e3 / args.steps, 1e-4)
        s_steps = int(min(max(args.sustained_seconds / est, args.steps), 20000)) + 1
        s_sampler = ClockSampler(local_rank)
        if rank == 0:
            s_sampler.start()
            time.sleep(0.2)
        s_marks = []
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sw0 = time.time()
        s0.record()
        for i in range(s_steps):
            one_step(s_marks if i % 8 == 0 else None)      # K4 phase events on every 8th step
        s1.record()
        barrier()
        sw1 = time.time()
        s_ms = s0.elapsed_time(s1)
        k4 = [s_marks[j * 7 + 2].elapsed_time(s_marks[j * 7 + 3]) for j in range(len(s_marks) // 7)]
        sustained = {"steps": s_steps, "ms_total": s_ms, "k4_ms": float(np.median(k4)),
                     "clocks": s_sampler.stop(sw0, sw1) if rank == 0 else None}

    # ---- side measurement: K4 in the other tensor-core mode on the same states + argmax agreement ------
    other = "tc_bf16" if args.value_mode != "tc_bf16" else "tc_fp16x2"
    sim.orca(); sim.lookahead(); sim.value(); sim.select()
    ref_arg = sim.argmax.clone()
    sim.set_value_mode(other)
    sim.value()
    o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    o0.record()
    for _ in range(5):
        sim.value()
    o1.record()
    sim.select()
    torch.cuda.synchronize()
    other_ms = o0.elapsed_time(o1) / 5
    other_agree = float((sim.argmax == ref_arg).float().mean().item())
    sim.set_value_mode(args.value_mode)

    # ---- e2e: the same step through the host-facing API (pinned host buffers) ------------
    h_pv = torch.empty_like(sim.hum_pv, device="cpu").pin_memory()
    h_rob = torch.empty_like(sim.rob_pv, device="cpu").pin_memory()
    h_out = {k: torch.empty_like(getattr(sim, k), device="cpu").pin_memory()
             for k in ("reward", "done", "event", "argmax")}
    h_pv.copy_(sim.hum_pv); h_rob.copy_(sim.rob_pv)
    torch.cuda.synchronize()
    h2d = h_pv.numel() * 4 + h_rob.numel() * 4
    d2h = 2 * h2d + sum(t.numel() * t.element_size() for t in h_out.values())

    def e2e_step():
        """One step through the batched API a user calls (BatchedEnv.decide_batch / step_batch / reset_done), the
        caller's observation arriving in pinned HOST buffers and the result going back to them, every step."""
        sim.hum_pv.copy_(h_pv, non_blocking=True)       # the caller's observation / robot state -> device
        sim.rob_pv.copy_(h_rob, non_blocking=True)
        idx = env.decide_batch()
        env.step_batch(action_idx=idx)
        h_pv.copy_(sim.hum_pv, non_blocking=True)       # new observation, reward, done, info -> host
        h_rob.copy_(sim.rob_pv, non_blocking=True)
        for k, t in h_out.items():
            t.copy_(getattr(sim, k), non_blocking=True)
        torch.cuda.synchronize()                        # the host consumes the result every step
        env.reset_done()
        h_pv.copy_(sim.hum_pv, non_blocking=True)       # (the re-generated episodes' first observation)
        h_rob.copy_(sim.rob_pv, non_blocking=True)
        torch.cuda.synchronize()

    e2e_steps = max(3, min(args.steps, 10))
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- sim-only path: ORCA + committed step in one launch, L2 flushed between iterations ----
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    zero_idx = torch.zeros(N, dtype=torch.int32, device=dev)
    sim_ms, sim_iters = 0.0, 30
    for it in range(sim_iters + 3):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sim.step(action_idx=zero_idx, fused_orca=True)
        b.record()
        torch.cuda.synchronize()
        if it >= 3:
            sim_ms += a.elapsed_time(b)
        env.reset_done()
    del flush

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    elapsed_ms = allmax(elapsed_ms)
    e2e_s = allmax(e2e_s)
    sim_ms = allmax(sim_ms)
    value_ms = allmax(phase_ms["value"])
    if sustained is not None:
        sustained["ms_total"] = allmax(sustained["ms_total"])
        sustained["k4_ms"] = allmax(sustained["k4_ms"])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    total_eps = N * world
    step_s = elapsed_ms / 1e3 / args.steps
    peaks = measured_peaks()
    fl = flops_per_eval(weights, n_rows) * N * N_ACTIONS            # per GPU per value phase
    achieved_tf = fl / (value_ms / 1e3 / args.steps) / 1e12
    sim_step_s = sim_ms / 1e3 / sim_iters
    sim_bytes = N * (48 * H + 90)
    sim_flops = N * H * 1000.0               # SURVEY 8d: ~1.0 kFLOP per human-step (ORCA LP at 9 neighbours)
    fp32_peak = 148 * 128 * 2 * 1.965e9      # SURVEY 8d: 148 SMs x 128 lanes x 2 x 1.965 GHz = 74 TFLOP/s
    if sustained is not None:
        s_step = sustained["ms_total"] / 1e3 / sustained["steps"]
        sustained = {"seconds": sustained["ms_total"] / 1e3, "steps": sustained["steps"], "ms_per_step": s_step * 1e3,
                     "value": total_eps * (H + 1) / s_step, "unit": UNIT,
                     "lookahead_evals_per_sec": total_eps * N_ACTIONS / s_step,
                     "k4_ms": sustained["k4_ms"], "k4_tflops": fl / (sustained["k4_ms"] / 1e3) / 1e12,
                     "k4_frac_of_peak": fl / (sustained["k4_ms"] / 1e3) / 1e12 / peaks["tensor_tflops"],
                     "clocks": sustained["clocks"],
                     "note": "back-to-back steps for >= %.1f s: the board reaches its power cap and the SM clock settles "
                             "below the maximum; the headline value above is the driver's --steps region" % args.sustained_seconds}
    line = {
        "metric": METRIC, "value": total_eps * (H + 1) / step_s, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": shape.name, "episodes_per_gpu": N, "humans": H, "static_discs": shape.Smax,
                   "what_is_measured": "value = POLICY-IN-THE-LOOP agent-steps/s: every step is a full decision (ORCA, "
                                       "81-action lookahead, value network, argmax) + the committed env.step + fresh scenes "
                                       "for finished episodes (device generator); sim_only = SURVEY 8d(i), the committed-step "
                                       "path alone, which is what north_star's 1e8 agent-steps/s is stated on",
                   "rows_per_state": n_rows, "D": cfg.D, "actions": N_ACTIONS, "weights": wsrc,
                   "parallelism": "episodes sharded over %d GPU(s), no data-path collective" % world,
                   "input_path": ("fused: K3 leaves 48 B per (episode, action), K4's crew builds the rotated joint-state rows "
                                  "from the state; the %.0f MB N*A*n*D input is never written" % (N * N_ACTIONS * n_rows * cfg.D * 4 / 1e6))
                   if fused else "materialised: K3 writes N*A*n*D floats, K4 reads them",
                   "l2": "per-step working set %.0f MB (%s) exceeds the 126 MB L2; sim_only flushes L2 between iterations" % (
                       (joint_mb + 48e-6 * N * N_ACTIONS) if fused else N * N_ACTIONS * n_rows * cfg.D * 4 / 1e6 + joint_mb,
                       "pooled per-state features written by the entity kernel and read by mlp3, + the lookahead records" if fused
                       else "value-net input + pooled features")},
        "lookahead_evals_per_sec": total_eps * N_ACTIONS / step_s,
        "phase_ms_per_step": {k: v / args.steps for k, v in phase_ms.items()},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"kernel": {"fp32": "K4 value network: value_entity_kernel + value_mlp3_kernel (fp32 FFMA)",
                                "tc_fp32": "K4 value network: tc_entity_kernel<3> + tc_mlp3_kernel<3> (tcgen05, bf16x3 "
                                           "operand splitting = 6 MMAs per product, fp32-accurate)",
                                "tc_fp16x2": "K4 value network: tc_entity_kernel<2> + tc_mlp3_kernel<2> (tcgen05, fp16x2 "
                                             "operand splitting = 3 MMAs per product, fp32-accurate)",
                                "tc_bf16": "K4 value network: tc_entity_kernel<1> + tc_mlp3_kernel<1> (tcgen05, bf16 operands)"
                                }[args.value_mode],
                     "bound": "tensor", "achieved": achieved_tf, "peak": peaks["tensor_tflops"], "unit": "TFLOP/s",
                     "frac": achieved_tf / peaks["tensor_tflops"], "traffic": (ROOFLINE_TRAFFIC_FUSED if fused else ROOFLINE_TRAFFIC).get(args.value_mode) if args.workload == "cfg2" and N == 4096 else None,
                     "peak_source": peaks["source"],
                     # the driver's --steps region lasts ~0.15 s (boost clocks): the same achieved figure against the
                     # measured BURST peak; the sustained-against-sustained pair is sustained.k4_frac_of_peak
                     "burst_peak": peaks["tensor_tflops_burst"],
                     "frac_of_burst_peak": achieved_tf / peaks["tensor_tflops_burst"] if peaks["tensor_tflops_burst"] else None,
                     "mma_issue_factor": {"fp32": 0, "tc_fp32": 6, "tc_fp16x2": 3, "tc_bf16": 1}[args.value_mode],
                     "note": "achieved = algorithmic FLOPs 2*(n*M_e+M_s) per (episode, action) / K4 time from CUDA events "
                             "inside the timed region.  The fp32-accurate modes issue mma_issue_factor fp16/bf16 MMAs per "
                             "product, so the tensor pipe executes that multiple of the algorithmic FLOPs: "
                             "tensor-pipe-equivalent fraction ~ frac * mma_issue_factor."},
        "value_mode": args.value_mode,
        "other_value_mode": {"mode": other, "k4_ms": other_ms, "achieved_tflops": fl / (other_ms / 1e3) / 1e12,
                             "argmax_agreement_with_%s" % args.value_mode: other_agree},
        "sim_only": {"agent_steps_per_sec": total_eps * (H + 1) / sim_step_s, "ms_per_step": sim_step_s * 1e3,
                     "launches_per_step": 2,   # K1 (half a warp per human) then K2 (warp per episode), one ebc_orca_step call
                     "roofline": {"bound": "hbm", "achieved": sim_bytes / sim_step_s / 1e9, "peak": peaks["hbm_gbs"],
                                  "unit": "GB/s", "frac": sim_bytes / sim_step_s / 1e9 / peaks["hbm_gbs"],
                                  "alu_achieved_tflops": sim_flops / sim_step_s / 1e12, "alu_peak_tflops": fp32_peak / 1e12,
                                  "alu_frac": sim_flops / sim_step_s / fp32_peak,
                                  "note": "SURVEY 8d asks for both roofs: 48*H+90 algorithmic bytes per episode-step against "
                                          "the measured HBM copy bandwidth, and ~1.0 kFLOP per human-step (ORCA LP) against the "
                                          "74 TFLOP/s FP32 roof; at this size the launch is latency / instruction-issue bound"}},
        "sustained": sustained,
        "e2e": {"value": total_eps * (H + 1) / (e2e_s / e2e_steps), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps},
    }
    if not args.no_cpu_baseline and world == 1:           # rank 0 at N = 1 only
        threads = os.cpu_count() or 1
        sample = max(4 * threads, 32)
        # a bounded sample of the same loop: whole steps until >= 10 s of wall time (<= 64 steps), every host thread busy
        rate, dt, n_cpu = cpu_oracle_rate(shape, cfg, weights, sample, 64, threads, kin=cfg.robot_kinematics, min_seconds=10.0)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "%d episodes x %d full steps (decision over %d actions + env.step) of %s, %.1f s on %d threads"
                                          % (sample, n_cpu, N_ACTIONS, shape.name, dt, threads)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
