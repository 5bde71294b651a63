"""rl/train.py — imitation-learning warm-up + RL (rl/train.py:22-42,99-276 of the reference), same flags,
same artefacts (`output.log`, `il_model.pth`, `rl_model_{episode}.pth`, configs copied into --output_dir).

    python -m rl.train --env_config E --policy sarl --policy_config P --train_config T --output_dir OUT [--gpu]
    python -m torch.distributed.run --nproc-per-node N -m rl.train ...        # one process per GPU

What changed versus the reference: the 8-process pool (rl/utils/parallel_explorer.py) is a batch of
`--episodes_per_iter` episodes per GPU on the device; with W ranks every rank samples its own seeds, the
value-network gradient is all-reduced over NCCL once per optimizer step and the evaluation counters are
all-gathered.  Replay memory, optimizer state and epsilon are not checkpointed (like the reference).

Walls-aware humans come from the env INI, not a flag: with `[sim] orca_obstacles = true` (this project's key, off by
default like the reference) humans avoid the scene's walls, and so does the ORCA robot that imitation learning
follows (ebc_robot_orca).  rl.test and rl.test_parallel read the same key from the env INI they are given."""
import argparse
import configparser
import copy
import logging
import os
import shutil
import sys

import torch

VAL_EPISODE_START = 100000


def parse_arguments(argv=None):
    p = argparse.ArgumentParser("Parse configuration file")
    p.add_argument("--env_config", type=str, default="configs/env_configs/env.config")
    p.add_argument("--policy", type=str, default="sarl")
    p.add_argument("--policy_config", type=str, default="configs/policy_configs/policy.config")
    p.add_argument("--train_config", type=str, default="configs/train_configs/train.config")
    p.add_argument("--output_dir", type=str, default="data/output")
    p.add_argument("--weights", type=str)
    p.add_argument("--resume", default=False, action="store_true")
    p.add_argument("--resume_iteration", type=int, default=0)
    p.add_argument("--end_iteration", type=int, default=1000000)
    p.add_argument("--gpu", default=False, action="store_true")
    p.add_argument("--debug", default=False, action="store_true")
    p.add_argument("--episodes_per_iter", type=int, default=8, help="episodes sampled per RL iteration and per GPU "
                   "(the reference's PROCESSES_NUM = 8)")
    return p.parse_args(argv)


def _dist():
    import torch.distributed as dist
    if "RANK" in os.environ and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        dist.init_process_group(backend)
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def prepare_output_dir(args, rank):
    """Copy the three configs into output_dir (train.py:45-80); on resume re-read them from there."""
    names = {"env_config": "env.config", "policy_config": "policy.config", "train_config": "train.config"}
    if rank == 0:
        os.makedirs(args.output_dir, exist_ok=True)
        if not args.resume:
            for attr, name in names.items():
                shutil.copy(getattr(args, attr), os.path.join(args.output_dir, name))
    for attr, name in names.items():
        dst = os.path.join(args.output_dir, name)
        if args.resume or rank == 0:
            setattr(args, attr, dst if os.path.exists(dst) else getattr(args, attr))


def run_train(args):
    from rl.utils.explorer import Explorer
    from rl.utils.memory import ReplayMemory
    from rl.utils.trainer import Trainer
    from rl.utils.utils import configure_environment_and_robot, configure_policy
    rank, world = _dist()
    prepare_output_dir(args, rank)
    handlers = [logging.StreamHandler(sys.stdout)]
    if rank == 0:
        handlers.append(logging.FileHandler(os.path.join(args.output_dir, "output.log"), mode="a" if args.resume else "w"))
    logging.basicConfig(level=logging.DEBUG if args.debug else logging.INFO, handlers=handlers,
                        format="%(asctime)s, %(levelname)s: %(message)s", datefmt="%Y-%m-%d %H:%M:%S", force=True)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    logging.info("Using device: %s (rank %d of %d)", device, rank, world)

    policy = configure_policy(args)
    policy.set_device(device)
    tc = configparser.RawConfigParser()
    tc.read(args.train_config)
    rl_lr = tc.getfloat("train", "rl_learning_rate")
    train_batches = tc.getint("train", "train_batches")
    train_episodes = tc.getint("train", "train_episodes")
    target_update_interval = tc.getint("train", "target_update_interval")
    evaluation_interval = tc.getint("train", "evaluation_interval")
    capacity = tc.getint("train", "capacity")
    eps_start, eps_end = tc.getfloat("train", "epsilon_start"), tc.getfloat("train", "epsilon_end")
    eps_decay = tc.getfloat("train", "epsilon_decay")
    checkpoint_interval = tc.getint("train", "checkpoint_interval")
    algo = tc.get("train", "optimizer_algorithm", fallback="sgd")
    batch_size = tc.getint("trainer", "batch_size")

    k = args.episodes_per_iter
    env = configure_environment_and_robot(args.env_config, policy, k, device)
    val_size = env.scene.case_size["val"]
    model = policy.get_model()
    memory = ReplayMemory(capacity, device=device)
    trainer = Trainer(model, memory, device, batch_size, policy=policy)
    explorer = Explorer(env, None, device, memory, policy.gamma, target_policy=policy)
    il_path = os.path.join(args.output_dir, "il_model.pth")
    episode = 0
    if args.resume:
        path = os.path.join(args.output_dir, "rl_model_%d.pth" % args.resume_iteration)
        if not os.path.exists(path):
            raise FileNotFoundError("RL weights does not exist: %s" % path)
        model.load_state_dict(torch.load(path, map_location=device))
        policy.weights_version += 1
        episode = args.resume_iteration
        logging.info("Load reinforcement learning trained weights. Resume training from %d", episode)
    elif os.path.exists(il_path) and args.weights is None:
        model.load_state_dict(torch.load(il_path, map_location=device))
        policy.weights_version += 1
        logging.info("Load imitation learning trained weights.")
    else:
        # ---- imitation learning (train.py:99-143): ORCA robot, discounted returns, supervised epochs ----
        il_episodes = tc.getint("imitation_learning", "il_episodes")
        il_epochs = tc.getint("imitation_learning", "il_epochs")
        il_lr = tc.getfloat("imitation_learning", "il_learning_rate")
        trainer.set_optimizer(il_lr, algo)
        safety = 0.0 if env.robot.visible else tc.getfloat("imitation_learning", "safety_space")
        policy.set_phase("train")
        seeds = [env.COUNTER_OFFSET["train"] + rank + world * i for i in range(-(-il_episodes // world))]
        explorer.run_k_episodes(len(seeds), "train", update_memory=True, imitation_learning=True, seeds=seeds,
                                safety_space=safety)
        trainer.optimize_epoch(il_epochs)
        if rank == 0:
            torch.save(model.state_dict(), il_path)
        logging.info("Finish imitation learning. Weights saved.")
        logging.info("Experience set size: %d/%d", len(memory), memory.capacity)
    explorer.update_target_model(model)

    # ---- reinforcement learning (train.py:212-273) ------------------------------------------------------------
    trainer.set_optimizer(rl_lr, algo)
    policy.set_phase("train")
    last_eval = None
    while episode < min(train_episodes, args.end_iteration):
        if episode < eps_decay:
            epsilon = eps_start + (eps_end - eps_start) / eps_decay * episode
        else:
            epsilon = eps_end
        policy.set_epsilon(epsilon)
        if evaluation_interval and episode % evaluation_interval < k * world and last_eval != episode // evaluation_interval:
            last_eval = episode // evaluation_interval
            policy.set_phase("val")
            vs = [VAL_EPISODE_START + rank + world * i for i in range(-(-val_size // world))]
            explorer.run_k_episodes(len(vs), "val", episode=episode, seeds=vs)
            policy.set_phase("train")
        # scene_number = episode, no phase offset (parallel_explorer.py:43-52 -> scene_generator.py:356-360)
        seeds = [episode + rank * k + i for i in range(k)]
        explorer.run_k_episodes(k, "train", update_memory=True, episode=episode, seeds=seeds, epsilon=epsilon,
                                store_all=True)
        trainer.optimize_batch(train_batches)
        episode += k * world
        if episode % target_update_interval < k * world:
            explorer.update_target_model(model)
        if checkpoint_interval and episode % checkpoint_interval < k * world and rank == 0:
            torch.save(model.state_dict(), os.path.join(args.output_dir, "rl_model_%d.pth" % episode))
    if rank == 0:
        torch.save(model.state_dict(), os.path.join(args.output_dir, "rl_model_%d.pth" % episode))
    return episode


def main(argv=None):
    try:
        run_train(parse_arguments(argv))
    finally:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
