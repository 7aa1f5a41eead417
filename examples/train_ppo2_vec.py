#!/usr/bin/env python
"""PPO2 on a vector env, entirely on the device: the vector form of
demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py (collection loop :186-216, learn :219-222) and of
PPO2-4-UavFntsmcParamPos/train.py.  Under torchrun every rank owns a shard of the instances and gradients are
all-reduced (DPPO2 as synchronous data parallelism).  ``--algo ppo`` trains with the PPO v1 learner instead (VecPPO:
normalised Monte-Carlo returns, full-batch epochs of the joint loss), the learner of the PPO v1 demos such as
PPO-4-UavHoverOuterLoop (``--env uav_hover``).  ``--algo dqn`` trains DQN (``--double``: Double DQN) on the discrete
FlightAttitudeSimulatorDiscrete (``--env fas_discrete``) with VecDQN: epsilon-greedy collection into a device replay
ring, keyed mini-batches, one GPU.

    python examples/train_ppo2_vec.py --env cartpole_angleonly --envs 4096 --iters 30
    python examples/train_ppo2_vec.py --algo ppo --env uav_hover --envs 65536 --steps 32 --iters 20
    python examples/train_ppo2_vec.py --algo dqn --env fas_discrete --envs 4096 --iters 300 --collect 2 --updates 8 --eval-envs 4096
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 examples/train_ppo2_vec.py --env soi
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import reinforcementlearningplatform_b200 as rlp  # noqa: E402
from reinforcementlearningplatform_b200 import dist as D  # noqa: E402
from reinforcementlearningplatform_b200.dqn import VecDQN, q_net  # noqa: E402
from reinforcementlearningplatform_b200.ppo import VecPPO  # noqa: E402
from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets  # noqa: E402

ENVS = {
    "cartpole_angleonly": (lambda **kw: rlp.CartPoleAngleOnly(variant="ppo2", **kw), dict(std=1.2, mean_act="identity")),
    "soi": (lambda **kw: rlp.SecondOrderIntegration(**kw), dict(std=0.8, mean_act="identity")),
    "fas": (lambda **kw: rlp.Flight_Attitude_Simulator(variant="ppo2", **kw), dict(std=0.8, mean_act="identity")),
    "uav_pos": (lambda **kw: rlp.UavPosCtrlRL(random_trajectory=True, **kw), dict(std=0.45, mean_act="relu")),
    # BASELINE config #5: the DPPO2 copy of UGVForwardObstacleAvoidance (41-dim observation with the 37-ray laser);
    # under torchrun this is DPPO2 as synchronous data parallelism (flat gradient all-reduce per mini-batch)
    "ugvo": (lambda **kw: rlp.UGVForwardObstacleAvoidance(variant="dppo2", **kw), dict(std=0.8, mean_act="identity")),
    # K-UAVR's UavHover (12 observations, 3 accelerations + 3 torques), the env of the PPO v1 UavRobust demos
    "uav_hover": (lambda **kw: rlp.uav_hover(**kw), dict(std=0.5, mean_act="identity")),
    # K-FASD, the discrete-action env of the DQN-family demos (--algo dqn only)
    "fas_discrete": (lambda **kw: rlp.FlightAttitudeSimulatorDiscrete(**kw), None),
}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", default="cartpole_angleonly", choices=sorted(ENVS))
    ap.add_argument("--algo", default="ppo2", choices=("ppo2", "ppo", "dqn"),
                    help="ppo2: VecPPO2 (GAE, mini-batches, gradient clip); ppo: VecPPO (the v1 learner); dqn: VecDQN")
    ap.add_argument("--envs", type=int, default=4096, help="instances in total (sharded over ranks)")
    ap.add_argument("--steps", type=int, default=64, help="time steps per rollout (buffer_size)")
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--epochs", type=int, default=8)
    ap.add_argument("--seed", type=int, default=3407)   # the reference script's seed (train.py:36)
    ap.add_argument("--eval-envs", type=int, default=0,
                    help="after the last iteration, run the deterministic policy for one episode on this many instances "
                         "in total (sharded over ranks)")
    ap.add_argument("--double", action="store_true", help="dqn: Double DQN targets")
    ap.add_argument("--memory", type=int, default=64, help="dqn: replay ring rows (memory_capacity)")
    ap.add_argument("--batch", type=int, default=4096, help="dqn: samples per update")
    ap.add_argument("--collect", type=int, default=4, help="dqn: collection steps per iteration")
    ap.add_argument("--updates", type=int, default=4, help="dqn: updates per iteration")
    ap.add_argument("--epsilon", type=float, default=0.1, help="dqn: exploration probability")
    args = ap.parse_args(argv)
    if (args.algo == "dqn") != (ENVS[args.env][1] is None):
        ap.error("--algo dqn trains the discrete-action env fas_discrete, the PPO learners the continuous ones")
    rank, world, local = D.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    torch.manual_seed(args.seed)
    n_local, off = D.shard(args.envs, rank, world)
    make, net_kw = ENVS[args.env]
    if args.algo == "dqn":
        return _train_dqn(args, world, dev, make)
    env = make(n_envs=n_local, device=dev, dtype=torch.float64, io_dtype=torch.float32, auto_reset=True, seed=args.seed,
               env_index_offset=off)
    actor, critic = reference_nets(env.state_dim, env.action_dim, dev, init_std=net_kw["std"], mean_act=net_kw["mean_act"])
    agent = (VecPPO2 if args.algo == "ppo2" else VecPPO)(
        env, actor, critic, {"buffer_size": args.steps, "K_epochs": args.epochs, "mini_batch_size": 16384},
        std=net_kw["std"], seed=args.seed, track_episodes=True)
    env.reset(True)
    log = []
    for it in range(args.iters):
        t0 = time.perf_counter()
        mean_r = agent.collect()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        episodes = agent.episodes.summary()          # the episodes that ended in this rollout, raw rewards
        agent.episodes.reset_stats()
        losses = agent.learn()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        done_rate = float(agent.buffer.done.float().mean())
        timeout_share = float(((agent.buffer.flag == env.TIMEOUT_FLAG) & (agent.buffer.done != 0)).float().sum() /
                              max(1.0, float(agent.buffer.done.sum())))
        row = {"iter": it, "mean_reward": mean_r, "done_rate": done_rate, "timeout_share": timeout_share,
               "collect_env_steps_per_s": args.steps * n_local * world / (t1 - t0), "learn_s": t2 - t1, **losses,
               "episodes": episodes["episodes"], "mean_episode_return": episodes["mean_return"],
               "mean_episode_length": episodes["mean_length"], "flag_counts": episodes["flag_counts"]}
        log.append(row)
        if rank == 0:
            print(json.dumps(row))
    if args.eval_envs > 0:
        n_eval, off_eval = D.shard(args.eval_envs, rank, world)
        eval_env = make(n_envs=n_eval, device=dev, dtype=torch.float64, io_dtype=torch.float32, auto_reset=True,
                        seed=args.seed + 1, env_index_offset=off_eval)
        ev = agent.evaluate_episodes(eval_env, max_steps=100000)
        ev = {k: v for k, v in ev.items() if not torch.is_tensor(v)}
        log.append({"eval": ev})
        if rank == 0:
            print(json.dumps({"eval": ev}))
    if world > 1:
        torch.distributed.destroy_process_group()
    return log


def _train_dqn(args, world, dev, make):
    """Per iteration: --collect epsilon-greedy steps of all instances into the ring, then --updates DQN updates; the log
    row holds the loss and the episodes that ended in the iteration.  --eval-envs: the greedy policy before and after."""
    if world > 1:
        raise SystemExit("--algo dqn runs on one GPU")
    env = make(n_envs=args.envs, device=dev, dtype=torch.float64, io_dtype=torch.float32, auto_reset=True, seed=args.seed)
    agent = VecDQN(env, q_net(env.state_dim, env.action_num[0], dev),
                   {"memory_capacity": args.memory, "batch_size": args.batch, "double_dqn": args.double},
                   epsilon=args.epsilon, seed=args.seed, track_episodes=True)

    def evaluate():
        eval_env = make(n_envs=args.eval_envs, device=dev, dtype=torch.float64, io_dtype=torch.float32, auto_reset=True,
                        seed=args.seed + 1)
        return {k: v for k, v in agent.evaluate_episodes(eval_env, max_steps=100000).items() if not torch.is_tensor(v)}

    log = []
    if args.eval_envs > 0:
        log.append({"eval_untrained": evaluate()})
        print(json.dumps(log[-1]))
    for it in range(args.iters):
        t0 = time.perf_counter()
        agent.collect(args.collect)
        episodes = agent.episodes.summary()
        agent.episodes.reset_stats()
        losses = agent.learn(args.updates) or {"loss": None}
        torch.cuda.synchronize()
        row = {"iter": it, "valid_rows": agent.valid_rows, "s": time.perf_counter() - t0, **losses,
               "episodes": episodes["episodes"], "mean_episode_return": episodes["mean_return"],
               "mean_episode_length": episodes["mean_length"], "flag_counts": episodes["flag_counts"]}
        log.append(row)
        print(json.dumps(row))
    if args.eval_envs > 0:
        log.append({"eval": evaluate()})
        print(json.dumps(log[-1]))
    return log


if __name__ == "__main__":
    main()
