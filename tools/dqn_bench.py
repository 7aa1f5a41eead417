#!/usr/bin/env python
"""Cost of K-DQN (b200_dqn_act, one VecDQN collection step, one VecDQN update) -> profiles/dqn/.

    python tools/dqn_bench.py [--n 1048576] [--out profiles/dqn]

1. b200_dqn_act on 2^20 FlightAttitudeSimulatorDiscrete observations with the 2-64-64-46 Q-net of dqn.q_net, against
   torch eager on the same net (the Linear stack, argmax, torch.rand and the epsilon choice).
2. One collection step of VecDQN (b200_dqn_act + the K-FASD step kernel into the replay ring) at 2^20 instances.
3. One update (target + gradient + reduction + Adam) at mini-batches of 4096 and 16,384, against float32 torch autograd
   of the same statement (gather, target forward, online forward, mse_loss, backward, torch.optim.Adam).
Every figure: CUDA events around blocks of calls after a warm-up, the median of 5 blocks, in ms per call.  The ring's
working set (64 rows x 2^20 instances) is larger than L2 for the updates' gathers; the act kernel's 8 MB of
observations are not (the same input every call, as in a collection loop that reads the row the step just wrote).
The card's name, power limit and SM clock limit are recorded with the numbers."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def median_ms(fn, calls, blocks=5, warmup=3):
    """median over `blocks` of (CUDA-event time of `calls` back-to-back calls) / calls"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(blocks):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(calls):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / calls)
    return float(np.median(out)), [round(x, 5) for x in out]


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--memory", type=int, default=64)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "dqn"))
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("dqn_bench: needs a CUDA device")
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.dqn import q_net
    dev = torch.device("cuda")
    n = args.n
    env = rlp.FlightAttitudeSimulatorDiscrete(n_envs=n, device=dev, dtype=torch.float64, io_dtype=torch.float32,
                                              auto_reset=True, seed=1)
    A = env.action_num[0]
    torch.manual_seed(0)
    net = q_net(env.state_dim, A, dev)
    res = {"device": card(), "n": n, "net": [env.state_dim, 64, 64, A], "unit": "ms per call, median of 5 blocks"}

    # 1. act
    agent = rlp.VecDQN(env, net, {"memory_capacity": args.memory, "batch_size": 4096, "learn_start": 1}, epsilon=0.1)
    obs = (torch.rand(env.state_dim, n, device=dev) - 0.5).contiguous()
    idx = torch.empty(n, dtype=torch.int32, device=dev)
    val = torch.empty(1, n, device=dev)
    step = [0]

    def act():
        agent.act(obs, idx, val, 0.1, step[0])
        step[0] += 1
    res["act_kernel_ms"], res["act_kernel_blocks"] = median_ms(act, 50)
    net_t = copy_net(net)
    obs_t = obs.t().contiguous()

    def act_torch():
        with torch.no_grad():
            greedy = net_t(obs_t).argmax(1)
            explore = torch.rand(n, device=dev) < 0.1
            rnd = torch.randint(0, A, (n,), device=dev)
            i = torch.where(explore, rnd, greedy)
            agent.table[i].view(1, -1)
    res["act_torch_ms"], res["act_torch_blocks"] = median_ms(act_torch, 50)

    # 2. one collection step (act + K-FASD step into the ring)
    agent.collect(args.memory)     # fill the ring once
    res["collect_step_ms"], res["collect_step_blocks"] = median_ms(lambda: agent.collect(1), 50)

    # 3. one update
    for M in (4096, 16384):
        agent.batch_size = M
        agent.workspace = torch.zeros(int(agent._lib.b200_dqn_workspace_bytes(C.byref(agent._q), M)),
                                      dtype=torch.uint8, device=dev)
        u = [0]

        def update():
            agent.grad_step(agent.sample_key(u[0]))
            agent.adam_step()
            u[0] += 1
        res[f"update_{M}_ms"], res[f"update_{M}_blocks"] = median_ms(update, 100)
        tq, tt = copy_net(net), copy_net(net)
        opt = torch.optim.Adam(tq.parameters(), lr=1e-3, eps=1e-8)
        R, N = agent.R, n

        def update_torch():
            pos = torch.randint(0, (R - 1) * N, (M,), device=dev)
            row, i = pos // N, pos % N
            s, s_ = agent.s[row, :, i], agent.s_[row, :, i]
            r, a, done = agent.r[row, i], agent.a[row, i].long(), agent.done[row, i]
            with torch.no_grad():
                y = r + 0.99 * (1 - done.float()) * tt(s_).max(1).values
            loss = torch.nn.functional.mse_loss(tq(s).gather(1, a[:, None])[:, 0], y)
            opt.zero_grad()
            loss.backward()
            opt.step()
        res[f"update_{M}_torch_ms"], res[f"update_{M}_torch_blocks"] = median_ms(update_torch, 100)

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "dqn_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    rows = [("b200_dqn_act, 2^20 instances", "act_kernel_ms", "act_torch_ms"),
            ("collection step (act + K-FASD), 2^20 instances", "collect_step_ms", None),
            ("update (target + grad + reduce + Adam), 4096 samples", "update_4096_ms", "update_4096_torch_ms"),
            ("update, 16,384 samples", "update_16384_ms", "update_16384_torch_ms")]
    lines = ["# K-DQN timings", "",
             f"`python tools/dqn_bench.py` on {res['device']} (name, power limit, SM clock limit as nvidia-smi reports "
             "them).  CUDA events around blocks of back-to-back calls after a warm-up; median of 5 blocks, ms per call.",
             "Net: dqn.q_net(2, 46) = 2-64-64-46, tanh.  The torch column is float32 eager / autograd of the same "
             "statement on the same net (tools/dqn_bench.py).", "",
             "| what | K-DQN (ms) | torch (ms) |", "|---|---|---|"]
    for name, k, t in rows:
        lines.append(f"| {name} | {res[k]:.4f} | {'' if t is None else f'{res[t]:.4f}'} |")
    with open(os.path.join(args.out, "README.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print(json.dumps(res))


def copy_net(net):
    import copy
    c = copy.deepcopy(net)
    for p in c.parameters():
        p.data = p.data.clone()
    return c


if __name__ == "__main__":
    main()
