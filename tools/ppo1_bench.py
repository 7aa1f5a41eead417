#!/usr/bin/env python
"""Cost of the PPO v1 update (VecPPO.learn: K-RET with statistics, b200_ppo1_grad, b200_adam_step) -> profiles/ppo1/.

    python tools/ppo1_bench.py [--n 262144] [--T 32] [--epochs 8] [--ab-lib path/to/other/libb200env.so]

1. VecPPO.learn() on a collected uav_hover rollout (the K-UAVR env of the PPO v1 demos, reference_nets): CUDA events
   around whole learn() calls; in a separate profiled run, the device time of every kernel, grouped as returns +
   statistics + normalisation, ppo1_advantage_kernel, ppo2_grad_kernel, ppo2_reduce_kernel and adam_kernel.
2. The same v1 epoch in float32 torch autograd (copies of the nets, the same full batch, torch.optim.Adam with two
   parameter groups), timed the same way.
3. With --ab-lib: b200_ppo2_grad of this build against another build of the library (e.g. the parent commit's) at 4096
   and 16,384 samples, alternating the two libraries, five runs each; per run the median of 200 launches.
The card's name, power limit and SM clock limit are recorded with the numbers."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

GROUPS = {"mc_returns_kernel": "returns+stats+norm", "gae_stats_reduce_kernel": "returns+stats+norm",
          "adv_normalize_kernel": "returns+stats+norm", "ppo1_advantage_kernel": "advantage",
          "ppo2_grad_kernel": "grad", "ppo2_reduce_kernel": "reduce", "adam_kernel": "adam"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def timed(fn, reps):
    """CUDA events around each call, after one warm-up call: list of milliseconds"""
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


def kernel_split(fn, calls):
    """device time per kernel group per call, from a torch.profiler run of `calls` calls"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    split, other = {}, 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0:
            continue
        g = next((v for k, v in GROUPS.items() if k in e.key), None)
        if g is None:
            other += t
        else:
            split[g] = split.get(g, 0.0) + t
    res = {k: v / 1000.0 / calls for k, v in split.items()}
    res["other"] = other / 1000.0 / calls
    return res


def learn_bench(n, T, epochs, reps):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo import VecPPO
    from reinforcementlearningplatform_b200.ppo2 import reference_nets
    env = rlp.uav_hover(n_envs=n, io_dtype=torch.float32, auto_reset=True, seed=1)
    torch.manual_seed(0)
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=0.5, mean_act="identity")
    agent = VecPPO(env, actor, critic, {"buffer_size": T, "K_epochs": epochs}, std=0.5, seed=1)
    env.reset(True)
    agent.collect()
    ms = timed(agent.learn, reps)
    split = kernel_split(agent.learn, 3)
    res = {"instances": n, "T": T, "samples": n * T, "epochs": epochs, "learn_ms": ms,
           "learn_ms_median": float(np.median(ms)), "epoch_ms_median": float(np.median(ms)) / epochs,
           "kernel_ms_per_learn": split,
           "kernel_ms_per_epoch": {k: (v / epochs if k in ("advantage", "grad", "reduce", "adam") else v)
                                   for k, v in split.items()}}

    # the same epoch in float32 torch autograd, on copies of the nets
    import copy
    buf = agent.buffer
    B = n * T
    flat = lambda x: x.permute(0, 2, 1).reshape(B, -1)
    s, a, a_lp = flat(buf.s).contiguous(), flat(buf.a).contiguous(), flat(buf.a_lp).sum(1, keepdim=True).contiguous()
    from reinforcementlearningplatform_b200 import gae
    st = torch.zeros(3, dtype=torch.float64, device="cuda")
    ret = gae.mc_returns(buf.r, buf.done, agent.gamma, stats=st)
    ret_hat = gae.normalize_advantage(ret, st, eps=1e-7).reshape(B, 1)
    at, ct = copy.deepcopy(actor), copy.deepcopy(critic)
    for p in list(at.parameters()) + list(ct.parameters()):
        p.data = p.data.clone()
    opt = torch.optim.Adam([{"params": at.parameters(), "lr": 1e-4}, {"params": ct.parameters(), "lr": 1e-3}], eps=1e-8)
    sd = torch.full((env.action_dim,), 0.5, device="cuda")

    def torch_epoch():
        v = ct(s)
        adv = (ret_hat - v).detach()
        mean = at(s)
        lp = (-((a - mean) ** 2) / (2 * sd * sd) - torch.log(sd) - math.log(math.sqrt(2 * math.pi))).sum(1, keepdim=True)
        ratio = torch.exp(lp - a_lp)
        surr = torch.min(ratio * adv, torch.clamp(ratio, 0.8, 1.2) * adv)
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(sd)).sum()
        loss = (-surr).mean() + 0.5 * ((v - ret_hat) ** 2).mean() - 0.01 * ent
        opt.zero_grad()
        loss.backward()
        opt.step()

    tms = timed(torch_epoch, reps)
    res["torch_autograd_epoch_ms"] = tms
    res["torch_autograd_epoch_ms_median"] = float(np.median(tms))
    res["speedup_per_epoch"] = res["torch_autograd_epoch_ms_median"] / res["epoch_ms_median"]
    return res


def ab_bench(other_path, runs=5, launches=200):
    """b200_ppo2_grad of this library (A) against `other_path` (B), the reference 6-64-64-32-8 / 6-64-32-1 nets,
    mini-batches of 4096 and 16,384 samples drawn by the keyed permutation of a 64 x 4096 rollout"""
    from reinforcementlearningplatform_b200 import _lib
    from reinforcementlearningplatform_b200.learn import FusedPPO2Update
    from reinforcementlearningplatform_b200.ppo2 import reference_nets
    libs = {"this": _lib.load(), "other": C.CDLL(os.path.abspath(other_path))}
    vp, f32, sz = C.c_void_p, C.c_float, C.c_size_t
    libs["other"].b200_ppo2_grad.restype = C.c_int
    libs["other"].b200_ppo2_grad.argtypes = [vp, vp, vp, f32, vp, vp, vp, f32, f32, vp, vp, vp, vp, sz, vp]
    torch.manual_seed(0)
    T, S, A, N = 64, 6, 8, 4096
    actor, critic = reference_nets(S, A, "cuda", init_std=0.45)
    upd = FusedPPO2Update(actor, critic, 0.45, np.zeros(A), np.full(A, 5.0), "relu")
    g = torch.Generator(device="cuda").manual_seed(1)
    s = torch.rand(T, S, N, device="cuda", generator=g).contiguous()
    a = (5 * torch.rand(T, A, N, device="cuda", generator=g)).contiguous()
    a_lp = (-1.5 - 0.5 * torch.rand(T, A, N, device="cuda", generator=g)).contiguous()
    adv = torch.randn(T, N, device="cuda", generator=g).contiguous()
    vt = torch.randn(T, N, device="cuda", generator=g).contiguous()
    am, cm = upd.params.mlp(0, upd.out_act), upd.params.mlp(1, 0)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    o = upd.params.net_off[1]
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {}
    for count in (4096, 16384):
        b = upd._batch(s, a, a_lp, adv, vt, 0, count, perm_key=5)
        grads = {}

        def call(lib):
            return lib.b200_ppo2_grad(C.byref(b), C.byref(am), C.byref(cm), upd.std, None, p(upd.a_min), p(upd.a_max),
                                      upd.eps_clip, upd.entropy_coef, p(upd.grad), C.c_void_p(upd.grad.data_ptr() + 4 * o),
                                      p(upd.loss), p(upd.workspace), upd.workspace.numel(), stream)

        for name, lib in libs.items():
            assert call(lib) == 0
            torch.cuda.synchronize()
            grads[name] = (upd.grad.clone(), upd.loss.clone())
        same = torch.equal(grads["this"][0], grads["other"][0]) and torch.equal(grads["this"][1], grads["other"][1])
        runs_us = {k: [] for k in libs}
        for r in range(runs):
            for name in (("this", "other") if r % 2 == 0 else ("other", "this")):
                lib = libs[name]
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(launches + 1)]
                for _ in range(20):
                    call(lib)
                ev[0].record()
                for i in range(launches):
                    call(lib)
                    ev[i + 1].record()
                ev[-1].synchronize()
                per = [ev[i].elapsed_time(ev[i + 1]) * 1000.0 for i in range(launches)]
                runs_us[name].append(float(np.median(per)))
        out[str(count)] = {"bit_identical": bool(same), "us_per_launch": runs_us,
                           "median_us": {k: float(np.median(v)) for k, v in runs_us.items()},
                           "spread_us": {k: float(max(v) - min(v)) for k, v in runs_us.items()}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=262144)
    ap.add_argument("--T", type=int, default=32)
    ap.add_argument("--epochs", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--ab-lib", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ppo1", "ppo1_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ppo1_bench needs a CUDA device"
    res = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    res["learn"] = learn_bench(args.n, args.T, args.epochs, args.reps)
    if args.ab_lib:
        res["ab_ppo2_grad"] = ab_bench(args.ab_lib)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
