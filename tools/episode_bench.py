"""K-EPISODE cost, measured in one process on one GPU:

1. the episode scan (b200_episode_scan with statistics, i.e. the scan kernel and the one-block reduction) against K-RET
   (b200_mc_returns) on the same [64, 2^20] float32 reward / u8 done arrays (plus the i32 flag column for the scan),
   alternating the two, median over blocks of launches timed with CUDA events.  The arrays (604 MB) exceed the L2;
2. VecPPO2.collect() on UavPosCtrlRL with 2^20 instances and T = 16, with episode tracking on and off, alternated.

Prints the card's name, power limit and maximum SM clock (nvidia-smi, a read-only query) and one JSON object.
    python tools/episode_bench.py [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def time_blocks(fns, blocks, reps):
    """alternate the callables block by block; per-call milliseconds, median over blocks"""
    ev = lambda: torch.cuda.Event(enable_timing=True)
    out = {k: [] for k in fns}
    for _ in range(blocks):
        for k, fn in fns.items():
            a, b = ev(), ev()
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            b.synchronize()
            out[k].append(a.elapsed_time(b) / reps)
    return {k: statistics.median(v) for k, v in out.items()}, out


def scan_vs_ret(T=64, N=1 << 20, blocks=9, reps=50):
    from reinforcementlearningplatform_b200 import EpisodeTracker, _lib
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(1)
    r = torch.randn((T, N), generator=g, device="cuda", dtype=torch.float32)
    dn = torch.rand((T, N), generator=g, device="cuda") < 0.01
    done = dn.to(torch.uint8)
    flag = torch.randint(0, 4, (T, N), generator=g, device="cuda", dtype=torch.int32)
    ret = torch.empty((T, N), dtype=torch.float32, device="cuda")
    tr = EpisodeTracker(N, "cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    scr = tr._scratch
    episode = lambda: lib.b200_episode_scan(_lib.F32, T, N, p(r), p(done), p(flag), p(tr.acc_return), p(tr.acc_length),
                                            p(tr.ep_return), p(tr.ep_length), p(tr.ep_flag), 0, p(tr.stats), p(scr),
                                            scr.numel() * 8, stream)
    mc = lambda: lib.b200_mc_returns(_lib.F32, T, N, p(r), p(done), 0.99, p(ret), stream)
    assert episode() == 0 and mc() == 0
    torch.cuda.synchronize()
    med, raw = time_blocks({"episode_scan": episode, "mc_returns": mc}, blocks, reps)
    by_ep = T * N * 9 + N * 2 * (8 + 4)           # r f32 + done u8 + flag i32; carry read and written
    by_mc = T * N * 9                              # r f32 + done u8 read, f32 return written
    return {"shape": [T, N], "reps_per_block": reps, "blocks": blocks,
            "episode_scan_ms": med["episode_scan"], "mc_returns_ms": med["mc_returns"],
            "ratio_episode_over_mc_returns": med["episode_scan"] / med["mc_returns"],
            "episode_scan_GBps": by_ep / med["episode_scan"] / 1e6, "mc_returns_GBps": by_mc / med["mc_returns"] / 1e6,
            "episode_scan_ms_blocks": raw["episode_scan"], "mc_returns_ms_blocks": raw["mc_returns"]}


def collect_overhead(N=1 << 20, T=16, rounds=9, warmup=2):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    agents = {}
    for track in (False, True):
        env = rlp.UavPosCtrlRL(n_envs=N, random_trajectory=True, io_dtype=torch.float32, auto_reset=True, seed=5)
        torch.manual_seed(0)
        actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=0.45)
        agents[track] = VecPPO2(env, actor, critic, {"buffer_size": T}, std=0.45, seed=1, track_episodes=track)
        env.reset(True)
    for _ in range(warmup):
        for a in agents.values():
            a.collect()
    torch.cuda.synchronize()
    med, raw = time_blocks({"off": agents[False].collect, "on": agents[True].collect}, rounds, 1)
    s = agents[True].episodes.summary()
    return {"env": "UavPosCtrlRL", "n_envs": N, "T": T, "rounds": rounds, "collect_ms_off": med["off"],
            "collect_ms_on": med["on"], "overhead_pct": 100.0 * (med["on"] / med["off"] - 1.0),
            "collect_ms_off_rounds": raw["off"], "collect_ms_on_rounds": raw["on"],
            "episodes_tracked": s["episodes"]}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args(argv)
    assert torch.cuda.is_available(), "episode_bench.py measures on a CUDA device"
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "scan": scan_vs_ret(),
           "collect": collect_overhead()}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
