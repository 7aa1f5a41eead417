#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched environment engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload uav_pos|uav_att|cartpole] [--impl reference]
                    [--dump-outputs DIR]

Default workload = config #4 of BASELINE.json: UavFntsmcParam position tracking (quadrotor RK4 + FNTSMC outer and
inner loops), 1,048,576 instances per GPU, fp64, 8 fresh gains per instance per step, auto-reset on.  One "step" is
one launch of the fused step kernel over all instances of this rank.  Instances shard independently over ranks (weak
scaling, no data-path collective); the timed region is bracketed by barrier + synchronize and the reported time is
the max over ranks.  Exactly K steps are timed, in up to 5 blocks.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned to its caller (current_state,
next_state, policy_state, reward, is_terminal, terminal_flag, time) as DIR/<name>.npy, instances first, float64 or
float32; at most 64 MB in all, so larger batches are cut to a fixed sample of instances (their indices in
DIR/instance_index.npy).  Actions and initial states are seeded: the same arguments give the same inputs on every run,
so the files of two builds can be compared one to one.

The JSON line carries, besides the contract keys: `roofline` (the binding resource of the step kernel -- the FP64 pipe
for the UAV / cart-pole kernels -- with the HBM view beside it; DRAM traffic and executed-instruction counts are parsed at
run time from the committed ncu summaries under profiles/), `repeats` (the blocks the K timed steps ran in: median and
spread of their time per step), `cpu_baseline` (the UNMODIFIED Python reference on every host core, one process per
core, from the byte-compiled staging oracle/_ref, and the C port beside it), `e2e` (same metric through the public
VecEnv API with host buffers: pinned H2D of the actions and D2H of next_state / reward / done every step, plus a raw
cudaMemcpyAsync probe of the same bytes), `clocks`, `gpu_launches`, and `also` (the other configs of BASELINE.json; under torchrun every rank
takes part in the sharded ones -- config #3's rollout + GAE + statistics all-reduce, config #5's DPPO2 iteration).

`--impl reference` times the reference's own Python loop (oracle/_ref, or the tree RLP_REFERENCE names) on all host
cores and never imports the product package.

Nothing is written into the source tree: no bytecode caches either, so the tree may be read-only.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import glob
import re
import subprocess
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

# algorithmic HBM bytes per env-step (fp64), derived in DESIGN.md section 4 from the kernel's loads/stores:
#   uav_pos: state 21 fields R+W (12 ODE, 3 sigma_o1, 3 s1, 3 att_ref) + 12 gains W + 12 trajectory R + 8 action R
#            + time R+W + 6 next_obs + reward W (8 B each) + done (1) + flag (4)
ALGO_BYTES = {
    "uav_pos": (21 * 2 + 12 + 12 + 8 + 2 + 6 + 1) * 8 + 5,
    "uav_att": (9 * 2 + 12 + 9 + 8 + 2 + 6 + 1) * 8 + 5,
    "cartpole": (4 * 2 + 1 + 2 + 4 + 1) * 8 + 5,
    # ugvo: 5 kinematic states R+W, target + n_obs + 16 obstacles R, 2 actions, time R+W, obs 41 + next_obs 41 + reward W
    "ugvo": (5 * 2 + 3 + 48 + 2 + 2 + 41 + 41 + 1) * 8 + 5,
    "soi": (4 * 2 + 2 + 2 + 4 + 4 + 1) * 8 + 5,
    "fas": (2 * 2 + 1 + 2 + 2 + 2 + 1) * 8 + 5,
    # generic families: state fields R+W, action R, time R+W, next_obs + policy obs W, reward W (8 B each) + done + flag
    "fas_discrete": (2 * 2 + 1 + 2 + 2 + 2 + 1) * 8 + 5,
    "ballbalancer": (4 * 2 + 1 + 2 + 3 + 3 + 1) * 8 + 5,
    "twolink": (8 * 2 + 2 + 2 + 6 + 6 + 6 + 1) * 8 + 5,   # + current_state (not a pure function of the state)
    "ugv": (5 * 2 + 2 + 2 + 4 + 4 + 1) * 8 + 5,
    # UavRobust hover: 12 ODE + 3 s1 + 3 att_ref + 3 dot_att_ref R+W, 3 pos_ref R, 6 action, time, 3 x 12 obs, reward
    "uavr_hover": (21 * 2 + 3 + 6 + 2 + 12 * 3 + 1) * 8 + 5,
}
# algorithmic fp64 work per env-step (weighted flops, SURVEY.md section 8d convention), used for the fp64-pipe view
ALGO_FLOPS = {"uav_pos": 5100.0, "uav_att": 3300.0, "cartpole": 3100.0, "ugvo": 54000.0, "soi": 125.0, "fas": 570.0}
PROFILED_ENVS = {"uav_pos": 1 << 20, "uav_att": 1 << 20, "cartpole": 65536, "ugvo": 262144}   # tools/profile_all.sh sizes


def profile_facts(workload):
    """What the committed ncu summaries say about the step kernel of `workload`: DRAM bytes per launch
    (dram__bytes_read + write of the `--set full` capture) and the executed instruction mix per env-step
    (profiles/tools/op_hist.py).  Parsed at run time from profiles/r*/<workload>_final_{keys,ophist}.txt, newest round
    first, so that the roofline follows the profile that is committed, not a constant pasted into this file."""
    unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
    for d in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*")), reverse=True):
        keys, hist = os.path.join(d, f"{workload}_final_keys.txt"), os.path.join(d, f"{workload}_final_ophist.txt")
        if not os.path.exists(keys):
            continue
        out = {"src": os.path.relpath(keys, ROOT), "profiled_envs": PROFILED_ENVS.get(workload)}
        traffic = 0.0
        for line in open(keys):
            m = re.match(r"(dram__bytes_(?:read|write)\.sum)\s+(\w+)\s+\['([0-9.eE+-]+)'\]", line)
            if m:
                traffic += float(m.group(3)) * unit.get(m.group(2), 1.0)
            m = re.match(r"(sm__pipe_fp64_cycles_active\S*|smsp__issue_active\S*|gpu__time_duration\.sum)\s+\S+\s+\['([0-9.eE+-]+)'\]", line)
            if m:
                out[m.group(1)] = float(m.group(2))
        out["dram_bytes"] = traffic or None
        if os.path.exists(hist):
            per = {}
            for line in open(hist):
                m = re.match(r"(\w+)\s+\d+\s+[0-9.]+%\s+per-thread\s+([0-9.]+)", line)
                if m:
                    per[m.group(1)] = float(m.group(2))
            out["fp64_pipe_inst"] = sum(per.get(k, 0.0) for k in ("DFMA", "DMUL", "DADD", "DSETP"))
            out["fp64_flops"] = 2 * per.get("DFMA", 0.0) + per.get("DMUL", 0.0) + per.get("DADD", 0.0)
            out["hist_src"] = os.path.relpath(hist, ROOT)
        return out
    return None


WORKLOADS = {
    "uav_pos": dict(n=1 << 20, desc="UavFntsmcParam position tracking, dt=0.02, time_max=10, 8 gains~U(0,5)/step"),
    "uav_att": dict(n=1 << 20, desc="UavFntsmcParam attitude tracking, dt=0.02, time_max=10, 8 gains~U(0,3)/step"),
    "cartpole": dict(n=65536, desc="CartPole (angle+position) RK4 time-loop step, force~U(-8,8)"),
    "ugvo": dict(n=262144, desc="UGVForwardObstacleAvoidance DPPO2 variant, dt=0.05, 15 circles, one 37-ray scan per step (the pre-step scan is the previous step's post-step scan)"),
    "soi": dict(n=1 << 20, desc="SecondOrderIntegration (ENV), RK4 step"),
    "fas": dict(n=1 << 20, desc="Flight_Attitude_Simulator (PPO2 variant), RK4 time-loop step"),
    "fas_discrete": dict(n=1 << 20, desc="FlightAttitudeSimulatorDiscrete, 2 RK4 steps/period, force from the discrete action set"),
    "ballbalancer": dict(n=1 << 20, desc="BallBalancer1D, RK4 time-loop step"),
    "twolink": dict(n=1 << 20, desc="TwoLinkManipulator, RK4 step with in-register 2x2 solve"),
    "ugv": dict(n=1 << 20, desc="UGVForward, RK4 step"),
    "uavr_hover": dict(n=1 << 20, desc="UavRobust uav_hover (acceleration + torque actions), dt=0.01"),
}


def make_env(workload, n, device, offset, dtype=torch.float64, host_only=False, io_dtype=None):
    import reinforcementlearningplatform_b200 as rlp
    kw = dict(n_envs=n, device=device, dtype=dtype, seed=2024, env_index_offset=offset, auto_reset=True,
              host_only=host_only, io_dtype=io_dtype)
    if workload == "uav_pos":
        return rlp.UavPosCtrlRL(random_trajectory=True, **kw)
    if workload == "uav_att":
        return rlp.UavAttCtrlRL(random_trajectory=True, **kw)
    if workload == "cartpole":
        return rlp.CartPole(**kw)
    if workload == "ugvo":
        return rlp.UGVForwardObstacleAvoidance(variant="dppo2", **kw)
    if workload == "soi":
        return rlp.SecondOrderIntegration(**kw)
    if workload == "fas":
        return rlp.Flight_Attitude_Simulator(variant="ppo2", **kw)
    simple = {"fas_discrete": rlp.FlightAttitudeSimulatorDiscrete, "ballbalancer": rlp.BallBalancer1D,
              "twolink": rlp.TwoLinkManipulator, "ugv": rlp.UGVForward, "uavr_hover": rlp.uav_hover}
    if workload in simple:
        return simple[workload](**kw)
    raise SystemExit(f"unknown workload {workload}")


def action_pool(env, n, pool, device, dtype, seed):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    ar = torch.as_tensor(np.asarray(env.action_range, dtype=np.float64), device=device)
    lo, hi = ar[:, 0].view(1, -1, 1), ar[:, 1].view(1, -1, 1)
    u = torch.rand((pool, ar.shape[0], n), generator=g, device=device, dtype=torch.float64)
    return (lo + (hi - lo) * u).to(dtype).contiguous()


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample_once(self):
        """One NVML reading.  Also called from the main thread right after the timed launches have been enqueued (the
        GPU is then busy with them for tens of milliseconds), so the clocks line never depends on thread scheduling."""
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self.stop_flag and self.nv is not None:
            self.sample_once()
            time.sleep(0.01)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def timed_steps(env, pool, steps, warmup, dist_on, sampler=None, dis_pool=None):
    import torch.distributed as dist
    P = pool.shape[0]
    dis = (lambda k: dis_pool[k % dis_pool.shape[0]]) if dis_pool is not None else (lambda k: None)
    for k in range(warmup):
        env.step_soa(pool[k % P], dis(k))
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        env.step_soa(pool[(warmup + k) % P], dis(warmup + k))
    e1.record()
    if sampler is not None:  # the launches are enqueued, the GPU is executing them: read the clocks under load
        for _ in range(3):
            sampler.sample_once()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist_on:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    return ms


DUMP_LIMIT = 63_000_000   # bytes of array data written by --dump-outputs: with the .npy headers, under 64 MB


def dump_outputs(env, out_dir, seed=0):
    """What the caller of the last step_soa receives, as out_dir/<name>.npy ([instances, ...], float64 or float32).  When
    the whole batch would exceed DUMP_LIMIT, a fixed sample of instances (drawn from `seed`, sorted) is written instead,
    with its indices in instance_index.npy."""
    outs = {"current_state": env.current_state, "next_state": env.next_state, "policy_state": env.policy_state,
            "reward": env.reward, "is_terminal": env.is_terminal, "terminal_flag": env.terminal_flag, "time": env.time}
    outs = {k: (v if v.dtype in (torch.float64, torch.float32) else v.to(torch.float32)) for k, v in outs.items()}
    n = env.n_envs
    per_instance = 8 + sum(v[0].numel() * v.element_size() for v in outs.values())   # + the index column
    k = min(n, DUMP_LIMIT // per_instance)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
    sel = torch.as_tensor(idx, device=env.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "instance_index.npy"), idx.astype(np.float64))
    for name, v in outs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v.index_select(0, sel).cpu().numpy())


# Shards of the host-buffer path (timed_e2e): shard c's copies overlap shard c+1's kernel.  Measured on one B200 at 1 M
# instances (tools/e2e_sweep.py): 1 shard 0.76e9, 2 shards 1.30e9, 3 shards 1.29e9, 4 shards 1.21e9, 8 shards 1.07e9
# env-steps/s against 1.46e9 for the bare copies -- two shards already keep both directions of the link busy, more only add
# host <-> device hand-overs; CUDA graphs around a shard's step change nothing (the host is not the limit).
E2E_SHARDS = 2


def timed_e2e(workload, n, steps, warmup, dist_on, seed, device, offset, dtype, chunks=E2E_SHARDS, io_dtype=None):
    """Same metric through the public API with HOST buffers.  Every step, for every instance: the actions are copied
    from pinned host memory, the step kernel runs, and policy_state / reward / is_terminal are read back to pinned host
    memory, where the host waits for them before it issues that instance's next action.  The batch is split into
    `chunks` independent VecEnv shards on their own CUDA streams so that shard c's copies overlap shard c+1's kernel
    (PCIe is full duplex); the dependency action(t+1) <- result(t) is kept per shard."""
    import torch.distributed as dist
    nc = n // chunks
    envs, streams = [], []
    for c in range(chunks):
        e = make_env(workload, nc, device, offset + c * nc, dtype, io_dtype=io_dtype)
        e.reset(True)
        envs.append(e)
        streams.append(torch.cuda.Stream(device=device))
    A, S = envs[0].action_dim, envs[0].state_dim
    dtype = io_dtype or dtype  # element type of every host <-> device buffer below
    rng = np.random.default_rng(seed)
    ar = np.asarray(envs[0].action_range, dtype=np.float64)
    host_a = [[torch.from_numpy(rng.uniform(ar[:, :1], ar[:, 1:], size=(A, nc))).to(dtype).pin_memory() for _ in range(2)]
              for _ in range(chunks)]
    dev_a = [torch.empty((A, nc), dtype=dtype, device=device) for _ in range(chunks)]
    h_obs = [torch.empty((S, nc), dtype=dtype).pin_memory() for _ in range(chunks)]
    h_rew = [torch.empty((nc,), dtype=dtype).pin_memory() for _ in range(chunks)]
    h_done = [torch.empty((nc,), dtype=torch.uint8).pin_memory() for _ in range(chunks)]
    ready = [torch.cuda.Event() for _ in range(chunks)]
    torch.cuda.synchronize()

    def one(k):
        for c in range(chunks):
            if k > 0:
                ready[c].synchronize()  # the host-side policy needs shard c's previous result before acting on it
            with torch.cuda.stream(streams[c]):
                dev_a[c].copy_(host_a[c][k & 1], non_blocking=True)
                envs[c].step_soa(dev_a[c])
                h_obs[c].copy_(envs[c]._reset_obs, non_blocking=True)
                h_rew[c].copy_(envs[c]._reward, non_blocking=True)
                h_done[c].copy_(envs[c]._done, non_blocking=True)
                ready[c].record(streams[c])

    for k in range(warmup):
        one(k)
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        one(warmup + k)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3  # host clock around fully synchronised work (copies on several streams)
    if dist_on:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    el = torch.tensor([], dtype=dtype).element_size()
    return ms, chunks * nc, A * chunks * nc * el, (S * nc + nc) * chunks * el + chunks * nc


def cpu_port(workload, n, steps, threads, seed=2024):
    """The C restatement of the reference (oracle/, kind "port") on the host cores: bounded sample."""
    from oracle import oracle
    from reinforcementlearningplatform_b200 import _lib
    host = make_env(workload, n, "cuda", 0, host_only=True)
    sf, od, ad, dd = _lib.dims(host.ENV_ID, host.VARIANT)
    orc = oracle.OracleEnv(host.ENV_ID, host._params, n, sf, od, ad, dd, seed=seed, auto_reset=True, nthreads=threads)
    orc.reset()
    rng = np.random.default_rng(seed)
    ar = np.asarray(host.action_range, dtype=np.float64)
    acts = [rng.uniform(ar[:, :1], ar[:, 1:], size=(ad, n)) for _ in range(4)]
    orc.step(acts[0])  # warm-up (page faults, thread pool)
    t0 = time.perf_counter()
    for k in range(steps):
        orc.step(acts[k % 4])
    dt = time.perf_counter() - t0
    return n * steps / dt, dt


def reference_tree():
    """Where the UNMODIFIED Python reference can be imported from: the tree RLP_REFERENCE names, else the byte-compiled
    staging made by oracle/stage_reference.py."""
    for d in (os.environ.get("RLP_REFERENCE"), os.path.join(ROOT, "oracle", "_ref")):
        if d and os.path.isdir(os.path.join(d, "environment")):
            return d
    return None


def reference_python(workload, seconds, procs):
    """The reference's own Python step loop (oracle/bench_reference_python.py --worker: e.g. the body of
    PPO2-4-UavFntsmcParamPos/train.py:290-297 with uniform random gains, reset(True) on terminal) in `procs` processes at
    once, one per host core, OMP_NUM_THREADS=1 like the reference sets it (DPPO2-4-UGVForwardObstacleAvoidance/
    train.py:22).  Returns aggregate env-steps/s, per-core mean and the tree the modules came from."""
    tree = reference_tree()
    if tree is None:
        return None
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", RLP_REFERENCE=tree,
               CUDA_VISIBLE_DEVICES="", PYTHONDONTWRITEBYTECODE="1")
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "bench_reference_python.py"), "--worker", workload,
           "--seconds", str(seconds)]
    ps = [subprocess.Popen(cmd + ["--seed", str(k + 1)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, env=env, text=True)
          for k in range(procs)]
    rates = []
    for q in ps:
        out, _ = q.communicate(timeout=600)
        try:
            d = json.loads(out.strip().splitlines()[-1])
            rates.append(d["steps"] / d["seconds"])
        except Exception:
            pass
    if not rates:
        return None
    return {"value": float(sum(rates)), "unit": "env-steps/s", "cores": len(rates), "per_core": float(np.mean(rates)),
            "kind": "reference", "tree": os.path.relpath(tree, ROOT) if tree.startswith(ROOT) else tree,
            "sample": f"{len(rates)} processes x {seconds:g} s of the reference's Python step loop (200 warm-up steps), "
                      "uniform random actions, reset(True) on terminal"}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores -- the unmodified
    Python classes (byte-compiled staging oracle/_ref on the GPU box), one process per core.  Nothing of the product
    package is imported here.  Only if no reference tree exists at all does this arm fall back to the C port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # a "step" of this arm = one env-step on every core; --steps K is honoured as K seconds-long windows, bounded
    seconds = float(min(max(args.steps * 0.25, 3.0), 30.0))
    reference_python(args.workload, min(1.0, seconds), cores)         # warm-up: page in numpy / cv2 on every core
    ref = reference_python(args.workload, seconds, cores)
    if ref is not None:
        val = ref["value"]
        base = ref
        envs, per_step = ref["cores"], ref["cores"] / val * 1e3
    else:
        threads = cores
        n = min(WORKLOADS[args.workload]["n"], 1 << 17)
        for _ in range(max(args.warmup, 1)):
            cpu_port(args.workload, n, 1, threads)
        val, dt = cpu_port(args.workload, n, args.steps, threads)
        base = {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "port",
                "sample": f"{n} instances x {args.steps} steps, OpenMP over instances (no reference tree found)"}
        envs, per_step = n, dt * 1e3 / args.steps
    line = {
        "impl": "reference", "metric": "env-steps/sec", "value": val, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "envs": envs, "desc": WORKLOADS[args.workload]["desc"],
                   "note": "one env instance per host core, all cores at once; a step = one env-step on every core"},
        "cpu_baseline": base,
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def copy_probe(n, A, S, steps, dev, dist_on, chunks=E2E_SHARDS):
    """The bytes of one e2e step moved by plain cudaMemcpyAsync (torch copy_ of pinned float32 buffers, one call per
    buffer), no kernel in between, same shard / stream structure: what the host link alone allows at this GPU count."""
    import torch.distributed as dist
    nc = n // chunks
    streams = [torch.cuda.Stream(device=dev) for _ in range(chunks)]
    h_a = [torch.empty((A, nc), dtype=torch.float32).pin_memory() for _ in range(chunks)]
    d_a = [torch.empty((A, nc), dtype=torch.float32, device=dev) for _ in range(chunks)]
    d_o = [torch.empty((S + 1, nc), dtype=torch.float32, device=dev) for _ in range(chunks)]
    h_o = [torch.empty((S + 1, nc), dtype=torch.float32).pin_memory() for _ in range(chunks)]
    d_d = [torch.empty((nc,), dtype=torch.uint8, device=dev) for _ in range(chunks)]
    h_d = [torch.empty((nc,), dtype=torch.uint8).pin_memory() for _ in range(chunks)]

    def one():
        for c in range(chunks):
            with torch.cuda.stream(streams[c]):
                d_a[c].copy_(h_a[c], non_blocking=True)
                h_o[c].copy_(d_o[c], non_blocking=True)
                h_d[c].copy_(d_d[c], non_blocking=True)
    for _ in range(3):
        one()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    if dist_on:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def also_workloads(args, dev, dtype, peaks):
    """Short device-resident measurements of the other single-GPU configs (same timing rules, fewer steps)."""
    out = []
    hbm = peaks.get("hbm_gbs", 6650.0)
    for w in ("cartpole", "soi", "fas", "ugvo", "fas_discrete", "ballbalancer", "twolink", "ugv", "uavr_hover"):
        if w == args.workload:
            continue
        n = WORKLOADS[w]["n"]
        env = make_env(w, n, dev, 0, dtype)
        env.reset(True)
        pool = action_pool(env, n, 4, dev, dtype, seed=7)
        steps = 20 if w == "ugvo" else 100
        ms = timed_steps(env, pool, steps, 5, False)
        per = ms * 1e-3 / steps
        out.append({"workload": w, "envs": n, "value": n / per, "unit": "env-steps/s", "ms_per_step": ms / steps,
                    "hbm_frac": ALGO_BYTES[w] * n / per / 1e9 / hbm, "desc": WORKLOADS[w]["desc"]})
        if w == "ugvo":
            # the line above covers the first steps of fresh episodes, where few instances terminate; once episodes end at
            # their steady-state rate (~4 % of the instances per step) the map rejection sampling of the auto-reset launch
            # costs as much as the step kernel: measured separately after 60 more steps
            ms = timed_steps(env, pool, 60, 60, False)
            per = ms * 1e-3 / 60
            out.append({"workload": "ugvo_steady", "envs": n, "value": n / per, "unit": "env-steps/s", "ms_per_step": ms / 60,
                        "hbm_frac": ALGO_BYTES[w] * n / per / 1e9 / hbm,
                        "desc": WORKLOADS[w]["desc"] + "; steps 85-145 of the batch: auto-resets at their steady-state rate"})
        del env, pool
        torch.cuda.empty_cache()
    # fp32 mode (state, arithmetic and I/O in float32; tolerances: tests/helpers.py FP32_TOL) of the headline workload
    # and of config #2 (CartPole, fp64 vs fp32)
    for w in (args.workload, "cartpole"):
        n = WORKLOADS[w]["n"]
        env = make_env(w, n, dev, 0, torch.float32)
        env.reset(True)
        pool = action_pool(env, n, 4, dev, torch.float32, seed=7)
        ms = timed_steps(env, pool, 100, 5, False)
        per = ms * 1e-3 / 100
        out.append({"workload": w + ":f32", "envs": n, "value": n / per, "unit": "env-steps/s", "ms_per_step": ms / 100,
                    "hbm_frac": ALGO_BYTES[w] / 2.0 * n / per / 1e9 / hbm, "desc": WORKLOADS[w]["desc"] + " [fp32 mode]"})
        del env, pool
        torch.cuda.empty_cache()
    # config #3: GAE over a 2048-step rollout, 131072 env columns per GPU
    from reinforcementlearningplatform_b200 import gae as G
    T, N = 2048, 131072
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    mk = lambda: torch.randn((T, N), generator=g, device=dev, dtype=torch.float32)
    r, vs, vsn = mk(), mk(), mk()
    done = (torch.rand((T, N), generator=g, device=dev) < 0.002).float()
    succ = done * (torch.rand((T, N), generator=g, device=dev) < 0.5).float()
    for _ in range(3):
        adv, vt, st = G.gae(r, vs, vsn, done, succ, 0.99, 0.95)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    reps = 10
    for _ in range(reps):
        adv, vt, st = G.gae(r, vs, vsn, done, succ, 0.99, 0.95)
    e1.record()
    torch.cuda.synchronize()
    per = e0.elapsed_time(e1) * 1e-3 / reps
    out.append({"workload": "gae", "T": T, "N": N, "value": T * N / per, "unit": "elements/s", "ms_per_step": per * 1e3,
                "hbm_frac": 28.0 * T * N / per / 1e9 / hbm,
                "desc": "PPO2 GAE reverse scan + (sum, sum^2, n) statistics, float32, time-major [T, N]"})
    del r, vs, vsn, done, succ, adv, vt
    torch.cuda.empty_cache()
    # the kernels either side of the step (SURVEY 8f): GAE over the rollout's own u8 / i32 columns, PPO v1 returns,
    # running normalisation, and the batched actor + critic forward (tensor cores, 3xTF32, and the FP32-FMA version)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import microbench
    descs = {"gae_flags": "K-GAE over the device-resident rollout (u8 done, i32 flag)", "mc_returns": "PPO v1 Monte-Carlo returns",
             "norm": "running mean/std normalisation of a [6, 4 M] float32 batch (statistics + merge/apply)",
             "policy": "actor 6-64-64-32-8 + critic 6-64-32-1 forward, sample, clamp, log-prob for 1 M instances (tcgen05 UMMA, activations in TMEM, 3xTF32 split)",
             "policy_fp32": "the same forward on the FP32 FMA pipe",
             "gae_small_seq": "K-GAE on the reference's own rollout shape (T = 2048, 8 columns): one thread per column, 2048 dependent steps",
             "gae_small_scan": "the same with acc_mode 2: warp-level scan along time (32 steps per trip composed by shuffles)",
             "learn": "K-LEARN: one 16,384-sample mini-batch of the PPO2 update (both nets: forward, loss, backward, "
                      "fixed-order reduction, clip + Adam) out of a 64 x 16,384 device rollout",
             "learn_torch": "the same mini-batch update by torch autograd + torch.optim.Adam (round 1's learner)"}
    for kind, desc in descs.items():
        m = microbench.run(kind, 10, dev=dev)
        m["hbm_frac"] = m["achieved_gbs"] / hbm
        m["desc"] = desc
        out.append(m)
        torch.cuda.empty_cache()
    # the whole on-device collection step of a PPO2 iteration (ppo2.VecPPO2.collect): K-POLICY -> step kernel (rows of
    # the rollout buffer written in place) -> K-NORM on the reward, 1 M UavFntsmcParam-pos instances, 16-step rollout
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    n = WORKLOADS["uav_pos"]["n"]
    env = make_env("uav_pos", n, dev, 0, torch.float64, io_dtype=torch.float32)
    env.reset(True)
    actor, critic = reference_nets(env.state_dim, env.action_dim, dev, init_std=0.45)
    agent = VecPPO2(env, actor, critic, {"buffer_size": 16, "K_epochs": 1}, std=0.45)
    agent.collect()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    agent.collect()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    out.append({"workload": "ppo2_collect_uav_pos", "T": 16, "envs": n, "value": 16 * n / (ms * 1e-3), "unit": "env-steps/s",
                "ms_per_step": ms / 16, "desc": "policy forward (3xTF32) + fused UAV step + reward normalisation per time step, "
                                                 "everything device-resident (float32 I/O, fp64 state and arithmetic)"})
    del agent, env
    torch.cuda.empty_cache()
    return out


def also_sharded(args, dev, dtype, world, rank, group_on):
    """The configs of BASELINE.json that shard over GPUs, run by EVERY rank at every GPU count (rank 0 reports; times are
    the max over ranks):
      #3  rollout_soi / rollout_fas: 131,072 instances per GPU x 2048 steps written in place into the time-major buffer,
          then K-GAE and the global advantage normalisation (3-double all-reduce) -- Proximal_Policy_Optimization2.py:88-100;
      #5  dppo2_ugvo: one DPPO2 iteration of UGVForwardObstacleAvoidance with the demo's 41-256-256 nets: K-POLICY (tcgen05,
          streamed weights) -> step kernel -> reward normalisation for T steps, then K-GAE + statistics all-reduce and
          k_epo = 6 full-batch epochs with one flat-gradient all-reduce per net and epoch (Distributed_PPO2.py:86-104 made
          synchronous).  T = 16 instead of the demo's 300-step buffer: the update runs on torch autograd (not this repo's
          kernels) and would otherwise dominate the bench's wall time;
      #4  uav_att, uav_pos at 2 M instances per GPU, uav_pos with an injected disturbance buffer."""
    import torch.distributed as dist
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, dppo2_nets
    out = []

    def maxr(x):
        if not group_on:
            return float(x)
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for w, T, N, cfg in (("soi", 2048, 131072, "#3"), ("fas", 2048, 131072, "#3"), ("cartpole", 1000, 65536, "#2")):
        ms_roll, ms_gae = rollout_pipeline(w, N, T, dev, group_on, offset=rank * N)
        ms_roll, ms_gae = maxr(ms_roll), maxr(ms_gae)
        out.append({"workload": f"rollout_{w}", "T": T, "envs_per_gpu": N, "n_gpus": world,
                    "value": world * T * N / ((ms_roll + ms_gae) * 1e-3), "rollout_value": world * T * N / (ms_roll * 1e-3),
                    "unit": "env-steps/s", "ms_rollout": ms_roll, "ms_gae_allreduce_norm": ms_gae,
                    "desc": f"config {cfg}, {WORKLOADS[w]['desc']}: {T}-step rollout into the device buffer by ONE "
                            "b200env_rollout launch (state in registers), K-GAE, 3-double all-reduce, normalise"})
        torch.cuda.empty_cache()
    # config #5
    N, T = WORKLOADS["ugvo"]["n"], 16
    env = make_env("ugvo", N, dev, rank * N, torch.float64, io_dtype=torch.float32)
    env.reset(True)
    ar = np.asarray(env.action_range, dtype=np.float64)
    actor, critic = dppo2_nets(env.state_dim, env.action_dim, ar[:, 0], ar[:, 1], dev)
    agent = VecPPO2(env, actor, critic, {"buffer_size": T, "K_epochs": 6, "using_mini_batch": False, "a_lr": 2e-5,
                                          "c_lr": 2e-4, "use_lr_decay": False}, std=actor.std, seed=3)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    agent.collect()
    agent.learn()
    torch.cuda.synchronize()
    if group_on:
        dist.barrier()
    ev[0].record()
    agent.collect()
    ev[1].record()
    agent.learn()
    ev[2].record()
    torch.cuda.synchronize()
    ms_c, ms_l = maxr(ev[0].elapsed_time(ev[1])), maxr(ev[1].elapsed_time(ev[2]))
    out.append({"workload": "dppo2_ugvo", "T": T, "envs_per_gpu": N, "n_gpus": world,
                "value": world * T * N / ((ms_c + ms_l) * 1e-3), "collect_value": world * T * N / (ms_c * 1e-3),
                "unit": "env-steps/s", "ms_collect": ms_c, "ms_learn": ms_l, "grad_allreduces": 12,
                "desc": "config #5: UGVForwardObstacleAvoidance (DPPO2 variant) x 41-256-256 nets; collect = K-POLICY + step "
                        "+ reward normalisation per time step; learn = K-GAE + statistics all-reduce + 6 full-batch epochs "
                        "(torch autograd) with one flat-gradient all-reduce per net and epoch"})
    del agent, env, actor, critic
    torch.cuda.empty_cache()
    # a whole PPO2 iteration on config #4's env and the reference's nets, nothing but this repo's kernels between the
    # first observation and the updated weights: collect (K-POLICY -> step kernel -> K-NORM, T steps) and learn (critic
    # values by K-POLICY, K-GAE, statistics all-reduce, K_epochs x mini-batches of K-LEARN with one flat-gradient
    # all-reduce per mini-batch when sharded)
    from reinforcementlearningplatform_b200.ppo2 import reference_nets
    N, T, K, mb = 1 << 18, 32, 4, 1 << 16
    env = make_env("uav_pos", N, dev, rank * N, torch.float64, io_dtype=torch.float32)
    env.reset(True)
    actor, critic = reference_nets(env.state_dim, env.action_dim, dev, init_std=0.45)
    agent = VecPPO2(env, actor, critic, {"buffer_size": T, "K_epochs": K, "mini_batch_size": mb, "use_lr_decay": False},
                    std=0.45, seed=5)
    assert agent.fused is not None
    agent.collect()
    agent.learn()
    torch.cuda.synchronize()
    if group_on:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    agent.collect()
    ev[1].record()
    agent.learn()
    ev[2].record()
    torch.cuda.synchronize()
    ms_c, ms_l = maxr(ev[0].elapsed_time(ev[1])), maxr(ev[1].elapsed_time(ev[2]))
    n_upd = K * (-(-T * N // mb))
    out.append({"workload": "ppo2_iter_uav_pos", "T": T, "envs_per_gpu": N, "n_gpus": world, "K_epochs": K, "mini_batch": mb,
                "value": world * T * N / ((ms_c + ms_l) * 1e-3), "collect_value": world * T * N / (ms_c * 1e-3),
                "learn_samples_per_s": world * K * T * N / (ms_l * 1e-3), "unit": "env-steps/s", "ms_collect": ms_c,
                "ms_learn": ms_l, "updates": n_upd, "us_per_update": ms_l * 1e3 / n_upd,
                "desc": "config #4 env + the reference's 6-64-64-32-8 / 6-64-32-1 nets: one full PPO2 iteration on device; "
                        "learn = K-POLICY critic values + K-GAE + K-LEARN (grad, reduce, clip + Adam launches per "
                        "mini-batch, flat-gradient all-reduce in between when sharded); no torch autograd"})
    del agent, env, actor, critic
    torch.cuda.empty_cache()
    # config #4 variants
    for name, w, n, with_dis in (("uav_att", "uav_att", 1 << 20, False), ("uav_pos_2M", "uav_pos", 1 << 21, False),
                                 ("uav_pos_dis", "uav_pos", 1 << 20, True)):
        env = make_env(w, n, dev, rank * n, dtype)
        env.reset(True)
        pool = action_pool(env, n, 4, dev, dtype, seed=rank + 7)
        dis = None
        if with_dis:  # sinusoid + noise force disturbance per instance, 4 rotating buffers (UavRobust/ref_cmd.py:46-61 style)
            g = torch.Generator(device=dev)
            g.manual_seed(rank + 9)
            dis = (0.5 * torch.randn((4, env._dd, n), generator=g, device=dev, dtype=torch.float64)).to(dtype).contiguous()
        ms = timed_steps(env, pool, 40, 5, group_on, dis_pool=dis)
        out.append({"workload": name, "envs_per_gpu": n, "n_gpus": world, "value": world * n * 40 / (ms * 1e-3),
                    "unit": "env-steps/s", "ms_per_step": ms / 40,
                    "desc": WORKLOADS[w]["desc"] + (" + injected disturbance [3, N] per step" if with_dis else "")})
        del env, pool, dis
        torch.cuda.empty_cache()
    return out


def exchange_times(dev, reps=50):
    """The only collectives of the path (SURVEY 8e, config #5), timed on the device over NCCL: the DPPO2 gradient
    average as one all-reduce of a flat fp32 buffer (154 k parameters of the 41-256-256-{2,1} demo nets, and 9.5 k of
    the 6-64-64-32 / 6-64-32 nets), the 3-double advantage statistics, the 3 x dim doubles of the normaliser."""
    import torch.distributed as dist
    out = {}
    for name, t in (("grad_allreduce_154k_fp32", torch.zeros(154_000, dtype=torch.float32, device=dev)),
                    ("grad_allreduce_9k5_fp32", torch.zeros(9_500, dtype=torch.float32, device=dev)),
                    ("adv_stats_3xf64", torch.zeros(3, dtype=torch.float64, device=dev))):
        for _ in range(5):
            dist.all_reduce(t)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dist.all_reduce(t)
        e1.record()
        torch.cuda.synchronize()
        us = torch.tensor([e0.elapsed_time(e1) * 1e3 / reps], device=dev, dtype=torch.float64)
        dist.all_reduce(us, op=dist.ReduceOp.MAX)
        out[name] = {"us": float(us.item()), "bytes": t.numel() * t.element_size()}
    g = torch.zeros(dist.get_world_size(), 3, 6, dtype=torch.float64, device=dev)
    b = torch.zeros(1, 3, 6, dtype=torch.float64, device=dev)
    for _ in range(5):
        dist.all_gather_into_tensor(g, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dist.all_gather_into_tensor(g, b)
    e1.record()
    torch.cuda.synchronize()
    us = torch.tensor([e0.elapsed_time(e1) * 1e3 / reps], device=dev, dtype=torch.float64)
    dist.all_reduce(us, op=dist.ReduceOp.MAX)
    out["norm_stats_allgather_18xf64"] = {"us": float(us.item()), "bytes": 144}
    return out


def rollout_pipeline(workload, n, T, dev, dist_on, seed=5, offset=0):
    """config #3: a T-step rollout written by the step kernel straight into a device-resident time-major float32
    buffer (rollout.RolloutBuffer), then K-GAE over it and the global advantage normalisation (3-double all-reduce when
    sharded).  V(s), V(s') are synthetic N(0,1) columns (the critic is outside the hot path).  Returns the times of the
    two stages in ms."""
    import reinforcementlearningplatform_b200 as rlp
    env = make_env(workload, n, dev, offset, torch.float64, io_dtype=torch.float32)
    env.reset(True)
    buf = rlp.RolloutBuffer(T, env)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    ar = torch.as_tensor(np.asarray(env.action_range, dtype=np.float64), device=dev, dtype=torch.float32)
    lo, hi = ar[:, 0].view(1, -1, 1), ar[:, 1].view(1, -1, 1)
    buf.a.copy_(lo + (hi - lo) * torch.rand(buf.a.shape, generator=g, device=dev, dtype=torch.float32))
    vs = torch.randn((T, n), generator=g, device=dev, dtype=torch.float32)
    vsn = torch.randn((T, n), generator=g, device=dev, dtype=torch.float32)
    buf.collect(env, 0, 8)  # warm-up
    buf.gae(vs, vsn, 0.99, 0.95)
    torch.cuda.synchronize()
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    buf.collect(env)  # b200env_rollout: all T steps in one call (one fused kernel for SOI / FAS)
    e[1].record()
    adv, vt = buf.gae(vs, vsn, 0.99, 0.95)
    e[2].record()
    torch.cuda.synchronize()
    return e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000, help="timed steps of the headline workload, split into up to 5 blocks")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="uav_pos", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="instances per GPU (default: the config's)")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / e2e / also (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    torch.cuda.set_device(local)
    if dist_on:
        # NCCL prints "NCCL version ..." on stdout when the communicator is created: route fd 1 to stderr around the
        # initialisation (and the first collective), so that stdout carries exactly ONE JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    n = args.envs or WORKLOADS[args.workload]["n"]
    dev = torch.device("cuda", local)

    env = make_env(args.workload, n, dev, rank * n, dtype)
    env.reset(True)
    pool = action_pool(env, n, 4, dev, dtype, seed=rank + 1)
    sampler = ClockSampler(local)
    sampler.start()
    # the K timed steps, in up to five blocks (each between barrier + synchronize, CUDA events, max over ranks): `value`
    # comes from the median block's time per step, the spread is reported
    REPEATS = min(5, args.steps)
    sizes = [args.steps // REPEATS + (r < args.steps % REPEATS) for r in range(REPEATS)]
    blocks = [timed_steps(env, pool, k, args.warmup if r == 0 else 1, dist_on, sampler) for r, k in enumerate(sizes)]
    clocks = sampler.result()
    per_step = [b_ / k for b_, k in zip(blocks, sizes)]
    ms_step = float(np.median(per_step))
    value = world * n / (ms_step * 1e-3)
    per_launch_s = ms_step * 1e-3
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)
    el = 8 if dtype == torch.float64 else 4
    algo_bytes = ALGO_BYTES[args.workload] * el / 8.0 * n
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    achieved_gbs = algo_bytes / per_launch_s / 1e9
    from reinforcementlearningplatform_b200 import _lib
    fma_peak = _lib.measure_fma_peak(_lib.F64 if el == 8 else _lib.F32)  # TFLOP/s, live, this GPU
    facts = profile_facts(args.workload) if el == 8 else None
    hbm_view = {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                "algorithmic_bytes": algo_bytes, "peak_source": "measured" if "hbm_gbs" in peaks else "fallback"}
    kernel = f"{args.workload}_step_kernel<{'double' if el == 8 else 'float'}>"
    compute_bound = args.workload not in ("soi", "fas", "fas_discrete")
    if compute_bound and facts and facts.get("fp64_flops"):
        # binding resource = the FP64 pipe: executed fp64 flops (DFMA = 2) per env-step from the committed SASS histogram
        # x instances / launch time against the FMA peak measured live; `frac_pipe_slots` counts every fp64-pipe
        # instruction as one issue slot of that pipe (peak / 2 instructions per second)
        ach = facts["fp64_flops"] * n / per_launch_s / 1e12
        roofline = {"bound": "fp64_pipe", "achieved": ach, "peak": fma_peak, "unit": "TFLOP/s", "frac": ach / fma_peak,
                    "frac_pipe_slots": facts["fp64_pipe_inst"] * n / per_launch_s / 1e12 / (fma_peak / 2.0),
                    "peak_source": "b200_measure_fma_peak, live (8 independent FMA chains per thread)",
                    "executed_per_env_step": {"fp64_flops": facts["fp64_flops"], "fp64_pipe_inst": facts["fp64_pipe_inst"],
                                              "src": facts.get("hist_src")},
                    "ncu_fp64_pipe_active_pct": facts.get("sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active"),
                    "weighted_algorithmic_tflops": ALGO_FLOPS.get(args.workload, float("nan")) * n / per_launch_s / 1e12,
                    "hbm": hbm_view}
    else:
        roofline = dict(hbm_view, bound="hbm")
        roofline["fp64_pipe"] = {"peak_tflops_fma": fma_peak,
                                 "weighted_algorithmic_tflops": ALGO_FLOPS.get(args.workload, float("nan")) * n / per_launch_s / 1e12}
    same_size = facts and facts.get("profiled_envs") == n
    roofline.update({"traffic": facts["dram_bytes"] if (facts and same_size) else None,
                     "traffic_source": facts["src"] if (facts and same_size) else None, "kernel": kernel})
    line = {
        "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": args.workload, "envs_per_gpu": n, "desc": WORKLOADS[args.workload]["desc"],
                   "auto_reset": True, "parallelism": f"env-shard x{world}",
                   "l2": "per-step working set (state + action + outputs) exceeds the 126 MB L2; 4 rotating action buffers"
                   if n >= (1 << 19) else "working set fits L2 (config size); launch-bound"},
        "repeats": {"blocks": REPEATS, "steps_per_block": sizes, "ms_per_step": per_step, "median_ms_per_step": ms_step,
                    "spread": (max(per_step) - min(per_step)) / ms_step},
        "roofline": roofline,
        "clocks": clocks, "gpu_launches": args.steps,
    }
    if not args.no_extras:
        A_dim, S_dim = env.action_dim, env.state_dim
        del env, pool
        torch.cuda.empty_cache()
        # the host-timed region is short (0.8 ms per step): 100 steps per block and the median of three blocks keep one-off
        # host hiccups (a page fault, a scheduler tick) out of the number
        e_steps = max(100, args.steps)
        e_runs = [timed_e2e(args.workload, n, e_steps, 5, dist_on, rank + 11, dev, rank * n, dtype, io_dtype=torch.float32)
                  for _ in range(3)]
        e_ms, e_n, h2d, d2h = sorted(e_runs, key=lambda r: r[0])[1]
        p_ms = sorted(copy_probe(n, A_dim, S_dim, e_steps, dev, dist_on) for _ in range(3))[1]
        e_val = world * e_n * e_steps / (e_ms * 1e-3)
        line["e2e"] = {"value": e_val, "unit": "env-steps/s", "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "io_dtype": "f32", "state_and_arithmetic": args.dtype, "steps": e_steps,
                       "blocks_ms_per_step": [r[0] / e_steps for r in e_runs],
                       "copy_probe": {"value": world * e_n * e_steps / (p_ms * 1e-3), "unit": "env-steps/s-equivalent",
                                      "h2d_gbs": world * h2d * e_steps / (p_ms * 1e-3) / 1e9,
                                      "d2h_gbs": world * d2h * e_steps / (p_ms * 1e-3) / 1e9,
                                      "what": "the same pinned buffers moved by one cudaMemcpyAsync each (torch copy_), no "
                                              f"kernel in between, same {E2E_SHARDS} shards / streams"},
                       "frac_of_copy_probe": p_ms / e_ms,
                       "api": f"VecEnv.step_soa on {E2E_SHARDS} shards / {E2E_SHARDS} streams: pinned host float32 actions in (the reference's "
                              "actor emits float32), float32 policy_state + reward and u8 is_terminal out every step; "
                              "state and arithmetic stay in the env dtype; the host waits for a shard's result before "
                              "its next action"}
        if dtype == torch.float64 and world == 1:
            f_ms, f_n, fh, fd = timed_e2e(args.workload, n, e_steps, 3, dist_on, rank + 11, dev, rank * n, dtype)
            line["e2e_f64_io"] = {"value": world * f_n * e_steps / (f_ms * 1e-3), "unit": "env-steps/s",
                                  "h2d_bytes_per_step": fh, "d2h_bytes_per_step": fd, "io_dtype": "f64"}
        also = also_sharded(args, dev, dtype, world, rank, dist_on)          # every rank takes part
        if rank == 0 and world == 1:
            also += also_workloads(args, dev, dtype, peaks)
        if rank == 0:
            line["also"] = also
        if rank == 0 and world == 1:
            threads = os.cpu_count() or 1
            ref = reference_python(args.workload, 4.0, threads)
            cn = min(n, 1 << 17)
            cval, cdt = cpu_port(args.workload, cn, 40, threads)
            csteps = int(min(max(40 * 6.0 / max(cdt, 1e-3), 40), 4000))  # ~6 s of CPU work
            cval, cdt = cpu_port(args.workload, cn, csteps, threads)
            port = {"value": cval, "unit": "env-steps/s", "cores": threads, "kind": "port",
                    "sample": f"{cn} instances x {csteps} steps ({cdt:.1f} s), C restatement of the reference (oracle/), "
                              "OpenMP over instances"}
            if ref is not None:
                line["cpu_baseline"] = dict(ref, port=port, reference_python=ref)
            else:
                line["cpu_baseline"] = dict(port, reference_python=None,
                                            note="no reference tree (oracle/_ref not staged): C port only")
    if dist_on:
        line["exchange"] = exchange_times(dev)
    if rank == 0:
        print(json.dumps(line))
    if dist_on:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
