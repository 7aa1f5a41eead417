"""Device-resident micro-benchmarks of the scan / normalisation kernels (K-GAE, K-RET, K-NORM) for ncu captures and
for the `also` block of bench.py.  python tools/microbench.py gae|gae_flags|mc_returns|norm [reps]"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def run(kind, reps=10, T=2048, N=131072, dev="cuda"):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200 import gae as G
    g = torch.Generator(device=dev)
    g.manual_seed(3)
    mk = lambda: torch.randn((T, N), generator=g, device=dev, dtype=torch.float32)
    if kind in ("gae", "gae_flags", "mc_returns"):
        r, vs, vsn = mk(), mk(), mk()
        dn = torch.rand((T, N), generator=g, device=dev) < 0.002
        done_u8 = dn.to(torch.uint8)
        flag = (dn & (torch.rand((T, N), generator=g, device=dev) < 0.5)).to(torch.int32) * 3
        done, succ = dn.float(), (dn & (flag != 3)).float()
        if kind == "gae":
            fn, nbytes = (lambda: G.gae(r, vs, vsn, done, succ, 0.99, 0.95)), 28.0
        elif kind == "gae_flags":
            fn, nbytes = (lambda: G.gae_flags(r, vs, vsn, done_u8, flag, 3, 0.99, 0.95)), 25.0
        else:
            fn, nbytes = (lambda: G.mc_returns(r, done_u8, 0.99)), 9.0
        units = T * N
    elif kind in ("gae_small_seq", "gae_small_scan"):
        # the reference's own rollout shape (one env, T = 2048) and a handful of envs: sequential column walk vs warp scan
        Ts, Ns = 2048, int(os.environ.get("GAE_N", "8"))
        mk2 = lambda: torch.randn((Ts, Ns), generator=g, device=dev, dtype=torch.float32)
        r, vs, vsn = mk2(), mk2(), mk2()
        done = (torch.rand((Ts, Ns), generator=g, device=dev) < 0.002).float()
        mode = 2 if kind == "gae_small_scan" else 1
        fn, nbytes, units = (lambda: G.gae(r, vs, vsn, done, done, 0.99, 0.95, acc_mode=mode)), 28.0, Ts * Ns
    elif kind == "norm":
        dim, n = 6, 1 << 22  # 6 x 4 M float32 = 100 MB per pass: larger than what L2 keeps between the two kernels
        x = torch.randn((dim, n), generator=g, device=dev, dtype=torch.float32)
        y = torch.empty_like(x)
        nz = rlp.Normalization(dim, device=dev, sync=False)
        fn, nbytes, units = (lambda: nz.normalize_soa(x, out=y)), 12.0, dim * n
    elif kind == "policy_wide":
        # the 41-256-256-{2,1} nets of the DPPO2 UGV-FOA demo (train.py:26-107), 262,144 instances (config #5 per GPU)
        S, A, n = 41, 2, 1 << 18
        torch.manual_seed(0)
        mk_l = lambda i, o: torch.nn.Linear(i, o).to(dev)
        actor = [mk_l(S, 256), mk_l(256, 256), mk_l(256, A)]
        critic = [mk_l(S, 256), mk_l(256, 256), mk_l(256, 1)]
        pol = rlp.GaussianPolicy(actor, critic, [-3.0, -6.28], [3.0, 6.28], [1.0, 2.09], device=dev,
                                 actor_out_act="tanh_range")
        obs = torch.randn((S, n), generator=g, device=dev, dtype=torch.float32)
        outs = pol(obs)
        fn = lambda: pol(obs, action=outs["action"], log_prob=outs["log_prob"], value=outs["value"])
        flops = 2.0 * (2 * (S * 256 + 256 * 256) + 256 * A + 256)
        nbytes, units = (S + 2 * A + 1) * 4.0, n
    elif kind in ("policy", "policy_fp32"):
        # the reference's PPOActor_Gaussian / PPOCritic shapes for UavFntsmcParamPos (state 6, 8 gains), 1 M instances
        S, A, n = 6, 8, 1 << 20
        torch.manual_seed(0)
        mk_l = lambda i, o: torch.nn.Linear(i, o).to(dev)
        actor = [mk_l(S, 64), mk_l(64, 64), mk_l(64, 32), mk_l(32, A)]
        critic = [mk_l(S, 64), mk_l(64, 32), mk_l(32, 1)]
        pol = rlp.GaussianPolicy(actor, critic, [0.0] * A, [5.0] * A, 0.45, device=dev,
                                 precision={"policy": "umma", "policy_fp32": "fp32"}[kind])
        obs = torch.randn((S, n), generator=g, device=dev, dtype=torch.float32)
        outs = pol(obs)
        fn = lambda: pol(obs, action=outs["action"], log_prob=outs["log_prob"], value=outs["value"])
        flops = 2.0 * (S * 64 + 64 * 64 + 64 * 32 + 32 * A + S * 64 + 64 * 32 + 32)
        nbytes, units = (S + 2 * A + 1) * 4.0, n
    elif kind in ("learn", "learn_torch"):
        # one mini-batch of the PPO2 update on the reference nets (6-64-64-32-8 / 6-64-32-1) out of a 64 x 16384 rollout:
        # K-LEARN (grad + reduce + clip/Adam launches) vs the torch autograd restatement of PPO2.py:102-131
        from reinforcementlearningplatform_b200.learn import FusedPPO2Update
        from reinforcementlearningplatform_b200.ppo2 import reference_nets
        S, A, Tn, Nn, mb = 6, 8, 64, 16384, int(os.environ.get("MB", "16384"))
        torch.manual_seed(0)
        actor, critic = reference_nets(S, A, dev, init_std=0.45)
        rn = lambda *sh: torch.randn(sh, generator=g, device=dev, dtype=torch.float32)
        s, a, a_lp, adv, vt = rn(Tn, S, Nn), rn(Tn, A, Nn).abs(), -1.0 - rn(Tn, A, Nn).abs() * 0.1, rn(Tn, Nn), rn(Tn, Nn)
        if kind == "learn":
            upd = FusedPPO2Update(actor, critic, 0.45, [0.0] * A, [5.0] * A, "relu")
            state = {"j": 0}
            def fn():
                upd.grad_step(s, a, a_lp, adv, vt, (state["j"] * mb) % (Tn * Nn - mb), mb, perm_key=7)
                upd.adam_step()
                state["j"] += 1
        else:
            import math
            oa = torch.optim.Adam(actor.parameters(), lr=1e-4, eps=1e-5)
            oc = torch.optim.Adam(critic.parameters(), lr=1e-3, eps=1e-5)
            sf, af = s.permute(0, 2, 1).reshape(Tn * Nn, S), a.permute(0, 2, 1).reshape(Tn * Nn, A)
            lpf, advf, vtf = a_lp.permute(0, 2, 1).reshape(Tn * Nn, A).sum(1, keepdim=True), adv.reshape(-1, 1), vt.reshape(-1, 1)
            def fn():
                idx = torch.randint(0, Tn * Nn, (mb,), device=dev)
                mean = actor(sf[idx])
                lp = -((af[idx] - mean) ** 2) / (2 * 0.45 ** 2) - math.log(0.45) - math.log(math.sqrt(2 * math.pi))
                ratios = torch.exp(lp.sum(1, keepdim=True) - lpf[idx])
                la = (-torch.min(ratios * advf[idx], torch.clamp(ratios, 0.8, 1.2) * advf[idx])).mean()
                oa.zero_grad(); la.backward(); torch.nn.utils.clip_grad_norm_(actor.parameters(), 0.5); oa.step()
                lc = torch.nn.functional.mse_loss(vtf[idx], critic(sf[idx]))
                oc.zero_grad(); lc.backward(); torch.nn.utils.clip_grad_norm_(critic.parameters(), 0.5); oc.step()
        flops = 3 * 2.0 * (S * 64 + 64 * 64 + 64 * 32 + 32 * A + S * 64 + 64 * 32 + 32)
        nbytes, units = (S + 2 * A + 2) * 4.0, mb
    else:
        raise SystemExit(f"unknown kind {kind}")
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    per = e0.elapsed_time(e1) * 1e-3 / reps
    res = {"workload": kind, "value": units / per, "unit": "elements/s", "ms_per_step": per * 1e3,
           "algorithmic_bytes_per_element": nbytes, "achieved_gbs": nbytes * units / per / 1e9}
    if kind.startswith("policy"):
        res.update({"unit": "instances/s", "flops_per_instance": flops, "achieved_tflops_fp32": flops * units / per / 1e12})
    if kind.startswith("learn"):
        res.update({"unit": "samples/s", "flops_per_sample": flops, "achieved_tflops_fp32": flops * units / per / 1e12,
                    "mini_batch": units})
    return res


if __name__ == "__main__":
    print(json.dumps(run(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 10)))
