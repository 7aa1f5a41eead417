"""Small invocations of the kernels that share data across threads (shared memory / warp votes / TMEM), for
compute-sanitizer:  compute-sanitizer --tool racecheck|memcheck python tools/sanitize_targets.py [ugvo norm policy_umma]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import reinforcementlearningplatform_b200 as rlp  # noqa: E402

which = sys.argv[1:] or ["ugvo", "norm", "policy_umma"]
dev = "cuda"
if "ugvo" in which:  # block-cooperative ray casting + warp-vote rejection sampler (auto-reset list)
    env = rlp.UGVForwardObstacleAvoidance(variant="dppo2", n_envs=777, device=dev, auto_reset=True, seed=3)
    env.reset(True)
    ar = torch.as_tensor(np.asarray(env.action_range), device=dev)
    for t in range(4):
        a = ar[:, :1] + (ar[:, 1:] - ar[:, :1]) * torch.rand(2, 777, device=dev, dtype=torch.float64)
        env.step_soa(a.contiguous())
    torch.cuda.synchronize()
    print("ugvo ok", float(env.reward.sum()))
if "norm" in which:  # last-block reduction
    nz = rlp.Normalization(6, device=dev, sync=False)
    x = torch.randn(6, 50000, device=dev)
    y = torch.empty_like(x)
    for _ in range(3):
        nz.normalize_soa(x, out=y)
    torch.cuda.synchronize()
    print("norm ok", float(y.std()))
mk = lambda i, o: torch.nn.Linear(i, o).to(dev)
if "policy_umma" in which:
    actor = [mk(6, 64), mk(64, 64), mk(64, 32), mk(32, 8)]
    critic = [mk(6, 64), mk(64, 32), mk(32, 1)]
    pol = rlp.GaussianPolicy(actor, critic, [0.0] * 8, [5.0] * 8, 0.45)
    out = pol(torch.randn(6, 3000, device=dev))
    torch.cuda.synchronize()
    print("policy umma ok", float(out["value"].mean()))
    a2, c2 = [mk(41, 256), mk(256, 256), mk(256, 2)], [mk(41, 256), mk(256, 256), mk(256, 1)]
    pol = rlp.GaussianPolicy(a2, c2, [-3.0, -6.28], [3.0, 6.28], [1.0, 2.09], actor_out_act="tanh_range")
    out = pol(torch.randn(41, 700, device=dev))
    torch.cuda.synchronize()
    print("policy umma wide ok", float(out["value"].mean()))
