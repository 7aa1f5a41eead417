"""Batched Gaussian actor / critic forward on device (kernel K-POLICY, csrc/policy_umma.cu; policy.cu).

``GaussianPolicy`` runs ``Proximal_Policy_Optimization2.choose_action`` (algorithm/policy_base/
Proximal_Policy_Optimization2.py:69-76) for all N instances at once on the engine's own buffers: the policy-state
buffer of a ``VecEnv`` built with ``io_dtype=torch.float32`` goes in (``[state_dim, N]``), the action buffer the step
kernel reads comes out (``[action_dim, N]``), together with the per-dimension log-probabilities and, optionally, the
critic value -- one launch, no host round trip.  The weights are read straight from the ``torch.nn.Linear`` parameters
of the caller's actor / critic modules (the reference's ``PPOActor_Gaussian`` / ``PPOCritic``, utils/classes.py:529-615,
the 256-wide copies of demonstration/DPPO2/DPPO2-4-UGVForwardObstacleAvoidance/train.py:26-107, or any tanh MLP of up to
4 layers).  The default kernel (tcgen05 / TMEM, ``precision="umma"``) multiplies from a packed copy of the weights in the
tensor core's operand layout; the copy is refreshed automatically whenever a parameter tensor has been modified in
place (``Tensor._version``), i.e. after every optimizer step, so callers never see stale weights.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib


def linear_layers(module) -> list:
    """The ``nn.Linear`` layers of a reference-style net in forward order (fc1, fc2, [fc3], [mean_layer])."""
    names = [n for n in ("fc1", "fc2", "fc3", "fc4", "mean_layer") if hasattr(module, n)]
    if names:
        return [getattr(module, n) for n in names]
    return [m for m in module.modules() if isinstance(m, torch.nn.Linear)]


def gaussian_std(std, device=None, out: Optional[torch.Tensor] = None):
    """``(std, std_vec)`` as K-POLICY and K-LEARN take them: a scalar std is ``(float, None)``; one value per action
    dimension is ``(1.0, float32 tensor on device)`` -- no kernel reads the scalar then.  ``out``: the ``std_vec`` of an
    existing head, overwritten in place instead of allocating a new one."""
    arr = np.asarray(std.detach().cpu() if torch.is_tensor(std) else std, dtype=np.float32).reshape(-1)
    if arr.size == 1:
        return float(arr[0]), None
    if out is None:
        return 1.0, torch.as_tensor(arr, device=device).contiguous()
    out.copy_(torch.as_tensor(arr, device=out.device))
    return 1.0, out


def gaussian_head(std, a_min, a_max, out_act: str, device):
    """The Gaussian action head of an actor, as K-POLICY and K-LEARN read it: ``(out_act code, a_min, a_max, std,
    std_vec)`` with the action clamp as float32 device tensors and ``std, std_vec`` from :func:`gaussian_std`."""
    bound = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float32), device=device).contiguous()
    return (_lib.OUT_ACT[out_act], bound(a_min), bound(a_max), *gaussian_std(std, device))


class GaussianPolicy:
    def __init__(self, actor_layers: Optional[Sequence], critic_layers: Optional[Sequence], a_min, a_max, std: float,
                 device="cuda", seed: int = 0, env_index_offset: int = 0, actor_out_act: str = "relu",
                 precision: str = "umma"):
        """``actor_layers`` / ``critic_layers``: sequences of ``torch.nn.Linear`` (CUDA, float32) or modules accepted by
        :func:`linear_layers`.  ``a_min, a_max``: action clamp (``actor.a_min / a_max``); ``std``: ``actor.std``, a float
        or one value per action dimension (the DPPO2 demos' ``init_std`` vector; "umma" only).
        ``actor_out_act``: "relu" (PPOActor_Gaussian.forward, utils/classes.py:563-569), "identity", or "tanh_range"
        (``tanh(mean_layer) * gain + off`` of the DPPO2 demo nets).
        ``precision``: "umma" (tcgen05 tensor cores + TMEM, 3xTF32 split, layers up to 256 wide; default) or "fp32"
        (FMA pipe, sums in k order, layers <= 64: the reference the tests compare "umma" with)."""
        if precision not in ("umma", "fp32"):
            raise ValueError(f"precision must be 'umma' or 'fp32', not {precision!r}")
        self.precision = precision
        self._lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: device must be a CUDA device")
        as_list = lambda x: None if x is None else (list(x) if isinstance(x, (list, tuple)) else linear_layers(x))
        self.actor, self.critic = as_list(actor_layers), as_list(critic_layers)
        self.out_act, self.a_min, self.a_max, self.std, self.std_vec = gaussian_head(std, a_min, a_max, actor_out_act,
                                                                                     self.device)
        if self.std_vec is not None and self.precision != "umma":
            raise ValueError("a per-dimension std needs precision='umma'")
        self._ws = None          # packed weights (precision "umma")
        self._ws_versions = None
        self.seed, self.env_index_offset, self.step = int(seed), int(env_index_offset), 0
        if self.actor:
            self.state_dim, self.action_dim = self.actor[0].in_features, self.actor[-1].out_features
        else:
            self.state_dim, self.action_dim = self.critic[0].in_features, 0

    def forward(self, obs_soa: torch.Tensor, noise: Optional[torch.Tensor] = None, *, action: torch.Tensor = None,
                log_prob: torch.Tensor = None, mean: torch.Tensor = None, value: torch.Tensor = None,
                want_mean: bool = False):
        """``obs_soa [state_dim, N]`` float32 contiguous -> dict(action [A, N], log_prob [A, N], mean?, value [N]?).
        ``noise [A, N]``: inject N(0, 1) draws (parity tests); default: in-kernel Philox draw for this ``step``.
        Output tensors may be passed in (rows of a rollout buffer) to be written in place."""
        if not (obs_soa.is_cuda and obs_soa.dtype == torch.float32 and obs_soa.is_contiguous()
                and obs_soa.dim() == 2 and obs_soa.shape[0] == self.state_dim):
            raise ValueError(f"obs must be a contiguous float32 CUDA [{self.state_dim}, N] tensor")
        n, A, dev = obs_soa.shape[1], self.action_dim, obs_soa.device
        out = {}
        am = cm = None
        if self.actor:
            am = _lib.mlp(self.actor, self.out_act)
            out["action"] = action if action is not None else torch.empty(A, n, dtype=torch.float32, device=dev)
            out["log_prob"] = log_prob if log_prob is not None else torch.empty(A, n, dtype=torch.float32, device=dev)
            if want_mean or mean is not None:
                out["mean"] = mean if mean is not None else torch.empty(A, n, dtype=torch.float32, device=dev)
            if noise is not None and not (noise.shape == (A, n) and noise.dtype == torch.float32 and noise.is_contiguous()):
                raise ValueError("noise must be a contiguous float32 [A, N] tensor")
        if self.critic:
            cm = _lib.mlp(self.critic, 0)
            out["value"] = value if value is not None else torch.empty(n, dtype=torch.float32, device=dev)
        if self.precision == "umma":
            self._forward_umma(n, am, cm, obs_soa, noise, out)
            if noise is None:
                self.step += 1
            return out
        p = _lib.ptr
        with torch.cuda.device(dev):
            _lib.check(self._lib.b200_policy_forward(
                n, None if am is None else C.byref(am), None if cm is None else C.byref(cm), p(obs_soa), p(self.a_min),
                p(self.a_max), self.std, p(noise), self.seed, self.step, self.env_index_offset, 0,  # B200_POLICY_FP32
                p(out.get("action")),
                p(out.get("log_prob")), p(out.get("mean")), p(out.get("value")), _lib.stream(dev)), "b200_policy_forward")
        if noise is None:
            self.step += 1
        return out

    def _param_versions(self):
        return tuple((t.data_ptr(), t._version) for layers in (self.actor, self.critic) if layers
                     for lin in layers for t in (lin.weight, lin.bias))

    def refresh(self, am=None, cm=None):
        """(Re)pack the weights into the tensor core's operand layout (b200_policy_pack).  Called automatically by
        ``forward`` when a parameter changed in place; call it yourself after replacing ``.data`` of a parameter."""
        am = am if am is not None or not self.actor else _lib.mlp(self.actor, self.out_act)
        cm = cm if cm is not None or not self.critic else _lib.mlp(self.critic, 0)
        ra, rc = (None if am is None else C.byref(am)), (None if cm is None else C.byref(cm))
        need = int(self._lib.b200_policy_workspace_bytes(ra, rc))
        if need == 0:
            raise _lib.B200EnvError("b200_policy_workspace_bytes: net not supported (layers <= 256 wide, heads <= 16)")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)   # torch allocations are 512 B aligned
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_policy_pack(ra, rc, _lib.ptr(self._ws), self._ws.numel(), _lib.stream(self.device)),
                       "b200_policy_pack")
        self._ws_versions = self._param_versions()

    def _forward_umma(self, n, am, cm, obs_soa, noise, out):
        if self._ws is None or self._ws_versions != self._param_versions():
            self.refresh(am, cm)
        p = _lib.ptr
        dev = obs_soa.device
        with torch.cuda.device(dev):
            _lib.check(self._lib.b200_policy_forward_packed(
                n, None if am is None else C.byref(am), None if cm is None else C.byref(cm),
                p(self._ws), self._ws.numel(), p(obs_soa), p(self.a_min), p(self.a_max), self.std,
                p(self.std_vec), p(noise), self.seed, self.step, self.env_index_offset, p(out.get("action")),
                p(out.get("log_prob")), p(out.get("mean")), p(out.get("value")), _lib.stream(dev)),
                "b200_policy_forward_packed")

    __call__ = forward
