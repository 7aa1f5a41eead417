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
        self.out_act = {"identity": 0, "relu": 1, "tanh_range": 2}[actor_out_act]
        self.a_min = torch.as_tensor(np.asarray(a_min, dtype=np.float32), device=self.device).contiguous()
        self.a_max = torch.as_tensor(np.asarray(a_max, dtype=np.float32), device=self.device).contiguous()
        std_arr = np.asarray(std, dtype=np.float32).reshape(-1)
        self.std_vec = None
        if std_arr.size > 1:
            if self.precision != "umma":
                raise ValueError("a per-dimension std needs precision='umma'")
            self.std_vec = torch.as_tensor(std_arr, device=self.device).contiguous()
            self.std = 1.0
        else:
            self.std = float(std_arr[0])
        self._ws = None          # packed weights (precision "umma")
        self._ws_versions = None
        self.seed, self.env_index_offset, self.step = int(seed), int(env_index_offset), 0
        if self.actor:
            self.state_dim, self.action_dim = self.actor[0].in_features, self.actor[-1].out_features
        else:
            self.state_dim, self.action_dim = self.critic[0].in_features, 0

    def _mlp(self, layers, out_act) -> _lib.MLP:
        m = _lib.MLP()
        m.n_layers = len(layers)
        if not 1 <= len(layers) <= 4:
            raise ValueError("1..4 linear layers")
        m.dims[0] = layers[0].in_features
        for l, lin in enumerate(layers):
            w, b = lin.weight, lin.bias
            if not (w.is_cuda and w.dtype == torch.float32 and w.is_contiguous() and b is not None and b.is_contiguous()):
                raise _lib.B200EnvError("policy layers must be contiguous float32 CUDA nn.Linear with bias")
            m.dims[l + 1] = lin.out_features
            m.w[l], m.b[l] = w.data_ptr(), b.data_ptr()
        m.out_act = out_act
        return m

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
            am = self._mlp(self.actor, self.out_act)
            out["action"] = action if action is not None else torch.empty(A, n, dtype=torch.float32, device=dev)
            out["log_prob"] = log_prob if log_prob is not None else torch.empty(A, n, dtype=torch.float32, device=dev)
            if want_mean or mean is not None:
                out["mean"] = mean if mean is not None else torch.empty(A, n, dtype=torch.float32, device=dev)
            if noise is not None and not (noise.shape == (A, n) and noise.dtype == torch.float32 and noise.is_contiguous()):
                raise ValueError("noise must be a contiguous float32 [A, N] tensor")
        if self.critic:
            cm = self._mlp(self.critic, 0)
            out["value"] = value if value is not None else torch.empty(n, dtype=torch.float32, device=dev)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        if self.precision == "umma":
            self._forward_umma(n, am, cm, obs_soa, noise, out)
            if noise is None:
                self.step += 1
            return out
        with torch.cuda.device(dev):
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(self._lib.b200_policy_forward(
                n, None if am is None else C.byref(am), None if cm is None else C.byref(cm), p(obs_soa), p(self.a_min),
                p(self.a_max), self.std, p(noise), self.seed, self.step, self.env_index_offset, 0,  # B200_POLICY_FP32
                p(out.get("action")),
                p(out.get("log_prob")), p(out.get("mean")), p(out.get("value")), stream), "b200_policy_forward")
        if noise is None:
            self.step += 1
        return out

    def _param_versions(self):
        return tuple((t.data_ptr(), t._version) for layers in (self.actor, self.critic) if layers
                     for lin in layers for t in (lin.weight, lin.bias))

    def refresh(self, am=None, cm=None):
        """(Re)pack the weights into the tensor core's operand layout (b200_policy_pack).  Called automatically by
        ``forward`` when a parameter changed in place; call it yourself after replacing ``.data`` of a parameter."""
        am = am if am is not None or not self.actor else self._mlp(self.actor, self.out_act)
        cm = cm if cm is not None or not self.critic else self._mlp(self.critic, 0)
        ra, rc = (None if am is None else C.byref(am)), (None if cm is None else C.byref(cm))
        need = int(self._lib.b200_policy_workspace_bytes(ra, rc))
        if need == 0:
            raise _lib.B200EnvError("b200_policy_workspace_bytes: net not supported (layers <= 256 wide, heads <= 16)")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)   # torch allocations are 512 B aligned
        with torch.cuda.device(self.device):
            stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            _lib.check(self._lib.b200_policy_pack(ra, rc, C.c_void_p(self._ws.data_ptr()), self._ws.numel(), stream),
                       "b200_policy_pack")
        self._ws_versions = self._param_versions()

    def _forward_umma(self, n, am, cm, obs_soa, noise, out):
        if self._ws is None or self._ws_versions != self._param_versions():
            self.refresh(am, cm)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        dev = obs_soa.device
        with torch.cuda.device(dev):
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(self._lib.b200_policy_forward_packed(
                n, None if am is None else C.byref(am), None if cm is None else C.byref(cm),
                C.c_void_p(self._ws.data_ptr()), self._ws.numel(), p(obs_soa), p(self.a_min), p(self.a_max), self.std,
                p(self.std_vec), p(noise), self.seed, self.step, self.env_index_offset, p(out.get("action")),
                p(out.get("log_prob")), p(out.get("mean")), p(out.get("value")), stream), "b200_policy_forward_packed")

    __call__ = forward
