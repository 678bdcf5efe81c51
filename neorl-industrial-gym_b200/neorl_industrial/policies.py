"""Learned policies that run inside the fused rollout kernel.

``MLPPolicy`` is the deterministic actor of an offline-RL agent (TD3+BC, IQL, CQL: one or two ReLU hidden layers of 64, 128
or 256 units, tanh or identity output). ``env.rollout(T, mlp)``, ``rollouts.evaluate_policy_device(env, T, policy=mlp)`` and
``NativeEnv.rollout_steps_device(..., POLICY_MLP)`` after ``NativeEnv.set_mlp_policy(mlp)`` evaluate it on the tensor cores
inside the K-step rollout (NIG_POLICY_MLP, include/nig_b200.h). ``predict`` is the same network in numpy with the same bf16
rounding, so the object also works as an agent for ``evaluate_with_safety`` / ``rollouts.evaluate_agent_batched``.

Numeric contract (also in include/nig_b200.h): weights and every layer's input are rounded to bf16 (nearest even), products
are summed in fp32 (on the device in the tensor core's order, here in fp64 and rounded once), biases and activations are
applied in fp32. Device actions therefore match ``predict`` to a tolerance, not bit for bit.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

HIDDEN_WIDTHS = (64, 128, 256)
OUTPUT_ACTIVATIONS = ("tanh", "identity")


def bf16_round(x) -> np.ndarray:
    """float32 -> nearest-even bfloat16, returned as float32 (NaN stays NaN, overflow goes to inf)."""
    x = np.ascontiguousarray(x, np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    out = (r & 0xFFFFFFFF).astype(np.uint32).view(np.float32)
    return np.where(np.isnan(x), x, out).astype(np.float32)


def _as_f32(x, what: str) -> np.ndarray:
    """A float32 COPY of an fp32 / fp64 / bf16 array or tensor (never a view of the caller's memory: a CPU fp32 torch
    parameter's .numpy() shares it); fp16, fp8 and integer weights are rejected."""
    if hasattr(x, "detach"):                         # torch tensor
        import torch
        if x.dtype not in (torch.float32, torch.float64, torch.bfloat16):
            raise ValueError(f"{what}: dtype {x.dtype} is not supported (float32, float64 or bfloat16)")
        x = x.detach().to("cpu", torch.float32).numpy()
    a = np.asarray(x)
    if a.dtype not in (np.float32, np.float64):
        raise ValueError(f"{what}: dtype {a.dtype} is not supported (float32 or float64)")
    return np.array(a, np.float32, order="C", copy=True)


class MLPPolicy:
    """Deterministic MLP actor: ``a = out_act(W_L relu(... relu(W_1 x + b_1) ...) + b_L)``, ``x = (s - obs_mean) / obs_std``.

    ``weights`` are ``[out, in]`` matrices in ``nn.Linear`` order (one or two hidden layers, then the output layer),
    ``biases`` the matching vectors (None = zeros). The object is a snapshot: it copies every array it is given, so a module
    that keeps training after ``from_torch`` does not change it, and ``NativeEnv.use_mlp_policy`` / ``env.rollout`` /
    ``evaluate_policy_device`` upload it once. To evaluate newer weights, build a new ``MLPPolicy``."""

    is_trained = True

    def __init__(self, weights: Sequence, biases: Optional[Sequence] = None, output_activation: str = "tanh",
                 obs_mean=None, obs_std=None):
        ws = [_as_f32(w, f"weight {k}") for k, w in enumerate(weights)]
        if len(ws) not in (2, 3):
            raise ValueError(f"{len(ws) - 1} hidden layers: 1 or 2 are supported")
        if any(w.ndim != 2 for w in ws):
            raise ValueError("every weight must be a 2-D [out, in] matrix")
        for k in range(1, len(ws)):
            if ws[k].shape[1] != ws[k - 1].shape[0]:
                raise ValueError(f"layer {k} takes {ws[k].shape[1]} inputs, layer {k - 1} gives {ws[k - 1].shape[0]}")
        for w in ws[:-1]:
            if w.shape[0] not in HIDDEN_WIDTHS:
                raise ValueError(f"hidden width {w.shape[0]} is not supported ({HIDDEN_WIDTHS})")
        if biases is None:
            biases = [None] * len(ws)
        if len(biases) != len(ws):
            raise ValueError("one bias per layer (or None)")
        bs = []
        for k, (w, b) in enumerate(zip(ws, biases)):
            b = np.zeros(w.shape[0], np.float32) if b is None else _as_f32(b, f"bias {k}")
            if b.shape != (w.shape[0],):
                raise ValueError(f"bias {k} has shape {b.shape}, expected ({w.shape[0]},)")
            bs.append(b)
        if output_activation not in OUTPUT_ACTIVATIONS:
            raise ValueError(f"output activation {output_activation!r} is not supported {OUTPUT_ACTIVATIONS}")
        self.weights, self.biases, self.output_activation = ws, bs, output_activation
        self.in_dim, self.out_dim = ws[0].shape[1], ws[-1].shape[0]
        self.hidden = [w.shape[0] for w in ws[:-1]]
        self.obs_mean = None if obs_mean is None else _as_f32(obs_mean, "obs_mean").reshape(self.in_dim)
        self.obs_inv_std = None
        if obs_std is not None:
            std = _as_f32(obs_std, "obs_std").reshape(self.in_dim)
            self.obs_inv_std = (np.float32(1.0) / std).astype(np.float32)

    @classmethod
    def from_torch(cls, module, obs_mean=None, obs_std=None) -> "MLPPolicy":
        """From an ``nn.Sequential`` of ``Linear`` / ``ReLU`` layers, optionally ending in ``Tanh``; anything else raises."""
        import torch.nn as nn
        if not isinstance(module, nn.Sequential):
            raise ValueError(f"expected an nn.Sequential of Linear / ReLU (/ Tanh), got {type(module).__name__}")
        layers = list(module)
        out_act = "identity"
        if layers and isinstance(layers[-1], nn.Tanh):
            out_act, layers = "tanh", layers[:-1]
        ws, bs = [], []
        for k, layer in enumerate(layers):
            want_linear = k % 2 == 0
            if want_linear and type(layer) is nn.Linear:
                ws.append(layer.weight)
                bs.append(layer.bias)
            elif not want_linear and type(layer) is nn.ReLU:
                continue
            else:
                raise ValueError(f"unsupported module at position {k}: {layer!r} (expected "
                                 f"{'Linear' if want_linear else 'ReLU'})")
        if not ws or len(layers) % 2 == 0:
            raise ValueError("the network must end with a Linear layer (optionally followed by Tanh)")
        return cls(ws, bs, out_act, obs_mean=obs_mean, obs_std=obs_std)

    def _input(self, obs: np.ndarray) -> np.ndarray:
        x = np.asarray(obs, np.float32)
        if self.obs_mean is not None:
            x = (x - self.obs_mean).astype(np.float32)
        if self.obs_inv_std is not None:
            x = (x * self.obs_inv_std).astype(np.float32)
        return x

    def predict(self, obs, deterministic: bool = True) -> np.ndarray:
        """Actions [..., A] (before the env's clip to [-1, 1]) with the device's roundings; products summed in fp64."""
        x = self._input(obs)
        shape = x.shape[:-1]
        x = x.reshape(-1, self.in_dim)
        n_layers = len(self.weights)
        with np.errstate(invalid="ignore", over="ignore"):
            for k, (w, b) in enumerate(zip(self.weights, self.biases)):
                y = (bf16_round(x).astype(np.float64) @ bf16_round(w).astype(np.float64).T).astype(np.float32)
                y = (y + b).astype(np.float32)
                if k < n_layers - 1:
                    y = np.where(y < 0, np.float32(0), y)           # ReLU; NaN stays NaN like torch.relu
                x = y
            if self.output_activation == "tanh":
                x = np.tanh(x).astype(np.float32)
        return x.reshape(shape + (self.out_dim,))

    def native_struct(self):
        """The nig_mlp_t of this network (keeps the arrays it points to alive on the returned object)."""
        from . import _native as N
        m = N.Mlp()
        m.n_hidden = len(self.hidden)
        for k, h in enumerate(self.hidden):
            m.hidden[k] = h
        m.output_activation = N.MLP_OUT_TANH if self.output_activation == "tanh" else N.MLP_OUT_IDENTITY
        m.in_dim, m.out_dim = self.in_dim, self.out_dim
        for k, (w, b) in enumerate(zip(self.weights, self.biases)):
            m.weight[k], m.bias[k] = w.ctypes.data, b.ctypes.data
        m.obs_mean = None if self.obs_mean is None else self.obs_mean.ctypes.data
        m.obs_inv_std = None if self.obs_inv_std is None else self.obs_inv_std.ctypes.data
        m._keep = (self.weights, self.biases, self.obs_mean, self.obs_inv_std)
        return m
