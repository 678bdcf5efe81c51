"""MLPPolicy without a GPU: conversion from torch, rejection of networks outside the supported family, the numpy forward
pass against the torch module, and the ctypes mirror of nig_mlp_t against include/nig_b200.h."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn as nn

import neorl_industrial as ni
from neorl_industrial import _native as N
from neorl_industrial.policies import bf16_round
from test_gpu_mlp_policy import assert_within, fp64_forward

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def actor(S=12, A=3, hidden=(256, 256), tanh=True, seed=0):
    torch.manual_seed(seed)
    layers, d = [], S
    for h in hidden:
        layers += [nn.Linear(d, h), nn.ReLU()]
        d = h
    layers.append(nn.Linear(d, A))
    if tanh:
        layers.append(nn.Tanh())
    return nn.Sequential(*layers)


@pytest.mark.parametrize("hidden,tanh", [((64,), True), ((128, 256), False), ((256, 256), True)])
def test_from_torch_and_predict(hidden, tanh):
    net = actor(24, 7, hidden, tanh)
    mean = np.linspace(-1, 1, 24).astype(np.float32)
    std = np.linspace(0.5, 2, 24).astype(np.float32)
    pol = ni.MLPPolicy.from_torch(net, obs_mean=mean, obs_std=std)
    assert pol.hidden == list(hidden) and (pol.in_dim, pol.out_dim) == (24, 7) and pol.is_trained
    assert pol.output_activation == ("tanh" if tanh else "identity")
    obs = np.random.default_rng(1).normal(0, 2, (500, 24)).astype(np.float32)
    got = pol.predict(obs, deterministic=True)
    with torch.no_grad():
        want = net(torch.from_numpy(pol._input(obs))).numpy().astype(np.float64)
    # the derived bound of the device tests: bf16 rounding of the bf16 network's layer inputs, widened by the rounding of
    # weights and inputs that the torch module's own fp32 forward does not do
    _, bound = fp64_forward(pol, obs)
    _, wide = fp64_forward(pol, obs, weight_rounding=True)
    assert_within(got, want, wide + bound, "predict vs the torch module")
    assert got.shape == (500, 7) and pol.predict(obs[0]).shape == (7,)


def test_policy_is_a_snapshot_of_the_module():
    """MLPPolicy copies the weights: training the module further changes neither the policy nor its predictions."""
    net = actor(hidden=(64, 64), tanh=False)
    pol = ni.MLPPolicy.from_torch(net, obs_mean=np.zeros(12, np.float32), obs_std=np.ones(12, np.float32))
    obs = np.random.default_rng(2).normal(0, 1, (50, 12)).astype(np.float32)
    before, w0 = pol.predict(obs), pol.weights[0].copy()
    with torch.no_grad():
        for p in net.parameters():
            p.add_(1.0)
    assert np.array_equal(pol.weights[0], w0) and np.array_equal(pol.predict(obs), before)
    w = np.ones((64, 12), np.float32)
    pol2 = ni.MLPPolicy([w, np.ones((3, 64), np.float32)])
    w[:] = 5.0
    assert (pol2.weights[0] == 1.0).all()


def test_bf16_round_is_nearest_even():
    x = np.array([1.0, 1.00390625, 1.01171875, 1.0078125 + 2 ** -9, -3.0e38, 3.4e38, np.inf, np.nan, -0.0], np.float32)
    want = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    got = bf16_round(x)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))


@pytest.mark.parametrize("module,match", [
    (nn.Sequential(nn.Linear(12, 64), nn.Tanh(), nn.Linear(64, 3)), "position 1"),                      # other activation
    (nn.Sequential(nn.Linear(12, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU(),
                   nn.Linear(64, 3)), "hidden layers"),                                                  # 3 hidden layers
    (nn.Sequential(nn.Linear(12, 96), nn.ReLU(), nn.Linear(96, 3)), "hidden width"),                     # width
    (nn.Sequential(nn.Linear(12, 64), nn.ReLU()), "end with a Linear"),
    (nn.Linear(12, 3), "nn.Sequential"),
    (nn.Sequential(nn.Linear(12, 64), nn.ReLU(), nn.Linear(64, 3), nn.Sigmoid()), "position 3"),
])
def test_from_torch_rejects_unsupported(module, match):
    with pytest.raises(ValueError, match=match):
        ni.MLPPolicy.from_torch(module)


def test_rejects_other_dtypes_and_shapes():
    with pytest.raises(ValueError, match="not supported"):
        ni.MLPPolicy.from_torch(actor(hidden=(64,)).half())
    w = [np.zeros((64, 12), np.float16), np.zeros((3, 64), np.float32)]
    with pytest.raises(ValueError, match="not supported"):
        ni.MLPPolicy(w)
    with pytest.raises(ValueError, match="takes"):
        ni.MLPPolicy([np.zeros((64, 12), np.float32), np.zeros((3, 128), np.float32)])
    with pytest.raises(ValueError, match="bias"):
        ni.MLPPolicy([np.zeros((64, 12), np.float32), np.zeros((3, 64), np.float32)], [np.zeros(63, np.float32), None])
    with pytest.raises(ValueError, match="output activation"):
        ni.MLPPolicy([np.zeros((64, 12), np.float32), np.zeros((3, 64), np.float32)], output_activation="sigmoid")
    pol = ni.MLPPolicy.from_torch(actor(hidden=(64,)).to(torch.bfloat16))             # bf16 weights are exact in fp32
    assert pol.weights[0].dtype == np.float32


def test_nan_propagates_like_torch():
    net = actor(hidden=(64, 64), tanh=False)
    pol = ni.MLPPolicy.from_torch(net)
    obs = np.zeros((3, 12), np.float32)
    obs[1, 4] = np.nan
    got = pol.predict(obs)
    with torch.no_grad():
        want = net(torch.from_numpy(obs)).numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got[1]).all() and not np.isnan(got[[0, 2]]).any()


def test_mlp_struct_matches_header(tmp_path):
    """ctypes mirror of nig_mlp_t == what a C compiler makes of include/nig_b200.h, and the new symbols are bound."""
    src = tmp_path / "mlp.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "nig_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu %d %d\\n", sizeof(nig_mlp_t), offsetof(nig_mlp_t, hidden),'
                   ' offsetof(nig_mlp_t, out_dim), offsetof(nig_mlp_t, weight), offsetof(nig_mlp_t, bias),'
                   ' offsetof(nig_mlp_t, obs_inv_std), NIG_POLICY_MLP, NIG_ABI_VERSION); return 0;}\n')
    exe = tmp_path / "mlp"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(N.Mlp), N.Mlp.hidden.offset, N.Mlp.out_dim.offset, N.Mlp.weight.offset, N.Mlp.bias.offset,
            N.Mlp.obs_inv_std.offset, N.POLICY_MLP, N.ABI_VERSION]
    assert got == want, (got, want)
    m = ni.MLPPolicy.from_torch(actor(hidden=(128, 64))).native_struct()
    assert (m.n_hidden, list(m.hidden), m.output_activation, m.in_dim, m.out_dim) == (2, [128, 64], N.MLP_OUT_TANH, 12, 3)
    assert m.weight[2] and m.bias[0] and m.obs_mean is None
    assert "nig_set_mlp_policy" in N.SYMBOLS and "nig_selftest_mlp" in N.SYMBOLS
