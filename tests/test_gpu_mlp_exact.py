"""NIG_POLICY_MLP on exactly representable networks: the tensor-core forward pass pinned bit for bit.

Every weight matrix is integers times a power of two, the layer-1 inputs are integers times 2^-4 (also after the
normalisation: a grid-valued mean and a power-of-two inverse std) and the hidden biases lie on their layer's product grid.
Every product of a layer is then a multiple of g = grid(bf16 inputs) * grid(bf16 weights), and while sum |w x| < 2^22 g for
every row, every partial sum in any order is an fp32-representable multiple of g: the tensor core's result does not depend
on its summation order and equals the exact sum. What is left to round is what the numeric contract of include/nig_b200.h
specifies: the bf16 nearest-even rounding of every layer's input (hidden pre-activations of hundreds to thousands of grid
units, so exact ties are frequent and truncation or round-half-away changes almost every row), the fp32 bias add (the
output bias is an arbitrary fp32 value), ReLU and tanhf. So identity outputs are compared bit for bit and tanh outputs to
tanhf's documented 2 ulp (tanh.approx.f32 is about 2^-11 relative, thousands of ulp).

The reference asserts the exactness condition for every layer before anything is compared, so a generator change that
leaves the exact regime fails instead of weakening the test (test_generator_is_exact checks it on the CPU for every env and
width pair, against fp32 sums in random orders).

Cases: every env x every width pair (one or two hidden layers of 64, 128, 256) x {identity, tanh} x {with, without
normalisation}; 128-row tile edges and a NaN row that padding lanes shadow; full tensor-memory occupancy per TMEM class,
every row bit for bit; the NULL bias / normalisation pointers of the C ABI; two handles of different TMEM widths running
concurrently on two streams."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from neorl_industrial.policies import MLPPolicy, bf16_round
from util import KINDS, assert_bits_equal, ulp_diff

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

S_A = {"reactor": (12, 3), "grid": (32, 8), "robot": (24, 7)}
WIDTHS = [(h,) for h in (64, 128, 256)] + [(a, b) for a in (64, 128, 256) for b in (64, 128, 256)]
EXACT_LIMIT = 2.0 ** 22          # sum |w x| / g below this: every partial sum is an fp32 multiple of g, in any order
TANH_ULP = 2                     # CUDA's documented maximum error of tanhf


def wid(hidden):
    return "x".join(str(h) for h in hidden)


def lsb_exponent(a):
    """log2 of the largest power of two that divides every finite non-zero element of the float32 array a."""
    a = np.ascontiguousarray(a, np.float32)
    a = a[np.isfinite(a) & (a != 0)]
    if not a.size:
        return 0
    u = a.view(np.uint32).astype(np.int64)
    e = (u >> 23) & 0xFF
    m = (u & 0x7FFFFF) | np.where(e > 0, 0x800000, 0)
    return int((np.maximum(e, 1) - 150 + np.log2(m & -m).astype(np.int64)).min())


def _forward(x, ws, bs, n_hidden, hidden_round=bf16_round, order_rng=None):
    """Layers (ws, bs) on fp32 inputs x: bf16(x) . bf16(W)^T, asserted exact, summed in fp64 (or, with order_rng, in fp32 in a
    random order of K); then the fp32 bias add; layers below n_hidden add ReLU and round the next input with hidden_round.
    Rows with a non-finite input are not checked for exactness (NaN propagates)."""
    for k, (w, b) in enumerate(zip(ws, bs)):
        xb, wb = bf16_round(x), bf16_round(w)
        fin = np.isfinite(xb).all(1)
        g = 2.0 ** (lsb_exponent(xb[fin]) + lsb_exponent(wb))
        mag = np.abs(xb[fin]).astype(np.float64) @ np.abs(wb).astype(np.float64).T
        assert (mag < EXACT_LIMIT * g).all(), \
            f"layer {k} leaves the exact regime: sum |w x| reaches 2^{np.log2(mag.max() / g):.2f} g"
        if order_rng is None:
            with np.errstate(invalid="ignore"):
                z = (xb.astype(np.float64) @ wb.astype(np.float64).T).astype(np.float32)
        else:
            z = np.zeros((xb.shape[0], wb.shape[0]), np.float32)
            with np.errstate(invalid="ignore"):
                for j in order_rng.permutation(xb.shape[1]):
                    z = (z + xb[:, j:j + 1] * wb[None, :, j]).astype(np.float32)
        y = (z + b).astype(np.float32)
        if k < n_hidden:
            y = np.where(y < 0, np.float32(0), y)
            x = hidden_round(y)
        else:
            x = y
    return x


def exact_forward(pol, obs, **kw):
    """The network's output layer before its activation (fp32), exact for the networks of exact_mlp."""
    return _forward(pol._input(obs), pol.weights, pol.biases, len(pol.hidden), **kw)


def exact_mlp(rng, S, A, hidden, n, norm=False):
    """(weights, biases, obs, obs_mean, obs_std) of an exactly representable network and n observations of it.

    x0 = m 2^-4 with |m| <= 64, or with probability 1/8 256 <= |m| < 1024 (9 or 10 significant bits: bf16(x0) rounds, half
    the 9-bit values are ties). Layer 1: integers in [-8, 8] times 2^-3; later hidden layers: integers in [-1, 1] times 2^-3
    with about 16 non-zero inputs per unit; hidden biases: integers in [-128, 512) on the layer's product grid. The output
    weights are integers in [-1, 1] scaled by the power of two that puts the 99th percentile of |W3 x| at about 2; the output
    bias is uniform in [-1, 1] (fp32). norm: obs = x0 std + mean with std a power of two per column and mean a multiple of
    2^-6, so that (obs - mean) / std == x0 exactly."""
    m = rng.integers(-64, 65, (n, S))
    big = rng.random((n, S)) < 0.125
    m = np.where(big, rng.choice([-1, 1], (n, S)) * rng.integers(256, 1024, (n, S)), m)
    x0 = (m * 2.0 ** -4).astype(np.float32)
    dims = [S, *hidden, A]
    ws, bs, e_x = [], [], -4
    for k in range(len(hidden)):
        shape = (dims[k + 1], dims[k])
        w = rng.integers(-8, 9, shape) if k == 0 else rng.integers(-1, 2, shape) * (rng.random(shape) < 16.0 / dims[k])
        ws.append((w * 2.0 ** -3).astype(np.float32))
        e_x -= 3
        bs.append((rng.integers(-128, 512, dims[k + 1]) * 2.0 ** e_x).astype(np.float32))
    w = rng.integers(-1, 2, (A, dims[-2])).astype(np.float64)
    z = _forward(x0, ws, bs, len(hidden)).astype(np.float64) @ w.T
    ws.append((w * 2.0 ** -np.round(np.log2(np.percentile(np.abs(z), 99) / 2))).astype(np.float32))
    bs.append(rng.uniform(-1, 1, A).astype(np.float32))
    if not norm:
        return ws, bs, x0, None, None
    std = (2.0 ** rng.integers(-2, 4, S)).astype(np.float32)
    mean = (rng.integers(-640, 641, S) * 2.0 ** -6).astype(np.float32)
    obs = (x0 * std + mean).astype(np.float32)
    assert np.array_equal(((obs - mean) * (np.float32(1) / std)).astype(np.float32), x0)
    return ws, bs, obs, mean, std


def policy(net, activation):
    ws, bs, _, mean, std = net
    return MLPPolicy(ws, bs, activation, obs_mean=mean, obs_std=std)


def seeded(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def truncate_bf16(x):
    x = np.ascontiguousarray(x, np.float32)
    return (x.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32)


def round_half_away_bf16(x):
    x = np.ascontiguousarray(x, np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    return ((((u + 0x8000) >> 16) << 16) & 0xFFFFFFFF).astype(np.uint32).view(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# the generator, without a GPU
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_generator_is_exact(name):
    """For every width pair: the networks satisfy the exactness condition (asserted inside _forward), an fp32 forward pass
    summing in random orders gives the same bits as the reference, outputs exceed +-1 without saturating tanh, and the
    hidden rounding is decisive: truncating to bf16 changes at least 90 % of the rows, rounding half away from zero 30 %."""
    S, A = S_A[name]
    for hidden in WIDTHS:
        for norm in (False, True):
            rng = seeded(name, hidden, norm)
            net = exact_mlp(rng, S, A, hidden, 512, norm)
            pol, obs = policy(net, "identity"), net[2]
            ref = exact_forward(pol, obs)
            for _ in range(2):
                assert_bits_equal(exact_forward(pol, obs, order_rng=rng), ref, f"{name} {hidden}: random summation order")
            assert 1.0 < np.abs(ref).max() < 8.0 and np.mean(np.abs(ref) > 1) > 0.05, (name, hidden, np.abs(ref).max())
            for fn, share in ((truncate_bf16, 0.9), (round_half_away_bf16, 0.3)):
                changed = (exact_forward(pol, obs, hidden_round=fn) != ref).any(1).mean()
                assert changed >= share, (name, hidden, fn.__name__, changed)


# ---------------------------------------------------------------------------------------------------------------------
# the device
@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    return ni, N, torch


def check_device(env, pol, obs, what):
    """nig_selftest_mlp of pol == the exact reference: bit for bit (identity) or within TANH_ULP of tanh (tanh)."""
    env.set_mlp_policy(pol)
    dev = env.selftest_mlp(obs)
    y = exact_forward(pol, obs)
    if pol.output_activation == "identity":
        assert_bits_equal(dev, y, what)
    else:
        want = np.tanh(y.astype(np.float64)).astype(np.float32)
        assert np.array_equal(np.isnan(dev), np.isnan(want)), f"{what}: NaN pattern"
        ok = ~np.isnan(want)
        d = ulp_diff(dev[ok], want[ok])
        assert d.max() <= TANH_ULP, f"{what}: {np.count_nonzero(d > TANH_ULP)} outputs more than {TANH_ULP} ulp from " \
                                    f"tanh (worst {d.max()} ulp)"
    return dev


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", WIDTHS, ids=wid)
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_exact_network(mods, name, hidden):
    """Every env's S / A, every width pair, identity and tanh, without and with normalisation: 1,000 rows (7 full tiles and
    a partial one)."""
    ni, N, torch = mods
    S, A = S_A[name]
    env = ni.NativeEnv(KINDS[name], 1, device=0, seed=1)
    for norm in (False, True):
        net = exact_mlp(seeded(name, hidden, norm), S, A, hidden, 1_000, norm)
        for act in ("identity", "tanh"):
            check_device(env, policy(net, act), net[2], f"{name} {wid(hidden)} {act} norm={norm}")
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_tile_edges(mods, name):
    """n = 1, 127, 128, 129, 255, 257 rows, and 129 rows with row 0 all NaN: padding lanes shadow row 0, so only row 0 may
    be NaN (and every other row keeps its bits)."""
    ni, N, torch = mods
    S, A = S_A[name]
    hidden = {"reactor": (256,), "grid": (64, 256), "robot": (256, 128)}[name]
    env = ni.NativeEnv(KINDS[name], 1, device=0, seed=1)
    net = exact_mlp(seeded(name, "edges"), S, A, hidden, 257, norm=True)
    for act in ("identity", "tanh"):
        pol = policy(net, act)
        for n in (1, 127, 128, 129, 255, 257):
            check_device(env, pol, net[2][:n], f"{name} {act} n={n}")
        obs = net[2][:129].copy()
        obs[0] = np.nan
        dev = check_device(env, pol, obs, f"{name} {act} NaN row 0")
        assert np.isnan(dev[0]).all() and not np.isnan(dev[1:]).any()
    env.close()


def full_occupancy_rows(torch, hidden):
    """Two full waves of CTAs at the most CTAs per SM that the tensor memory serves, plus a partial tile:
    2 * SMs * (512 / columns) * 128 + 77 (151,629 / 75,853 / 37,965 rows at widths 64 / 128 / 256 on 148 SMs)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return 2 * sms * (512 // (2 * max(hidden))) * 128 + 77


@pytest.mark.gpu
@pytest.mark.parametrize("name,hidden", [("reactor", (64, 64)), ("robot", (128, 128)), ("grid", (256, 256))],
                         ids=["tmem128", "tmem256", "tmem512"])
def test_full_occupancy(mods, name, hidden):
    """Every row bit for bit (identity) and within TANH_ULP (tanh) while every SM holds as many CTAs as its 512 TMEM
    columns serve (4 at width 64, 2 at 128, 1 at 256), for two waves."""
    ni, N, torch = mods
    S, A = S_A[name]
    n = full_occupancy_rows(torch, hidden)
    env = ni.NativeEnv(KINDS[name], 1, device=0, seed=1)
    net = exact_mlp(seeded(name, "full"), S, A, hidden, n, norm=True)
    for act in ("identity", "tanh"):
        check_device(env, policy(net, act), net[2], f"{name} {wid(hidden)} {act} n={n}")
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [(128,), (256, 64)], ids=wid)
def test_null_bias_and_normalisation_pointers(mods, hidden):
    """nig_set_mlp_policy with bias[l] = NULL and obs_mean / obs_inv_std = NULL == explicit zero biases, zero mean and unit
    inverse std, bit for bit; in between, the same weights with non-zero biases and a normalisation are uploaded on the
    same handle, so that an upload that left the previous network in place would fail."""
    ni, N, torch = mods
    import ctypes as C
    S, A = S_A["robot"]
    env = ni.NativeEnv(KINDS["robot"], 1, device=0, seed=1)
    ws, bs, obs, _, _ = exact_mlp(seeded("null", hidden), S, A, hidden, 300)
    zeros = MLPPolicy(ws, [np.zeros_like(b) for b in bs], "identity", obs_mean=np.zeros(S, np.float32),
                      obs_std=np.ones(S, np.float32))
    explicit = check_device(env, zeros, obs, "explicit zero biases, zero mean, unit std")
    other = MLPPolicy(ws, bs, "identity", obs_mean=np.full(S, 0.5, np.float32), obs_std=np.full(S, 0.5, np.float32))
    assert not np.array_equal(check_device(env, other, obs, "non-zero biases, normalised"), explicit)
    m = zeros.native_struct()
    for k in range(len(ws)):
        m.bias[k] = None
    m.obs_mean = m.obs_inv_std = None
    N.check(N.lib().nig_set_mlp_policy(env._h, C.byref(m)))
    assert_bits_equal(env.selftest_mlp(obs), explicit, "NULL biases and normalisation")
    env.close()


CONCURRENT = r"""
import json, sys
import numpy as np
sys.path[:0] = [{root!r}, {root!r} + "/tests", {root!r} + "/neorl-industrial-gym_b200"]
import torch
import neorl_industrial as ni
from neorl_industrial import _native as N
from torch.profiler import ProfilerActivity, profile
from test_gpu_mlp_exact import S_A, exact_mlp, full_occupancy_rows, seeded
from util import assert_bits_equal

K = 64
runs = []
for kind, name, hidden, n in ((0, "reactor", (64, 64), full_occupancy_rows(torch, (64, 64))), (1, "grid", (256, 256), 37_965)):
    env = ni.NativeEnv(kind, n, device=0, seed=6, max_episode_steps=40)
    st = env.reset_host()
    env.track_extrema(True)
    S, A = S_A[name]
    ws, bs = exact_mlp(seeded("concurrent", name), S, A, hidden, 4_096)[:2]
    env.set_mlp_policy(ni.MLPPolicy(ws, bs, "tanh", obs_mean=st.mean(0), obs_std=st.std(0) + 1e-3))
    runs.append(dict(env=env, name=name, start=env.get_state_host(), tick=(env.tick, env.epoch), rs=env.empty()))
torch.cuda.synchronize()

def restart(r):
    r["env"].set_state_host(*r["start"])
    r["env"].set_tick(*r["tick"])
    r["env"].clear_stats()

def result(r):
    env = r["env"]
    return env.get_state_host(), r["rs"][:env.n].cpu().numpy().copy(), env.read_stats(), env.read_extrema()

alone = []
for r in runs:
    restart(r)
    r["env"].rollout_device(K, N.POLICY_MLP, reward_sum=r["rs"])
    torch.cuda.synchronize()
    alone.append(result(r))
for r in runs:
    restart(r)
streams = [torch.cuda.Stream() for _ in runs]
gate, ready = torch.cuda.Stream(), torch.cuda.Event()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    # both launches wait for one event behind a ~10 ms spin, so that the host's time between the two calls cannot
    # serialise them: the device sees both at once
    with torch.cuda.stream(gate):
        torch.cuda._sleep(20_000_000)
        ready.record(gate)
    for r, s in zip(runs, streams):
        s.wait_event(ready)
        with torch.cuda.stream(s):
            r["env"].rollout_device(K, N.POLICY_MLP, reward_sum=r["rs"])
    torch.cuda.synchronize()
prof.export_chrome_trace(sys.argv[1])
for r, a in zip(runs, alone):
    b, w = result(r), r["name"] + ": concurrent vs alone"
    for k in range(4):
        assert_bits_equal(b[0][k], a[0][k], f"{{w}}: state part {{k}}")
    assert_bits_equal(b[1], a[1], f"{{w}}: per-env reward sum")
    assert np.array_equal(b[2][0], a[2][0]) and np.allclose(b[2][1], a[2][1], rtol=1e-12, atol=0), (w, b[2], a[2])
    assert b[3] == a[3] and a[3][0] is not None, (w, b[3], a[3])
    assert a[2][0][1] > 0, (w, "no episode finished")
    r["env"].close()
print("concurrent ok")
"""


@pytest.mark.gpu
def test_two_tmem_widths_concurrently(tmp_path):
    """A reactor handle with a width-64 network (128 TMEM columns, 4 CTAs per SM) at full-occupancy size and a PowerGrid
    handle with a 256-256 network (512 columns) run K steps on two streams, released together by one event: states,
    per-env reward sums, statistics and extrema equal each handle's run alone from the same state and tick. The kernel
    intervals are recorded with torch.profiler (in a child process: profiler sessions early in a suite can leave later
    ones empty) and must overlap, so that the test cannot silently stop testing concurrency."""
    trace = tmp_path / "trace.json"
    out = subprocess.run([sys.executable, "-c", CONCURRENT.format(root=ROOT), str(trace)], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0 and "concurrent ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
    events = json.loads(trace.read_text())["traceEvents"]
    spans = {}
    for e in events:
        if e.get("ph") == "X" and "rollout_mlp_kernel" in e.get("name", ""):
            env = "Reactor" if "Reactor" in e["name"] else "Grid" if "Grid" in e["name"] else None
            spans.setdefault(env, []).append((float(e["ts"]), float(e["ts"]) + float(e["dur"])))
    assert set(spans) == {"Reactor", "Grid"} and all(len(v) == 1 for v in spans.values()), spans
    (r0, r1), (g0, g1) = spans["Reactor"][0], spans["Grid"][0]
    assert r0 < g1 and g0 < r1, f"the two rollouts did not overlap: reactor {r0:.1f}..{r1:.1f} us, grid {g0:.1f}..{g1:.1f} us"
