"""The on-device get_dataset writer beyond its default path: dataset_kernel<Env, CONS_GENERIC, ...> for constraint sets
(SafetyWrapper bounds, re-ordered or removed built-ins), scan_lengths_kernel with more than one episode per scan thread,
truncation inside a dataset with both terminals conventions, the UNIFORM and ZERO policies with and without store_clip,
the qualities tests/test_gpu_dataset.py does not run, null optional outputs, and the length-probe cache across a re-seed.
Every case compares every written array, n_written and nig_dataset_size with the CPU oracle (spec-exp mode) bit for bit,
so the scan's offsets are checked through the rows they place. Every output has rows past the dataset's end, filled with a
sentinel that must survive. A dispatch witness records kernel names so that these tests cannot lose their target
silently."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import KINDS, assert_bits_equal, kernel_names, oracle_dataset, template_args

pytestmark = pytest.mark.gpu

ENV_CLASS = {"reactor": "ChemicalReactorEnv", "grid": "PowerGridEnv", "robot": "RobotAssemblyEnv"}
ENV_T = {"reactor": "Reactor", "grid": "Grid", "robot": "Robot"}
CONS_GENERIC, CONS_DEFAULT = 0, 1                  # nig_kernels.cuh
SENTINEL = 0xA5                                    # fill byte of every output (0xA5A5A5A5 is a finite float)
SLACK = 37                                         # rows past the dataset's end in every output
OPTIONAL = ("timeouts", "next_observations", "safety")


@pytest.fixture(scope="module")
def mods():
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from oracle import oracle as O
    return ni, N, O, torch


def _policy(ni, name, quality):
    """(n_steps, policy, PolicyParams) of get_dataset(quality)."""
    _, n_steps, policy, pp = getattr(ni, ENV_CLASS[name]).dataset_policy(quality)
    return n_steps, policy, pp


def _write(torch, env, n_ep, n_steps, policy, pp, incl, cap, optional=True):
    """nig_dataset into outputs of `cap` rows (optional=False: without timeouts, next_observations and safety), every byte
    set to SENTINEL first. Checks that the rows from n_written on still hold it; returns host copies of the written rows
    and n_written."""
    dev = env.torch_device()
    f32, u8 = torch.float32, torch.uint8
    spec = {"observations": ((cap, env.S), f32), "actions": ((cap, env.A), f32), "rewards": ((cap,), f32),
            "terminals": ((cap,), u8), "timeouts": ((cap,), u8), "next_observations": ((cap, env.S), f32),
            "safety": ((cap,), u8)}
    out = {}
    for k, (shape, dt) in spec.items():
        if optional or k not in OPTIONAL:
            out[k] = torch.empty(shape, dtype=dt, device=dev)
            out[k].view(u8).fill_(SENTINEL)
    written = env.dataset_device(n_ep, n_steps, policy, pp, out, cap, incl)
    torch.cuda.synchronize()
    host = {k: v.cpu().numpy() for k, v in out.items()}
    for k, v in host.items():
        assert (v[written:].view(np.uint8) == SENTINEL).all(), f"{k}: a row past n_written = {written} was written"
    return {k: v[:written] for k, v in host.items()}, written


def _check(got, m, written, ref, lens, what):
    assert m == written == int(lens.sum()) == len(ref["rewards"]), (what, m, written, int(lens.sum()))
    for k in ("observations", "actions", "rewards", "next_observations"):
        if k in got:
            assert_bits_equal(got[k], ref[k], f"{what}: {k}")
    assert_bits_equal(got["terminals"], ref["terminals"].astype(np.uint8), f"{what}: terminals")
    if "safety" in got:
        assert_bits_equal(got["safety"], ref["safety"], f"{what}: safety")
    if "timeouts" in got:
        assert not got["timeouts"].any(), what


def _run(mods, name, n_ep, n_steps, policy, pp, *, seed, incl, cons=None, max_steps=None, env0=0, optional=True,
         threads=1, what=""):
    """One dataset from a fresh one-env handle against the oracle; returns the oracle's rows and episode lengths."""
    ni, N, O, torch = mods
    kind = KINDS[name]
    env = ni.NativeEnv(kind, 1, device=0, seed=seed, env_id_offset=env0, max_episode_steps=max_steps, constraints=cons)
    m = env.dataset_size(n_ep, n_steps, policy, pp)
    got, written = _write(torch, env, n_ep, n_steps, policy, pp, incl, m + SLACK, optional)
    env.close()
    kw = {} if cons is None else {"builtin": False, "extra_cons": _ocons(O, cons)}
    ref, lens = oracle_dataset(O, kind, n_ep, n_steps, policy, pp, seed, 0, env0, incl, max_episode_steps=max_steps,
                               threads=threads, **kw)
    _check(got, m, written, ref, lens, what or name)
    return ref, lens


def _ocons(O, cons):
    return [O.Con(c.kind, c.id, c.si, c.ai, c.coef, c.lo, c.hi, c.penalty, c.critical) for c in cons]


def _builtins(N, kind, order=(0, 1, 2)):
    from neorl_industrial.vector import make_constraint
    spec = N.env_spec(kind)
    return [make_constraint(N.CON_BUILTIN, cid=k, penalty=spec.constraints[k].penalty,
                            critical=bool(spec.constraints[k].critical)) for k in order]


# ---------------------------------------------------------------------------------------------------------------------
# 1. dispatch witness
def _dispatch_names():
    """Prints, as JSON, the kernel names torch.profiler records for one small dataset per env and constraint set."""
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N
    from neorl_industrial.vector import make_constraint
    out = {}
    for name in ENV_T:
        kind = KINDS[name]
        _, policy, pp = _policy(ni, name, "mixed")
        bound = make_constraint(N.CON_BOUND, si=0, lo=-1.0, hi=1.0, penalty=-5.0)
        for label, cons in (("default", None), ("appended", _builtins(N, kind) + [bound]),
                            ("reordered", _builtins(N, kind, (2, 0, 1))), ("removed", _builtins(N, kind, (0, 2)))):
            env = ni.NativeEnv(kind, 1, device=0, seed=1, constraints=cons)

            def call():
                m = env.dataset_size(64, 20, policy, pp)
                _write(torch, env, 64, 20, policy, pp, True, m + SLACK)
            out[f"{name} {label}"] = sorted(kernel_names(torch, call))
            env.close()
    print(json.dumps(out))


def test_dataset_dispatch_witness():
    """A constraint set other than the env's default one runs both passes of dataset_kernel<Env, CONS_GENERIC, ...>; the
    default set runs CONS_DEFAULT; the scan runs between them. The names are recorded in a child process: profiler
    sessions started this early in the suite's process made the later witnesses of test_gpu_rollout_flavours.py and
    test_gpu_step_flavours.py record no kernels (torch 2.11, CUDA 12.8)."""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    code = (f"import sys; sys.path[:0] = {[root, os.path.join(root, 'neorl-industrial-gym_b200'), here]!r}; "
            "import test_gpu_dataset_flavours as t; t._dispatch_names()")
    flags = ["-s"] if sys.flags.no_user_site else []
    run = subprocess.run([sys.executable, *flags, "-c", code], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-8000:]
    got = json.loads(run.stdout.strip().splitlines()[-1])
    if not any(template_args(names, "dataset_kernel") for names in got.values()):
        pytest.skip("torch.profiler recorded no CUDA kernel in the child process (no CUPTI activity records)")
    for case, names in got.items():
        c = CONS_DEFAULT if case.endswith("default") else CONS_GENERIC
        env_t = ENV_T[case.split()[0]]
        assert template_args(names, "dataset_kernel") == {(env_t, str(c), "false"), (env_t, str(c), "true")}, (case, names)
        assert any("scan_lengths_kernel" in x for x in names), (case, names)


# ---------------------------------------------------------------------------------------------------------------------
# 2. constraint sets
def _cons_set(N, O, name, which, n_steps, policy, pp):
    """Constraint sets for the dataset kernels. The bands sit at quantiles of the rows of a default-set dataset, so that
    the plain band fires in about a fifth of the rows and the critical one ends episodes now and then."""
    from neorl_industrial.vector import make_constraint
    kind = KINDS[name]
    ref, _ = oracle_dataset(O, kind, 40, n_steps, policy, pp, 11, 0, 0, True)
    s = ref["observations"]
    s = s[np.isfinite(s).all(1)]
    f32 = lambda x: float(np.float32(x))
    q = lambda si, p: f32(np.quantile(s[:, si], p))
    band = make_constraint(N.CON_BOUND, si=0, lo=q(0, 0.1), hi=q(0, 0.9), penalty=-40.0)
    if which == "appended":      # SafetyWrapper: the built-ins, then a state band and a band with an action term
        return _builtins(N, kind) + [band, make_constraint(N.CON_BOUND, si=0, ai=0, coef=f32(0.1), lo=q(0, 0.2),
                                                           hi=q(0, 0.8), penalty=-15.0)]
    if which == "critical_nan":  # a critical band that ends episodes, then a NaN bound that every row violates
        return _builtins(N, kind) + [
            make_constraint(N.CON_BOUND, si=1, lo=q(1, 0.002), hi=q(1, 0.998), penalty=-60.0, critical=True),
            make_constraint(N.CON_BOUND, si=0, lo=q(0, 0.5), hi=float("nan"), penalty=-3.0)]
    if which == "reordered":
        return _builtins(N, kind, (2, 0, 1)) + [band]
    return _builtins(N, kind, (0, 2)) + [band]         # "removed": built-in 1 left out


@pytest.mark.parametrize("which", ["appended", "critical_nan", "reordered", "removed"])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_constraint_sets_vs_oracle(mods, name, which):
    ni, N, O, torch = mods
    n_steps, policy, pp = _policy(ni, name, "mixed")
    n_steps = min(n_steps, 300)
    cons = _cons_set(N, O, name, which, n_steps, policy, pp)
    ref, lens = _run(mods, name, 300, n_steps, policy, pp, seed=23, incl=name == "reactor", cons=cons, env0=777,
                     what=f"{name} {which}")
    saf = ref["safety"].astype(np.int64)
    assert ((saf >> (len(cons) - 1)) & 1).any(), "no row violates the last constraint"
    if which == "critical_nan":
        assert ((saf >> 4) & 1).all(), "the NaN bound must be violated in every row"
        ends = ref["terminals"] & (((saf >> 3) & 1) == 1)
        assert ends.any(), "the critical band ended no episode"


def test_safety_wrapper_get_dataset(mods):
    """The public path: SafetyWrapper(make(...), [BoundConstraint(...)]).get_dataset(..., extensions=True) == the oracle
    with the built-ins followed by the same bounds; a callable (host-evaluated) constraint makes get_dataset raise."""
    ni, N, O, torch = mods
    from neorl_industrial.safety import BoundConstraint, SafetyWrapper
    env = SafetyWrapper(ni.make("ChemicalReactor-v0", seed=31), [
        BoundConstraint("temperature band", 0, 305.0, 325.0, penalty=-100.0),
        BoundConstraint("pressure with feed", 1, 1.0e5, 2.6e5, penalty=-37.5, action_index=1, action_coef=1.0e4)])
    d = env.get_dataset("mixed", n_episodes=150, extensions=True)
    n_steps, policy, pp = _policy(ni, "reactor", "mixed")
    extra = [O.bound_con(0, np.float32(305.0), np.float32(325.0), -100.0),
             O.bound_con(1, np.float32(1.0e5), np.float32(2.6e5), -37.5, ai=1, coef=np.float32(1.0e4))]
    ref, lens = oracle_dataset(O, O.REACTOR, 150, n_steps, policy, pp, 31, 0, 0, True, extra_cons=extra)
    assert len(d["rewards"]) == int(lens.sum())
    for k in ("observations", "actions", "rewards", "next_observations", "safety"):
        assert_bits_equal(d[k], ref[k], k)
    assert_bits_equal(d["terminals"], ref["terminals"], "terminals")
    assert not d["timeouts"].any()
    assert ((ref["safety"] >> 3) & 1).any() and ((ref["safety"] >> 4) & 1).any()
    env.unwrap().close()
    host = SafetyWrapper(ni.make("ChemicalReactor-v0", seed=31), [lambda s, a: s[0] < 340.0])
    with pytest.raises(NotImplementedError, match="host-evaluated"):
        host.get_dataset("mixed", n_episodes=10)
    host.unwrap().close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. scan sizes
@pytest.mark.parametrize("n_ep", [1023, 1024, 1025, 4099, 50_000])
def test_scan_sizes_vs_oracle(mods, n_ep):
    """PowerGrid 'mixed' episodes are short and vary widely in length (about 5.5 steps): the one-block scan takes
    ceil(n / 1024) = 1, 1, 2, 5 and 49 lengths per thread, idle threads at the tail, and the dataset kernels several waves."""
    ni, N, O, torch = mods
    _, policy, pp = _policy(ni, "grid", "mixed")
    _, lens = _run(mods, "grid", n_ep, 40, policy, pp, seed=41, incl=False, env0=n_ep, threads=O.max_threads())
    assert lens.min() < 5 and lens.max() > 20


def test_scan_reactor_over_1024_episodes(mods):
    ni, N, O, torch = mods
    _, policy, pp = _policy(ni, "reactor", "mixed")
    _run(mods, "reactor", 2_500, 60, policy, pp, seed=43, incl=True, threads=O.max_threads())


# ---------------------------------------------------------------------------------------------------------------------
# 4. truncation
@pytest.mark.parametrize("incl", [True, False])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_truncation_inside_dataset(mods, name, incl):
    """Handles created with an episode cap below n_steps: episodes that reach the cap end TRUNCATED, and their last row's
    terminal follows terminals_include_truncation."""
    ni, N, O, torch = mods
    _, policy, pp = _policy(ni, name, "mixed")
    cap, n_steps = {"reactor": (250, 300), "grid": (6, 80), "robot": (37, 80)}[name]     # some episodes end before the cap
    ref, lens = _run(mods, name, 200, n_steps, policy, pp, seed=47, incl=incl, max_steps=cap, what=f"{name} cap {cap}")
    assert lens.max() == cap and (lens < cap).any()
    last = ref["terminals"][(np.cumsum(lens) - 1)[lens == cap]]       # (an episode may also terminate on its last step)
    assert last.all() if incl else not last.all()


def test_robot_mixed_reaches_its_episode_cap(mods):
    """RobotAssembly 'mixed' at its real n_steps of 1,000 = its episode cap: a few episodes run into it."""
    ni, N, O, torch = mods
    n_steps, policy, pp = _policy(ni, "robot", "mixed")
    assert n_steps == 1000
    _, lens = _run(mods, "robot", 250, n_steps, policy, pp, seed=7, incl=False)
    assert (lens == 1000).sum() >= 2


# ---------------------------------------------------------------------------------------------------------------------
# 5. policies and qualities
@pytest.mark.parametrize("clip", [0.0, 0.5])
@pytest.mark.parametrize("policy", ["UNIFORM", "ZERO"])
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_uniform_and_zero_policies(mods, name, policy, clip):
    ni, N, O, torch = mods
    pp = N.PolicyParams()
    pp.store_clip = clip
    pol = {"UNIFORM": N.POLICY_UNIFORM, "ZERO": N.POLICY_ZERO}[policy]
    ref, _ = _run(mods, name, 200, 150, pol, pp, seed=53, incl=name != "grid", what=f"{name} {policy} clip {clip}")
    a = np.abs(ref["actions"])
    if policy == "ZERO":
        assert (a == 0).all()
    else:
        assert a.max() == 0.5 if clip else 0.99 < a.max() <= 1.0


@pytest.mark.parametrize("name,quality,n_ep", [("reactor", "medium", 150), ("grid", "random", 200), ("grid", "medium", 200),
                                               ("robot", "random", 150), ("robot", "medium", 150)])
def test_remaining_qualities(mods, name, quality, n_ep):
    """The get_dataset qualities tests/test_gpu_dataset.py does not run, at their real n_steps."""
    ni, N, O, torch = mods
    n_steps, policy, pp = _policy(ni, name, quality)
    _run(mods, name, n_ep, n_steps, policy, pp, seed=59, incl=name == "reactor", env0=4096, what=f"{name} {quality}")


# ---------------------------------------------------------------------------------------------------------------------
# 6. output combinations
@pytest.mark.parametrize("name", ["reactor", "grid", "robot"])
def test_null_optional_outputs(mods, name):
    """timeouts, next_observations and safety all null: the required arrays are the same, nothing past n_written."""
    ni, N, O, torch = mods
    n_steps, policy, pp = _policy(ni, name, "mixed")
    _run(mods, name, 120, min(n_steps, 300), policy, pp, seed=61, incl=True, optional=False, what=f"{name} required only")


# ---------------------------------------------------------------------------------------------------------------------
# 7. the length-probe cache across a re-seed
def test_stale_probe_after_set_seed(mods):
    """nig_dataset_size with seed A, nig_set_seed(B), nig_dataset: the dataset of seed B, not B's episodes at A's row
    offsets. The outputs hold 2 x max(total A, total B) + n_steps rows, so that a stale probe cannot write past them."""
    ni, N, O, torch = mods
    n_steps, policy, pp = _policy(ni, "grid", "mixed")
    n_ep = 400
    env = ni.NativeEnv(KINDS["grid"], 1, device=0, seed=71)
    m_a = env.dataset_size(n_ep, n_steps, policy, pp)
    env.set_seed(72)
    ref, lens = oracle_dataset(O, O.GRID, n_ep, n_steps, policy, pp, 72, 0, 0, False)
    assert m_a != int(lens.sum())
    got, written = _write(torch, env, n_ep, n_steps, policy, pp, False, 2 * max(m_a, int(lens.sum())) + n_steps)
    m_b = env.dataset_size(n_ep, n_steps, policy, pp)       # the next dataset (gen 1) of seed B
    env.close()
    _check(got, written, written, ref, lens, "after set_seed")
    fresh = ni.NativeEnv(KINDS["grid"], 1, device=0, seed=72)
    same, _ = _write(torch, fresh, n_ep, n_steps, policy, pp, False, written + SLACK)
    fresh.close()
    for k, v in same.items():
        assert_bits_equal(got[k], v, f"re-seeded handle vs a fresh one: {k}")
    _, lens1 = oracle_dataset(O, O.GRID, n_ep, n_steps, policy, pp, 72, 1, 0, False)
    assert m_b == int(lens1.sum())


def test_stale_probe_through_get_dataset(mods):
    """episodes_for_transitions leaves its final count as the cached probe; env.reset(seed=B) then get_dataset(n_episodes=
    that count) must write seed B's dataset. Seeds A and B are chosen so that even B's episodes at A's row offsets stay
    inside the arrays get_dataset sizes from a stale probe (checked below with the oracle's lengths)."""
    ni, N, O, torch = mods
    from neorl_industrial.datasets import episodes_for_transitions
    seed_a, seed_b = 81, 82
    env = ni.make("PowerGrid-v0", seed=seed_a)
    n_steps, policy, pp = _policy(ni, "grid", "mixed")
    n_ep = episodes_for_transitions(env.native, 2_000, n_steps, policy, pp)
    _, lens_a = oracle_dataset(O, O.GRID, n_ep, n_steps, policy, pp, seed_a, 0, 0, False)
    ref, lens = oracle_dataset(O, O.GRID, n_ep, n_steps, policy, pp, seed_b, 0, 0, False)
    off_a = np.cumsum(lens_a) - lens_a
    assert (off_a + lens <= lens_a.sum()).all() and lens_a.sum() != lens.sum()
    env.reset(seed=seed_b)
    d = env.get_dataset("mixed", n_episodes=n_ep, extensions=True)
    env.close()
    assert len(d["rewards"]) == int(lens.sum()), (len(d["rewards"]), int(lens.sum()), int(lens_a.sum()))
    for k in ("observations", "actions", "rewards", "next_observations", "safety"):
        assert_bits_equal(d[k], ref[k], k)
    assert_bits_equal(d["terminals"], ref["terminals"], "terminals")
