"""CPU tests of the C-ABI boundary: the library loads, exports every symbol include/nig_b200.h declares,
struct layouts agree, metadata is right, and without a GPU every compute entry point fails LOUDLY
(no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import neorl_industrial as ni
from neorl_industrial import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "nig_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"NIG_API\s+[\w\s\*]+?\b(nig_\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    names = declared_symbols()
    assert len(names) >= 30
    raw = C.CDLL(N.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} declared in include/nig_b200.h but not exported by libnig_b200.so"
    assert set(names) == set(N.SYMBOLS), set(names) ^ set(N.SYMBOLS)


def test_abi_version_and_specs():
    lib = N.lib()
    assert lib.nig_abi_version() == N.ABI_VERSION
    expect = {0: (12, 3, 2, 500), 1: (32, 8, 23, 1000), 2: (24, 7, 0, 1000)}
    pens = {0: [(-100, 1), (-50, 1), (-25, 0)], 1: [(-50, 1), (-30, 1), (-20, 0)], 2: [(-100, 1), (-200, 1), (-50, 0)]}
    for kind, (s, a, nz, ms) in expect.items():
        sp = N.env_spec(kind)
        assert (sp.state_dim, sp.action_dim, sp.noise_dim, sp.max_episode_steps, sp.n_constraints) == (s, a, nz, ms, 3)
        got = [(sp.constraints[k].penalty, sp.constraints[k].critical) for k in range(3)]
        assert got == pens[kind]
    with pytest.raises(ValueError):
        N.env_spec(7)


def test_struct_sizes_match_header(tmp_path):
    """ctypes mirrors == what a C compiler makes of include/nig_b200.h (sizes and a few telling offsets)."""
    import subprocess
    src = tmp_path / "sizes.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "nig_b200.h"\n'
        'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(nig_constraint_t), sizeof(nig_config_t),'
        ' sizeof(nig_policy_params_t), sizeof(nig_step_io_t), sizeof(nig_rollout_t), sizeof(nig_rollout_host_t),'
        ' sizeof(nig_dataset_out_t), sizeof(nig_env_spec_t), sizeof(nig_baseline_t), offsetof(nig_policy_params_t, baseline),'
        ' offsetof(nig_rollout_host_t, reward_sum)); return 0;}\n')
    exe = tmp_path / "sizes"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(N.Constraint), C.sizeof(N.Config), C.sizeof(N.PolicyParams), C.sizeof(N.StepIO), C.sizeof(N.Rollout),
            C.sizeof(N.RolloutHost), C.sizeof(N.DatasetOut), C.sizeof(N.EnvSpec), C.sizeof(N.Baseline),
            N.PolicyParams.baseline.offset, N.RolloutHost.reward_sum.offset]
    assert got == want, (got, want)
    assert C.sizeof(N.Constraint) == 36 and C.sizeof(N.Config) == 48 + 8 * 36


def test_make_registry_errors():
    with pytest.raises(ValueError, match="Unknown environment 'Nope-v0'. Available: "):
        ni.make("Nope-v0")
    with pytest.raises(NotImplementedError):
        ni.make("AdvancedPowerGrid-v0")


def test_no_gpu_means_loud_failure():
    if N.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ni.make("ChemicalReactor-v0")
    with pytest.raises(ValueError):
        ni.make("ChemicalReactor-v0", device="cpu")


def test_create_rejects_env_ids_beyond_32_bits():
    """Global env ids are 32-bit: nig_create refuses env_id_offset < 0 and env_id_offset + n_envs > 2^32 before it looks
    for a device, so the range check answers NIG_ERR_INVALID with or without a GPU; the last valid offset passes it."""
    lib = N.lib()

    def create(n, off):
        cfg = N.Config()
        cfg.env_kind, cfg.device, cfg.n_envs, cfg.env_id_offset, cfg.n_constraints = N.ENV_CHEMICAL_REACTOR, 0, n, off, -1
        h = C.c_void_p()
        rc = lib.nig_create(C.byref(cfg), C.byref(h))
        if h.value:
            lib.nig_destroy(h)
        return rc
    for n, off in ((100, (1 << 32) - 99), (1, 1 << 32), (1 << 31, (1 << 31) + 1), (5, -1), (5, -(1 << 40))):
        assert create(n, off) == N.ERR_INVALID, (n, off)
        assert "2^32" in N.lib().nig_last_error().decode(), (n, off)
    for n, off in ((100, (1 << 32) - 100), (1, (1 << 32) - 1)):
        assert create(n, off) in (N.OK, N.ERR_NO_DEVICE), (n, off)
    with pytest.raises(ValueError, match="2\\^32"):
        ni.NativeEnv(N.ENV_POWER_GRID, 10, env_id_offset=(1 << 32) - 9)


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing in the product may import, include, link or dlopen it."""
    pkg = os.path.join(ROOT, "neorl-industrial-gym_b200")
    bad = re.compile(r"(import\s+oracle|from\s+oracle|libnig_oracle|nig_oracle|oracle\.py|[\"'<]\.*/*oracle/|orc_[a-z_]+\()")
    checked = 0
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                src = open(os.path.join(dirpath, f)).read()
                src = src.replace("nothing under oracle/ is ever imported", "")     # the loader's own statement of this rule
                assert not bad.search(src), os.path.join(dirpath, f)
                checked += 1
    assert checked >= 12


def test_types_and_spaces():
    sm = ni.SafetyMetrics(2, 3, 1, 1, 2 / 3)
    assert abs(sm.satisfaction_rate - 2 / 3) < 1e-12 and sm.violation_severity == {}
    c = ni.BoundConstraint("t_band", 0, 280, 320, penalty=-100, action_index=0, action_coef=0.1)
    assert c.check_fn(np.array([300.0] + [0] * 11, np.float32), np.zeros(3, np.float32))
    assert not c.check_fn(np.array([320.0] + [0] * 11, np.float32), np.ones(3, np.float32))
    assert c._native[0] == "bound"
    from neorl_industrial.spaces import Box
    b = Box(-1.0, 1.0, (3,), np.float32, seed=0)
    x = b.sample()
    assert x.dtype == np.float32 and x.shape == (3,) and b.contains(x)
    bm = ni.BatchedSafetyMetrics(np.array([0, 1, 3, 7], np.uint8), 3, 0b011)
    assert bm.violation_count.tolist() == [0, 1, 2, 3] and bm.critical_violations.tolist() == [0, 1, 2, 2]
    assert bm[2].constraints_satisfied == 1


def test_extrema_keys_decode_in_order():
    """nig_decode_extrema inverts the order-preserving int64 keys the rollout kernel keeps for return_min / return_max
    (utils.py:131-132): key(x) restated in numpy here, monotone in x, the maximum of the keys decodes to the extremum."""
    def key(x):
        b = np.array(x, np.float64).view(np.uint64)
        k = np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))
        return (k >> np.uint64(1)).astype(np.int64)

    rng = np.random.default_rng(3)
    xs = np.concatenate([rng.normal(0, 1e4, 4000), rng.normal(0, 1e-3, 100), [0.0, 1e300, -1e300]])
    order = np.argsort(xs, kind="stable")
    ks = key(xs)
    assert (np.diff(ks[order]) >= 0).all() and (ks > 0).all()
    assert key(-0.0) < key(0.0) < key(5e-324 * 4)
    keys = np.array([key(-xs).max(), ks.max()], np.int64)
    lo, hi = ni.NativeEnv.decode_extrema(keys)
    assert np.isclose(lo, xs.min(), rtol=3e-16, atol=0) and np.isclose(hi, xs.max(), rtol=3e-16, atol=0)
    assert ni.NativeEnv.decode_extrema(np.zeros(2, np.int64)) == (None, None)


def test_normal_table_headers_are_the_generators_output(tmp_path):
    """csrc/nig_normal_table.h and oracle/nig_normal_table.h hold the same numbers, and they are what
    tools/fit_normal_table.py produces today (the table is data of the math spec: library and oracle must not drift)."""
    import importlib.util
    a = open(os.path.join(ROOT, "neorl-industrial-gym_b200", "csrc", "nig_normal_table.h")).read()
    b = open(os.path.join(ROOT, "oracle", "nig_normal_table.h")).read()
    strip = lambda t: t.split("*/", 1)[1]
    assert strip(a) == strip(b)
    spec = importlib.util.spec_from_file_location("fit_normal_table", os.path.join(ROOT, "tools", "fit_normal_table.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    tab, err_abs, _ = mod.build()
    out = tmp_path / "t.h"
    mod.emit(tab, str(out), "CUDA library")
    assert out.read_text() == a
    assert tab.shape == (513, 4) and err_abs < 6e-7


def test_library_and_oracle_share_one_normal_table():
    """csrc/nig_normal_table.h and oracle/nig_normal_table.h are two emissions of tools/fit_normal_table.py: the same
    numbers (a silent divergence would show up as baffling bit-level parity failures)."""
    strip = lambda t: [l for l in t.splitlines() if not l.lstrip().startswith(("//", "/*", "*"))]
    a = open(os.path.join(ROOT, "neorl-industrial-gym_b200", "csrc", "nig_normal_table.h")).read()
    b = open(os.path.join(ROOT, "oracle", "nig_normal_table.h")).read()
    assert strip(a) == strip(b)


def test_bench_reference_arm_runs_without_a_gpu():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm) needs no GPU: one JSON line with the
    contract's keys, the same metric / unit as the GPU arm, `impl: reference`, a cpu_baseline block and an e2e block."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("env-steps/sec (ChemicalReactor-v0") and line["value"] > 2e3
    # the reference's own Python loop (oracle/_ref, made by oracle/make_ref.py) when present, else the C port
    import bench
    from oracle import make_ref
    assert line["cpu_baseline"]["kind"] == ("reference" if make_ref.available() else "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["config"] == bench.bench_config(1)                  # the CUDA arm prints the same object
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["gpu_launches"] == 0 and line["vs_baseline"] is None


def test_reference_copy_is_byte_identical_and_not_in_history():
    """oracle/_ref, where oracle/make_ref.py made it, holds the seven hot-path reference modules byte for byte (SHA-256
    manifest; compared with the reference tree too when that exists), and it is git-ignored: reference sources never
    enter this repo's history."""
    import subprocess
    from oracle import make_ref
    if make_ref.available():
        assert make_ref.verify()
    r = subprocess.run(["git", "-C", ROOT, "check-ignore", "-q", "oracle/_ref/MANIFEST.json"])
    if r.returncode in (0, 1):                                      # 128: not a git checkout (a copy of the tree)
        assert r.returncode == 0
    tracked = subprocess.run(["git", "-C", ROOT, "ls-files", "oracle/_ref"], capture_output=True, text=True)
    assert tracked.stdout.strip() == ""


def test_bench_has_no_literal_throughput_numbers():
    """every baseline figure bench.py prints is measured in the same run (VERDICT r01: a hard-coded 12,177 steps/s)."""
    import re
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert "12177" not in src and "9,378" not in src and "9378" not in src
    assert not re.search(r'"value":\s*[0-9]', src)
