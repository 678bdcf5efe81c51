"""Exhaustive CPU proof of three shortcuts in the reactor's fused rollout loop (reactor_fast_steps_v, nig_kernels.cuh), against
the oracle's own math spec (tests/fast_exp_check.c is compiled together with oracle/nig_oracle.c):
  * the shortened exp of the loop (spec_expf_small_v: no clamps, rint by the 1.5 * 2^23 shift, one multiply by 2^n)
    returns the bits of spec_expf for every binary32 in [-6, 6], both zeros included;
  * the episode-end cat / 100 by the constant division equals the IEEE quotient for every cat Reactor::reset can draw;
  * the uniform-policy actions (Reactor::uniform_from_words, one add on the random mantissa bits) equal the fma form.
The GPU parity tests compare the kernels themselves with the oracle; this pins the whole input range of all three."""
import os
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "fast_exp_check.c")
# the oracle's flags (oracle/Makefile): no contraction, fmaf as one instruction
CFLAGS = ["-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-fopenmp", "-Wall", "-Wno-unused-function"]


def test_fast_loop_exp_and_reset_division_are_exact(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    assert cc, "a C compiler is needed (the oracle is built with gcc too)"
    exe = str(tmp_path / "fast_exp_check")
    subprocess.check_call([cc, *CFLAGS, "-o", exe, SRC, "-lm"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "exp: 2172649474 values in [-6, 6], 0 mismatches" in out.stdout, out.stdout
    assert " 0 mismatches of cat / 100" in out.stdout, out.stdout
    assert "uniform actions: 0 mismatches" in out.stdout, out.stdout
