"""Shared helpers for the parity tests."""
import glob
import io
import os

import numpy as np

GOLDEN_FILE_LIMIT = 1_000_000     # bytes per fixture file; a larger set is stored as parts <stem>.1.npz, <stem>.2.npz, ...


def save_golden(path_stem, **arrays):
    """np.savez_compressed to <path_stem>.npz, or, when that file would exceed GOLDEN_FILE_LIMIT, whole arrays spread in
    order over the parts <path_stem>.<k>.npz. Replaces whatever <path_stem>.npz / parts an earlier run left."""
    def packed(d):
        buf = io.BytesIO()
        np.savez_compressed(buf, **d)
        return buf.getvalue()

    parts = [packed(arrays)]
    if len(parts[0]) > GOLDEN_FILE_LIMIT:
        parts, cur = [], {}
        for k, v in arrays.items():
            if cur and len(packed({**cur, k: v})) > GOLDEN_FILE_LIMIT:
                parts.append(packed(cur))
                cur = {}
            cur[k] = v
        parts.append(packed(cur))
    for old in glob.glob(path_stem + ".npz") + glob.glob(path_stem + ".[0-9]*.npz"):
        os.remove(old)
    names = [path_stem + ".npz"] if len(parts) == 1 else [f"{path_stem}.{k}.npz" for k in range(1, len(parts) + 1)]
    for name, data in zip(names, parts):
        assert len(data) <= GOLDEN_FILE_LIMIT, (name, len(data))
        with open(name, "wb") as f:
            f.write(data)


def load_golden(golden_dir, stem):
    """The arrays of <stem>.npz, or of all its parts <stem>.<k>.npz (save_golden), as one dict."""
    base = os.path.join(golden_dir, stem)
    paths = glob.glob(base + ".npz") + sorted(glob.glob(base + ".[0-9]*.npz"), key=lambda p: int(p.split(".")[-2]))
    assert paths, f"no golden fixture {base}.npz"
    out = {}
    for p in paths:
        with np.load(p) as z:
            for k in z.files:
                assert k not in out, (p, k)
                out[k] = z[k]
    return out


def ulp_diff(a, b):
    """Distance in units-in-the-last-place between two float32 arrays (0 == bit-identical up to +-0)."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, -(ai & 0x7FFFFFFF), ai)
    bi = np.where(bi < 0, -(bi & 0x7FFFFFFF), bi)
    return np.abs(ai - bi)


def assert_bits_equal(a, b, what=""):
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.dtype == np.float32:
        # +-0 compare equal; a NaN matches a NaN (IEEE 754 leaves sign / payload of a generated NaN to the implementation:
        # x86 yields 0xffc00000 for inf - inf, the GPU 0x7fffffff)
        same = (a.view(np.uint32) == b.view(np.uint32)) | ((a == 0) & (b == 0)) | (np.isnan(a) & np.isnan(b))
    else:
        same = a == b
    if not same.all():
        idx = np.argwhere(~same)[:5]
        raise AssertionError(f"{what}: {np.count_nonzero(~same)} / {same.size} elements differ, first at {idx.tolist()}: "
                             f"{a[tuple(idx[0])]!r} vs {b[tuple(idx[0])]!r}")


KINDS = {"reactor": 0, "grid": 1, "robot": 2}
ENV_IDS = {"reactor": "ChemicalReactor-v0", "grid": "PowerGrid-v0", "robot": "RobotAssembly-v0"}


# ---------------------------------------------------------------------------------------------------------------------
# oracle tracking shared by the kernel-flavour tests (test_gpu_rollout_flavours.py, test_gpu_step_flavours.py)
def popcount8(v):
    return np.unpackbits(np.ascontiguousarray(v, np.uint8)[:, None], axis=1).sum(1, dtype=np.int64)


class Track:
    """Steps the oracle one tick at a time and keeps what a fused launch reports: per-env reward sum (fp32, sequential
    within the launch), violation and done counts; and, over a statistics window (up to clear()), successes, episode
    length sum / square, the fp64 return sum / square, the fp64 reward sum and the return extrema. Returns accumulate in
    the env's accumulator type (fp32 reactor, fp64 grid / robot); a NaN return is skipped by the extrema like the kernels'
    compare-selects skip it."""

    def __init__(self, orc, name):
        self.orc, self.reactor = orc, name == "reactor"
        self.acc_t = np.float32 if self.reactor else np.float64
        self.ep_ret = np.zeros(orc.n, self.acc_t)
        self.clear()

    def clear(self):
        self.orc.stats[:] = 0
        self.succ = self.len_sum = self.len_sq = 0
        self.ret_sum = self.ret_sq = self.rew_sum = 0.0
        self.ret_abs = self.rew_abs = 0.0           # sums of magnitudes (tolerance scale of the fp64 sums)
        self.lo, self.hi = np.inf, -np.inf

    def observe(self, r, fl, vm, steps_before):
        """Books one oracle step (its reward, flags and violation mask; the episode steps before it) into the running
        returns and the window; returns the env mask of finished episodes."""
        if not self.reactor:
            self.rew_sum += float(r.astype(np.float64).sum())
            self.rew_abs += float(np.nansum(np.abs(r.astype(np.float64))))
        self.ep_ret = (self.ep_ret + r.astype(self.acc_t)).astype(self.acc_t)
        done = (fl & 3) > 0
        if done.any():
            er = self.ep_ret[done].astype(np.float64)
            ln = (steps_before[done] + 1).astype(np.int64)
            self.ret_sum += float(er.sum()); self.ret_sq += float((er * er).sum())
            self.ret_abs += float(np.nansum(np.abs(er)))
            self.succ += int((er > 0).sum()); self.len_sum += int(ln.sum()); self.len_sq += int((ln * ln).sum())
            fin = er[~np.isnan(er)]
            if fin.size:
                self.lo, self.hi = min(self.lo, float(fin.min())), max(self.hi, float(fin.max()))
            self.ep_ret[done] = 0
        return done

    def step(self, a, **kw):
        """One oracle step (OracleEnv.step keywords) booked by observe(); returns what the oracle returned."""
        steps_before = self.orc.ep_step.copy()
        out = self.orc.step(a, **kw)
        self.observe(out[1], out[2], out[3], steps_before)
        return out

    def launch(self, K, policy):
        orc, n = self.orc, self.orc.n
        rsum = np.zeros(n, np.float32)
        vcnt = np.zeros(n, np.int64)
        dcnt = np.zeros(n, np.int64)
        for _ in range(K):
            a = policy()
            steps_before = orc.ep_step.copy()
            _, r, fl, vm = orc.step(a, want_next_obs=False)
            rsum = (rsum + r).astype(np.float32)
            vcnt += popcount8(vm)
            dcnt += self.observe(r, fl, vm, steps_before)
        if self.reactor:            # the kernels add each env's fp32 launch sum to the fp64 reward-sum slot
            self.rew_sum += float(rsum.astype(np.float64).sum())
        return rsum, vcnt, dcnt


def _close(got, want, rtol, atol, what):
    if np.isnan(want):
        assert np.isnan(got), (what, got, want)
    else:
        np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=what)


def compare_state(env, orc, what):
    st, ep_step, ep_viol, done = env.get_state_host()
    assert_bits_equal(st, orc.state, f"{what}: state")
    assert_bits_equal(ep_step, orc.ep_step, f"{what}: episode step")
    assert_bits_equal(ep_viol, orc.ep_viol, f"{what}: episode violations")
    assert_bits_equal(done, orc.done_latch.astype(bool), f"{what}: done latch")


def compare_stats(N, counters, sums, tr, ncons, extrema, what, lohi=None, reward_sum=True):
    """Counters [:6], per-constraint counters, episode statistics and fp64 sums of one window against the tracker
    (reward_sum=False: not the fp64 reward-sum slot, which only the fused rollouts fill)."""
    orc = tr.orc
    assert counters[:6].tolist() == orc.stats[:6].tolist(), (what, counters[:8], orc.stats[:8])
    assert counters[N.ST_CON0:N.ST_CON0 + ncons].tolist() == orc.stats[8:8 + ncons].tolist(), what
    assert (int(counters[N.ST_SUCCESSES]), int(counters[N.ST_EP_LEN_SUM]), int(counters[N.ST_EP_LEN_SQ])) == \
        (tr.succ, tr.len_sum, tr.len_sq), what
    # grid / robot: the kernels sum unrounded fp64 rewards, the oracle hands them back rounded to fp32 (relative 6e-8
    # each): bounded by the magnitude of what was summed, as sums of mixed signs may cancel
    rtol, atol = (1e-9, 1e-6) if tr.reactor else (1e-6, 1e-3)
    _close(sums[0], tr.ret_sum, rtol, atol + rtol * tr.ret_abs, f"{what}: return sum")
    _close(sums[1], tr.ret_sq, rtol, atol, f"{what}: return square sum")
    if reward_sum:
        _close(sums[N.ST_F_REWARD_SUM - 24], tr.rew_sum, rtol, atol + rtol * tr.rew_abs, f"{what}: reward sum")
    if lohi is not None:
        lo, hi = lohi
        if not extrema or tr.lo == np.inf:
            assert lo is None and hi is None, what
        else:
            tol = 1e-15 if tr.reactor else 1e-6
            np.testing.assert_allclose([lo, hi], [tr.lo, tr.hi], rtol=tol, atol=0 if tr.reactor else 1e-3, err_msg=what)


def adversarial(O, kind, rng, s0, n, max_steps, clean_from=None):
    """Entry states that spoil whole warps of the loop invariants of the dedicated kernels (see test_gpu_round2.py),
    episodes about to be truncated, NaN states (and grid states that overflow to NaN) that truncate on their first step,
    so that a NaN return reaches the fp64 sums of the first launch only. Special envs are drawn from [0, clean_from)."""
    st = s0.copy()
    ep_step = np.zeros(n, np.int32)
    m = n if clean_from is None else clean_from

    def some(k):
        return rng.choice(m, k, replace=False)
    if kind == O.REACTOR:
        st[some(40), 8] = 1.0                      # e-stop already tripped
        st[some(40), 9] = 1.0                      # alarm latched (inside the invariant)
        st[some(10), 8] = 0.3                      # fractional and negative-zero latches
        st[some(10), 9] = 0.7
        st[some(10), 8] = -0.0
        st[some(10), 9] = -0.0
        st[some(30), 0] = rng.uniform(350.0, 356.0, 30).astype(np.float32)     # over the temperature limit
        st[some(30), 1] = rng.uniform(5.0e5, 5.2e5, 30).astype(np.float32)     # around the pressure limit
        st[some(10), 0] = 150.0                    # outside the 200 .. 350 K entry range
        st[some(10), 5] = rng.choice([0.0, 1e-35, 49.0, 50.0, 3e30], 10).astype(np.float32)
        st[some(5), 4] = 0.0
    elif kind == O.GRID:
        st[some(40), 0] = rng.uniform(-1.2, 1.2, 40).astype(np.float32)
        st[some(6), 0] = np.array([0.5, -0.5, 1.0, -1.0, -0.0, 0.49999997], np.float32)
        i = some(40); st[i, 1 + rng.integers(0, 8, 40)] = rng.uniform(0.88, 1.12, 40).astype(np.float32)
        i = some(30); st[i, 9 + rng.integers(0, 8, 30)] = rng.choice([0.0, -0.0, 100.0, 99.5, 0.4, 100.5, -3.0, 1e-30], 30).astype(np.float32)
        i = some(20); st[i, 17 + rng.integers(0, 8, 20)] = rng.choice([0.0, -0.0, 1e-20, 0.3, 1e30, 3e38, -2.0], 20).astype(np.float32)
        brink = i                                  # (huge generation overflows to inf / NaN: truncate these on the first step)
        w = 32 * 7                                 # one warp with zero imbalance and zero frequency (division guard)
        st[w:w + 32, 0] = 0.0; st[w:w + 32, 9:17] = 50.0; st[w:w + 32, 17:25] = 50.0
    else:
        i = some(40); st[i, :3] = rng.uniform(-0.9, 0.9, (40, 3)).astype(np.float32)        # end effector near / past the workspace
        i = some(40); st[i, 7 + rng.integers(0, 7, 40)] = rng.uniform(-np.pi, np.pi, 40).astype(np.float32)
        i = some(30); st[i, 18 + rng.integers(0, 3, 30)] = rng.choice([0.0, -0.0, 49.9, 50.0, 79.0, 81.0, -60.0], 30).astype(np.float32)
    ep_step[some(200)] = rng.integers(max(0, max_steps - 60), max_steps, 200)
    nan = some(3)
    st[nan, 0] = np.nan
    ep_step[nan] = max_steps - 1
    if kind == O.GRID:
        ep_step[brink] = max_steps - 1
    return st, ep_step
