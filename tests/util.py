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
