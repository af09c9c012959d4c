"""Outputs of the reference's own native kernels on the tests' seeded inputs, stored in tests/golden/ref_kernels_golden.npz
(made by tests/golden/make_ref_kernels_golden.py), and the two forms the file uses for outputs too large to store as they are:
  * keep lists of greedy NMS over boxes with unique scores: one bit per box, in descending score order (keep_bits);
  * large float arrays: the SHA-256 of all their bytes plus every 100th value (sampled), checked by assert_bit_equal."""
import hashlib
from pathlib import Path

import numpy as np

PATH = Path(__file__).resolve().parent / "golden" / "ref_kernels_golden.npz"


def ref(key):
    return np.load(PATH)[key]


def digest(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def keep_bits(keep, scores):
    order = np.argsort(-scores, kind="stable")
    bits = np.isin(order, keep)
    assert np.array_equal(order[bits], keep), "keep list not in descending score order"
    return np.packbits(bits)


def keep_from_bits(bits, scores):
    order = np.argsort(-scores, kind="stable")
    return order[np.unpackbits(bits, count=len(scores)).astype(bool)]


def sampled(a):
    flat = np.ascontiguousarray(a).ravel()
    return {"sha256": digest(flat), "every100": flat[::100].copy()}


def assert_bit_equal(got, key):
    """got equals, bit for bit, the float32 array stored under key in the sampled form."""
    flat = np.ascontiguousarray(got, dtype=np.float32).ravel()
    want = ref(f"{key}/every100")
    bad = 100 * np.flatnonzero(flat[::100].view(np.uint32) != want.view(np.uint32))
    assert bad.size == 0, (f"{key}: {bad.size} of {want.size} sampled values differ bitwise; first at {bad[:5]}: "
                           f"{flat[bad[:5]]} vs {want[bad[:5] // 100]}")
    assert np.array_equal(digest(flat), ref(f"{key}/sha256")), f"{key}: values differ bitwise outside the sample"
