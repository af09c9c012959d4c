"""CPU tests: the oracle against the committed golden vectors, among them the keep lists of the reference's own CPU
extension (tests/refgolden.py)."""
from pathlib import Path

import numpy as np
import pytest

import oracle
from tests.boxgen import rboxes, degenerate_pairs
from tests.refgolden import keep_from_bits, ref

ROOT = Path(__file__).resolve().parents[1]
PIN_CASES = [(400, 250, 0.4, 0), (1500, 800, 0.3, 1), (900, 5000, 0.45, 2), (257, 100, 0.6, 3)]


def test_oracle_matches_golden_keep_lists():
    g = np.load(ROOT / "tests" / "golden" / "nms_golden.npz")
    names = sorted({x.split("/")[0] for x in g.files})
    assert len(names) >= 9
    for k in names:
        d, s, thr = g[f"{k}/dets"], g[f"{k}/scores"], float(g[f"{k}/thr"])
        assert np.array_equal(oracle.nms_rotated(d, s, thr, mode=0), g[f"{k}/keep_cpu"]), k
        # fixtures are margin-checked, so the CUDA rule (`>`, device hull order) agrees too
        assert np.array_equal(oracle.nms_rotated(d, s, thr, mode=1), g[f"{k}/keep_cpu"]), k


def test_oracle_matches_golden_iou_values():
    g = np.load(ROOT / "tests" / "golden" / "iou_golden.npz")
    assert np.array_equal(oracle.iou_pairs(g["a"], g["b"], 0).view(np.uint32), g["iou_host"].view(np.uint32))
    assert np.array_equal(oracle.iou_pairs(g["a"], g["b"], 1).view(np.uint32), g["iou_devorder"].view(np.uint32))
    # geometry known answers: identical boxes -> 1, disjoint -> 0, zero area -> 0
    a = np.array([[10, 10, 20, 10, 0.3], [0, 0, 1e-8, 1e-8, 0], [5, 5, 2, 2, 0], [0, 0, 4, 2, 0]], np.float32)
    b = np.array([[10, 10, 20, 10, 0.3], [0, 0, 1, 1, 0], [50, 50, 2, 2, 0], [1, 0, 4, 2, 0]], np.float32)
    v = oracle.iou_pairs(a, b, 0)
    assert abs(v[0] - 1.0) < 1e-6 and v[1] == 0.0 and v[2] == 0.0 and abs(v[3] - 0.6) < 1e-6


@pytest.mark.parametrize("n,span,thr,seed", PIN_CASES)
def test_oracle_pinned_to_reference_cpu_extension(n, span, thr, seed):
    d, s, _ = rboxes(n, span, seed, n_classes=4)
    want = keep_from_bits(ref(f"cpu_keep/{n}_{span}_{thr}_{seed}"), s)
    assert np.array_equal(oracle.nms_rotated(d, s, thr, mode=0), want)


def test_obb_nms_wrapper_semantics():
    d = np.array([[1, 1, 1e-4, 5, 0], [20, 20, 5, 3, 0], [20, 20, 5, 3, 0.01], [90, 90, 4, 4, 0]], np.float32)
    s = np.array([0.99, 0.5, 0.6, 0.1], np.float32)
    assert oracle.obb_nms(d, s, 0.4, 1).tolist() == [2, 3]
    assert oracle.obb_nms(d[:1], s[:1], 0.4, 1).tolist() == []
    assert oracle.nms_rotated(np.zeros((0, 5), np.float32), np.zeros(0, np.float32), 0.4).tolist() == []
