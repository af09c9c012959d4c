"""GPU parity of the float polygon NMS / rotated-box overlaps (csrc/poly_f32.cu; SURVEY rows A14, B4) against the reference's
own kernels, DOTA_devkit/poly_nms_gpu/*.cu compiled unmodified for sm_100a (oracle/build_ref.build_polygpu), whose outputs on
the seeded inputs below are stored in tests/golden/ref_kernels_golden.npz (tests/refgolden.py): IoU matrices bit for bit, keep
lists equal - through the devkit's host-pointer C ABI (`_poly_nms`, `_overlaps`), and through the device-pointer ops behind
nms_rotated_ext.nms_poly."""
import ctypes

import numpy as np
import pytest
import torch

from tests.boxgen import rboxes
from tests.polygen import merge_dets
from tests.refgolden import assert_bit_equal, ref

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


OVERLAP_CASES = ((0, 300, 257, 600.0), (1, 64, 1000, 200.0), (2, 1, 1, 50.0))
POLY_NMS_CASES = [(1, 0, 0.3), (63, 1, 0.1), (64, 2, 0.3), (65, 3, 0.5), (3000, 4, 0.3), (5000, 5, 0.1)]


def _rboxes5(n, span, seed, degenerate=True):
    d, _, _ = rboxes(n, span, seed, class_offset=False, theta_grid=False)
    if degenerate and n >= 8:
        d[1] = d[0]                      # identical boxes
        d[2, 2:4] = 0.0                  # zero-area box: union == 0 against itself -> (inter + 1) / (union + 1)
        d[3] = d[2]
        d[4, 4] = 0.0                    # axis-aligned
        d[5] = d[4]
        d[5, 0] += d[4, 2]               # touching along an edge
        d[6, 2:4] = 1e-3                 # tiny
    return d


def overlap_inputs(seed, n, k, span):
    b, q = _rboxes5(n, span, seed), _rboxes5(k, span, 100 + seed)
    if n > 8 and k > 8:
        q[:8] = b[:8]
    return b, q


def test_overlaps_bit_exact_host_abi_and_device_op():
    from yolov5_obb_b200.devkit import poly_overlaps, poly_overlaps_device
    for seed, n, k, span in OVERLAP_CASES:
        b, q = overlap_inputs(seed, n, k, span)
        got = poly_overlaps(b, q)
        assert got.shape == (n, k)
        assert_bit_equal(got, f"overlaps/{seed}")
        assert (got > 0.05).mean() > 0.01, "the case must contain overlapping pairs"
        dev = poly_overlaps_device(torch.from_numpy(b).to(DEV), torch.from_numpy(q).to(DEV)).cpu().numpy()
        assert np.array_equal(dev.view(np.uint32), got.view(np.uint32))


def _sorted_dets(n, seed):
    d = merge_dets(n, seed).astype(np.float32)
    return np.ascontiguousarray(d[np.argsort(-d[:, 8], kind="stable")])


@pytest.mark.parametrize("n,seed,thr", POLY_NMS_CASES)
def test_poly_nms_keep_lists_equal_reference(n, seed, thr):
    from yolov5_obb_b200 import _lib
    from yolov5_obb_b200.devkit import poly_gpu_nms
    from yolov5_obb_b200.nms_rotated import nms_poly, poly_nms
    d = _sorted_dets(n, seed)
    want = ref(f"poly_nms/{n}_{seed}_{thr}")
    assert n < 100 or 0 < len(want) < n
    # (1) the devkit's host-pointer C ABI (K3 contract: the caller's order is the processing order)
    got = np.zeros(n, np.int32)
    gnum = ctypes.c_int(0)
    _lib.lib().y5obb_devkit_poly_nms(got.ctypes.data, ctypes.addressof(gnum), d.ctypes.data, n, 9, thr, 0)
    assert gnum.value == len(want) and np.array_equal(got[:gnum.value], want)
    # (2) the .pyx-level function on UNSORTED input (host argsort as the .pyx) and (3) the device op behind nms_poly (K2): both
    # return indices into the caller's order
    perm = np.random.default_rng(seed).permutation(n)
    shuffled = np.ascontiguousarray(d[perm])
    exp = [int(np.flatnonzero(perm == i)[0]) for i in want]          # where the kept sorted rows sit in the shuffled array
    assert poly_gpu_nms(shuffled, thr) == exp
    k2 = nms_poly(torch.from_numpy(shuffled).to(DEV), thr).cpu().tolist()
    assert k2 == exp
    dets_k, inds = poly_nms(torch.from_numpy(shuffled).to(DEV), thr)
    assert inds.cpu().tolist() == exp and dets_k.shape == (len(exp), 9)


def test_poly_nms_edge_cases():
    from yolov5_obb_b200.nms_rotated import nms_poly, poly_nms
    assert nms_poly(torch.zeros((0, 9), device=DEV), 0.3).numel() == 0
    with pytest.raises(NotImplementedError):
        poly_nms(torch.zeros((3, 9)), 0.3)                            # CPU tensor: the reference raises too (wrapper.py:62-63)
    with pytest.raises(RuntimeError):
        nms_poly(torch.zeros((3, 8), device=DEV), 0.3)
    # all-identical polygons: only the top score survives; disjoint polygons: all survive, in score order
    one = np.array([0, 0, 10, 0, 10, 10, 0, 10], np.float32)
    same = np.concatenate([np.tile(one, (70, 1)), np.linspace(0.1, 0.9, 70, dtype=np.float32)[:, None]], 1)
    assert nms_poly(torch.from_numpy(same).to(DEV), 0.5).cpu().tolist() == [69]
    apart = same.copy()
    apart[:, 0:8:2] += (np.arange(70, dtype=np.float32) * 50)[:, None]
    assert nms_poly(torch.from_numpy(apart).to(DEV), 0.5).cpu().tolist() == list(range(69, -1, -1))
