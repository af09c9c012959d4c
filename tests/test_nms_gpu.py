"""GPU parity tests for the rotated-NMS path, called through the C ABI (ctypes -> liby5obb.so).

Oracles, strongest first:
  1. the reference's own kernels compiled for sm_100a (nms_rotated_cuda = K1 + host scan, and the
     single_box_iou_rotated device function): bit-exact.  Their outputs on the seeded inputs below are stored in
     tests/golden/ref_kernels_golden.npz (tests/refgolden.py).
  2. oracle/liboracle.so — scalar C++ restatement (no FMA): IoU within 1e-5, keep lists equal on
     inputs whose decisive IoUs are not within 1e-4 of the threshold.
  3. tests/golden/*.npz — fixtures produced by the reference CPU extension (tests/golden/make_golden.py).
"""
from pathlib import Path

import numpy as np
import pytest
import torch

import oracle
from tests.boxgen import rboxes, degenerate_pairs
from tests.refgolden import assert_bit_equal, keep_from_bits, ref

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
DEV = "cuda:0"


KEEP_CASES = [(1, 100, 0), (63, 200, 1), (64, 200, 2), (65, 200, 3), (1000, 300, 4), (5000, 1024, 5), (30000, 1024, 6),
              (4097, 16384, 7)]
THRESHOLDS = [0.1, 0.2, 0.45, 0.7]


def _nms(d, s, thr, **kw):
    from yolov5_obb_b200.nms_rotated import nms_rotated
    return nms_rotated(torch.from_numpy(d).to(DEV), torch.from_numpy(s).to(DEV), thr, **kw).cpu().numpy()


def _our_iou_pairs(a, b):
    from yolov5_obb_b200.nms_rotated import rbox_iou_pairs
    return rbox_iou_pairs(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV)).cpu().numpy()


def _near_pairs(n, seed, theta_grid):
    """Pairs that actually overlap: b is a perturbed copy of a."""
    rng = np.random.default_rng(seed)
    a, _, _ = rboxes(n, 1024, seed, class_offset=True, theta_grid=theta_grid)
    b = a.copy()
    b[:, :2] += rng.normal(0, 1, (n, 2)).astype(np.float32) * (a[:, 3:4] * 0.5)
    b[:, 2:4] *= rng.uniform(0.6, 1.5, (n, 2)).astype(np.float32)
    if theta_grid:
        b[:, 4] = ((rng.integers(0, 180, n) - 90) / 180 * 3.141592).astype(np.float32)
    else:
        b[:, 4] += rng.normal(0, 0.3, n).astype(np.float32)
    same = rng.random(n) < 0.05
    b[same] = a[same]  # exact duplicates
    return a, b


@pytest.mark.parametrize("theta_grid", [True, False])
def test_iou_bitexact_vs_reference_device_function(theta_grid):
    a, b = _near_pairs(400_000, 11, theta_grid)
    ours = _our_iou_pairs(a, b)
    assert_bit_equal(ours, f"iou/{int(theta_grid)}")
    assert (ours > 0).mean() > 0.5, "pairs should mostly overlap"


def test_iou_degenerate_bitexact_and_vs_cpu_oracle():
    a, b = degenerate_pairs()
    ours, want = _our_iou_pairs(a, b), ref("iou_degenerate")
    assert np.array_equal(ours.view(np.uint32), want.view(np.uint32)), (ours, want)
    # the CPU restatement agrees except on the last 4 pairs (one rectangle written two ways: all edges
    # parallel/coincident), where FMA contraction changes which candidate points survive — there the
    # reference's own CPU and CUDA builds disagree with each other as well
    cpu = oracle.iou_pairs(a, b, variant=1)
    np.testing.assert_allclose(ours[:-4], cpu[:-4], rtol=0, atol=2e-5)


def test_iou_vs_cpu_oracle_tolerance():
    a, b = _near_pairs(50_000, 5, True)
    ours = _our_iou_pairs(a, b)
    cpu = oracle.iou_pairs(a, b, variant=1)
    np.testing.assert_allclose(ours, cpu, rtol=0, atol=1e-5)  # FMA contraction only


@pytest.mark.parametrize("n,span,seed", KEEP_CASES)
def test_keep_bitexact_vs_reference_cuda_kernel(n, span, seed):
    d, s, _ = rboxes(n, span, seed)
    ours = _nms(d, s, 0.4)
    want = keep_from_bits(ref(f"keep/{n}_{span}_{seed}"), s)
    assert ours.dtype == np.int64
    assert np.array_equal(ours, want), f"n={n}: {len(ours)} vs {len(want)} kept"


def threshold_case():
    return rboxes(8000, 600, 21, n_classes=3)


@pytest.mark.parametrize("thr", THRESHOLDS)
def test_keep_thresholds_vs_reference_cuda_kernel(thr):
    d, s, _ = threshold_case()
    ours = _nms(d, s, thr)
    assert np.array_equal(ours, keep_from_bits(ref(f"thr/{thr}"), s))
    assert len(ours) < 8000  # something is suppressed


def _margin_ok(d, s, thr, keep, mode):
    """True if no decisive IoU (kept i vs any later j) lies within 1e-4 of thr — computed with the CPU oracle."""
    order = np.argsort(-s, kind="stable")
    kept = set(keep.tolist())
    ki = [i for i in order if i in kept]
    # sample: all kept x all boxes is too much for large n; tests call this on n <= 2000
    A = np.repeat(d[ki], len(d), 0)
    B = np.tile(d, (len(ki), 1))
    v = oracle.iou_pairs(A, B, variant=mode)
    return not np.any(np.abs(v - thr) < 1e-4)


@pytest.mark.parametrize("strict", [True, False])
def test_keep_vs_cpu_oracle_both_comparison_rules(strict):
    mode = 1 if strict else 0
    for seed in range(33, 60):
        d, s, _ = rboxes(1500, 400, seed, n_classes=2)
        exp = oracle.nms_rotated(d, s, 0.3, mode=mode)
        if _margin_ok(d, s, 0.3, exp, mode):
            break
    else:
        pytest.skip("no seed without a decisive IoU within 1e-4 of the threshold")
    ours = _nms(d, s, 0.3, strict_gt=strict)
    assert np.array_equal(ours, exp)


def test_ge_vs_gt_differ_on_exact_threshold():
    # two identical boxes: IoU == 1.0 exactly; thr = 1.0 separates `>` from `>=`
    d = np.array([[10, 10, 8, 4, 0.3], [10, 10, 8, 4, 0.3]], np.float32)
    s = np.array([0.9, 0.8], np.float32)
    iou = _our_iou_pairs(d[:1], d[1:])
    if iou[0] != 1.0:
        pytest.skip(f"self IoU rounds to {iou[0]!r}")
    assert _nms(d, s, 1.0, strict_gt=True).tolist() == [0, 1]
    assert _nms(d, s, 1.0, strict_gt=False).tolist() == [0]


def test_golden_fixtures():
    g = np.load(ROOT / "tests" / "golden" / "nms_golden.npz")
    for k in sorted({x.split("/")[0] for x in g.files}):
        d, s, thr = g[f"{k}/dets"], g[f"{k}/scores"], float(g[f"{k}/thr"])
        if k.startswith("kat"):
            # SURVEY 8(c) known-answer boxes: 2 and 3 are the same square written two ways, a degenerate
            # pair on which the reference's own CPU and CUDA arithmetic disagree (FMA contraction), so the
            # device result is pinned to the reference CUDA kernel, not to the CPU fixture
            assert np.array_equal(_nms(d, s, thr, strict_gt=True), keep_from_bits(ref(f"kat/{k}"), s)), k
            continue
        # fixtures hold the reference CPU extension's keep (>=, host hull); margin-checked at creation
        ours = _nms(d, s, thr, strict_gt=False)
        assert np.array_equal(ours, g[f"{k}/keep_cpu"]), k


def test_edge_cases():
    from yolov5_obb_b200.nms_rotated import nms_rotated, obb_nms
    e = torch.zeros((0, 5), device=DEV)
    assert nms_rotated(e, torch.zeros(0, device=DEV), 0.4).numel() == 0
    dd, ii = obb_nms(e, torch.zeros(0, device=DEV), 0.4)
    assert dd.shape == (0, 5) and ii.numel() == 0
    # all too small -> nothing (nms_rotated_wrapper.py:33-34)
    d = torch.tensor([[1, 1, 1e-4, 5, 0], [2, 2, 5, 1e-5, 0]], device=DEV)
    dd, ii = obb_nms(d, torch.tensor([0.5, 0.6], device=DEV), 0.4)
    assert ii.numel() == 0 and dd.shape == (0, 5)
    # some too small: indices refer to the unfiltered input (wrapper.py:36-42), inds is a CPU tensor
    d = torch.tensor([[1, 1, 1e-4, 5, 0], [20, 20, 5, 3, 0], [20, 20, 5, 3, 0.01], [90, 90, 4, 4, 0]], device=DEV)
    s = torch.tensor([0.99, 0.5, 0.6, 0.1], device=DEV)
    dd, ii = obb_nms(d, s, 0.4)
    assert ii.device.type == "cpu" and ii.dtype == torch.int64
    assert ii.tolist() == [2, 3]
    assert torch.equal(dd.cpu(), d.cpu()[ii])
    # ties: lower index first
    d = torch.tensor([[0, 0, 2, 2, 0], [100, 0, 2, 2, 0], [200, 0, 2, 2, 0]], device=DEV, dtype=torch.float32)
    s = torch.tensor([0.5, 0.5, 0.5], device=DEV)
    assert nms_rotated(d, s, 0.4).tolist() == [0, 1, 2]
    # numpy path (wrapper.py:20-24) returns numpy
    dn, sn, _ = rboxes(100, 100, 9)
    dd, ii = obb_nms(dn, sn, 0.4, device_id=0)
    assert isinstance(ii, np.ndarray) and np.array_equal(ii, oracle.obb_nms(dn, sn, 0.4, mode=1))
    # wrong device -> loud failure, no CPU fallback
    with pytest.raises(RuntimeError):
        nms_rotated(torch.zeros((3, 5)), torch.zeros(3), 0.4)


def test_batched_equals_per_image():
    from yolov5_obb_b200 import _lib
    L = _lib.lib()
    B = 5
    parts = [rboxes(n, 500, 40 + i) for i, n in enumerate([700, 0, 64, 3000, 129])]
    d = np.concatenate([p[0] for p in parts])
    s = np.concatenate([p[1] for p in parts])
    img = np.concatenate([np.full(len(p[0]), i, np.int32) for i, p in enumerate(parts)])
    perm = np.random.default_rng(0).permutation(len(d))  # image ids arrive in any order
    d, s, img = d[perm], s[perm], img[perm]
    td, ts, ti = (torch.from_numpy(x).to(DEV) for x in (d, s, img))
    n = len(d)
    keep = torch.empty(n, dtype=torch.int64, device=DEV)
    cnt = torch.empty(B, dtype=torch.int64, device=DEV)
    off = torch.empty(B + 1, dtype=torch.int64, device=DEV)
    ws = torch.empty(L.y5obb_nms_workspace_bytes(n, B, 3000), dtype=torch.uint8, device=DEV)
    for max_keep in (0, 50):
        rc = L.y5obb_nms_rotated_batched_f32(td.data_ptr(), ts.data_ptr(), ti.data_ptr(), n, B, 3000, 0.4, 1, max_keep,
                                             keep.data_ptr(), cnt.data_ptr(), off.data_ptr(), ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        cnt_h, off_h, keep_h = cnt.cpu().numpy(), off.cpu().numpy(), keep.cpu().numpy()
        for b in range(B):
            idx = np.flatnonzero(img == b)
            exp = idx[oracle.nms_rotated(d[idx], s[idx], 0.4, mode=1)] if len(idx) else np.zeros(0, np.int64)
            if max_keep:
                exp = exp[:max_keep]
            got = keep_h[off_h[b]:off_h[b] + cnt_h[b]]
            assert np.array_equal(got, exp), (b, max_keep, len(got), len(exp))
    # capacity violation is reported, not overrun: claim max_per_image = 64 while an image holds 3000
    ws2 = torch.empty(L.y5obb_nms_workspace_bytes(n, B, 64), dtype=torch.uint8, device=DEV)
    rc = L.y5obb_nms_rotated_batched_f32(td.data_ptr(), ts.data_ptr(), ti.data_ptr(), n, B, 64, 0.4, 1, 0,
                                         keep.data_ptr(), cnt.data_ptr(), off.data_ptr(), ws2.data_ptr(), ws2.numel(),
                                         torch.cuda.current_stream().cuda_stream)
    assert rc == 0 and (cnt.cpu().numpy() == -1).all()


def cluster_case():
    """Five images of 45 000, 0, 64, 5 000 and 41 000 boxes, their image ids in a seeded random order."""
    sizes = [45000, 0, 64, 5000, 41000]
    parts = [rboxes(n, 1024, 60 + i) for i, n in enumerate(sizes)]
    d = np.concatenate([p[0] for p in parts])
    s = np.concatenate([p[1] for p in parts])
    img = np.concatenate([np.full(len(p[0]), i, np.int32) for i, p in enumerate(parts)])
    perm = np.random.default_rng(1).permutation(len(d))
    return d[perm], s[perm], img[perm], len(sizes)


def test_batched_cluster_scan_equals_reference_kernel():
    """Images with >= 40 960 boxes take the cluster form of the greedy scan (k_reduce_cluster: 8 CTAs per image sharing the
    removed-set through distributed shared memory), smaller ones the single CTA - in the same batched call.  Checker: the
    reference's own CUDA kernel K1 per image (stored keep lists; the CPU oracle needs n x kept pair tests, minutes at this
    size), with and without max_keep."""
    from yolov5_obb_b200 import _lib
    L = _lib.lib()
    d, s, img, B = cluster_case()
    td, ts, ti = (torch.from_numpy(x).to(DEV) for x in (d, s, img))
    n = len(d)
    keep = torch.empty(n, dtype=torch.int64, device=DEV)
    cnt = torch.empty(B, dtype=torch.int64, device=DEV)
    off = torch.empty(B + 1, dtype=torch.int64, device=DEV)
    ws = torch.empty(L.y5obb_nms_workspace_bytes(n, B, 45000), dtype=torch.uint8, device=DEV)
    exp = []
    for b in range(B):
        idx = np.flatnonzero(img == b)
        exp.append(idx[keep_from_bits(ref(f"cluster/{b}"), s[idx])])
    for max_keep in (0, 700):
        rc = L.y5obb_nms_rotated_batched_f32(td.data_ptr(), ts.data_ptr(), ti.data_ptr(), n, B, 45000, 0.4, 1, max_keep,
                                             keep.data_ptr(), cnt.data_ptr(), off.data_ptr(), ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        cnt_h, off_h, keep_h = cnt.cpu().numpy(), off.cpu().numpy(), keep.cpu().numpy()
        for b in range(B):
            want = exp[b][:max_keep] if max_keep else exp[b]
            got = keep_h[off_h[b]:off_h[b] + cnt_h[b]]
            assert np.array_equal(got, want), (b, max_keep, len(got), len(want))


def test_full_size_properties():
    """BASELINE config 4 at full size (200k boxes, 15 classes): size-independent properties.
    idempotence: NMS of the kept set keeps everything; sortedness: keep is score-descending;
    independence: no two kept boxes overlap above thr (sampled); class separation: per-class NMS of a
    class subset equals the restriction of the global keep."""
    n = 200_000
    d, s, cls = rboxes(n, 1024, 77)
    keep = _nms(d, s, 0.4)
    assert len(np.unique(keep)) == len(keep)
    assert np.all(np.diff(s[keep]) < 0)
    again = _nms(d[keep], s[keep], 0.4)
    assert np.array_equal(again, np.arange(len(keep)))
    for c in (0, 7, 14):
        idx = np.flatnonzero(cls == c)
        sub = idx[_nms(d[idx], s[idx], 0.4)]
        assert np.array_equal(sub, keep[cls[keep] == c])
    # the top-scoring box of every class is always kept
    for c in range(15):
        idx = np.flatnonzero(cls == c)
        assert idx[np.argmax(s[idx])] in set(keep.tolist())
    # sparse worst case: nothing suppressed
    d2, s2, _ = rboxes(100_000, 2_000_000, 78, class_offset=False)
    k2 = _nms(d2, s2, 0.4)
    exp_sparse = np.argsort(-s2, kind="stable")
    assert len(k2) > 99_000 and np.array_equal(k2, exp_sparse[np.isin(exp_sparse, k2)])
