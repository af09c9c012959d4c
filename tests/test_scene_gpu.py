"""GPU tests of whole-scene detection (yolov5_obb_b200/scene.py):
1. the scene stem (y5obb_stem_s2d_scene_u8) is bit-identical to host crops + y5obb_stem_s2d_u8;
2. the segmented polygon NMS keeps, per segment, exactly what the single-list device NMS and the host oracle keep;
3. the merge stage reproduces the reference devkit's merged lines (tests/golden/scene_golden.npz);
4. SceneDetector.detect equals the host composition of the existing pieces, exactly."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import scene_ref
from tests.test_scene_cpu import golden_lines

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
DEV = "cuda:0"
TILE = 1024


def _scene(h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, generator=g)


def _s2d(B):
    return torch.zeros((B, TILE // 2, TILE // 2 + 2, 16), dtype=torch.bfloat16, device=DEV)


@pytest.mark.parametrize("hw", [(600, 800), (1024, 1024), (1111, 2057), (3000, 4000)])
def test_stem_scene_bit_equal_to_host_crop(hw):
    from yolov5_obb_b200 import _lib
    from yolov5_obb_b200.scene import split_origins
    h, w = hw
    scene = _scene(h, w, h * 7 + w)
    org = split_origins(h, w, TILE, 200)
    n, B = len(org), len(org) + 3            # three invalid tiles at the tail
    origins = torch.zeros((B, 2), dtype=torch.int32)
    origins[:n] = torch.tensor(org, dtype=torch.int32)
    L, st = _lib.lib(), _lib.stream_ptr(DEV)
    got = _s2d(B)
    sd = scene.to(DEV)
    _lib.check(L.y5obb_stem_s2d_scene_u8(sd.data_ptr(), h, w, origins.to(DEV).data_ptr(), B, n, TILE, got.data_ptr(), 1, st),
               "y5obb_stem_s2d_scene_u8")
    crops = np.zeros((B, 3, TILE, TILE), np.uint8)
    crops[:n] = scene_ref.crop_tiles(scene.numpy(), org, TILE)
    x = torch.from_numpy(crops).to(DEV)
    want = _s2d(B)
    _lib.check(L.y5obb_stem_s2d_u8(x.data_ptr(), want.data_ptr(), B, TILE, TILE, 1, st), "y5obb_stem_s2d_u8")
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert not got[n:].any()
    # the cases cover interior tiles (away from every edge), edge tiles and tiles clamped back inside the scene
    if h > 2 * TILE:
        assert any(0 < l and l + TILE < w and 0 < u and u + TILE < h for l, u in org)
    if w > TILE:
        assert org[-1][0] == w - TILE


def _segments(sizes, seed):
    """Rows of several segments, interleaved: dets [n, 9] fp64, seg int32 [n]."""
    from tests.polygen import merge_dets
    rng = np.random.default_rng(seed)
    parts = [merge_dets(k, seed=seed + s) if k else np.zeros((0, 9)) for s, k in enumerate(sizes)]
    D = np.concatenate(parts, 0)
    seg = np.concatenate([np.full(k, s, np.int32) for s, k in enumerate(sizes)])
    perm = rng.permutation(len(D))
    return D[perm], seg[perm]


@pytest.mark.parametrize("thr", [0.1, 0.2, 0.5])
def test_segmented_nms_equals_per_segment_nms(thr):
    from yolov5_obb_b200.devkit import py_cpu_nms_poly_fast
    from yolov5_obb_b200.scene import poly_nms_segmented
    sizes = [1, 63, 64, 0, 65, 2100, 0, 7, 300, 128, 2, 0] + [5] * 20
    D, seg = _segments(sizes, seed=int(thr * 10))
    Dd, segd = torch.from_numpy(D).to(DEV), torch.from_numpy(seg).to(DEV)
    keep, off = poly_nms_segmented(Dd, segd, sizes, thr)
    off = off.cpu().tolist()
    keep = keep[:off[-1]].cpu().numpy()
    assert off[0] == 0 and all(a <= b for a, b in zip(off, off[1:]))
    for s, k in enumerate(sizes):
        idx = np.where(seg == s)[0]
        got = keep[off[s]:off[s + 1]]
        assert len(idx) == k
        if k == 0:
            assert len(got) == 0
            continue
        alone = py_cpu_nms_poly_fast(torch.from_numpy(D[idx]).to(DEV), thr).cpu().numpy()
        assert got.tolist() == idx[alone].tolist(), (s, k)
        if k <= 300:
            assert got.tolist() == idx[scene_ref.nms_poly_stable(D[idx], thr)].tolist(), (s, k)


def test_merge_stage_reproduces_reference_lines():
    from yolov5_obb_b200.scene import merge_tiles
    G = np.load(ROOT / "tests" / "golden" / "scene_golden.npz")
    names, nc = G["scene_names"].tolist(), int(G["nc"])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    merged = merge_tiles(t(G["det7"]), t(G["counts"]), t(G["origins"]), t(G["scene_of"]), len(names), nc, 0.2)
    got = {}
    for s, name in enumerate(names):
        r = merged[s].cpu().numpy()
        assert np.all(np.diff(r[:, 9]) >= 0)   # grouped by class, ascending
        for c in range(nc):
            rc = r[r[:, 9] == c]
            if len(rc):
                got[(name, c)] = scene_ref.format_lines(name, rc[:, :9])
    assert got == golden_lines(G)


def _host_composition(model, scenes, det_kw, batch, merge_iou):
    """host crop -> existing detect_records + non_max_suppression_obb -> rbox2poly + offsets -> py_cpu_nms_poly_fast per
    (scene, class), all with the existing entry points."""
    from yolov5_obb_b200.devkit import py_cpu_nms_poly_fast
    from yolov5_obb_b200.general import non_max_suppression_obb
    from yolov5_obb_b200.rboxs_utils import rbox2poly
    from yolov5_obb_b200.scene import split_origins
    nc = model.model[-1].nc
    tiles, where = [], []
    for k, s in enumerate(scenes):
        org = split_origins(s.shape[0], s.shape[1], TILE, 200)
        tiles.append(scene_ref.crop_tiles(s.cpu().numpy(), org, TILE))
        where += [(k, l, u) for l, u in org]
    tiles = np.concatenate(tiles, 0)
    rows = []   # (scene, cls, [9] fp64) in tile order, row order
    for b0 in range(0, len(tiles), batch):
        x = np.zeros((batch, 3, TILE, TILE), np.uint8)
        x[:len(tiles[b0:b0 + batch])] = tiles[b0:b0 + batch]
        packed, counts = non_max_suppression_obb(model.detect_records(torch.from_numpy(x).to(DEV)), return_packed=True, **det_kw)
        for j in range(min(batch, len(tiles) - b0)):
            d = packed[j, :counts[j]]
            k, l, u = where[b0 + j]
            poly = rbox2poly(d[:, :5].contiguous()).double()
            poly[:, 0::2] += l
            poly[:, 1::2] += u
            r9 = torch.cat([poly, d[:, 5:6].double()], 1)
            rows += [(k, int(c), r9[i]) for i, c in enumerate(d[:, 6].tolist())]
    out = []
    for k in range(len(scenes)):
        parts = []
        for c in range(nc):
            seg = [r for s, cc, r in rows if s == k and cc == c]
            if seg:
                D = torch.stack(seg)
                kept = D[py_cpu_nms_poly_fast(D, merge_iou)]
                parts.append(torch.cat([kept, torch.full((len(kept), 1), float(c), dtype=torch.float64, device=DEV)], 1))
        out.append(torch.cat(parts, 0) if parts else torch.zeros((0, 10), dtype=torch.float64, device=DEV))
    return out


def test_scene_detector_equals_host_composition():
    from tests.modelgen import calibrated_bench_model
    from tests.tilegen import synth_tiles
    from yolov5_obb_b200.scene import SceneDetector
    model = calibrated_bench_model("s", nc=15, seed=0, conf=0.25).to(DEV)
    # two scenes, 6 + 9 tiles: 15 tiles in batches of 4 (not a multiple; batches span both scenes)
    scenes = []
    for k, (h, w) in enumerate([(1500, 2600), (2000, 2000)]):
        img = synth_tiles(1, max(h, w), seed=50 + k)[0, :, :h, :w]
        scenes.append(img.flip(0).permute(1, 2, 0).contiguous().to(DEV))   # RGB CHW -> BGR HWC
    kw = dict(conf_thres=0.25, iou_thres=0.4, max_det=1500, multi_label=True)
    det = SceneDetector(model, batch=4, merge_iou=0.2, **kw)
    want = _host_composition(model, scenes, kw, 4, 0.2)
    assert sum(len(w) for w in want) > 0
    for _ in range(2):   # the second call replays the captured plan and post-process graphs
        got = det.detect(scenes)
        assert len(got) == 2
        for g, w in zip(got, want):
            assert g.dtype == torch.float64 and g.shape[1] == 10
            assert torch.equal(g, w), (g.shape, w.shape)
    one = det.detect(scenes[1])
    assert torch.equal(one[0], want[1])
