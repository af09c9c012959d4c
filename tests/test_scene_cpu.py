"""CPU tests of whole-scene detection (yolov5_obb_b200/scene.py): the tile origins and the host restatement of the merge
(oracle/scene_ref.py) against what the reference's own DOTA devkit code produced (tests/golden/scene_golden.npz, written by
tests/golden/make_scene_golden.py), and argument checking."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import scene_ref
from yolov5_obb_b200.scene import SceneDetector, split_origins

ROOT = Path(__file__).resolve().parents[1]


def _golden():
    return np.load(ROOT / "tests" / "golden" / "scene_golden.npz")


def golden_lines(G):
    """{(scene name, class): [merged line, ...]} of the reference's per-class merged files."""
    out = {}
    for c in range(int(G["nc"])):
        for line in G[f"lines{c}"].tolist():
            out.setdefault((line.split(" ", 1)[0], c), []).append(line)
    return out


def test_split_origins_equal_imgsplit():
    G = _golden()
    off = 0
    for (h, w), k in zip(G["split_sizes"].tolist(), G["split_counts"].tolist()):
        want = [tuple(p) for p in G["split_origins"][off:off + k].tolist()]
        off += k
        assert split_origins(h, w, 1024, 200) == want, (h, w)
        assert scene_ref.split_origins(h, w, 1024, 200) == want, (h, w)


def test_split_origins_examples():
    assert [l for l, _ in split_origins(500, 4000)] == [0, 824, 1648, 2472, 2976]
    assert [l for l, _ in split_origins(500, 1848)] == [0, 824]
    assert split_origins(1024, 1024) == [(0, 0)]
    assert split_origins(600, 800) == [(0, 0)]


def test_oracle_merge_equals_reference_lines():
    G = _golden()
    names = G["scene_names"].tolist()
    nc = int(G["nc"])
    tiles = [G["det7"][t, :G["counts"][t]] for t in range(len(G["counts"]))]
    rows = scene_ref.tiles_to_scene(tiles, G["origins"].tolist())
    sid = np.repeat(G["scene_of"], G["counts"])
    merged = scene_ref.merge(rows, sid, len(names), nc, 0.2)
    want = golden_lines(G)
    got = {}
    for s, name in enumerate(names):
        for c in range(nc):
            r = merged[s][merged[s][:, 9] == c]
            if len(r):
                got[(name, c)] = scene_ref.format_lines(name, r[:, :9])
    assert got == want


@pytest.mark.parametrize("bad", [dict(gap=1024), dict(gap=2000), dict(gap=-1)])
def test_split_origins_rejects_bad_gap(bad):
    with pytest.raises(ValueError):
        split_origins(2000, 2000, 1024, **bad)


@pytest.mark.parametrize("hw", [(0, 100), (100, 0), (-5, 10)])
def test_split_origins_rejects_empty_scene(hw):
    with pytest.raises(ValueError):
        split_origins(*hw)


def _model():
    from tests.modelgen import build_mirror
    return build_mirror("n", nc=15, seed=0)


def test_scene_detector_rejects_bad_configuration():
    m = _model()
    with pytest.raises(ValueError):
        SceneDetector(m, subsize=1000)          # not a multiple of the max stride 32
    with pytest.raises(ValueError):
        SceneDetector(m, subsize=1024, gap=1024)
    with pytest.raises(ValueError):
        SceneDetector(m, batch=0)
    m.train()
    with pytest.raises(RuntimeError):
        SceneDetector(m)


def test_scene_detector_rejects_bad_scenes():
    det = SceneDetector(_model())
    with pytest.raises(RuntimeError):           # a CPU tensor: there is no CPU path
        det.detect(torch.zeros((100, 100, 3), dtype=torch.uint8))
    with pytest.raises(TypeError):
        det.detect(np.zeros((100, 100, 3), np.uint8))
    with pytest.raises(TypeError):
        det.detect(torch.zeros((100, 100, 3), dtype=torch.float32))
    with pytest.raises(ValueError):              # CHW instead of HWC
        det.detect(torch.zeros((3, 100, 100), dtype=torch.uint8))
    with pytest.raises(ValueError):
        det.detect(torch.zeros((100, 100), dtype=torch.uint8))
