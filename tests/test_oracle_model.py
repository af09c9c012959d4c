"""CPU tests: the mirror Model's parameters/initialisation and the fp32 oracle forward against
golden outputs of the REFERENCE model (tests/golden/model_golden.npz, made by make_model_golden.py)."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import model_ref
from tests.modelgen import build_mirror

ROOT = Path(__file__).resolve().parents[1]
G = np.load(ROOT / "tests" / "golden" / "model_golden.npz")


@pytest.mark.parametrize("size", ["n", "s"])
def test_mirror_init_and_oracle_forward_match_reference(size):
    m = build_mirror(size, nc=15, seed=0)
    # same constructor order -> same RNG stream -> bit-identical parameters (incl. Detect bias init, yolo.py:223-232)
    psum = sum(p.double().sum().item() for p in m.parameters())
    assert abs(psum - float(G[f"{size}/param_sum"])) < 1e-9 * max(1.0, abs(psum))
    x = torch.from_numpy(G[f"{size}/x"])
    pred, _ = model_ref.forward(m, x)
    ref = torch.from_numpy(G[f"{size}/pred"])
    assert pred.shape == ref.shape == (1, 3 * (8 * 12 + 4 * 6 + 2 * 3), 200)
    # 1e-5, or 16 float32 ulps of the value where that is more: the box columns reach ~400 px, where one ulp is 3e-5, and
    # the CPU convolutions' summation order (thread count, instruction set) moves them by a few ulps - one thread instead
    # of eight: up to 4.7 ulps; an fp64 forward differs from the stored fp32 output by up to 3
    tol = (16 * torch.finfo(torch.float32).eps * ref.abs()).clamp_min(1e-5)
    assert ((pred - ref).abs() < tol).all(), (pred - ref).abs().max().item()


def test_model_structure_mirrors_reference():
    from yolov5_obb_b200 import yolo as Y
    for size, nparams in (("n", 2027752), ("s", 7545544), ("m", 21655272), ("x", 87523240)):  # reference Model Summary lines
        m = Y.Model(f"yolov5{size}.yaml", ch=3, nc=15)
        assert sum(p.numel() for p in m.parameters()) == nparams
        assert m.stride.tolist() == [8.0, 16.0, 32.0]
        det = m.model[-1]
        assert det.no == 200 and det.na == 3 and det.nl == 3
        assert m.save == [4, 6, 10, 14, 17, 20, 23]
    with pytest.raises(RuntimeError):
        m.eval()(torch.zeros(1, 3, 64, 64))  # CPU tensor: no fallback
