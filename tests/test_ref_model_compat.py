"""INTEGRATION.md B3: the engine plans a model from module class NAMES and a fixed set of attributes, so it accepts the
reference's own `models.yolo.Model` object as well as the mirror.  The engine's view of the reference Model (n / s / m) is
stored in tests/golden/ref_model_view.json (tests/golden/make_ref_model_golden.py); the mirror built from the same yaml must
give the identical view attribute by attribute, and a state_dict of the reference's names and shapes must load into it
strictly."""
import json
from pathlib import Path

import torch

from yolov5_obb_b200.yolo import Model as MirrorModel

ROOT = Path(__file__).resolve().parents[1]


def conv_view(m):
    """what engine._conv_params / add_conv read of a Conv module"""
    c = m.conv
    return ("Conv", c.in_channels, c.out_channels, tuple(c.kernel_size), tuple(c.stride), tuple(c.padding), c.groups,
            c.bias is None, type(m.bn).__name__, float(m.bn.eps), type(m.act).__name__)


def engine_view(model):
    out = []
    for m in model.model:
        kind = type(m).__name__
        f = m.f if isinstance(m.f, int) else tuple(m.f)
        row = [kind, m.i, f]
        if kind == "Conv":
            row.append(conv_view(m))
        elif kind == "C3":
            row += [conv_view(m.cv1), conv_view(m.cv2), conv_view(m.cv3),
                    tuple((type(b).__name__, conv_view(b.cv1), conv_view(b.cv2), bool(b.add)) for b in m.m)]
        elif kind == "SPPF":
            k = getattr(m, "k", None)          # (the mirror keeps k, the reference the nn.MaxPool2d: engine.py reads either)
            if k is None:
                k = m.m.kernel_size if isinstance(m.m.kernel_size, int) else m.m.kernel_size[0]
                assert (m.m.stride, m.m.padding) == (1, k // 2)
            row += [conv_view(m.cv1), conv_view(m.cv2), k]
        elif kind == "Upsample":
            row += [m.scale_factor, m.mode]
        elif kind == "Concat":
            row.append(m.d)
        elif kind == "Detect":
            row += [m.nc, m.no, m.nl, m.na, tuple(m.anchors.shape), [round(float(s), 6) for s in m.stride],
                    [round(float(a), 5) for a in m.anchors.flatten()],
                    tuple((c.in_channels, c.out_channels, tuple(c.kernel_size)) for c in m.m)]
        else:
            raise AssertionError(f"module kind {kind} is not one the engine plans")
        out.append(tuple(row))
    return out


def describe(model):
    """What the check compares, in the form the JSON file holds: the engine's view, the strides, and per state_dict entry its
    name, shape and whether it is a parameter (not a buffer)."""
    params = {k for k, _ in model.named_parameters()}
    return json.loads(json.dumps({
        "stride": [round(float(s), 6) for s in model.stride],
        "engine_view": engine_view(model),
        "state_dict": [[k, list(v.shape), k in params] for k, v in model.state_dict().items()],
    }))


def test_engine_view_of_reference_model_equals_mirror():
    golden = json.loads((ROOT / "tests" / "golden" / "ref_model_view.json").read_text())
    for size in ("n", "s", "m"):
        ref = golden[size]
        torch.manual_seed(0)
        mir = MirrorModel(f"yolov5{size}.yaml", ch=3, nc=15)
        got = describe(mir)
        assert len(ref["engine_view"]) == len(got["engine_view"]), (len(ref["engine_view"]), len(got["engine_view"]))
        for ra, rb in zip(ref["engine_view"], got["engine_view"]):
            assert ra == rb, f"yolov5{size}: the engine would see\n  reference {ra}\n  mirror    {rb}"
        assert got["stride"] == ref["stride"]
        assert got["state_dict"] == ref["state_dict"]
        mir.load_state_dict({k: torch.zeros(shape) for k, shape, _ in ref["state_dict"]}, strict=True)
