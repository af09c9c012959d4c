"""INTEGRATION.md B3, option 2 ("keep the reference Model object, replace _forward_once by InferenceEngine"): the engine
identifies modules by class NAME and reads a fixed set of attributes (engine.py).  This script imports the REFERENCE package
(tests/golden/ref_import.py), builds the reference's Model for yolov5n / s / m and writes ref_model_view.json: the engine's
view of it (tests/test_ref_model_compat.engine_view), its strides, and the name, shape and kind of every state_dict entry.
tests/test_ref_model_compat.py checks the mirror against that file.  Re-run:  python tests/golden/make_ref_model_golden.py"""
import json
import sys
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
import ref_import  # noqa: E402

ref_import.setup()
sys.path.insert(0, str(HERE.parents[1]))
from models.yolo import Model as RefModel  # noqa: E402  (the reference)
from tests.test_ref_model_compat import describe  # noqa: E402


def main():
    sizes = []
    for size in ("n", "s", "m"):
        torch.manual_seed(0)
        d = describe(RefModel(f"models/yolov5{size}.yaml", ch=3, nc=15))
        # one layer / one state_dict entry per line
        parts = [f'  "{k}": ' + (json.dumps(v) if k == "stride" else
                                 "[\n" + ",\n".join("   " + json.dumps(r, separators=(",", ":")) for r in v) + "\n  ]")
                 for k, v in d.items()]
        sizes.append(f' "{size}": {{\n' + ",\n".join(parts) + "\n }")
        print(f"yolov5{size}: {len(d['engine_view'])} layers, {len(d['state_dict'])} state_dict entries")
    (HERE / "ref_model_view.json").write_text("{\n" + ",\n".join(sizes) + "\n}\n")


if __name__ == "__main__":
    main()
