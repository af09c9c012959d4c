"""Golden data for whole-scene detection (yolov5_obb_b200/scene.py), produced by the REFERENCE's own DOTA devkit code:

* split: DOTA_devkit/ImgSplit_multi_process.py splitbase.SplitSingle (rate 1, subsize 1024, gap 200) on blank scenes of
  several sizes with an empty label file; the patch names it writes (name__1__left___up) give the tile origins.
  shapely is not needed without labels: shapely.geometry is stubbed (only constructed, never used).
* merge: DOTA_devkit/ResultMerge_multi_process.py mergesingle(dst, py_cpu_nms_poly_fast, class_file) on per-class result files
  of seeded tile detections (several scenes, several tiles per scene, objects across tile borders, distinct scores), written
  at full precision so that only the reference's own rounding (coordinates 0.1, conf 0.01) applies.  Its polyiou SWIG module
  does not import on Python 3.12, so DOTA_devkit.polyiou is a shim over the reference's polyiou.cpp compiled by
  oracle/build_ref.py (as make_poly_golden.py uses it).
Rows whose coordinates fall within 1e-3 of a 0.05 rounding boundary are re-drawn, so a last-bit difference of a sin / cos
implementation cannot change a stored line.
python tests/golden/make_scene_golden.py"""
import glob
import os
import re
import sys
import tempfile
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
REF = Path("/root/reference")
sys.path.insert(0, str(ROOT))
from oracle import rbox_ref  # noqa: E402
from oracle.build_ref import build_polyiou, load_polyiou  # noqa: E402

SPLIT_SIZES = [(600, 800), (1024, 1024), (1111, 2057), (3000, 4000), (1024, 1848), (1025, 1023), (2500, 1300)]
NC = 3
MAX_DET = 64
SCENES = [("P0001", 1500, 2600), ("P0002", 900, 700), ("P0003", 2300, 2300)]


def _import_devkit():
    sys.path.insert(0, str(REF))
    sys.path.insert(0, str(REF / "DOTA_devkit"))
    shapely = types.ModuleType("shapely")
    geometry = types.ModuleType("shapely.geometry")

    class Polygon:  # constructed by savepatches, never used without labels
        def __init__(self, *a, **k):
            pass
    geometry.Polygon = Polygon
    shapely.geometry = geometry
    sys.modules["shapely"], sys.modules["shapely.geometry"] = shapely, geometry
    assert build_polyiou()
    lib = load_polyiou()

    def iou_poly(p, q):
        a, b, o = np.ascontiguousarray(p, np.float64), np.ascontiguousarray(q, np.float64), np.zeros(1)
        lib.ref_iou_poly_pairs(a.ctypes.data, b.ctypes.data, o.ctypes.data, 1)
        return float(o[0])
    poly = types.ModuleType("DOTA_devkit.polyiou")
    poly.VectorDouble = list
    poly.iou_poly = iou_poly
    sys.modules["DOTA_devkit.polyiou"] = poly
    import ImgSplit_multi_process as split
    import ResultMerge_multi_process as merge
    return split, merge


def make_split(split):
    import cv2
    work = Path(tempfile.mkdtemp(prefix="scene_split_"))
    (work / "in" / "images").mkdir(parents=True)
    (work / "in" / "labelTxt").mkdir()
    base = split.splitbase(str(work / "in"), str(work / "out"), gap=200, subsize=1024, num_process=1)
    origins = []
    for h, w in SPLIT_SIZES:
        name = f"blank_{h}x{w}"
        cv2.imwrite(str(work / "in" / "images" / (name + ".png")), np.zeros((h, w, 3), np.uint8))
        (work / "in" / "labelTxt" / (name + ".txt")).write_text("")
        base.SplitSingle(name, 1, ".png")
        got = []
        for f in glob.glob(str(work / "out" / "images" / (name + "__*.png"))):
            m = re.search(r"__1__(\d+)___(\d+)\.png$", f)
            got.append((int(m.group(1)), int(m.group(2))))
        origins.append(sorted(got))  # the loop's order: left outer, up inner, both increasing
    base.pool.close()
    return origins


def _near_boundary(v):
    f = np.abs(v * 10.0 - np.floor(v * 10.0) - 0.5)
    return bool((f < 1e-2).any())


def make_tiles(seed=0):
    """Per scene: objects in scene pixels, reported by every tile that contains their centre (tile coordinates, jittered)."""
    from yolov5_obb_b200.scene import split_origins
    rng = np.random.default_rng(seed)
    det7, origins, scene_of = [], [], []
    used_scores = set()
    for s, (_, h, w) in enumerate(SCENES):
        objs = [(rng.uniform(0, w), rng.uniform(0, h), rng.uniform(15, 120), rng.uniform(0.3, 1.0), rng.uniform(-np.pi / 2, np.pi / 2),
                 int(rng.integers(0, NC))) for _ in range(40)]
        # clusters: several objects near each other (suppression inside one tile as well as across tiles)
        for k in range(12):
            cx, cy, l, r, th, c = objs[k]
            objs.append((cx + rng.normal(0, 6), cy + rng.normal(0, 6), l * rng.uniform(0.8, 1.2), r, th + rng.normal(0, 0.1), c))
        for left, up in split_origins(h, w):
            rows = []
            for cx, cy, l, r, th, c in objs:
                x, y = cx - left + rng.normal(0, 1.5), cy - up + rng.normal(0, 1.5)
                if not (0 <= x < 1024 and 0 <= y < 1024) or len(rows) >= MAX_DET:
                    continue
                while True:
                    row = np.array([x, y, l * rng.uniform(0.95, 1.05), l * r, np.clip(th + rng.normal(0, 0.02), -np.pi / 2, np.pi / 2 - 1e-3),
                                    rng.uniform(0.02, 0.99), c], np.float32)
                    poly = rbox_ref.rbox2poly(row[None, :5]).astype(np.float64)[0]
                    poly[0::2] += left
                    poly[1::2] += up
                    if float(row[5]) not in used_scores and not _near_boundary(poly):
                        break
                used_scores.add(float(row[5]))
                rows.append(row)
            t = np.zeros((MAX_DET, 7), np.float32)
            if rows:
                t[:len(rows)] = np.stack(rows)
            det7.append((t, len(rows)))
            origins.append((left, up))
            scene_of.append(s)
    D = np.stack([t for t, _ in det7])
    counts = np.array([k for _, k in det7], np.int64)
    return D, counts, np.array(origins, np.int32), np.array(scene_of, np.int32)


def make_merge(merge, D, counts, origins, scene_of):
    work = Path(tempfile.mkdtemp(prefix="scene_merge_"))
    (work / "src").mkdir()
    (work / "dst").mkdir()
    lines = {}
    for c in range(NC):
        src = work / "src" / f"Task1_class{c}.txt"
        with open(src, "w") as f:
            for t in range(len(D)):
                name, (left, up) = SCENES[scene_of[t]][0], origins[t]
                for r in D[t, :counts[t]]:
                    if int(r[6]) != c:
                        continue
                    poly = rbox_ref.rbox2poly(r[None, :5])[0]
                    vals = " ".join(repr(float(v)) for v in poly)
                    f.write(f"{name}__1__{left}___{up} {repr(float(r[5]))} {vals}\n")
        merge.mergesingle(str(work / "dst"), merge.py_cpu_nms_poly_fast, str(src))
        lines[c] = (work / "dst" / f"Task1_class{c}.txt").read_text().splitlines()
    return lines


def main():
    cwd = os.getcwd()
    split, merge = _import_devkit()
    os.chdir(cwd)
    origins_split = make_split(split)
    D, counts, origins, scene_of = make_tiles()
    lines = make_merge(merge, D, counts, origins, scene_of)
    out = {
        "split_sizes": np.array(SPLIT_SIZES, np.int64),
        "split_counts": np.array([len(o) for o in origins_split], np.int64),
        "split_origins": np.array([p for o in origins_split for p in o], np.int64),
        "det7": D, "counts": counts, "origins": origins, "scene_of": scene_of,
        "scene_names": np.array([s[0] for s in SCENES]), "nc": np.int64(NC),
    }
    for c in range(NC):
        out[f"lines{c}"] = np.array(lines[c], dtype=str)
    np.savez_compressed(HERE / "scene_golden.npz", **out)
    print({k: getattr(v, "shape", v) for k, v in out.items()})


if __name__ == "__main__":
    main()
