"""Whole-scene detection throughput: SceneDetector.detect (device crop + one plan + device merge) against the host composition
of the existing pieces (host crop + upload, Model.detect_records + non_max_suppression_obb per batch, rbox2poly + offsets,
one device polygon NMS call per (scene, class) segment), in the same process and alternating.  yolov5s (nc 15, the seeded
calibrated benchmark model), batch 16, DOTA submission settings (conf 0.01, IoU 0.4, max_det 1500, merge IoU 0.2), seeded
synthetic 4000^2 (25 tiles) and 8000^2 (100 tiles) scenes.  Times are host clocks around work that ends in a device
synchronise, after warm-up; the merge stage is also timed alone (CUDA events) with its segment and pair counts.
python tools/time_scene.py [--reps 5] [--out profiles/r3_scene_time.json]"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import scene_ref  # noqa: E402
from tests.modelgen import calibrated_bench_model  # noqa: E402
from tests.tilegen import synth_tiles  # noqa: E402
from yolov5_obb_b200.devkit import py_cpu_nms_poly_fast  # noqa: E402
from yolov5_obb_b200.general import non_max_suppression_obb  # noqa: E402
from yolov5_obb_b200.rboxs_utils import rbox2poly  # noqa: E402
from yolov5_obb_b200.scene import SceneDetector, merge_tiles, split_origins  # noqa: E402

DEV = "cuda:0"
KW = dict(conf_thres=0.01, iou_thres=0.4, max_det=1500, multi_label=True)
B, TILE, NC = 16, 1024, 15


def host_composition(model, scene, keep_tiles=None):
    org = split_origins(scene.shape[0], scene.shape[1], TILE, 200)
    tiles = scene_ref.crop_tiles(scene.cpu().numpy(), org, TILE)
    segs = {}
    for b0 in range(0, len(tiles), B):
        x = np.zeros((B, 3, TILE, TILE), np.uint8)
        x[:len(tiles[b0:b0 + B])] = tiles[b0:b0 + B]
        packed, counts = non_max_suppression_obb(model.detect_records(torch.from_numpy(x).to(DEV)), return_packed=True, **KW)
        if keep_tiles is not None:
            keep_tiles.append((packed.clone(), counts))
        for j in range(min(B, len(tiles) - b0)):
            d = packed[j, :counts[j]]
            poly = rbox2poly(d[:, :5].contiguous()).double()
            poly[:, 0::2] += org[b0 + j][0]
            poly[:, 1::2] += org[b0 + j][1]
            r9 = torch.cat([poly, d[:, 5:6].double()], 1)
            cls = d[:, 6].long()
            for c in cls.unique().tolist():
                segs.setdefault(c, []).append(r9[cls == c])
    out = []
    for c in sorted(segs):
        D = torch.cat(segs[c], 0)
        out.append(D[py_cpu_nms_poly_fast(D, 0.2)])
    return out


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_scene_time.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_scene.py measures on a CUDA device; none is present")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    model = calibrated_bench_model("s", nc=NC, seed=0).to(DEV)
    det = SceneDetector(model, batch=B)
    res = dict(gpu=gpu, torch=torch.__version__, model="yolov5s nc=15 (tests.modelgen.calibrated_bench_model seed 0)",
               batch=B, subsize=TILE, gap=200, settings=KW, merge_iou=0.2, reps=a.reps, scenes={})
    for side in (4000, 8000):
        scene = synth_tiles(1, side, seed=7)[0].flip(0).permute(1, 2, 0).contiguous().to(DEV)
        n_tiles = len(split_origins(side, side, TILE, 200))
        for _ in range(2):   # warm-up: plans, graphs, workspaces
            det.detect(scene)
            host_composition(model, scene)
        t_dev, t_host = [], []
        for _ in range(a.reps):   # alternating
            t_dev += timed(lambda: det.detect(scene), 1)
            t_host += timed(lambda: host_composition(model, scene), 1)
        out = det.detect(scene)[0]
        # the merge stage alone, on this scene's tile detections
        tiles = []
        host_composition(model, scene, keep_tiles=tiles)
        det7 = torch.cat([p for p, _ in tiles], 0)[:n_tiles].contiguous()
        counts = torch.tensor([c for _, cs in tiles for c in cs][:n_tiles], dtype=torch.int64, device=DEV)
        org = torch.tensor(split_origins(side, side, TILE, 200), dtype=torch.int32, device=DEV)
        sid = torch.zeros(n_tiles, dtype=torch.int32, device=DEV)
        merge_tiles(det7, counts, org, sid, 1, NC)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ms = []
        for _ in range(a.reps):
            ev[0].record()
            merge_tiles(det7, counts, org, sid, 1, NC)
            ev[1].record()
            torch.cuda.synchronize()
            ms.append(ev[0].elapsed_time(ev[1]))
        cls = []
        for p, cs in tiles:
            for j, c in enumerate(cs):
                cls.append(p[j, :c, 6].long().cpu())
        cls = torch.cat(cls[:n_tiles]) if cls else torch.zeros(0, dtype=torch.long)
        hist = torch.bincount(cls, minlength=NC).tolist()
        mp = side * side / 1e6
        md, mh = float(np.median(t_dev)), float(np.median(t_host))
        res["scenes"][f"{side}x{side}"] = dict(
            tiles=n_tiles, detections=int(out.shape[0]), tile_rows=int(sum(hist)),
            segments=int(sum(1 for k in hist if k)), pairs=int(sum(k * (k - 1) // 2 for k in hist)),
            detect_s=t_dev, host_composition_s=t_host, detect_median_s=md, host_median_s=mh,
            detect_scenes_per_s=1 / md, detect_mpix_per_s=mp / md, host_scenes_per_s=1 / mh, host_mpix_per_s=mp / mh,
            merge_ms=ms, merge_median_ms=float(np.median(ms)))
        print(json.dumps({k: v for k, v in res["scenes"][f"{side}x{side}"].items() if not isinstance(v, list)}))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps(dict(gpu=gpu, out=a.out)))


if __name__ == "__main__":
    main()
