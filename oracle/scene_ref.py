"""Whole-scene detection chain of the DOTA devkit restated on the host — TEST INFRASTRUCTURE for yolov5_obb_b200/scene.py
(never imported by the product package).

  split_origins   DOTA_devkit/ImgSplit_multi_process.py:252-273 (SplitSingle's loop at rate 1)
  crop_tiles      :122-132 saveimagepatches (zero padding at the bottom and right) + BGR -> RGB, NCHW uint8
  tiles_to_scene  utils/rboxs_utils.py:106-126 rbox2poly (oracle.rbox_ref) + ResultMerge_multi_process.py:175-182 poly2origpoly
  merge           ResultMerge_multi_process.py:62-123 py_cpu_nms_poly_fast per (scene, class), oracle.poly_ref arithmetic,
                  with the lower-index-first rule for tied scores (the reference's argsort()[::-1] takes the higher index)
  format_lines    the merged files' text (:220-234): conf rounded to 0.01, coordinates to 0.1"""
import numpy as np

from . import poly_ref, rbox_ref


def split_origins(h, w, subsize=1024, gap=200):
    slide = subsize - gap
    out, left = [], 0
    while left < w:
        if left + subsize >= w:
            left = max(w - subsize, 0)
        up = 0
        while up < h:
            if up + subsize >= h:
                up = max(h - subsize, 0)
            out.append((left, up))
            if up + subsize >= h:
                break
            up += slide
        if left + subsize >= w:
            break
        left += slide
    return out


def crop_tiles(scene_bgr, origins, subsize):
    """[H, W, 3] uint8 BGR -> [len(origins), 3, subsize, subsize] uint8 RGB, zero outside the scene."""
    out = np.zeros((len(origins), 3, subsize, subsize), np.uint8)
    for k, (left, up) in enumerate(origins):
        sub = scene_bgr[up:up + subsize, left:left + subsize]
        out[k, :, :sub.shape[0], :sub.shape[1]] = sub[:, :, ::-1].transpose(2, 0, 1)
    return out


def tiles_to_scene(tile_dets, origins):
    """Per tile [n, 7] (cx, cy, l, s, theta, conf, cls) -> [N, 10] fp64 (scene polygon, conf, cls), tile after tile."""
    rows = []
    for d, (left, up) in zip(tile_dets, origins):
        d = np.asarray(d, np.float32).reshape(-1, 7)
        poly = rbox_ref.rbox2poly(d[:, :5]).astype(np.float64)
        poly[:, 0::2] += left
        poly[:, 1::2] += up
        rows.append(np.concatenate([poly, d[:, 5:7].astype(np.float64)], 1))
    return np.concatenate(rows, 0) if rows else np.zeros((0, 10))


def nms_poly_stable(dets, thresh, iou=poly_ref.iou_poly):
    """py_cpu_nms_poly_fast with descending score, ties -> lower index first."""
    dets = np.asarray(dets, np.float64).reshape(-1, 9)
    obbs = dets[:, :8]
    x1, y1 = obbs[:, 0::2].min(1), obbs[:, 1::2].min(1)
    x2, y2 = obbs[:, 0::2].max(1), obbs[:, 1::2].max(1)
    areas = (x2 - x1 + 1) * (y2 - y1 + 1)
    order = np.argsort(-dets[:, 8], kind="stable")
    keep = []
    while order.size > 0:
        i = order[0]
        keep.append(int(i))
        rest = order[1:]
        w = np.maximum(0.0, np.minimum(x2[i], x2[rest]) - np.maximum(x1[i], x1[rest]))
        h = np.maximum(0.0, np.minimum(y2[i], y2[rest]) - np.maximum(y1[i], y1[rest]))
        hb = w * h
        with np.errstate(invalid="ignore", divide="ignore"):
            ovr = hb / (areas[i] + areas[rest] - hb)
        for j in np.where(ovr > 0)[0]:
            ovr[j] = iou(obbs[i], obbs[rest[j]])
        order = rest[ovr <= thresh]
    return keep


def merge(rows10, scene_ids, n_scenes, nc, thresh=0.2, nms=nms_poly_stable):
    """[N, 10] scene rows with their scene ids -> per scene [n, 10]: class after class, keep order within."""
    rows10 = np.asarray(rows10, np.float64).reshape(-1, 10)
    scene_ids = np.asarray(scene_ids)
    out = []
    for s in range(n_scenes):
        parts = []
        for c in range(nc):
            idx = np.where((scene_ids == s) & (rows10[:, 9] == c))[0]
            if idx.size:
                parts.append(rows10[idx[nms(rows10[idx, :9], thresh)]])
        out.append(np.concatenate(parts, 0) if parts else np.zeros((0, 10)))
    return out


def format_lines(name, rows9):
    """The merged file's lines of one scene (ResultMerge_multi_process.py:220-234)."""
    lines = []
    for r in rows9:
        bbox = [round(float(v), 1) for v in r[:8]]
        lines.append(name + " " + str(round(float(r[8]), 2)) + " " + " ".join(map(str, bbox)))
    return lines
