"""Whole-scene DOTA detection on the device: the reference's submission chain

  DOTA_devkit/ImgSplit_multi_process.py:226-273  split every scene into subsize x subsize patches (rate 1, overlap `gap`)
  val.py --task test (conf 0.01, IoU 0.4, max_det 1500)  detect on every patch, rbox2poly -> JSON (val.py:226-232, 50-67)
  tools/TestJson2VocClassTxt.py  regroup by class
  DOTA_devkit/ResultMerge_multi_process.py:175-236  poly2origpoly + py_cpu_nms_poly_fast (nms_thresh 0.2) per (scene, class)

as one call: the stem crops the tiles from the scene tensors (csrc/aux_kernels.cu y5obb_stem_s2d_scene_u8), the tiles run
through ONE inference plan in batches, and the merge (csrc/poly_nms.cu y5obb_tiles_to_scene_f64 +
y5obb_poly_nms_segmented_f64) runs every (scene, class) NMS at once.  Between the first tile batch and the merge the host
reads the device once: the per-batch candidate totals of the post-process (overflow check) and the (scene, class) row
histogram that sizes the merge workspace.

Not covered: rates other than 1 (the devkit's multi-scale split resizes with cv2.INTER_CUBIC), label cropping for training,
the text rounding of the JSON step (polygon to 0.1, score to 1e-5: the merge here works on unrounded values) and file I/O."""
from typing import List, Sequence, Tuple, Union

import torch

from . import _lib
from .general import non_max_suppression_obb


def split_origins(h: int, w: int, subsize: int = 1024, gap: int = 200) -> List[Tuple[int, int]]:
    """(left, up) of every patch of an h x w scene, in the devkit's order (left outer, up inner): SplitSingle's loop
    (ImgSplit_multi_process.py:252-273) at rate 1.  Edge patches are moved back inside the scene; a scene smaller than a patch
    gives the single origin (0, 0) and is zero-padded at the bottom and right."""
    h, w, subsize, gap = int(h), int(w), int(subsize), int(gap)
    if h <= 0 or w <= 0 or subsize <= 0:
        raise ValueError(f"scene {h}x{w} and patch size {subsize} must be positive")
    if gap < 0 or gap >= subsize:
        raise ValueError(f"gap {gap} must be in [0, subsize={subsize})")
    slide = subsize - gap
    out = []
    left = 0
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


def tiles_to_scene(det7: torch.Tensor, counts: torch.Tensor, origins: torch.Tensor, scene_of: torch.Tensor, n_scenes: int,
                   nc: int, stats: torch.Tensor):
    """Tile detections [T, max_det, 7] (counts int64 [T]) -> scene-space rows dets9 [T * max_det, 9] fp64 and segment ids
    (scene * nc + class) int32, compacted tile after tile.  Writes the (scene, class) row histogram into stats[:-1] and the row
    count into stats[-1] (int64 device view of n_scenes * nc + 1 elements); nothing is read back."""
    T, max_det = det7.shape[0], det7.shape[1]
    dev = det7.device
    dets9 = torch.empty((T * max_det, 9), dtype=torch.float64, device=dev)
    seg = torch.empty(T * max_det, dtype=torch.int32, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        st = _lib.stream_ptr(dev)
        ws = _lib.workspace(L.y5obb_tiles_to_scene_workspace_bytes(T), dev, f"scene_gather:{st}")
        _lib.check(L.y5obb_tiles_to_scene_f64(det7.data_ptr(), counts.data_ptr(), T, max_det, origins.data_ptr(),
                                              scene_of.data_ptr(), n_scenes, nc, dets9.data_ptr(), seg.data_ptr(),
                                              stats[-1:].data_ptr(), stats.data_ptr(), ws.data_ptr(), ws.numel(), st),
                   "y5obb_tiles_to_scene_f64")
    return dets9, seg


def poly_nms_segmented(dets9: torch.Tensor, seg: torch.Tensor, seg_counts: Sequence[int], thresh: float):
    """py_cpu_nms_poly_fast (ResultMerge_multi_process.py:62-123) on every segment at once: dets9 [>= n, 9] fp64, seg int32
    [>= n] segment ids, seg_counts the HOST list of rows per segment (n = their sum).  Returns (keep int64 [n], offsets int64
    [S + 1]) on the device, nothing read back: segment s keeps keep[offsets[s]:offsets[s + 1]], indices into dets9 in
    descending score order; keep[offsets[S]:] is unused."""
    counts = torch.tensor([int(k) for k in seg_counts], dtype=torch.int64)
    S, n = counts.numel(), int(counts.sum())
    dev = dets9.device
    keep = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    offsets = torch.empty(S + 1, dtype=torch.int64, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        st = _lib.stream_ptr(dev)
        nbytes = L.y5obb_poly_nms_segmented_workspace_bytes(counts.data_ptr(), S)
        if nbytes == 0:
            raise RuntimeError(f"segmented polygon NMS: a segment of {int(counts.max())} rows exceeds the greedy scan's limit")
        ws = _lib.workspace(nbytes, dev, f"scene_merge:{st}")
        _lib.check(L.y5obb_poly_nms_segmented_f64(dets9.data_ptr(), seg.data_ptr(), n, counts.data_ptr(), S, float(thresh),
                                                  keep.data_ptr(), offsets.data_ptr(), ws.data_ptr(), ws.numel(), st),
                   "y5obb_poly_nms_segmented_f64")
    return keep[:n], offsets


def _scene_rows(dets9, seg, keep, offsets, n_scenes, nc):
    """Kept rows as per-scene [n, 10] fp64 tensors (x1 y1 ... x4 y4, conf, cls): class after class, keep order within."""
    bounds = offsets[::nc].tolist()   # segment s * nc starts scene s (the read that shapes the results)
    keep = keep[:bounds[-1]]
    rows = torch.empty((keep.numel(), 10), dtype=torch.float64, device=dets9.device)
    rows[:, :9] = dets9.index_select(0, keep)
    rows[:, 9] = seg.index_select(0, keep).remainder(nc)
    return [rows[bounds[s]:bounds[s + 1]] for s in range(n_scenes)]


def merge_tiles(det7: torch.Tensor, counts: torch.Tensor, origins: torch.Tensor, scene_of: torch.Tensor, n_scenes: int, nc: int,
                merge_iou: float = 0.2) -> List[torch.Tensor]:
    """The merge stage alone (ResultMerge_multi_process.py:175-236 at rate 1): tile detections [T, max_det, 7] with counts
    int64 [T], origins int32 [T, 2] (left, up) and scene ids int32 [T] (< 0: ignored) on one device -> per scene [n, 10] fp64
    (x1 y1 ... x4 y4, conf, cls) in scene pixels, grouped by class in ascending order, descending score within a class."""
    stats = torch.empty(n_scenes * nc + 1, dtype=torch.int64, device=det7.device)
    dets9, seg = tiles_to_scene(det7.float().contiguous(), counts.long().contiguous(), origins.int().contiguous(),
                                scene_of.int().contiguous(), n_scenes, nc, stats)
    hist = stats[:-1].tolist()
    keep, offsets = poly_nms_segmented(dets9, seg, hist, merge_iou)
    return _scene_rows(dets9, seg, keep, offsets, n_scenes, nc)


class SceneDetector:
    """Detections of whole DOTA scenes: `detect(scene)` = the reference's split -> val.py --task test -> class files ->
    ResultMerge chain, on the device.  Defaults are those of that chain's DOTA submission settings."""

    def __init__(self, model, subsize: int = 1024, gap: int = 200, batch: int = 16, conf_thres: float = 0.01,
                 iou_thres: float = 0.4, max_det: int = 1500, merge_iou: float = 0.2, multi_label: bool = True, classes=None,
                 agnostic: bool = False):
        if model.training:
            raise RuntimeError("SceneDetector needs the model in eval() mode")
        smax = int(max(model.stride))
        if int(subsize) <= 0 or int(subsize) % smax:
            raise ValueError(f"subsize {subsize} must be a positive multiple of the model's max stride {smax}")
        if int(gap) < 0 or int(gap) >= int(subsize):
            raise ValueError(f"gap {gap} must be in [0, subsize={subsize})")
        if int(batch) < 1:
            raise ValueError("batch must be >= 1")
        self.model, self.subsize, self.gap, self.batch = model, int(subsize), int(gap), int(batch)
        self.nc = int(model.model[-1].nc)
        self.merge_iou = float(merge_iou)
        self.kw = dict(conf_thres=conf_thres, iou_thres=iou_thres, classes=classes, agnostic=agnostic, multi_label=multi_label,
                       max_det=int(max_det))

    @staticmethod
    def _check(scenes):
        for s in scenes:
            if not isinstance(s, torch.Tensor):
                raise TypeError("a scene must be a torch.Tensor")
            if s.dtype != torch.uint8:
                raise TypeError(f"a scene must be uint8 (cv2.imread's BGR pixels), got {s.dtype}")
            if s.dim() != 3 or s.shape[2] != 3 or s.shape[0] == 0 or s.shape[1] == 0:
                raise ValueError(f"a scene must be [H, W, 3] (HWC, BGR), got {tuple(s.shape)}")
            _lib.require_cuda(s, "scene")
        if len({s.device for s in scenes}) > 1:
            raise ValueError("all scenes of one call must be on the same device")

    def _batch_runs(self, b, tile_scene):
        """(scenes, tile counts) of batch b: its valid tiles grouped into consecutive runs of one scene."""
        runs = []
        for s in tile_scene[b * self.batch:(b + 1) * self.batch]:
            if runs and runs[-1][0] == s:
                runs[-1][1] += 1
            else:
                runs.append([s, 1])
        return runs

    def detect(self, scenes: Union[torch.Tensor, Sequence[torch.Tensor]]) -> List[torch.Tensor]:
        """scenes: one uint8 CUDA tensor [H, W, 3] (BGR, as cv2.imread returns it) or a list of them.  Returns per scene a
        float64 device tensor [n, 10] = (x1 y1 x2 y2 x3 y3 x4 y4, conf, cls) in scene pixels, grouped by class in ascending
        order and in descending score within a class: the content and order of the reference's merged per-class files."""
        scenes = [scenes] if isinstance(scenes, torch.Tensor) else list(scenes)
        if not scenes:
            return []
        self._check(scenes)
        scenes = [s.contiguous() for s in scenes]
        dev, S, B, nc = scenes[0].device, len(scenes), self.batch, self.nc
        origins, tile_scene = [], []
        for k, s in enumerate(scenes):
            o = split_origins(s.shape[0], s.shape[1], self.subsize, self.gap)
            origins += o
            tile_scene += [k] * len(o)
        T = len(origins)
        nb = (T + B - 1) // B
        Tp = nb * B
        origins_h = torch.zeros((Tp, 2), dtype=torch.int32)
        origins_h[:T] = torch.tensor(origins, dtype=torch.int32)
        scene_of_h = torch.full((Tp,), -1, dtype=torch.int32)
        scene_of_h[:T] = torch.tensor(tile_scene, dtype=torch.int32)
        origins_d, scene_of_d = origins_h.to(dev), scene_of_h.to(dev)   # uploaded before the first batch
        det_all = torch.empty((Tp, self.kw["max_det"], 7), dtype=torch.float32, device=dev)
        # one int64 buffer read back once: [candidate totals per batch | rows per tile | (scene, class) histogram | rows]
        info = torch.empty(nb + Tp + S * nc + 1, dtype=torch.int64, device=dev)
        counts_d, stats = info[nb:nb + Tp], info[nb + Tp:]
        caps = []
        with torch.cuda.device(dev):
            for b in range(nb):
                packed, counts, cap = self._run_batch(b, scenes, tile_scene, origins_d, "async")
                det_all[b * B:(b + 1) * B].copy_(packed)
                counts_d[b * B:(b + 1) * B].copy_(counts[:B])
                info[b:b + 1].copy_(counts[B:B + 1])
                caps.append(cap)
            dets9, seg = tiles_to_scene(det_all, counts_d, origins_d, scene_of_d, S, nc, stats)
            host = info.tolist()   # the one read between the first batch and the merge
            rerun = False
            for b in range(nb):
                c = host[nb + b * B:nb + (b + 1) * B]
                if host[b] > caps[b] or host[b] < 0 or any(k < 0 for k in c):
                    # rare: more candidates than the post-process's optimistic capacity -> this batch again, blocking
                    # (DetectPipeline._finish does the same)
                    packed, cnt = self._run_batch(b, scenes, tile_scene, origins_d, True)
                    det_all[b * B:(b + 1) * B].copy_(packed)
                    counts_d[b * B:(b + 1) * B].copy_(torch.tensor(cnt, dtype=torch.int64))
                    rerun = True
            if rerun:
                dets9, seg = tiles_to_scene(det_all, counts_d, origins_d, scene_of_d, S, nc, stats)
                host = info.tolist()
            keep, offsets = poly_nms_segmented(dets9, seg, host[nb + Tp:nb + Tp + S * nc], self.merge_iou)
            return _scene_rows(dets9, seg, keep, offsets, S, nc)

    def _run_batch(self, b, scenes, tile_scene, origins_d, return_packed):
        B = self.batch
        runs = self._batch_runs(b, tile_scene)
        rec = self.model.detect_records_tiles([scenes[s] for s, _ in runs], origins_d[b * B:(b + 1) * B], [k for _, k in runs],
                                              self.subsize)
        return non_max_suppression_obb(rec, return_packed=return_packed, **self.kw)
