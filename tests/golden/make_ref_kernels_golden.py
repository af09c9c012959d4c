"""Generates ref_kernels_golden.npz: the outputs of the REFERENCE's own native kernels (built by oracle/build_ref.py into
oracle/_ref) on the seeded inputs of the tests that compare with them.  Needs those builds and a GPU (sm_100a).
Re-run:  python tests/golden/make_ref_kernels_golden.py [OUT.npz]

  cpu_keep/{n}_{span}_{thr}_{seed}  nms_rotated_cpu keep lists           tests/test_oracle_nms.py (pins the C++ oracle)
  keep/{n}_{span}_{seed}, thr/{thr}, kat/{name}, cluster/{image}
                                     nms_rotated_cuda (K1) keep lists      tests/test_nms_gpu.py
  iou/{theta_grid}, iou_degenerate   single_box_iou_rotated<float>         tests/test_nms_gpu.py
  overlaps/{seed}, poly_nms/{n}_{seed}_{thr}
                                     DOTA_devkit poly_nms_gpu _overlaps / _poly_nms   tests/test_poly_f32_gpu.py
Keep lists are stored as keep_bits, iou/* and overlaps/* in the sampled form (tests/refgolden.py).
"""
import ctypes
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle.build_ref import OUT as REF_LIBS, load_polygpu, load_ref  # noqa: E402
from tests.boxgen import rboxes, degenerate_pairs  # noqa: E402
from tests.refgolden import keep_bits, sampled  # noqa: E402
from tests import test_nms_gpu as t_nms, test_oracle_nms as t_oracle, test_poly_f32_gpu as t_poly  # noqa: E402

DEV = "cuda:0"


def ref_iou_pairs(a, b):
    L = ctypes.CDLL(str(REF_LIBS / "libref_iou.so"))
    L.ref_iou_pairs.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_long, ctypes.c_void_p]
    L.ref_iou_pairs.restype = ctypes.c_int
    ta, tb = torch.from_numpy(a).to(DEV).contiguous(), torch.from_numpy(b).to(DEV).contiguous()
    out = torch.empty(a.shape[0], dtype=torch.float32, device=DEV)
    torch.cuda.synchronize()
    assert L.ref_iou_pairs(ta.data_ptr(), tb.data_ptr(), out.data_ptr(), a.shape[0], None) == 0
    torch.cuda.synchronize()
    return out.cpu().numpy()


def main(path):
    ref = load_ref()
    cuda_nms = lambda d, s, thr: ref.nms_rotated_cuda(torch.from_numpy(d).to(DEV), torch.from_numpy(s).to(DEV), thr).cpu().numpy()
    out = {}
    for n, span, thr, seed in t_oracle.PIN_CASES:
        d, s, _ = rboxes(n, span, seed, n_classes=4)
        keep = ref.nms_rotated_cpu(torch.from_numpy(d), torch.from_numpy(s), thr).numpy()
        out[f"cpu_keep/{n}_{span}_{thr}_{seed}"] = keep_bits(keep, s)
    for n, span, seed in t_nms.KEEP_CASES:
        d, s, _ = rboxes(n, span, seed)
        out[f"keep/{n}_{span}_{seed}"] = keep_bits(cuda_nms(d, s, 0.4), s)
    d, s, _ = t_nms.threshold_case()
    for thr in t_nms.THRESHOLDS:
        out[f"thr/{thr}"] = keep_bits(cuda_nms(d, s, thr), s)
    g = np.load(ROOT / "tests" / "golden" / "nms_golden.npz")
    for k in sorted({x.split("/")[0] for x in g.files if x.startswith("kat")}):
        out[f"kat/{k}"] = keep_bits(cuda_nms(g[f"{k}/dets"], g[f"{k}/scores"], float(g[f"{k}/thr"])), g[f"{k}/scores"])
    d, s, img, B = t_nms.cluster_case()
    for b in range(B):
        idx = np.flatnonzero(img == b)
        out[f"cluster/{b}"] = keep_bits(cuda_nms(d[idx], s[idx], 0.4) if len(idx) else np.zeros(0, np.int64), s[idx])

    for theta_grid in (True, False):
        a, b = t_nms._near_pairs(400_000, 11, theta_grid)
        for name, v in sampled(ref_iou_pairs(a, b)).items():
            out[f"iou/{int(theta_grid)}/{name}"] = v
    out["iou_degenerate"] = ref_iou_pairs(*degenerate_pairs())

    ref_poly_nms, ref_overlaps = load_polygpu()
    for seed, n, k, span in t_poly.OVERLAP_CASES:
        b, q = t_poly.overlap_inputs(seed, n, k, span)
        want = np.zeros((n, k), np.float32)
        ref_overlaps(want.ctypes.data, b.ctypes.data, q.ctypes.data, n, k, 0)
        for name, v in sampled(want).items():
            out[f"overlaps/{seed}/{name}"] = v
    for n, seed, thr in t_poly.POLY_NMS_CASES:
        d = t_poly._sorted_dets(n, seed)
        keep = np.zeros(n, np.int32)
        num = ctypes.c_int(0)
        ref_poly_nms(keep.ctypes.data, ctypes.addressof(num), d.ctypes.data, n, 9, thr, 0)
        out[f"poly_nms/{n}_{seed}_{thr}"] = keep[:num.value].copy()

    np.savez_compressed(path, **out)
    for k, v in out.items():
        print(k, v.dtype, v.shape)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else Path(__file__).resolve().parent / "ref_kernels_golden.npz")
