"""Inference plan: turns a yolo.Model into a fixed sequence of sm_100a kernel launches.

Layout decisions (all NHWC bf16):
  * every tensor is a channel slice of some buffer; a producer whose output feeds a Concat
    (models/common.py:267-274) stores directly at its channel offset in the concat buffer;
  * nn.Upsample(2x nearest) is a second store of the producing conv's epilogue (out2x);
  * C3 (models/common.py:126-138): cv1 and cv2 share the input, so they run as ONE GEMM with
    concatenated output channels [cv1 | cv2] written into the block's concat buffer; the Bottleneck
    chain then updates channels [0, c_) in place (1x1 -> tmp, 3x3 + residual -> back), cv3 reads the
    whole buffer;
  * SPPF (:181-196): cv1 -> channels [0,c_) of a 4c_ buffer, one pooling kernel fills the rest;
  * the stem Conv(3, c, 6, 2, 2) runs as a 3x3 conv over a 2x2 space-to-depth copy of the image;
  * Detect (models/yolo.py:49-81): one GEMM per level whose epilogue permutes, applies sigmoid and the
    grid/anchor decode and writes fp32 rows of the final [B, A, no] tensor.
BatchNorm is folded into the conv weights exactly as utils/torch_utils.py:192-212 (fuse_conv_and_bn).
"""
import ctypes
from typing import List, Optional

import torch

from . import _lib
from .conv import Conv as ConvOp, Slice, WindowView, pack_weights, MODE_DETECT
from . import yolo as Y


def fold_bn(conv: torch.nn.Conv2d, bn: Optional[torch.nn.BatchNorm2d]):
    """W' = diag(gamma / sqrt(var + eps)) W ; b' = beta - gamma * mean / sqrt(var + eps)  (+ conv bias).
    Host-side plan building: the arithmetic runs on CPU copies of the parameters (one D2H copy per tensor, no device
    kernels), the packed bf16 operands are uploaded once by the caller."""
    w = conv.weight.detach().float().cpu()
    b = conv.bias.detach().float().cpu() if conv.bias is not None else torch.zeros(w.shape[0])
    if bn is None:
        return w, b
    scale = bn.weight.detach().float().cpu() / torch.sqrt(bn.running_var.detach().float().cpu() + bn.eps)
    return w * scale.view(-1, 1, 1, 1), (b - bn.running_mean.detach().float().cpu()) * scale + bn.bias.detach().float().cpu()


def _conv_params(m):
    return fold_bn(m.conv, getattr(m, "bn", None))


def _kind(m) -> str:
    """Module kind by class NAME, so that the reference's own modules (models/common.py, models/yolo.py,
    torch.nn.Upsample) are accepted as well as the mirrors of yolo.py."""
    return type(m).__name__


def _is(m, name: str) -> bool:
    return _kind(m) == name


class InferenceEngine:
    def __init__(self, model: "Y.Model", B: int, H: int, W: int, device, conv_flags: int = 0, compact_detect: bool = False):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("InferenceEngine needs a CUDA device (sm_100a); there is no CPU path")
        det = model.model[-1]
        smax = int(max(model.stride))
        if H % smax or W % smax:
            raise RuntimeError(f"image size {H}x{W} must be a multiple of the max stride {smax}")
        self.device, self.B, self.H, self.W = device, B, H, W
        self.ops = []          # (callable taking stream ptr)
        import os
        self._calls, self._graph = 0, None
        self._use_graph = os.environ.get("Y5OBB_NO_GRAPH", "0") != "1"
        self.convs: List[ConvOp] = []
        self.keep = []         # buffers
        self.flops = 0.0
        self.hbm_bytes = 0.0
        L = _lib.lib()
        layers = list(model.model)
        n = len(layers)

        def src_of(i, f):
            return i - 1 if f == -1 else (f if f >= 0 else i + f)

        # ---- pass 1: channels and spatial size of every layer output
        ch, hw = [0] * n, [(0, 0)] * n
        for m in layers:
            i = m.i
            if _is(m, "Detect"):
                continue
            fs = [src_of(i, f) for f in ([m.f] if isinstance(m.f, int) else m.f)]
            in_hw = (H, W) if i == 0 else hw[fs[0]]
            if _is(m, "Conv"):
                s, k, p = m.conv.stride[0], m.conv.kernel_size[0], m.conv.padding[0]
                ch[i] = m.conv.out_channels
                hw[i] = ((in_hw[0] + 2 * p - k) // s + 1, (in_hw[1] + 2 * p - k) // s + 1)
            elif _is(m, "C3"):
                ch[i], hw[i] = m.cv3.conv.out_channels, in_hw
            elif _is(m, "SPPF"):
                ch[i], hw[i] = m.cv2.conv.out_channels, in_hw
            elif _is(m, "Upsample"):
                ch[i], hw[i] = ch[fs[0]], (in_hw[0] * 2, in_hw[1] * 2)
            elif _is(m, "Concat"):
                ch[i], hw[i] = sum(ch[f] for f in fs), in_hw
                assert all(hw[f] == in_hw for f in fs)

        arena = {"buf": None, "used": 0}

        def new(h, w, c):
            # zeros, once: the pixel-pair view of stride-2 convs may read channels of a buffer before their
            # producer ran (they meet zero weights, but must be finite).  Carved from a few large zeroed chunks
            # (one fill each) instead of one allocation + fill per tensor.
            n = B * h * w * c
            n_al = (n + 127) // 128 * 128   # 256-byte aligned starts (TMA wants 16)
            if arena["buf"] is None or arena["used"] + n_al > arena["buf"].numel():
                arena["buf"] = torch.zeros(max(n_al, 128 << 20), dtype=torch.bfloat16, device=device)
                arena["used"] = 0
                self.keep.append(arena["buf"])
            t = arena["buf"][arena["used"]:arena["used"] + n].view(B, h, w, c)
            arena["used"] += n_al
            return t

        # ---- pass 2: who feeds a concat
        feeds = {}
        cat_buf = {}
        for m in layers:
            if _is(m, "Concat"):
                cat_buf[m.i] = new(hw[m.i][0], hw[m.i][1], ch[m.i])
                off = 0
                for f in m.f:
                    s = src_of(m.i, f)
                    if s in feeds:
                        raise RuntimeError("a layer feeding two Concats is not in the shipped yamls")
                    feeds[s] = (m.i, off)
                    off += ch[s]
        out: List[Optional[Slice]] = [None] * n
        up_of = {}  # producer conv index -> Slice receiving the up-sampled copy
        for m in layers:
            i = m.i
            if _is(m, "Detect"):
                continue
            if _is(m, "Concat"):
                out[i] = Slice.full(cat_buf[i])
            elif _is(m, "Upsample"):
                if i not in feeds:
                    raise RuntimeError("nn.Upsample must feed a Concat (v6.0 head pattern)")
                j, off = feeds[i]
                src = src_of(i, m.f)
                if not _is(layers[src], "Conv"):
                    raise RuntimeError("nn.Upsample must follow a Conv (v6.0 head pattern)")
                up_of[src] = Slice(cat_buf[j], off, ch[i])
                out[i] = up_of[src]
            elif i in feeds:
                j, off = feeds[i]
                out[i] = Slice(cat_buf[j], off, ch[i])
            else:
                out[i] = Slice.full(new(hw[i][0], hw[i][1], ch[i]))

        self.out_slices = out   # per top-level layer: where its output lives (tests read them for teacher-forced parity)

        def add_conv(x, w, b, k, s, p, act, dst: Optional[Slice] = None, res=None, out2x=None, detd=None):
            wp, bp = pack_weights(w.cpu(), b.cpu(), MODE_DETECT if detd else 0, detd["no"] if detd else 0)   # packed on the host
            if act and not detd:
                bp = bp * 0.5   # the SiLU epilogue wants 0.5 * bias (Y5OBB_CONV_BIAS_HALVED)
            op = ConvOp(x, wp.to(device), bp.to(device), w.shape[0], k, s, p, act, out=dst, res=res, out2x=out2x, det=detd,
                        flags=conv_flags, bias_prehalved=True)
            self.convs.append(op)
            info = op.info()
            self.flops += info["flops"]
            self.hbm_bytes += info["hbm_bytes"]
            h = op._h
            self.ops.append(lambda st, h=h: L.y5obb_conv_run(h, st))

        # ---- pass 3: emit ops
        # space-to-depth image with one zero pixel of padding left and right of every row: the stem's three
        # horizontal taps are then 48 CONTIGUOUS channels of an overlapping-window view (pixel stride 16)
        self.x_s2d = torch.zeros((B, H // 2, W // 2 + 2, 16), dtype=torch.bfloat16, device=device)
        self.keep.append(self.x_s2d)
        for m in layers:
            i = m.i
            if _is(m, "Detect"):
                break
            fs = [src_of(i, f) for f in ([m.f] if isinstance(m.f, int) else m.f)]
            if _is(m, "Conv"):
                w, b = _conv_params(m)
                k, s, p = m.conv.kernel_size[0], m.conv.stride[0], m.conv.padding[0]
                act = isinstance(m.act, torch.nn.SiLU)
                if i == 0:
                    if (k, s, p, w.shape[1]) != (6, 2, 2, 3):
                        raise RuntimeError("layer 0 must be the v6.0 stem Conv(3, c, 6, 2, 2)")
                    # w2[co, (dy*2+dx)*3 + c, ty, tx] = w[co, c, 2*ty+dy, 2*tx+dx]   (3x3/s1/p1 over the s2d image)
                    w2 = torch.zeros((w.shape[0], 16, 3, 3))
                    for dy in range(2):
                        for dx in range(2):
                            w2[:, (dy * 2 + dx) * 3:(dy * 2 + dx) * 3 + 3] = w[:, :, dy::2, dx::2]
                    # w3[co, tx*16 + ch, ty, 0] = w2[co, ch, ty, tx]   (3x1 over 48-channel windows)
                    w3 = w2.permute(0, 3, 1, 2).reshape(w.shape[0], 48, 3, 1).contiguous()
                    Wp = W // 2 + 2
                    win = WindowView(buf=self.x_s2d, ptr=self.x_s2d.data_ptr(), pix_stride=16, row_stride=Wp * 16,
                                     img_stride=(H // 2) * Wp * 16, B=B, H=H // 2, W=W // 2, C=48, hbm_c=16)
                    add_conv(win, w3, b, (3, 1), 1, (1, 0), act, out[i])
                else:
                    add_conv(out[fs[0]], w, b, k, s, p, act, out[i], out2x=up_of.get(i))
            elif _is(m, "C3"):
                x = out[fs[0]]
                c_ = m.cv1.conv.out_channels
                cat = Slice.full(new(hw[i][0], hw[i][1], 2 * c_))
                tmp = Slice.full(new(hw[i][0], hw[i][1], c_))
                w1, b1 = _conv_params(m.cv1)
                w2, b2 = _conv_params(m.cv2)
                add_conv(x, torch.cat([w1, w2], 0), torch.cat([b1, b2], 0), 1, 1, 0, True, cat)
                chain = Slice(cat.buf, 0, c_)
                for bt in m.m:
                    wa, ba = _conv_params(bt.cv1)
                    wb, bb = _conv_params(bt.cv2)
                    add_conv(chain, wa, ba, 1, 1, 0, True, tmp)
                    add_conv(tmp, wb, bb, 3, 1, 1, True, chain, res=chain if bt.add else None)
                w3, b3 = _conv_params(m.cv3)
                add_conv(cat, w3, b3, 1, 1, 0, True, out[i])
            elif _is(m, "SPPF"):
                x = out[fs[0]]
                # the pooling kernel is the 5x5 / stride 1 / pad 2 window of every shipped yaml (common.py:183-196); the mirror
                # keeps `k`, the reference's module keeps the nn.MaxPool2d as `m`
                pk = getattr(m, "k", None)
                if pk is None and hasattr(m, "m"):
                    pk = m.m.kernel_size if isinstance(m.m.kernel_size, int) else m.m.kernel_size[0]
                if pk != 5:
                    raise RuntimeError(f"SPPF with a {pk}x{pk} pooling window is not planned (the kernel is 5x5)")
                c_ = m.cv1.conv.out_channels
                cat4 = new(hw[i][0], hw[i][1], 4 * c_)
                w1, b1 = _conv_params(m.cv1)
                add_conv(x, w1, b1, 1, 1, 0, True, Slice(cat4, 0, c_))
                hh, ww = hw[i]
                ptr, ps = cat4.data_ptr(), cat4.shape[3]
                self.ops.append(lambda st, ptr=ptr, ps=ps, hh=hh, ww=ww, c_=c_: L.y5obb_sppf_pool(ptr, ps, B, hh, ww, c_, st))
                self.hbm_bytes += 2.0 * B * hh * ww * c_ * 4
                w2, b2 = _conv_params(m.cv2)
                add_conv(Slice.full(cat4), w2, b2, 1, 1, 0, True, out[i])
            # Concat / Upsample emit nothing

        # ---- Detect
        self.no, self.na = det.no, det.na
        rows = [det.na * hw[f][0] * hw[f][1] for f in det.f]
        self.rows_total = sum(rows)
        # compact_detect: the Detect epilogue writes (cx, cy, w, h, obj, cls[nc], theta index) records - all that
        # non_max_suppression_obb reads of a row - instead of the [B, A, no] tensor (96 B instead of 800 B per anchor row)
        self.compact_detect = bool(compact_detect)
        self.rec_w = ((det.nc + 6) + 3) // 4 * 4
        self.nc = det.nc
        self.pred = torch.empty((B, self.rows_total, self.rec_w if compact_detect else det.no), dtype=torch.float32, device=device)
        row_off = 0
        for l, f in enumerate(det.f):
            mi = det.m[l]
            stride = float(det.stride[l])
            anchors_px = (det.anchors[l].detach().float().cpu() * stride).flatten().tolist()
            add_conv(out[f], mi.weight.detach().float().cpu(), mi.bias.detach().float().cpu(), 1, 1, 0, False,
                     detd=dict(out=self.pred, rows_per_image=self.rows_total, row_off=row_off, no=det.no,
                               decode=2 if compact_detect else True,
                               stride=stride, anchors_px=anchors_px))
            row_off += rows[l]
        self.hbm_bytes += 4.0 * B * self.rows_total * det.no + 4.0 * B * 3 * H * W + 2.0 * self.x_s2d.numel()
        self.n_launches = len(self.ops) + 1

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: [B,3,H,W] fp32 in [0,1] (or uint8 0..255) on this engine's device -> pred [B, A, no] fp32
        (engine-owned buffer, overwritten by the next call)."""
        _lib.require_cuda(x, "x")
        if tuple(x.shape) != (self.B, 3, self.H, self.W):
            raise RuntimeError(f"engine was planned for {(self.B, 3, self.H, self.W)}, got {tuple(x.shape)}")
        st = _lib.stream_ptr(self.device)
        L = _lib.lib()
        with torch.cuda.device(self.device):
            if x.dtype == torch.uint8:  # raw image: the caller-side `/ 255` is folded into the layout pass
                x = x.contiguous()
                _lib.check(L.y5obb_stem_s2d_u8(x.data_ptr(), self.x_s2d.data_ptr(), self.B, self.H, self.W, 1, st),
                           "y5obb_stem_s2d_u8")
            else:
                x = x.contiguous().float()
                _lib.check(L.y5obb_stem_s2d(x.data_ptr(), self.x_s2d.data_ptr(), self.B, self.H, self.W, 1, st),
                           "y5obb_stem_s2d")
            self._replay()
        return self.pred

    def forward_tiles(self, scene, origins: torch.Tensor, n_valid) -> torch.Tensor:
        """Runs the plan on B tiles cropped from whole scenes on the device (DOTA_devkit/ImgSplit_multi_process.py:226-273 at
        rate 1, without the patch files): scene is one uint8 [H, W, 3] BGR tensor (cv2.imread's layout) or a list of them,
        origins an int32 [B, 2] device tensor of tile (left, up), n_valid the number of tiles cut from each scene (an int, or
        one per scene; their tiles are consecutive in origins).  Tiles after the last valid one are zero.  Pixels outside a
        scene are zero (the devkit's padding), channels are flipped to RGB and scaled by 1/255 exactly as forward() does for a
        uint8 batch.  Returns the same engine-owned buffer as forward()."""
        scenes = [scene] if isinstance(scene, torch.Tensor) else list(scene)
        counts = [int(n_valid)] if isinstance(n_valid, int) else [int(k) for k in n_valid]
        if self.H != self.W or len(scenes) != len(counts) or not scenes:
            raise RuntimeError("forward_tiles needs a square plan and one tile count per scene")
        if tuple(origins.shape) != (self.B, 2) or origins.dtype != torch.int32 or not origins.is_contiguous():
            raise RuntimeError(f"origins must be a contiguous int32 [{self.B}, 2] tensor")
        _lib.require_cuda(origins, "origins")
        if any(k < 0 for k in counts) or sum(counts) > self.B:
            raise RuntimeError(f"tile counts {counts} do not fit a batch of {self.B}")
        st = _lib.stream_ptr(self.device)
        L = _lib.lib()
        with torch.cuda.device(self.device):
            b0 = 0
            for s, k in zip(scenes, counts):
                _lib.require_cuda(s, "scene")
                if s.dtype != torch.uint8 or s.dim() != 3 or s.shape[2] != 3 or not s.is_contiguous():
                    raise RuntimeError("a scene must be a contiguous uint8 [H, W, 3] tensor")
                if k:
                    _lib.check(L.y5obb_stem_s2d_scene_u8(s.data_ptr(), s.shape[0], s.shape[1], origins[b0].data_ptr(), k, k,
                                                         self.H, self.x_s2d[b0].data_ptr(), 1, st), "y5obb_stem_s2d_scene_u8")
                b0 += k
            if b0 < self.B:   # padding tiles: zeros (no scene pixel is read)
                _lib.check(L.y5obb_stem_s2d_scene_u8(scenes[0].data_ptr(), 1, 1, origins.data_ptr(), self.B - b0, 0, self.H,
                                                     self.x_s2d[b0].data_ptr(), 1, st), "y5obb_stem_s2d_scene_u8")
            self._replay()
        return self.pred

    def _replay(self):
        """The op list after the layout pass: the layer sequence is fixed (same buffers every call), so from the third call on
        it is replayed as one CUDA graph - the layout pass stays outside because it reads the caller's tensor
        (Y5OBB_NO_GRAPH=1 disables)."""
        self._calls += 1
        if self._use_graph and self._calls > 2:
            if self._graph is None:
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, capture_error_mode="thread_local"):
                    self._run_ops(_lib.stream_ptr(self.device))
                self._graph = g
            self._graph.replay()
        else:
            self._run_ops(_lib.stream_ptr(self.device))

    def _run_ops(self, st):
        for op in self.ops:
            rc = op(st)
            if rc:
                _lib.check(rc, "engine op")
