"""Host-side mirror of the reference model interface, executed by the sm_100a engine.

Mirrors /root/reference/models/yolo.py (Model :95-268, Detect :33-92, parse_model :271-323) and the
building blocks of /root/reference/models/common.py (Conv :37-49, Bottleneck :94-104, C3 :126-138,
SPPF :181-196, Concat :267-274): same constructor arguments, same module/parameter names (so a
reference state_dict loads unchanged), same forward() return values.  The modules here only HOLD
parameters; all arithmetic runs in csrc/ through the C ABI (engine.py).  There is no PyTorch compute
path in this package — the fp32 torch restatement used by the tests lives in oracle/model_ref.py.
"""
import math
from copy import deepcopy
from pathlib import Path

import torch
import torch.nn as nn

# ---------------------------------------------------------------------------------------------
# configuration (values of models/yolov5{n,s,m,l,x}.yaml, generated rather than stored)
# ---------------------------------------------------------------------------------------------
_SCALES = {"n": (0.33, 0.25), "s": (0.33, 0.50), "m": (0.67, 0.75), "l": (1.0, 1.0), "x": (1.33, 1.25)}
_ANCHORS = [[10, 13, 16, 30, 33, 23], [30, 61, 62, 45, 59, 119], [116, 90, 156, 198, 373, 326]]  # P3/8, P4/16, P5/32


def yolov5_cfg(size: str = "s", nc: int = 80) -> dict:
    """The v6.0 CSPDarknet + PANet layout (models/yolov5s.yaml:13-48) for a given scale letter."""
    gd, gw = _SCALES[size]
    backbone = [[-1, 1, "Conv", [64, 6, 2, 2]]]                      # 0  P1/2
    for width, depth in ((128, 3), (256, 6), (512, 9), (1024, 3)):   # 1-8: stride-2 conv + C3 per stage
        backbone += [[-1, 1, "Conv", [width, 3, 2]], [-1, depth, "C3", [width]]]
    backbone += [[-1, 1, "SPPF", [1024, 5]]]                          # 9
    head = []
    for width, skip in ((512, 6), (256, 4)):                          # top-down: 10-17
        head += [[-1, 1, "Conv", [width, 1, 1]], [-1, 1, "nn.Upsample", [None, 2, "nearest"]],
                 [[-1, skip], 1, "Concat", [1]], [-1, 3, "C3", [width, False]]]
    for width, skip in ((256, 14), (512, 10)):                        # bottom-up: 18-23
        head += [[-1, 1, "Conv", [width, 3, 2]], [[-1, skip], 1, "Concat", [1]], [-1, 3, "C3", [2 * width, False]]]
    head += [[[17, 20, 23], 1, "Detect", ["nc", "anchors"]]]          # 24
    return dict(nc=nc, depth_multiple=gd, width_multiple=gw, anchors=deepcopy(_ANCHORS), backbone=backbone, head=head)


def make_divisible(x, divisor):
    return math.ceil(x / divisor) * divisor


def autopad(k, p=None):
    return k // 2 if p is None else p


# ---------------------------------------------------------------------------------------------
# parameter containers (names match the reference modules)
# ---------------------------------------------------------------------------------------------
class _NoTorchPath(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError(f"{type(self).__name__} holds parameters only; run the model through "
                           "yolov5_obb_b200.yolo.Model.forward (sm_100a engine) — there is no PyTorch fallback")


class Conv(_NoTorchPath):
    def __init__(self, c1, c2, k=1, s=1, p=None, g=1, act=True):
        super().__init__()
        assert g == 1, "grouped convs are not used by yolov5{n,s,m,l,x}.yaml"
        self.conv = nn.Conv2d(c1, c2, k, s, autopad(k, p), groups=g, bias=False)
        self.bn = nn.BatchNorm2d(c2)
        self.act = nn.SiLU() if act is True else nn.Identity()


class Bottleneck(_NoTorchPath):
    def __init__(self, c1, c2, shortcut=True, g=1, e=0.5):
        super().__init__()
        c_ = int(c2 * e)
        self.cv1 = Conv(c1, c_, 1, 1)
        self.cv2 = Conv(c_, c2, 3, 1, g=g)
        self.add = shortcut and c1 == c2


class C3(_NoTorchPath):
    def __init__(self, c1, c2, n=1, shortcut=True, g=1, e=0.5):
        super().__init__()
        c_ = int(c2 * e)
        self.cv1 = Conv(c1, c_, 1, 1)
        self.cv2 = Conv(c1, c_, 1, 1)
        self.cv3 = Conv(2 * c_, c2, 1)
        self.m = nn.Sequential(*(Bottleneck(c_, c_, shortcut, g, e=1.0) for _ in range(n)))


class SPPF(_NoTorchPath):
    def __init__(self, c1, c2, k=5):
        super().__init__()
        assert k == 5
        c_ = c1 // 2
        self.cv1 = Conv(c1, c_, 1, 1)
        self.cv2 = Conv(c_ * 4, c2, 1, 1)
        self.k = k


class Concat(_NoTorchPath):
    def __init__(self, dimension=1):
        super().__init__()
        self.d = dimension


class Upsample(_NoTorchPath):
    """nn.Upsample(None, 2, 'nearest') placeholder (no parameters)."""

    def __init__(self, size=None, scale_factor=2, mode="nearest"):
        super().__init__()
        assert size is None and scale_factor == 2 and mode == "nearest"
        self.scale_factor, self.mode = scale_factor, mode


class Detect(_NoTorchPath):
    stride = None

    def __init__(self, nc=80, anchors=(), ch=(), inplace=True):
        super().__init__()
        self.nc = nc
        self.no = nc + 5 + 180  # models/yolo.py:40
        self.nl = len(anchors)
        self.na = len(anchors[0]) // 2
        self.register_buffer("anchors", torch.tensor(anchors).float().view(self.nl, -1, 2))
        self.m = nn.ModuleList(nn.Conv2d(x, self.no * self.na, 1) for x in ch)
        self.inplace = inplace


_MODULES = {"Conv": Conv, "C3": C3, "SPPF": SPPF, "Concat": Concat, "nn.Upsample": Upsample, "Detect": Detect}


def parse_model(d: dict, ch: list):
    """models/yolo.py:271-323 for the module types the shipped yamls use."""
    anchors, nc, gd, gw = d["anchors"], d["nc"], d["depth_multiple"], d["width_multiple"]
    na = (len(anchors[0]) // 2) if isinstance(anchors, list) else anchors
    no = na * (nc + 185)
    layers, save, c2 = [], [], ch[-1]
    for i, (f, n, m, args) in enumerate(d["backbone"] + d["head"]):
        name = m if isinstance(m, str) else m.__name__
        if name not in _MODULES:
            raise RuntimeError(f"module {name!r} is outside the hot path (only {sorted(_MODULES)} are built)")
        cls = _MODULES[name]
        args = [nc if a == "nc" else anchors if a == "anchors" else (None if a == "None" else a) for a in args]
        n_ = max(round(n * gd), 1) if n > 1 else n
        if cls in (Conv, C3, SPPF):
            c1, c2 = ch[f], args[0]
            if c2 != no:
                c2 = make_divisible(c2 * gw, 8)
            args = [c1, c2, *args[1:]]
            if cls is C3:
                args.insert(2, n_)
                n_ = 1
        elif cls is Concat:
            c2 = sum(ch[x] for x in f)
        elif cls is Detect:
            args.append([ch[x] for x in f])
            if isinstance(args[1], int):
                args[1] = [list(range(args[1] * 2))] * len(f)
        else:
            c2 = ch[f]
        assert n_ == 1, "repeated non-C3 modules do not occur in the shipped yamls"
        m_ = cls(*args)
        m_.i, m_.f, m_.type = i, f, name
        m_.np = sum(x.numel() for x in m_.parameters())
        save.extend(x % i for x in ([f] if isinstance(f, int) else f) if x != -1)
        layers.append(m_)
        if i == 0:
            ch = []
        ch.append(c2)
    return nn.Sequential(*layers), sorted(save)


class _TrainFn(torch.autograd.Function):
    """Training-mode forward / backward of the whole network as one autograd node (what train.py:324-333 drives):
    forward = train_engine.TrainEngine.forward, backward = train_backward.BackwardPlan.run.  The parameters are
    inputs of the node so that autograd accumulates their gradients into `.grad` itself."""

    @staticmethod
    def forward(ctx, eng, x, *params):
        outs = eng.forward(x, getattr(eng, "_refresh_next", False))
        ctx.eng, ctx.params = eng, params
        return tuple(o.detach() for o in outs)

    @staticmethod
    def backward(ctx, *grads):
        plan = ctx.eng.backward(list(grads))
        # one clone of the flat buffer: autograd may keep the returned views as .grad (zero_grad(set_to_none=True) makes
        # that copy-free), and the plan rewrites its own buffer every step
        flat = plan.flat.clone()
        ctx.eng.last_grad_flat = flat
        views = {p: flat[o:o + p.numel()].view(p.shape) for p, o in zip(plan.params, plan.offsets)}
        return (None, None) + tuple(views.get(p) for p in ctx.params)


class Model(nn.Module):
    """Drop-in for models/yolo.py:95 Model: Model(cfg, ch=3, nc=None, anchors=None); forward(x[B,3,H,W] in [0,1])
    -> eval: (pred[B, sum(3*H_i*W_i), nc+185] fp32, None); train: list of 3 [B,3,H_i,W_i,nc+185] logits."""

    def __init__(self, cfg="yolov5s.yaml", ch=3, nc=None, anchors=None):
        super().__init__()
        if isinstance(cfg, dict):
            self.yaml = deepcopy(cfg)
        else:
            p = Path(str(cfg))
            if p.exists():  # a reference-style yaml file
                import yaml
                self.yaml_file = p.name
                with open(p, encoding="ascii", errors="ignore") as f:
                    self.yaml = yaml.safe_load(f)
            else:  # "yolov5s.yaml" / "yolov5s" / "s"
                key = p.stem.replace("yolov5", "")
                if key not in _SCALES:
                    raise FileNotFoundError(cfg)
                self.yaml_file = f"yolov5{key}.yaml"
                self.yaml = yolov5_cfg(key)
        ch = self.yaml["ch"] = self.yaml.get("ch", ch)
        if nc and nc != self.yaml["nc"]:
            self.yaml["nc"] = nc
        if anchors:
            self.yaml["anchors"] = round(anchors)
        self.model, self.save = parse_model(deepcopy(self.yaml), ch=[ch])
        self.names = [str(i) for i in range(self.yaml["nc"])]
        self.inplace = self.yaml.get("inplace", True)

        m = self.model[-1]
        assert isinstance(m, Detect)
        m.inplace = self.inplace
        m.stride = torch.tensor(self._strides())  # the reference probes a 256x256 forward (yolo.py:121-123)
        m.anchors /= m.stride.view(-1, 1, 1)
        self.stride = m.stride
        self._initialize_biases()
        for mod in self.modules():  # utils/torch_utils.py:154-166 initialize_weights
            if isinstance(mod, nn.BatchNorm2d):
                mod.eps = 1e-3
                mod.momentum = 0.03
        self._engines = {}
        self._fused = False
        self._generation = 0

    def _bump_generation(self):
        """Explicit staleness signal for the inference plans: called by everything that writes parameters or statistics
        through raw pointers (training forwards, the fused optimizer step, a start-up broadcast), which tensor version
        counters do not see."""
        self._generation = getattr(self, "_generation", 0) + 1

    def _strides(self):
        s, out = [], {}
        for m in self.model:
            f = m.f if isinstance(m.f, int) else m.f[0]
            src = (m.i - 1 if f == -1 else f)
            cur = out.get(src, 1.0) if m.i > 0 else 1.0
            if isinstance(m, Conv) and m.conv.stride[0] == 2:
                cur *= 2
            elif isinstance(m, Upsample):
                cur /= 2
            out[m.i] = cur
        det = self.model[-1]
        for j in det.f:
            s.append(float(out[j]))
        return s

    def _initialize_biases(self, cf=None):  # models/yolo.py:223-232 (touches the 180 theta channels too)
        m = self.model[-1]
        for mi, s in zip(m.m, m.stride):
            b = mi.bias.view(m.na, -1)
            b.data[:, 4] += math.log(8 / (640 / s) ** 2)
            b.data[:, 5:] += math.log(0.6 / (m.nc - 0.999999)) if cf is None else torch.log(cf / cf.sum())
            mi.bias = torch.nn.Parameter(b.view(-1), requires_grad=True)

    def fuse(self):
        """models/yolo.py:246-254.  BN folding happens when an engine packs weights (engine.py uses
        fuse_conv_and_bn arithmetic, utils/torch_utils.py:192-212); this only records the request."""
        self._fused = True
        return self

    def invalidate(self):
        """Drop every plan (packed weights, buffers, captured graphs); the next forward re-plans."""
        self._engines.clear()
        self._sig_tensors = None

    def __deepcopy__(self, memo):
        """copy.deepcopy(model) (ModelEMA, checkpoints): parameters and buffers are copied, the device plans are not."""
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        skip = ("_engines", "_last_train_engine", "_sig_tensors", "_sig_nbt")
        new.__dict__ = {k: deepcopy(v, memo) for k, v in self.__dict__.items() if k not in skip}
        new._engines = {}
        new._sig_tensors = None
        return new

    def _apply(self, fn, *args, **kwargs):  # .to() / .cuda() / .float(): the plans point at the old storages
        if getattr(self, "_engines", None):
            self._engines.clear()
        self._sig_tensors = None
        return super()._apply(fn, *args, **kwargs)

    def forward(self, x, augment=False, profile=False, visualize=False):
        if augment or profile or visualize:
            raise RuntimeError("augment/profile/visualize are host tooling outside the hot path")
        if self.training:
            from .train_engine import TrainEngine
            key = ("train", tuple(x.shape), x.device.index)
            eng = self._engines.get(key)
            refresh = eng is not None          # an existing plan re-packs the (possibly updated) parameters first
            if eng is None:
                eng = self._engines[key] = TrainEngine(self, x.shape[0], x.shape[2], x.shape[3], x.device)
            eng._refresh_next = refresh
            self._last_train_engine = eng
            self._bump_generation()  # running statistics move (the captured graph bumps no version counter)
            if not torch.is_grad_enabled():
                return eng.forward(x, refresh)
            params = [p for p in self.parameters() if p.requires_grad]
            return list(_TrainFn.apply(eng, x, *params))
        from .engine import InferenceEngine
        key = (tuple(x.shape), x.device.index)
        eng = self._engines.get(key)
        # The inference plan folds BatchNorm into packed bf16 weights when it is built.  Parameters and statistics that
        # were updated in place since then (optimizer / EMA steps, load_state_dict, a training forward) show up in the
        # tensors' version counters or in num_batches_tracked: the plan is then rebuilt (val after every epoch, train.py:352).
        sig = self._weights_signature()
        if eng is None or eng._weights_sig != sig:
            eng = self._engines[key] = InferenceEngine(self, x.shape[0], x.shape[2], x.shape[3], x.device)
            eng._weights_sig = sig
        return eng.forward(x), None

    def detect_records(self, x, slot: int = 0):
        """Eval-mode forward for the fused post-process: instead of the [B, A, nc+185] tensor the Detect epilogue writes, per
        anchor row, the compact record (cx, cy, w, h, obj, cls[nc], theta index) - everything non_max_suppression_obb reads
        (utils/general.py:781-832) - so 96 B instead of 800 B per row cross HBM, once instead of three times.  Returns a
        general.DetectRecords, accepted by yolov5_obb_b200.general.non_max_suppression_obb in place of the prediction
        tensor (bit-identical detections: same sigmoid / decode arithmetic, same first-maximum theta rule).
        `slot` selects one of several independent plans of the same shape (own activation and record buffers, own captured
        graph): batches in flight on DIFFERENT streams must use different slots (pipeline.DetectPipeline does)."""
        if self.training:
            raise RuntimeError("detect_records is an inference entry point (model.eval())")
        from .general import DetectRecords
        eng = self._records_engine(tuple(x.shape), x.device, slot)
        return DetectRecords(eng.forward(x), eng.nc)

    def detect_records_tiles(self, scene, origins, n_valid, tile: int, slot: int = 0):
        """detect_records on tiles cut from whole scenes on the device (InferenceEngine.forward_tiles): scene a uint8
        [H, W, 3] BGR tensor or a list of them, origins int32 [B, 2] (left, up) on their device, n_valid tiles per scene (an
        int or one per scene), the rest of the batch padding.  Runs the plan detect_records uses for a [B, 3, tile, tile]
        batch (same buffers, same captured graph) and returns its records."""
        if self.training:
            raise RuntimeError("detect_records_tiles is an inference entry point (model.eval())")
        from .general import DetectRecords
        eng = self._records_engine((origins.shape[0], 3, int(tile), int(tile)), origins.device, slot)
        return DetectRecords(eng.forward_tiles(scene, origins, n_valid), eng.nc)

    def _records_engine(self, shape, device, slot):
        from .engine import InferenceEngine
        key = ("records", tuple(shape), device.index) + ((int(slot),) if slot else ())
        eng = self._engines.get(key)
        sig = self._weights_signature()
        if eng is None or eng._weights_sig != sig:
            eng = self._engines[key] = InferenceEngine(self, shape[0], shape[2], shape[3], device, compact_detect=True)
            eng._weights_sig = sig
        return eng

    def _weights_signature(self):
        tr = getattr(self, "_sig_tensors", None)
        if tr is None:
            tr = self._sig_tensors = list(self.parameters()) + [b for b in self.buffers() if b.dtype.is_floating_point]
            self._sig_nbt = [b for n, b in self.named_buffers() if n.endswith("num_batches_tracked")]
        # (the training kernels write running statistics through raw pointers: they bump num_batches_tracked, which a
        # torch op increments, so the sum of its version counters moves with every training forward)
        return (sum(t._version for t in tr), sum(t._version for t in self._sig_nbt), id(tr[0]) if tr else 0,
                getattr(self, "_generation", 0))
