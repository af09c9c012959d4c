"""Backward pass of the training plan (train_engine.TrainEngine): what autograd + cuDNN do under
`scaler.scale(loss).backward()` (/root/reference/train.py:333) for the Conv/C3/SPPF/Concat/Upsample/Detect graph,
as a fixed sequence of sm_100a kernel launches.

Per Conv module (y = [res +] silu(bn(conv(x))), reverse order):
   gy (+ 2x-up-sampled copy's gradient folded in)  --y5obb_bn_silu_bwd-->  dz, dgamma, dbeta, residual pass-through
   dz, x  --y5obb_wgrad (both read in place, NHWC)-->  dW (tensor cores, split-K)
   dz     --conv_tc_kernel with transposed / flipped weights (dgrad; stride 2: over the zero-stuffed dz)-->  gx (+=)
Gradient buffers mirror the activation buffers; whether a contribution overwrites or accumulates is decided
statically when the plan is built (first writer of a channel range overwrites).
Parameter gradients land in views of ONE flat fp32 buffer owned by the plan (run() returns it); the autograd
Function in yolo.py hands them to autograd, which accumulates into `.grad` (so GradScaler / DDP hooks see them).
"""
from typing import Dict, List, Optional

import torch

from . import _lib
from .conv import Conv as ConvOp, Slice, pack_weights, tiling, MODE_DETECT
from .train_ops import Wgrad


class _Written:
    """Which channel ranges of each gradient buffer already hold a contribution in this backward pass."""

    def __init__(self):
        self.r: Dict[int, List] = {}

    def contribute(self, s: Slice) -> bool:
        """Returns True if the contribution must ACCUMULATE (range already written), False if it overwrites."""
        key = s.buf.data_ptr()
        lo, hi = s.c_off, s.c_off + s.C
        ranges = self.r.setdefault(key, [])
        overlap = [(a, b) for a, b in ranges if a < hi and lo < b]
        if not overlap:
            ranges.append((lo, hi))
            return False
        covered = sorted(overlap)
        pos = lo
        for a, b in covered:
            if a > pos:
                raise RuntimeError("gradient range partially written: unsupported graph")
            pos = max(pos, b)
        if pos < hi:
            raise RuntimeError("gradient range partially written: unsupported graph")
        return True

    def covered(self, s: Slice) -> bool:
        key = s.buf.data_ptr()
        lo, hi = s.c_off, s.c_off + s.C
        pos = lo
        for a, b in sorted(self.r.get(key, [])):
            if a <= pos < b:
                pos = b
        return pos >= hi


class BackwardPlan:
    def __init__(self, eng):
        self.eng = eng
        dev = eng.device
        B = eng.B
        L = _lib.lib()
        self._L = L
        self.gbuf: Dict[int, torch.Tensor] = {}
        self.steps = []  # (name, closure(stream))
        # The weight gradients are leaves of the backward chain (bn_bwd(l) -> {wgrad(l), dgrad(l)} -> bn_bwd(l-1) -> ...): they
        # run on a second stream, each ordered after the kernel that produced its dz, and are joined before the few
        # re-mapping copies at the end - so wgrad_kernel (tensor-bound, one 60 KB CTA per SM) shares the SMs with the
        # HBM-bound BatchNorm backward passes and fills the tails of the dgrad launches.  Every wgrad reads buffers nothing
        # writes after its producer (its own dz, the saved activation) and accumulates into its own slice of the flat
        # gradient buffer, so only the interleaving changes.
        self.side = torch.cuda.Stream(dev)
        self.prof = None  # set to {} to collect per-step-kind device times (ms) during run()

        def add(tag, fn):
            self.steps.append((tag, fn))

        self.keep = []
        self.flops = 0.0
        written = _Written()
        det = eng.model.model[-1]

        def gslice(s: Slice) -> Slice:
            k = s.buf.data_ptr()
            if k not in self.gbuf:
                self.gbuf[k] = torch.zeros_like(s.buf)
            return Slice(self.gbuf[k], s.c_off, s.C)

        def f32(n):
            t = torch.zeros(n, dtype=torch.float32, device=dev)
            self.keep.append(t)
            return t

        def bf(*shape):
            t = torch.zeros(shape, dtype=torch.bfloat16, device=dev)
            self.keep.append(t)
            return t

        # one flat fp32 buffer holds every parameter gradient (model.parameters() order): the kernels write into
        # views of it, a data-parallel job all-reduces it in one call
        self.params = [p for p in eng.model.parameters()]
        self.offsets, n = [], 0
        for p in self.params:
            self.offsets.append(n)
            n += (p.numel() + 3) // 4 * 4  # 16-byte aligned views
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.pgrad: Dict[torch.nn.Parameter, torch.Tensor] = {
            p: self.flat[o:o + p.numel()].view(p.shape) for p, o in zip(self.params, self.offsets)}

        def grad_of(p: torch.nn.Parameter) -> torch.Tensor:
            return self.pgrad[p]

        self._grad_of = grad_of

        def add_dgrad(dz_slice: Slice, w_dgrad, k, pad, gx: Slice, name):
            """gx (+)= conv(dz, w_dgrad) with stride 1."""
            acc = written.contribute(gx)
            wp, bp = pack_weights(w_dgrad, None)
            op = ConvOp(dz_slice, wp, bp, w_dgrad.shape[0], k, 1, pad, False, out=gx, res=gx if acc else None)
            self.flops += op.info()["flops"]
            add("dgrad", lambda st, h=op._h: _lib.check(L.y5obb_conv_run(h, st), name))
            return op, wp

        # ---------------- Detect levels ----------------
        self.det_grads_in = [torch.zeros_like(o) for o in eng.det_out]  # static copies of dLoss/dpred (graph inputs)
        self._calls, self._graph = 0, None
        self.det_parts = []
        for l in range(det.nl):
            cv = eng.det_convs[l]
            xin: Slice = cv._keep[0]
            mi = det.m[l]
            H, W, Cin = xin.H, xin.W, xin.C
            bk, bn, cin_pad, cout_pad, nt = tiling(Cin, det.na * det.no, MODE_DETECT, det.no)
            dzd = bf(B, H, W, det.na * bn)
            s1, s2 = f32(det.na * bn), f32(det.na * bn)
            part = dict(l=l, dzd=dzd, s1=s1, bn=bn, Cin=Cin, mi=mi)
            self.det_parts.append(part)

            def pack_step(st, l=l, dzd=dzd, H=H, W=W, bn=bn):
                g = self.det_grads_in[l]
                _lib.check(L.y5obb_detect_grad_pack(g.data_ptr(), dzd.data_ptr(), B, det.na, H, W, det.no, bn, st), "detect_grad_pack")
            add("detect_pack", pack_step)
            # bias gradient = per-channel sums of dz
            add("detect_bias", lambda st, dzd=dzd, s1=s1, s2=s2, n=B * H * W, C=det.na * bn:
                              _lib.check(L.y5obb_bn_stats(dzd.data_ptr(), C, n, C, s1.data_ptr(), s2.data_ptr(), eng.scratch.data_ptr(),
                                                          eng.scratch.numel(), st), "detect bias grad"))
            wg = Wgrad(dzd.data_ptr(), det.na * bn, xin.ptr, xin.pix_stride, grad_of(mi.weight), B, det.na * bn, H, W, Cin, H, W,
                       1, 1, 0, keep=(dzd, xin.buf, self.flat), param_layout=True, co_group=(det.no, bn))
            self.keep.append(wg)
            self.flops += 2.0 * B * H * W * det.na * bn * Cin
            add("wgrad", lambda st, wg=wg: wg.run(st))
            # dgrad: gx (+)= dz @ W  (1x1): weights [Cout'=Cin][Cin'=na*bn]
            wT = torch.zeros((Cin, det.na * bn, 1, 1), device=dev)
            part["wT"] = wT
            op, wp = add_dgrad(Slice.full(dzd), wT, 1, 0, gslice(xin), "detect dgrad")
            part["dgrad_wp"] = wp
            self.keep.append(op)

        # ---------------- conv layers, reverse ----------------
        self.conv_parts = []
        for lay in reversed(eng.layers):
            if isinstance(lay, tuple):
                _, cat4, hh, ww, c_ = lay
                gc = gslice(Slice.full(cat4))
                npix = B * hh * ww
                t2, t1, t0 = f32(npix * c_), f32(npix * c_), f32(npix * c_)
                ps = cat4.shape[3]
                base, gbase = cat4.data_ptr(), gc.buf.data_ptr()

                def pool_bwd(st, base=base, gbase=gbase, ps=ps, c_=c_, hh=hh, ww=ww, t2=t2, t1=t1, t0=t0, npix=npix):
                    t2.zero_(); t1.zero_(); t0.zero_()
                    # y3 = m(y2): gradient of y3 routed into y2
                    _lib.check(L.y5obb_maxpool5_bwd(base + 2 * (2 * c_), ps, None, gbase + 2 * (3 * c_), ps, t2.data_ptr(), B, hh, ww, c_, st), "pool bwd 3")
                    _lib.check(L.y5obb_maxpool5_bwd(base + 2 * (1 * c_), ps, t2.data_ptr(), gbase + 2 * (2 * c_), ps, t1.data_ptr(), B, hh, ww, c_, st), "pool bwd 2")
                    _lib.check(L.y5obb_maxpool5_bwd(base, ps, t1.data_ptr(), gbase + 2 * (1 * c_), ps, t0.data_ptr(), B, hh, ww, c_, st), "pool bwd 1")
                    _lib.check(L.y5obb_add_f32_to_bf16(t0.data_ptr(), gbase, ps, npix, c_, 1, st), "pool bwd add")
                if not written.covered(gc):
                    raise RuntimeError("SPPF gradient not ready")
                add("pool_bwd", pool_bwd)
                continue

            mod, z, y = lay.mod, lay.z, lay.y
            conv, bn = mod.conv, mod.bn
            k, s, p = conv.kernel_size[0], conv.stride[0], conv.padding[0]
            Cout, Hh, Ww = z.C, z.H, z.W
            npix = B * Hh * Ww
            gy = gslice(y)
            if lay.y2x is not None:  # fold the up-sampled copy's gradient into gy
                g2 = gslice(lay.y2x)
                acc = written.contribute(gy)
                add("upsample_bwd", lambda st, g2=g2, gy=gy, npix=npix, C=Cout, W=Ww, acc=acc:
                                  _lib.check(L.y5obb_upsample2x_bwd(g2.ptr, g2.pix_stride, gy.ptr, gy.pix_stride, npix, C, W, int(acc), st), "upsample bwd"))
            if not written.covered(gy):
                names = {id(mm): nn_ for nn_, mm in eng.model.named_modules()}
                raise RuntimeError(f"gradient of {names.get(id(mod))}'s output [{y.c_off}, {y.c_off + y.C}) of a "
                                   f"{tuple(y.buf.shape)} buffer is not produced before it is consumed; written: "
                                   f"{written.r.get(gy.buf.data_ptr())}")
            dz = bf(B, Hh, Ww, Cout)
            s1, s2 = f32(Cout), f32(Cout)
            gres, gacc = None, 0
            if lay.res is not None:
                gres = gslice(lay.res)
                gacc = int(written.contribute(gres))
            part = dict(lay=lay, dz=dz)
            self.conv_parts.append(part)

            dg, db = grad_of(bn.weight), grad_of(bn.bias)

            def bn_bwd(st, lay=lay, z=z, gy=gy, dz=dz, s1=s1, s2=s2, gres=gres, gacc=gacc, npix=npix, C=Cout, dg=dg, db=db):
                _lib.check(L.y5obb_bn_silu_bwd(z.ptr, z.pix_stride, gy.ptr, gy.pix_stride, npix, C, lay.scale.data_ptr(),
                                               lay.shift.data_ptr(), lay.mean.data_ptr(), lay.invstd.data_ptr(), int(lay.act),
                                               s1.data_ptr(), s2.data_ptr(), dz.data_ptr(), C,
                                               gres.ptr if gres else None, gres.pix_stride if gres else 0, gacc,
                                               dg.data_ptr(), db.data_ptr(), 0, eng.scratch.data_ptr(), eng.scratch.numel(), st),
                           "bn_silu_bwd")
            add("bn_bwd", bn_bwd)

            # ---- wgrad (straight from the NHWC buffers)
            x = lay.x
            if lay.stem:  # the forward's view: a 3x1 conv over 48-channel windows (3 horizontal taps x 16 s2d channels)
                Wp = eng.W // 2 + 2
                Hi, Wi, Cin_w = eng.H // 2, eng.W // 2, 48
                kw_, sw_, pw_ = (3, 1), 1, (1, 0)
                x_ptr, x_ps, x_keep = eng.x_s2d.data_ptr(), 16, eng.x_s2d
                x_strides = (Wp * 16, (eng.H // 2) * Wp * 16)
            else:
                Hi, Wi, Cin_w = x.H, x.W, x.C
                kw_, sw_, pw_ = k, s, p
                x_ptr, x_ps, x_keep = x.ptr, x.pix_stride, x.buf
                x_strides = (0, 0)
            ntap = kw_[0] * kw_[1] if isinstance(kw_, tuple) else kw_ * kw_
            if lay.stem:  # gradient over the space-to-depth form, re-mapped to [Cout,3,6,6] at the end of run()
                dw = f32(3 * Cout * 48)
                part["stem_dw"] = dw
                add("zero", lambda st, dw=dw: dw.zero_())
                wg = Wgrad(dz.data_ptr(), Cout, x_ptr, x_ps, dw, B, Cout, Hh, Ww, Cin_w, Hi, Wi, kw_, sw_, pw_, keep=(dz, x_keep),
                           x_strides=x_strides)
            else:
                wg = Wgrad(dz.data_ptr(), Cout, x_ptr, x_ps, grad_of(conv.weight), B, Cout, Hh, Ww, Cin_w, Hi, Wi, kw_, sw_, pw_,
                           keep=(dz, x_keep, self.flat), param_layout=True)
            self.keep.append(wg)
            self.flops += 2.0 * npix * Cout * Cin_w * ntap
            add("wgrad", lambda st, wg=wg: wg.run(st))

            # ---- dgrad
            if not lay.stem:
                gx = gslice(x)
                w_d = torch.zeros((x.C, Cout, k, k), device=dev)  # filled by refresh()
                part["w_d"] = w_d
                if s == 1:
                    op, wp = add_dgrad(Slice.full(dz), w_d, k, k - 1 - p, gx, "dgrad")
                    part["dgrad_wp"] = wp
                    self.keep.append(op)
                elif k == 3 and p == 1 and x.H % 2 == 0 and x.W % 2 == 0:
                    # Output pixels of parity (ph, pw) only see the taps of matching parity: four 1- / 2-tap stride-1
                    # convolutions of dz, each written to every other pixel of gx - 9 tap-GEMMs per 4 outputs instead of
                    # the 36 of the zero-stuffed form.
                    acc = written.contribute(gx)
                    ps = gx.pix_stride
                    part["dgrad_s2"] = []
                    for ph in range(2):
                        for pw in range(2):
                            kh2, kw2 = (2 if ph else 1), (2 if pw else 1)
                            wp, bp = pack_weights(torch.zeros((x.C, Cout, kh2, kw2), device=dev), None)
                            geom = dict(h=Hh, w=Ww, off=(ph * x.W + pw) * ps, pix=2 * ps, row=2 * x.W * ps, img=x.H * x.W * ps)
                            op = ConvOp(Slice.full(dz), wp, bp, x.C, (kh2, kw2), 1, (0, 0), False, out=gx,
                                        res=gx if acc else None, out_geom=geom)
                            self.flops += op.info()["flops"]
                            add("dgrad", lambda st, h=op._h: _lib.check(L.y5obb_conv_run(h, st), "dgrad s2 phase"))
                            part["dgrad_s2"].append((ph * 2 + pw, wp))
                            self.keep.append(op)
                else:
                    dzup = bf(B, x.H, x.W, Cout)
                    add("zero_stuff", lambda st, dz=dz, dzup=dzup, npix=npix, C=Cout, W=Ww:
                                      _lib.check(L.y5obb_zero_stuff2x(dz.data_ptr(), C, dzup.data_ptr(), C, npix, C, W, st), "zero_stuff"))
                    op, wp = add_dgrad(Slice.full(dzup), w_d, k, k - 1 - p, gx, "dgrad s2")
                    part["dgrad_wp"] = wp
                    self.keep.append(op)
        self.refresh()

    # ------------------------------------------------------------------------------------------
    def pack_entries(self):
        """(kind, fp32 parameter, packed bf16 buffer, group_real, group_pad) of every data-gradient weight buffer."""
        from .train_ops import PACK_DGRAD, PACK_DETECT_DGRAD, PACK_DGRAD_S2
        det = self.eng.model.model[-1]
        ent = [(PACK_DETECT_DGRAD, part["mi"].weight.data, part["dgrad_wp"], det.no, part["bn"]) for part in self.det_parts]
        ent += [(PACK_DGRAD, part["lay"].mod.conv.weight.data, part["dgrad_wp"], 0, 0) for part in self.conv_parts
                if "dgrad_wp" in part]
        for part in self.conv_parts:
            for phase, wp in part.get("dgrad_s2", ()):
                ent.append((PACK_DGRAD_S2, part["lay"].mod.conv.weight.data, wp, phase, 0))
        return ent

    def refresh(self):
        """Pack the data-gradient weights (W transposed, taps flipped) from the current parameters."""
        from .train_ops import PackPlan
        PackPlan(self.pack_entries(), self.eng.device).run()

    def run(self, grads: List[torch.Tensor]):
        """grads: dLoss/dp for the 3 Detect outputs (fp32, same shapes as TrainEngine.det_out)."""
        eng = self.eng
        det = eng.model.model[-1]
        st = _lib.stream_ptr(eng.device)
        with torch.cuda.device(eng.device), torch.no_grad():
            for l in range(det.nl):
                g = grads[l]
                if g is None:
                    self.det_grads_in[l].zero_()
                else:
                    self.det_grads_in[l].copy_(g)
            if self.prof is not None or not eng.use_graph:
                self._launch_all(st)
            else:  # first run eager, second captured, then ONE graph launch replaces ~700 kernel launches
                self._calls += 1
                if self._calls == 1:
                    self._launch_all(st)
                else:
                    if self._graph is None:
                        torch.cuda.synchronize(eng.device)
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g, capture_error_mode="thread_local"):
                            self._launch_all(_lib.stream_ptr(eng.device))
                        self._graph = g
                    self._graph.replay()
        return self.flat

    def _launch_all(self, st):
        eng = self.eng
        det = eng.model.model[-1]
        with torch.no_grad():
            self.flat.zero_()
            if self.prof is None:
                cur, side = torch.cuda.current_stream(eng.device), self.side
                side.wait_stream(cur)                       # fork (after the flat buffer was zeroed)
                for tag, step in self.steps:
                    if tag in ("wgrad", "zero"):            # ("zero": the stem's own dw buffer, cleared on the wgrad's stream)
                        ev = torch.cuda.Event()
                        ev.record(cur)                      # the step before it on the main chain produced its dz
                        side.wait_event(ev)
                        with torch.cuda.stream(side):
                            step(side.cuda_stream)
                    else:
                        step(st)
                cur.wait_stream(side)                       # join: the copies below read the weight gradients
            else:  # debug: CUDA events around every step, summed per kind (and listed per wgrad / dgrad layer)
                evs = []
                for tag, step in self.steps:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    step(st)
                    e1.record()
                    evs.append((tag, e0, e1))
                torch.cuda.synchronize()
                self.prof = {}
                for tag, e0, e1 in evs:
                    self.prof.setdefault(tag, []).append(e0.elapsed_time(e1))
            # ---- the few gradients that need a re-mapping (tiny tensors)
            for part in self.det_parts:
                mi, bn = part["mi"], part["bn"]
                self.pgrad[mi.bias].copy_(part["s1"].view(det.na, bn)[:, :det.no].reshape(-1))
            for part in self.conv_parts:
                if "stem_dw" in part:  # dw[ty][co][tx * 16 + (dy*2+dx)*3 + c] is the gradient of w[co, c, 2ty+dy, 2tx+dx]
                    conv = part["lay"].mod.conv
                    dw = part["stem_dw"].view(3, conv.out_channels, 3, 16).permute(1, 3, 0, 2)  # [co, ch16, ty, tx]
                    g = self.pgrad[conv.weight]
                    for dy in range(2):
                        for dx in range(2):
                            g[:, :, dy::2, dx::2].copy_(dw[:, (dy * 2 + dx) * 3:(dy * 2 + dx) * 3 + 3])
        return self.flat
