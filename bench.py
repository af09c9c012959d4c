#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its single-GPU configuration.

Workload (config.workload): configs[1] = yolov5s-OBB inference, batch 16, 1024x1024 synthetic DOTA-shaped
tiles, the three stages the reference's `val.py --task speed` times (val.py:183-207): pre-process
(uint8 -> normalised), inference (Model.forward), NMS (non_max_suppression_obb, conf 0.25 / IoU 0.45,
val.py:378-383).  Metric: images/s.

  value      whole-job images/s with the uint8 batch already resident in HBM (device timing, CUDA events,
             max over ranks); the step is Model.detect_records + non_max_suppression_obb: Model.forward with the Detect rows
             written as the compact records the post-process reads (checked equal to Model.forward + NMS before timing)
  e2e        the same step through the public API from PINNED HOST memory: H2D of the uint8 batch and D2H
             of the detections inside the timed region
  roofline   conv_tc_kernel (tcgen05 implicit GEMM), the dominant kernel: algorithmic conv FLOPs per launch
             / mean launch duration measured with CUDA events around every launch in the timed steps,
             against MEASURED_PEAKS.json's burst bf16 figure (frac) and its sustained one (frac_sustained)
  parity     the benchmarked plan checked against the fp32 oracle before anything is timed (bf16-noise-floor rule), and the
             fused Detect-records plan checked equal to Model.forward + non_max_suppression_obb
  nms        the other half of the metric: rotated-NMS boxes/s and pair-IoUs/s, 1k-200k candidates, beside the reference's own
             CUDA kernel K1 on the same GPU and its CPU kernel
  extra.eager_torch_b200   the reference's GPU path restated with eager PyTorch/cuDNN fp16 + K1 on this GPU (the bar, not the target);
  train.eager_torch_b200   the same for the training step (autocast + GradScaler + SGD)
  cpu_baseline   the oracle port (fp32 torch restatement of the reference's eager CPU path + the reference's
             own CPU NMS kernel from oracle/_ref when present) on the host cores, bounded sample

  train      the train-step leg of the metric ("train+infer"): yolov5m-OBB, 8 tiles of 1024x1024 per GPU (configs[2]'s per-GPU
             share), one optimisation step = forward (batch-stat BN) + ComputeLoss + backward + [NCCL all-reduce of the
             flat gradient, N>1] + SGD-Nesterov + EMA; device-timed value, e2e with H2D of the uint8 batch + targets and
             D2H of the loss, achieved fraction of the tensor peak on the algorithmic 3x-forward FLOPs, and the CPU
             restatement of train.py --device cpu beside it

--dump-outputs DIR writes what the timed step returned for its last batch (detections.npy, detections_per_image.npy): the
inputs and weights are seeded, so two builds can be compared output for output.

--impl reference runs that CPU arm alone (rank 0 only under torchrun).  N>1 = independent replicas, one
b16 batch per GPU (the path shards by image batch, no data-path collective): weak scaling.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

MODEL, BATCH, IMG, NC = "s", 16, 1024, 15
TRAIN_MODEL, TRAIN_BATCH, TRAIN_TARGETS_PER_IMG = "m", 8, 24   # BASELINE configs[2]: yolov5m, b64 over 8 GPUs = 8 img / GPU
TRAIN_GFLOP_PER_IMG = {"n": 3 * 12.70, "s": 3 * 44.60, "m": 384.0, "l": 3 * 284.09, "x": 1592.3}  # SURVEY §8(d): fprop+dgrad+wgrad
CONF, IOU, MAX_DET = 0.25, 0.45, 1500
FWD_GFLOP_PER_IMG = 44.60  # BASELINE.md §2 (conv-only forward, yolov5s @1024, nc=15)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default=MODEL)
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the train-step leg (the `train` object of the JSON line)")
    ap.add_argument("--train-model", default=TRAIN_MODEL)
    ap.add_argument("--train-batch", type=int, default=TRAIN_BATCH)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--no-nms-sweep", action="store_true", help="skip the rotated-NMS boxes/s sweep (the `nms` object)")
    ap.add_argument("--no-eager", action="store_true", help="skip the eager-PyTorch-on-this-GPU bar (`extra.eager_torch_b200`)")
    ap.add_argument("--no-extra-models", action="store_true", help="skip the yolov5m b16 inference line (`extra.yolov5m_b16_inference`)")
    ap.add_argument("--no-parity-gate", action="store_true", help="skip the engine-vs-oracle check of the benchmarked plan")
    ap.add_argument("--slots", type=int, default=2, help="batches in flight per GPU, one stream + one plan each (DetectPipeline slots)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the detections of the last timed step to DIR/*.npy")
    return ap.parse_args()


def peaks():
    """MEASURED_PEAKS.json (driver-written): HBM copy bandwidth and cuBLAS bf16 throughput, burst and sustained.  The conv
    launches are timed one by one with CUDA events inside a region of a few tens of milliseconds at the full 1965 MHz clock
    (no power capping, see `clocks`), so the BURST figure is the denominator of roofline.frac; the sustained one is reported
    beside it (frac_sustained) and is the denominator of the multi-second train leg."""
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(tflops=float(d.get("bf16_tflops", 1590.0)), tflops_sustained=float(d.get("bf16_tflops_sustained", 1400.0)),
                    hbm=float(d.get("hbm_gbs", 6650.0)), src="measured (MEASURED_PEAKS.json: burst bf16 for frac, sustained for frac_sustained)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line), through NVML
    (nvidia_ml_py) from a thread every 20 ms; nvidia-smi's own polling loop takes longer to start than a short run lasts."""

    def __init__(self, index):
        self.rows, self.ok, self._stop = [], False, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            phys = index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                ids = [v for v in vis.split(",") if v.strip() != ""]
                if index < len(ids) and ids[index].strip().isdigit():
                    phys = int(ids[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception as e:  # pragma: no cover
            self.err = f"{type(e).__name__}: {e}"

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:
                try:
                    self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                      nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
                except Exception:
                    pass
            self._stop.wait(0.02)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"NVML unavailable ({getattr(self, 'err', '')})"], "samples": 0}
        self._stop.set()
        self.t.join(timeout=1)
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= int(r[1])
        names = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4),
                 ("hw_power_brake_slowdown", 0x80)]
        reasons = [n for n, b in names if bits & b]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm)}


def synth_batch(batch, seed):
    """uint8 DOTA-shaped synthetic tiles (tests/tilegen.py), on the host (pinned by the caller).  Four distinct
    seeded tiles are tiled to the batch: generation is host-side Python and not part of any timed region."""
    import torch
    from tests.tilegen import synth_tiles
    base = synth_tiles(min(batch, 4), IMG, seed)
    reps = (batch + base.shape[0] - 1) // base.shape[0]
    return base.repeat(reps, 1, 1, 1)[:batch].contiguous()


def build_model(size, device=None):
    """Seeded random-init yolov5-OBB (no checkpoints exist offline), calibrated identically on every arm so
    that the NMS stage sees a DOTA-like few thousand candidates per tile (tests/modelgen.py)."""
    from tests.modelgen import calibrated_bench_model
    m = calibrated_bench_model(size, nc=NC, seed=0, conf=CONF)
    return m.to(device) if device is not None else m


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's eager CPU path (+ the reference's own CPU NMS kernel)
# ------------------------------------------------------------------------------------------------
def cpu_arm(size, batch, steps, warmup, budget_s=25.0, use_ref_nms=False):
    import torch
    from oracle import model_ref
    from oracle.postprocess import non_max_suppression_obb as cpu_nms
    torch.set_grad_enabled(False)
    m = build_model(size)
    cores = torch.get_num_threads()
    b = 1  # bounded sample: one tile per step of the same workload
    x8 = synth_batch(b, 0)
    kind = "port"
    nms_note = "C++ oracle rotated NMS (1 thread)"
    if use_ref_nms:  # the reference's own nms_rotated_cpu kernel, compiled from /root/reference into oracle/_ref
        try:
            import oracle.postprocess as pp
            from oracle.build_ref import load_ref
            ref = load_ref()

            def ref_obb_nms(dets, scores, thr, mode=0):
                import numpy as np
                d, s_ = torch.from_numpy(np.ascontiguousarray(dets)), torch.from_numpy(np.ascontiguousarray(scores))
                ok = ~(d[:, 2:4].min(1)[0] < 0.001)  # nms_rotated_wrapper.py:32-39
                idx = torch.arange(d.shape[0])[ok]
                return idx[ref.nms_rotated_cpu(d[ok], s_[ok], float(thr))].numpy()

            pp._oracle_obb_nms = ref_obb_nms
            nms_note = "the reference's own nms_rotated_cpu extension (oracle/_ref, 1 thread)"
        except Exception as e:  # pragma: no cover
            nms_note += f" [oracle/_ref unavailable: {type(e).__name__}]"

    split = [0.0, 0.0, 0.0]  # the reference's three timers (val.py:183-207): pre-process, inference, NMS

    def step():
        t = [time.perf_counter()]
        x = x8.float() / 255                      # pre-process (val.py:187-188)
        t.append(time.perf_counter())
        pred, _ = model_ref.forward(m, x)         # inference
        t.append(time.perf_counter())
        r = cpu_nms(pred, CONF, IOU, multi_label=True, max_det=MAX_DET, nms_mode=0)  # NMS (CPU rule >=)
        t.append(time.perf_counter())
        for i in range(3):
            split[i] = t[i + 1] - t[i]            # the last step's split is reported
        return r

    t0 = time.perf_counter()
    step()                                   # warm-up (page-in, thread pools); a second one only if steps are short
    per = time.perf_counter() - t0
    if per < 15.0 and min(warmup, 2) > 1:
        t0 = time.perf_counter()
        step()
        per = time.perf_counter() - t0
    if per > 45.0:  # one step already exceeds the budget (the reference's quadratic single-thread CPU NMS): report it
        n, dt, cold = 1, per, " (the single, un-warmed step: one step exceeds the time budget)"
    else:
        n = max(1, min(steps, int(budget_s / max(per, 1e-3))))
        t0 = time.perf_counter()
        for _ in range(n):
            step()
        dt, cold = (time.perf_counter() - t0) / n, ""
    return dict(value=b / dt, unit="images/s", cores=cores, kind=kind, ms_per_step=dt * 1e3, steps=n,
                split_ms={"pre": split[0] * 1e3, "inference": split[1] * 1e3, "nms": split[2] * 1e3},
                value_without_nms=b / max(split[0] + split[1], 1e-9),
                sample=f"yolov5{size} fp32 eager-torch restatement of the reference CPU path + {nms_note}, "
                       f"{n} steps of 1 tile 1024x1024 (of the b{batch} workload){cold}, torch {torch.__version__}, {cores} threads")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_arm(args.model, args.batch, args.steps, args.warmup, budget_s=60.0, use_ref_nms=True)
    line = {
        "impl": "reference", "metric": "images/s", "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus,
        "steps": cb["steps"], "warmup": min(args.warmup, 2), "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "split_ms", "value_without_nms")},
        "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "split_ms shows where the CPU step goes: the reference's nms_rotated_cpu is single-threaded and quadratic in "
                "the candidate count (SURVEY 2.3), so this arm's images/s is dominated by NMS on the synthetic tiles' "
                "candidate load; value_without_nms is pre-process + inference alone",
    }
    if not args.no_train:  # the train-step leg of the metric on the same CPU arm (train.py --device cpu restated)
        tb = cpu_train_arm(args.train_model, budget_s=45.0)
        line["train"] = {"impl": "reference", "workload": f"yolov5{args.train_model}-OBB train step (forward, ComputeLoss, backward, "
                         "SGD-Nesterov) on the host cores, 1 tile 1024x1024 per step", "value": tb["value"], "unit": "images/s",
                         "ms_per_step": tb["ms_per_step"], "cpu_baseline": {k: tb[k] for k in ("value", "unit", "cores", "kind", "sample")}}
    print(json.dumps(line), flush=True)


def workload_config(args):
    return {"workload": f"yolov5{args.model}-OBB inference b{args.batch} 1024x1024 (BASELINE configs[1], val.py --task speed: "
                        f"pre-process + Model.forward + non_max_suppression_obb conf {CONF} iou {IOU} multi_label)",
            "batch_per_gpu": args.batch, "imgsz": IMG, "nc": NC, "parallelism": f"replicas x{args.gpus} (no collective)",
            "in_flight": f"our arm: {getattr(args, 'slots', 1)} batches per GPU, each on its own stream with its own plan (DetectPipeline "
                         "slots); ms_per_step = timed region / steps (throughput time, not the latency of one batch: see "
                         "single_stream).  The reference arm processes one batch at a time",
            "l2": "per-step working set (activations > 3 GB) exceeds the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------------
# train-step leg (BASELINE metric "train+infer"; configs[2] per-GPU share: yolov5m, 8 tiles of 1024x1024 per GPU)
# ------------------------------------------------------------------------------------------------
def train_inputs(batch, rank):
    import torch
    from tests.lossgen import synth_targets
    imgs = synth_batch(batch, seed=100 + rank)
    tg = torch.from_numpy(synth_targets(batch, TRAIN_TARGETS_PER_IMG * batch, IMG, nc=NC, seed=200 + rank))
    return imgs, tg


def cpu_train_arm(size, budget_s=30.0):
    """The reference's CPU training path (train.py --device cpu: eager fp32 torch forward, ComputeLoss, autograd
    backward, SGD-Nesterov step) restated by the oracle, 1 tile per step on the host cores — a bounded sample."""
    import torch
    from oracle import model_ref, loss_ref
    from tests.modelgen import build_mirror
    m = build_mirror(size, nc=NC, seed=0).train()
    det = m.model[-1]
    hyp = loss_ref.scaled_hyp(loss_ref.DEFAULT_HYP, det.nl, NC, IMG)
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.937, nesterov=True)
    imgs, tg = train_inputs(1, 0)
    cores = torch.get_num_threads()

    def step():
        with torch.enable_grad():
            pred = model_ref.forward_with_grad(m, imgs.float() / 255, training=True)
            loss, _ = loss_ref.compute_loss(pred, tg, det.anchors, det.stride, hyp, NC)
            loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    t0 = time.perf_counter()
    step()
    per = time.perf_counter() - t0
    n = max(1, min(5, int(budget_s / max(per, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    dt = (time.perf_counter() - t0) / n
    return dict(value=1.0 / dt, unit="images/s", cores=cores, kind="port", ms_per_step=dt * 1e3,
                sample=f"yolov5{size} fp32 eager-torch restatement of train.py --device cpu (forward, ComputeLoss, autograd "
                       f"backward, SGD-Nesterov), {n} steps of 1 tile 1024x1024, {cores} threads")


def eager_train_arm(size, dev, batch, steps=5, warmup=2):
    """The reference's own GPU training step restated with eager PyTorch on this GPU (train.py:318-336: amp.autocast forward +
    ComputeLoss, GradScaler backward, SGD-Nesterov step; cudnn.benchmark; no EMA update, which only flatters this bar): the bar
    the hand-written step has to beat on its own box, not the target."""
    import torch
    from oracle import model_ref, loss_ref
    from tests.modelgen import build_mirror
    torch.backends.cudnn.benchmark = True
    m = build_mirror(size, nc=NC, seed=0).train().to(dev)
    det = m.model[-1]
    hyp = loss_ref.scaled_hyp(loss_ref.DEFAULT_HYP, det.nl, NC, IMG)
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.937, nesterov=True)
    scaler = torch.amp.GradScaler("cuda")
    imgs, tg = train_inputs(batch, 0)
    imgs, tg = imgs.to(dev), tg.to(dev)
    anchors, stride = det.anchors.to(dev), det.stride.to(dev)

    def step():
        with torch.enable_grad():
            with torch.autocast("cuda", dtype=torch.float16):
                pred = model_ref.forward_with_grad(m, imgs.float() / 255, training=True)
            loss, _ = loss_ref.compute_loss([p.float() for p in pred], tg, anchors, stride, hyp, NC)
            scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        opt.zero_grad(set_to_none=True)
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(steps):
        last = step()
    torch.cuda.synchronize(dev)
    dt = (time.perf_counter() - t0) / steps
    return {"value": batch / dt, "unit": "images/s", "ms_per_step": dt * 1e3, "steps": steps, "loss_last": float(last),
            "what": f"eager PyTorch {torch.__version__} / cuDNN {torch.backends.cudnn.version()}: yolov5{size} train step on this GPU, "
                    f"{batch} tiles 1024x1024, torch.autocast(fp16) forward + fp32 ComputeLoss + GradScaler backward + SGD-Nesterov "
                    "(train.py:318-336), cudnn.benchmark=True, NCHW, no EMA; wall clock with a synchronize around the timed steps"}


def run_train_leg(args, dev, world, rank, dist, pk):
    """One optimisation step per 'step': forward, ComputeLoss, backward, [NCCL all-reduce of the flat gradient],
    SGD-Nesterov + EMA (yolov5_obb_b200.train_step.TrainStep = the loop body of train.py:296-342)."""
    import torch
    from tests.modelgen import build_mirror
    from yolov5_obb_b200.train_step import TrainStep
    size, TB = args.train_model, args.train_batch
    m = build_mirror(size, nc=NC, seed=0).train().to(dev)
    # configs[2] is a b64 job (8 tiles on each of 8 GPUs): nominal batch 64 -> the reference's `accumulate` is 1, i.e. every
    # step ends with the optimizer + EMA update (a b8 single-GPU job would only step the optimizer every 8th batch)
    # warm-up as train.py:305-316 (nw = max(round(3 epochs x batches), 1000) -> 1000 here): lr ramps from 0 (biases: from 0.1)
    ts = TrainStep(m, batch_size=64, imgsz=IMG, warmup_iters=1000)
    imgs_h, tg_h = train_inputs(TB, rank)
    imgs_h, tg_h = imgs_h.pin_memory(), tg_h.pin_memory()
    imgs_d, tg_d = imgs_h.to(dev), tg_h.to(dev)
    steps = max(1, args.train_steps)
    losses, first_loss = [], []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(n, e2e):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if e2e:  # the public loop over HOST batches (TrainStep.run: inputs from pinned host memory every step - the copy of
            # batch i+1 overlaps step i - and every step's loss read back to the host)
            for loss, items in ts.run((imgs_h, tg_h) for _ in range(n)):
                losses.append(float(loss))
        else:
            for _ in range(n):
                loss, items = ts.step(imgs_d, tg_d)
                if not first_loss:
                    first_loss.append(float(loss.cpu()))    # the very first optimisation step (warm-up region, untimed)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / n

    run(max(3, min(args.warmup, 5)), False)
    ms_dev = run(steps, False)
    ms_e2e = run(steps, True)
    value = world * TB / (ms_dev / 1e3)
    flops_img = TRAIN_GFLOP_PER_IMG[size] * 1e9
    out = {
        "workload": f"yolov5{size}-OBB train step, {TB} tiles 1024x1024 per GPU (BASELINE configs[2] per-GPU share): Model.forward "
                    f"(batch-stat BN) + ComputeLoss + backward + {'NCCL all-reduce of the flat gradient + ' if world > 1 else ''}"
                    "SGD-Nesterov + EMA",
        "value": value, "unit": "images/s", "ms_per_step": ms_dev, "steps": steps, "global_batch": TB * world,
        "e2e": {"value": world * TB / (ms_e2e / 1e3), "unit": "images/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(imgs_h.numel() + tg_h.numel() * 4), "d2h_bytes_per_step": 4},
        "tensor": {"algorithmic_TFLOP_per_step_per_gpu": flops_img * TB / 1e12,
                   "achieved_TFLOPs_per_gpu": flops_img * TB / (ms_dev / 1e3) / 1e12, "peak": pk["tflops_sustained"],
                   "peak_note": "sustained bf16 (the train leg runs for seconds)",
                   "frac": flops_img * TB / (ms_dev / 1e3) / 1e12 / pk["tflops_sustained"]},
        "loss_first_last": [first_loss[0], losses[-1]] if losses else None,
        "loss_note": "loss of the first optimisation step of the run and of the last timed one, same repeated batch; lr warm-up as "
                     "train.py:305-316 (SGD-Nesterov lr0 0.01, momentum 0.8 -> 0.937, bias lr from 0.1)",
        "targets_per_step": int(tg_h.shape[0]), "dtype": "bf16 activations/gradients, fp32 accumulation and master weights",
    }
    del ts, m
    torch.cuda.empty_cache()
    return out



# ------------------------------------------------------------------------------------------------
# rotated-NMS leg of the metric (BASELINE configs[3]): boxes/s and pair-IoUs/s, 1k-200k candidates, 15 classes, IoU 0.4
# ------------------------------------------------------------------------------------------------
NMS_SIZES = (1000, 2000, 5000, 10000, 20000, 50000, 100000, 200000)
NMS_THR, NMS_CLASSES = 0.4, 15


def nms_sweep(dev, seeds=(0, 1, 2), cpu_budget_s=25.0):
    """SURVEY §8(d): N candidates of 15 classes in one 1024^2 frame ("dense": realistic suppression) and in a 16384^2 frame
    ("sparse": nothing suppressed, worst case for the pair count), unique scores, thr 0.4.  Per (layout, N), median over
    the seeds:  ours through the reference-facing op nms_rotated(dets, scores, thr) on class-OFFSET boxes (the reference's
    own mode, general.py:849-851) and through the segmented op on raw boxes; the reference's CUDA kernel K1
    (nms_rotated_cuda.cu compiled from /root/reference into oracle/_ref) on the same GPU and inputs, keep lists compared;
    the reference's CPU kernel for the sizes a time budget allows."""
    import ctypes
    import numpy as np
    import torch
    from tests.boxgen import rboxes
    from yolov5_obb_b200 import _lib
    from yolov5_obb_b200.nms_rotated import nms_rotated, nms_rotated_batched
    L = _lib.lib()
    ref = None
    try:
        from oracle.build_ref import load_ref
        ref = load_ref()
    except Exception as e:  # pragma: no cover
        ref_err = f"{type(e).__name__}: {e}"

    def wall(fn):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize(dev)
        return (time.perf_counter() - t0) * 1e3, r

    rows, cpu_left = [], cpu_budget_s
    for layout, span in (("dense", 1024.0), ("sparse", 16384.0)):
        for n in NMS_SIZES:
            t_off, t_seg, t_ref, stages, kept, equal, seg_same = [], [], [], [], [], [], []
            pairs = 0
            for seed in seeds:
                d, sc, cls = rboxes(n, span, 1000 * seed + 17, n_classes=NMS_CLASSES, class_offset=False)
                cnt = np.bincount(cls, minlength=NMS_CLASSES).astype(np.int64)
                pairs = int((cnt * (cnt - 1) // 2).sum())
                d_off = d.copy()
                d_off[:, :2] += cls[:, None].astype(np.float32) * np.float32(4096)
                td, to, ts_, tc = (torch.from_numpy(a).to(dev) for a in (d, d_off, sc, cls.astype(np.int32)))
                nms_rotated(to, ts_, NMS_THR)                                   # warm-up (workspace growth, first launch)
                L.y5obb_nms_debug_stage_timing(1)
                ms, keep = wall(lambda: nms_rotated(to, ts_, NMS_THR))
                st4 = (ctypes.c_float * 4)()
                if L.y5obb_nms_debug_stage_ms(st4) == 0:
                    stages.append([float(v) for v in st4])
                L.y5obb_nms_debug_stage_timing(0)
                t_off.append(ms)
                kept.append(int(keep.numel()))
                nms_rotated_batched(td, ts_, tc, NMS_CLASSES, NMS_THR)
                ms2, (k2, c2, o2) = wall(lambda: nms_rotated_batched(td, ts_, tc, NMS_CLASSES, NMS_THR))
                t_seg.append(ms2)
                # the segmented result, merged back into one score-ordered list, is the offset-mode keep set
                c2h, o2h = c2.tolist(), o2.tolist()
                seg_keep = torch.cat([k2[o2h[g]:o2h[g] + c2h[g]] for g in range(NMS_CLASSES)])
                seg_keep = seg_keep[torch.argsort(ts_[seg_keep], descending=True)]
                # informational: raw-coordinate boxes are MORE exact than the reference's offset ones (fp32 centres lose up
                # to 0.004 px at 57 344), and in the sparse frame (16 384 > 4 096) offset classes overlap - so the two modes
                # answer slightly different questions at large N
                seg_same.append(bool(torch.equal(seg_keep, keep)))
                if ref is not None:
                    ref.nms_rotated_cuda(to[: min(n, 2000)], ts_[: min(n, 2000)], NMS_THR)
                    ms3, kref = wall(lambda: ref.nms_rotated_cuda(to, ts_, NMS_THR))
                    t_ref.append(ms3)
                    equal.append(bool(torch.equal(kref, keep)))
            med = lambda v: float(np.median(v)) if v else None
            stg = [float(np.median([s_[i] for s_ in stages])) for i in range(4)] if stages else None
            row = {"layout": layout, "n": n, "pairs_algorithmic": pairs, "kept": int(np.median(kept)),
                   "ms": med(t_off), "boxes_per_s": n / (med(t_off) / 1e3), "pair_ious_per_s": pairs / (med(t_off) / 1e3),
                   "GBps_on_24B_per_box": 24.0 * n / (med(t_off) / 1e3) / 1e9,
                   "stage_ms": dict(zip(("sort", "plan_prep", "k_tiles", "k_reduce"), stg)) if stg else None,
                   "segmented_ms": med(t_seg), "segmented_boxes_per_s": n / (med(t_seg) / 1e3),
                   "reference_k1_ms": med(t_ref), "speedup_vs_reference_k1": (med(t_ref) / med(t_off)) if t_ref else None,
                   "keep_list_equals_reference_k1": all(equal) if equal else None,
                   "segmented_equals_offset_mode": all(seg_same)}
            # the reference's CPU kernel (single thread, quadratic): only while the time budget lasts
            if ref is not None and n <= 10000 and cpu_left > 0:
                est = 1.7e-6 * (n * n / 2 if layout == "sparse" else n * max(row["kept"], 1))
                if est < cpu_left:
                    d, sc, cls = rboxes(n, span, 17, n_classes=NMS_CLASSES, class_offset=True)
                    t0 = time.perf_counter()
                    kc = ref.nms_rotated_cpu(torch.from_numpy(d), torch.from_numpy(sc), NMS_THR)
                    dt = time.perf_counter() - t0
                    cpu_left -= dt
                    row["reference_cpu_ms"] = dt * 1e3
                    row["reference_cpu_kept"] = int(kc.numel())
            rows.append(row)
    big = [r for r in rows if r["n"] == 200000 and r["layout"] == "dense"][0]
    return {"workload": "rotated-NMS + rotated-IoU sweep (BASELINE configs[3]): N candidate rboxes, 15 classes, IoU 0.4, unique "
                        "scores, seeds 0-2 (median); dense = one 1024^2 frame, sparse = 16384^2 frame; class-offset boxes "
                        "through nms_rotated (the reference's mode), raw boxes through the segmented op",
            "metric": "rotated-NMS boxes/s", "value": big["boxes_per_s"], "unit": "boxes/s", "at": "dense, N = 200000",
            "timing": "wall clock around the op with a device synchronize on both sides (the op returns a variable-length "
                      "tensor: one 8-byte host read inside); stage_ms from CUDA events inside the op",
            "reference_k1": "utils/nms_rotated/src/nms_rotated_cuda.cu compiled unmodified (oracle/_ref), same GPU, same "
                            "inputs" if ref is not None else f"unavailable ({ref_err})",
            "all_keep_lists_equal_reference_k1": all(r["keep_list_equals_reference_k1"] for r in rows) if ref is not None else None,
            "rows": rows}


# ------------------------------------------------------------------------------------------------
# parity gate of the benchmarked plan, and the eager-PyTorch bar on the same GPU
# ------------------------------------------------------------------------------------------------
def parity_gate(model_cpu, x_u8_dev, pred, sample=(0, -1)):
    """The exact plan the timing runs (b16 x 1024^2: its own tile geometry, stem padding, 16 images per grid) against the
    fp32 oracle (oracle/model_ref on the host, test infrastructure) on sampled images of the batch.
    The calibrated benchmark model is 'alive' (BatchNorm statistics of a real tile, Detect rows rescaled ~50x): it amplifies
    storage rounding layer by layer, so the yardstick is MEASURED - the oracle itself with bf16 storage emulated
    (emulate_bf16=True) against the fp32 oracle.  Per Detect level the device's relative L2 distance to fp32 must stay below
    2x that floor + 3e-3, and its `obj > conf` candidate mask must agree with fp32 no worse than the emulation's does - 0.1.
    (Layer-by-layer, chaos-free evidence for this plan: tests/test_engine_gpu.py::test_bench_plan_teacher_forced.)"""
    import torch
    from oracle import model_ref
    B = x_u8_dev.shape[0]
    idx = sorted({i % B for i in sample})
    x = x_u8_dev[idx].cpu().float() / 255
    want, _ = model_ref.forward(model_cpu, x)
    emu, _ = model_ref.forward(model_cpu, x, emulate_bf16=True)
    got = pred[idx].float().cpu()
    det = model_cpu.model[-1]
    H = x.shape[2]
    rows = [det.na * (H // int(s)) ** 2 for s in det.stride.tolist()]
    out, o, ok = {"images": idx, "rule": "rel_l2 < 2 * bf16_floor + 3e-3 per level; mask IoU >= floor's - 0.1", "levels": []}, 0, True
    for l, r in enumerate(rows):
        g, w, e = got[:, o:o + r], want[:, o:o + r], emu[:, o:o + r]
        rel, floor = ((g - w).norm() / w.norm()).item(), ((e - w).norm() / w.norm()).item()
        out["levels"].append({"stride": int(det.stride[l]), "rel_l2": rel, "bf16_floor": floor})
        ok = ok and rel < 2.0 * floor + 3e-3
        o += r
    cw = want[..., 4] > CONF

    def iou(t):
        c = t[..., 4] > CONF
        return (c & cw).sum().item() / max((c | cw).sum().item(), 1)

    out["obj_candidate_mask_iou"], out["obj_candidate_mask_iou_bf16_floor"] = iou(got), iou(emu)
    out["candidates_engine_vs_oracle"] = [int((got[..., 4] > CONF).sum()), int(cw.sum())]
    out["ok"] = bool(ok and out["obj_candidate_mask_iou"] >= out["obj_candidate_mask_iou_bf16_floor"] - 0.1)
    if not out["ok"]:
        raise RuntimeError(f"parity gate failed: the benchmarked plan disagrees with the fp32 oracle: {out}")
    return out


def eager_torch_arm(model_cpu, x_u8_dev, steps, warmup):
    """The reference's own GPU path restated (oracle/eager_ref.py: fused fp16 model through cuDNN with cudnn.benchmark, Detect,
    the per-image non_max_suppression_obb loop over the reference's CUDA kernel K1) on this GPU, same tiles, same step
    definition (pre-process + inference + NMS).  The bar SURVEY §2.3 L1 names - not the target."""
    import torch
    from oracle.eager_ref import EagerFusedModel
    from oracle.postprocess import non_max_suppression_obb as loop_nms, ref_obb_nms_cuda
    from oracle.build_ref import load_ref
    dev = x_u8_dev.device
    ref = load_ref()
    nms_fn = ref_obb_nms_cuda(ref)
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        em = EagerFusedModel(model_cpu, dev, half=True)

        def step():
            x = x_u8_dev.half() / 255                                   # val.py:187-188
            pred = em.forward(x)                                        # val.py:191
            return loop_nms(pred, CONF, IOU, multi_label=True, max_det=MAX_DET, nms_fn=nms_fn), pred

        for _ in range(max(warmup, 3)):
            step()
        torch.cuda.synchronize(dev)
        t_inf = t_nms = 0.0
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        t0 = time.perf_counter()
        n_det = 0
        for _ in range(steps):
            e[0].record()
            pred = em.forward(x_u8_dev.half() / 255)
            e[1].record()
            dets = loop_nms(pred, CONF, IOU, multi_label=True, max_det=MAX_DET, nms_fn=nms_fn)
            e[2].record()
            torch.cuda.synchronize(dev)
            t_inf += e[0].elapsed_time(e[1])
            t_nms += e[1].elapsed_time(e[2])
            n_det = sum(d.shape[0] for d in dets)
        dt = (time.perf_counter() - t0) / steps
    finally:
        torch.backends.cudnn.benchmark = old
    B = x_u8_dev.shape[0]
    return {"value": B / dt, "unit": "images/s", "ms_per_step": dt * 1e3, "inference_ms": t_inf / steps, "nms_ms": t_nms / steps,
            "steps": steps, "detections_per_image": n_det / B, "dtype": "fp16 (model.half(), val.py:128,142)",
            "what": "eager PyTorch " + torch.__version__ + " / cuDNN " + str(torch.backends.cudnn.version()) +
                    ", cudnn.benchmark=True, NCHW, BatchNorm folded (Conv.forward_fuse); non_max_suppression_obb per-image loop "
                    "with the reference's nms_rotated_cuda (K1 + N^2/8-byte mask D2H + host scan); same GPU, tiles and step "
                    "definition; timed by wall clock with a synchronize per step (its NMS synchronises anyway)"}

# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, packed, counts, batch):
    """What a caller of the timed step receives for one batch: detections.npy = the rows (cx, cy, l, s, theta, conf, cls) of
    every image, image after image; detections_per_image.npy = how many rows belong to each image."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    n = counts[:batch].cpu().numpy()
    rows = packed.cpu().numpy()
    np.save(out / "detections.npy", np.concatenate([rows[b, :k] for b, k in enumerate(n)]).astype(np.float32))
    np.save(out / "detections_per_image.npy", n.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from yolov5_obb_b200 import _lib
    from yolov5_obb_b200.general import non_max_suppression_obb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly ONE JSON line: until it is printed, file descriptor 1 points at stderr, so that whatever native
    # libraries write to stdout (NCCL's "NCCL version ..." banner at communicator creation) cannot end up in front of it
    sys.stdout.flush()
    _saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    import copy
    model_cpu = build_model(args.model)
    model = copy.deepcopy(model_cpu).to(dev)
    # every replica processes the same seeded tile set: the NMS stage is data dependent (candidates per tile), and with four
    # distinct tiles per batch a per-rank seed made rank 1's step 12 % longer than rank 0's - sample noise, not scaling
    x_host = synth_batch(B, seed=0).pin_memory()
    x_dev = x_host.to(dev)
    pred0, _ = model(x_dev)                 # Model.forward: the [B, A, no] tensor of the reference API
    pred0 = pred0.clone()
    rec0 = model.detect_records(x_dev)      # the timed plan: same network, Detect rows as compact records
    eng = model._engines[("records", tuple(x_dev.shape), dev.index)]
    # the number below is only worth reporting if THIS plan computes the right thing: compare it with the oracle first
    parity = None
    if not args.no_parity_gate and rank == 0:
        parity = parity_gate(model_cpu, x_dev, pred0)
        # ... and the fused plan (records) must give the detections of Model.forward + non_max_suppression_obb: box / obj /
        # class columns bit-equal, theta index = the tensor's argmax up to near-ties of its tanh.approx sigmoid
        # (tests/recordcheck.py); with those rows patched the two detection lists must be IDENTICAL
        from tests.recordcheck import check_records
        pred_p, near_ties = check_records(pred0, rec0.data, NC)
        d_full = non_max_suppression_obb(pred_p, CONF, IOU, multi_label=True, max_det=MAX_DET)
        d_rec = non_max_suppression_obb(rec0, CONF, IOU, multi_label=True, max_det=MAX_DET)
        parity["fused_records_equal_model_forward_plus_nms"] = all(torch.equal(a, b) for a, b in zip(d_full, d_rec))
        parity["theta_near_tie_rows"] = near_ties
        parity["rows"] = int(pred0.shape[0] * pred0.shape[1])
        if not parity["fused_records_equal_model_forward_plus_nms"]:
            raise RuntimeError("the fused Detect-records plan and Model.forward + non_max_suppression_obb disagree")
    conv_flops = [c.info()["flops"] for c in eng.convs]
    n_conv = len(eng.convs)
    st = _lib.stream_ptr(dev)
    L = _lib.lib()
    conv_handles = {c._h.value for c in eng.convs}

    from yolov5_obb_b200.pipeline import DetectPipeline
    pipe = DetectPipeline(model, CONF, IOU, MAX_DET, multi_label=True, device=dev, slots=args.slots)
    last = {}

    def step_device():
        """pre-process + forward + NMS of one resident batch through the public pipeline object (DetectPipeline.submit =
        Model.detect_records + non_max_suppression_obb on the next slot's stream); the result stays on the device as the packed
        ([B, max_det, 7], rows per image) pair, so consecutive steps queue back to back (no host read per step) and
        `slots` batches are in flight at once."""
        slot = pipe._next
        last[slot] = pipe.submit(x_dev)
        return last[slot]

    def step_single():
        """the same step with ONE batch in flight, on the current stream (what round 1 and the first half of round 2 timed)"""
        rec = model.detect_records(x_dev)   # Model.forward with the Detect rows written as compact records (fused post-process)
        return non_max_suppression_obb(rec, CONF, IOU, multi_label=True, max_det=MAX_DET, return_packed="async")

    def run_e2e(steps):
        """`steps` batches from pinned host memory through the public pipeline API: H2D of batch i+1 overlaps the
        compute of batch i; the D2H of every batch's detections is inside the loop."""
        n = 0
        for dets in pipe(x_host for _ in range(steps)):
            n += sum(d.shape[0] for d in dets)
        return n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, pipeline=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if pipeline is not None:
            pipeline.fork()     # the slot streams start after e0 ...
        r = None
        for _ in range(steps):
            r = fn()
        if pipeline is not None:
            pipeline.join()     # ... and e1 is recorded after every slot stream has finished its last batch
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, r

    # nvidia-smi takes ~100 ms to start: launch it before the warm-up so that it is sampling (every 100 ms) while
    # the timed region runs; warm-up and timed steps are the same load
    sampler = ClockSampler(local) if rank == 0 else None
    # one blocking call first: it sizes the candidate capacity for this workload (sticky hint, general._CAP_HINT)
    non_max_suppression_obb(model.detect_records(x_dev), CONF, IOU, multi_label=True, max_det=MAX_DET)
    n_warm = max(args.warmup, 3) * pipe.slots    # every slot captures its graphs on its third call
    pipe.fork()
    for _ in range(n_warm):
        dets = step_device()
    pipe.join()
    ms_total, dets = timed(step_device, args.steps, pipe)
    clocks = sampler.stop() if sampler else None
    for dd in last.values():                     # the last batch of every slot
        rows = dd[1].tolist()
        if rows[B] > dd[2] or min(rows) < 0:
            raise RuntimeError("NMS candidate capacity exceeded in the timed steps: the measurement would be invalid")
    det_per_img = float(sum(rows[:B])) / B
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dets[0], dets[1], B)   # the last timed step's batch
    ms_step = ms_total / args.steps
    # the same step with one batch in flight (for the comparison with earlier rounds, and as the step the per-launch
    # roofline shares refer to)
    for _ in range(3):
        step_single()
    ms_single, _ = timed(step_single, min(args.steps, 20))
    ms_single /= min(args.steps, 20)
    # where the step goes (a few extra steps with events between the two public calls; not part of the timed region)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    bd = [0.0, 0.0]
    host_s = 0.0
    torch.cuda.synchronize()
    for _ in range(5):
        t0 = time.perf_counter()
        ev[0].record()
        rec = model.detect_records(x_dev)
        ev[1].record()
        non_max_suppression_obb(rec, CONF, IOU, multi_label=True, max_det=MAX_DET, return_packed="async")
        ev[2].record()
        host_s += time.perf_counter() - t0
        torch.cuda.synchronize()
        bd[0] += ev[0].elapsed_time(ev[1])
        bd[1] += ev[1].elapsed_time(ev[2])
    breakdown = {"forward_ms": bd[0] / 5, "post_process_ms": bd[1] / 5, "host_enqueue_ms": host_s / 5 * 1e3,
                 "note": "one batch in flight, events between the two public calls"}
    value = world * B / (ms_step / 1e3)

    run_e2e(3)
    pipe.h2d_bytes = pipe.d2h_bytes = 0
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_e2e(args.steps)
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_e2e = float(tt.item())
    d2h = pipe.d2h_bytes // args.steps
    e2e_value = world * B / (ms_e2e / args.steps / 1e3)

    # roofline leg: CUDA events around every conv launch of the timed steps (same stream, after warm-up)
    pk = peaks()
    steps_r = min(args.steps, 5)
    evs = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_conv)]
           for _ in range(steps_r)]
    x_f = x_dev
    torch.cuda.synchronize()
    for s in range(steps_r):
        _lib.check(L.y5obb_stem_s2d_u8(x_f.data_ptr(), eng.x_s2d.data_ptr(), B, IMG, IMG, 1, st), "s2d")
        ci = 0
        for op in eng.ops:
            h = op.__defaults__[0] if op.__defaults__ else None
            is_conv = isinstance(h, type(eng.convs[0]._h)) and h.value in conv_handles
            if is_conv:
                evs[s][ci][0].record()
            op(st)
            if is_conv:
                evs[s][ci][1].record()
                ci += 1
    torch.cuda.synchronize()
    conv_ms = [sum(evs[s][i][0].elapsed_time(evs[s][i][1]) for s in range(steps_r)) / steps_r for i in range(n_conv)]
    tot_conv_ms = sum(conv_ms)
    ach_tflops = sum(conv_flops) / (tot_conv_ms / 1e3) / 1e12
    traffic, traffic_src = None, None
    tp = ROOT / "profiles" / "r2_conv_traffic.json"   # dram__bytes_read+write per launch from one `ncu --set full` capture
    if tp.exists() and args.model == MODEL and B == BATCH:
        tj = json.loads(tp.read_text())
        traffic, traffic_src = tj["dram_bytes_per_launch_mean"], tj["source"]
    roof = {"bound": "tensor", "kernel": "conv_tc_kernel", "achieved": ach_tflops, "peak": pk["tflops"],
            "unit": "TFLOP/s", "frac": ach_tflops / pk["tflops"], "frac_sustained": ach_tflops / pk["tflops_sustained"],
            "peak_sustained": pk["tflops_sustained"], "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": eng.hbm_bytes / n_conv, "peak_source": pk["src"],
            "launches_per_step": n_conv, "flops_per_launch": sum(conv_flops) / n_conv,
            "mean_launch_us": tot_conv_ms / n_conv * 1e3, "conv_share_of_step": tot_conv_ms / ms_single,
            "conv_share_note": "sum of the conv launches / the single-stream step (launches timed one batch in flight)",
            "hbm_view": {"algorithmic_GB_per_step": eng.hbm_bytes / 1e9,
                         "achieved_GBps": eng.hbm_bytes / (tot_conv_ms / 1e3) / 1e9, "peak_GBps": pk["hbm"]}}

    # the other half of the metric (rotated-NMS boxes/s) and the eager-PyTorch bar: single-GPU runs only, rank 0
    nms, eager = None, None
    if world == 1 and not args.no_nms_sweep:
        nms = nms_sweep(dev)
    if world == 1 and not args.no_eager:
        try:
            eager = eager_torch_arm(model_cpu, x_dev, steps=min(args.steps, 10), warmup=3)
        except Exception as e:  # the bar needs oracle/_ref (the reference's K1): report its absence, never fake it
            eager = {"unavailable": f"{type(e).__name__}: {e}"}

    # north_star's model at the same inference workload (yolov5m b16): reported beside the configs[1] line, same step definition
    extra_m = None
    if world == 1 and args.model == MODEL and not args.no_extra_models:
        try:
            mm = copy.deepcopy(build_model("m")).to(dev)
            non_max_suppression_obb(mm.detect_records(x_dev), CONF, IOU, multi_label=True, max_det=MAX_DET)   # capacity hint

            pipe_m = DetectPipeline(mm, CONF, IOU, MAX_DET, multi_label=True, device=dev, slots=args.slots)

            def step_m():
                return pipe_m.submit(x_dev)
            pipe_m.fork()
            for _ in range(4 * pipe_m.slots):
                dm = step_m()
            pipe_m.join()
            ms_m, dm = timed(step_m, min(args.steps, 20), pipe_m)
            eng_m = mm._engines[("records", tuple(x_dev.shape), dev.index)]
            ms_m /= min(args.steps, 20)
            extra_m = {"workload": "yolov5m-OBB inference b16 1024x1024 (north_star's model; same step: pre-process + Model.forward + NMS)",
                       "value": B / (ms_m / 1e3), "unit": "images/s", "ms_per_step": ms_m,
                       "conv_algorithmic_TFLOP_per_step": eng_m.flops / 1e12,
                       "whole_step_TFLOPs": eng_m.flops / (ms_m / 1e3) / 1e12, "detections_per_image": float(sum(dm[1].tolist()[:B])) / B}
            del mm, eng_m, pipe_m
            torch.cuda.empty_cache()
        except Exception as e:  # pragma: no cover
            extra_m = {"unavailable": f"{type(e).__name__}: {e}"}

    # train-step leg (all ranks take part: the gradient all-reduce is the path's one exchange step)
    train = None
    pipe_slots = pipe.slots
    if not args.no_train:
        del pipe
        last.clear()
        model._engines.clear()
        torch.cuda.empty_cache()
        train = run_train_leg(args, dev, world, rank, dist, pk)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": "images/s", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic (seeded DOTA-shaped uint8 tiles, seeded random-init weights with calibrated BN/Detect statistics)",
        "config": workload_config(args),
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": int(x_host.numel()),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e / args.steps,
                "api": "yolov5_obb_b200.pipeline.DetectPipeline (pinned host uint8 in, per-image host detections out; "
                       f"{pipe_slots} batches in flight on their own streams, H2D of batch i+1 on a copy stream, host read-out of "
                       "batch i-slots while the later ones compute)"},
        "single_stream": {"ms_per_step": ms_single, "value": world * B / (ms_single / 1e3), "unit": "images/s",
                          "what": "the same device-resident step with ONE batch in flight on one stream"},
        "gpu_launches": (1 + len(eng.ops) + 25) * args.steps,  # layout pass + conv / pool launches + the post-process kernels (profiles/r2_launches_infer.csv: 79 per step)
        "detections_per_image": det_per_img, "step_breakdown": breakdown,
        "clocks": clocks, "roofline": roof,
    }
    if parity is not None:
        line["parity"] = parity
    if nms is not None:
        line["nms"] = nms
    if eager is not None or extra_m is not None:
        line["extra"] = {}
        if eager is not None:
            line["extra"]["eager_torch_b200"] = eager
        if extra_m is not None:
            line["extra"]["yolov5m_b16_inference"] = extra_m
    if not args.no_cpu_baseline and world == 1:
        cb = cpu_arm(args.model, B, args.steps, args.warmup)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "split_ms", "value_without_nms")}
    if train is not None:
        line["train"] = train
        if world == 1 and not args.no_eager:
            try:
                train["eager_torch_b200"] = eager_train_arm(args.train_model, dev, train.get("global_batch", 8))
            except Exception as e:  # pragma: no cover
                train["eager_torch_b200"] = {"unavailable": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
        if not args.no_cpu_baseline and world == 1:
            tb = cpu_train_arm(args.train_model)
            train["cpu_baseline"] = {k: tb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(_saved_stdout, 1)
    os.close(_saved_stdout)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
