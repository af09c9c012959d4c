"""CPU checks of bench.py's contract pieces that need no GPU: argument defaults, the workload description, the roofline
denominators, the clock sampler's behaviour without NVML, the synthetic inputs, and the files --dump-outputs writes."""
import json
import sys

import numpy as np
import torch

import bench


def test_defaults_and_workload_description(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    a = bench.parse()
    assert (a.gpus, a.impl, a.model, a.batch) == (1, "ours", "s", 16) and a.warmup >= 3 and a.steps >= 1
    assert (a.train_model, a.train_batch) == ("m", 8)           # BASELINE configs[2]: yolov5m, 8 tiles per GPU
    cfg = bench.workload_config(a)
    assert "yolov5s-OBB inference b16 1024x1024" in cfg["workload"] and cfg["imgsz"] == 1024 and "l2" in cfg
    assert a.slots == 2 and "2 batches per GPU" in cfg["in_flight"]   # the pipelined step is declared in the config
    json.dumps(cfg)


def test_peaks_and_clock_sampler_degrade_gracefully():
    pk = bench.peaks()
    assert pk["tflops"] > 100 and pk["hbm"] > 1000 and isinstance(pk["src"], str)
    c = bench.ClockSampler(0).stop()                            # no GPU here: a reasoned null, never an exception
    assert set(c) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    json.dumps(c)


def test_synthetic_inputs_are_seeded_and_shaped():
    x = bench.synth_batch(3, seed=1)
    assert x.dtype == torch.uint8 and tuple(x.shape) == (3, 3, 1024, 1024)
    assert torch.equal(x, bench.synth_batch(3, seed=1)) and not torch.equal(x[0], bench.synth_batch(3, seed=2)[0])
    imgs, tg = bench.train_inputs(2, rank=0)
    assert imgs.dtype == torch.uint8 and tuple(imgs.shape) == (2, 3, 1024, 1024)
    assert tg.shape == (2 * bench.TRAIN_TARGETS_PER_IMG, 187) and tg[:, 0].max() < 2 and tg[:, 1].max() < bench.NC
    assert abs(float(tg[0, 7:].max()) - 1.0) < 1e-6             # a CSL row peaks at 1


def test_dump_outputs_writes_the_detections_per_image(monkeypatch, tmp_path):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "7", "--dump-outputs", str(tmp_path / "out")])
    a = bench.parse()
    assert a.steps == 7 and a.dump_outputs == str(tmp_path / "out")
    packed = torch.arange(2 * 4 * 7, dtype=torch.float32).reshape(2, 4, 7)    # [B, max_det, 7], rows past the count unused
    counts = torch.tensor([3, 1, 99])                                          # per image, then the candidate total
    bench.dump_outputs(a.dump_outputs, packed, counts, 2)
    det = np.load(tmp_path / "out" / "detections.npy")
    per = np.load(tmp_path / "out" / "detections_per_image.npy")
    assert det.dtype == np.float32 and per.dtype == np.float64
    assert per.tolist() == [3.0, 1.0]
    assert np.array_equal(det, np.concatenate([packed[0, :3].numpy(), packed[1, :1].numpy()]))
