"""Stand-alone timing of the wgrad kernel on training-sized layers (debug aid)."""
import sys, torch
from yolov5_obb_b200.train_ops import Wgrad
DEV = "cuda:0"
CASES = [(8, 48, 48, 256, 256, 3, 1), (8, 96, 96, 128, 128, 3, 1), (8, 48, 96, 512, 512, 3, 2), (8, 192, 192, 64, 64, 3, 1),
         (8, 384, 768, 64, 64, 3, 2), (8, 768, 768, 32, 32, 1, 1), (8, 96, 48, 256, 256, 1, 1), (8, 192, 96, 128, 128, 1, 1)]
sel = [int(v) for v in sys.argv[1:]] or range(len(CASES))
for (B, Cin, Cout, H, W, k, s) in [CASES[i] for i in sel]:
    p = k // 2
    Ho, Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    x = torch.randn(B, H, W, Cin, device=DEV).bfloat16()
    dz = torch.randn(B, Ho, Wo, Cout, device=DEV).bfloat16()
    dw = torch.zeros((Cout, Cin, k, k), dtype=torch.float32, device=DEV)
    wg = Wgrad(dz.data_ptr(), Cout, x.data_ptr(), Cin, dw, B, Cout, Ho, Wo, Cin, H, W, k, s, p, keep=(x, dz), param_layout=True)
    for _ in range(3):
        wg.run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        wg.run()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 100
    fl = 2.0 * B * Ho * Wo * Cout * Cin * k * k
    print(f"{Cin}->{Cout} k{k} s{s} {Ho}x{Wo}: {us:7.1f} us  {fl / us / 1e6:6.1f} TF/s", flush=True)
