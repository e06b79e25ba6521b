"""GPU probe: pinned D2H / H2D bandwidth and the host link topology."""
import os
import torch
for mb in (28.7, 256.0):
    n = int(mb * 1e6)
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    for name, a, b in (("D2H", h, d), ("H2D", d, h)):
        for _ in range(2):
            a.copy_(b, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            a.copy_(b, non_blocking=True)
        e1.record(); torch.cuda.synchronize()
        print("%s %.1f MB pinned: %.1f GB/s" % (name, mb, n * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9))
os.system("nvidia-smi topo -m 2>&1 | head -20")
