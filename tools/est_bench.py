"""Times the estimator stages (CUDA events, device-resident) on N synthetic 12 MP frames: maps (box filters) and fit
(radix select + score3 + masked sums), self and collab."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yond_public_b200 as Y  # noqa: E402
from yond_public_b200 import nlf  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 8
flat = float(sys.argv[2]) if len(sys.argv) > 2 else 0.0  # fraction of the frame height that is saturated (constant 1.0): lap == 0 there
H, W = 3024, 4032
g = torch.Generator(device="cuda").manual_seed(0)
x = torch.rand((n, 1, H, W), device="cuda", generator=g) * 0.5
if flat > 0:
    x[:, :, :int(H * flat)] = 1.0
y = (x.reshape(n, H, W) * 0.9 + 0.01).contiguous()
est = nlf._estimator()


def timeit(fn, reps=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


px = n * H * W
t_self = timeit(lambda: est.estimate_dev(x, None, 29))
t_collab = timeit(lambda: est.estimate_dev(x, y, 29, y_mosaic=True))
print(f"frames {n} (flat {flat}): self estimate {t_self:.3f} ms ({px * 16 / t_self / 1e6:.0f} GB/s of 16 B/px maps only), collab {t_collab:.3f} ms")
