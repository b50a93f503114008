"""Times single conv layers (tcgen05 kernel): the mean conv_tc_kernel duration over N yond_conv2d calls, read from
torch.profiler's CUDA activities.  `python tools/conv_microbench.py [N]`; MB_B sets the batch, MB_CASES=i,j selects cases."""
import ctypes as C
import os
import sys

import numpy as np
import torch
from torch.autograd import DeviceType
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from yond_public_b200 import _lib  # noqa: E402

lib = _lib.load()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 20
B = int(os.environ.get("MB_B", "256"))
CASES = [  # mode, H, W, cin0, cin1, cout, act, res, dual
    (0, 128, 128, 32, 0, 32, 2, False, False), (0, 128, 128, 32, 0, 32, 0, True, False), (2, 128, 128, 32, 0, 64, 0, False, True),
    (0, 64, 64, 64, 0, 64, 2, False, False), (1, 128, 128, 32, 32, 32, 0, False, True), (3, 64, 64, 64, 0, 32, 0, False, False),
    (0, 32, 32, 128, 0, 128, 2, False, False), (0, 16, 16, 256, 0, 256, 2, False, False), (0, 8, 8, 512, 0, 512, 2, False, False),
]
sel = os.environ.get("MB_CASES")
for i, (mode, H, W, c0, c1, co, act, res, dual) in enumerate(CASES):
    if sel and str(i) not in sel.split(","):
        continue
    cin = c0 + c1
    dev = "cuda"
    s0 = torch.randn(B, H, W, c0, device=dev).to(torch.bfloat16)
    s1 = torch.randn(B, H, W, c1, device=dev).to(torch.bfloat16) if c1 else None
    if mode == 3:
        w = np.random.randn(cin, co, 2, 2).astype(np.float32) * 0.05
        Ho, Wo = 2 * H, 2 * W
    else:
        k = 1 if mode == 1 else 3
        w = np.random.randn(co, cin, k, k).astype(np.float32) * 0.05
        Ho, Wo = (H // 2, W // 2) if mode == 2 else (H, W)
    out0 = torch.empty(B, Ho, Wo, co, device=dev, dtype=torch.bfloat16)
    out1 = torch.empty_like(out0) if dual else None
    r = torch.randn(B, Ho, Wo, co, device=dev).to(torch.bfloat16) if res else None
    bias = torch.zeros(co, device=dev)
    sc = torch.ones(B, co, device=dev) if act == 2 else None
    p = _lib.ptr

    def call():
        rc = lib.yond_conv2d(mode, 0, B, H, W, c0, c1, p(s0), p(s1), co, w.ctypes.data_as(C.c_void_p), p(bias), p(sc), p(sc), act,
                             0.2, p(r), p(out0), p(out1), _lib.stream_ptr())
        assert rc == 0, lib.yond_last_error()

    call()  # warm-up: module load, tensor-map encoder
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(N):
            call()
    us = [e.time_range.elapsed_us() for e in prof.events() if e.device_type == DeviceType.CUDA and "conv_tc_kernel" in e.name]
    assert len(us) == N, f"expected {N} conv_tc_kernel launches, profiler saw {len(us)}"
    print(f"case {i}: mode={mode} B={B} HxW={H}x{W} Cin={c0}+{c1} Cout={co}: {sum(us) / N:.2f} us/launch")
