import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from noisynet_b200 import _lib, ops
from noisynet_b200._lib import NOISE_EXTERNAL
B = 512
dev = torch.device("cuda:0")
s_a = 5.0 / 15.0
x = torch.randint(0, 16, (B, 65, 14, 14), device=dev).float() * s_a
w_raw = torch.randn(120, 65, 5, 5, device=dev) * 0.1
wq = ops.quantize_fwd(w_raw, 4, -1.0, 1.0, 0.0)
scale = ops.tensor_stats(x)[0:1]
for _ in range(3):
    r = ops.noisy_conv_fwd(x, wq, w_raw, None, 1, 0, noise_mode=NOISE_EXTERNAL, current=1.0, scale_dev=scale, precision="bf16",
                           a_code_scale=s_a, w_code_scale=1.0 / 15.0, want_y=False)
gy = torch.randn_like(r["y_noisy"])
for _ in range(3):
    ops.conv_dgrad(gy, wq, x.shape, precision="bf16", w_code_scale=1.0 / 15.0)
torch.cuda.synchronize()
for _ in range(3):
    ops.conv_wgrad(gy, x, wq.shape, precision="bf16", a_code_scale=s_a)
xf = torch.randint(0, 16, (B, 3000, 1, 1), device=dev).float() * s_a
gyf = torch.randn(B, 390, 1, 1, device=dev)
for _ in range(3):
    ops.conv_wgrad(gyf, xf, (390, 3000, 1, 1), precision="bf16", a_code_scale=s_a)
torch.cuda.synchronize()
