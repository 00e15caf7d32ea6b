"""Launch each hot contraction of the batch-512 step a few times (for ncu captures: conv1 forward / wgrad on the in-place
kernels, conv2 forward / dgrad / wgrad on the TMA kernels)."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from noisynet_b200 import ops
from noisynet_b200._lib import NOISE_EXTERNAL, NOISE_MERGED
B = 512
dev = torch.device("cuda:0")
s_a = 5.0 / 15.0
x1 = torch.randint(0, 16, (B, 3, 32, 32), device=dev).float() * (1.0 / 15.0)
w1_raw = torch.randn(65, 3, 5, 5, device=dev) * 0.1
w1 = ops.quantize_fwd(w1_raw, 4, -1.0, 1.0, 0.0)
sc1 = ops.tensor_stats(w1_raw)[1:2]
x2 = torch.randint(0, 16, (B, 65, 14, 14), device=dev).float() * s_a
w2_raw = torch.randn(120, 65, 5, 5, device=dev) * 0.1
w2 = ops.quantize_fwd(w2_raw, 4, -1.0, 1.0, 0.0)
sc2 = ops.tensor_stats(x2)[0:1]
for _ in range(3):
    r1 = ops.noisy_conv_fwd(x1, w1, w1_raw, None, 1, 0, noise_mode=NOISE_MERGED, current=1.0, scale_dev=sc1, precision="bf16",
                            a_code_scale=1.0 / 15.0, w_code_scale=1.0 / 15.0, want_y=False)
    r2 = ops.noisy_conv_fwd(x2, w2, w2_raw, None, 1, 0, noise_mode=NOISE_EXTERNAL, current=1.0, scale_dev=sc2, precision="bf16",
                            a_code_scale=s_a, w_code_scale=1.0 / 15.0, want_y=False)
gy1 = torch.randn_like(r1["y_noisy"])
gy2 = torch.randn_like(r2["y_noisy"])
for _ in range(3):
    ops.conv_dgrad(gy2, w2, x2.shape, precision="bf16", w_code_scale=1.0 / 15.0)
    ops.conv_wgrad(gy2, x2, w2.shape, precision="bf16", a_code_scale=s_a)
    ops.conv_wgrad(gy1, x1, w1.shape, precision="bf16", a_code_scale=1.0 / 15.0)
torch.cuda.synchronize()
