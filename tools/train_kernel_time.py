"""Average duration of the training-step kernels (CUDA events around isolated calls): python tools/train_kernel_time.py"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import stribor_b200 as st

rows, d = 1 << 18, 128
dev = torch.device('cuda')
torch.manual_seed(0)
layer = st.Coupling(st.Spline(d, 16, latent_net=st.net.MLP(d, [64], d * 47), lower=-4, upper=4, spline_type='quadratic'),
                    mask='ordered_right_half').to(dev)
x = torch.randn(rows, d, device=dev, requires_grad=True)
for _ in range(3):
    y, ld = layer.inverse_and_log_det_jacobian(x)
    (y.sum() + ld.sum()).backward()
torch.cuda.synchronize()
e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
n = 10
tf = tb = 0.0
for _ in range(n):
    e[0].record()
    y, ld = layer.inverse_and_log_det_jacobian(x)
    e[1].record()
    loss = y.sum() + ld.sum()
    torch.cuda.synchronize()
    e[0].synchronize()
    tf += e[0].elapsed_time(e[1])
    e[1].record()
    loss.backward()
    e[2].record()
    torch.cuda.synchronize()
    tb += e[1].elapsed_time(e[2])
print(f'forward {tf / n:.3f} ms, backward (incl. host-side ops) {tb / n:.3f} ms per layer at {rows} rows')
