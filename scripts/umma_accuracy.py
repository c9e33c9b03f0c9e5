"""Experiment (GPU): error of the tcgen05 3xTF32 projection vs fp64, by K."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gnn_tableextraction_b200 import ops

DEV = "cuda"
def padded(t):
    o = ops.empty_padded(t.shape[0], t.shape[1], DEV); o.copy_(t); return o
def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max()).item()
def mask(t):
    return (t.view(torch.int32) & -8192).view(torch.float32)

for fin in (32, 64, 128, 218, 256):
    for exact in (False, True):
        g = torch.Generator().manual_seed(fin)
        n, fo = 20000, 218
        x1, x2 = torch.randn(n, fin, generator=g), torch.randn(n, fin, generator=g)
        W = (torch.rand(fo, 2 * fin, generator=g) - 0.5) * (2.0 / (2 * fin) ** 0.5)
        if exact:
            x1, x2, W = mask(x1), mask(x2), mask(W)
        z64 = torch.cat([x1, x2], 1).double() @ W.double().t()
        pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
        z, _, _, _ = ops.umma_linear_fwd(padded(x1), padded(x2), fin, pack, None, fo)
        zf = ops.linear_fwd(padded(x1), padded(x2), W.to(DEV), None)
        d = (z.double().cpu() - z64)
        print(f"K={2*fin:4d} tf32-exact-inputs={exact!s:5}  umma {rel(z, z64):.2e}  ffma {rel(zf, z64):.2e}  "
              f"umma mean signed err*sign(z) {(d * z64.sign()).mean().item() / z64.abs().max().item():+.2e}")
