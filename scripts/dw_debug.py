import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gnn_tableextraction_b200 import ops
DEV="cuda"
def padded(t):
    o = ops.empty_padded(t.shape[0], t.shape[1], DEV); o.copy_(t); return o
for (n,fo,k) in [(32,128,32),(64,128,32),(512,128,64),(1000,218,218)]:
    g=torch.Generator().manual_seed(1)
    dz=torch.randn(n,fo,generator=g); x=torch.randn(n,k,generator=g)
    dW=torch.full((fo,k),7.0,device=DEV)
    ops.umma_linear_bwd_weight(padded(dz), padded(x), None, dW, None)
    ref=dz.double().t()@x.double()
    out=dW.double().cpu()
    err=((out-ref).abs().max()/ref.abs().max()).item()
    print(f"n={n} fo={fo} k={k}: err {err:.3e} out[0,:4]={out[0,:4].tolist()} ref[0,:4]={ref[0,:4].tolist()} absmax out {out.abs().max().item():.3e}")
    # structured probe: dz = e_r0 (single nonzero row), x = arange
    dz2=torch.zeros(n,fo); dz2[3,5]=1.0
    x2=torch.arange(n*k,dtype=torch.float32).reshape(n,k)/16
    ops.umma_linear_bwd_weight(padded(dz2), padded(x2), None, dW, None)
    o=dW.cpu()
    nz=o.nonzero()
    print("   probe nonzeros:", nz[:6].tolist(), "values", [round(o[i,j].item(),3) for i,j in nz[:6].tolist()], "expected row 5 =", x2[3,:4].tolist())
