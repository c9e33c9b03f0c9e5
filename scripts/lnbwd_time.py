import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gnn_tableextraction_b200 import ops
DEV="cuda"; n,f=153600,218
dy=ops.empty_padded(n,f,DEV); dy.normal_(); z=ops.empty_padded(n,f,DEV); z.normal_()
mean=torch.zeros(n,device=DEV); rstd=torch.ones(n,device=DEV); g=torch.ones(f,device=DEV); b=torch.zeros(f,device=DEV)
dg=torch.empty(f,device=DEV); db=torch.empty(f,device=DEV); dc=torch.empty(f,device=DEV)
fn=lambda: ops.layernorm_act_bwd(dy,z,mean,rstd,g,b,True,dg,db,False,dz_colsum=dc)
for _ in range(3): fn()
torch.cuda.synchronize()
e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20): fn()
e1.record(); torch.cuda.synchronize()
ms=e0.elapsed_time(e1)/20
print("ln bwd us", ms*1e3, "GB/s", 12*n*f/ms/1e6)
