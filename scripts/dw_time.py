import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gnn_tableextraction_b200 import ops
DEV="cuda"
n,fo,k=153600,218,218
dz=ops.empty_padded(n,fo,DEV); dz.normal_()
x1=ops.empty_padded(n,k,DEV); x1.normal_()
x2=ops.empty_padded(n,k,DEV); x2.normal_()
dW=torch.empty(fo,2*k,device=DEV)
for _ in range(3): ops.umma_linear_bwd_weight(dz,x1,x2,dW,None)
torch.cuda.synchronize()
e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10): ops.umma_linear_bwd_weight(dz,x1,x2,dW,None)
e1.record(); torch.cuda.synchronize()
print("dW ms", e0.elapsed_time(e1)/10)
