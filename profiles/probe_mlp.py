import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pivotcvae_b200 import ops
B=1024
g=torch.Generator(device="cuda").manual_seed(0)
x=torch.randn(B,27,generator=g,device="cuda")
dims=[27,256,256,8]
layers=[]
for i in range(3):
    layers.append((torch.randn(dims[i+1],dims[i],generator=g,device="cuda")*0.1, torch.zeros(dims[i+1],device="cuda"), 1 if i<2 else 0))
for _ in range(3): ops.mlp_forward([ops.Dense(x)], layers, B)
torch.cuda.synchronize()
s,e=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
s.record()
for _ in range(50): ops.mlp_forward([ops.Dense(x)], layers, B)
e.record(); torch.cuda.synchronize()
print("mlp block B=%d: %.2f us"%(B, s.elapsed_time(e)/50*1000))
