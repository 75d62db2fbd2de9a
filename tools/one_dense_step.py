import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cave_b200 import cave_forward_backward
dev = torch.device("cuda:0")
d, m, B = 1225, 1024, 1184
g = torch.Generator(device=dev).manual_seed(d * 7 + m)
A = torch.randn((B, m, d), generator=g, device=dev)
c = torch.randn((B, d), generator=g, device=dev, dtype=torch.float64)
for _ in range(2):
    out = cave_forward_backward(c, A, 1.0, 0, reduction="none", want_status=True, dense=True)
torch.cuda.synchronize()
print("ok", float(out["loss_i"].sum()))
