import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cave_b200 import cave_forward_backward, pack_constraints, synth
dev = torch.device("cuda:0")
insts = synth.make_batch("tsp50", 4096, seed=1000)
A = synth.densify(insts, device=dev)
pred = torch.tensor(synth.predictions(insts, 1000, "uniform"), device=dev)
pack = pack_constraints(A)
for mi in (1, 2, 3, 4, 6, 200):
    fn = lambda: cave_forward_backward(pred, A, -1.0, 1, 0.2, "mean", pack=pack, max_iter=mi)
    for _ in range(3): fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(5): fn()
    e1.record(); torch.cuda.synchronize()
    print(f"max_iter={mi:4d}: solve kernel {e0.elapsed_time(e1)/5:7.3f} ms")
