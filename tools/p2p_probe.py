import sys, os
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import torch
x = torch.ones(1 << 20, device="cuda:1"); y = x.to("cuda:0"); torch.cuda.synchronize()
print("peer access 0<->1:", torch.cuda.can_device_access_peer(0, 1))
sys.argv = ["x", "sp5", "4096", "0", "1000"]
exec(open(os.path.join(HERE, "seed_probe_structured.py")).read())
