import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "warp-transducer_b200"))
from warprnnt_pytorch.joint import AddJointRNNTLoss
dev = torch.device("cuda:0")
N, T, L, V = 128, 150, 20, 5000
U = L + 1
trans = torch.rand((N, T, V), device=dev, requires_grad=True)
pred = torch.rand((N, U, V), device=dev, requires_grad=True)
labels = torch.as_tensor(np.random.default_rng(1).integers(1, V, size=(N, L)).astype(np.int32)).to(dev)
tl = torch.full((N,), T, dtype=torch.int32, device=dev)
ul = torch.full((N,), L, dtype=torch.int32, device=dev)
f = AddJointRNNTLoss()
for _ in range(2):
    trans.grad = pred.grad = None
    f(trans, pred, labels, tl, ul).backward()
torch.cuda.synchronize()
