"""Long CTA pipelines (many tiles / graphs per CTA): writes the forward output and the VJP gradients of a big batch to an .npz.
usage: stress_long.py out.npz [graphs=8192] [K=5]   (run against two builds, MHO_LIB=..., and compare)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, bench
from multihop_offload_b200 import ChebNet, GraphBatch, LayerSpec
out = sys.argv[1]; graphs = int(sys.argv[2]) if len(sys.argv) > 2 else 8192; K = int(sys.argv[3]) if len(sys.argv) > 3 else 5
w = bench.make_workload(graphs, 0, None, K=K)
dev = torch.device("cuda:0")
net = ChebNet([LayerSpec(K, 32, 32, 2, 0.2)], device=dev)
net.set_weights([(w["W"], w["b"])])
b = GraphBatch(w["graph_off"], w["rowptr"], w["colidx"], None, device=dev)
X = torch.from_numpy(w["X"]).to(dev)
Y = net.forward(b, X)
torch.manual_seed(1)
dY = torch.randn_like(Y)
Y2, saved = net.forward(b, X, save=True)
gpg, gsum, _ = net.backward(b, X, Y2, saved, dY)
gpg2, gsum2, _ = net.backward(b, X, Y2, saved, dY)
torch.cuda.synchronize()
assert torch.equal(Y, Y2) and torch.equal(gpg, gpg2) and torch.equal(gsum, gsum2), "not repeatable"
print("tiles", b.n_tiles, "graphs", graphs, "nan", bool(torch.isnan(Y).any()), bool(torch.isnan(gpg).any()))
np.savez(out, Y=Y.cpu().numpy(), gsum=gsum.cpu().numpy(), g0=gpg[::97].cpu().numpy())
