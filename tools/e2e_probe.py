"""e2e probe: time mho_cheb_forward_host on the benchmark batch from page-locked buffers."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, bench
from multihop_offload_b200 import ChebNet, LayerSpec
from multihop_offload_b200._lib import pinned_like
w = bench.make_workload(1024)
net = ChebNet([LayerSpec(5, 32, 32, 2, 0.2)], device="cuda:0")
n = int(w["graph_off"][-1])
X = np.random.default_rng(0).standard_normal((n, 32)).astype(np.float32)
bufs = {k: pinned_like(np.ascontiguousarray(v)) for k, v in dict(g=w["graph_off"].astype(np.int32), r=w["rowptr"].astype(np.int32), c=w["colidx"].astype(np.int32), x=X).items()}
Y = pinned_like(np.zeros((n, 32), np.float32))
def step():
    net.forward_host(bufs["g"].array, bufs["r"].array, bufs["c"].array, None, bufs["x"].array, Y.array)
for _ in range(5): step()
t = time.perf_counter()
for _ in range(30): step()
print("us/step %.1f" % ((time.perf_counter() - t) / 30 * 1e6))
