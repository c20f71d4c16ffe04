"""Debug probe for the fp16-parts forward kernel (cheb_forward_f16.cu): one 32->32 layer, K given on the command line,
small and full-size batches, with bit rows and with CSR input; prints the per-graph error against the fp64 oracle."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import chebnet_oracle as O
from helpers import rel_err, oracle_batch_forward, random_weights
from multihop_offload_b200 import ChebNet, GraphBatch, LayerSpec

Ks = [int(a) for a in sys.argv[1:]] or [5]
rng = np.random.default_rng(0)
for K in Ks:
    for sizes, tag in (([20, 50, 110, 64, 30, 100, 128, 3, 5], "small"), (list(rng.choice(np.arange(20, 111, 10), size=96)), "96 graphs")):
        mats = O.make_batch(sizes, seed0=1000)
        specs = [LayerSpec(K, 32, 32)]
        ws = random_weights(specs, rng)
        net = ChebNet(specs, device="cuda:0"); net.set_weights(ws)
        for bits in (True, False):
            batch = GraphBatch.from_scipy(mats, tile_rows=128, device="cuda:0")
            if not bits:
                batch.dev.pop("adj_bits", None); batch._struct_cache = {}
            X = rng.normal(size=(batch.total_nodes, 32)) * (3.0 if tag == "small" else 1.0)
            Xd = torch.from_numpy(X.astype(np.float32)).cuda()
            t0 = time.time()
            Y = net.forward(batch, Xd)
            torch.cuda.synchronize()
            Y = Y.cpu().numpy()
            ref, sc = oracle_batch_forward(mats, X, ws, [s.act for s in specs], 0.2, return_scale=True)
            goff = np.concatenate([[0], np.cumsum([m.shape[0] for m in mats])])
            err = rel_err(Y, ref, goff, sc)
            print("K=%d %-10s bits=%s tiles=%d  rel err %.3g  nan %d  (%.1f ms)" % (K, tag, bits, batch.n_tiles, err, int(np.isnan(Y).sum()), 1e3 * (time.time() - t0)), flush=True)
            if not (err < 1e-5):
                for g in range(len(mats)):
                    a, b = goff[g], goff[g + 1]
                    e = np.abs(Y[a:b] - ref[a:b]).max() / max(np.abs(ref[a:b]).max(), sc[g], 1e-30)
                    if not (e < 1e-5): print("   graph %d n=%d rows [%d,%d) err %.3g  Y %s ref %s" % (g, b - a, a, b, e, Y[a, :3], ref[a, :3]))
