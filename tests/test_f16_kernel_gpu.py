"""GPU parity of the second-generation tensor-core forward (csrc/cheb_forward_f16.cu): one 32 -> 32 ChebConv layer,
2 <= K <= 10, binary operator, through the C-ABI, against the fp64 oracle (numpy) and the plain-C oracle.

Tolerance (north_star): 1e-5 relative, per graph, |y - y_ref|_inf / max(|y_ref|_inf, |z_ref|_inf)."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import chebnet_oracle as O
from helpers import oracle_batch_forward, random_weights, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _forward(torch, specs, ws, mats, X, bits=True):
    from multihop_offload_b200 import ChebNet, GraphBatch
    net = ChebNet(specs, device="cuda:0")
    net.set_weights(ws)
    batch = GraphBatch.from_scipy(mats, tile_rows=128, device="cuda:0")
    if not bits:
        batch.dev.pop("adj_bits", None)
        batch._struct_cache = {}
    Y = net.forward(batch, torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)).cuda())
    torch.cuda.synchronize()
    return Y.cpu().numpy(), batch, net


@pytest.mark.parametrize("K", [2, 3, 4, 5, 6, 8, 10])
def test_single_layer_all_orders(torch_cuda, K):
    """Random BA batches (several tiles per CTA for the small K), relu / leaky / none, bit rows and CSR input."""
    from multihop_offload_b200 import LayerSpec
    rng = np.random.default_rng(100 + K)
    sizes = rng.choice(np.arange(20, 111, 10), size=(700 if K <= 5 else 200))
    mats = O.make_batch(sizes, seed0=5000 + K)
    n = int(sizes.sum())
    for act in (O.ACT_LEAKY, O.ACT_RELU, O.ACT_NONE):
        specs = [LayerSpec(K, 32, 32, act, 0.2)]
        ws = random_weights(specs, rng)
        X = rng.normal(size=(n, 32))
        ref, zs = oracle_batch_forward(mats, X, ws, [act], 0.2, return_scale=True)
        for bits in (True, False):
            Y, batch, _ = _forward(torch_cuda, specs, ws, mats, X, bits)
            err = rel_err(Y, ref, batch.graph_off, zs)
            assert err < TOL, (K, act, bits, err)


def test_magnitudes_and_degenerate_graphs(torch_cuda):
    """The fp16 parts are scaled per row (X W) and per GRAPH and step (Clenshaw; mho_batch_t.tile_graph0): graphs of wildly
    different magnitude inside ONE tile, zero rows, all-zero graphs, a star graph (max degree n - 1: the loosest degree
    bound), a graph without edges, tiny graphs.  Without tile_graph0 the library falls back to the bf16 x 3 kernel."""
    from multihop_offload_b200 import LayerSpec
    rng = np.random.default_rng(7)

    def star(n):
        A = sp.lil_matrix((n, n))
        A[0, 1:] = 1.0
        A[1:, 0] = 1.0
        return sp.csr_matrix(A)

    def path(n):
        return sp.csr_matrix(sp.diags([np.ones(n - 1), np.ones(n - 1)], [-1, 1]))

    mats = [O.ba_adjacency(50, 2, 1), O.ba_adjacency(60, 2, 2),          # one tile, two graphs
            star(110), path(3), path(2), sp.csr_matrix((40, 40)),         # hub, tiny, edgeless
            O.ba_adjacency(30, 2, 3), O.ba_adjacency(30, 2, 4), O.ba_adjacency(30, 2, 5), O.ba_adjacency(30, 2, 6),
            star(128), O.ba_adjacency(100, 2, 7)]
    sizes = [m.shape[0] for m in mats]
    off = np.concatenate([[0], np.cumsum(sizes)])
    for K in (2, 5, 7):
        specs = [LayerSpec(K, 32, 32, O.ACT_LEAKY, 0.2)]
        ws = random_weights(specs, rng)
        X = rng.normal(size=(off[-1], 32))
        X[off[0]:off[1]] *= 1e-6          # tile mates nine orders of magnitude apart
        X[off[1]:off[2]] *= 1e+3
        X[off[9]:off[10]] *= 1e+2
        X[off[6]:off[7]] *= 1e-20         # tiny but normal
        X[off[7]:off[8]] *= 1e+18
        X[off[8]:off[9]] = 0.0            # an all-zero graph
        X[off[11]:off[11] + 10] = 0.0     # zero rows inside a graph
        X[off[2]] = 0.0; X[off[2], 3] = 5.0   # a single non-zero on the hub
        ref, zs = oracle_batch_forward(mats, X, ws, [s.act for s in specs], 0.2, return_scale=True)
        for bits in (True, False):
            Y, batch, _ = _forward(torch_cuda, specs, ws, mats, X, bits)
            assert np.isfinite(Y).all(), (K, bits)
            per = [np.abs(Y[off[g]:off[g + 1]] - ref[off[g]:off[g + 1]]).max() / max(np.abs(ref[off[g]:off[g + 1]]).max(), zs[g], 1e-30)
                   for g in range(len(mats))]
            assert max(per) < TOL, (K, bits, ["%d:%.2e" % (g, e) for g, e in enumerate(per) if e >= TOL])
    # without tile_graph0 the batch takes the first-generation kernel (bf16 x 3 parts, no scales): same answers
    from multihop_offload_b200 import ChebNet, GraphBatch
    specs = [LayerSpec(5, 32, 32, O.ACT_LEAKY, 0.2)]
    ws = random_weights(specs, rng)
    X = rng.normal(size=(off[-1], 32))
    X[off[0]:off[1]] *= 30.0
    ref, zs = oracle_batch_forward(mats, X, ws, [s.act for s in specs], 0.2, return_scale=True)
    net = ChebNet(specs, device="cuda:0"); net.set_weights(ws)
    batch = GraphBatch.from_scipy(mats, tile_rows=128, device="cuda:0")
    batch.dev.pop("tile_graph0", None); batch._struct_cache = {}
    Y = net.forward(batch, torch_cuda.from_numpy(X.astype(np.float32)).cuda()).cpu().numpy()
    assert rel_err(Y, ref, batch.graph_off, zs) < TOL


def test_weight_magnitudes(torch_cuda):
    """The weight image is scaled by a power of two per layer; zero kernels, tiny and large kernels, zero slices."""
    from multihop_offload_b200 import LayerSpec
    rng = np.random.default_rng(8)
    mats = O.make_batch([64, 64, 100, 20, 110], seed0=40)
    n = sum(m.shape[0] for m in mats)
    X = rng.normal(size=(n, 32))
    specs = [LayerSpec(5, 32, 32, O.ACT_NONE, 0.2)]
    for scale, kill in ((1e-12, None), (1e+6, None), (1.0, 4), (1.0, 0), (0.0, None)):
        W = rng.uniform(-1, 1, size=(5, 32, 32)) * scale
        if kill is not None:
            W[kill] = 0.0
        ws = [(W, rng.normal(size=32) * 0.1)]
        ref, zs = oracle_batch_forward(mats, X, ws, [O.ACT_NONE], 0.2, return_scale=True)
        Y, batch, _ = _forward(torch_cuda, specs, ws, mats, X)
        assert np.isfinite(Y).all()
        assert rel_err(Y, ref, batch.graph_off, np.maximum(zs, 1e-30)) < TOL, (scale, kill)


def test_bench_workload_every_graph_vs_c_oracle(torch_cuda):
    """The exact benchmark workload (bench.make_workload(1024): leaky_relu, tile-packing order), ALL 1024 graphs, with
    bit rows and with CSR input, against the plain-C fp64 oracle (oracle/cheb_oracle.c)."""
    sys.path.insert(0, ROOT)
    import bench
    import c_oracle
    from multihop_offload_b200 import ChebNet, GraphBatch, LayerSpec
    w = bench.make_workload(1024)
    ws = [(w["W"], w["b"])]
    ref = c_oracle.stack_forward(w["graph_off"], w["rowptr"], w["colidx"], None, ws, [2], 0.2, w["X"].astype(np.float64), 0)
    net = ChebNet([LayerSpec(5, 32, 32, 2, 0.2)], device="cuda:0")
    net.set_weights(ws)
    Xd = torch_cuda.from_numpy(w["X"]).cuda()
    for bits in (True, False):
        batch = GraphBatch(w["graph_off"], w["rowptr"], w["colidx"], None, device="cuda:0")
        if not bits:
            batch.dev.pop("adj_bits", None)
            batch._struct_cache = {}
        Y = net.forward(batch, Xd).cpu().numpy()
        worst = 0.0
        for g in range(1024):
            a, b = int(w["graph_off"][g]), int(w["graph_off"][g + 1])
            worst = max(worst, np.abs(Y[a:b] - ref[a:b]).max() / np.abs(ref[a:b]).max())
        assert worst < TOL, (bits, worst)
    # two launches in flight on two streams (what bench.py captures) give the same bits as a lone launch
    s1, s2 = torch_cuda.cuda.Stream(), torch_cuda.cuda.Stream()
    Y1 = torch_cuda.empty_like(Xd); Y2 = torch_cuda.empty_like(Xd)
    torch_cuda.cuda.synchronize()
    with torch_cuda.cuda.stream(s1):
        net.forward(batch, Xd, out=Y1)
    with torch_cuda.cuda.stream(s2):
        net.forward(batch, Xd, out=Y2)
    torch_cuda.cuda.synchronize()
    assert torch_cuda.equal(Y1, Y2) and np.array_equal(Y1.cpu().numpy(), Y)


def test_forward_after_optimizer_replay_uses_new_weights(torch_cuda):
    """mho_adam_replay rewrites the fp32 parameters in place: every cached weight image (walk, dense, f16) is stale after
    it.  forward -> optimizer.apply -> forward must match the oracle with the UPDATED weights on every forward path."""
    from multihop_offload_b200 import ChebNet, GraphBatch, LayerSpec, reference_stack
    from multihop_offload_b200.optim import KerasAdamReplay
    rng = np.random.default_rng(11)
    mats = O.make_batch([40, 50, 100, 64], seed0=9)
    n = sum(m.shape[0] for m in mats)
    k3 = reference_stack(K=3)[:-1] + [LayerSpec(3, 32, 1, O.ACT_NONE)]   # (a final relu over raw-adjacency K = 3 layers is dead for most seeds)
    for specs, f_in in (([LayerSpec(5, 32, 32)], 32), (reference_stack(K=1), 4), (k3, 4)):
        net = ChebNet(specs, device="cuda:0")
        ws0 = random_weights(specs, rng, 0.5)
        ws0[-1] = (ws0[-1][0], np.abs(ws0[-1][1]) + 2.0)   # keep a final relu alive
        net.set_weights(ws0)
        opt = KerasAdamReplay(net, learning_rate=5e-2)
        batch = GraphBatch.from_scipy(mats, device="cuda:0")
        X = rng.normal(size=(n, f_in))
        Xd = torch_cuda.from_numpy(X.astype(np.float32)).cuda()
        acts = [s.act for s in specs]
        Y0 = net.forward(batch, Xd).cpu().numpy()
        g = torch_cuda.from_numpy(rng.normal(size=(3, net.n_params)).astype(np.float32)).cuda()
        opt.apply(g)
        Y1 = net.forward(batch, Xd).cpu().numpy()
        ws1 = net.get_weights()
        ref1, zs = oracle_batch_forward(mats, X, ws1, acts, 0.2, return_scale=True)
        assert np.abs(Y1 - Y0).max() > 1e-4 * np.abs(Y0).max(), "the update must change the output"
        tol = TOL if len(specs) == 1 or specs[0].K == 1 else 5e-5   # deep K > 1 stacks: fp32 round-off amplification
        assert rel_err(Y1, ref1, batch.graph_off, zs) < tol, [s.K for s in specs]


def test_long_pipelines_many_tiles_per_cta(torch_cuda):
    """8192 graphs = ~4750 tiles: sixteen tiles per CTA through the warp-specialised kernel's hand-offs (named barriers,
    monotonic counters, double-buffered staging), and the same batch through the eight-warp kernel path (CSR input) -
    against the plain-C oracle, K = 5 and K = 3."""
    sys.path.insert(0, ROOT)
    import bench
    import c_oracle
    from multihop_offload_b200 import ChebNet, GraphBatch, LayerSpec
    for K in (5, 3):
        w = bench.make_workload(8192, 0, None, K=K)
        ws = [(w["W"], w["b"])]
        ref = c_oracle.stack_forward(w["graph_off"], w["rowptr"], w["colidx"], None, ws, [2], 0.2, w["X"].astype(np.float64), 0)
        net = ChebNet([LayerSpec(K, 32, 32, 2, 0.2)], device="cuda:0")
        net.set_weights(ws)
        Xd = torch_cuda.from_numpy(w["X"]).cuda()
        outs = []
        for bits in (True, False):
            batch = GraphBatch(w["graph_off"], w["rowptr"], w["colidx"], None, device="cuda:0")
            if not bits:
                batch.dev.pop("adj_bits", None)
                batch._struct_cache = {}
            Y = net.forward(batch, Xd)
            Yb = net.forward(batch, Xd)
            assert torch_cuda.equal(Y, Yb)
            outs.append(Y.cpu().numpy())
        off = w["graph_off"]
        den = np.maximum.reduceat(np.abs(ref).max(axis=1), off[:-1].astype(np.int64))
        for Y in outs:
            err = np.maximum.reduceat(np.abs(Y - ref).max(axis=1), off[:-1].astype(np.int64)) / den
            assert err.max() < TOL, (K, err.max(), int(err.argmax()))
        assert np.array_equal(outs[0], outs[1]), "the two kernels run the same arithmetic"
