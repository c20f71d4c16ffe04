"""GPU parity: VJP (mho_cheb_backward) and optimizer replay (mho_adam_replay) vs the fp64 oracle."""
import glob
import os

import numpy as np
import pytest
import scipy.sparse as sp

import chebnet_oracle as O
from helpers import random_weights, rel_err

pytestmark = pytest.mark.gpu
GTOL = 2e-5  # gradients: sums over all nodes of a graph in fp32 vs fp64


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _oracle_grads(mats, X, ws, acts, dY, slope=0.2):
    outs, gs, dxs, o = [], [], [], 0
    for A in mats:
        n = A.shape[0]
        y, cache = O.cheb_stack_forward(A, X[o:o + n], ws, acts, slope, return_cache=True)
        g, dx = O.cheb_stack_backward(A, ws, cache, dY[o:o + n], slope)
        outs.append(y); gs.append(O.flatten_params(g)); dxs.append(dx)
        o += n
    return np.concatenate(outs), np.stack(gs), np.concatenate(dxs)


def _run_bwd(torch, specs, ws, mats, X, dY, binary=None):
    from multihop_offload_b200 import ChebNet, GraphBatch
    net = ChebNet(specs, device="cuda:0"); net.set_weights(ws)
    batch = GraphBatch.from_scipy(mats, binary=binary, device="cuda:0")
    Xd = torch.from_numpy(X.astype(np.float32)).cuda()
    Y, saved = net.forward(batch, Xd, save=True)
    gpg, gsum, dX = net.backward(batch, Xd, Y, saved, torch.from_numpy(dY.astype(np.float32)).cuda(), need_dx=True)
    torch.cuda.synchronize()
    return Y.cpu().numpy(), gpg.cpu().numpy(), gsum.cpu().numpy(), dX.cpu().numpy(), batch


def test_backward_random_stacks(torch_cuda):
    from multihop_offload_b200 import LayerSpec, reference_stack
    rng = np.random.default_rng(5)
    configs = [
        (reference_stack(K=1), "raw-adj", 0.5),
        (reference_stack(K=3), "cheb-lap", 1.0),
        ([LayerSpec(5, 32, 32)], "cheb-lap", 1.0),
        ([LayerSpec(4, 7, 13), LayerSpec(2, 13, 20, O.ACT_NONE), LayerSpec(3, 20, 5, O.ACT_RELU)], "cheb-lap", 1.0),
        ([LayerSpec(2, 32, 32), LayerSpec(1, 32, 32), LayerSpec(6, 32, 2, O.ACT_RELU)], "cheb-lap", 1.0),
    ]
    for specs, op, scale in configs:
        sizes = rng.choice([20, 33, 47, 64, 100, 110, 200], size=9)
        mats = O.make_batch(sizes, seed0=int(rng.integers(1 << 20)), operator=op)
        n = int(sizes.sum())
        X = rng.normal(size=(n, specs[0].f_in))
        ws = random_weights(specs, rng, scale, bias=0.2)
        dY = rng.normal(size=(n, specs[-1].f_out))
        acts = [s.act for s in specs]
        Y, gpg, gsum, dX, batch = _run_bwd(torch_cuda, specs, ws, mats, X, dY)
        yr, gr, dxr = _oracle_grads(mats, X, ws, acts, dY)
        tag = [(s.K, s.f_in, s.f_out) for s in specs]
        for gi in range(len(mats)):
            assert rel_err(gpg[gi], gr[gi]) < GTOL, (tag, gi, rel_err(gpg[gi], gr[gi]))
        assert rel_err(gsum, gr.sum(0)) < GTOL, tag
        assert rel_err(dX, dxr, batch.graph_off) < GTOL, (tag, rel_err(dX, dxr, batch.graph_off))


def test_backward_non_symmetric_weighted(torch_cuda):
    from multihop_offload_b200 import LayerSpec
    rng = np.random.default_rng(11)
    specs = [LayerSpec(4, 32, 16), LayerSpec(3, 16, 4, O.ACT_RELU)]
    ws = random_weights(specs, rng, 0.8, bias=0.2)
    mats = []
    for i in range(7):
        n = int(rng.integers(3, 90))
        A = sp.random(n, n, min(1.0, 5.0 / n), random_state=100 + i, format="csr")
        A.data[:] = rng.uniform(-0.3, 0.3, size=A.nnz)
        mats.append(A)
    n = sum(m.shape[0] for m in mats)
    X = rng.normal(size=(n, 32)); dY = rng.normal(size=(n, 4))
    Y, gpg, gsum, dX, batch = _run_bwd(torch_cuda, specs, ws, mats, X, dY, binary=False)
    assert not batch.symmetric
    yr, gr, dxr = _oracle_grads(mats, X, ws, [s.act for s in specs], dY)
    for gi in range(len(mats)):
        assert rel_err(gpg[gi], gr[gi]) < GTOL
    assert rel_err(dX, dxr, batch.graph_off) < GTOL


def test_backward_golden_rollout_cases(torch_cuda, golden_dir):
    """Shipped checkpoint x shipped networks: gradient of the weights seeded through the queue head."""
    from multihop_offload_b200 import reference_stack
    for tag, K, ykey, gkey in (("BAT800", 1, "lam", "grad_flat"), ("K3", 3, "lam_K3", "grad_flat_K3")):
        w = np.load(os.path.join(golden_dir, "weights_%s.npz" % tag))
        ws = [(w["W%d" % i], w["b%d" % i]) for i in range(5)]
        for f in sorted(glob.glob(os.path.join(golden_dir, "case*.npz"))):
            z = np.load(f)
            n = z["X"].shape[0]
            A = sp.csr_matrix((z["vals"], z["colidx"], z["rowptr"]), shape=(n, n))
            dY = z["g_lam"] if K == 1 else z["dY_K3"]
            Y, gpg, gsum, dX, _ = _run_bwd(torch_cuda, reference_stack(K=K), ws, [A], z["X"], dY)
            assert rel_err(Y, z[ykey]) < 1e-5
            assert rel_err(gpg[0], z[gkey]) < GTOL, (tag, os.path.basename(f), rel_err(gpg[0], z[gkey]))
            if K == 3:
                assert rel_err(dX, z["dX_K3"]) < GTOL


def test_backward_rejects_invalid_layer_stacks(torch_cuda):
    """mho_cheb_backward checks the layer stack as mho_cheb_forward does: widths that do not chain and an unknown activation
    are MHO_ERR_INVALID, and nothing is launched.  The batch has no graphs and the gradient buffers are NULL, so an accepted
    stack would not launch or write anything either."""
    import ctypes as C
    from multihop_offload_b200 import _lib
    ctx = _lib.Context.get(0)
    buf = torch_cuda.zeros(4096, dtype=torch_cuda.float32, device="cuda:0")
    offs = torch_cuda.zeros(1, dtype=torch_cuda.int32, device="cuda:0")
    b = _lib.mho_batch_t()
    b.graph_off = offs.data_ptr(); b.rowptr = offs.data_ptr(); b.max_tile_rows = 1
    p = buf.data_ptr()
    before = ctx.launch_count()
    for layers in ([(3, 32, 16, O.ACT_LEAKY), (2, 8, 1, O.ACT_RELU)],   # f_in 8 != previous f_out 16
                   [(3, 32, 32, 3)]):                                  # act 3 does not exist
        arr = (_lib.mho_layer_t * len(layers))(*[_lib.mho_layer_t(K, fi, fo, act, 0.2, p, p) for K, fi, fo, act in layers])
        rc = ctx.lib.mho_cheb_backward(ctx.handle, C.byref(b), arr, len(layers), p, p, p, p, None, None, None, None)
        assert rc == -1, (layers, rc)   # MHO_ERR_INVALID
    assert ctx.launch_count() == before


def test_adam_replay_matches_keras_semantics(torch_cuda):
    from multihop_offload_b200 import ChebNet, reference_stack
    from multihop_offload_b200.optim import KerasAdamReplay
    rng = np.random.default_rng(3)
    for K, lr, decay in ((1, 1e-4, 1.0), (3, 1e-2, 0.9), (2, 1e-6, 1.0)):
        specs = reference_stack(K=K)
        ws = random_weights(specs, rng, 1.5, bias=0.4)   # some columns exceed max_norm -> constraint active
        net = ChebNet(specs, device="cuda:0"); net.set_weights(ws)
        opt = KerasAdamReplay(net, learning_rate=lr, decay_rate=decay)
        flat0 = O.flatten_params(ws)
        opt.set_master(flat0)
        n_steps = 23
        grads = rng.normal(size=(n_steps, net.n_params)) * rng.choice([0.01, 1.0, 30.0], size=(n_steps, 1))
        g32 = grads.astype(np.float32)
        shapes = []
        for s in specs:
            shapes += [(s.K, s.f_in, s.f_out), (s.f_out,)]
        ref = O.KerasAdam(shapes, lr=lr, decay_rate=decay)
        params, o = [], 0
        for sh in shapes:
            sz = int(np.prod(sh)); params.append(flat0[o:o + sz].reshape(sh).copy()); o += sz
        # two calls (10 + 13 steps) to exercise the iteration counter
        opt.apply(torch_cuda.from_numpy(g32[:10]).cuda()); opt.apply(torch_cuda.from_numpy(g32[10:]).cuda())
        torch_cuda.cuda.synchronize()
        for s in range(n_steps):
            gl, o = [], 0
            for sh in shapes:
                sz = int(np.prod(sh)); gl.append(g32[s, o:o + sz].astype(np.float64).reshape(sh)); o += sz
            ref.apply(params, gl)
        want = np.concatenate([p.ravel() for p in params])
        got = opt.get_master()
        np.testing.assert_allclose(got, want, rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(net.get_flat(), want.astype(np.float32), rtol=0, atol=0)
        assert opt.iterations == n_steps
