"""CPU: the oracle against the committed golden vectors and algebraic invariants."""
import glob
import os

import numpy as np
import scipy.sparse as sp

import chebnet_oracle as O


def _weights(golden_dir, tag):
    z = np.load(os.path.join(golden_dir, "weights_%s.npz" % tag))
    n = len([k for k in z.files if k.startswith("W")])
    return [(z["W%d" % i], z["b%d" % i]) for i in range(n)]


def _case_adj(z):
    n = z["X"].shape[0]
    return sp.csr_matrix((z["vals"], z["colidx"], z["rowptr"]), shape=(n, n))


def test_shipped_checkpoint_shapes(golden_dir):
    for tag in ("BAT800", "BAT950"):
        ws = _weights(golden_dir, tag)
        assert [W.shape for W, _ in ws] == [(1, 4, 32), (1, 32, 32), (1, 32, 32), (1, 32, 32), (1, 32, 1)]
        assert sum(W.size + b.size for W, b in ws) == 3361


def test_golden_cases_reproduce(golden_dir):
    ws = _weights(golden_dir, "BAT800")
    ws3 = _weights(golden_dir, "K3")
    files = sorted(glob.glob(os.path.join(golden_dir, "case*.npz")))
    assert len(files) >= 6
    for f in files:
        z = np.load(f)
        A = _case_adj(z)
        lam, cache = O.cheb_stack_forward(A, z["X"], ws, return_cache=True)
        np.testing.assert_allclose(lam, z["lam"], rtol=1e-12, atol=1e-12)
        assert (lam >= 0).all()
        n = A.shape[0]
        Ai = sp.csr_matrix((z["adj_i_vals"], z["adj_i_colidx"], z["adj_i_rowptr"]),
                           shape=(len(z["link_rates"]),) * 2)
        ld, nd, hc = O.queue_head_forward(lam, z["maps_ol_el"], z["maps_on_el"], z["link_rates"], z["cf_degs"],
                                          z["proc_bws"], Ai, int(z["T"]), return_cache=True)
        np.testing.assert_allclose(ld, z["link_delay"], rtol=1e-12)
        np.testing.assert_allclose(nd, z["node_delay"], rtol=1e-12)
        D = O.delay_matrix(ld, nd, int(z["num_nodes"]), z["edges"], z["link_matrix"], z["comp_nodes"], True)
        np.testing.assert_array_equal(np.isnan(D), np.isnan(z["delay_mtx_bug"]))
        np.testing.assert_allclose(np.nan_to_num(D), np.nan_to_num(z["delay_mtx_bug"]), rtol=1e-12)
        lam3 = O.cheb_stack_forward(A, z["X"], ws3)
        np.testing.assert_allclose(lam3, z["lam_K3"], rtol=1e-11, atol=1e-11)


def test_k1_is_independent_of_the_operator(golden_dir):
    """Spektral default K=1: the adjacency is never multiplied (SURVEY fact 0.3)."""
    ws = _weights(golden_dir, "BAT800")
    z = np.load(os.path.join(golden_dir, "case0.npz"))
    A = _case_adj(z)
    lam = O.cheb_stack_forward(A, z["X"], ws)
    lam2 = O.cheb_stack_forward(sp.identity(A.shape[0], format="csr") * 3.0, z["X"], ws)
    np.testing.assert_array_equal(lam, lam2)


def test_chebyshev_polynomials_on_diagonal_operator():
    rng = np.random.default_rng(0)
    d = rng.uniform(-1, 1, size=9)
    A = sp.diags(d).tocsr()
    X = rng.normal(size=(9, 3))
    Ts = O.cheb_basis(A, X, 7)
    for k, T in enumerate(Ts):
        coef = np.zeros(k + 1); coef[k] = 1
        np.testing.assert_allclose(T, np.polynomial.chebyshev.chebval(d, coef)[:, None] * X, atol=1e-12)


def test_permutation_equivariance():
    rng = np.random.default_rng(1)
    A = O.ba_adjacency(25, 2, 3)
    X = rng.normal(size=(25, 4))
    ws = O.glorot_weights([4, 8, 1], 3, rng)
    ws = [(W, b + 0.2) for W, b in ws]
    perm = rng.permutation(25)
    P = sp.csr_matrix((np.ones(25), (np.arange(25), perm)), shape=(25, 25))
    y = O.cheb_stack_forward(A, X, ws)
    yp = O.cheb_stack_forward(P @ A @ P.T, P @ X, ws)
    np.testing.assert_allclose(yp, P @ y, atol=1e-10)


def test_vjp_matches_finite_differences():
    rng = np.random.default_rng(2)
    A = O.ba_adjacency(14, 2, 5)
    A = 0.15 * (A + sp.random(14, 14, 0.1, random_state=3, format="csr"))  # NON-symmetric, well-conditioned for FD
    X = rng.normal(size=(14, 4))
    ws = O.glorot_weights([4, 6, 6, 2], 4, rng)
    ws = [(W, rng.normal(size=b.shape) * 0.1 + 0.3) for W, b in ws]
    Y, cache = O.cheb_stack_forward(A, X, ws, return_cache=True)
    dY = rng.normal(size=Y.shape)
    grads, dX = O.cheb_stack_backward(A, ws, cache, dY)

    def f():
        return float((O.cheb_stack_forward(A, X, ws) * dY).sum())

    eps = 1e-6
    for li, (W, b) in enumerate(ws):
        for _ in range(4):
            idx = tuple(rng.integers(0, s) for s in W.shape)
            old = W[idx]; W[idx] = old + eps; fp = f(); W[idx] = old - eps; fm = f(); W[idx] = old
            assert abs((fp - fm) / (2 * eps) - grads[li][0][idx]) <= 1e-5 * (1 + abs(grads[li][0][idx]))
        j = int(rng.integers(0, b.size))
        old = b[j]; b[j] = old + eps; fp = f(); b[j] = old - eps; fm = f(); b[j] = old
        assert abs((fp - fm) / (2 * eps) - grads[li][1][j]) <= 1e-5 * (1 + abs(grads[li][1][j]))
    old = X[3, 1]; X[3, 1] = old + eps; fp = f(); X[3, 1] = old - eps; fm = f(); X[3, 1] = old
    assert abs((fp - fm) / (2 * eps) - dX[3, 1]) <= 1e-5 * (1 + abs(dX[3, 1]))


def test_queue_head_vjp_matches_finite_differences(golden_dir):
    z = np.load(os.path.join(golden_dir, "case0.npz"))
    L = len(z["link_rates"])
    Ai = sp.csr_matrix((z["adj_i_vals"], z["adj_i_colidx"], z["adj_i_rowptr"]), shape=(L, L))
    lam = z["lam"].copy()
    rng = np.random.default_rng(5)

    def run(lm):
        return O.queue_head_forward(lm, z["maps_ol_el"], z["maps_on_el"], z["link_rates"], z["cf_degs"],
                                    z["proc_bws"], Ai, int(z["T"]), return_cache=True)

    ld, nd, hc = run(lam)
    g_ld, g_nd = rng.normal(size=ld.shape), rng.normal(size=nd.shape)
    g = O.queue_head_vjp(hc, g_ld, g_nd, lam.shape[0], z["maps_ol_el"], z["maps_on_el"])
    np.testing.assert_allclose(g, z["g_lam"] * 0 + g)  # shape check
    eps = 1e-6
    for i in rng.choice(lam.shape[0], size=12, replace=False):
        lp, lm_ = lam.copy(), lam.copy()
        lp[i] += eps; lm_[i] -= eps
        a, b, _ = run(lp); c, d, _ = run(lm_)
        fd = ((a - c) * g_ld).sum() / (2 * eps) + ((b - d) * g_nd).sum() / (2 * eps)
        assert abs(fd - g[i, 0]) <= 1e-5 * (1 + abs(g[i, 0])), (i, fd, g[i, 0])


def test_keras_adam_clipnorm_and_max_norm():
    rng = np.random.default_rng(3)
    shapes = [(1, 4, 8), (8,)]
    params = [rng.normal(size=s) * 2 for s in shapes]
    opt = O.KerasAdam(shapes, lr=0.1)
    for _ in range(5):
        grads = [rng.normal(size=s) * 10 for s in shapes]
        opt.apply(params, grads)
    # max_norm(axis=0): kernel is clamped elementwise for K=1, bias by its L2 norm
    assert np.abs(params[0]).max() <= 1.0 + 1e-6
    assert np.sqrt((params[1] ** 2).sum()) <= 1.0 + 1e-6


def test_tf_bundle_reader_matches_golden_when_reference_present(golden_dir):
    """tests/golden/ckpt_BAT800 is the reference's shipped model_ChebConv_BAT800_a5_c5_ACO_agent, byte for byte (SHA-256
    of the reference's files below); read back, it holds the golden weights."""
    import hashlib
    ref = os.path.join(golden_dir, "ckpt_BAT800")
    shipped = {"checkpoint": "fd8cedf447ada3326c854af6fcdf33c8e714bbae68ee9cbf79b235f5129d1c17",
               "cp-0000.ckpt.data-00000-of-00001": "5f17759de8bd7c342383b0da157cde055dfbfe7f5e5d67a6e2a02fe9bba42df4",
               "cp-0000.ckpt.index": "97e5b9767c44c10ac1295eef488d19296bd8d53ba67a3fd8676c517373046108"}
    for name, digest in shipped.items():
        with open(os.path.join(ref, name), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, name
    ws = O.load_reference_weights(ref)
    gold = _weights(golden_dir, "BAT800")
    for (W, b), (Wg, bg) in zip(ws, gold):
        np.testing.assert_array_equal(W, Wg)
        np.testing.assert_array_equal(b, bg)
