"""GPU: mho_env_step (csrc/env_step.cu) bit for bit against the reference's recorded offloading() / local_compute() +
run() (tests/golden/env_cases.npz) and against the numpy oracle on random synthetic items; per-item status of
malformed items; argument checks."""
import ctypes as C

import networkx as nx
import numpy as np
import pytest
import scipy.sparse as sp

import env_oracle
from test_env_step import assert_same, golden_cases

pytestmark = pytest.mark.gpu


def test_kernel_matches_recording_in_one_batch(golden_dir):
    from multihop_offload_b200 import env_step as ES
    cases = list(golden_cases(golden_dir))
    net, items = ES.merge([(c[0], c[1]) for c in cases])
    got = ES.launch(net, items)
    want = env_oracle.env_step(net, items)
    assert_same(got, want, "merged")
    # and each case's slice equals the reference's recording
    jo, io_ = 0, 0
    for c, (_, it, rec) in enumerate(cases):
        nj, ni = int(it["job_off"][-1]), it["n_items"]
        for k in ("dst", "nhop", "delay_est", "delay_emp"):
            assert np.array_equal(got[k][jo:jo + nj], rec[k], equal_nan=True), (c, k)
        assert np.all(got["status"][io_:io_ + ni] == 0)
        jo += nj; io_ += ni
    for k in ("delay_links", "delay_nodes", "unit"):
        assert np.array_equal(got[k], np.concatenate([r[k] for _, _, r in cases]), equal_nan=True), k


class SynthEnv:
    """An AdhocCloud-shaped network: BA connectivity graph, its line graph as conflict graph."""

    def __init__(self, n, seed, rng, n_servers=6):
        g = nx.barabasi_albert_graph(n, 2, seed=seed)
        self.graph_c = g
        self.num_nodes = n
        gi = nx.line_graph(g)
        self.link_list = list(gi.nodes)
        self.num_links = len(self.link_list)
        self.adj_c = sp.csr_matrix(nx.adjacency_matrix(g))
        self.adj_i = sp.csr_matrix(nx.adjacency_matrix(gi, nodelist=self.link_list))
        self.cf_degs = np.asarray(self.adj_i.sum(axis=0)).flatten()
        self.link_rates = np.round(rng.uniform(0, 30, self.num_links))
        self.servers = sorted(int(x) for x in rng.choice(n, n_servers, replace=False))
        self.proc_bws = rng.uniform(0.5, 3, n)
        self.proc_bws[self.servers] = rng.uniform(5, 20, n_servers)
        self.T = 1000
        hop = dict(nx.all_pairs_shortest_path_length(g))
        self.hop = np.array([[hop[a].get(b, np.inf) for b in range(n)] for a in range(n)], np.float64)


def _random_items(env, rng, n_items):
    from multihop_offload_b200 import env_step as ES
    n = env.num_nodes
    sps, items = [], []
    for i in range(n_items):
        if i % 6 == 5:   # arbitrary positive matrices: many walks never arrive
            s = rng.uniform(0.01, 5.0, (n, n))
        else:            # shortest-path lengths of random (rounded: ties) edge weights
            w = rng.uniform(0.5, 5.0, env.graph_c.number_of_edges())
            w = np.round(w) if i % 3 == 0 else w
            for (a, b), x in zip(env.graph_c.edges, w):
                env.graph_c[a][b]["w"] = float(x)
            d = dict(nx.all_pairs_dijkstra_path_length(env.graph_c, weight="w"))
            s = np.array([[d[a].get(b, np.inf) for b in range(n)] for a in range(n)])
        np.fill_diagonal(s, rng.uniform(0.0, 0.05, n))
        sps.append(s)
        J = int(rng.choice([0, 1, 3, 7, 8, 9, 40, 129, 300]))
        src = rng.integers(0, n, J).astype(np.int32)
        items.append(ES.EnvItem(ES.LOCAL if i % 4 == 1 else ES.GREEDY, i, src, rng.uniform(0.01, 2.0, J),
                                rng.choice([100.0, 50.0, 7.5], J), rng.choice([1.0, 2.0, 0.5], J)))
    return sps, items


def test_kernel_matches_oracle_random_items():
    from multihop_offload_b200 import env_step as ES
    rng = np.random.default_rng(21)
    batches = []
    for k, n in enumerate((12, 60, 200)):
        env = SynthEnv(n, 40 + k, rng)
        net = ES.network_arrays(env, env.hop)
        sps, items = _random_items(env, rng, 12)
        batches.append((net, ES.item_arrays(net, sps, items)))
    net, items = ES.merge(batches)
    got = ES.launch(net, items)
    want = env_oracle.env_step(net, items)
    assert np.any(want["status"] == 0)
    assert_same(got, want, "random")
    # a plan over one network: the same numbers through EnvPlan.step
    env = SynthEnv(30, 3, rng)
    sps, its = _random_items(env, rng, 5)
    plan = ES.EnvPlan(env, env.hop)
    res = plan.step(sps, its)
    o = env_oracle.env_step(plan.net, ES.item_arrays(plan.net, sps, its))
    assert np.array_equal(np.concatenate([r.delay_emp for r in res]), o["delay_emp"], equal_nan=True)


def test_status_of_malformed_items_leaves_others_intact():
    from multihop_offload_b200 import env_step as ES
    rng = np.random.default_rng(4)
    env = SynthEnv(40, 8, rng)
    good = ES.network_arrays(env, env.hop)
    broken = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in good.items()}
    broken["adj_link"][:] = -1                      # no adjacency entry has a link
    n = env.num_nodes
    src = np.array([v for v in range(n) if v not in env.servers][:5], np.int32)
    jobs = (src, np.full(5, 0.1), np.full(5, 100.0), np.full(5, 1.0))
    base = env.hop.copy()                           # hop distances: every walk reaches its server
    cyc = -env.hop                                  # every step leads away from the server: a walk cycles
    for m in (base, cyc):
        np.fill_diagonal(m, 100.0)                  # local execution is expensive ...
        m[env.servers, env.servers] = 0.01          # ... and the servers are fast
    it_good = [ES.EnvItem(ES.GREEDY, 0, *jobs), ES.EnvItem(ES.GREEDY, 1, *jobs), ES.EnvItem(ES.LOCAL, 0, *jobs)]
    net, items = ES.merge([(good, ES.item_arrays(good, [base, cyc], it_good)),
                           (broken, ES.item_arrays(broken, [base], [ES.EnvItem(ES.GREEDY, 0, *jobs)]))])
    got = ES.launch(net, items)
    want = env_oracle.env_step(net, items)
    st = got["status"]
    assert st[0] == ES._lib.ENV_OK and st[2] == ES._lib.ENV_OK
    assert st[1] == want["status"][1] == ES._lib.ENV_ROUTE_LOOP
    assert st[3] == want["status"][3] == ES._lib.ENV_NO_LINK
    for k in ("dst", "nhop", "delay_est", "delay_emp"):
        assert np.array_equal(got[k][:5], want[k][:5], equal_nan=True), k
        assert np.array_equal(got[k][10:15], want[k][10:15], equal_nan=True), k
    assert np.all(got["dst"][5:10] == -1) and np.all(np.isnan(got["delay_emp"][15:20]))


def test_invalid_arguments():
    import torch
    from multihop_offload_b200 import _lib
    from multihop_offload_b200 import env_step as ES
    lib = _lib.load_library()
    ctx = _lib.Context.get(0)
    rng = np.random.default_rng(1)
    env = SynthEnv(10, 1, rng)
    plan = ES.EnvPlan(env, env.hop)
    dev, keep = ES.upload_net(plan.net, "cuda:0")
    it = _lib.mho_env_items_t()
    out = _lib.mho_env_out_t()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.mho_env_step(None, C.byref(dev), C.byref(it), C.byref(out), st) == -1
    assert lib.mho_env_step(ctx.handle, None, C.byref(it), C.byref(out), st) == -1
    it.n_items = -1
    assert lib.mho_env_step(ctx.handle, C.byref(dev), C.byref(it), C.byref(out), st) == -1
    it.n_items = 0
    assert lib.mho_env_step(ctx.handle, C.byref(dev), C.byref(it), C.byref(out), st) == 0   # empty batch: nothing to do
    it.n_items = 1
    assert lib.mho_env_step(ctx.handle, C.byref(dev), C.byref(it), C.byref(out), st) == -1  # NULL item arrays / outputs
    t = torch.zeros(64, dtype=torch.float64, device="cuda:0")
    p = t.data_ptr()
    it = _lib.mho_env_items_t(1, 1, p, p, p, p, p, p, p, p, p)
    out = _lib.mho_env_out_t(p, p, p, p, p, None, 0, None, None, None, None, None, None, p)
    assert lib.mho_env_step(ctx.handle, C.byref(dev), C.byref(it), C.byref(out), st) == -1  # routes without offsets
    out = _lib.mho_env_out_t(p, p, p, p, None, None, 0, None, None, None, None, None, None, p)
    it.max_jobs = _lib.ENV_MAX_JOBS + 1
    assert lib.mho_env_step(ctx.handle, C.byref(dev), C.byref(it), C.byref(out), st) == -2  # MHO_ERR_TOO_LARGE
    assert ctx.launch_count() >= 0
    torch.cuda.synchronize()
