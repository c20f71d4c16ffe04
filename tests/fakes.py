"""Test doubles (tests/ only): an oracle-backed stand-in for ChebNet / KerasAdamReplay so that the HOST
logic of the agent and drivers can be exercised on the CPU box against the reference's real simulator.
The product never imports this; on a GPU the real libmho path is tested in test_agent_gpu.py."""
import sys
import types

import numpy as np
import scipy.sparse as sp
import torch

import chebnet_oracle as O


class OracleChebNet:
    def __init__(self, specs, device="cpu", params=None, seed=0):
        self.specs = list(specs)
        self.device = "cpu"
        self.n_params = int(sum(s.n_params for s in self.specs))
        rng = np.random.default_rng(seed)
        ws = O.glorot_weights([self.specs[0].f_in] + [s.f_out for s in self.specs], self.specs[0].K, rng)
        self.params = torch.zeros(self.n_params, dtype=torch.float64)
        self.set_weights(ws)

    def set_flat(self, flat):
        self.params.copy_(torch.as_tensor(np.asarray(flat, dtype=np.float64).ravel()))

    def get_flat(self):
        return self.params.numpy().copy()

    def set_weights(self, ws):
        self.set_flat(O.flatten_params(ws))

    def get_weights(self):
        return O.unflatten_params(self.get_flat(), [(s.K, s.f_in, s.f_out) for s in self.specs])

    def weights_changed(self):
        pass

    def _mats(self, batch):
        out = []
        for a, b in zip(batch.graph_off[:-1], batch.graph_off[1:]):
            z0, z1 = batch.rowptr[a], batch.rowptr[b]
            vals = np.ones(z1 - z0) if batch.vals is None else batch.vals[z0:z1]
            out.append(sp.csr_matrix((vals, batch.colidx[z0:z1] - a, batch.rowptr[a:b + 1] - z0), shape=(b - a, b - a)))
        return out

    def forward(self, batch, X, save=False, out=None, per_graph_tiles=False):
        ws, acts = self.get_weights(), [s.act for s in self.specs]
        Xn = X.numpy().astype(np.float64)
        ys, caches, o = [], [], 0
        for A in self._mats(batch):
            n = A.shape[0]
            y, c = O.cheb_stack_forward(A, Xn[o:o + n], ws, acts, self.specs[0].slope, return_cache=True)
            ys.append(y); caches.append(c); o += n
        Y = torch.as_tensor(np.concatenate(ys, 0))
        return (Y, caches) if save else Y

    def backward(self, batch, X, Y, saved, dY, need_dx=False, need_sum=True):
        ws = self.get_weights()
        g, o = [], 0
        dYn = dY.numpy().astype(np.float64)
        for A, cache in zip(self._mats(batch), saved):
            n = A.shape[0]
            grads, _ = O.cheb_stack_backward(A, ws, cache, dYn[o:o + n], self.specs[0].slope)
            g.append(O.flatten_params(grads)); o += n
        gpg = torch.as_tensor(np.stack(g))
        return gpg, (gpg.sum(0) if need_sum else None), None


class OracleAdam:
    def __init__(self, net, learning_rate=1e-4, clipnorm=1.0, max_norm=1.0, decay_rate=1.0, decay_steps=100, **kw):
        self.net = net
        shapes = []
        for s in net.specs:
            shapes += [(s.K, s.f_in, s.f_out), (s.f_out,)]
        self.shapes = shapes
        self.opt = O.KerasAdam(shapes, lr=learning_rate, clipnorm=clipnorm, max_norm=max_norm, decay_rate=decay_rate,
                               decay_steps=decay_steps)
        self.iterations = 0
        self.master = net.params

    def set_master(self, flat):
        self.net.set_flat(flat)

    def get_master(self):
        return self.net.get_flat()

    def apply(self, grads):
        if grads.dim() == 1:
            grads = grads.unsqueeze(0)
        for g in grads.numpy():
            flat = self.net.get_flat()
            ps, gs, o = [], [], 0
            for sh in self.shapes:
                n = int(np.prod(sh)); ps.append(flat[o:o + n].reshape(sh)); gs.append(g[o:o + n].reshape(sh)); o += n
            self.opt.apply(ps, gs)
            self.net.set_flat(np.concatenate([p.ravel() for p in ps]))
            self.iterations += 1


class FakeGraphBatch:
    """GraphBatch without libmho's planner (CPU tests of host logic only)."""

    def __init__(self, graph_off, rowptr, colidx, vals):
        self.graph_off, self.rowptr, self.colidx, self.vals = graph_off, rowptr, colidx, vals
        self.n_graphs = len(graph_off) - 1
        self.total_nodes = int(graph_off[-1])

    @classmethod
    def from_scipy(cls, mats, device=None, **kw):
        g, rp, ci, va = O.concat_batch(mats)
        return cls(g, rp, ci, va)


def install(monkeypatch):
    """Swap the libmho-backed classes inside the agent module for the oracle-backed doubles."""
    import multihop_offload_b200.gnn_offloading_agent as mod
    monkeypatch.setattr(mod, "ChebNet", OracleChebNet)
    monkeypatch.setattr(mod, "KerasAdamReplay", OracleAdam)
    monkeypatch.setattr(mod, "GraphBatch", FakeGraphBatch)
    return mod


def install_apsp(monkeypatch):
    """A ``util`` module whose all_pairs_shortest_paths (the reference's src/util.py:101-110, which the agent imports on the
    CPU) is the oracle's Dijkstra, pinned bit for bit against the reference's own outputs in test_apsp.py."""
    import apsp_oracle

    def all_pairs_shortest_paths(graph, weight=None):
        edges = list(graph.edges)
        w = None if weight is None else [graph[a][b][weight] for a, b in edges]
        return apsp_oracle.apsp_lengths(graph.number_of_nodes(), edges, w)

    mod = types.ModuleType("util")
    mod.all_pairs_shortest_paths = all_pairs_shortest_paths
    monkeypatch.setitem(sys.modules, "util", mod)


class RecordedStep:
    """One forward_backward() step recorded against the reference's simulator (tests/golden/agent_case_n20.npz, written by
    oracle/make_golden_agent.py): `obj` and `env` carry the fields the agent reads; env.offloading() checks that the agent
    hands over the shortest-path matrices of the recording and sets the routes the simulator chose from them, env.run()
    returns the recorded delays."""

    def __init__(self, z):
        import networkx as nx
        self.z = z
        n_ext = z["X"].shape[0]
        A = sp.csr_matrix((z["gi_vals"], z["gi_colidx"], z["gi_rowptr"]), shape=(n_ext, n_ext))
        self.adj, self.X = A, z["X"]
        obj = types.SimpleNamespace(gi_ext=nx.from_scipy_sparse_array(A), num_edges_ext=n_ext,
                                    edge_self_loop=z["X"][:, 0], edge_rate_ext=z["X"][:, 1], jobs_arrivals=z["X"][:, 2],
                                    edge_as_server=z["X"][:, 3], maps_ol_el=z["maps_ol_el"], maps_on_el=z["maps_on_el"],
                                    link_list_ext=[tuple(int(v) for v in e) for e in z["link_list_ext"]])
        env = types.SimpleNamespace()
        env.num_nodes, env.T, env.num_links = int(z["num_nodes"]), int(z["T"]), int(z["num_links"])
        env.link_rates, env.cf_degs, env.proc_bws, env.link_matrix = z["link_rates"], z["cf_degs"], z["proc_bws"], z["link_matrix"]
        L = env.num_links
        env.adj_i = sp.csr_matrix((z["adj_i_vals"], z["adj_i_colidx"], z["adj_i_rowptr"]), shape=(L, L))
        g = nx.Graph()
        g.add_nodes_from(range(env.num_nodes))
        g.add_edges_from([tuple(int(v) for v in e) for e in z["edges"]])
        env.graph_c = g
        env.num_jobs = len(z["job_source"])
        env.jobs = [types.SimpleNamespace(source_node=int(s), arrival_rate=float(r), ul_data=float(u), dl_data=float(d))
                    for s, r, u, d in zip(z["job_source"], z["job_rate"], z["job_ul"], z["job_dl"])]
        env.flows = []
        env.offloading, env.run = self.offloading, self.run
        self.obj, self.env = obj, env

    def offloading(self, sp_gnn, sp_hop, explore=0.0):
        z = self.z
        np.testing.assert_allclose(sp_gnn, z["sp_gnn"], rtol=1e-9, atol=0)
        np.testing.assert_array_equal(sp_hop, z["sp_hop"])
        assert explore == float(z["explore"])
        off = z["flow_route_off"]
        self.env.flows = [types.SimpleNamespace(dst=int(d), route=[int(v) for v in z["flow_route"][a:b]])
                          for d, a, b in zip(z["flow_dst"], off[:-1], off[1:])]
        return None, None

    def run(self):
        z = self.z
        return z["delay_links"].copy(), z["delay_nodes"].copy(), z["delay_unit"].copy()
