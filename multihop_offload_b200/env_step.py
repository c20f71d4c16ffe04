"""Batched environment step on the GPU (mho_env_step): the replacement of the reference's per-instance
``AdhocCloud.offloading(sp, hop)`` / ``local_compute(dproc)`` followed by ``AdhocCloud.run()`` (src/offloading_v3.py:363-550)
and the drivers' ``delay_emp = nansum(delay_links, 0) + nansum(delay_nodes, 0)``.

``EnvPlan`` flattens the instance-invariant constants of one network (an ``AdhocCloud``-shaped object: ``adj_c``,
``adj_i``, ``link_list``, ``servers``, ``link_rates``, ``cf_degs``, ``proc_bws``, ``T``) plus its hop-count matrix into
the arrays of ``mho_env_t``, once; ``EnvPlan.for_env`` caches it on the env.  ``step(sps, items)`` evaluates a batch of
items - each an ``EnvItem(mode, sp, src, rate, ul, dl)`` whose ``sp`` indexes the list of n x n shortest-path blocks - in
one launch and returns one ``EnvResult`` per item.  The results are bit-identical to the reference (see csrc/env_step.cu).
"""
from __future__ import annotations

import collections
import ctypes as C

import numpy as np
import scipy.sparse as sp_

from . import _lib

GREEDY, LOCAL = _lib.ENV_GREEDY, _lib.ENV_LOCAL
STATUS = {_lib.ENV_OK: "ok", _lib.ENV_ROUTE_LOOP: "route loop", _lib.ENV_NO_LINK: "no link", _lib.ENV_BAD_ITEM: "bad item"}

EnvItem = collections.namedtuple("EnvItem", "mode sp src rate ul dl")
EnvResult = collections.namedtuple("EnvResult", "status dst nhop delay_est delay_emp routes delay_links delay_nodes unit")


def jobs_of(env):
    """(src, rate, ul, dl) of env.jobs in job order."""
    jobs = env.jobs[:env.num_jobs] if env.jobs else []
    return (np.array([j.source_node for j in jobs], np.int32), np.array([j.arrival_rate for j in jobs], np.float64),
            np.array([j.ul_data for j in jobs], np.float64), np.array([j.dl_data for j in jobs], np.float64))


def network_arrays(env, hop):
    """The mho_env_t arrays of one network (a batch of one; LOCAL ids)."""
    n, L = int(env.num_nodes), int(env.num_links)
    lidx = {}
    for i, (a, b) in enumerate(env.link_list):
        lidx.setdefault((int(a), int(b)), i)
    A = sp_.csr_matrix(env.adj_c)
    rowptr, cols, links = [0], [], []
    for v in range(n):
        row = A.indices[A.indptr[v]:A.indptr[v + 1]]
        vals = A.data[A.indptr[v]:A.indptr[v + 1]]
        for u in row[vals != 0]:                  # np.nonzero(adj_c[v]): stored order, explicit zeros skipped
            u = int(u)
            cols.append(u)
            links.append(lidx.get((v, u), lidx.get((u, v), -1)))
        rowptr.append(len(cols))
    Ai = sp_.csc_matrix(env.adj_i)                # busy * adj_i reads the columns, neighbours ascending
    Ai.sum_duplicates()
    Ai.sort_indices()
    assert Ai.shape == (L, L) and np.all(Ai.data == 1), "the conflict graph must be binary"
    hop = np.ascontiguousarray(hop, dtype=np.float64)
    assert hop.shape == (n, n)
    return dict(
        n_nets=1, max_nodes=n, max_links=L,
        node_off=np.array([0, n], np.int32), link_off=np.array([0, L], np.int32),
        server_off=np.array([0, len(env.servers)], np.int32), servers=np.asarray(env.servers, np.int32).reshape(-1),
        adj_rowptr=np.asarray(rowptr, np.int32), adj_col=np.asarray(cols, np.int32), adj_link=np.asarray(links, np.int32),
        link_rates=np.asarray(env.link_rates, np.float64).reshape(-1), cf_degs=np.asarray(env.cf_degs, np.float64).reshape(-1),
        proc_bws=np.asarray(env.proc_bws, np.float64).reshape(-1),
        cf_rowptr=Ai.indptr.astype(np.int32), cf_col=Ai.indices.astype(np.int32),
        hop=hop.reshape(-1), hop_off=np.array([0], np.int64), T=np.array([float(env.T)], np.float64))


def item_arrays(net, sps, items):
    """The mho_env_items_t arrays plus the output offsets (every item on network 0 of `net`)."""
    n, L = int(net["max_nodes"]), int(net["max_links"])
    J = np.array([len(it.src) for it in items], np.int64)
    job_off = np.concatenate([[0], np.cumsum(J)]).astype(np.int32)
    cat = lambda k, dt: np.concatenate([np.asarray(getattr(it, k), dt).reshape(-1) for it in items]) if items else np.zeros(0, dt)  # noqa: E731
    spm = np.concatenate([np.ascontiguousarray(s, dtype=np.float64).reshape(-1) for s in sps]) if len(sps) else np.zeros(0)
    for s in sps:
        assert np.shape(s) == (n, n)
    ex = lambda a: np.concatenate([[0], np.cumsum(a)[:-1]]).astype(np.int64) if len(a) else np.zeros(0, np.int64)  # noqa: E731
    return dict(
        n_items=len(items), max_jobs=int(J.max()) if len(J) else 0,
        net=np.zeros(len(items), np.int32), mode=np.array([it.mode for it in items], np.int32), job_off=job_off,
        sp=spm, sp_off=np.array([int(it.sp) * n * n for it in items], np.int64),
        src=cat("src", np.int32), rate=cat("rate", np.float64), ul=cat("ul", np.float64), dl=cat("dl", np.float64),
        route_stride=n + 1, routes_off=ex(J * (n + 1)), links_off=ex(J * L), nodes_off=ex(J * n),
        unit_off=np.arange(len(items), dtype=np.int64) * n * n)


OUTPUTS = ("routes", "delay_links", "delay_nodes", "unit")


def merge(batches):
    """One (net, items) pair from several (network_arrays(), item_arrays()) pairs, each holding ONE network: networks,
    items and output offsets are concatenated so that the merged batch runs in one launch."""
    net, items = {}, {}
    nk = ("node_off", "link_off", "server_off")
    base = dict(node_off=0, link_off=0, server_off=0, adj=0, cf=0, hop=0, net=0, job=0, sp=0,
                routes_off=0, links_off=0, nodes_off=0, unit_off=0)
    parts = {k: [] for k in ("node_off", "link_off", "server_off", "servers", "adj_rowptr", "adj_col", "adj_link", "link_rates",
                             "cf_degs", "proc_bws", "cf_rowptr", "cf_col", "hop", "hop_off", "T", "net", "mode", "job_off", "sp",
                             "sp_off", "src", "rate", "ul", "dl", "routes_off", "links_off", "nodes_off", "unit_off")}
    stride = max(int(it["route_stride"]) for _, it in batches)
    for g, (N, I) in enumerate(batches):
        for k in nk:
            parts[k].append(N[k][:-1] + base[k])
        parts["adj_rowptr"].append(N["adj_rowptr"][:-1] + base["adj"])
        parts["cf_rowptr"].append(N["cf_rowptr"][:-1] + base["cf"])
        parts["hop_off"].append(N["hop_off"] + base["hop"])
        for k in ("servers", "adj_col", "adj_link", "link_rates", "cf_degs", "proc_bws", "cf_col", "hop", "T"):
            parts[k].append(N[k])
        parts["net"].append(I["net"] + base["net"])
        parts["job_off"].append(I["job_off"][:-1] + base["job"])
        parts["sp_off"].append(I["sp_off"] + base["sp"])
        for k in ("mode", "sp", "src", "rate", "ul", "dl"):
            parts[k].append(I[k])
        nj = int(I["job_off"][-1])
        J = np.diff(I["job_off"]).astype(np.int64)
        parts["routes_off"].append(np.concatenate([[0], np.cumsum(J * stride)[:-1]]).astype(np.int64) + base["routes_off"])
        for k in ("links_off", "nodes_off", "unit_off"):
            parts[k].append(I[k] + base[k])
        n, L = int(N["node_off"][-1]), int(N["link_off"][-1])
        for k in nk:
            base[k] += int(N[k][-1])
        base["adj"] += int(N["adj_rowptr"][-1]); base["cf"] += int(N["cf_rowptr"][-1]); base["hop"] += N["hop"].size
        base["net"] += int(N["n_nets"]); base["job"] += nj; base["sp"] += I["sp"].size
        base["routes_off"] += nj * stride; base["links_off"] += int(np.sum(J * L)) if I["n_items"] else 0
        base["nodes_off"] += int(np.sum(J * n)) if I["n_items"] else 0
        base["unit_off"] += int(I["n_items"]) * n * n
    cat = lambda k, dt: np.concatenate(parts[k]).astype(dt)  # noqa: E731
    i32 = ("node_off", "link_off", "server_off", "servers", "adj_rowptr", "adj_col", "adj_link", "cf_rowptr", "cf_col",
           "net", "mode", "job_off", "src")
    for k in parts:
        dt = np.int32 if k in i32 else (np.int64 if k.endswith("_off") else np.float64)
        (items if k in ("net", "mode", "job_off", "sp", "sp_off", "src", "rate", "ul", "dl", "routes_off", "links_off",
                        "nodes_off", "unit_off") else net)[k] = cat(k, dt)
    for k, tot in (("node_off", "node_off"), ("link_off", "link_off"), ("server_off", "server_off"), ("adj_rowptr", "adj"),
                   ("cf_rowptr", "cf")):
        net[k] = np.append(net[k], base[tot]).astype(np.int32)
    items["job_off"] = np.append(items["job_off"], base["job"]).astype(np.int32)
    net.update(n_nets=base["net"], max_nodes=max(int(N["max_nodes"]) for N, _ in batches),
               max_links=max(int(N["max_links"]) for N, _ in batches))
    items.update(n_items=int(sum(int(I["n_items"]) for _, I in batches)), max_jobs=max(int(I["max_jobs"]) for _, I in batches),
                 route_stride=stride)
    return net, items


def output_sizes(net, items):
    """Element counts of the flat outputs of a batch."""
    ni, nj = int(items["n_items"]), int(items["job_off"][-1])
    noff, loff = np.asarray(net["node_off"]), np.asarray(net["link_off"])
    g = np.asarray(items["net"], np.int64)
    J = np.diff(items["job_off"]).astype(np.int64)
    n, L = (noff[g + 1] - noff[g]).astype(np.int64), (loff[g + 1] - loff[g]).astype(np.int64)
    end = lambda off, size: int(np.max(np.asarray(off) + size)) if ni else 0  # noqa: E731
    return dict(routes=nj * int(items["route_stride"]), delay_links=end(items["links_off"], J * L),
                delay_nodes=end(items["nodes_off"], J * n), unit=end(items["unit_off"], n * n), jobs=nj, items=ni)


def bind(net, items, want=OUTPUTS, device="cuda:0", ctx=None, dev_net=None):
    """Uploads the item arrays and allocates the outputs of one batch; returns (call, outputs, sizes) where call()
    enqueues one mho_env_step launch on the current stream (the arrays stay alive with `call`)."""
    import torch
    ctx = ctx if ctx is not None else _lib.Context.get(torch.device(device).index or 0)
    if dev_net is None:
        dev_net = upload_net(net, device)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)  # noqa: E731
    d = {k: up(items[k]) for k in ("net", "mode", "job_off", "sp", "sp_off", "src", "rate", "ul", "dl",
                                   "routes_off", "links_off", "nodes_off", "unit_off")}
    sz = output_sizes(net, items)
    ni, nj = sz["items"], sz["jobs"]
    o = dict(dst=torch.empty(nj, dtype=torch.int32, device=device), nhop=torch.empty(nj, dtype=torch.int32, device=device),
             delay_est=torch.empty(nj, dtype=torch.float64, device=device),
             delay_emp=torch.empty(nj, dtype=torch.float64, device=device),
             status=torch.empty(ni, dtype=torch.int32, device=device))
    for k in want:
        o[k] = torch.empty(max(sz[k], 1), dtype=torch.int32 if k == "routes" else torch.float64, device=device)
    p = lambda k: o[k].data_ptr() if k in o else None  # noqa: E731
    q = lambda k: d[k].data_ptr() if d[k].numel() else None  # noqa: E731
    it = _lib.mho_env_items_t(ni, int(items["max_jobs"]), q("net"), q("mode"), q("job_off"), q("sp"), q("sp_off"),
                              q("src"), q("rate"), q("ul"), q("dl"))
    out = _lib.mho_env_out_t(p("dst"), p("nhop"), p("delay_est"), p("delay_emp"), p("routes"), q("routes_off"),
                             int(items["route_stride"]), p("delay_links"), q("links_off"), p("delay_nodes"),
                             q("nodes_off"), p("unit"), q("unit_off"), p("status"))

    def call():
        st = C.c_void_p(torch.cuda.current_stream(torch.device(device)).cuda_stream)
        _lib.check(ctx.lib.mho_env_step(ctx.handle, C.byref(dev_net[0]), C.byref(it), C.byref(out), st), "mho_env_step")
    call.keep = (d, dev_net)
    return call, o, sz


def launch(net, items, want=OUTPUTS, device="cuda:0", ctx=None, dev_net=None):
    """One mho_env_step launch over flat arrays (net: mho_env_t fields, items: mho_env_items_t fields plus the output
    offsets); returns the outputs as a dict of flat numpy arrays.  dev_net: a cached (mho_env_t, tensors) upload."""
    call, o, sz = bind(net, items, want, device, ctx, dev_net)
    call()
    res = {k: v.cpu().numpy() for k, v in o.items()}
    for k in want:
        res[k] = res[k][:sz[k]]
    return res


def upload_net(net, device):
    import torch
    keep = {k: torch.from_numpy(np.ascontiguousarray(v)).to(device) for k, v in net.items() if isinstance(v, np.ndarray)}
    ptr = lambda k: keep[k].data_ptr() if keep[k].numel() else None  # noqa: E731
    s = _lib.mho_env_t(int(net["n_nets"]), int(net["max_nodes"]), int(net["max_links"]),
                       *[ptr(k) for k in ("node_off", "link_off", "server_off", "servers", "adj_rowptr", "adj_col", "adj_link",
                                          "link_rates", "cf_degs", "proc_bws", "cf_rowptr", "cf_col", "hop", "hop_off", "T")])
    return s, keep


def device_run(plan, items, want):
    if plan._dev is None:
        plan._dev = upload_net(plan.net, plan.device)
    return launch(plan.net, items, want, plan.device, plan.ctx, plan._dev)


run = device_run   # the launch step() uses: (plan, item arrays, wanted optional outputs) -> flat outputs


class EnvPlan(object):
    def __init__(self, env, hop, device="cuda:0", ctx=None):
        self.net = network_arrays(env, hop)
        self.device = device
        self._ctx = ctx
        self._dev = None

    @classmethod
    def for_env(cls, env, hop, device="cuda:0", ctx=None):
        """The plan of `env`, built once and cached on the env object (the constants are instance-invariant)."""
        plan = env.__dict__.get("_mho_env_plan")
        if plan is None:
            plan = cls(env, hop, device, ctx)
            env.__dict__["_mho_env_plan"] = plan
        return plan

    @property
    def ctx(self):
        if self._ctx is None:
            import torch
            self._ctx = _lib.Context.get(torch.device(self.device).index or 0)
        return self._ctx

    def step(self, sps, items, want=OUTPUTS):
        """sps: list of n x n shortest-path blocks (diagonal = server unit delays); items: list of EnvItem.
        Returns one EnvResult per item (numpy; optional outputs not in `want` are None)."""
        want = tuple(k for k in OUTPUTS if k in want)
        ia = item_arrays(self.net, sps, items)
        o = run(self, ia, want)
        n, L = int(self.net["max_nodes"]), int(self.net["max_links"])
        res = []
        for i in range(len(items)):
            a, b = int(ia["job_off"][i]), int(ia["job_off"][i + 1])
            J = b - a
            get = lambda k, off, shape: o[k][off:off + int(np.prod(shape))].reshape(shape) if k in want else None  # noqa: E731
            res.append(EnvResult(int(o["status"][i]), o["dst"][a:b], o["nhop"][a:b], o["delay_est"][a:b], o["delay_emp"][a:b],
                                 get("routes", int(ia["routes_off"][i]), (J, n + 1)),
                                 get("delay_links", int(ia["links_off"][i]), (L, J)),
                                 get("delay_nodes", int(ia["nodes_off"][i]), (n, J)),
                                 get("unit", int(ia["unit_off"][i]), (n, n))))
        return res
