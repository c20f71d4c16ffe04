"""numpy restatement of mho_env_step (TEST INFRASTRUCTURE ONLY): AdhocCloud.offloading(sp, hop) with explore = 0 /
local_compute(dproc), then AdhocCloud.run() (src/offloading_v3.py:363-550) and the drivers' delay_emp, evaluated over
the flat arrays of the C-ABI (include/mho.h: mho_env_t, mho_env_items_t, mho_env_out_t; built by
multihop_offload_b200/env_step.py).  It uses the reference's own numpy operations in the same order, so its outputs
are bit-identical to the reference's; csrc/env_step.cu is checked against it.

    env_step(net, items, want) -> dict of flat outputs, the layout mho_env_step writes
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp_

OK, ROUTE_LOOP, NO_LINK, BAD_ITEM = 0, 1, 2, 3
GREEDY, LOCAL = 0, 1


def _network(net, g):
    n0, n1 = int(net["node_off"][g]), int(net["node_off"][g + 1])
    l0, l1 = int(net["link_off"][g]), int(net["link_off"][g + 1])
    s0, s1 = int(net["server_off"][g]), int(net["server_off"][g + 1])
    n, L = n1 - n0, l1 - l0
    arp = net["adj_rowptr"][n0:n1 + 1]
    crp = net["cf_rowptr"][l0:l1 + 1]
    lst = np.repeat(np.arange(L), np.diff(crp))   # column l of adj_i holds the neighbour list of link l
    adj_i = sp_.csr_matrix((np.ones(len(lst)), (net["cf_col"][crp[0]:crp[-1]], lst)), shape=(L, L))
    h0 = int(net["hop_off"][g])
    return dict(n=n, L=L, servers=list(int(x) for x in net["servers"][s0:s1]),
                nbrs=[(net["adj_col"][arp[v]:arp[v + 1]], net["adj_link"][arp[v]:arp[v + 1]]) for v in range(n)],
                link_rates=np.asarray(net["link_rates"][l0:l1], np.float64), cf_degs=np.asarray(net["cf_degs"][l0:l1], np.float64),
                proc_bws=np.asarray(net["proc_bws"][n0:n1], np.float64), adj_i=adj_i,
                hop=np.asarray(net["hop"][h0:h0 + n * n]).reshape(n, n), T=float(net["T"][g]))


def _item(N, mode, spm, src, rate, ul, dl):
    """-> (status, dst, nhop, est, routes, link_delay [L, J], node_delay [n, J], U [n, n])."""
    n, L, S = N["n"], N["L"], N["servers"]
    J = len(src)
    unit = np.diagonal(spm).copy()
    spz = spm.copy()
    np.fill_diagonal(spz, 0)
    dsts, nhops, ests, routes, hops = [], [], [], [], []
    for j in range(J):
        s = int(src[j])
        if mode == LOCAL:
            dsts.append(s); nhops.append(0); ests.append(np.max([unit[s] * ul[j], 1])); routes.append([s, s]); hops.append([])
            continue
        local = unit[s] * ul[j]
        uld = np.max([spz[s, S] * ul[j], N["hop"][s, S]], axis=0)
        dld = np.max([spz[S, s] * dl[j], N["hop"][S, s]], axis=0)
        pd = unit[S] * ul[j]
        proc = np.max([pd, np.ones_like(pd)], axis=0)
        srv = uld + dld + proc
        jidx = int(np.argmin(np.append(srv, local)))
        if jidx < len(S):
            dst = S[jidx]
            route, links, node = [s], [], s
            while node != dst:
                if len(route) - 1 >= n:
                    return (ROUTE_LOOP,)
                nbs, lks = N["nbrs"][node]
                if len(nbs) == 0:
                    return (NO_LINK,)
                k = int(np.argmin(spz[nbs, dst]))
                if lks[k] < 0 or lks[k] >= L:
                    return (NO_LINK,)
                node = int(nbs[k])
                route.append(node); links.append(int(lks[k]))
            dsts.append(dst); nhops.append(len(links)); ests.append(srv[jidx]); routes.append(route); hops.append(links)
        else:
            dsts.append(s); nhops.append(0); ests.append(local); routes.append([s, s]); hops.append([])
    # run()
    link_emp = np.full((L, J), np.nan)
    node_emp = np.full((n, J), np.nan)
    link_load = np.zeros_like(link_emp)
    srv_load = np.zeros((n,))
    for j in range(J):
        ul_rate, dl_rate = ul[j] * rate[j], dl[j] * rate[j]
        for lk in hops[j]:
            link_load[lk, j] += ul_rate + dl_rate
        srv_load[dsts[j]] += ul_rate
    lam = link_load.sum(axis=1)
    mu = N["link_rates"] / (N["cf_degs"] + 1)
    for _ in range(10):
        busy = np.clip(lam / mu, 0, 1.0)
        nb = busy * N["adj_i"]
        mu = N["link_rates"] * (1.0 / (1.0 + nb))
    U = np.full((n, n), np.nan)
    with np.errstate(divide="ignore", invalid="ignore"):
        for j in range(J):
            nh = float(nhops[j])
            n0 = int(src[j])
            for lk, n1 in zip(hops[j], routes[j][1:]):
                u = 1 / (mu[lk] - lam[lk])
                if mu[lk] - lam[lk] <= 0:
                    u = N["T"] * (lam[lk] / ((ul[j] + dl[j]) * mu[lk]))
                U[n0, n1] = U[n1, n0] = u
                link_emp[lk, j] = np.max([ul[j] * u, nh]) + np.max([dl[j] * u, nh])
                n0 = n1
            d = dsts[j]
            pb = N["proc_bws"][d]
            u = 1 / (pb - srv_load[d])
            if pb - srv_load[d] <= 0:
                u = N["T"] * (srv_load[d] / (ul[j] * pb))
            U[d, d] = u
            node_emp[d, j] = np.max([ul[j] * u, 1])
    return OK, dsts, nhops, ests, routes, link_emp, node_emp, U


def env_step(net, items, want=("routes", "delay_links", "delay_nodes", "unit")):
    """The outputs of mho_env_step for the flat arrays `net` (mho_env_t) and `items` (mho_env_items_t plus the output
    offsets and route_stride), as one dict of flat numpy arrays."""
    ni = int(items["n_items"])
    job_off = np.asarray(items["job_off"])
    nj = int(job_off[-1]) if ni else 0
    nets = {}
    out = dict(dst=np.zeros(nj, np.int32), nhop=np.zeros(nj, np.int32), delay_est=np.zeros(nj), delay_emp=np.zeros(nj),
               status=np.zeros(ni, np.int32))
    sizes = {}
    for i in range(ni):
        g = int(items["net"][i])
        if g not in nets:
            nets[g] = _network(net, g)
        N = nets[g]
        J = int(job_off[i + 1] - job_off[i])
        sizes["routes"] = max(sizes.get("routes", 0), int(items["routes_off"][i]) + J * int(items["route_stride"]))
        sizes["delay_links"] = max(sizes.get("delay_links", 0), int(items["links_off"][i]) + N["L"] * J)
        sizes["delay_nodes"] = max(sizes.get("delay_nodes", 0), int(items["nodes_off"][i]) + N["n"] * J)
        sizes["unit"] = max(sizes.get("unit", 0), int(items["unit_off"][i]) + N["n"] ** 2)
    for k in want:
        out[k] = np.full(sizes.get(k, 0), -1 if k == "routes" else np.nan, np.int32 if k == "routes" else np.float64)
    stride = int(items["route_stride"])
    for i in range(ni):
        g, mode = int(items["net"][i]), int(items["mode"][i])
        a, b = int(job_off[i]), int(job_off[i + 1])
        N = nets[g]
        n = N["n"]
        if mode not in (GREEDY, LOCAL) or b - a > int(items["max_jobs"]) or np.any((items["src"][a:b] < 0) | (items["src"][a:b] >= n)):
            out["status"][i] = BAD_ITEM
            continue
        o = int(items["sp_off"][i])
        spm = np.asarray(items["sp"][o:o + n * n], np.float64).reshape(n, n)
        r = _item(N, mode, spm, items["src"][a:b], items["rate"][a:b], items["ul"][a:b], items["dl"][a:b])
        out["status"][i] = r[0]
        if r[0] != OK:
            out["dst"][a:b] = -1; out["nhop"][a:b] = -1; out["delay_est"][a:b] = np.nan; out["delay_emp"][a:b] = np.nan
            continue
        _, dsts, nhops, ests, routes, le, ne, U = r
        out["dst"][a:b], out["nhop"][a:b], out["delay_est"][a:b] = dsts, nhops, ests
        out["delay_emp"][a:b] = np.nansum(le, axis=0) + np.nansum(ne, axis=0)
        J = b - a
        if "routes" in want:
            ro = int(items["routes_off"][i])
            for j, rt in enumerate(routes):
                out["routes"][ro + j * stride: ro + j * stride + len(rt)] = rt
        if "delay_links" in want:
            out["delay_links"][int(items["links_off"][i]):int(items["links_off"][i]) + N["L"] * J] = le.reshape(-1)
        if "delay_nodes" in want:
            out["delay_nodes"][int(items["nodes_off"][i]):int(items["nodes_off"][i]) + n * J] = ne.reshape(-1)
        if "unit" in want:
            out["unit"][int(items["unit_off"][i]):int(items["unit_off"][i]) + n * n] = U.reshape(-1)
    return out
