"""Shared pieces of the AdHoc_test / AdHoc_train drivers (restated from the reference's module-level
scripts src/AdHoc_test.py:82-178 and src/AdHoc_train.py:81-207).  The network simulator itself
(``offloading_v3.AdhocCloud``, ``util.all_pairs_shortest_paths``) is the reference's CPU code, out of
scope here and imported from the user's reference checkout (``--ref_src`` / ``MHO_REFERENCE_SRC``)."""
from __future__ import annotations

import copy
import os
import sys
import time
import types

import numpy as np
import scipy.io as sio
import scipy.sparse as sp


def import_reference_env(ref_src):
    """(AdhocCloud, all_pairs_shortest_paths) from the reference's src/ directory."""
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:  # plotting is never used by the drivers
                sys.modules[name] = types.ModuleType(name)
    if ref_src and ref_src not in sys.path:
        sys.path.insert(0, ref_src)
    try:
        from offloading_v3 import AdhocCloud
        from util import all_pairs_shortest_paths
    except ImportError as e:
        raise ImportError("the drivers need the reference's environment simulator: pass --ref_src=<reference>/src "
                          "or set MHO_REFERENCE_SRC (%s)" % e)
    return AdhocCloud, all_pairs_shortest_paths


def load_case(AdhocCloud, filepath, T):
    """AdHoc_test.py:84-109: environment of one shipped .mat network."""
    mat = sio.loadmat(filepath)
    net_cfg = mat['network'][0, 0]
    link_rates = mat["link_rate"].flatten()
    nodes_info = mat["nodes_info"]
    seed = int(net_cfg['seed'].flatten()[0])
    num_nodes = int(net_cfg['num_nodes'].flatten()[0])
    m = net_cfg['m'].flatten()[0]
    env = AdhocCloud(num_nodes, T, seed, cf_radius=0.0, gtype=filepath, trace=True)
    # networkx >= 3 returns sparse ARRAYS; offloading_v3.py:448,:503 rely on matrix semantics
    env.adj_c = sp.csr_matrix(env.adj_c)
    env.adj_i = sp.csr_matrix(env.adj_i)
    env.links_init(link_rates)
    for nidx in range(num_nodes):
        if nodes_info[nidx, 0] == 2:
            env.add_relay(nidx)
        elif nodes_info[nidx, 0] == 1:
            env.add_server(nidx, float(nodes_info[nidx, 1]))
        elif nodes_info[nidx, 0] == 0:
            env.proc_bws[nidx] = nodes_info[nidx, 1]
    return env, nodes_info, seed, num_nodes, m


def sample_jobs(env, nodes_info, arrival_scale):
    """AdHoc_test.py:113-121."""
    env.clear_all_jobs()
    mobile_nodes, = np.nonzero(nodes_info[:, 0] == 0)
    num_mobile = mobile_nodes.size
    mobile_nodes = np.random.permutation(mobile_nodes)
    num_jobs = np.random.randint(int(0.3 * num_mobile), num_mobile)
    arrival_rates = np.random.uniform(0.1, 0.5, (num_jobs,))
    for idx in range(num_jobs):
        env.add_job(mobile_nodes[idx], rate=arrival_scale * arrival_rates[idx])
    return num_jobs


def lookahead_instances(env, nodes_info, arrival_scale, n_instances, agent, apsp):
    """SURVEY 8f #3: job sets and GNN inputs of the next `n_instances` instances of a network WITHOUT disturbing the driver's
    random stream: the generator state is saved, the instances are sampled exactly as the per-instance loop will sample
    them (sample_jobs, then the draws each instance consumes before the next one: one np.random.uniform per job in each
    of the two env.offloading() calls - baseline and GNN, offloading_v3.py:416 - whose VALUES are irrelevant at
    explore = 0), their features are collected, the state is restored.  One GNN / head / shortest-path launch each
    for all of them (ACOAgent.forward_instances)."""
    state = np.random.get_state()
    feats, obj0, jobsets = [], None, []
    for _ in range(n_instances):
        num_jobs = sample_jobs(env, nodes_info, arrival_scale)
        obj = env.graph_expand()
        obj0 = obj0 or obj
        feats.append(agent.instance_features(obj))
        jobsets.append(_jobs_of(env))
        np.random.uniform(0, 1, size=2 * num_jobs)
    np.random.set_state(state)
    pre = agent.forward_instances(obj0, env, feats, apsp)
    env.__dict__.pop("_mho_env_steps", None)
    if use_device_env_step(agent):
        env_step_instances(env, agent, apsp, jobsets, pre)
    return pre


def use_device_env_step(agent):
    """On a CUDA device the environment step of the looked-ahead instances (baseline, local and GNN of each) runs as one
    mho_env_step launch; elsewhere the reference's simulator runs instance by instance."""
    return bool(getattr(agent, "_on_gpu", lambda: False)())


def _jobs_of(env):
    from .env_step import jobs_of
    return jobs_of(env)


def _jobs_key(jobs):
    return b"".join(np.ascontiguousarray(a).tobytes() for a in jobs)


def baseline_paths(env, agent, apsp):
    """AdHoc_test.py:129-136: the baseline's shortest-path matrix (link delays 1 / rate, processing delays 1 / proc_bw on
    the diagonal) and the hop counts.  Both depend on the network only, not on the job set."""
    dmtx_bl, dlist_bl, dproc_bl = env.dmtx_baseline()
    dproc_bl[dproc_bl <= 0] = float(env.T)
    for link, delay in zip(env.link_list, dlist_bl):
        src, dst = link
        env.graph_c[src][dst]["delay"] = delay if delay > 0 else float(env.T)
    if getattr(agent, "_on_gpu", lambda: False)():
        # same shortest-path matrices from mho_apsp (bit-identical to the reference's Dijkstra, SURVEY 8f #2)
        M = np.zeros((env.num_nodes, env.num_nodes))
        for (src, dst) in env.graph_c.edges:
            M[src, dst] = M[dst, src] = env.graph_c[src][dst]["delay"]
        sp_baseline, sp_hop = agent._shortest_paths(env, M, apsp)
    else:
        sp_baseline = apsp(env.graph_c, weight="delay")
        sp_hop = apsp(env.graph_c, weight=None)
    np.fill_diagonal(sp_baseline, dproc_bl)
    return sp_baseline, sp_hop


def env_step_instances(env, agent, apsp, jobsets, pre):
    """The environment side of the baseline, local and GNN methods of the looked-ahead instances of one network in ONE
    mho_env_step launch: offloading() / local_compute() + run() of every (instance, method) item, bit-identical to the
    reference.  jobsets: (src, rate, ul, dl) of each instance; pre: lookahead_instances()'s GNN shortest paths of the same
    instances.  The resulting delay_emp are kept on the env under (method, job set); run_method() returns them when the
    driver reaches that instance and method."""
    from .env_step import GREEDY, LOCAL, EnvItem, EnvPlan
    sp_bl, sp_hop = baseline_paths(env, agent, apsp)
    loc = np.zeros_like(sp_bl)
    np.fill_diagonal(loc, env.dmtx_baseline()[2])   # local_compute's dproc (AdHoc_test.py:140-141)
    sps, items = [sp_bl, loc], []
    for jobs, (delay_mtx_np, sp_gnn, _) in zip(jobsets, pre):
        sp_gnn = np.array(sp_gnn, copy=True)
        np.fill_diagonal(sp_gnn, np.diagonal(delay_mtx_np))
        sps.append(sp_gnn)
        items += [EnvItem(GREEDY, 0, *jobs), EnvItem(LOCAL, 1, *jobs), EnvItem(GREEDY, len(sps) - 1, *jobs)]
    plan = EnvPlan.for_env(env, sp_hop, device=getattr(agent, "device", "cuda:0"), ctx=getattr(getattr(agent, "net", None), "ctx", None))
    res = plan.step(sps, items, want=())
    bad = [i for i, r in enumerate(res) if r.status != 0]
    if bad:
        raise RuntimeError("mho_env_step: item %d of %s has status %d" % (bad[0], env.case_name, res[bad[0]].status))
    steps = {}
    for i, jobs in enumerate(jobsets):
        for k, method in enumerate(("baseline", "local", "GNN-pre")):
            steps[(method, _jobs_key(jobs))] = res[3 * i + k].delay_emp
    env.__dict__["_mho_env_steps"] = steps


def _precomputed_step(method, env, explore):
    """delay_emp of env_step_instances() for this method and the env's current job set, or None.  A hit consumes the
    draws the reference's offloading() would have consumed (one np.random.uniform per job, offloading_v3.py:416)."""
    steps = env.__dict__.get("_mho_env_steps")
    if not steps or explore != 0.0:
        return None
    emp = steps.pop((method, _jobs_key(_jobs_of(env))), None)
    if emp is not None and method != "local":
        np.random.uniform(0, 1, size=len(emp))
    return emp


def run_method(method, env, agent, apsp, explore=0.0, pre=None):
    """One of the methods of AdHoc_test.py:125-153 / AdHoc_train.py:124-157 -> (delay_emp, extras).
    pre: precomputed (delay matrix, shortest paths) of this instance from lookahead_instances (method "GNN-pre")."""
    extras = {}
    emp = _precomputed_step(method, env, explore)
    if emp is not None:
        return np.array(emp, copy=True), extras
    if method == "baseline":
        sp_baseline, sp_hop = baseline_paths(env, agent, apsp)
        env.offloading(sp_baseline, sp_hop)
        delay_links, delay_nodes, _ = env.run()
    elif method == "local":
        dmtx_bl, dlist_bl, dproc_bl = env.dmtx_baseline()
        env.local_compute(dproc_bl)
        delay_links, delay_nodes, _ = env.run()
    elif method == "GNN":
        obj = env.graph_expand()
        (_, delay_links, delay_nodes, _, _, loss_fn, loss_mse) = agent.forward_backward(obj, env, explore)
        extras = dict(loss_fn=loss_fn, loss_mse=loss_mse)
    elif method == "GNN-test":
        obj = env.graph_expand()
        delay_links, delay_nodes, _ = agent.forward_env(obj, env)
    elif method == "GNN-pre":
        delay_links, delay_nodes, _ = agent.env_step_from(pre, env)
    else:
        raise ValueError(method)
    delay_emp = np.nansum(delay_links, axis=0) + np.nansum(delay_nodes, axis=0)
    return delay_emp, extras


def result_row(base, method_key, method, runtime, delay_emp, delay_dict, env, num_jobs):
    """Row schema of AdHoc_test.py:160-176 ("Algo") / AdHoc_train.py:163-180 ("method")."""
    row = dict(base)
    row.update({
        "num_servers": len(env.servers), "num_relays": len(env.relays),
        "num_mobile": base["num_nodes"] - len(env.servers) - len(env.relays), "num_jobs": num_jobs,
        method_key: method, "runtime": runtime,
        "gap_2_bl": np.nanmean(delay_dict[method] - delay_dict["baseline"]),
        "gnn_bl_ratio": np.nanmean(delay_dict[method] / delay_dict["baseline"]),
        "tau": np.nanmean(delay_emp),
        "congest_jobs": np.count_nonzero(delay_emp > float(env.T)),
    })
    return row
