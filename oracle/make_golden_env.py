"""Writes tests/golden/env_cases.npz: the REFERENCE's own AdhocCloud.offloading() / local_compute() + run() (imported
from the read-only checkout through ref_env) on shipped networks and one synthetic one, recorded in the flat layout of
mho_env_step (multihop_offload_b200/env_step.py builds the inputs).

Cases: networks with N in {20, 50, 80, 110} from aco_data_ba_10, each with baseline, local and GNN shortest-path
matrices (the GNN delay matrices come from the oracle-backed agent of tests/fakes.py with the shipped BAT800 weights,
as in make_golden_agent.py) on four job sets: a sampled one, one with a high arrival scale (both congestion branches),
one job, and five jobs; the N = 110 network also once with link rates rounded to multiples of 10 (many argmin ties);
and a synthetic N = 200 BA network with 150 jobs.  Needs the reference checkout (MHO_REFERENCE_ROOT):

    python oracle/make_golden_env.py
"""
import os
import sys

import numpy as np
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import env_oracle  # noqa: E402
import fakes  # noqa: E402
import ref_env  # noqa: E402
from multihop_offload_b200 import env_step as ES  # noqa: E402


class _Patch:
    def setattr(self, obj, name, value):
        setattr(obj, name, value)


def baseline_sp(env, apsp):
    """AdHoc_test.py:129-136: the baseline shortest paths and the hop counts."""
    _, dlist, dproc = env.dmtx_baseline()
    dproc[dproc <= 0] = float(env.T)
    for (a, b), d in zip(env.link_list, dlist):
        env.graph_c[a][b]["delay"] = d if d > 0 else float(env.T)
    spb = apsp(env.graph_c, weight="delay")
    hop = apsp(env.graph_c, weight=None)
    np.fill_diagonal(spb, dproc)
    return spb, hop


def gnn_sp(agent, env, apsp):
    """gnn_offloading_agent.py:278-287: the GNN delay matrix -> shortest paths with its diagonal."""
    _, _, D = agent.forward(env.graph_expand(), env)
    for (a, b) in env.graph_c.edges:
        env.graph_c[a][b]["delay"] = D[a, b]
    s = apsp(env.graph_c, weight="delay")
    np.fill_diagonal(s, np.diagonal(D))
    return s


def reference_step(env, mode, spm, hop):
    """The reference's own calls for one item -> the outputs in the layout of one mho_env_step item."""
    if mode == ES.GREEDY:
        _, est = env.offloading(spm, hop)
    else:
        _, est = env.local_compute(np.diagonal(spm).copy())
    dl, dn, U = env.run()
    n = env.num_nodes
    routes = np.full((env.num_jobs, n + 1), -1, np.int32)
    for j, f in enumerate(env.flows):
        routes[j, :len(f.route)] = f.route
    return dict(dst=np.array([f.dst for f in env.flows], np.int32), nhop=np.array([f.nhop for f in env.flows], np.int32),
                delay_est=np.asarray(est, np.float64), delay_emp=np.nansum(dl, axis=0) + np.nansum(dn, axis=0),
                routes=routes.reshape(-1), delay_links=np.asarray(dl, np.float64).reshape(-1),
                delay_nodes=np.asarray(dn, np.float64).reshape(-1), unit=np.asarray(U, np.float64).reshape(-1))


def record(env, hop, sps, jobsets):
    """Runs every (job set, method) item through the reference; returns (net, items, outputs) flat arrays."""
    items, outs = [], []
    for jobs in jobsets:
        env.clear_all_jobs()
        for (s, r) in jobs:
            env.add_job(int(s), rate=float(r))
        src, rate, ul, dl = ES.jobs_of(env)
        for mode, k in ((ES.GREEDY, 0), (ES.LOCAL, 1), (ES.GREEDY, 2)):
            items.append(ES.EnvItem(mode, k, src, rate, ul, dl))
            outs.append(reference_step(env, mode, sps[k], hop))
    net = ES.network_arrays(env, hop)
    ia = ES.item_arrays(net, sps, items)
    rec = {k: np.concatenate([o[k] for o in outs]) for k in outs[0]}
    rec["status"] = np.zeros(len(items), np.int32)
    return net, ia, rec


def sampled_jobs(env, nodes_info, scale, num=None):
    mobile, = np.nonzero(nodes_info[:, 0] == 0)
    mobile = np.random.permutation(mobile)
    num = np.random.randint(int(0.3 * mobile.size), mobile.size) if num is None else num
    rates = np.random.uniform(0.1, 0.5, (num,))
    return [(mobile[i], scale * rates[i]) for i in range(num)]


def main():
    sys.argv = ["make_golden_env"]
    mod = fakes.install(_Patch())
    F = mod.FLAGS
    F.device, F.ref_src, F.T, F.K, F.fix_diag, F.learning_rate, F.training_set = "cpu", ref_env.REF_SRC, 1000, 1, False, 1e-4, "BAT800"
    AdhocCloud, apsp = ref_env.import_env()
    agent = mod.ACOAgent(F, 1000)
    agent.load(os.path.join(ROOT, "tests", "golden", "ckpt_BAT800"))
    data = os.path.join(ref_env.REF_ROOT, "data", "aco_data_ba_10")
    out, cases = {}, []
    names = ["aco_case_seed500_m2_n20_s4.mat", "aco_case_seed500_m2_n50_s6.mat", "aco_case_seed500_m2_n80_s11.mat",
             "aco_case_seed500_m2_n110_s18.mat", "aco_case_seed500_m2_n110_s18.mat"]
    for ci, name in enumerate(names):
        np.random.seed(100 + ci)
        env, nodes_info = ref_env.build_env(os.path.join(data, name))
        if ci == 4:   # coarse link rates: many equal path lengths
            env.link_rates = np.maximum(np.round(env.link_rates / 10.0) * 10.0, 10.0)
        spb, hop = baseline_sp(env, apsp)
        loc = np.zeros_like(spb)
        np.fill_diagonal(loc, env.dmtx_baseline()[2])
        jobsets = [sampled_jobs(env, nodes_info, 0.15), sampled_jobs(env, nodes_info, 1.5),
                   sampled_jobs(env, nodes_info, 0.15, 1), sampled_jobs(env, nodes_info, 0.15, 5)]
        env.clear_all_jobs()
        for (s, r) in jobsets[0]:
            env.add_job(int(s), rate=float(r))
        spg = gnn_sp(agent, env, apsp)
        cases.append(record(env, hop, [spb, loc, spg], jobsets))
    # synthetic N = 200 BA network, 150 jobs
    np.random.seed(7)
    env = AdhocCloud(200, 1000, 7, cf_radius=0.0, gtype="ba", pos="new")
    env.adj_c = sp.csr_matrix(env.adj_c)
    env.adj_i = sp.csr_matrix(env.adj_i)
    env.links_init(np.random.uniform(5, 40, env.num_links))
    roles = np.zeros(200, int)
    roles[np.random.choice(200, 30, replace=False)] = 1
    for v in range(200):
        if roles[v] == 1:
            env.add_server(v, float(np.random.uniform(5, 20)))
        else:
            env.proc_bws[v] = float(np.random.uniform(1, 3))
    nodes_info = np.stack([roles, env.proc_bws], 1)
    spb, hop = baseline_sp(env, apsp)
    loc = np.zeros_like(spb)
    np.fill_diagonal(loc, env.dmtx_baseline()[2])
    jobs = sampled_jobs(env, nodes_info, 0.15, 150)
    env.clear_all_jobs()
    for (s, r) in jobs:
        env.add_job(int(s), rate=float(r))
    spg = gnn_sp(agent, env, apsp)
    cases.append(record(env, hop, [spb, loc, spg], [jobs]))

    for ci, (net, ia, rec) in enumerate(cases):
        got = env_oracle.env_step(net, ia)
        for k, v in rec.items():
            assert np.array_equal(got[k], v, equal_nan=True), (ci, k)
        for k, v in net.items():
            out["c%d_net_%s" % (ci, k)] = np.asarray(v)
        for k, v in ia.items():
            out["c%d_items_%s" % (ci, k)] = np.asarray(v)
        for k, v in rec.items():
            out["c%d_out_%s" % (ci, k)] = np.asarray(v)
        L = int(net["max_links"])
        lam_hit = np.nanmax(rec["unit"]) if rec["unit"].size else 0
        print("case %d: n=%d L=%d items=%d jobs=%d max unit delay %.3g" % (ci, int(net["max_nodes"]), L, int(ia["n_items"]),
                                                                            int(ia["job_off"][-1]), lam_hit))
    out["n_cases"] = np.int32(len(cases))
    dst = os.path.join(ROOT, "tests", "golden", "env_cases.npz")
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    main()
