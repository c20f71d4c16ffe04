"""Writes tests/golden/agent_case_n20.npz: one ACOAgent.forward_backward() step against the REFERENCE's own simulator
(offloading_v3.AdhocCloud, imported from the read-only checkout), recorded at the agent / simulator boundary.

Stored: the fields of the expanded graph and of the environment the agent reads, the shortest-path matrices the agent
handed to env.offloading(), and what the simulator produced from them (routes of the jobs, env.run() delays).  The
GNN is the oracle-backed test double of tests/fakes.py, so the recording does not depend on libmho.
tests/test_agent_host.py replays it without the reference.  Needs the reference checkout (MHO_REFERENCE_ROOT):

    python oracle/make_golden_agent.py
"""
import os
import sys

import numpy as np
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import fakes  # noqa: E402
import ref_env  # noqa: E402


class _Patch:
    def setattr(self, obj, name, value):
        setattr(obj, name, value)


def csr_parts(A):
    A = sp.csr_matrix(A)
    A.sort_indices()
    return A.indptr.astype(np.int32), A.indices.astype(np.int32), A.data.astype(np.float64)


def main():
    sys.argv = ["make_golden_agent"]
    mod = fakes.install(_Patch())
    F = mod.FLAGS
    F.device, F.ref_src, F.T, F.K, F.fix_diag, F.learning_rate, F.training_set = "cpu", ref_env.REF_SRC, 1000, 1, False, 1e-4, "BAT800"
    AdhocCloud, _ = ref_env.import_env()
    from multihop_offload_b200.drivers_common import load_case, sample_jobs
    agent = mod.ACOAgent(F, 1000)
    agent.load(os.path.join(ROOT, "tests", "golden", "ckpt_BAT800"))
    fn = os.path.join(ref_env.REF_ROOT, "data", "aco_data_ba_10", "aco_case_seed500_m2_n20_s4.mat")
    env, nodes_info, seed, n, m = load_case(AdhocCloud, fn, 1000)
    np.random.seed(3)
    sample_jobs(env, nodes_info, 0.15)
    obj = env.graph_expand()
    adj, X = ref_env.gnn_inputs(obj)
    out = {}
    rp, ci, va = csr_parts(adj)
    out.update(gi_rowptr=rp, gi_colidx=ci, gi_vals=va, X=X, maps_ol_el=np.asarray(obj.maps_ol_el, np.int64),
               maps_on_el=np.asarray(obj.maps_on_el, np.int64), link_list_ext=np.asarray(obj.link_list_ext, np.int64))
    rp, ci, va = csr_parts(env.adj_i)
    out.update(adj_i_rowptr=rp, adj_i_colidx=ci, adj_i_vals=va, num_nodes=np.int64(env.num_nodes), T=np.int64(env.T),
               num_links=np.int64(env.num_links), link_rates=np.asarray(env.link_rates, np.float64),
               cf_degs=np.asarray(env.cf_degs), proc_bws=np.asarray(env.proc_bws, np.float64),
               link_matrix=np.asarray(env.link_matrix, np.int64), edges=np.asarray(list(env.graph_c.edges), np.int64))
    offloading, run = env.offloading, env.run

    def rec_offloading(sp_gnn, sp_hop, explore=0.0):
        out.update(sp_gnn=np.array(sp_gnn, copy=True), sp_hop=np.array(sp_hop, copy=True), explore=np.float64(explore))
        return offloading(sp_gnn, sp_hop, explore)

    def rec_run():
        dl, dn, du = run()
        out.update(delay_links=np.array(dl, copy=True), delay_nodes=np.array(dn, copy=True), delay_unit=np.array(du, copy=True))
        return dl, dn, du

    env.offloading, env.run = rec_offloading, rec_run
    agent.forward_backward(obj, env, 0.0)
    jobs = env.jobs[:env.num_jobs]
    flows = env.flows[:env.num_jobs]
    out.update(job_source=np.array([j.source_node for j in jobs], np.int64),
               job_rate=np.array([j.arrival_rate for j in jobs], np.float64),
               job_ul=np.array([j.ul_data for j in jobs], np.float64),
               job_dl=np.array([j.dl_data for j in jobs], np.float64),
               flow_dst=np.array([f.dst for f in flows], np.int64),
               flow_route=np.concatenate([np.asarray(f.route, np.int64) for f in flows]),
               flow_route_off=np.cumsum([0] + [len(f.route) for f in flows]).astype(np.int64))
    dst = os.path.join(ROOT, "tests", "golden", "agent_case_n20.npz")
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    main()
