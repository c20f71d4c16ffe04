"""CPU: host logic of the drop-in agent and drivers against the reference's REAL simulator.

The GNN is an oracle-backed test double (tests/fakes.py); what is under test is everything around it: flags, feature
assembly, queue head, bug-compatible delay matrix, environment coupling, critic, route gradient, VJP seeding, replay,
checkpoints and the CSV schema.  One agent step is replayed from a recording made against the reference's simulator
(tests/golden/agent_case_n20.npz); the tests that drive the simulator itself (the drivers, and the statistical pin that
replays the AdHoc_test protocol and compares mean tau of the GNN policy with the reference's shipped result CSV, SURVEY
App. E/F) need the reference checkout and skip without it."""
import os
import sys

import numpy as np
import pandas as pd
import pytest

import chebnet_oracle as O
import fakes
import ref_env

needs_reference = pytest.mark.skipif(not ref_env.available(), reason="drives the reference's simulator: reference checkout not present")
REF = ref_env.REF_ROOT


@pytest.fixture()
def agent_mod(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["test"])
    mod = fakes.install(monkeypatch)
    F = mod.FLAGS
    F.device = "cpu"
    F.ref_src = ref_env.REF_SRC
    F.T = 1000
    F.K = 1
    F.fix_diag = False
    F.learning_rate = 1e-4
    F.training_set = "BAT800"
    return mod


@pytest.fixture()
def shipped(golden_dir):
    """The reference's model_ChebConv_BAT800_a5_c5_ACO_agent (a byte copy, pinned in test_oracle.py)."""
    return os.path.join(golden_dir, "ckpt_BAT800")


def _agent(mod, ckpt, memory=1000):
    agent = mod.ACOAgent(mod.FLAGS, memory)
    agent.load(ckpt)
    return agent


def test_load_restores_shipped_weights_exactly(agent_mod, shipped):
    agent = _agent(agent_mod, shipped)
    ws = O.load_reference_weights(shipped)
    for (W, b), (W2, b2) in zip(agent.net.get_weights(), ws):
        np.testing.assert_array_equal(W, W2); np.testing.assert_array_equal(b, b2)
    assert len(agent.model.trainable_weights) == 10


@needs_reference
def test_statistical_pin_forward_env(agent_mod, shipped):
    """tau of the GNN policy, bug-compatible diagonal, vs the shipped CSV on the same network files."""
    from multihop_offload_b200.drivers_common import load_case, run_method, sample_jobs
    AdhocCloud, apsp = ref_env.import_env()
    agent = _agent(agent_mod, shipped)
    datadir = os.path.join(REF, "data", "aco_data_ba_100")
    names = sorted(os.listdir(datadir))
    pick = names[::len(names) // 30][:30]
    csv = pd.read_csv(os.path.join(REF, "out", "Adhoc_test_data_aco_data_ba_100_load_0.15_T_1000.csv"))
    pub = csv[csv.Algo == "GNN"].groupby("filename").tau.mean()
    pub_local = csv[csv.Algo == "local"].groupby("filename").tau.mean()
    np.random.seed(12345)
    d_gnn, d_loc, taus = [], [], []
    for fn in pick:
        env, nodes_info, seed, n, m = load_case(AdhocCloud, os.path.join(datadir, fn), 1000)
        tg, tl = [], []
        for _ in range(10):
            sample_jobs(env, nodes_info, 0.15)
            run_method("baseline", env, agent, apsp)
            dl, _ = run_method("local", env, agent, apsp)
            dg, _ = run_method("GNN-test", env, agent, apsp)
            tg.append(np.nanmean(dg)); tl.append(np.nanmean(dl))
        d_gnn.append(np.mean(tg) - pub[fn]); d_loc.append(np.mean(tl) - pub_local[fn]); taus.append(np.mean(tg))
    d_gnn, d_loc = np.array(d_gnn), np.array(d_loc)
    se = d_gnn.std(ddof=1) / np.sqrt(len(d_gnn))
    print("tau GNN %.3f  paired diff vs published %.3f +- %.3f ; local control %.3f" % (np.mean(taus), d_gnn.mean(), se, d_loc.mean()))
    # published overall 18.44 (bug-compatible); the aligned-diagonal variant sits near 14.0 (SURVEY App. E)
    assert abs(d_gnn.mean()) < max(4 * se, 1.2)
    assert abs(d_loc.mean()) < 1.2
    # job sampling noise is common to both policies: the GNN-vs-local gap is the sharper pin
    # (published -1.92; the aligned-diagonal variant would sit near -6.4)
    assert abs((d_gnn - d_loc).mean()) < 0.8
    assert 16.0 < np.mean(taus) < 21.0


@pytest.mark.slow
@needs_reference
def test_statistical_pin_150_files(agent_mod, shipped):
    """The same replay over 150 network files x 10 instances (SURVEY App. E's protocol; ~3 min on 8 cores): per-size tau
    table written to tests/golden/statistical_pin_150.json (committed), checked against the shipped CSV.
    Run with:  python -m pytest tests/test_agent_host.py -m slow -k 150 -s"""
    import json
    from multihop_offload_b200.drivers_common import load_case, run_method, sample_jobs
    AdhocCloud, apsp = ref_env.import_env()
    agent = _agent(agent_mod, shipped)
    datadir = os.path.join(REF, "data", "aco_data_ba_100")
    names = sorted(os.listdir(datadir))
    pick = names[3::len(names) // 150][:150]
    csv = pd.read_csv(os.path.join(REF, "out", "Adhoc_test_data_aco_data_ba_100_load_0.15_T_1000.csv"))
    pub = csv[csv.Algo == "GNN"].groupby("filename").tau.mean()
    pub_local = csv[csv.Algo == "local"].groupby("filename").tau.mean()
    pub_cong = csv[csv.Algo == "GNN"].groupby("filename")[["congest_jobs", "num_jobs"]].sum() if "num_jobs" in csv.columns else None
    np.random.seed(2024)
    rows = []
    for fn in pick:
        env, nodes_info, seed, n, m = load_case(AdhocCloud, os.path.join(datadir, fn), 1000)
        tg, tl = [], []
        for _ in range(10):
            sample_jobs(env, nodes_info, 0.15)
            run_method("baseline", env, agent, apsp)
            dl, _ = run_method("local", env, agent, apsp)
            dg, _ = run_method("GNN-test", env, agent, apsp)
            tg.append(np.nanmean(dg)); tl.append(np.nanmean(dl))
        rows.append(dict(file=fn, n=int(n), tau_gnn=float(np.mean(tg)), tau_local=float(np.mean(tl)),
                         pub_gnn=float(pub[fn]), pub_local=float(pub_local[fn])))
    df = pd.DataFrame(rows)
    d_gnn = (df.tau_gnn - df.pub_gnn).values
    d_loc = (df.tau_local - df.pub_local).values
    se = d_gnn.std(ddof=1) / np.sqrt(len(d_gnn))
    table = {"files": len(df), "instances_per_file": 10, "seed": 2024, "bug_compatible_diagonal": True,
             "tau_gnn_mean": float(df.tau_gnn.mean()), "tau_gnn_published_same_files": float(df.pub_gnn.mean()),
             "tau_local_mean": float(df.tau_local.mean()), "tau_local_published_same_files": float(df.pub_local.mean()),
             "paired_diff_gnn": {"mean": float(d_gnn.mean()), "se": float(se)},
             "paired_diff_local": {"mean": float(d_loc.mean()), "se": float(d_loc.std(ddof=1) / np.sqrt(len(d_loc)))},
             "per_size": {str(int(k)): {"tau_gnn": float(g.tau_gnn.mean()), "published": float(g.pub_gnn.mean()), "files": int(len(g))}
                          for k, g in df.groupby("n")}}
    print(json.dumps(table, indent=1))
    with open(os.path.join(os.path.dirname(__file__), "golden", "statistical_pin_150.json"), "w") as f:
        json.dump(table, f, indent=1)
    assert abs(d_gnn.mean()) < max(4 * se, 0.5)
    assert abs(d_loc.mean()) < 0.5
    assert abs((d_gnn - d_loc).mean()) < 0.4       # published GNN-vs-local gap -1.92; the aligned-diagonal variant sits near -6.4
    for k, g in df.groupby("n"):
        # 30 files per size: the per-file paired difference has a standard deviation of ~4 (heavy tail: congested jobs)
        assert abs(g.tau_gnn.mean() - g.pub_gnn.mean()) < 2.5, (k, g.tau_gnn.mean(), g.pub_gnn.mean())


def test_forward_backward_seeds_the_vjp_like_the_oracle(agent_mod, shipped, golden_dir, monkeypatch):
    """One step on aco_case_seed500_m2_n20_s4.mat (jobs of np.random.seed(3)), replayed from the recording."""
    fakes.install_apsp(monkeypatch)
    agent = _agent(agent_mod, shipped)
    step = fakes.RecordedStep(np.load(os.path.join(golden_dir, "agent_case_n20.npz")))
    obj, env = step.obj, step.env
    captured = {}
    orig = agent.vjp_from_grad_dist

    def spy(gd):
        captured["gd"] = np.array(gd, copy=True)
        captured["tape"] = agent._tape
        return orig(gd)

    agent.vjp_from_grad_dist = spy
    out = agent.forward_backward(obj, env, 0.0)
    assert len(out) == 7 and np.isfinite(out[5]) and len(agent.memory) == 1
    grad, loss, mse = agent.memory[0]
    gd = captured["gd"]
    assert gd.shape == (env.num_nodes, env.num_nodes) and np.isfinite(gd).all() and np.abs(gd).sum() > 0
    # independent restatement: oracle head VJP + oracle stack VJP on the same grad_dist
    adj, X = step.adj, step.X
    ws = agent.net.get_weights()
    lam, cache = O.cheb_stack_forward(adj, X.astype(np.float32).astype(np.float64), ws, return_cache=True)
    ld, nd, hc = O.queue_head_forward(lam, obj.maps_ol_el, obj.maps_on_el, env.link_rates, env.cf_degs, env.proc_bws,
                                      env.adj_i, env.T, return_cache=True)
    comp = np.nonzero(env.proc_bws > 0)[0]
    g_ld = np.zeros_like(ld); g_nd = np.zeros_like(nd)
    for (e0, e1) in env.graph_c.edges:
        g_ld[env.link_matrix[e0, e1], 0] += gd[e0, e1] + gd[e1, e0]
    g_nd[:, 0] = gd[comp, comp]
    g_lam = O.queue_head_vjp(hc, g_ld, g_nd, lam.shape[0], obj.maps_ol_el, obj.maps_on_el)
    grads, _ = O.cheb_stack_backward(adj, ws, cache, g_lam)
    want = O.flatten_params(grads)
    got = grad.numpy()
    # the agent hands dY to the GNN VJP in fp32 (the kernels' dtype): ~6e-8 relative
    assert np.abs(got - want).max() <= 1e-6 * max(np.abs(want).max(), 1e-30)


def test_replay_applies_gradients_sequentially_and_checkpoints_roundtrip(agent_mod, shipped, tmp_path):
    agent = _agent(agent_mod, shipped, memory=50)
    rng = np.random.default_rng(0)
    import torch
    assert np.isnan(agent.replay(4))
    for i in range(6):
        agent.memorize(torch.as_tensor(rng.normal(size=agent.net.n_params)), float(i), 0.0)
    w0 = agent.net.get_flat()
    eps0 = agent.epsilon
    loss = agent.replay(4)
    assert np.isfinite(loss) and agent.optimizer.iterations == 4
    assert agent.epsilon == pytest.approx(eps0 * agent_mod.FLAGS.epsilon_decay)
    assert np.abs(agent.net.get_flat() - w0).max() > 0
    path = str(tmp_path / "model_x" / "cp-0003.ckpt")
    agent.save(path)
    other = agent_mod.ACOAgent(agent_mod.FLAGS, 10)
    other.load(str(tmp_path / "model_x"))
    np.testing.assert_array_equal(other.net.get_flat(), agent.net.get_flat())


@needs_reference
def test_adhoc_test_driver_csv_schema(agent_mod, tmp_path, monkeypatch):
    from multihop_offload_b200 import AdHoc_test
    monkeypatch.setattr(AdHoc_test, "ACOAgent", agent_mod.ACOAgent)
    F = agent_mod.FLAGS
    F.datapath = os.path.join(REF, "data", "aco_data_ba_10")
    F.out = str(tmp_path / "out")
    F.modeldir = os.path.join(REF, "model")
    F.arrival_scale = 0.15
    F.max_files = 2
    F.seed = 1
    AdHoc_test.main()
    df = pd.read_csv(os.path.join(F.out, "Adhoc_test_data_aco_data_ba_10_load_0.15_T_1000.csv"))
    ref_cols = list(pd.read_csv(os.path.join(REF, "out", "Adhoc_test_data_aco_data_ba_100_load_0.15_T_1000.csv"), nrows=1).columns)
    assert list(df.columns) == ref_cols
    assert len(df) == 2 * 10 * 3 and set(df.Algo) == {"baseline", "local", "GNN"}
    assert np.isfinite(df.tau).all()


@needs_reference
def test_adhoc_test_driver_batched_instances_same_rows(agent_mod, tmp_path, monkeypatch):
    """--batch_instances (SURVEY 8f #3): the GNN side of the 10 instances of a file is evaluated ahead of the per-instance
    loop without disturbing the random stream - every CSV row except the wall-clock column is identical."""
    from multihop_offload_b200 import AdHoc_test
    monkeypatch.setattr(AdHoc_test, "ACOAgent", agent_mod.ACOAgent)
    F = agent_mod.FLAGS
    F.datapath = os.path.join(REF, "data", "aco_data_ba_10")
    F.modeldir = os.path.join(REF, "model")
    F.arrival_scale = 0.15
    F.max_files = 2
    F.seed = 7
    dfs = []
    for flag in (False, True):
        F.batch_instances = flag
        F.out = str(tmp_path / ("out%d" % flag))
        AdHoc_test.main()
        dfs.append(pd.read_csv(os.path.join(F.out, "Adhoc_test_data_aco_data_ba_10_load_0.15_T_1000.csv")).drop(columns=["runtime"]))
    F.batch_instances = False
    pd.testing.assert_frame_equal(dfs[0], dfs[1], check_exact=True)


@needs_reference
def test_adhoc_train_driver_replays_and_saves(agent_mod, tmp_path, monkeypatch):
    from multihop_offload_b200 import AdHoc_train, tf_bundle
    monkeypatch.setattr(AdHoc_train, "ACOAgent", agent_mod.ACOAgent)
    F = agent_mod.FLAGS
    F.datapath = os.path.join(REF, "data", "aco_data_ba_10")
    F.out = str(tmp_path / "out")
    F.modeldir = str(tmp_path / "model")
    F.arrival_scale = 0.15
    F.max_files = 2
    F.epochs = 1
    F.batch = 8
    F.seed = 2
    F.learning_rate = 1e-6
    AdHoc_train.main()
    df = pd.read_csv(os.path.join(F.out, "aco_training_data_aco_data_ba_10_load_0.15_T_1000.csv"))
    assert len(df) == 2 * 10 * 4 and set(df.method) == {"baseline", "local", "GNN", "GNN-test"}
    ck = tf_bundle.latest_checkpoint(os.path.join(F.modeldir, "model_ChebConv_BAT800_a5_c5_ACO_agent"))
    assert ck is not None and ck.endswith("cp-0000.ckpt")
    assert [W.shape for W, _ in tf_bundle.load_weights(ck)] == [(1, 4, 32), (1, 32, 32), (1, 32, 32), (1, 32, 32), (1, 32, 1)]


def test_fill_adj_bits_and_pack_order():
    """Host-side planning helpers of the tensor-core forward: bit rows == dense block, pack_order is a permutation
    that never needs more tiles than the given order."""
    import scipy.sparse as sp
    from multihop_offload_b200 import GraphBatch, pack_order
    rng = np.random.default_rng(5)
    sizes = rng.choice(np.arange(20, 111, 10), size=60)
    mats = []
    for n in sizes:
        a = (rng.random((n, n)) < 0.08).astype(np.float32)
        a = np.triu(a, 1); a = a + a.T
        mats.append(sp.csr_matrix(a))
    b = GraphBatch.from_scipy(mats, tile_rows=128)
    assert b.adj_bits is not None and b.adj_bits.shape == (b.total_nodes, 4)
    for t in range(b.n_tiles):
        n0, n1 = int(b.graph_off[b.tile_off[t]]), int(b.graph_off[b.tile_off[t + 1]])
        dense = np.zeros((n1 - n0, 128), dtype=bool)
        for i in range(n0, n1):
            cols = b.colidx[b.rowptr[i]:b.rowptr[i + 1]] - n0
            dense[i - n0, cols] = True
        bits = np.unpackbits(b.adj_bits[n0:n1].view(np.uint8), axis=1, bitorder="little").astype(bool)
        assert np.array_equal(bits, dense), t
    perm = pack_order(sizes, 128)
    assert sorted(perm.tolist()) == list(range(len(sizes)))
    packed = GraphBatch.from_scipy([mats[i] for i in perm], tile_rows=128)
    assert packed.n_tiles <= b.n_tiles
    assert packed.max_tile_rows <= 128
