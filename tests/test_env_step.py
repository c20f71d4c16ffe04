"""CPU: the numpy restatement of the environment step (oracle/env_oracle.py) against the reference's own
offloading() / local_compute() + run() - from the recording tests/golden/env_cases.npz (oracle/make_golden_env.py), and
live on randomly sampled instances when the reference checkout is present - and the batched environment step of
AdHoc_test --batch_instances with the oracle in place of the kernel."""
import os
import sys

import numpy as np
import pandas as pd
import pytest

import env_oracle
import ref_env

needs_reference = pytest.mark.skipif(not ref_env.available(), reason="drives the reference's simulator: reference checkout not present")


def golden_cases(golden_dir):
    z = np.load(os.path.join(golden_dir, "env_cases.npz"))
    for c in range(int(z["n_cases"])):
        pick = lambda pre: {k[len(pre):]: z[k] for k in z.files if k.startswith(pre)}  # noqa: E731
        net, items, out = pick("c%d_net_" % c), pick("c%d_items_" % c), pick("c%d_out_" % c)
        for k in ("n_nets", "max_nodes", "max_links"):
            net[k] = int(net[k])
        for k in ("n_items", "max_jobs", "route_stride"):
            items[k] = int(items[k])
        yield net, items, out


def assert_same(got, want, what=""):
    for k, v in want.items():
        assert got[k].shape == v.shape and np.array_equal(got[k], v, equal_nan=True), (what, k)


def test_oracle_matches_recording(golden_dir):
    n = 0
    for c, (net, items, out) in enumerate(golden_cases(golden_dir)):
        assert_same(env_oracle.env_step(net, items), out, c)
        n += items["n_items"]
    assert n == 63


def test_recording_covers_the_cases(golden_dir):
    cases = list(golden_cases(golden_dir))
    assert sorted({c[0]["max_nodes"] for c in cases}) == [20, 50, 80, 110, 200]
    J = np.concatenate([np.diff(c[1]["job_off"]) for c in cases])
    assert J.max() > 128 and 1 in J and np.any((J > 1) & (J < 8))
    modes = np.concatenate([c[1]["mode"] for c in cases])
    assert set(modes) == {0, 1}
    # the congestion branch of the servers fires: a load at or above the processing rate
    congested = 0
    for net, items, out in cases:
        for i in range(items["n_items"]):
            a, b = items["job_off"][i], items["job_off"][i + 1]
            load = np.zeros(net["max_nodes"])
            np.add.at(load, out["dst"][a:b], items["ul"][a:b] * items["rate"][a:b])
            congested += int(np.sum((load > 0) & (net["proc_bws"] - load <= 0)))
    assert congested > 0


@needs_reference
def test_oracle_matches_live_reference():
    """~200 instances sampled across the shipped datasets, each with the baseline, local and a third shortest-path matrix
    (random link delays, perturbed server delays): the oracle equals the reference's own offloading() / local_compute() +
    run().  An item on which the oracle reports a route loop is skipped: the reference's routing() never returns there."""
    sys.path.insert(0, os.path.dirname(env_oracle.__file__))
    import make_golden_env as G
    from multihop_offload_b200 import env_step as ES
    _, apsp = ref_env.import_env()
    rng = np.random.default_rng(11)
    names = []
    for d in ("aco_data_ba_10", "aco_data_ba_100"):
        p = os.path.join(ref_env.REF_ROOT, "data", d)
        if os.path.isdir(p):
            names += [os.path.join(p, f) for f in sorted(os.listdir(p))]
    files = [names[i] for i in rng.choice(len(names), size=min(20, len(names)), replace=False)]
    np.random.seed(5)
    count = loops = 0
    for f in files:
        env, nodes_info = ref_env.build_env(f)
        spb, hop = G.baseline_sp(env, apsp)
        loc = np.zeros_like(spb)
        np.fill_diagonal(loc, env.dmtx_baseline()[2])
        for (a, b) in env.graph_c.edges:   # shortest paths of random link delays: every greedy walk arrives
            env.graph_c[a][b]["delay"] = float(rng.uniform(0.01, 1.0))
        pert = apsp(env.graph_c, weight="delay")
        np.fill_diagonal(pert, np.diagonal(spb) * rng.uniform(0.5, 2.0, env.num_nodes))
        net = ES.network_arrays(env, hop)
        for _ in range(10):
            jobs = G.sampled_jobs(env, nodes_info, float(rng.choice([0.15, 0.5, 1.5])))
            env.clear_all_jobs()
            for (s, r) in jobs:
                env.add_job(int(s), rate=float(r))
            jv = ES.jobs_of(env)
            for mode, k in ((ES.GREEDY, 0), (ES.LOCAL, 1), (ES.GREEDY, 2)):
                items = ES.item_arrays(net, [[spb, loc, pert][k]], [ES.EnvItem(mode, 0, *jv)])
                got = env_oracle.env_step(net, items)
                if got["status"][0] == env_oracle.ROUTE_LOOP:   # the reference's routing() would never return
                    loops += 1
                    continue
                assert_same(got, dict(G.reference_step(env, mode, [spb, loc, pert][k], hop), status=np.zeros(1, np.int32)), f)
            count += 1
    assert count >= 200 and loops == 0, (count, loops)


@needs_reference
def test_adhoc_test_batched_env_step_same_rows(tmp_path, monkeypatch):
    """AdHoc_test --batch_instances with the batched environment step (the oracle standing in for mho_env_step): the
    simulator's run() is never called, and every CSV row except the wall-clock column, and the random stream after the
    run, equal the per-instance loop's - the job sets, the draws and the results match."""
    import fakes
    from multihop_offload_b200 import AdHoc_test, drivers_common, env_step
    monkeypatch.setattr(sys, "argv", ["test"])
    mod = fakes.install(monkeypatch)
    F = mod.FLAGS
    F.device, F.ref_src, F.T, F.K, F.fix_diag, F.learning_rate, F.training_set = "cpu", ref_env.REF_SRC, 1000, 1, False, 1e-4, "BAT800"
    monkeypatch.setattr(AdHoc_test, "ACOAgent", mod.ACOAgent)
    calls, sim_runs = [], []

    def oracle_run(plan, items, want):
        calls.append(items["n_items"])
        return env_oracle.env_step(plan.net, items, want)

    monkeypatch.setattr(env_step, "run", oracle_run)
    AdhocCloud, _ = ref_env.import_env()
    sim_run = AdhocCloud.run

    def counted_run(self):
        sim_runs.append(1)
        return sim_run(self)

    monkeypatch.setattr(AdhocCloud, "run", counted_run)
    F.datapath = os.path.join(ref_env.REF_ROOT, "data", "aco_data_ba_10")
    F.modeldir = os.path.join(ref_env.REF_ROOT, "model")
    F.arrival_scale = 0.15
    F.max_files = 2
    F.seed = 7
    F.batch_instances = True
    dfs, states, runs = [], [], []
    for device_step in (False, True):
        monkeypatch.setattr(drivers_common, "use_device_env_step", lambda agent: device_step)
        del sim_runs[:]
        F.out = str(tmp_path / ("out%d" % device_step))
        AdHoc_test.main()
        dfs.append(pd.read_csv(os.path.join(F.out, "Adhoc_test_data_aco_data_ba_10_load_0.15_T_1000.csv")).drop(columns=["runtime"]))
        states.append(np.random.get_state()[1].copy())
        runs.append(len(sim_runs))
    F.batch_instances = False
    assert calls == [30, 30]
    assert runs == [60, 0]
    assert len(dfs[1]) == 60
    pd.testing.assert_frame_equal(dfs[0], dfs[1], check_exact=True)
    assert np.array_equal(states[0], states[1])
