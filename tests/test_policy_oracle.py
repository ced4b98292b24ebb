"""The MAPPO restatement in oracle/policy_oracle.py against tests/golden/mappo.npz, which was recorded from the
UNMODIFIED reference modules (oracle/gen_policy_golden.py; src/agent/mappo_agent.py:6-44, 87-142): the masked,
renormalised distribution incl. its fall-back branches, Categorical's log-prob of the reference's sampled action,
the central critic.  Plus sanity properties of the GNN restatement (parity unpinned: torch_geometric is absent)."""
import os

import numpy as np

from conftest import ROOT
from oracle import policy_oracle as po
from oracle import sy_oracle as so

GOLD = np.load(os.path.join(ROOT, "tests", "golden", "mappo.npz"))


def _policy_sd(ci, pid):
    return {k: GOLD[f"c{ci}_p{pid}_{k}"] for k in ("actor.0.weight", "actor.0.bias", "actor.2.weight", "actor.2.bias")}


def test_mappo_distribution_and_log_prob_match_reference():
    branches = set()
    for ci, (n_agents, obs_size, hidden, n_nodes) in enumerate(GOLD["cases"].tolist()):
        for t in range(len(GOLD[f"c{ci}_obs"])):
            sd = _policy_sd(ci, int(GOLD[f"c{ci}_pid"][t]))
            mask, want = GOLD[f"c{ci}_mask"][t], GOLD[f"c{ci}_probs"][t]
            got = po.mappo_probs(GOLD[f"c{ci}_obs"][t], sd, mask, dtype=np.float32)
            np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-9)
            a = int(GOLD[f"c{ci}_action"][t])
            np.testing.assert_allclose(po.categorical_log_prob(got, a, np.float32), GOLD[f"c{ci}_logp"][t], rtol=2e-5, atol=2e-6)
            if mask.sum() == 0:
                branches.add("no mask")
                assert np.allclose(want, 1.0 / n_nodes)
            elif np.allclose(want[mask > 0], 1.0 / mask.sum()) and mask.sum() > 1:
                branches.add("uniform over mask")
            else:
                branches.add("softmax")
            assert want[mask == 0].sum() == 0 or mask.sum() == 0
    assert branches == {"no mask", "uniform over mask", "softmax"}


def test_critic_matches_reference():
    for ci in range(len(GOLD["cases"])):
        sd = {k: GOLD[f"c{ci}_{k}"] for k in ("critic.0.weight", "critic.0.bias", "critic.2.weight", "critic.2.bias")}
        got = [po.critic_value(x, sd) for x in GOLD[f"c{ci}_gobs"]]
        np.testing.assert_allclose(got, GOLD[f"c{ci}_values"], rtol=1e-5, atol=1e-6)


def test_mappo_sampler_follows_the_distribution():
    p = np.zeros(30, dtype=np.float32)
    p[[3, 7, 21]] = [0.2, 0.5, 0.3]
    draws = np.bincount([po.mappo_sample(p, 5, e, 0, 1) for e in range(4000)], minlength=30)
    assert set(np.nonzero(draws)[0]) == {3, 7, 21}
    np.testing.assert_allclose(draws[[3, 7, 21]] / 4000.0, [0.2, 0.5, 0.3], atol=0.03)


def test_gnn_restatement_properties():
    rng = np.random.default_rng(0)
    g = so.philox_sample_graph_once(1, 0, 0, 0, 20, 35)
    K = 4
    sd = {"conv1.W": rng.normal(size=(K, K)), "conv1.bias": rng.normal(size=K) * 0.1, "conv1.phi.lin.weight": rng.normal(size=(K, K)),
          "conv2.W": rng.normal(size=(K, K)), "conv2.bias": rng.normal(size=K) * 0.1, "conv2.phi.lin.weight": rng.normal(size=(K, K)),
          "output_layer.weight": rng.normal(size=(1, K)), "output_layer.bias": rng.normal(size=1)}
    x = po.graph_features(po.FEATURES_ENV, [3, 5, 9, 11], 3, 20, K)
    assert x.sum() == 4 and x[3, 0] == 1 and x[11, 3] == 1
    assert po.graph_features(po.FEATURES_ENV, [3, 5, 9, 11], -1, 20, K)[:, 0].sum() == 0
    xr = po.graph_features(po.FEATURES_REFERENCE, [3, 5, 9, 11], -1, 20, K)
    assert xr[19, 0] == 1 and xr[5, 1] == 1 and xr[5, 2] == 1 and xr[:, 3].sum() == 0  # utils.py:176-199 as written
    q = po.gnn_forward(x, g.edge_links, sd)
    assert q.shape == (20,) and np.isfinite(q).all()
    # a symmetric W has no antisymmetric part: W - W^T = 0, only the -gamma damping and the GCN term remain
    sd2 = dict(sd)
    sd2["conv1.W"] = sd["conv1.W"] + sd["conv1.W"].T
    sd3 = dict(sd)
    sd3["conv1.W"] = np.zeros((K, K))
    np.testing.assert_allclose(po.gnn_forward(x, g.edge_links, sd2), po.gnn_forward(x, g.edge_links, sd3), rtol=1e-12)
    # messages follow the stored edge direction only: reversing every edge changes the result
    assert not np.allclose(q, po.gnn_forward(x, g.edge_links[:, ::-1], sd))


def test_host_gcn_lists_reproduce_the_oracle_aggregation():
    """policy.gcn_in_edges (host logic of the policy kernels): aggregating with its in-edge lists and coefficients is
    GCNConv's normalised propagation as the oracle restates it (directed edge_links.T, self-loops, deg = 1 + in-degree)."""
    from student_mechanism_design_b200 import GraphSpec, gcn_in_edges

    rng = np.random.default_rng(3)
    graphs = [so.philox_sample_graph_once(5, g, 0, 0, 25, 45) for g in range(3)]
    specs = [GraphSpec(g.num_nodes, g.edge_links, g.edges) for g in graphs]
    in_ptr, in_src, in_coef, self_coef, stride = gcn_in_edges(specs)
    assert stride == max(len(g.edges) for g in graphs)
    for i, g in enumerate(graphs):
        n = g.num_nodes
        x = rng.normal(size=(n, 5))
        got = self_coef[i][:, None].astype(np.float64) * x
        for v in range(n):
            for e in range(in_ptr[i, v], in_ptr[i, v + 1]):
                got[v] += float(in_coef[i, e]) * x[in_src[i, e]]
        src, dst = g.edge_links[:, 0].astype(np.int64), g.edge_links[:, 1].astype(np.int64)
        deg = 1.0 + np.bincount(dst, minlength=n)
        dis = deg ** -0.5
        want = (dis * dis)[:, None] * x
        np.add.at(want, dst, (dis[src] * dis[dst])[:, None] * x[src])
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)
        assert in_ptr[i, -1] == len(g.edges) and (np.diff(in_ptr[i]) == np.bincount(dst, minlength=n)).all()


def _random_gnn_sd(rng, K):
    return {"conv1.W": rng.normal(size=(K, K)), "conv1.bias": rng.normal(size=K) * 0.1, "conv1.phi.lin.weight": rng.normal(size=(K, K)),
            "conv2.W": rng.normal(size=(K, K)), "conv2.bias": rng.normal(size=K) * 0.1, "conv2.phi.lin.weight": rng.normal(size=(K, K)),
            "output_layer.weight": rng.normal(size=(1, K)), "output_layer.bias": rng.normal(size=1)}


def test_gnn_two_independent_restatements_agree__parity_unpinned():
    """PARITY UNPINNED: torch_geometric (the reference's AntiSymmetricConv / GCNConv, gnn_agent.py:230-257) is not
    installed here, so no golden vector from the real module exists (oracle/gen_gnn_golden.py writes one wherever PyG
    is available).  Until then the dense NumPy restatement (`gnn_forward`) and a second one written independently as
    literal per-edge message passing in Python floats (`gnn_forward_message_passing`) must agree to 1e-12 on random
    graphs, weights and feature modes (hidden MrX, the reference's own feature quirk)."""
    rng = np.random.default_rng(11)
    for ci, (N, E, K) in enumerate([(12, 11, 3), (20, 35, 4), (40, 75, 7), (25, 50, 16)]):
        g = so.philox_sample_graph_once(3, ci, 0, 0, N, E)
        sd = _random_gnn_sd(rng, K)
        for t in range(4):
            pos = rng.choice(N, size=K, replace=False)
            mode = po.FEATURES_REFERENCE if t == 3 else po.FEATURES_ENV
            x = po.graph_features(mode, pos, -1 if t % 2 else int(pos[0]), N, K)
            a = po.gnn_forward(x, g.edge_links, sd)
            b = po.gnn_forward_message_passing(x, g.edge_links, sd)
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12)
    # a graph with parallel / reversed duplicates in the stored edge list: both count every stored edge once, in its direction
    links = np.asarray([[0, 1], [1, 0], [1, 2], [1, 2], [3, 2]])
    sd = _random_gnn_sd(rng, 3)
    x = po.graph_features(po.FEATURES_ENV, [0, 2, 3], 0, 4, 3)
    np.testing.assert_allclose(po.gnn_forward(x, links, sd), po.gnn_forward_message_passing(x, links, sd), rtol=1e-12, atol=1e-12)


def test_gnn_restatement_against_pyg_golden_when_present():
    """pins the GNN restatement as soon as tests/golden/gnn.npz (oracle/gen_gnn_golden.py, needs torch_geometric) exists"""
    import pytest

    path = os.path.join(ROOT, "tests", "golden", "gnn.npz")
    if not os.path.isfile(path):
        pytest.skip("tests/golden/gnn.npz absent (torch_geometric is not installed in the build image): GNN parity unpinned")
    gold = np.load(path)
    keys = ("conv1.W", "conv1.bias", "conv1.phi.lin.weight", "conv2.W", "conv2.bias", "conv2.phi.lin.weight", "output_layer.weight",
            "output_layer.bias")
    for ci in range(len(gold["cases"])):
        sd = {k: gold[f"c{ci}_{k}"] for k in keys}
        for x, q in zip(gold[f"c{ci}_x"], gold[f"c{ci}_q"]):
            np.testing.assert_allclose(po.gnn_forward(x.astype(np.float64), gold[f"c{ci}_edge_links"], sd), q, rtol=2e-5, atol=2e-6)


def test_batched_philox_matches_the_scalar_one():
    rng = np.random.default_rng(5)
    ctr = rng.integers(0, 2 ** 32, size=(4, 300), dtype=np.uint64)
    seed = (0xDEADBEEF << 32) | 0x12345678
    got = po.philox4x32_batched(*ctr, seed)
    for i in range(300):
        assert tuple(int(w[i]) for w in got) == so.philox4x32(tuple(int(c[i]) for c in ctr), (seed & 0xFFFFFFFF, seed >> 32))
    assert all(float(po.u01_batched(got[0])[i]) == po.u01(int(got[0][i])) for i in range(300))


def _pool_with_parallel_edges(N, E):
    """three graphs of one size; the last stores one edge twice and one reversed: both are separate GCN messages"""
    graphs = [so.philox_sample_graph_once(7, g, 0, 0, N, E) for g in range(3)]
    links = graphs[2].edge_links.copy()
    links[-1], links[-2] = links[0], links[1][::-1]
    return [graphs[0].edge_links, graphs[1].edge_links, links]


def test_batched_gnn_oracle_matches_both_scalar_restatements():
    """gnn_forward_batched (sparse aggregation, env chunks) == gnn_forward == gnn_forward_message_passing to 1e-12 on a
    few hundred envs of a pool with parallel edges, both feature modes, MrX hidden and revealed, both models."""
    rng = np.random.default_rng(12)
    N, E, K, B = 20, 35, 5, 240
    pool = _pool_with_parallel_edges(N, E)
    assert len({tuple(r) for r in pool[2].tolist()}) < len(pool[2])  # the pool does hold a parallel edge
    sds = [_random_gnn_sd(rng, K), _random_gnn_sd(rng, K)]
    pos = np.stack([rng.choice(N, size=K, replace=False) for _ in range(B)])
    pos[::7, 2] = pos[::7, 1]  # officers sharing a node
    rev = np.where(rng.random(B) < 0.5, -1, 3)
    gid = rng.integers(0, 3, size=B)
    for mode in (po.FEATURES_ENV, po.FEATURES_REFERENCE):
        q = po.gnn_forward_batched(mode, pos, rev, gid, pool, sds, N, chunk_floats=37 * N * K)  # several chunks per graph
        for b in range(B):
            x = po.graph_features(mode, pos[b], rev[b], N, K)
            np.testing.assert_array_equal(po.graph_features_batched(mode, pos[b: b + 1], rev[b: b + 1], N, K)[0], x)
            for m in range(2):
                np.testing.assert_allclose(q[b, m], po.gnn_forward(x, pool[gid[b]], sds[m]), rtol=1e-12, atol=1e-12)
                if b % 4 == 0:
                    np.testing.assert_allclose(q[b, m], po.gnn_forward_message_passing(x, pool[gid[b]], sds[m]), rtol=1e-12,
                                               atol=1e-12)
    assert (rev < 0).any() and (rev >= 0).any() and (gid == 2).any()


def test_batched_gnn_exploration_matches_gnn_select():
    rng = np.random.default_rng(2)
    B, A, N, seed, step, off = 300, 4, 30, (7 << 32) | 99, 17, 1000
    mask = rng.random((B, A, N)) < 0.12
    mask[::11, 1] = False  # agents without a move
    explored, act = po.gnn_explore_batched(mask, 0.4, 0.7, seed, off + np.arange(B), step)
    q = rng.normal(size=N)
    for b in range(B):
        for a in range(A):
            want, ex, _ = po.gnn_select(q, np.nonzero(mask[b, a])[0], 0.4 if a == 0 else 0.7, seed, off + b, step, a)
            assert ex == explored[b, a] and (act[b, a] == want if ex else act[b, a] == -1), (b, a)
    assert explored.any() and (~explored).any()


def test_batched_mappo_oracle_matches_mappo_probs():
    """mappo_forward_batched == mappo_probs to 1e-12 on a few hundred rows that take all three branches; the error scale
    is the documented sum of magnitudes"""
    rng = np.random.default_rng(4)
    R, D, H, N = 400, 6, 24, 33
    sd = {"actor.0.weight": rng.normal(size=(H, D)) * 0.4, "actor.0.bias": rng.normal(size=H) * 0.2,
          "actor.2.weight": rng.normal(size=(N, H)) * 0.2, "actor.2.bias": rng.normal(size=N)}
    sd["actor.2.bias"][:3] += 60.0  # the mass on masks without nodes 0..2 underflows 1e-8: uniform over the mask
    obs = rng.normal(size=(R, D))
    mask = rng.random((R, N)) < 0.15
    mask[::9] = False  # empty masks: uniform over all nodes
    mask[1::9, :3] = True
    out = po.mappo_forward_batched(obs, sd, mask, chunk=64)
    for r in range(R):
        np.testing.assert_allclose(out["probs"][r], po.mappo_probs(obs[r], sd, mask[r].astype(np.float64)), rtol=1e-12, atol=1e-15)
        h = np.abs(sd["actor.0.bias"]) + np.abs(sd["actor.0.weight"]) @ np.abs(obs[r])
        assert abs(out["scale"][r] - (np.abs(sd["actor.2.bias"]) + np.abs(sd["actor.2.weight"]) @ h).max()) <= 1e-12 * out["scale"][r]
    assert set(out["mode"].tolist()) == {po.MAPPO_SOFTMAX, po.MAPPO_UNIFORM_MASK, po.MAPPO_UNIFORM_ALL}
    gsd = {"critic.0.weight": rng.normal(size=(H, 3 * D)), "critic.0.bias": rng.normal(size=H), "critic.2.weight": rng.normal(size=(1, H)),
           "critic.2.bias": rng.normal(size=1)}
    x = rng.normal(size=(50, 3 * D))
    v, scale = po.critic_value_batched(x, gsd)
    np.testing.assert_allclose(v, [po.critic_value(r, gsd) for r in x], rtol=1e-12, atol=1e-12)
    assert (scale >= np.abs(v)).all()
