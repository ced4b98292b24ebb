"""The batched float64 belief oracle (oracle/belief_oracle.py) against the scalar oracle (sy_oracle.belief_update /
belief_cross_entropy) and against the C oracle's own belief trajectory.  CPU only."""
import numpy as np
import pytest

import belief_oracle as bo
import sy_oracle as so
import sy_oracle_c as oc
from student_mechanism_design_b200 import generate_graph_pool

RTOL = 1e-14
HUB_DEGREES = [0, 1, 3, 4, 5, 8, 9, 12, 13, 16, 17, 32, 33, 64, 255]


def _close(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, what
    assert np.array_equal(got == 0, want == 0), (what, "support")
    err = np.abs(got - want)
    bad = err > RTOL * np.abs(want)
    assert not bad.any(), (what, np.argwhere(bad)[:5].tolist(), float((err / np.maximum(np.abs(want), 1e-300)).max()))


def _graphs():
    return {
        "hub": bo.hub_graph(300, HUB_DEGREES, isolated=(40, 41, 77)),
        "random": generate_graph_pool(1, 64, 110, seed=3)[0],
        "isolated": bo.hub_graph(37, [2, 5], isolated=(0, 17, 36)),
    }


def _rows(N, rng):
    tiny = 10.0 ** rng.uniform(-25, 0, size=N)  # entries spanning 1e-25 .. 1
    tiny[rng.integers(N, size=N // 5)] = 0.0
    r = rng.random(N)
    return {
        "random": r / r.sum(),
        "sum_3_7": 3.7 * r / r.sum(),
        "zero": np.zeros(N),
        "tiny": tiny,
        "sparse": np.where(rng.random(N) < 0.1, rng.random(N), 0.0),
        "uniform": so.belief_uniform(N),
    }


def test_propagation_matrix_degrees():
    g = bo.hub_graph(300, HUB_DEGREES, isolated=(40, 41, 77))
    rp = so.Graph(g.num_nodes, g.edge_links, g.edges).csr()[0]
    deg = np.diff(rp)
    assert bo.max_degree(g) >= 255 and set(HUB_DEGREES) <= set(deg.tolist()) | {0}
    M = bo.propagation_matrix(g)
    # every column is a node's mass: it sums to 1 (split over the neighbours, or kept by an isolated node)
    np.testing.assert_allclose(np.asarray(M.sum(axis=0)).ravel(), 1.0, rtol=1e-14)
    for j in np.nonzero(deg == 0)[0]:
        assert M[j, j] == 1.0 and M[:, j].nnz == 1


@pytest.mark.parametrize("gname", ["hub", "random", "isolated"])
def test_propagate_and_hints_match_scalar_oracle(gname):
    g = _graphs()[gname]
    og = so.Graph(g.num_nodes, g.edge_links, g.edges)
    N = g.num_nodes
    rng = np.random.default_rng(7)
    rows = _rows(N, rng)
    hints = {"none": None, "empty": np.zeros(N, np.uint8), "all": np.ones(N, np.uint8),
             "random": (rng.random(N) < 0.3).astype(np.uint8)}
    prev = np.stack(list(rows.values()))
    B = len(prev)
    for hname, h in hints.items():
        hint = None if h is None else np.tile(h, (B, 1))
        got = bo.belief_step_batched(prev, [g], np.zeros(B, np.int64), np.full(B, bo.PROPAGATE), np.zeros(B, np.int64), hint)
        for b, rname in enumerate(rows):
            want = so.belief_update(prev[b], og, hint=None if h is None else np.nonzero(h)[0].tolist())
            _close(got[b], want, (gname, hname, rname))


def test_keep_uniform_delta_rows_and_mixed_graphs():
    gs = _graphs()
    pool = [gs["isolated"], bo.hub_graph(37, [9, 3], isolated=(5,), seed=1)]
    N, B = 37, 12
    rng = np.random.default_rng(1)
    prev = rng.random((B, N))
    prev[3] = 0.0
    gid = np.arange(B) % 2
    op = np.array([bo.KEEP, bo.UNIFORM, bo.DELTA, bo.PROPAGATE] * 3)
    x = rng.integers(N, size=B)
    got = bo.belief_step_batched(prev, pool, gid, op, x)
    for b in range(B):
        og = so.Graph(N, pool[gid[b]].edge_links, pool[gid[b]].edges)
        if op[b] == bo.KEEP:
            assert np.array_equal(got[b], prev[b])
        elif op[b] == bo.UNIFORM:
            assert np.array_equal(got[b], so.belief_uniform(N))
        elif op[b] == bo.DELTA:
            assert np.array_equal(got[b], so.belief_update(prev[b], og, reveal=x[b]))
        else:
            _close(got[b], so.belief_update(prev[b], og), b)
    assert np.array_equal(got[3], so.belief_uniform(N))  # zero row propagates to the uniform row


@pytest.mark.parametrize("gname", ["hub", "random", "isolated"])
def test_cross_entropy_matches_scalar_oracle(gname):
    g = _graphs()[gname]
    og = so.Graph(g.num_nodes, g.edge_links, g.edges)
    N = g.num_nodes
    rng = np.random.default_rng(11)
    prev = np.stack(list(_rows(N, rng).values()))
    B = len(prev)
    for x in (0, N // 2, N - 1):
        got = bo.belief_ce_batched(prev, [g], np.zeros(B, np.int64), np.full(B, x))
        want = [so.belief_cross_entropy(so.belief_update(prev[b], og), x) for b in range(B)]
        np.testing.assert_allclose(got, want, rtol=RTOL, atol=0)


@pytest.mark.parametrize("auto_reset,reveal", [(True, 3), (False, 4), (True, 0)])
def test_ops_from_c_oracle_reproduce_its_belief_trajectory(auto_reset, reveal):
    """The operation derived from the C oracle's state before and after each step, applied to its previous row, gives
    its next row: propagation, reveals, same-step auto-resets and frozen envs (no auto-reset), on a pool with a hub
    graph and isolated nodes."""
    N = 40
    pool = [bo.hub_graph(N, [0, 12, 17, 33], isolated=(9, 30)), generate_graph_pool(1, N, 70, seed=2)[0]]
    cfg = so.OracleConfig(num_police=2, agent_money=6, toll=1, belief=True, reveal_interval=reveal)
    B = 96
    gid = (np.arange(B) // 32) % 2
    ob = oc.CBatch(cfg, pool, B, seed=5, auto_reset=auto_reset, graph_id=gid.astype(np.int32))
    mats = [bo.propagation_matrix(g) for g in pool]
    seen = set()
    for s in range(30):
        prev, done, ep = ob.belief(), np.asarray(ob.done), np.asarray(ob.episode)
        ob.step(ob.sample_actions(s))
        op = bo.op_from_transition(done, ep, np.asarray(ob.episode), ob.revealed(), reveal, auto_reset)
        seen |= set(op.tolist())
        got = bo.belief_step_batched(prev, pool, np.asarray(ob.graph_id), op, ob.pos()[:, 0], mats=mats)
        _close(got, ob.belief(), ("step", s))
    want = {bo.PROPAGATE} | ({bo.UNIFORM} if auto_reset else {bo.KEEP}) | ({bo.DELTA} if reveal else set())
    assert want <= seen, seen


def test_ops_with_skipped_reveals_match_python_oracle():
    """Scheduled reveals that the batch's Philox draw skips propagate instead (OracleBatch.step with reveal_skip_prob)."""
    N = 30
    pool = generate_graph_pool(2, N, 50, seed=4)
    cfg = so.OracleConfig(num_police=2, agent_money=8, belief=True, reveal_interval=2, reveal_skip_prob=0.5)
    ob = so.OracleBatch.from_seed(cfg, [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in pool], 40, seed=3)
    skipped = 0
    for s in range(12):
        prev, done, ep = ob.belief(), list(ob.done), list(ob.episode)
        ob.step(ob.sample_actions(s))
        op = bo.op_from_transition(done, ep, ob.episode, ob.revealed(), 2, True)
        t = np.asarray([e.t for e in ob.envs])
        skipped += int(((t % 2 == 0) & (op == bo.PROPAGATE)).sum())
        got = bo.belief_step_batched(prev, pool, ob.graph_id, op, ob.pos()[:, 0])
        _close(got, ob.belief(), ("step", s))
    assert skipped > 0
