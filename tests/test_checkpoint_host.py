"""Re-keying the oracles mid-run (CPU only): `CBatch.set_seed` and `OracleBatch.seed` switched at the same step keep the
C and the Python oracle in step -- sampled actions, same-step auto-reset start nodes and graph choice, reveal-skip draws
-- and a `CBatch` restarted under a new seed equals one built with it.  These are the references tests/
test_gpu_checkpoint.py holds a re-seeded handle against."""
import numpy as np
import pytest

import sy_oracle as so
import sy_oracle_c as oc

N, E, P, MONEY, G, B = 30, 55, 3, 12, 5, 96
S1, S2 = 11, 2 ** 32 + 7


@pytest.fixture(scope="module")
def pool():
    import student_mechanism_design_b200.graphs as gr

    return [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in gr.generate_graph_pool(G, N, E, seed=3)]


def _cfg(skip=0.3):
    return so.OracleConfig(num_police=P, agent_money=MONEY, toll=1, belief=True, reveal_interval=2, reveal_skip_prob=skip,
                           max_timestep=14)


def _same_state(c, p, tag):
    assert np.array_equal(c.pos(), p.pos()), (tag, "pos")
    assert np.array_equal(c.money(), p.money()), (tag, "money")
    assert np.array_equal(c.timestep(), p.timestep()), (tag, "timestep")
    assert c.graph_id == p.graph_id, (tag, "graph_id")
    assert c.episode == p.episode, (tag, "episode")
    assert np.array_equal(c.visits(), p.visits()), (tag, "visits")
    assert np.array_equal(c.revealed(), p.revealed()), (tag, "revealed")
    assert np.array_equal(c.masks(), p.masks()), (tag, "masks")
    assert np.array_equal(c.node_features(), p.node_features()), (tag, "node_features")
    assert np.abs(c.belief() - p.belief()).max() <= 1e-12, (tag, "belief")


def _same_out(a, b, tag):
    assert a["reward"].tobytes() == b["reward"].tobytes(), (tag, "reward")
    for k in ("terminated", "truncated", "winner"):
        assert np.array_equal(a[k], b[k]), (tag, k)


@pytest.mark.parametrize("switch_at", [0, 23])
def test_c_and_python_oracle_switch_seeds_at_the_same_step(pool, switch_at):
    """60 steps of the random-valid policy over a 5-graph pool with resample_graph, reveal_skip_prob = 0.3 and same-step
    auto-reset; both oracles change from S1 to S2 before step `switch_at`.  A C oracle that keeps S1 diverges."""
    c = oc.CBatch(_cfg(), pool, B, seed=S1, auto_reset=True, resample_graph=True)
    p = so.OracleBatch.from_seed(_cfg(), pool, B, seed=S1, auto_reset=True, resample_graph=True)
    kept = oc.CBatch(_cfg(), pool, B, seed=S1, auto_reset=True, resample_graph=True)
    assert c.graph_id == p.graph_id and len(set(c.graph_id)) == G
    _same_state(c, p, "reset")
    skipped = resets = 0
    for s in range(60):
        if s == switch_at:
            c.set_seed(S2)
            p.seed = S2
            assert c.seed == S2 and c._c.seed == S2
        a = c.sample_actions(s)
        assert np.array_equal(a, p.sample_actions(s)), ("sampler", s)
        scheduled = (c.timestep() + 1) % 2 == 0
        want_c, want_p = c.step(a), p.step(a)
        _same_out(want_c, want_p, ("step", s))
        _same_state(c, p, ("step", s))
        ended = want_c["terminated"] | want_c["truncated"]
        skipped += int((scheduled & ~ended & (c.revealed() < 0)).sum())
        resets += int(ended.sum())
        kept.step(kept.sample_actions(s))
    assert skipped > 0 and resets > 0  # reveal skips and auto-resets happened under the new key
    assert not np.array_equal(kept.pos(), c.pos())


def test_c_oracle_reveal_skip_matches_python_and_zero_keeps_every_reveal(pool):
    """The C oracle's reveal-skip draw against the Python oracle's at p = 1 (every reveal skipped) and p = 0."""
    for skip in (1.0, 0.0):
        c = oc.CBatch(_cfg(skip), pool, B, seed=S1, auto_reset=True)
        p = so.OracleBatch.from_seed(_cfg(skip), pool, B, seed=S1, auto_reset=True)
        for s in range(12):
            a = c.sample_actions(s)
            _same_out(c.step(a), p.step(a), (skip, s))
            _same_state(c, p, (skip, s))
            on_schedule = c.timestep() % 2 == 0
            if skip == 1.0:
                assert (c.revealed() == -1).all()
            else:
                assert (c.revealed()[on_schedule & (c.timestep() > 0)] >= 0).all()


@pytest.mark.parametrize("s2", [0, 2 ** 32 + 7, 2 ** 64 - 1, -1])
def test_c_oracle_restarted_under_a_new_seed_equals_one_built_with_it(pool, s2):
    """set_seed + reset on a CBatch that ran 17 steps under S1 equals a CBatch built with s2, step for step (-1 is
    2^64 - 1)."""
    c = oc.CBatch(_cfg(), pool, B, seed=S1, auto_reset=True, resample_graph=True)
    for s in range(17):
        c.step(c.sample_actions(s))
    c.set_seed(s2)
    c.reset()
    fresh = oc.CBatch(_cfg(), pool, B, seed=s2 & (2 ** 64 - 1), auto_reset=True, resample_graph=True)
    _same_state(c, fresh, "restart")
    for s in range(30):
        a = c.sample_actions(s)
        assert np.array_equal(a, fresh.sample_actions(s)), ("sampler", s)
        _same_out(c.step(a), fresh.step(a), ("step", s))
        _same_state(c, fresh, ("step", s))
