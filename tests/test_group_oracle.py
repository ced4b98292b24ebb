"""CPU: the mechanism-group oracle (sy_oracle.OracleGroupBatch) keeps the conventions of a handle with groups -- one
group equal to the config is OracleBatch bit for bit, a group with fewer police plays exactly as an OracleBatch built
with that police count while its other agents carry the absent values, and the per-group statistics sum to the
total -- and the host refuses values that ctypes would wrap into int32 before the library is reached."""
import numpy as np
import pytest

import sy_oracle as so

N, E, P = 20, 30, 4


def _graphs(G=2):
    import random

    return [so.sample_connected_graph(N, E, random.Random(s), np.random.RandomState(s)) for s in range(G)]


def _cfg(**kw):
    d = dict(num_police=P, agent_money=12, toll=1, reveal_interval=3, reveal_skip_prob=0.5, belief=True, max_timestep=14)
    d.update(kw)
    return so.OracleConfig(**d)


VIEWS = ["pos", "money", "timestep", "visits", "masks", "node_features", "revealed", "belief"]


def _rollout(batches, steps, check):
    for s in range(steps):
        acts = [b.sample_actions(s) for b in batches]
        outs = [b.step(a) for b, a in zip(batches, acts)]
        check(s, acts, outs)


@pytest.mark.parametrize("mode", ["fp64", "fp32"])
def test_one_group_equals_oracle_batch(mode):
    graphs = _graphs()
    cfg = _cfg(reward_mode=mode)
    B = 40
    ref = so.OracleBatch.from_seed(cfg, graphs, B, seed=5, env_offset=3)
    grp = so.OracleGroupBatch.from_seed([cfg], [0] * B, P, graphs, B, seed=5, env_offset=3)

    def check(s, acts, outs):
        assert np.array_equal(acts[0], acts[1]), s
        for k in ("reward", "terminated", "truncated", "winner"):
            assert outs[0][k].tobytes() == outs[1][k].tobytes(), (s, k)
        for v in VIEWS:
            assert getattr(ref, v)().tobytes() == getattr(grp, v)().tobytes(), (s, v)
        assert ref.episode == grp.episode and ref.graph_id == grp.graph_id

    _rollout([ref, grp], 40, check)
    assert ref.finished == grp.finished and len(ref.finished) > 0
    assert ref.belief_ces == grp.belief_ces
    assert ref.expected_stats() == grp.expected_stats()


def test_fewer_police_follow_their_own_batch():
    """groups of 1 and 2 police (horizons 6 and 14, own budgets, tolls, reveal schedules and weights) inside a
    4-police layout: their columns 0..P_g equal an OracleBatch built with that config, the rest are absent"""
    graphs = _graphs()
    w = dict(so.DEFAULT_REWARD_WEIGHTS, Police_group=-2.0, Mrx_position=1e6)
    cfgs = [_cfg(num_police=1, max_timestep=6, agent_money=30, toll=0, reveal_interval=0),
            _cfg(num_police=2, reward_weights=w, reveal_skip_prob=1.0),
            _cfg()]
    B = 45
    gid = np.random.default_rng(1).integers(0, len(cfgs), B)
    grp = so.OracleGroupBatch.from_seed(cfgs, gid, P, graphs, B, seed=9)
    refs = [so.OracleBatch.from_seed(c, graphs, B, seed=9) for c in cfgs]
    rows = [np.nonzero(gid == g)[0] for g in range(len(cfgs))]

    def check(s, acts, outs):
        for g, (c, r) in enumerate(zip(cfgs, refs)):
            A_g, idx = c.num_police + 1, rows[g]
            assert np.array_equal(acts[0][idx, :A_g], acts[1 + g][idx]), (s, g)
            assert (acts[0][idx, A_g:] == -1).all()
            for k in ("terminated", "truncated", "winner"):
                assert np.array_equal(outs[0][k][idx], outs[1 + g][k][idx]), (s, g, k)
            assert outs[0]["reward"][idx, :A_g].tobytes() == outs[1 + g]["reward"][idx].tobytes(), (s, g)
            assert not outs[0]["reward"][idx, A_g:].any()
            for v, absent in (("pos", -1), ("money", 0), ("masks", False)):
                got, want = getattr(grp, v)()[idx], getattr(r, v)()[idx]
                assert np.array_equal(got[:, :A_g], want) and (got[:, A_g:] == absent).all(), (s, g, v)
            nf = grp.node_features()[idx]
            assert np.array_equal(nf[..., :A_g], r.node_features()[idx]) and not nf[..., A_g:].any(), (s, g)
            for v in ("timestep", "visits", "revealed", "belief"):
                assert np.array_equal(getattr(grp, v)()[idx], getattr(r, v)()[idx]), (s, g, v)

    _rollout([grp] + refs, 30, check)
    total, per = grp.expected_stats()
    assert all(v[so.STAT_EPISODES] > 0 for v in per)
    assert per[0][so.STAT_TRUNCATIONS] > 0  # the 6-step horizon


def test_group_stats_sum_to_total_and_match_the_episodes():
    graphs = _graphs(3)
    cfgs = [_cfg(num_police=1, agent_money=3, toll=2), _cfg(num_police=3, max_timestep=0), _cfg(agent_money=0), _cfg()]
    B = 64
    gid = np.arange(B) % len(cfgs)
    ob = so.OracleGroupBatch.from_seed(cfgs, gid, P, graphs, B, seed=2)
    for s in range(25):
        ob.step(ob.sample_actions(s))
    total, per = ob.expected_stats()
    assert len(total) == len(per[0]) == so.SY_NUM_STATS
    for k in range(14):
        assert total[k] == sum(v[k] for v in per), k
    assert total[so.STAT_ENV_STEPS] == B * 25
    fin = np.asarray(ob.finished, dtype=np.int64)
    assert total[so.STAT_EPISODES] == len(fin) > 0
    assert total[so.STAT_SUM_SQ_LENGTH] == int((fin[:, 0] ** 2).sum())
    assert total[so.STAT_SUM_EPISODE_BUDGET_SPENT] == int(fin[:, 2].sum())
    assert total[so.STAT_MRX_WINS] == total[so.STAT_TRUNCATIONS] + total[so.STAT_OUT_OF_MONEY]
    # budget 0: every police is skipped from the first step on, so those episodes end out of money after one step
    assert per[2][so.STAT_OUT_OF_MONEY] == per[2][so.STAT_EPISODES] == per[2][so.STAT_ENV_STEPS]
    # horizon 0: the second step times out unless a capture comes first
    assert per[1][so.STAT_TRUNCATIONS] > 0 and per[1][so.STAT_SUM_LENGTH] <= 2 * per[1][so.STAT_EPISODES]
    assert per[0][so.STAT_POLICE_MOVES] > 0 and per[0][so.STAT_SUM_BUDGET_SPENT] >= 3 * per[0][so.STAT_POLICE_MOVES]


# ------------------------------------------------------------------------------------------ host range checks
@pytest.mark.parametrize("kw", [dict(agent_money=2 ** 32 + 5), dict(agent_money=2 ** 31), dict(agent_money=-1),
                                dict(max_timestep=65534), dict(max_timestep=2 ** 32 + 250), dict(max_timestep=-1),
                                dict(reveal_interval=2 ** 32 + 1), dict(reveal_interval=-2),
                                dict(tolls=1048577), dict(tolls=2 ** 31 - 1), dict(tolls=2 ** 32), dict(tolls=0.5),
                                dict(num_envs=2 ** 32 + 4), dict(num_envs=0)])
def test_constructor_refuses_values_int32_would_wrap(kw):
    """raised before the CUDA check, so before any ctypes field is written"""
    from student_mechanism_design_b200 import BatchedScotlandYardEnv

    args = dict(num_envs=4, number_of_agents=2, agent_money=10)
    args.update(kw)
    key = next(iter(kw))
    with pytest.raises(ValueError, match=key):
        BatchedScotlandYardEnv(**args, graph_nodes=10, graph_edges=12)


@pytest.mark.parametrize("mech", [{"agent_money": 2 ** 32 + 5}, {"agent_money": 2 ** 31}, {"reveal_interval": 2 ** 32 + 1},
                                  {"reveal_interval": 2 ** 31}, {"agent_money": True}])
def test_pack_mechanism_refuses_values_int32_would_wrap(mech):
    import types

    from student_mechanism_design_b200 import DEFAULT_REWARD_WEIGHTS
    from student_mechanism_design_b200.env import pack_mechanism

    base = types.SimpleNamespace(reward_weights=dict(DEFAULT_REWARD_WEIGHTS), agent_money=10, reveal_interval=5,
                                 config=types.SimpleNamespace(reveal_skip_prob=0.0))
    with pytest.raises(ValueError, match=next(iter(mech))):
        pack_mechanism(mech, base)
    g = pack_mechanism({"agent_money": 2 ** 31 - 1, "reveal_interval": 2 ** 31 - 1}, base)
    assert (g.agent_money, g.reveal_interval) == (2 ** 31 - 1, 2 ** 31 - 1)


def test_bounds_agree_across_header_and_binding():
    import os
    import re

    from conftest import ROOT
    from student_mechanism_design_b200 import _cabi

    header = open(os.path.join(ROOT, "include", "sy_env.h")).read()
    assert int(re.search(r"#define SY_MAX_TIMESTEP (\d+)", header).group(1)) == _cabi.SY_MAX_TIMESTEP == 0xFFFF - 2
    assert int(re.search(r"#define SY_MAX_TOLL (\d+)", header).group(1)) == _cabi.SY_MAX_TOLL
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    assert "SY_MAX_TIMESTEP" in doc and "SY_MAX_TOLL" in doc
