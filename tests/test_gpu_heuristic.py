"""Heuristic opponents (sy_heuristic_actions) on the device, through the C ABI, against the CPU oracle
(heuristic_oracle.heuristic_actions): per step on the device state at c2 / c3 shapes (every kind), N = 1 000, a ragged batch,
a pool whose graphs mix inside a tile and 16 mechanism groups with mixed tolls, police counts and horizons; the random
and fully exploring kinds equal sy_sample_actions, NONE sides stay untouched and two half-batch handles equal one full
handle; 300-step evade-vs-chase rollouts equal the oracle rollout with and without groups (state, rewards, flags,
statistics); RolloutCollector steps deferred with chasing police; the chasers catch more often than random police,
an evading MrX is caught less often than a random one, and every refused argument returns its code."""
import ctypes as C

import numpy as np
import pytest

import heuristic_oracle as ho
import sy_oracle as so
from test_gpu_parity import _compare_out, _compare_state

pytestmark = pytest.mark.gpu

CODE = {None: ho.HEUR_NONE, "random": ho.HEUR_RANDOM, "evade": ho.HEUR_EVADE, "chase": ho.HEUR_CHASE,
        "chase_belief": ho.HEUR_CHASE_BELIEF}
SENTINEL = 12345


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _pkg():
    import student_mechanism_design_b200 as pkg

    return pkg


def _graphs(pool):
    return [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in pool]


def _env_rules(env):
    """(toll, police count) of every env"""
    B = env.num_envs
    if env.mechanisms is None:
        return np.full(B, env.tolls), np.full(B, env.number_of_agents)
    gid = env.group_id.cpu().numpy()
    m = env.mechanisms
    return np.array([m[g]["tolls"] for g in gid]), np.array([m[g]["number_of_agents"] for g in gid])


def _check(torch, env, graphs, h, step_counter, tag):
    """one call of `h` on the device state against the oracle fed the same state"""
    B, A = env.num_envs, env.num_agents
    pos, money = env.pos.cpu().numpy(), env.money.cpu().numpy()
    t, rev, gid = env.timestep.cpu().numpy(), env.mrx_revealed.cpu().numpy(), env.graph_id.cpu().numpy()
    belief = env.belief_map.cpu().numpy() if h.police == "chase_belief" else None
    ls0 = h.last_seen.cpu().numpy()
    out = torch.full((B, A), SENTINEL, dtype=torch.int64, device=env.device)
    got = h.act(out=out, step_counter=step_counter).cpu().numpy()
    tolls, npol = _env_rules(env)
    want, want_ls = ho.heuristic_actions(env.seed, env.env_offset + np.arange(B), step_counter, pos, money, t, rev, gid,
                                         graphs, tolls, npol, CODE[h.mrx], CODE[h.police], h._h.explore_mrx,
                                         h._h.explore_police, ls0, belief, np.full((B, A), SENTINEL))
    bad = np.argwhere(got != want)
    assert bad.size == 0, (tag, bad[:5].tolist(), got[tuple(bad[0])], want[tuple(bad[0])])
    np.testing.assert_array_equal(h.last_seen.cpu().numpy(), want_ls, err_msg=tag)
    return got


POLICIES = [("evade", "chase", 0.0, 0.0), ("random", "random", 0.0, 0.0), (None, "chase", 0.0, 0.3),
            ("evade", None, 0.25, 0.0)]
BELIEF_POLICIES = POLICIES + [("evade", "chase_belief", 0.0, 0.0), ("random", "chase_belief", 0.1, 0.1)]
P16 = 4
MECH16 = [dict(tolls=g % 4, number_of_agents=P16 - g % P16, max_timestep=6 + 3 * g, agent_money=12) for g in range(16)]
SHAPES = {
    "c2": dict(B=1024, N=50, E=110, P=3, money=10, G=2, kw=dict(reveal_interval=5), steps=14, pol=POLICIES),
    # (the oracle draws the random actions one by one: at 65 536 envs the random police are left to the other shapes)
    "c3": dict(B=65536, N=200, E=400, P=6, money=20, G=4, kw=dict(reveal_interval=5, tolls=1, belief=True), steps=7,
               pol=[("evade", "chase", 0.0, 0.0), ("evade", "chase_belief", 0.0, 0.05), ("random", None, 0.0, 0.0)]),
    "n1000": dict(B=4096, N=1000, E=1500, P=4, money=30, G=1, kw=dict(reveal_interval=4, belief=True), steps=6,
                  pol=BELIEF_POLICIES),
    "ragged": dict(B=1007, N=50, E=110, P=3, money=10, G=3, kw=dict(reveal_interval=3, tolls=1), steps=10, pol=POLICIES),
    "mixed_pool": dict(B=640, N=60, E=120, P=5, money=15, G=7, kw=dict(reveal_interval=3, resample_graph=True, belief=True),
                       steps=10, pol=BELIEF_POLICIES),
    "groups16": dict(B=2048, N=50, E=110, P=P16, money=12, G=3, kw=dict(reveal_interval=3, max_timestep=60), steps=14,
                     pol=POLICIES, mechs=MECH16),
}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_per_step_matches_oracle(torch_cuda, shape):
    torch, pkg = torch_cuda, _pkg()
    c = SHAPES[shape]
    pool = pkg.generate_graph_pool(c["G"], c["N"], c["E"], seed=3)
    env = pkg.BatchedScotlandYardEnv(c["B"], c["P"], c["money"], graphs=pool, seed=17, auto_reset=True, **c["kw"])
    if "mechs" in c:
        env.set_mechanisms(c["mechs"])
    env.reset()
    graphs = _graphs(pool)
    hs = [pkg.HeuristicPolicy(env, m, p, em, ep) for m, p, em, ep in c["pol"]]
    for s in range(c["steps"]):
        for h in hs:
            _check(torch, env, graphs, h, 1000 + s, (shape, s, h.mrx, h.police))
        env.step(env.sample_actions(step_counter=s))


def _c2(pkg, B=1024, env_offset=0, **kw):
    pool = pkg.generate_graph_pool(2, 50, 110, seed=3)
    args = dict(seed=21, auto_reset=True, reveal_interval=5, env_offset=env_offset)
    args.update(kw)
    return pkg.BatchedScotlandYardEnv(B, 3, 10, graphs=pool, **args)


def test_random_exploring_and_none_identities(torch_cuda):
    torch, pkg = torch_cuda, _pkg()
    env = _c2(pkg, tolls=1)
    env.set_mechanisms([dict(number_of_agents=3, tolls=0), dict(number_of_agents=2, tolls=2), dict(number_of_agents=1)])
    env.reset()
    rnd = pkg.HeuristicPolicy(env, "random", "random")
    explore = pkg.HeuristicPolicy(env, "evade", "chase", 1.0, 1.0)
    none = pkg.HeuristicPolicy(env, None, None)
    only_police = pkg.HeuristicPolicy(env, None, "chase")
    only_mrx = pkg.HeuristicPolicy(env, "evade", None)
    for s in range(8):
        want = env.sample_actions(step_counter=500 + s)
        assert torch.equal(rnd.act(step_counter=500 + s), want)
        assert torch.equal(explore.act(step_counter=500 + s), want)
        sent = torch.full_like(want, SENTINEL)
        assert (none.act(out=sent.clone(), step_counter=s) == SENTINEL).all()
        a = only_police.act(out=sent.clone(), step_counter=s)
        assert (a[:, 0] == SENTINEL).all() and (a[:, 1:] != SENTINEL).all()
        a = only_mrx.act(out=sent.clone(), step_counter=s)
        assert (a[:, 1:] == SENTINEL).all() and (a[:, 0] != SENTINEL).all()
        env.step(want)


def test_two_half_handles_equal_one_full_handle(torch_cuda):
    torch, pkg = torch_cuda, _pkg()
    full = _c2(pkg, 1024, 0)
    halves = [_c2(pkg, 512, 0), _c2(pkg, 512, 512)]
    envs = [full] + halves
    hs = [pkg.HeuristicPolicy(e, "evade", "chase", 0.2, 0.2) for e in envs]
    for e in envs:
        e.reset()
    for s in range(30):
        acts = [h.act(step_counter=s) for h in hs]
        assert torch.equal(acts[0], torch.cat(acts[1:]))
        assert torch.equal(hs[0].last_seen, torch.cat([h.last_seen for h in hs[1:]]))
        for e, a in zip(envs, acts):
            e.step(a)
    assert torch.equal(full.pos, torch.cat([e.pos for e in halves]))


@pytest.mark.parametrize("groups", [False, True])
def test_rollout_matches_oracle(torch_cuda, groups):
    """300 steps of evade vs chase (reveal on, auto-reset, belief off): actions, state, rewards, flags and statistics"""
    torch, pkg = torch_cuda, _pkg()
    B, P, T, money = 256, 3, 40, 12
    pool = pkg.generate_graph_pool(3, 40, 70, seed=8)
    tables = pkg.env.numpy_reward_tables(T)
    env = pkg.BatchedScotlandYardEnv(B, P, money, graphs=pool, seed=5, auto_reset=True, reveal_interval=3, tolls=1,
                                     max_timestep=T, keep_reward64=True, reward_tables=tables)
    graphs = _graphs(pool)
    kw = dict(exp_table=tables[0], cov_table=tables[1], reveal_interval=3)
    if groups:
        mechs = [dict(number_of_agents=3, tolls=1, max_timestep=T, agent_money=money),
                 dict(number_of_agents=2, tolls=0, max_timestep=25, agent_money=20),
                 dict(number_of_agents=1, tolls=2, max_timestep=T, agent_money=30),
                 dict(number_of_agents=3, tolls=3, max_timestep=10, agent_money=money)]
        gid = [b % 4 for b in range(B)]
        env.set_mechanisms(mechs, group_id=torch.as_tensor(np.asarray(gid, dtype=np.int32)))
        cfgs = [so.OracleConfig(num_police=m["number_of_agents"], agent_money=m["agent_money"], toll=m["tolls"],
                                max_timestep=m["max_timestep"], **kw) for m in mechs]
        ob = so.OracleGroupBatch.from_seed(cfgs, gid, P, graphs, B, seed=5)
    else:
        ob = so.OracleBatch.from_seed(so.OracleConfig(num_police=P, agent_money=money, toll=1, max_timestep=T, **kw),
                                      graphs, B, seed=5)
    env.reset()
    h = pkg.HeuristicPolicy(env, "evade", "chase")
    ls = np.full(B, -1, dtype=np.int32)
    c = {"mode": "fp64", "kw": {}}
    for s in range(300):
        a = h.act(step_counter=s)
        want_a, ls = ho.batch_heuristic_actions(ob, s, ho.HEUR_EVADE, ho.HEUR_CHASE, last_seen=ls)
        np.testing.assert_array_equal(a.cpu().numpy(), want_a, err_msg=str(s))
        np.testing.assert_array_equal(h.last_seen.cpu().numpy(), ls, err_msg=str(s))
        env.step(a)
        want = ob.step(want_a)
        _compare_state(env, ob, c, s)
        _compare_out(env, want, c, s)
    total, per = ob.expected_stats()
    assert total[so.STAT_EPISODES] > B  # episodes ended and restarted throughout
    assert list(env.stats().values())[:14] == total[:14]
    if groups:
        for g, st in enumerate(env.stats(by_group=True)):
            assert list(st.values())[:14] == per[g][:14], g


def test_collector_steps_deferred_with_chasing_police(torch_cuda):
    torch, pkg = torch_cuda, _pkg()
    envs = [_c2(pkg, 1024, tolls=1) for _ in range(2)]
    for e in envs:
        e.reset()
    deferred = []
    orig = envs[0].step_deferred
    envs[0].step_deferred = lambda a: (deferred.append(1), orig(a))[1]
    buf = pkg.RolloutCollector(envs[0], pkg.HeuristicPolicy(envs[0], "evade", "chase"), horizon=40).collect()
    assert len(deferred) == 40 and not envs[0].observations_pending
    h = pkg.HeuristicPolicy(envs[1], "evade", "chase")
    for t in range(40):
        a = h()
        assert torch.equal(buf["actions"][t], a), t
        envs[1].step(a)
        assert torch.equal(buf["reward"][t], envs[1].reward), t
    for name in ("pos", "money", "timestep", "mrx_revealed", "action_mask", "node_features", "agent_budget"):
        assert torch.equal(getattr(envs[0], name), getattr(envs[1], name)), name
    assert envs[0].stats() == envs[1].stats()


def test_chase_belief_refused_while_observations_are_pending(torch_cuda):
    torch, pkg = torch_cuda, _pkg()
    env = _c2(pkg, belief=True)
    env.reset()
    h = pkg.HeuristicPolicy(env, "evade", "chase_belief")
    assert not h.reads_state_only
    env.step_deferred(env.sample_actions())
    out = torch.full((env.num_envs, env.num_agents), SENTINEL, dtype=torch.int64, device=env.device)
    h.last_seen.fill_(7)
    with pytest.raises(pkg.SyError, match="pending"):
        h.act(out=out)
    torch.cuda.synchronize()
    assert (out == SENTINEL).all() and (h.last_seen == 7).all()
    env.flush_observations()
    h.act(out=out)
    assert (out != SENTINEL).all()


def _capture_rate(pkg, mrx, police, steps=250):
    """share of the finished episodes that end in a capture"""
    env = pkg.BatchedScotlandYardEnv(2048, 3, 20, graphs=pkg.generate_graph_pool(4, 50, 110, seed=3), seed=33,
                                     auto_reset=True, reveal_interval=3)
    env.reset()
    h = pkg.HeuristicPolicy(env, mrx, police)
    for _ in range(steps):
        env.step(h.act())
    st = env.stats()
    return st["police_wins"] / st["episodes"]


def test_heuristics_play_towards_their_goals(torch_cuda):
    """chasers catch MrX more often than random police; an evading MrX is caught less often than a random one"""
    pkg = _pkg()
    rate_rr = _capture_rate(pkg, "random", "random")
    rate_rc = _capture_rate(pkg, "random", "chase")
    rate_ec = _capture_rate(pkg, "evade", "chase")
    assert rate_rc > rate_rr + 0.05, (rate_rr, rate_rc)
    assert rate_ec < rate_rc - 0.05, (rate_rc, rate_ec)


def _raw_call(env, h, obs=None, step_counter=0, out=None):
    import torch

    out = torch.full((env.num_envs, env.num_agents), SENTINEL, dtype=torch.int64, device=env.device) if out is None else out
    return env._lib.sy_heuristic_actions(env._handle, C.byref(h), C.byref(env._state), C.byref(obs or env._obs),
                                         step_counter, out.data_ptr(), env._stream()), out


def _h(**kw):
    from student_mechanism_design_b200 import _cabi

    h = _cabi.SyHeuristic(C.sizeof(_cabi.SyHeuristic), ho.HEUR_EVADE, ho.HEUR_CHASE, 0, 0, None)
    for k, v in kw.items():
        setattr(h, k, v)
    return h


def test_errors(torch_cuda):
    torch, pkg = torch_cuda, _pkg()
    from student_mechanism_design_b200 import _cabi

    env = _c2(pkg)
    env.reset()
    assert _raw_call(env, _h())[0] == 0
    for kw in (dict(struct_bytes=32), dict(mrx_kind=ho.HEUR_CHASE), dict(mrx_kind=-1), dict(police_kind=ho.HEUR_EVADE),
               dict(police_kind=5), dict(explore_mrx=2 ** 32 + 1), dict(explore_police=2 ** 63),
               dict(police_kind=ho.HEUR_CHASE_BELIEF)):  # (the env has no belief map)
        rc, out = _raw_call(env, _h(**kw))
        assert rc == 1, kw  # SY_ERR_INVALID_ARGUMENT
        assert (out == SENTINEL).all(), kw
    assert _raw_call(env, _h(explore_mrx=2 ** 32, explore_police=2 ** 32))[0] == 0
    obs = _cabi.SyObs(env._obs.action_mask, env._obs.node_features, env._obs.agent_budget, None, None)
    assert _raw_call(env, _h(), obs=obs)[0] == 1
    # call order: graphs and reward tables first
    lib, cfg = env._lib, env.config
    for load_graphs in (False, True):
        handle = C.c_void_p()
        _cabi.check(lib.sy_create(C.byref(cfg), C.byref(handle)))
        try:
            if load_graphs:
                row_ptr, col, wgt, stride = pkg.pack_csr(env.graphs)
                _cabi.check(lib.sy_load_graphs(handle, env.num_graphs, row_ptr.ctypes.data, col.ctypes.data,
                                               wgt.ctypes.data, stride, env._stream()))
            else:
                exp_neg, cov = pkg.numpy_reward_tables()
                _cabi.check(lib.sy_set_reward_tables(handle, exp_neg.ctypes.data, len(exp_neg), cov.ctypes.data, len(cov),
                                                     env._stream()))
            out = torch.empty(env.num_envs, env.num_agents, dtype=torch.int64, device=env.device)
            rc = lib.sy_heuristic_actions(handle, C.byref(_h()), C.byref(env._state), C.byref(env._obs), 0, out.data_ptr(),
                                          env._stream())
            assert rc == 3, load_graphs
        finally:
            lib.sy_destroy(handle)
    # new mechanism groups: refused until the reset they require, as the steps are
    env.set_mechanisms([dict(number_of_agents=2), dict(number_of_agents=3)])
    assert _raw_call(env, _h())[0] == 3
    h = pkg.HeuristicPolicy(env, "evade", "chase")
    with pytest.raises(pkg.SyError, match="reset"):
        h.act()
    env.reset()
    assert _raw_call(env, _h())[0] == 0
    h.act()
    # host-side validation
    for kw in (dict(mrx="chase"), dict(police="evade"), dict(police="chase_belief"), dict(epsilon_mrx=1.5),
               dict(epsilon_police=float("nan"))):
        with pytest.raises(ValueError):
            pkg.HeuristicPolicy(env, **kw)
    B, A = env.num_envs, env.num_agents
    for bad in (torch.zeros(B, A, dtype=torch.int32, device=env.device), torch.zeros(B, A + 1, dtype=torch.int64, device=env.device),
                torch.zeros(B, A, dtype=torch.int64), torch.zeros(A, B, dtype=torch.int64, device=env.device).t()):
        with pytest.raises(ValueError):
            h.act(out=bad)
