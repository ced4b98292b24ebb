"""Mechanism groups against the CPU oracle (sy_oracle.OracleGroupBatch, the C oracle for the long horizons), not
against ungrouped handles that run the same kernel source.

Checked here: a 15-police handle whose groups put every mechanism key at its edges (police 1 and 15, horizons 0 / 1 /
the handle's, budgets 0 / 1 / 2^31 - 1, tolls 0 / above every budget / SY_MAX_TOLL, reveal intervals 0 / 1 / 7, skip
probabilities 0 / 0.5 / 1, weights with zeros, negatives, 1e6 and values fp32 cannot hold) follows the per-env oracle
after every step through the two-kernel, fused, deferred, replayed one-launch rollout and bulk-writer paths in both
reward modes, and with 1 024 one-env groups; stats() / metrics(), per group and in total, against the oracle's finished
episodes; the bounds of the statistics (budgets and squared lengths past int32 in whole tiles that end in one step, the
visit counters at the longest horizon), with and without groups; and the refusal of the values past each bound."""
import ctypes as C

import numpy as np
import pytest

import sy_oracle as so
from test_gpu_group_rules import _absent
from test_gpu_parity import _compare_out, _compare_state

pytestmark = pytest.mark.gpu

N, E, P, T = 40, 70, 15, 12  # the handle: 15 police (16 agents), horizon 12
BIG = 2 ** 31 - 1
MAX_TOLL = 1048576
W_ODD = dict(so.DEFAULT_REWARD_WEIGHTS, Police_distance=0.0, Police_group=-0.7, Police_position=1e6, Mrx_closest=1 / 3,
             Mrx_average=-1e6, Mrx_position=0.1, Police_coverage=-0.3, Police_proximity=1e-7, Police_overlap_penalty=2.5)
W_ZERO = {k: 0.0 for k in so.REWARD_WEIGHT_NAMES}
# every key at its edges; complete dicts, so that the oracle's configs can be built from them
EDGE_MECHS = [
    dict(number_of_agents=1, max_timestep=0, agent_money=0, tolls=0, reveal_interval=0, reveal_skip_prob=0.0,
         reward_weights=W_ZERO),
    dict(number_of_agents=15, max_timestep=1, agent_money=1, tolls=5000, reveal_interval=1, reveal_skip_prob=0.5,
         reward_weights=W_ODD),  # a toll above every budget (MrX's 1000 too): nobody ever moves
    dict(number_of_agents=7, max_timestep=T, agent_money=BIG, tolls=MAX_TOLL, reveal_interval=7, reveal_skip_prob=1.0,
         reward_weights=W_ODD),
    dict(number_of_agents=3, max_timestep=T, agent_money=40, tolls=2, reveal_interval=1, reveal_skip_prob=0.5,
         reward_weights=so.DEFAULT_REWARD_WEIGHTS),
    dict(number_of_agents=15, max_timestep=5, agent_money=BIG, tolls=0, reveal_interval=7, reveal_skip_prob=0.0,
         reward_weights=dict(W_ODD, Mrx_time=-2.0, Police_time=1e6)),
    dict(number_of_agents=2, max_timestep=1, agent_money=6, tolls=1, reveal_interval=0, reveal_skip_prob=1.0,
         reward_weights=W_ZERO),
]
AGENT_NAMES = ["pos", "money", "agent_budget", "reward", "reward64", "terminated", "truncated", "done_flags",
               "action_mask", "node_features"]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _pkg():
    import student_mechanism_design_b200 as pkg

    return pkg


def _ocfg(m, mode, tables, belief=True):
    return so.OracleConfig(num_police=m["number_of_agents"], agent_money=m["agent_money"], toll=m["tolls"],
                           reward_weights=dict(m["reward_weights"]), reward_mode=mode, max_timestep=m["max_timestep"],
                           reveal_interval=m["reveal_interval"], reveal_skip_prob=m["reveal_skip_prob"], belief=belief,
                           exp_table=tables[0], cov_table=tables[1])


def _grouped(torch, B, mechs, gid, mode, seed=7, nf_dtype="float32", G=3):
    """a grouped 15-police handle and the per-env oracle of the same batch"""
    pkg = _pkg()
    pool = pkg.generate_graph_pool(G, N, E, seed=4)
    tables = pkg.env.numpy_reward_tables(T)
    w = {k: torch.tensor(v, dtype=torch.float32) for k, v in so.DEFAULT_REWARD_WEIGHTS.items()} if mode == "fp32" else None
    env = pkg.BatchedScotlandYardEnv(B, P, 10, reward_weights=w, graphs=pool, seed=seed, auto_reset=True, tolls=1,
                                     reveal_interval=5, max_timestep=T, belief=True, belief_ce=True, keep_reward64=True,
                                     reward_mode=mode, reward_tables=tables, node_features_dtype=getattr(torch, nf_dtype))
    env.set_mechanisms(mechs, group_id=torch.as_tensor(np.asarray(gid, dtype=np.int32)))
    graphs = [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in pool]
    ob = so.OracleGroupBatch.from_seed([_ocfg(m, mode, tables) for m in mechs], gid, P, graphs, B, seed=seed)
    env.reset()
    return env, ob


def _check(env, ob, mechs, gid, mode, tag, dense=True):
    c = {"mode": mode, "kw": {"belief": dense}}
    if dense:
        _compare_state(env, ob, c, tag)
    else:  # deferred: the compact state only (the dense tensors lag one step, checked by the caller)
        for k in ("pos", "money", "timestep", "visits", "mrx_revealed"):
            want = getattr(ob, "revealed" if k == "mrx_revealed" else k)()
            assert np.array_equal(getattr(env, k).cpu().numpy(), want), (tag, k)
        assert np.array_equal(env.episode.cpu().numpy(), np.asarray(ob.episode, dtype=np.int32)), tag
    dev = env.device
    torch = __import__("torch")
    for g, m in enumerate(mechs):
        rows = torch.as_tensor(np.nonzero(np.asarray(gid) == g)[0], dtype=torch.int64, device=dev)
        if len(rows):
            names = AGENT_NAMES if dense else [k for k in AGENT_NAMES if k not in ("action_mask", "node_features")]
            _absent(env, rows, m["number_of_agents"], names, (tag, g))


def _check_out(env, want, mode, tag):
    _compare_out(env, want, {"mode": mode}, tag)


def _dense(ob):
    return ob.masks(), ob.node_features(), ob.belief()


def _check_dense(env, dense, tag):
    mask, nf, bel = dense
    assert np.array_equal(env.action_mask.cpu().numpy(), mask), tag
    assert np.array_equal(env.node_features.cpu().numpy(), nf), tag
    err = np.abs(env.belief_map.cpu().numpy().astype(np.float64) - bel).max()
    assert err <= 1e-6, (tag, err)


def _set_path(env, path):
    if path in ("two_kernels", "bulk"):
        env.set_option("step_kernel", "two_kernels")
        env.set_option("lagged_kernel", "off")
    if path == "bulk":
        env.set_option("writer_path", "bulk")
    elif path == "fused":
        env.set_option("step_kernel", "fused")


def _run(torch, env, ob, mechs, gid, mode, path, steps):
    _check(env, ob, mechs, gid, mode, "reset")
    if path == "graph":  # the replayed one-launch rollout: k steps per replay, the device's step counter
        k = 4
        graph, _ = env.capture_rollout(k)  # (its warm-up runs steps 0 .. k-1)
        for s in range(steps):
            if s >= k and s % k == 0:
                graph.replay()
            want = ob.step(ob.sample_actions(s))
            if s % k == k - 1:
                _check_out(env, want, mode, (path, s))
                _check(env, ob, mechs, gid, mode, (path, s))
        return
    for s in range(steps):
        acts = env.sample_actions(step_counter=s)
        a_h = acts.cpu().numpy()
        assert np.array_equal(a_h, ob.sample_actions(s)), ("sampler", s)
        if path == "deferred":
            before = _dense(ob)
            env.step_deferred(acts)
            want = ob.step(a_h)
            _check_out(env, want, mode, (path, s))
            _check(env, ob, mechs, gid, mode, (path, s), dense=False)
            _check_dense(env, before, (path, "pending", s))  # the dense tensors describe the state before the call
        else:
            env.step(acts)
            want = ob.step(a_h)
            _check_out(env, want, mode, (path, s))
            _check(env, ob, mechs, gid, mode, (path, s))
    if path == "deferred":
        env.flush_observations()
        _check(env, ob, mechs, gid, mode, (path, "flushed"))


def _episode_metrics(fin, budget, tolls_paid, eff_sum=None):
    """src/eval/metrics.py:168-232 straight from the oracle's finished episodes (length, winner, spent, ...)"""
    n = len(fin)
    if n == 0:
        return None
    length, win, spent = fin[:, 0].astype(np.float64), fin[:, 1], fin[:, 2].astype(np.float64)
    mrx = win == so.WINNER_MRX
    pol = win == so.WINNER_POLICE
    return dict(num_episodes=n, mrx_wins=int(mrx.sum()), police_wins=int(pol.sum()), win_rate=mrx.mean(),
                mean_episode_length=length.mean(), mean_budget_spent=spent.mean(),
                mean_budget_efficiency=spent.mean() / budget if eff_sum is None else eff_sum / n,
                mean_tolls_paid=tolls_paid / n, mean_time_to_catch=length[pol].mean() if pol.any() else 0.0,
                mean_survival_time=length[mrx].mean() if mrx.any() else 0.0,
                episode_length_std=length.std(), win_rate_std=float(np.sqrt(mrx.mean() * (1 - mrx.mean()))))


def _check_stats(env, ob, mechs):
    """stats() / metrics(), per group and in total, against the oracle: integers exactly, metrics to 1e-12"""
    total, per = ob.expected_stats()
    assert list(env.stats().values())[:14] == total[:14]
    got = env.stats(by_group=True)
    for g in range(len(mechs)):
        assert list(got[g].values())[:14] == per[g][:14], g
    fin = np.asarray(ob.finished, dtype=np.int64).reshape(-1, 5)
    budgets = [max(m["number_of_agents"] * m["agent_money"], 1) for m in mechs]
    paid = [m["tolls"] * per[g][so.STAT_POLICE_MOVES] for g, m in enumerate(mechs)]
    eff = sum(fin[fin[:, 4] == g][:, 2].sum() / budgets[g] for g in range(len(mechs)))
    wants = [_episode_metrics(fin[fin[:, 4] == g], budgets[g], paid[g]) for g in range(len(mechs))]
    wants.append(_episode_metrics(fin, None, sum(paid), eff_sum=eff))
    for want, have in zip(wants, env.metrics(by_group=True) + [env.metrics()]):
        if want is None:
            assert have["num_episodes"] == 0
            continue
        for k, v in want.items():
            assert have[k] == pytest.approx(v, rel=1e-12, abs=1e-12 if "std" not in k else 1e-9), k
    ces, cg = np.asarray(ob.belief_ces), np.asarray(ob.ce_groups)
    for g, m in enumerate(env.metrics(by_group=True)):
        if (cg == g).any():
            assert m["mean_belief_ce"] == pytest.approx(ces[cg == g].mean(), rel=1e-5, abs=1e-6), g


# ------------------------------------------------------------------------------------------ 1 + 2: every step path
@pytest.mark.parametrize("mode", ["fp64", "fp32"])
@pytest.mark.parametrize("path", ["two_kernels", "fused", "deferred", "graph", "bulk"])
def test_edge_groups_follow_the_oracle(torch_cuda, path, mode):
    """a ragged batch of 100 envs (three tiles and four envs), groups assigned at random, 20 steps (episodes of every
    group end and restart); then the statistics and metrics"""
    torch = torch_cuda
    B = 100
    gid = np.random.default_rng(11).integers(0, len(EDGE_MECHS), B).astype(np.int32)
    env, ob = _grouped(torch, B, EDGE_MECHS, gid, mode, nf_dtype="uint8" if path == "bulk" else "float32")
    _set_path(env, path)
    _run(torch, env, ob, EDGE_MECHS, gid, mode, path, 20)
    _check_stats(env, ob, EDGE_MECHS)
    total, per = ob.expected_stats()
    assert all(v[so.STAT_EPISODES] > 0 for v in per if v[so.STAT_ENV_STEPS])
    assert per[2][so.STAT_POLICE_MOVES] > 0 and total[so.STAT_TRUNCATIONS] > 0 and total[so.STAT_OUT_OF_MONEY] > 0
    env.close()


def test_1024_one_env_groups(torch_cuda):
    """1 024 groups drawn at random from the edge values, one env each (plus a few shared), assigned at random"""
    torch = torch_cuda
    rng = np.random.default_rng(5)
    mechs = []
    for _ in range(1024):
        m = {k: EDGE_MECHS[rng.integers(len(EDGE_MECHS))][k] for k in EDGE_MECHS[0]}
        if m["tolls"] > m["agent_money"] and m["tolls"] == MAX_TOLL:  # keep SY_MAX_TOLL with a budget that pays it
            m["agent_money"] = BIG
        mechs.append(m)
    B = 1100
    gid = np.concatenate([rng.permutation(1024), rng.integers(0, 1024, B - 1024)]).astype(np.int32)
    env, ob = _grouped(torch, B, mechs, gid, "fp64")
    _run(torch, env, ob, mechs, gid, "fp64", "two_kernels", 10)
    _check_stats(env, ob, mechs)
    env.close()


# ------------------------------------------------------------------------------------------ 3: bounds
def _island_graph(n, weight, seed):
    """node 0 and node 1 isolated (MrX, and a police that never moves); nodes 2 .. n-1 a ring with chords"""
    rng = np.random.default_rng(seed)
    ring = [(i, i + 1) for i in range(2, n - 1)] + [(n - 1, 2)]
    chords = [(i, i + 3) for i in range(2, n - 3, 2)]
    links = np.asarray(ring + chords, dtype=np.int32)
    w = np.full(len(links), weight) if weight else rng.integers(1, 5, len(links))
    return links, w.astype(np.int64)


def _island_env(torch, B, p, money, toll, horizon, graph, groups, mode="fp64"):
    """B envs on the island graph that end only by timeout, in the same step; `groups`: the mechanism is set as the
    one group of a handle with other constructor values, and the last env is in a second, idle group (so that the first
    tile holds 32 envs of the mechanism)"""
    pkg = _pkg()
    n = graph[0].max() + 1
    spec = pkg.GraphSpec(int(n), graph[0], graph[1])
    tables = pkg.env.numpy_reward_tables(horizon)
    kw = dict(graphs=[spec], seed=3, auto_reset=False, keep_reward64=True, reward_mode=mode, reward_tables=tables)
    if groups:
        env = pkg.BatchedScotlandYardEnv(B, p, 10, tolls=1, max_timestep=horizon, **kw)
        mech = dict(agent_money=money, tolls=toll, max_timestep=horizon)
        gid = np.zeros(B, dtype=np.int32)
        gid[-1] = 1
        env.set_mechanisms([mech, dict(agent_money=10, tolls=1, max_timestep=0)], group_id=torch.as_tensor(gid))
    else:
        env = pkg.BatchedScotlandYardEnv(B, p, money, tolls=toll, max_timestep=horizon, **kw)
        gid = None
    starts = np.zeros((B, p + 1), dtype=np.int32)
    starts[:, 1] = 1
    rng = np.random.default_rng(B + p)
    for b in range(B):
        starts[b, 2:] = 2 + rng.permutation(int(n) - 2)[: p - 1]
    env.reset(init_pos=starts)
    return env, spec, starts, gid, tables


@pytest.mark.parametrize("groups", [False, True])
@pytest.mark.parametrize("p", [6, 15])
def test_budget_sums_past_int32(torch_cuda, p, groups):
    """budget 2^31 - 1, toll SY_MAX_TOLL, weight-255 edges (the largest per-step charge), horizon 250: every env of the
    two tiles times out in the same step having spent up to 14 x 252 x (255 + SY_MAX_TOLL) ~ 3.7e9; the statistics
    against the oracle's episodes"""
    torch = torch_cuda
    B, horizon = 64, 250
    graph = _island_graph(p + 16, 255, p)
    env, spec, starts, gid, tables = _island_env(torch, B, p, BIG, MAX_TOLL, horizon, graph, groups)
    ocfg = so.OracleConfig(num_police=p, agent_money=BIG, toll=MAX_TOLL, max_timestep=horizon, exp_table=tables[0],
                           cov_table=tables[1])
    og = [so.Graph(spec.num_nodes, spec.edge_links, spec.edges)]
    if groups:
        idle = so.OracleConfig(num_police=p, agent_money=10, toll=1, max_timestep=0, exp_table=tables[0], cov_table=tables[1])
        ob = so.OracleGroupBatch([ocfg, idle], gid, p, og, [0] * B, starts, seed=3)
    else:
        ob = so.OracleBatch(ocfg, og, [0] * B, starts, seed=3)
    L = horizon + 2
    for chunk in (100, 100, L - 200):
        env.rollout_random(chunk)
    for s in range(L):
        want = ob.step(ob.sample_actions(s))
    _check_out(env, want, "fp64", "end")
    assert np.array_equal(env.pos.cpu().numpy(), ob.pos()) and np.array_equal(env.money.cpu().numpy(), ob.money())
    total, per = ob.expected_stats()
    main = per[0]
    assert main[so.STAT_TRUNCATIONS] == main[so.STAT_EPISODES] == B - int(groups)
    assert main[so.STAT_SUM_EPISODE_BUDGET_SPENT] > 2 ** 32  # past int32 in every tile
    assert list(env.stats().values())[:13] == total[:13]
    if groups:
        got = env.stats(by_group=True)
        assert [list(g.values())[:13] for g in got] == [v[:13] for v in per]
    env.close()


def _c_reference(graph, starts, p, money, horizon, steps):
    """the C oracle over `steps` random steps: final state, the rewards of the last step, the raw int32 visit counters
    and the police moves (position changes) -- it records no episodes"""
    import sy_oracle_c as soc

    B = starts.shape[0]
    og = [so.Graph(int(graph[0].max() + 1), graph[0], graph[1])]
    cb = soc.CBatch(so.OracleConfig(num_police=p, agent_money=money, max_timestep=horizon), og, B, seed=3,
                    auto_reset=False, start_positions=starts, graph_id=np.zeros(B, np.int32), with_obs=False)
    moves, want = np.zeros(B, np.int64), None
    prev = cb.pos()
    for s in range(steps):
        want = cb.step(cb.sample_actions(s))
        cur = cb.pos()
        moves += (cur[:, 1:] != prev[:, 1:]).sum(axis=1)
        prev = cur
    return cb, want, moves


@pytest.mark.parametrize("groups", [False, True])
@pytest.mark.parametrize("horizon", [8191, 65533])
def test_long_horizons(torch_cuda, horizon, groups):
    """horizon 8 191 (length 8 193: 32 squared lengths past int32) and SY_MAX_TIMESTEP (length 65 535: one squared
    length past int32), one tile ending in one step; the parked police's visit counter reaches 65 535 exactly, and the
    coverage term of the last running step equals the C oracle's"""
    torch = torch_cuda
    B, p, money = 32 + int(groups), 3, 10 ** 6
    graph = _island_graph(12, 0, 1)
    env, spec, starts, gid, _ = _island_env(torch, B, p, money, 0, horizon, graph, groups)
    L = horizon + 2
    done = 0
    while done < L - 1:  # every step but the last in chunks, then the last one alone
        k = min(4096, L - 1 - done)
        env.rollout_random(k)
        done += k
    main = np.ones(B, bool) if gid is None else gid == 0
    cb, want, moves = _c_reference(graph, starts, p, money, horizon, L - 1)
    r = env.reward64.cpu().numpy()
    assert r[main].tobytes() == want["reward"][main].tobytes()  # the shaped rewards of the last running step
    vis = env.visits.cpu().numpy().astype(np.int64)
    assert np.array_equal(vis[main], cb._visits[main]) and (vis[main, 1] == L - 1).all()
    env.rollout_random(1)
    prev = cb.pos()
    want = cb.step(cb.sample_actions(L - 1))
    moves += (cb.pos()[:, 1:] != prev[:, 1:]).sum(axis=1)
    assert want["truncated"][main].all()
    assert (env.visits.cpu().numpy()[main, 1] == L).all() and (cb._visits[main, 1] == L).all()  # 65 535 at the bound
    pos, mon = env.pos.cpu().numpy(), env.money.cpu().numpy()
    assert np.array_equal(pos[main], cb.pos()[main]) and np.array_equal(mon[main], cb.money()[main])
    nb = int(main.sum())
    spent = p * money * nb - int(cb.money()[main][:, 1:].astype(np.int64).sum())
    st = env.stats(by_group=True)[0] if groups else env.stats()
    assert st["episodes"] == st["truncations"] == st["mrx_wins"] == nb
    assert st["env_steps"] == nb * L
    assert st["sum_episode_length"] == nb * L and st["sum_length_mrx_wins"] == nb * L
    assert st["sum_sq_episode_length"] == nb * L * L
    assert st["sum_episode_budget_spent"] == st["sum_budget_spent"] == spent
    assert st["police_moves"] == int(moves[main].sum()) > 0
    env.close()


def test_values_past_each_bound_are_refused(torch_cuda):
    """sy_create refuses toll SY_MAX_TOLL + 1 and max_timestep SY_MAX_TIMESTEP + 1 (straight through the C ABI, past the
    host checks), and accepts both bounds"""
    pkg = _pkg()
    from student_mechanism_design_b200 import _cabi

    lib = _cabi.load_library()

    def create(**kw):
        cfg = _cabi.SyConfig()
        cfg.struct_bytes = C.sizeof(_cabi.SyConfig)
        cfg.device, cfg.num_envs, cfg.num_nodes, cfg.num_police = 0, 4, 10, 2
        cfg.agent_money, cfg.mrx_money, cfg.max_timestep = 10, 1000, 250
        for k, v in kw.items():
            setattr(cfg, k, v)
        h = C.c_void_p()
        rc = lib.sy_create(C.byref(cfg), C.byref(h))
        if rc == 0:
            lib.sy_destroy(h)
        return rc, lib.sy_last_error().decode()

    assert create(toll=_cabi.SY_MAX_TOLL)[0] == 0 and create(max_timestep=_cabi.SY_MAX_TIMESTEP)[0] == 0
    rc, msg = create(toll=_cabi.SY_MAX_TOLL + 1)
    assert rc == 1 and "toll" in msg and str(_cabi.SY_MAX_TOLL) in msg
    rc, msg = create(toll=BIG)
    assert rc == 1 and "toll" in msg
    rc, msg = create(max_timestep=_cabi.SY_MAX_TIMESTEP + 1)
    assert rc == 1 and "max_timestep" in msg and str(_cabi.SY_MAX_TIMESTEP) in msg
    with pytest.raises(ValueError, match="tolls"):
        pkg.BatchedScotlandYardEnv(4, 2, 10, tolls=_cabi.SY_MAX_TOLL + 1, graph_nodes=10, graph_edges=12)
    with pytest.raises(ValueError, match="max_timestep"):
        pkg.BatchedScotlandYardEnv(4, 2, 10, max_timestep=_cabi.SY_MAX_TIMESTEP + 1, graph_nodes=10, graph_edges=12)
    # the groups are bounded by the handle's values
    env = pkg.BatchedScotlandYardEnv(4, 2, 10, max_timestep=_cabi.SY_MAX_TIMESTEP, graph_nodes=10, graph_edges=12)
    with pytest.raises(ValueError, match="max_timestep"):
        env.set_mechanisms([{"max_timestep": _cabi.SY_MAX_TIMESTEP + 1}])
    with pytest.raises(ValueError, match="tolls"):
        env.set_mechanisms([{"tolls": _cabi.SY_MAX_TOLL + 1}])
    env.close()
