"""Mechanism groups (sy_set_groups / sy_group_stats, env.set_mechanisms): one handle evaluating several mechanisms.

Checked here: a group equal to the handle's config changes no byte of any output, through every step path; envs of a
group with its own weights / budget / reveal schedule follow exactly the trajectory of an ungrouped handle with that
config (Philox is keyed by the global env index alone), for interleaved, random and contiguous assignments; the
per-group statistics equal the statistics of those separate handles and sum to the handle-wide vector; two half
shards with the default assignment add up to the full batch; the lifecycle errors; metrics(by_group=True); the
out-of-bounds canaries."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, E, P, MONEY = 40, 60, 3, 10
BELIEF_TOL = 1e-6
STATE = ["pos", "money", "timestep", "graph_id", "episode", "done", "visits", "agent_budget", "mrx_revealed"]
RESULT = ["reward", "reward64", "terminated", "truncated", "done_flags", "winner", "status"]
DENSE = ["action_mask", "node_features"]

MECHS = [
    dict(reward_weights={"Police_time": 0.5, "Mrx_time": -0.25, "Police_distance": 0.7}, agent_money=0, reveal_interval=0),
    dict(reward_weights={"Mrx_closest": 1.5, "Police_overlap_penalty": 0.3}, agent_money=1, reveal_interval=3),
    dict(agent_money=4, reveal_interval=5),
    dict(reward_weights={"Police_time": 0.125, "Mrx_time": 0.75}, agent_money=20, reveal_interval=3),
    dict(reward_weights={"Police_coverage": 2.0}, agent_money=MONEY, reveal_interval=5, reveal_skip_prob=0.5),
]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _pool():
    import student_mechanism_design_b200 as pkg

    return pkg.generate_graph_pool(2, N, E, seed=0)


def _env(B, pool, *, money=MONEY, reveal=5, weights=None, skip=0.0, env_offset=0, reward_mode="fp64", **kw):
    import student_mechanism_design_b200 as pkg

    return pkg.BatchedScotlandYardEnv(B, P, money, reward_weights=weights, graphs=pool, seed=7, auto_reset=True, tolls=1,
                                      belief=True, belief_ce=True, reveal_interval=reveal, keep_reward64=True,
                                      reward_mode=reward_mode, reveal_skip_prob=skip, env_offset=env_offset, **kw)


def _config_of(mech):
    """constructor arguments of an ungrouped handle that runs mechanism `mech`"""
    import student_mechanism_design_b200 as pkg

    w = dict(pkg.DEFAULT_REWARD_WEIGHTS)
    w.update(mech.get("reward_weights", {}))
    return dict(money=mech.get("agent_money", MONEY), reveal=mech.get("reveal_interval", 5), weights=w,
                skip=mech.get("reveal_skip_prob", 0.0))


def _rows(env, names, rows=None):
    out = {}
    for k in names:
        t = getattr(env, k)
        if t is None:
            continue
        a = t.cpu().numpy()
        out[k] = a if rows is None else a[rows]
    return out


def _equal(a, b, tag):
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, (tag, k)
        if a[k].tobytes() != b[k].tobytes():  # bytes: float64 rewards compared bit for bit
            bad = np.argwhere(a[k] != b[k])
            raise AssertionError(f"{tag} {k}: {len(bad)} mismatches, first at {bad[:1].tolist()}")


def _belief_close(a, b, tag, tol=BELIEF_TOL):
    err = np.abs(a.belief_map.cpu().numpy().astype(np.float64) - b.belief_map.cpu().numpy().astype(np.float64)).max()
    assert err <= tol, (tag, "belief_map", err)


def _set_path(env, path):
    if path == "two_kernels":
        env.set_option("step_kernel", "two_kernels")
        env.set_option("lagged_kernel", "off")
    elif path == "fused":
        env.set_option("step_kernel", "fused")


def _lockstep(ref, grp, steps, path, tag, dense_exact):
    """step both envs with the same sampled actions through `path` and compare everything after every step"""
    ref.reset()
    grp.reset()
    _equal(_rows(ref, STATE + DENSE), _rows(grp, STATE + DENSE), (tag, "reset"))
    if path == "graph":
        g1, _ = ref.capture_rollout(5)
        g2, _ = grp.capture_rollout(5)
        for r in range(steps // 5):
            g1.replay()
            g2.replay()
            _equal(_rows(ref, STATE + RESULT + DENSE), _rows(grp, STATE + RESULT + DENSE), (tag, "replay", r))
            _belief_close(ref, grp, (tag, r), 0.0 if dense_exact else BELIEF_TOL)
        return
    for s in range(steps):
        a1, a2 = ref.sample_actions(step_counter=s), grp.sample_actions(step_counter=s)
        assert np.array_equal(a1.cpu().numpy(), a2.cpu().numpy()), (tag, "sampler", s)
        if path == "deferred":
            ref.step_deferred(a1)
            grp.step_deferred(a2)
            _equal(_rows(ref, STATE + RESULT), _rows(grp, STATE + RESULT), (tag, "deferred", s))
        else:
            ref.step(a1)
            grp.step(a2)
            _equal(_rows(ref, STATE + RESULT + DENSE), _rows(grp, STATE + RESULT + DENSE), (tag, s))
            _belief_close(ref, grp, (tag, s), 0.0 if dense_exact else BELIEF_TOL)
    ref.flush_observations()
    grp.flush_observations()
    _equal(_rows(ref, STATE + DENSE), _rows(grp, STATE + DENSE), (tag, "flushed"))
    _belief_close(ref, grp, (tag, "flushed"), 0.0 if dense_exact else BELIEF_TOL)


@pytest.mark.parametrize("reward_mode", ["fp64", "fp32"])
@pytest.mark.parametrize("path", ["two_kernels", "fused", "deferred", "graph"])
@pytest.mark.parametrize("C", [1, 7])
def test_identity_groups_change_nothing(torch_cuda, C, path, reward_mode):
    """C groups equal to the config, interleaved: byte-equal to a handle without groups, both handles running `path`
    (two-kernel step, fused step, deferred steps through the lagged kernel, replayed one-launch rollout graph) --
    the grouped handle through the GROUPS instantiation of that path -- statistics included"""
    torch = torch_cuda
    pool = _pool()
    B = 997
    w = None
    if reward_mode == "fp32":
        import student_mechanism_design_b200 as pkg

        w = {k: torch.tensor(v, dtype=torch.float32) for k, v in pkg.DEFAULT_REWARD_WEIGHTS.items()}
    ref, grp = _env(B, pool, weights=w, reward_mode=reward_mode), _env(B, pool, weights=w, reward_mode=reward_mode)
    _set_path(ref, path)
    _set_path(grp, path)
    grp.set_mechanisms([{}] * C)
    assert grp.mechanisms[0]["agent_money"] == MONEY and grp.group_id.shape == (B,)
    _lockstep(ref, grp, 60, path, (C, path, reward_mode), dense_exact=True)
    assert ref.stats() == grp.stats()
    per = grp.stats(by_group=True)
    assert len(per) == C
    assert {k: sum(g[k] for g in per) for k in per[0]} == grp.stats()


def _against_separate_handles(torch, B, gid, steps, tag):
    """grouped handle with MECHS and assignment gid vs one ungrouped handle per mechanism, same seed and offset: env b
    of the grouped handle must follow env b of handle gid[b]"""
    pool = _pool()
    grp = _env(B, pool)
    grp.set_mechanisms(MECHS, group_id=torch.as_tensor(gid, dtype=torch.int32))
    refs = [_env(B, pool, **_config_of(m)) for m in MECHS]
    grp.reset()
    for r in refs:
        r.reset()
    counts = [dict.fromkeys(COUNTED, 0) for _ in MECHS]  # per group, aggregated on the host from per-env outcomes
    for s in range(steps):
        acts = grp.sample_actions(step_counter=s)
        grp.step(acts)
        got = _rows(grp, STATE + RESULT + DENSE)
        bel = grp.belief_map.cpu().numpy()
        for g, r in enumerate(refs):
            rows = np.nonzero(gid == g)[0]
            ra = r.sample_actions(step_counter=s)
            assert np.array_equal(ra.cpu().numpy()[rows], acts.cpu().numpy()[rows]), (tag, "sampler", g, s)
            t_before = r.timestep.cpu().numpy()[rows]
            r.step(ra)
            _count(counts[g], t_before, r.status.cpu().numpy()[rows], r.winner.cpu().numpy()[rows])
            want = _rows(r, STATE + RESULT + DENSE, rows)
            _equal({k: v[rows] for k, v in got.items()}, want, (tag, g, s))
            err = np.abs(bel[rows].astype(np.float64) - r.belief_map.cpu().numpy()[rows].astype(np.float64)).max()
            assert err <= BELIEF_TOL, (tag, g, s, err)
    return grp, refs, counts


# statistics that follow from the per-env outcomes alone (auto-reset: every env steps every step)
COUNTED = ["env_steps", "episodes", "mrx_wins", "police_wins", "truncations", "out_of_money", "sum_episode_length",
           "sum_sq_episode_length", "sum_length_police_wins", "sum_length_mrx_wins"]


def _count(c, t_before, status, winner):
    fin = (status & 3) != 0  # SY_STATUS_TERMINATED | SY_STATUS_TRUNCATED
    length = (t_before + 1).astype(np.int64)
    c["env_steps"] += len(status)
    c["episodes"] += int(fin.sum())
    c["mrx_wins"] += int((fin & (winner == 1)).sum())
    c["police_wins"] += int((fin & (winner == 2)).sum())
    c["truncations"] += int(((status & 2) != 0).sum())
    c["out_of_money"] += int((((status & 1) != 0) & (winner == 1)).sum())
    c["sum_episode_length"] += int(length[fin].sum())
    c["sum_sq_episode_length"] += int((length[fin] ** 2).sum())
    c["sum_length_police_wins"] += int(length[fin & (winner == 2)].sum())
    c["sum_length_mrx_wins"] += int(length[fin & (winner == 1)].sum())


@pytest.mark.parametrize("assign", ["modulo", "random"])
def test_distinct_groups_follow_their_config(torch_cuda, assign):
    """five different mechanisms (non-zero *_time weights, budgets 0 / 1 / 4 / 20, reveal 0 / 3 / 5) on a ragged
    batch, assigned b % C and at random, 60 steps"""
    B = 4099
    C = len(MECHS)
    gid = np.arange(B) % C if assign == "modulo" else np.random.default_rng(3).integers(0, C, B)
    grp, refs, counts = _against_separate_handles(torch_cuda, B, gid.astype(np.int32), 60, assign)
    # per-group statistics against the outcomes of the group's envs, aggregated on the host: a statistic credited to
    # the wrong group of a mixed warp shows here
    per = grp.stats(by_group=True)
    for g in range(C):
        assert {k: per[g][k] for k in COUNTED} == counts[g], (assign, g)
    assert sum(c["episodes"] for c in counts) > 0 and all(c["env_steps"] > 0 for c in counts)
    assert {k: sum(x[k] for x in per) for k in per[0]} == grp.stats()
    m = grp.metrics(by_group=True)
    assert len(m) == C and set(m[0]) == set(grp.metrics())
    for g in range(C):
        c = counts[g]
        assert (m[g]["num_episodes"], m[g]["mrx_wins"], m[g]["police_wins"]) == (c["episodes"], c["mrx_wins"], c["police_wins"])
        if c["episodes"]:
            assert m[g]["mean_episode_length"] == c["sum_episode_length"] / c["episodes"]


def test_decomposition_contiguous_blocks(torch_cuda):
    """contiguous group blocks on one graph (different reveal_skip_prob included) vs C handles with env_offset = block
    start: outputs byte-equal; stats(by_group=True)[g] == handle g's stats(); sum over groups == stats()"""
    torch = torch_cuda
    import student_mechanism_design_b200 as pkg

    pool = pkg.generate_graph_pool(1, N, E, seed=0)
    sizes = [96, 64, 160, 33, 200]
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    B = int(sum(sizes))
    gid = np.repeat(np.arange(len(sizes)), sizes).astype(np.int32)
    mechs = [dict(m, reveal_skip_prob=p) for m, p in zip(MECHS, [0.0, 0.25, 0.5, 0.0, 0.9])]
    grp = _env(B, pool)
    grp.set_mechanisms(mechs, group_id=torch.as_tensor(gid))
    refs = [_env(n, pool, env_offset=int(s), **_config_of(m)) for n, s, m in zip(sizes, starts, mechs)]
    grp.reset()
    for r in refs:
        r.reset()
    for s in range(60):
        grp.step(grp.sample_actions(step_counter=s))
        got = _rows(grp, STATE + RESULT + DENSE + ["belief_map"])
        for g, r in enumerate(refs):
            r.step(r.sample_actions(step_counter=s))
            sl = slice(int(starts[g]), int(starts[g]) + sizes[g])
            _equal({k: v[sl] for k, v in got.items()}, _rows(r, STATE + RESULT + DENSE + ["belief_map"]), ("block", g, s))
    per = grp.stats(by_group=True)
    for g, r in enumerate(refs):
        assert per[g] == r.stats(), g
    assert {k: sum(x[k] for x in per) for k in per[0]} == grp.stats()


def test_shards_sum_to_full_batch(torch_cuda):
    """two half handles with the default assignment ((env_offset + b) % C), summed per group, equal one full handle"""
    pool = _pool()
    B, C = 2048, 16
    mechs = [dict(agent_money=4 + g, reveal_interval=g % 4) for g in range(C)]
    full, lo, hi = _env(B, pool), _env(B // 2, pool), _env(B // 2, pool, env_offset=B // 2)
    for e in (full, lo, hi):
        e.set_mechanisms(mechs)
        e.reset()
        e.rollout_random(40, step_counter=0)
    f = full.stats(by_group=True)
    a, b = lo.stats(by_group=True), hi.stats(by_group=True)
    assert [{k: x[k] + y[k] for k in x} for x, y in zip(a, b)] == f
    assert np.array_equal(full.pos.cpu().numpy(), np.concatenate([lo.pos.cpu().numpy(), hi.pos.cpu().numpy()]))


def test_lifecycle_and_errors(torch_cuda):
    torch = torch_cuda
    import ctypes as C

    import student_mechanism_design_b200 as pkg
    from student_mechanism_design_b200 import _cabi

    pool = _pool()
    B = 256
    env, fresh = _env(B, pool), _env(B, pool)
    env.reset()
    env.set_mechanisms(MECHS)
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):  # the library's text: a full reset is owed
        env.step(env.sample_actions())
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):
        _cabi.check(env._lib.sy_rollout_random(env._handle, 2, 0, env.sample_actions().data_ptr(), C.byref(env._state),
                                               C.byref(env._obs), C.byref(env._out), env._stream()))
    part = torch.ones(B, dtype=torch.bool)
    part[B // 2:] = False
    with pytest.raises(pkg.SyError, match="cover every env"):  # a partial reset is refused in Python ...
        env.reset(reset_mask=part)
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):  # ... and does not count in the library
        m = part.to(device=env.device, dtype=torch.uint8)
        _cabi.check(env._lib.sy_reset(env._handle, m.data_ptr(), None, None, 0, C.byref(env._state), C.byref(env._obs),
                                      env._stream()))
        env.step(env.sample_actions())
    env.reset()
    env.step(env.sample_actions())

    def raw(groups, ids=None, n=None):
        arr = (_cabi.SyGroup * max(len(groups), 1))(*groups)
        return _cabi.check(env._lib.sy_set_groups(env._handle, len(groups) if n is None else n, arr,
                                                  None if ids is None else ids.data_ptr(), env._stream()))

    good = pkg.env.pack_mechanism({}, env)
    cases = []
    g = pkg.env.pack_mechanism({}, env); g.struct_bytes = 8; cases.append(([g], None, "SyGroup size mismatch"))
    g = pkg.env.pack_mechanism({}, env); g.agent_money = -1; cases.append(([g], None, "negative agent_money"))
    g = pkg.env.pack_mechanism({}, env); g.reveal_interval = -2; cases.append(([g], None, "negative agent_money / reveal_interval"))
    g = pkg.env.pack_mechanism({}, env); g.reveal_skip_prob = 1.5; cases.append(([g], None, "reveal_skip_prob"))
    g = pkg.env.pack_mechanism({}, env); g.reward_weights[3] = float("nan"); cases.append(([g], None, "not finite"))
    cases.append(([good, good], torch.full((B,), 2, dtype=torch.int32, device=env.device), "group ids outside"))
    cases.append(([good], None, "num_groups must be in"))
    for groups, ids, msg in cases:
        with pytest.raises(pkg.SyError, match=msg):
            raw(groups, ids, n=2000 if msg.startswith("num_groups") else None)
    # the rejected calls kept the groups: steps still run, per-group statistics still fold with C = 5
    env.step(env.sample_actions())
    with pytest.raises(pkg.SyError, match="sy_group_stats"):
        _cabi.check(env._lib.sy_group_stats(env._handle, 3, env.group_stats_vec.data_ptr(), env._stream()))
    assert len(env.stats(by_group=True)) == len(MECHS)
    sd = env.state_dict()
    assert "group_id" in sd and "group_stats_vec" in sd
    # clearing: bit-identical to a fresh handle from the next full reset on
    env.set_mechanisms(None)
    assert env.mechanisms is None and env.group_id is None and "group_id" not in env.state_dict()
    env.reset(restart=True)
    fresh.reset()
    for s in range(30):
        env.step(env.sample_actions(step_counter=s))
        fresh.step(fresh.sample_actions(step_counter=s))
        _equal(_rows(env, STATE + RESULT + DENSE + ["belief_map"]), _rows(fresh, STATE + RESULT + DENSE + ["belief_map"]), ("cleared", s))


def test_packing_rejects_bad_dicts(torch_cuda):
    pool = _pool()
    env = _env(64, pool)
    for bad, exc in [({"agent_money": -1}, ValueError), ({"reveal_interval": 1.5}, ValueError),
                     ({"reveal_skip_prob": 2.0}, ValueError), ({"reward_weights": {"nope": 1.0}}, KeyError),
                     ({"toll": 1}, KeyError), ({"reward_weights": {"Mrx_time": float("inf")}}, ValueError)]:
        with pytest.raises(exc):
            env.set_mechanisms([bad])
    with pytest.raises(ValueError):
        env.set_mechanisms([])


def test_replay_after_new_groups_is_refused(torch_cuda):
    """a rollout graph captured under other groups must be recaptured; the recaptured one runs the new groups"""
    import student_mechanism_design_b200 as pkg

    pool = _pool()
    env = _env(500, pool)
    env.reset()
    graph, _ = env.capture_rollout(4)
    graph.replay()
    env.set_mechanisms(MECHS)
    with pytest.raises(pkg.SyError, match="capture it again"):
        graph.replay()
    env.reset(reset_mask=torch_cuda.ones(500, dtype=torch_cuda.bool, device=env.device))  # an all-set mask is a full reset
    graph, _ = env.capture_rollout(4)
    graph.replay()
    env.set_mechanisms([dict(agent_money=3)])
    with pytest.raises(pkg.SyError, match="capture it again"):
        graph.replay()
    env.reset()
    graph, _ = env.capture_rollout(4)
    graph.replay()
    assert len(env.stats(by_group=True)) == 1


def test_guards_with_groups(torch_cuda):
    pool = _pool()
    env = _env(333, pool, guard_bytes=4096)
    env.set_mechanisms(MECHS)
    env.reset()
    for s in range(20):
        env.step(env.sample_actions(step_counter=s))
    env.rollout_random(10)
    env.stats(by_group=True)
    env.check_guards()
