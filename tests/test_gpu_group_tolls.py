"""Per-group tolls (sy_set_group_tolls, the `tolls` key of env.set_mechanisms): each env pays its mechanism group's toll
in every place a move's legality is decided.

Checked here: tolls equal to the config change no byte of any output through every step path; envs of groups with
their own tolls (and budgets) follow exactly the trajectory of an ungrouped handle built with that toll -- state,
results, action_mask, node_features and sampled actions after every step, the belief map to 1e-6 -- on ragged, mixed
batches and on the paths the small case does not reach (mixed graphs in a tile, 1-row mask images, batches over one
wave, the one-launch rollout, the host-buffer calls, the benchmarked shapes); per-group statistics and mean_tolls_paid;
shards; the agents' valid moves; the lifecycle of sy_set_group_tolls; the out-of-bounds canaries."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, E, P, MONEY = 40, 60, 3, 10
BELIEF_TOL = 1e-6
STATE = ["pos", "money", "timestep", "graph_id", "episode", "done", "visits", "agent_budget", "mrx_revealed"]
RESULT = ["reward", "reward64", "terminated", "truncated", "done_flags", "winner", "status"]
DENSE = ["action_mask", "node_features"]
ABOVE = 1000  # a toll above every budget: nobody of that group can ever move
# (toll, agent_money) of the distinct groups
TOLL_MECHS = [dict(tolls=0, agent_money=MONEY), dict(tolls=1, agent_money=4), dict(tolls=2, agent_money=20),
              dict(tolls=3, agent_money=7), dict(tolls=ABOVE, agent_money=MONEY)]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _pool(G=2, n=N, e=E):
    import student_mechanism_design_b200 as pkg

    return pkg.generate_graph_pool(G, n, e, seed=0)


def _env(B, pool, *, toll=1, money=MONEY, p=P, reward_mode="fp64", weights=None, env_offset=0, **kw):
    import student_mechanism_design_b200 as pkg

    kw.setdefault("belief", True)
    kw.setdefault("belief_ce", kw["belief"])
    return pkg.BatchedScotlandYardEnv(B, p, money, reward_weights=weights, graphs=pool, seed=7, auto_reset=True,
                                      tolls=toll, reveal_interval=5, keep_reward64=True, reward_mode=reward_mode,
                                      env_offset=env_offset, **kw)


def _raw_tolls(env, tolls):
    """sy_set_group_tolls straight through the C ABI (returns the status code)"""
    arr = (C.c_int32 * max(len(tolls), 1))(*tolls)
    return env._lib.sy_set_group_tolls(env._handle, len(tolls), arr, env._stream())


def _bits(t):
    """a tensor as integers of the same width, so that floats compare bit for bit"""
    import torch

    if t.dtype in (torch.float32, torch.float64):
        return t.view(torch.int32 if t.dtype == torch.float32 else torch.int64)
    return t


def _equal(grp, ref, names, rows, tag):
    """outputs `names` of `grp` and `ref` equal on `rows` (LongTensor on the device, or None = all), byte for byte"""
    for k in names:
        a, b = getattr(grp, k), getattr(ref, k)
        if a is None:
            assert b is None, (tag, k)
            continue
        if rows is not None:
            a, b = a.index_select(0, rows), b.index_select(0, rows)
        if not _bits(a).equal(_bits(b)):
            bad = (_bits(a) != _bits(b)).nonzero()
            raise AssertionError(f"{tag} {k}: {bad.shape[0]} mismatches, first at {bad[:1].tolist()}")


def _belief_close(grp, ref, rows, tag, tol=BELIEF_TOL):
    if grp.belief_map is None:
        return
    a, b = grp.belief_map, ref.belief_map
    if rows is not None:
        a, b = a.index_select(0, rows), b.index_select(0, rows)
    err = (a.double() - b.double()).abs().max().item() if a.numel() else 0.0
    assert err <= tol, (tag, "belief_map", err)


def _set_path(env, path):
    if path in ("two_kernels", "bulk"):
        env.set_option("step_kernel", "two_kernels")
        env.set_option("lagged_kernel", "off")
    if path == "bulk":
        env.set_option("writer_path", "bulk")
    elif path == "fused":
        env.set_option("step_kernel", "fused")


# ------------------------------------------------------------------------------------------ identity
@pytest.mark.parametrize("reward_mode", ["fp64", "fp32"])
@pytest.mark.parametrize("path", ["two_kernels", "fused", "deferred", "graph", "bulk"])
@pytest.mark.parametrize("toll", [0, 1])
def test_identity_tolls_equal_to_config(torch_cuda, toll, path, reward_mode):
    """three groups whose tolls equal the config's, given explicitly (also straight through sy_set_group_tolls): byte-equal
    to a handle without groups through `path`, statistics included"""
    torch = torch_cuda
    pool = _pool()
    B = 997
    w = None
    if reward_mode == "fp32":
        import student_mechanism_design_b200 as pkg

        w = {k: torch.tensor(v, dtype=torch.float32) for k, v in pkg.DEFAULT_REWARD_WEIGHTS.items()}
    ref, grp = (_env(B, pool, toll=toll, weights=w, reward_mode=reward_mode) for _ in range(2))
    for e in (ref, grp):
        _set_path(e, path)
    grp.set_mechanisms([{"tolls": toll}, {"tolls": float(toll)}, {}])
    assert [m["tolls"] for m in grp.mechanisms] == [toll] * 3 and grp._env_toll is None
    assert _raw_tolls(grp, [toll] * 3) == 0
    ref.reset()
    grp.reset()
    _equal(grp, ref, STATE + DENSE, None, "reset")
    if path == "graph":
        g1, _ = ref.capture_rollout(5)
        g2, _ = grp.capture_rollout(5)
        for r in range(12):
            g1.replay()
            g2.replay()
            _equal(grp, ref, STATE + RESULT + DENSE, None, ("replay", r))
            _belief_close(grp, ref, None, r, 0.0)
    else:
        for s in range(60):
            a1, a2 = ref.sample_actions(step_counter=s), grp.sample_actions(step_counter=s)
            assert a1.equal(a2), ("sampler", s)
            if path == "deferred":
                ref.step_deferred(a1)
                grp.step_deferred(a2)
                _equal(grp, ref, STATE + RESULT, None, ("deferred", s))
            else:
                ref.step(a1)
                grp.step(a2)
                _equal(grp, ref, STATE + RESULT + DENSE, None, s)
                _belief_close(grp, ref, None, s, 0.0)
        ref.flush_observations()
        grp.flush_observations()
        _equal(grp, ref, STATE + DENSE, None, "flushed")
    assert ref.stats() == grp.stats()
    assert ref.metrics()["mean_tolls_paid"] == grp.metrics()["mean_tolls_paid"]


# ------------------------------------------------------------------------------------------ distinct tolls
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


class _Pair:
    """a grouped handle with `mechs` assigned by `gid` and one ungrouped handle per mechanism (its toll and budget),
    same seed and offset: env b of the grouped handle must follow env b of handle gid[b]"""

    def __init__(self, torch, B, mechs, gid, pool, count=False, **kw):
        self.torch, self.B, self.gid = torch, B, np.asarray(gid, dtype=np.int32)
        self.grp = _env(B, pool, **kw)
        self.grp.set_mechanisms(mechs, group_id=torch.as_tensor(self.gid))
        self.refs = [_env(B, pool, toll=m.get("tolls", 1), money=m.get("agent_money", MONEY), **kw) for m in mechs]
        dev = self.grp.device
        self.rows = [torch.as_tensor(np.nonzero(self.gid == g)[0], dtype=torch.int64, device=dev) for g in range(len(mechs))]
        self.counts = [dict.fromkeys(COUNTED, 0) for _ in mechs] if count else None
        for e in [self.grp] + self.refs:
            e.reset()

    @property
    def envs(self):
        return [self.grp] + self.refs

    def compare(self, names, tag, belief=True):
        for g, r in enumerate(self.refs):
            _equal(self.grp, r, names, self.rows[g], (tag, g))
            if belief:
                _belief_close(self.grp, r, self.rows[g], (tag, g))

    def step(self, s, dense=True):
        acts = self.grp.sample_actions(step_counter=s)
        t_before = self.grp.timestep.cpu().numpy() if self.counts is not None else None
        self.grp.step(acts)
        for g, r in enumerate(self.refs):
            ra = r.sample_actions(step_counter=s)
            rows = self.rows[g]
            assert ra.index_select(0, rows).equal(acts.index_select(0, rows)), ("sampler", g, s)
            r.step(ra)
            if self.counts is not None:
                idx = rows.cpu().numpy()
                _count(self.counts[g], t_before[idx], self.grp.status.cpu().numpy()[idx], self.grp.winner.cpu().numpy()[idx])
        self.compare(STATE + RESULT + (DENSE if dense else []), ("step", s), belief=dense)


def _gids(B, C, assign):
    return (np.arange(B) % C if assign == "modulo" else np.random.default_rng(3).integers(0, C, B)).astype(np.int32)


@pytest.mark.parametrize("assign", ["modulo", "random"])
def test_distinct_tolls_follow_their_config(torch_cuda, assign):
    """tolls 0 / 1 / 2 / 3 / above every budget with different budgets on a ragged batch (4 099 envs), assigned b % C
    and at random (every warp mixes tolls), 60 steps; then per-group statistics and mean_tolls_paid"""
    B, C_ = 4099, len(TOLL_MECHS)
    pr = _Pair(torch_cuda, B, TOLL_MECHS, _gids(B, C_, assign), _pool(), count=True)
    for s in range(60):
        pr.step(s)
    grp = pr.grp
    per = grp.stats(by_group=True)
    for g in range(C_):
        assert {k: per[g][k] for k in COUNTED} == pr.counts[g], (assign, g)
    assert all(c["episodes"] > 0 for c in pr.counts)
    assert {k: sum(x[k] for x in per) for k in per[0]} == grp.stats()
    # the group above every budget never moves a police officer and never pays; the others do
    assert per[-1]["police_moves"] == 0 and per[-1]["sum_budget_spent"] == 0
    assert all(per[g]["police_moves"] > 0 for g in range(C_ - 1))
    m = grp.metrics(by_group=True)
    for g, mech in enumerate(TOLL_MECHS):
        assert m[g]["mean_tolls_paid"] == mech["tolls"] * per[g]["police_moves"] / per[g]["episodes"], g
        assert m[g]["num_episodes"] == pr.counts[g]["episodes"]
    paid = sum(mech["tolls"] * per[g]["police_moves"] for g, mech in enumerate(TOLL_MECHS))
    assert grp.metrics()["mean_tolls_paid"] == paid / grp.stats()["episodes"]
    # spending: every police move of group g costs its edge weight plus toll_g
    for g, mech in enumerate(TOLL_MECHS):
        assert per[g]["sum_budget_spent"] >= (1 + mech["tolls"]) * per[g]["police_moves"]


@pytest.mark.parametrize("driver", ["deferred", "rollout", "fused"])
def test_distinct_tolls_in_kernel_draws(torch_cuda, driver):
    """the next-action draw inside the lagged and one-launch rollout kernels (4 099 envs: one CTA per tile, at most one
    per SM), and the fused step, with mixed tolls"""
    B = 4099
    pr = _Pair(torch_cuda, B, TOLL_MECHS, _gids(B, len(TOLL_MECHS), "random"), _pool())
    if driver == "fused":
        for e in pr.envs:
            _set_path(e, "fused")
        for s in range(30):
            pr.step(s)
        return
    for k in range(6):
        for e in pr.envs:
            if driver == "rollout":
                e.rollout_random(5, step_counter=5 * k)
            else:
                for s in range(5):
                    e.step_deferred(e.sample_actions(step_counter=5 * k + s))
        pr.compare(STATE + RESULT, (driver, k), belief=False)
    for e in pr.envs:
        e.flush_observations()
    pr.compare(STATE + DENSE, (driver, "flushed"))


def test_mixed_graphs_in_a_tile(torch_cuda):
    """resample_graph: after auto-resets the envs of a tile sit on different graphs, so the writers, the in-kernel draw
    and the sampler take their unstaged paths"""
    B = 1000
    pool = _pool(G=4)
    pr = _Pair(torch_cuda, B, TOLL_MECHS, _gids(B, len(TOLL_MECHS), "random"), pool, resample_graph=True)
    for s in range(40):
        pr.step(s)
    gids = pr.grp.graph_id.cpu().numpy()[: B // 32 * 32].reshape(-1, 32)
    assert (gids != gids[:, :1]).any(axis=1).sum() > 0  # some tile sits on more than one graph
    for k in range(4):
        for e in pr.envs:
            e.rollout_random(5, step_counter=100 + 5 * k)
        pr.compare(STATE + RESULT, ("rollout", k), belief=False)
    for e in pr.envs:
        e.flush_observations()
    pr.compare(STATE + DENSE, "flushed")


def test_one_row_mask_images(torch_cuda):
    """A * N > 4096: the writers assemble one action_mask row per image"""
    n, p = 600, 7  # A * N = 4 800
    pool = _pool(G=1, n=n, e=1200)
    B = 300
    mechs = [dict(tolls=0), dict(tolls=2, agent_money=6), dict(tolls=ABOVE)]
    pr = _Pair(torch_cuda, B, mechs, _gids(B, 3, "modulo"), pool, p=p)
    for s in range(25):
        pr.step(s)
    for e in pr.envs:
        _set_path(e, "bulk")
    for s in range(25, 35):
        pr.step(s)


def test_batch_over_one_wave(torch_cuda):
    """random rollouts of a batch larger than one wave (step and sampler as separate launches)"""
    B = 12000
    mechs = [dict(tolls=0), dict(tolls=3), dict(tolls=2, agent_money=5), dict(tolls=ABOVE)]
    pr = _Pair(torch_cuda, B, mechs, _gids(B, 4, "random"), _pool())
    for k in range(4):
        for e in pr.envs:
            e.rollout_random(5, step_counter=5 * k)
        pr.compare(STATE + RESULT, ("rollout", k), belief=False)
        for e in pr.envs:
            e.flush_observations()
        pr.compare(DENSE, ("rollout", k))


def test_host_buffer_calls(torch_cuda):
    """step_host / sample_actions_host / host_rollout_random with mixed tolls"""
    torch = torch_cuda
    B = 500
    pr = _Pair(torch, B, TOLL_MECHS, _gids(B, len(TOLL_MECHS), "random"), _pool())
    for s in range(20):
        got = pr.grp.sample_actions_host(step_counter=s).clone()
        pr.grp.step_host(got)
        for g, r in enumerate(pr.refs):
            want = r.sample_actions_host(step_counter=s).clone()
            idx = pr.rows[g].cpu()
            assert got.index_select(0, idx).equal(want.index_select(0, idx)), ("sample_actions_host", g, s)
            r.step_host(want)
        pr.compare(STATE + RESULT + DENSE, ("step_host", s))
    for e in pr.envs:
        e.host_rollout_random(10, step_counter=100)
    pr.compare(STATE + DENSE, "host_rollout_random")


# ------------------------------------------------------------------------------------------ benchmarked shapes
def _bench_env(B, n, e, toll, **kw):
    import student_mechanism_design_b200 as pkg

    return pkg.BatchedScotlandYardEnv(B, 6, 20, graph_nodes=n, graph_edges=e, seed=0, num_graphs=1, tolls=toll, belief=True,
                                      reveal_interval=5, auto_reset=True, device="cuda:0", **kw)


@pytest.mark.parametrize("shape", ["c3", "c4"])
def test_benchmarked_shapes(torch_cuda, shape):
    """c3 (65 536 envs, N = 200, belief + reveal) for 25 steps and c4 (32 768 envs, N = 1000: the observation grid's
    tail split) for a few, four toll groups interleaved, each group against an ungrouped handle with its toll"""
    torch = torch_cuda
    B, n, e, steps = (65536, 200, 400, 25) if shape == "c3" else (32768, 1000, 2000, 4)
    tolls = [0, 1, 2, 3]
    grp = _bench_env(B, n, e, 1)
    grp.set_mechanisms([{"tolls": t} for t in tolls])
    rows = [torch.arange(g, B, 4, device=grp.device) for g in range(4)]
    refs = [_bench_env(B, n, e, t) for t in tolls]
    for x in [grp] + refs:
        x.reset()
    for s in range(steps):
        acts = grp.sample_actions(step_counter=s)
        grp.step(acts)
        for g, ref in enumerate(refs):
            ra = ref.sample_actions(step_counter=s)
            assert acts.index_select(0, rows[g]).equal(ra.index_select(0, rows[g])), (shape, "sampler", g, s)
            ref.step(ra)
            _equal(grp, ref, STATE + RESULT + DENSE, rows[g], (shape, tolls[g], s))
            _belief_close(grp, ref, rows[g], (shape, tolls[g], s))
    for x in [grp] + refs:
        x.close()


def test_shards_sum_to_full_batch(torch_cuda):
    """two half handles with the default assignment, summed per group, equal one full handle"""
    pool = _pool()
    B, C_ = 2048, 16
    mechs = [dict(tolls=g % 4, agent_money=4 + g) for g in range(C_)]
    full, lo, hi = _env(B, pool), _env(B // 2, pool), _env(B // 2, pool, env_offset=B // 2)
    for e in (full, lo, hi):
        e.set_mechanisms(mechs)
        e.reset()
        e.rollout_random(40, step_counter=0)
    f = full.stats(by_group=True)
    a, b = lo.stats(by_group=True), hi.stats(by_group=True)
    assert [{k: x[k] + y[k] for k in x} for x, y in zip(a, b)] == f
    assert np.array_equal(full.pos.cpu().numpy(), np.concatenate([lo.pos.cpu().numpy(), hi.pos.cpu().numpy()]))
    mf, ma, mb = full.metrics(by_group=True), lo.metrics(by_group=True), hi.metrics(by_group=True)
    for g in range(C_):
        assert mf[g]["num_episodes"] == ma[g]["num_episodes"] + mb[g]["num_episodes"]


# ------------------------------------------------------------------------------------------ agents
def _advance(pr, steps):
    for s in range(steps):
        pr.step(s, dense=False)


@pytest.mark.parametrize("features", ["env", "reference"])
def test_gnn_act_with_group_tolls(torch_cuda, features):
    import student_mechanism_design_b200 as pkg

    B = 2000
    pr = _Pair(torch_cuda, B, TOLL_MECHS, _gids(B, len(TOLL_MECHS), "random"), _pool(), belief=False)
    pols = [pkg.GNNPolicy(e, features=features, seed=5) for e in pr.envs]
    for k in range(6):
        _advance(pr, 3)
        for eps in ((0.3, 0.5), (0.0, 0.0)):  # explore and exploit
            got = pols[0].act(*eps, step_counter=k)
            for g, pol in enumerate(pols[1:]):
                want = pol.act(*eps, step_counter=k)
                rows = pr.rows[g]
                assert got.index_select(0, rows).equal(want.index_select(0, rows)), (features, eps, k, g)


@pytest.mark.parametrize("tensor_cores", [True, False])
def test_mappo_act_with_group_tolls(torch_cuda, tensor_cores):
    import student_mechanism_design_b200 as pkg

    B = 2000
    pr = _Pair(torch_cuda, B, TOLL_MECHS, _gids(B, len(TOLL_MECHS), "random"), _pool(), belief=False)
    A = P + 1
    pols = [pkg.MappoPolicy(e, obs_size=A, hidden_size=64, seed=2) for e in pr.envs]
    for pol in pols:
        pol.tensor_cores = tensor_cores
    for k in range(6):
        _advance(pr, 3)
        got, lp = pols[0].act(step_counter=k)
        for g, pol in enumerate(pols[1:]):
            want, wlp = pol.act(step_counter=k)
            rows = pr.rows[g]
            assert got.index_select(0, rows).equal(want.index_select(0, rows)), (tensor_cores, k, g)
            assert _bits(lp.index_select(0, rows)).equal(_bits(wlp.index_select(0, rows))), (tensor_cores, k, g)


def test_rollout_collector_with_gnn(torch_cuda):
    """RolloutCollector with GNNPolicy: the deferred path, the policy reading the headroom budgets"""
    import student_mechanism_design_b200 as pkg

    B = 1500
    pr = _Pair(torch_cuda, B, TOLL_MECHS, _gids(B, len(TOLL_MECHS), "random"), _pool(), belief=False)
    trajs = []
    for e in pr.envs:
        pol = pkg.GNNPolicy(e, seed=1)
        pol.epsilon = (0.2, 0.4)
        trajs.append(pkg.RolloutCollector(e, pol, 30).collect())
    for g in range(len(TOLL_MECHS)):
        rows = pr.rows[g]
        for k, v in trajs[0].items():
            if not torch_cuda.is_tensor(v) or v.dim() < 2 or v.shape[1] != B:
                continue
            assert _bits(v.index_select(1, rows)).equal(_bits(trajs[g + 1][k].index_select(1, rows))), (k, g)
    pr.compare(STATE, "after collect", belief=False)


# ------------------------------------------------------------------------------------------ lifecycle
def test_lifecycle_and_errors(torch_cuda):
    torch = torch_cuda
    import student_mechanism_design_b200 as pkg
    from student_mechanism_design_b200 import _cabi

    pool = _pool()
    B = 256
    env = _env(B, pool)
    env.reset()
    with pytest.raises(pkg.SyError, match="no mechanism groups"):
        _cabi.check(_raw_tolls(env, [0]))
    env.set_mechanisms([dict(tolls=0), dict(tolls=ABOVE)])
    env.reset()
    env.step(env.sample_actions())
    for tolls, msg in [([0], "num_groups 1"), ([0, 0, 0], "num_groups 3"), ([-1, 0], "outside"),
                       ([0, _cabi.SY_MAX_TOLL + 1], "outside")]:
        with pytest.raises(pkg.SyError, match=msg):
            _cabi.check(_raw_tolls(env, tolls))
    env.step_deferred(env.sample_actions())
    with pytest.raises(pkg.SyError, match="pending"):
        _cabi.check(_raw_tolls(env, [1, 1]))
    env.flush_observations()
    env.step(env.sample_actions())  # the rejected calls owe no reset
    assert _raw_tolls(env, [_cabi.SY_MAX_TOLL, 0]) == 0
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):
        env.step(env.sample_actions())
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):
        _cabi.check(env._lib.sy_rollout_random(env._handle, 2, 0, env.sample_actions().data_ptr(), C.byref(env._state),
                                               C.byref(env._obs), C.byref(env._out), env._stream()))
    # rejected calls keep the previous tolls: [SY_MAX_TOLL, 0] behave like ungrouped handles with those tolls
    with pytest.raises(pkg.SyError, match="outside"):
        _cabi.check(_raw_tolls(env, [-5, 2]))
    env.reset(restart=True)  # (episode counters from 0, as on the fresh reference handles)
    refs = [_env(B, pool, toll=_cabi.SY_MAX_TOLL), _env(B, pool, toll=0)]
    rows = [torch.arange(g, B, 2, device=env.device) for g in range(2)]
    for r in refs:
        r.reset()
    for s in range(20):
        env.step(env.sample_actions(step_counter=s))
        for g, r in enumerate(refs):
            r.step(r.sample_actions(step_counter=s))
            _equal(env, r, STATE + RESULT + DENSE, rows[g], ("kept", g, s))
    # sy_set_groups gives every group the config's toll again: bit-identical to a handle without groups
    env.set_mechanisms([{}, {}])
    assert env._env_toll is None
    plain = _env(B, pool)
    env.reset(restart=True)
    plain.reset()
    for s in range(30):
        env.step(env.sample_actions(step_counter=s))
        plain.step(plain.sample_actions(step_counter=s))
        _equal(env, plain, STATE + RESULT + DENSE, None, ("restored", s))
    # clearing the groups: bit-identical to a fresh handle
    env.set_mechanisms([dict(tolls=3)])
    env.reset()
    env.step(env.sample_actions())
    env.set_mechanisms(None)
    assert env.mechanisms is None and env._env_toll is None
    fresh = _env(B, pool)
    env.reset(restart=True)
    fresh.reset()
    for s in range(30):
        env.step(env.sample_actions(step_counter=s))
        fresh.step(fresh.sample_actions(step_counter=s))
        _equal(env, fresh, STATE + RESULT + DENSE + ["belief_map"], None, ("cleared", s))


def test_replay_after_new_tolls_is_refused(torch_cuda):
    import student_mechanism_design_b200 as pkg

    pool = _pool()
    env = _env(500, pool)
    env.set_mechanisms([dict(tolls=0), dict(tolls=2)])
    env.reset()
    graph, _ = env.capture_rollout(4)
    graph.replay()
    env.set_mechanisms([dict(tolls=3), dict(tolls=2)])
    with pytest.raises(pkg.SyError, match="capture it again"):
        graph.replay()
    env.reset()
    graph, _ = env.capture_rollout(4)
    graph.replay()
    assert [m["tolls"] for m in env.mechanisms] == [3, 2]


def test_guards_with_group_tolls(torch_cuda):
    pool = _pool()
    env = _env(333, pool, guard_bytes=4096)
    env.set_mechanisms(TOLL_MECHS)
    env.reset()
    for s in range(20):
        env.step(env.sample_actions(step_counter=s))
    env.rollout_random(10)
    env.stats(by_group=True)
    env.check_guards()
