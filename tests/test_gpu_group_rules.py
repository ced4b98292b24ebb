"""Per-group police count and episode horizon (sy_set_group_rules, the `number_of_agents` / `max_timestep` keys of
env.set_mechanisms).

Checked here: rules equal to the config change no byte of any output through every step path; agents 0..P_g of an env
of a group with P_g police and horizon T_g follow exactly the trajectory of an ungrouped handle built with
number_of_agents = P_g and max_timestep = T_g -- state, results, action_mask rows, node_features columns (both dtypes)
and sampled actions after every step, the belief map to 1e-6 -- while its agents past P_g carry exactly the absent
values of include/sy_env.h; on ragged, mixed batches and on the paths the small case does not reach (the in-kernel
draws, mixed graphs in a tile, 1-row mask images, batches over one wave, the host-buffer calls, the benchmarked shapes,
15 police); per-group statistics; shards; partial resets and init_pos; the policies' refusal; the lifecycle of
sy_set_group_rules; the out-of-bounds canaries."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, E, P, MONEY = 40, 60, 3, 10
BELIEF_TOL = 1e-6
ENV_STATE = ["timestep", "graph_id", "episode", "done", "visits", "mrx_revealed"]
ENV_RESULT = ["winner", "status"]
# per-agent outputs and the dimension of their agent index
AGENT_DIM = {"pos": 1, "money": 1, "agent_budget": 1, "reward": 1, "reward64": 1, "terminated": 1, "truncated": 1,
             "done_flags": 1, "action_mask": 1, "node_features": 2}
AGENT_STATE = ["pos", "money", "agent_budget"]
AGENT_RESULT = ["reward", "reward64", "terminated", "truncated", "done_flags"]
DENSE = ["action_mask", "node_features"]
STATE = ENV_STATE + AGENT_STATE
RESULT = ENV_RESULT + AGENT_RESULT
# (police, horizon) with budgets and tolls.  Groups 0, 1 and 4 get budgets that last past their horizon (at most 5 per
# move), so their episodes end by truncation too and not only by capture or by the police going broke
RULE_MECHS = [dict(number_of_agents=1, max_timestep=15, agent_money=200),
              dict(number_of_agents=2, max_timestep=40, agent_money=250),
              dict(number_of_agents=3, max_timestep=250), dict(number_of_agents=1, max_timestep=40, agent_money=4, tolls=2),
              dict(number_of_agents=2, max_timestep=15, agent_money=100, tolls=0)]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _pool(G=2, n=N, e=E):
    import student_mechanism_design_b200 as pkg

    return pkg.generate_graph_pool(G, n, e, seed=0)


def _env(B, pool, *, toll=1, money=MONEY, p=P, max_timestep=250, reward_mode="fp64", weights=None, env_offset=0, **kw):
    import student_mechanism_design_b200 as pkg

    kw.setdefault("belief", True)
    kw.setdefault("belief_ce", kw["belief"])
    return pkg.BatchedScotlandYardEnv(B, p, money, reward_weights=weights, graphs=pool, seed=7, auto_reset=True,
                                      tolls=toll, reveal_interval=5, keep_reward64=True, reward_mode=reward_mode,
                                      env_offset=env_offset, max_timestep=max_timestep, **kw)


def _raw_rules(env, police, horizon):
    """sy_set_group_rules straight through the C ABI (returns the status code); None = a NULL array"""
    n = len(police) if police is not None else (len(horizon) if horizon is not None else len(env.mechanisms))
    arr = lambda v: None if v is None else (C.c_int32 * max(len(v), 1))(*v)  # noqa: E731
    return env._lib.sy_set_group_rules(env._handle, n, arr(police), arr(horizon), env._stream())


def _bits(t):
    """a tensor as integers of the same width, so that floats compare bit for bit"""
    import torch

    if t.dtype in (torch.float32, torch.float64):
        return t.view(torch.int32 if t.dtype == torch.float32 else torch.int64)
    if t.dtype == torch.bool:
        return t.view(torch.uint8)
    return t


def _raise(a, b, tag, k):
    if not _bits(a).equal(_bits(b)):
        bad = (_bits(a) != _bits(b)).nonzero()
        raise AssertionError(f"{tag} {k}: {bad.shape[0]} mismatches, first at {bad[:1].tolist()}")


def _equal(grp, ref, names, rows, tag):
    """outputs `names` of `grp` and `ref` equal on `rows` (LongTensor on the device, or None = all), byte for byte; for
    per-agent outputs the columns of ref's agents"""
    for k in names:
        a, b = getattr(grp, k), getattr(ref, k)
        if a is None:
            assert b is None, (tag, k)
            continue
        if rows is not None:
            a, b = a.index_select(0, rows), b.index_select(0, rows)
        if k in AGENT_DIM:
            a = a.narrow(AGENT_DIM[k], 0, b.shape[AGENT_DIM[k]])
        _raise(a, b, tag, k)


def _absent(env, rows, police, names, tag):
    """the agents past `police` of the envs `rows` carry exactly the absent values of include/sy_env.h"""
    torch = __import__("torch")
    A = env.num_agents
    if police + 1 == A:
        return
    for k in names:
        t = getattr(env, k)
        if t is None:
            continue
        d = AGENT_DIM[k]
        x = t.index_select(0, rows).narrow(d, police + 1, A - police - 1)
        if k == "pos":
            want = torch.full_like(x, -1)
        elif k in ("terminated", "truncated", "done_flags"):  # the env's own flags
            want = t.index_select(0, rows).narrow(1, 0, 1).expand_as(x)
        else:
            want = torch.zeros_like(x)
        _raise(x, want, tag, ("absent", k))


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
def test_identity_rules_equal_to_config(torch_cuda, path, reward_mode):
    """three groups whose police count and horizon equal the config's, given through the keys (and straight through
    sy_set_group_rules): byte-equal to a handle without groups through `path`, statistics included"""
    torch = torch_cuda
    pool = _pool()
    B = 997
    w = None
    if reward_mode == "fp32":
        import student_mechanism_design_b200 as pkg

        w = {k: torch.tensor(v, dtype=torch.float32) for k, v in pkg.DEFAULT_REWARD_WEIGHTS.items()}
    ref, grp = (_env(B, pool, weights=w, reward_mode=reward_mode, max_timestep=30) for _ in range(2))
    for e in (ref, grp):
        _set_path(e, path)
    grp.set_mechanisms([{"number_of_agents": P, "max_timestep": 30}, {"number_of_agents": float(P)}, {}])
    assert [(m["number_of_agents"], m["max_timestep"]) for m in grp.mechanisms] == [(P, 30)] * 3
    assert grp._env_police is None
    assert _raw_rules(grp, [P] * 3, [30] * 3) == 0
    assert _raw_rules(grp, None, None) == 0
    ref.reset()
    grp.reset()
    names = STATE + DENSE
    _equal(grp, ref, names, None, "reset")
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
    assert ref.stats()["truncations"] > 0
    m1, m2 = ref.metrics(), grp.metrics()
    # (the aggregate budget efficiency is summed per group: equal up to the order of the float additions)
    assert {k: v for k, v in m1.items() if k != "mean_budget_efficiency"} == \
        {k: v for k, v in m2.items() if k != "mean_budget_efficiency"}
    assert m1["mean_budget_efficiency"] == pytest.approx(m2["mean_budget_efficiency"], rel=1e-12)


# ------------------------------------------------------------------------------------------ decomposition
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
    """a grouped handle (p police) with `mechs` assigned by `gid` and one ungrouped handle per mechanism (its police
    count, horizon, toll and budget), same seed and offset: agents 0..P_g of env b of the grouped handle must follow
    env b of handle gid[b], its other agents must be absent"""

    def __init__(self, torch, B, mechs, gid, pool, count=False, p=P, **kw):
        self.torch, self.B, self.gid, self.p = torch, B, np.asarray(gid, dtype=np.int32), p
        self.grp = _env(B, pool, p=p, **kw)
        self.grp.set_mechanisms(mechs, group_id=torch.as_tensor(self.gid))
        self.police = [m.get("number_of_agents", p) for m in mechs]
        self.refs = [_env(B, pool, p=m.get("number_of_agents", p), max_timestep=m.get("max_timestep", 250),
                          toll=m.get("tolls", 1), money=m.get("agent_money", MONEY), **kw) for m in mechs]
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
            _absent(self.grp, self.rows[g], self.police[g], [k for k in names if k in AGENT_DIM], (tag, g))
            if belief:
                _belief_close(self.grp, r, self.rows[g], (tag, g))

    def check_actions(self, acts, ref_acts, g, tag):
        rows, pg = self.rows[g], self.police[g]
        a = acts.index_select(0, rows)
        assert a.narrow(1, 0, pg + 1).equal(ref_acts.index_select(0, rows)), ("sampler", g, tag)
        assert bool((a.narrow(1, pg + 1, self.p - pg) == -1).all()), ("absent action", g, tag)

    def step(self, s, dense=True):
        acts = self.grp.sample_actions(step_counter=s)
        t_before = self.grp.timestep.cpu().numpy() if self.counts is not None else None
        # absent agents' actions are ignored whatever they hold
        garbage = acts.clone()
        for g, pg in enumerate(self.police):
            if pg < self.p:
                garbage[self.rows[g], pg + 1:] = self.torch.randint(-3, N + 3, (len(self.rows[g]), self.p - pg),
                                                                    device=acts.device)
        self.grp.step(garbage)
        for g, r in enumerate(self.refs):
            ra = r.sample_actions(step_counter=s)
            self.check_actions(acts, ra, g, s)
            r.step(ra)
            if self.counts is not None:
                idx = self.rows[g].cpu().numpy()
                _count(self.counts[g], t_before[idx], self.grp.status.cpu().numpy()[idx], self.grp.winner.cpu().numpy()[idx])
        self.compare(STATE + RESULT + (DENSE if dense else []), ("step", s), belief=dense)


def _gids(B, C, assign):
    return (np.arange(B) % C if assign == "modulo" else np.random.default_rng(3).integers(0, C, B)).astype(np.int32)


@pytest.mark.parametrize("nf_dtype", ["float32", "uint8"])
@pytest.mark.parametrize("assign", ["modulo", "random"])
def test_rules_follow_their_config(torch_cuda, assign, nf_dtype):
    """police 1 / 2 / 3 with horizons 15 / 40 / 250, tolls and budgets, on a ragged batch (4 099 envs), assigned b % C and
    at random (every warp mixes police counts), 64 steps; then per-group statistics and budget efficiency"""
    torch = torch_cuda
    B, C_ = 4099, len(RULE_MECHS)
    pr = _Pair(torch, B, RULE_MECHS, _gids(B, C_, assign), _pool(), count=True,
               node_features_dtype=getattr(torch, nf_dtype))
    for s in range(64):
        pr.step(s)
    grp = pr.grp
    per = grp.stats(by_group=True)
    for g in range(C_):
        assert {k: per[g][k] for k in COUNTED} == pr.counts[g], (assign, g)
        assert per[g]["police_moves"] > 0 and per[g]["sum_budget_spent"] >= per[g]["police_moves"]
    assert all(c["episodes"] > 0 for c in pr.counts)
    assert all(pr.counts[g]["truncations"] > 0 for g in (0, 1, 4)), [c["truncations"] for c in pr.counts]  # horizons
    assert {k: sum(x[k] for x in per) for k in per[0]} == grp.stats()
    m = grp.metrics(by_group=True)
    for g, mech in enumerate(RULE_MECHS):
        budget = mech["number_of_agents"] * mech.get("agent_money", MONEY)
        assert m[g]["mean_budget_efficiency"] == per[g]["sum_episode_budget_spent"] / per[g]["episodes"] / budget, g
    eff = sum(per[g]["sum_episode_budget_spent"] / (mech["number_of_agents"] * mech.get("agent_money", MONEY))
              for g, mech in enumerate(RULE_MECHS))
    assert grp.metrics()["mean_budget_efficiency"] == eff / grp.stats()["episodes"]


@pytest.mark.parametrize("driver", ["deferred", "rollout", "fused"])
def test_rules_in_kernel_draws(torch_cuda, driver):
    """the next-action draw inside the lagged and one-launch rollout kernels (4 099 envs: one CTA per tile), and the fused
    step, with mixed police counts and horizons"""
    B = 4099
    pr = _Pair(torch_cuda, B, RULE_MECHS, _gids(B, len(RULE_MECHS), "random"), _pool())
    if driver == "fused":
        for e in pr.envs:
            _set_path(e, "fused")
        for s in range(30):
            pr.step(s)
        return
    for k in range(8):
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
    pr = _Pair(torch_cuda, B, RULE_MECHS, _gids(B, len(RULE_MECHS), "random"), pool, resample_graph=True)
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
    mechs = [dict(number_of_agents=1, max_timestep=20), dict(number_of_agents=4, tolls=2, agent_money=6), dict()]
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
    mechs = [dict(number_of_agents=1, max_timestep=15), dict(number_of_agents=2), dict(agent_money=5, max_timestep=40),
             dict(number_of_agents=2, tolls=3, max_timestep=15)]
    pr = _Pair(torch_cuda, B, mechs, _gids(B, 4, "random"), _pool())
    for k in range(4):
        for e in pr.envs:
            e.rollout_random(5, step_counter=5 * k)
        pr.compare(STATE + RESULT, ("rollout", k), belief=False)
        for e in pr.envs:
            e.flush_observations()
        pr.compare(DENSE, ("rollout", k))


def test_host_buffer_calls(torch_cuda):
    """step_host / sample_actions_host / host_rollout_random with mixed police counts"""
    torch = torch_cuda
    B = 500
    pr = _Pair(torch, B, RULE_MECHS, _gids(B, len(RULE_MECHS), "random"), _pool())
    for s in range(20):
        got = pr.grp.sample_actions_host(step_counter=s).clone()
        pr.grp.step_host(got)
        for g, r in enumerate(pr.refs):
            want = r.sample_actions_host(step_counter=s).clone()
            idx, pg = pr.rows[g].cpu(), pr.police[g]
            sel = got.index_select(0, idx)
            assert sel.narrow(1, 0, pg + 1).equal(want.index_select(0, idx)), ("sample_actions_host", g, s)
            assert bool((sel.narrow(1, pg + 1, P - pg) == -1).all())
            r.step_host(want)
        pr.compare(STATE + RESULT + DENSE, ("step_host", s))
    for e in pr.envs:
        e.host_rollout_random(10, step_counter=100)
    pr.compare(STATE + DENSE, "host_rollout_random")


# ------------------------------------------------------------------------------------------ larger shapes
def _bench_env(B, n, e, p, max_timestep=250, **kw):
    import student_mechanism_design_b200 as pkg

    return pkg.BatchedScotlandYardEnv(B, p, 20, graph_nodes=n, graph_edges=e, seed=0, num_graphs=1, tolls=1, belief=True,
                                      reveal_interval=5, auto_reset=True, device="cuda:0", max_timestep=max_timestep,
                                      keep_reward64=True, **kw)


@pytest.mark.parametrize("shape", ["c3", "c4", "p15"])
def test_larger_shapes(torch_cuda, shape):
    """c3 (65 536 envs, N = 200, belief + reveal) and c4 (32 768 envs, N = 1000: the observation grid's tail split) with
    6 police and groups of 1..6 police interleaved; 15 police (MAXA = 16) with groups of 1..15.  Each group against an
    ungrouped handle with its police count (and, for some, a shorter horizon)"""
    torch = torch_cuda
    B, n, e, steps, p = {"c3": (65536, 200, 400, 25, 6), "c4": (32768, 1000, 2000, 4, 6),
                         "p15": (4096 + 7, 101, 190, 30, 15)}[shape]
    police = list(range(1, p + 1))
    horizon = [15 if k % 3 == 0 else 250 for k in police]
    C_ = len(police)
    grp = _bench_env(B, n, e, p)
    grp.set_mechanisms([{"number_of_agents": k, "max_timestep": t} for k, t in zip(police, horizon)])
    rows = [torch.arange(g, B, C_, device=grp.device) for g in range(C_)]
    refs = [_bench_env(B, n, e, k, max_timestep=t) for k, t in zip(police, horizon)]
    for x in [grp] + refs:
        x.reset()
    for s in range(steps):
        acts = grp.sample_actions(step_counter=s)
        grp.step(acts)
        for g, ref in enumerate(refs):
            ra = ref.sample_actions(step_counter=s)
            sel = acts.index_select(0, rows[g])
            assert sel.narrow(1, 0, police[g] + 1).equal(ra.index_select(0, rows[g])), (shape, "sampler", g, s)
            assert bool((sel.narrow(1, police[g] + 1, p - police[g]) == -1).all())
            ref.step(ra)
            _equal(grp, ref, STATE + RESULT + DENSE, rows[g], (shape, police[g], s))
            _absent(grp, rows[g], police[g], AGENT_STATE + AGENT_RESULT + DENSE, (shape, police[g], s))
            _belief_close(grp, ref, rows[g], (shape, police[g], s))
    for x in [grp] + refs:
        x.close()


# ------------------------------------------------------------------------------------------ statistics and resets
def test_shards_sum_to_full_batch(torch_cuda):
    """two half handles with the default assignment, summed per group, equal one full handle"""
    pool = _pool()
    B, C_ = 2048, 12
    mechs = [dict(number_of_agents=1 + g % 3, max_timestep=(15, 40, 250)[g % 3], agent_money=4 + g) for g in range(C_)]
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


def test_partial_resets_and_init_pos(torch_cuda):
    """reset(reset_mask) of a third of the envs, and init_pos with garbage in the absent columns (ignored, read back as
    -1), against the ungrouped handles given the same masks and the live columns"""
    torch = torch_cuda
    B = 1000
    pr = _Pair(torch, B, RULE_MECHS, _gids(B, len(RULE_MECHS), "random"), _pool())
    for s in range(10):
        pr.step(s)
    mask = torch.arange(B, device=pr.grp.device) % 3 == 0
    for e in pr.envs:
        e.reset(reset_mask=mask)
    pr.compare(STATE + DENSE, "partial reset")
    for s in range(10, 20):
        pr.step(s)
    # explicit start nodes: distinct nodes for the live columns, garbage past each env's police
    rng = np.random.default_rng(11)
    ip = np.stack([rng.permutation(N)[: P + 1] for _ in range(B)]).astype(np.int32)
    garbage = ip.copy()
    for g, pg in enumerate(pr.police):
        idx = pr.rows[g].cpu().numpy()
        garbage[np.ix_(idx, np.arange(pg + 1, P + 1))] = rng.integers(-1000, 1000, (len(idx), P - pg))
    pr.grp.reset(init_pos=garbage)
    for g, r in enumerate(pr.refs):
        r.reset(init_pos=np.ascontiguousarray(ip[:, : pr.police[g] + 1]))
    pr.compare(STATE + DENSE, "init_pos")
    for s in range(20, 40):
        pr.step(s)


# ------------------------------------------------------------------------------------------ agents
def test_policies_refuse_mixed_police_counts(torch_cuda):
    """GNNPolicy / MappoPolicy raise before any launch while some group's police count differs; a RolloutCollector with a
    logits policy runs (absent agents: an all-zero mask row samples -1); equal police counts are accepted"""
    torch = torch_cuda
    import student_mechanism_design_b200 as pkg

    pool = _pool()
    B = 600
    env = _env(B, pool, belief=False)
    gnn, mappo = pkg.GNNPolicy(env, seed=1), pkg.MappoPolicy(env, obs_size=P + 1, hidden_size=64, seed=2)
    env.set_mechanisms(RULE_MECHS)
    env.reset()
    launches = env._lib.sy_launch_count()
    for call in (lambda: gnn.act(0.1, 0.1), gnn.q_values, gnn, mappo.act):
        with pytest.raises(ValueError, match="number_of_agents"):
            call()
    assert env._lib.sy_launch_count() == launches
    assert gnn.step_counter == 0 and mappo.step_counter == 0
    logits = lambda obs: torch.zeros(B, P + 1, N, device=env.device)  # noqa: E731
    traj = pkg.RolloutCollector(env, logits, 20).collect()
    acts = traj["actions"]
    gid = env.group_id.long()
    police = torch.tensor([m["number_of_agents"] for m in RULE_MECHS], device=env.device)[gid]
    absent = torch.arange(P + 1, device=env.device).view(1, 1, -1) > police.view(1, -1, 1)
    assert bool((acts[absent.expand_as(acts)] == -1).all())
    assert bool((acts[~absent.expand_as(acts)] >= 0).any())
    assert bool((env.pos[torch.arange(P + 1, device=env.device).view(1, -1) > police.view(-1, 1)] == -1).all())
    env.set_mechanisms([{"max_timestep": 20, "number_of_agents": P}, {}])  # same police count: the agents work
    env.reset()
    gnn.act(0.0, 0.0)
    mappo.act()


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
        _cabi.check(_raw_rules(env, [1], [250]))
    env.set_mechanisms([dict(), dict(tolls=2)])
    env.reset()
    env.step(env.sample_actions())
    for police, horizon, msg in [([1], [250], "num_groups 1"), ([1, 1, 1], None, "num_groups 3"),
                                 ([0, 1], None, "outside"), ([1, P + 1], None, "outside"), (None, [-1, 3], "outside"),
                                 (None, [250, 251], "outside"), ([-3, 2], [10, 10], "outside")]:
        with pytest.raises(pkg.SyError, match=msg):
            _cabi.check(_raw_rules(env, police, horizon))
    env.step_deferred(env.sample_actions())
    with pytest.raises(pkg.SyError, match="pending"):
        _cabi.check(_raw_rules(env, [1, 2], [20, 20]))
    env.flush_observations()
    env.step(env.sample_actions())  # the rejected calls owe no reset
    assert _raw_rules(env, [2, 1], [20, 250]) == 0
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):
        env.step(env.sample_actions())
    with pytest.raises(pkg.SyError, match="mechanism groups changed"):
        _cabi.check(env._lib.sy_rollout_random(env._handle, 2, 0, env.sample_actions().data_ptr(), C.byref(env._state),
                                               C.byref(env._obs), C.byref(env._out), env._stream()))
    # rejected calls keep the previous values, and the call clears nothing else (the tolls stay): [2 police, T 20, toll 1]
    # and [1 police, T 250, toll 2] behave like ungrouped handles with those values
    with pytest.raises(pkg.SyError, match="outside"):
        _cabi.check(_raw_rules(env, [3, 0], [5, 5]))
    env.reset(restart=True)  # (episode counters from 0, as on the fresh reference handles)
    refs = [_env(B, pool, p=2, max_timestep=20), _env(B, pool, p=1, toll=2)]
    rows = [torch.arange(g, B, 2, device=env.device) for g in range(2)]
    for r in refs:
        r.reset()
    for s in range(40):
        env.step(env.sample_actions(step_counter=s))
        for g, r in enumerate(refs):
            r.step(r.sample_actions(step_counter=s))
            _equal(env, r, STATE + RESULT + DENSE, rows[g], ("kept", g, s))
            _absent(env, rows[g], 2 - g, AGENT_STATE + AGENT_RESULT + DENSE, ("kept", g, s))
    # sy_set_groups gives every group the config's police count and horizon again: bit-identical to no groups
    env.set_mechanisms([{}, {}])
    assert env._env_police is None
    plain = _env(B, pool)
    env.reset(restart=True)
    plain.reset()
    for s in range(30):
        env.step(env.sample_actions(step_counter=s))
        plain.step(plain.sample_actions(step_counter=s))
        _equal(env, plain, STATE + RESULT + DENSE, None, ("restored", s))
    # clearing the groups: bit-identical to a fresh handle
    env.set_mechanisms([dict(number_of_agents=1, max_timestep=5)])
    env.reset()
    env.step(env.sample_actions())
    env.set_mechanisms(None)
    assert env.mechanisms is None and env._env_police is None
    fresh = _env(B, pool)
    env.reset(restart=True)
    fresh.reset()
    for s in range(30):
        env.step(env.sample_actions(step_counter=s))
        fresh.step(fresh.sample_actions(step_counter=s))
        _equal(env, fresh, STATE + RESULT + DENSE + ["belief_map"], None, ("cleared", s))


def test_replay_after_new_rules_is_refused(torch_cuda):
    import student_mechanism_design_b200 as pkg

    pool = _pool()
    env = _env(500, pool)
    env.set_mechanisms([dict(number_of_agents=1), dict(number_of_agents=2)])
    env.reset()
    graph, _ = env.capture_rollout(4)
    graph.replay()
    env.set_mechanisms([dict(number_of_agents=3), dict(max_timestep=10)])
    with pytest.raises(pkg.SyError, match="capture it again"):
        graph.replay()
    env.reset()
    graph, _ = env.capture_rollout(4)
    graph.replay()
    assert [m["number_of_agents"] for m in env.mechanisms] == [3, 3]


# ------------------------------------------------------------------------------------------ canaries
GUARD_SHAPES = [  # (N, E, P, B, belief, reveal, tolls), as tests/test_gpu_guards.py
    (13, 20, 2, 33, True, 3, 1),
    (101, 190, 15, 45, True, 4, 1),
    (200, 400, 6, 4096 + 19, True, 5, 1),
    (333, 600, 4, 300, True, 5, 1),
]
GUARD_VARIANTS = ["default", "bulk", "fused", "split", "lagged"]


@pytest.mark.parametrize("variant", GUARD_VARIANTS)
@pytest.mark.parametrize("shape", GUARD_SHAPES, ids=lambda s: f"N{s[0]}P{s[2]}")
def test_guards_with_fewer_police(torch_cuda, shape, variant):
    """no write outside any buffer with groups of fewer police (and short horizons), both node_features dtypes"""
    torch = torch_cuda
    import student_mechanism_design_b200 as pkg

    N_, E_, P_, B, belief, reveal, tolls = shape
    mechs = [dict(number_of_agents=1 + k % P_, max_timestep=(7, 250, 20)[k % 3]) for k in range(max(P_, 3))]
    for nf_dtype in (torch.float32, torch.uint8):
        env = pkg.BatchedScotlandYardEnv(B, P_, 9, graph_nodes=N_, graph_edges=E_, num_graphs=3, seed=5, auto_reset=True,
                                         tolls=tolls, belief=belief, reveal_interval=reveal, keep_reward64=True,
                                         node_features_dtype=nf_dtype, guard_bytes=4096)
        if variant == "bulk":
            env.set_option("step_kernel", "two_kernels")
            env.set_option("writer_path", "bulk")
        elif variant == "fused":
            env.set_option("step_kernel", "fused")
        elif variant == "split":
            env.set_option("step_kernel", "two_kernels")
            env.set_option("nf_fill", "on")
        elif variant == "lagged":
            env.set_option("step_kernel", "two_kernels")
            env.set_option("lagged_kernel", "on")
        env.set_mechanisms(mechs)
        env.reset()
        env.check_guards()
        for s in range(12):
            acts = env.sample_actions(step_counter=s)
            if variant == "lagged":
                env.step_deferred(acts)
            else:
                env.step(acts)
        env.flush_observations()
        env.check_guards()
        env.rollout_random(5, step_counter=100)
        env.check_guards()
        env.step_host(env.sample_actions_host(step_counter=200))
        mask = (torch.arange(B, device=env.device) % 3 == 0)
        env.reset(reset_mask=mask)
        torch.cuda.synchronize()
        env.check_guards()
        assert bool(env.action_mask.any()) and bool((env.pos == -1).any())
        env.close()
