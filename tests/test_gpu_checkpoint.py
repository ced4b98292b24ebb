"""Checkpoint, rewind and re-seed of the batched env: `state_dict` / `load_state_dict`, `set_seed` / `reset(seed=...)`.

Every resume is held against a twin handle that runs the same pool, seed and actions without interruption: after every
step (every call of a multi-step path) the two agree byte for byte on the state (`pos`, `money`, `timestep`,
`graph_id`, `episode`, `done`, `visits`, `mrx_revealed`, `agent_budget`), the dense observations (`action_mask`,
`node_features`, `belief_map`) and the results (`reward`, `reward64`, the flags, `status`, `winner`), and at the end
on `stats()` / `metrics()` (per group too).  The twin itself follows the C oracle (belief within BELIEF_TOL), the
Python OracleGroupBatch for mechanism groups, and heuristic_oracle / policy_oracle for the policies' draws.

Covered: every step path on both sides of the checkpoint (fused, two kernels, bulk writers, deferred with and without
the lagged kernel, the one-launch rollout and the per-step rollout, a replayed CUDA graph, the host-buffer calls) at
c2, c3 (ragged 4 099 envs and the full 65 536), N = 1 000, 15 police, uint8 node features, frozen envs and a 5-graph
pool with graph resampling and reveal skips; a dict taken while observations are pending and one loaded into a handle
with pending observations; rewinding a handle (with and without mechanism groups, with and without a stats() call in
between); resuming on three uneven shards; re-keying by reset(seed=...), set_seed mid-episode and the torchrl adapter;
and the refused loads and replays."""
import io

import numpy as np
import pytest

import heuristic_oracle as ho
import policy_oracle as po
import sy_oracle as so
import sy_oracle_c as oc
from test_gpu_fullsize import BELIEF_TOL, _compare, _same, _threads, torch_cuda  # noqa: F401

pytestmark = pytest.mark.gpu

U64 = 2 ** 64 - 1
S1 = 5
SEEDS = [0, 2 ** 32 + 7, U64, -1]
SHAPES = {
    "c2": dict(N=50, E=110, P=3, money=10, B=1024, toll=0, belief=False, reveal=5),
    "c3": dict(N=200, E=400, P=6, money=20, B=4099, toll=1, belief=True, reveal=5),
    "c3_full": dict(N=200, E=400, P=6, money=20, B=65536, toll=1, belief=True, reveal=5),
    "c4": dict(N=1000, E=2000, P=6, money=20, B=1024, toll=1, belief=True, reveal=5),
    "p15": dict(N=120, E=300, P=15, money=12, B=777, toll=1, belief=True, reveal=4),
    "u8": dict(N=50, E=110, P=3, money=10, B=1500, toll=1, belief=True, reveal=3, nf="uint8"),
    "frozen": dict(N=30, E=60, P=2, money=6, B=300, toll=1, belief=True, reveal=2, auto_reset=False, max_t=6),
    "pool": dict(N=50, E=110, P=4, money=12, B=1024, toll=1, belief=True, reveal=3, graphs=5, resample=True, skip=0.3),
}
STATE = ("pos", "money", "timestep", "graph_id", "episode", "done", "visits", "mrx_revealed", "agent_budget")
DENSE = ("action_mask", "node_features", "belief_map")
RESULTS = ("reward", "reward64", "terminated", "truncated", "done_flags", "status", "winner")
DEFAULT_OPTIONS = dict(step_kernel="auto", writer_path="lsu", lagged_kernel="auto", rollout_kernel="on")
# path -> the options that force it (where AUTO would pick another one)
PATHS = {
    "fused": dict(step_kernel="fused"),
    "two_kernels": dict(step_kernel="two_kernels"),
    "bulk": dict(step_kernel="two_kernels", writer_path="bulk"),
    "lagged": dict(lagged_kernel="on"),
    "unlagged": dict(lagged_kernel="off"),
    "rollout": dict(rollout_kernel="on"),
    "per_step": dict(rollout_kernel="off", lagged_kernel="off"),
    "graph": dict(),
    "host": dict(),
}
SEG = 3  # steps per rollout call / graph replay


def _pkg():
    import student_mechanism_design_b200 as pkg

    return pkg


def _pool(sh, seed=0):
    return _pkg().generate_graph_pool(sh.get("graphs", 1), sh["N"], sh["E"], seed=seed)


def _env(sh, pool, seed=S1, **over):
    torch = __import__("torch")
    kw = dict(graphs=pool, seed=seed, auto_reset=sh.get("auto_reset", True), tolls=sh["toll"], belief=sh["belief"],
              belief_ce=sh["belief"], reveal_interval=sh["reveal"], keep_reward64=True,
              resample_graph=sh.get("resample", False), reveal_skip_prob=sh.get("skip", 0.0),
              max_timestep=sh.get("max_t", 250), node_features_dtype=getattr(torch, sh.get("nf", "float32")))
    kw.update(over)
    B = kw.pop("num_envs", sh["B"])
    return _pkg().BatchedScotlandYardEnv(B, kw.pop("num_police", sh["P"]), sh["money"], **kw)


def _oracle(sh, pool, seed=S1):
    cfg = so.OracleConfig(num_police=sh["P"], agent_money=sh["money"], toll=sh["toll"], belief=sh["belief"],
                          reveal_interval=sh["reveal"], reveal_skip_prob=sh.get("skip", 0.0),
                          max_timestep=sh.get("max_t", 250))
    B, resample = sh["B"], sh.get("resample", False)
    gid = None if resample else ((np.arange(B) // 32) % sh.get("graphs", 1)).astype(np.int32)
    return oc.CBatch(cfg, pool, B, seed=seed & U64, auto_reset=sh.get("auto_reset", True), resample_graph=resample,
                     threads=_threads(), graph_id=gid)


class _Follower:
    """The C oracle driven with the env's default sampler counters 0, 1, 2, ..."""

    def __init__(self, ob):
        self.ob, self.counter, self.want = ob, 0, None

    def to(self, counter):
        while self.counter < counter:
            self.want = self.ob.step(self.ob.sample_actions(self.counter))
            self.counter += 1

    def check(self, env, tag):
        self.to(env._sample_counter)
        pending = env.observations_pending
        _compare(env, self.ob, self.want, env.belief_on and not pending, tag, dense=not pending)
        _same(env.done, self.ob._done, (tag, "done"))


def _snap(env, keys=STATE + DENSE + RESULTS):
    return {k: getattr(env, k).cpu().numpy().copy() for k in keys if getattr(env, k) is not None}


def _equal(a, b, tag):
    assert a.keys() == b.keys(), (tag, sorted(a), sorted(b))
    for k in a:
        if a[k].tobytes() != b[k].tobytes():
            bad = np.argwhere(a[k] != b[k])
            raise AssertionError(f"{tag} {k}: {len(bad)} entries differ, first at {bad[0].tolist()}: "
                                 f"{a[k][tuple(bad[0])]} vs {b[k][tuple(bad[0])]}")


def _set_path(env, path):
    for k, v in dict(DEFAULT_OPTIONS, **PATHS[path]).items():
        env.set_option(k, v)


def _run(env, path, calls):
    """`calls` calls of `path` with the env's default sampler counters; yields after each one"""
    torch = __import__("torch")
    _set_path(env, path)
    graph = counter = None
    for i in range(calls):
        if path in ("fused", "two_kernels", "bulk"):
            env.step(env.sample_actions())
        elif path in ("lagged", "unlagged"):
            env.step_deferred(env.sample_actions())
        elif path in ("rollout", "per_step"):
            env.rollout_random(SEG)
        elif path == "graph":
            if graph is None:
                graph, counter = env.capture_rollout(SEG)  # its warm-up call is the first SEG steps
            else:
                graph.replay()
            # the counter tensor is the caller's: the next default draw continues after the replayed steps
            env._sample_counter = int(counter.item())
        elif i % 2 == 0:
            env.step_host(env.sample_actions_host())
        else:
            env.host_rollout_random(2, flags="per_agent")
        torch.cuda.synchronize()
        yield i


def _roundtrip(sd):
    torch = __import__("torch")
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    return torch.load(buf)


def _same_stats(a, b, tag, groups=False):
    assert a.stats() == b.stats(), tag
    assert a.metrics() == b.metrics(), tag
    if groups:
        assert a.stats(by_group=True) == b.stats(by_group=True), tag
        assert a.metrics(by_group=True) == b.metrics(by_group=True), tag


def _oracle_stats(env, ob, tag):
    """the handle's step and episode counts against the oracle (auto-reset batches)"""
    st = env.stats()
    assert st["env_steps"] == env.num_envs * ob.counter, tag
    assert st["episodes"] == int(np.asarray(ob.ob._episode).sum()), tag


RESUME_CASES = [
    ("c2", "fused", "two_kernels"), ("c2", "rollout", "graph"), ("c2", "host", "lagged"),
    ("c3", "two_kernels", "bulk"), ("c3", "lagged", "unlagged"), ("c3", "per_step", "host"),
    ("c3", "graph", "per_step"), ("c3", "unlagged", "fused"), ("c3", "rollout", "lagged"),
    ("c3_full", "lagged", "two_kernels"),
    ("c4", "unlagged", "two_kernels"), ("p15", "fused", "lagged"), ("u8", "bulk", "fused"),
    ("frozen", "two_kernels", "rollout"), ("pool", "lagged", "fused"), ("pool", "host", "graph"),
    ("pool", "per_step", "bulk"),
]


@pytest.mark.parametrize("shape,before,after", RESUME_CASES)
def test_restored_handle_continues_like_its_uninterrupted_twin(torch_cuda, shape, before, after):
    """The twin runs `before`, its state_dict goes through torch.save / torch.load into a fresh handle that was never
    reset, and both run `after` with default sampler counters: byte-equal after every call, the twin on the oracle."""
    sh = SHAPES[shape]
    big = sh["B"] > 10000
    calls = (2, 2) if big else (6, 6)
    pool = _pool(sh)
    twin, restored = _env(sh, pool), _env(sh, pool)
    ob = _Follower(_oracle(sh, pool))
    twin.reset()
    ob.check(twin, "reset")
    for i in _run(twin, before, calls[0]):
        ob.check(twin, (before, i))
    sd = twin.state_dict()
    assert not twin.observations_pending  # the dict holds the dense observations of the current state
    ob.check(twin, "saved")
    for k in STATE + DENSE:
        if k in sd:
            assert sd[k].cpu().numpy().tobytes() == getattr(twin, k).cpu().numpy().tobytes(), k
    assert int(sd["sample_counter"]) == twin._sample_counter == ob.counter
    restored.load_state_dict(_roundtrip(sd))
    assert restored._sample_counter == twin._sample_counter and restored.config.seed == twin.config.seed
    _equal(_snap(restored, STATE + DENSE), _snap(twin, STATE + DENSE), "loaded")
    for i, _ in zip(_run(twin, after, calls[1]), _run(restored, after, calls[1])):
        _equal(_snap(restored), _snap(twin), (after, i))
        if not big or i == calls[1] - 1:
            ob.check(twin, (after, i))
    twin.flush_observations()
    restored.flush_observations()
    _equal(_snap(restored), _snap(twin), "flushed")
    ob.check(twin, "flushed")
    _same_stats(restored, twin, "stats")
    if sh.get("auto_reset", True):
        _oracle_stats(twin, ob, "oracle stats")
    twin.close()
    restored.close()


@pytest.mark.parametrize("shape", ["c2", "c3"])
def test_save_while_pending_and_load_while_pending(torch_cuda, shape):
    """A dict taken right after step_deferred equals, dense tensors and belief included, a twin that stepped plainly
    (the same observation kernel wrote both).  Loaded into a fresh handle and into a handle that has observations of
    its own pending, it continues exactly like that twin, statistics included."""
    sh = SHAPES[shape]
    pool = _pool(sh)
    plain, deferred, fresh, busy = (_env(sh, pool) for _ in range(4))
    for e in (plain, fresh, busy):
        _set_path(e, "two_kernels")
    _set_path(deferred, "lagged")
    ob = _oracle(sh, pool)
    plain.reset()
    deferred.reset()
    busy.reset(seed=99)
    for s in range(9):
        a = plain.sample_actions(step_counter=s)
        plain.step(a)
        deferred.step_deferred(a)
        busy.step_deferred(busy.sample_actions(step_counter=s))
        want = ob.step(ob.sample_actions(s))
    assert deferred.observations_pending and busy.observations_pending
    sd = deferred.state_dict()
    _compare(plain, ob, want, sh["belief"], "plain twin")
    for k in STATE + DENSE:
        if k in sd:
            assert sd[k].cpu().numpy().tobytes() == getattr(plain, k).cpu().numpy().tobytes(), ("dict", k)
    fresh.load_state_dict(sd)
    busy.load_state_dict(sd)
    assert not busy.observations_pending
    _set_path(deferred, "two_kernels")
    for h in (fresh, busy, deferred):
        _equal(_snap(h, STATE + DENSE), _snap(plain, STATE + DENSE), "loaded")
    for s in range(9, 17):
        a = plain.sample_actions(step_counter=s)
        for h in (plain, deferred, fresh, busy):
            h.step(a)
        want = ob.step(ob.sample_actions(s))
        for h, name in ((deferred, "saved"), (fresh, "fresh"), (busy, "busy")):
            _equal(_snap(h), _snap(plain), (name, s))
    _compare(plain, ob, want, sh["belief"], "end")
    for h in (deferred, fresh, busy):
        _same_stats(h, plain, "stats")
    for h in (plain, deferred, fresh, busy):
        h.close()


@pytest.mark.parametrize("path", ["two_kernels", "lagged", "rollout"])
@pytest.mark.parametrize("stats_between", [False, True])
def test_rewind_in_the_same_handle(torch_cuda, path, stats_between):
    """save at t, run k, load, rerun the same k: both passes are byte-identical, and stats() counts the k steps once
    (equal to a twin that ran t + k steps) whether or not stats() was called between the save and the load."""
    sh = SHAPES["c3"]
    pool = _pool(sh)
    h, twin = _env(sh, pool), _env(sh, pool)
    ob = _Follower(_oracle(sh, pool))
    for e in (h, twin):
        e.reset()
        for _ in _run(e, path, 4):
            pass
    sd = h.state_dict()
    twin.flush_observations()  # what state_dict does to `h`
    first = [_snap(h) for _ in _run(h, path, 5)]
    if stats_between:
        h.stats()
    h.load_state_dict(sd)
    assert h._sample_counter == int(sd["sample_counter"])
    second = [_snap(h) for _ in _run(h, path, 5)]
    for i, (a, b) in enumerate(zip(first, second)):
        _equal(b, a, ("second pass", i))
    for i, _ in enumerate(_run(twin, path, 5)):
        _equal(_snap(twin), second[i], ("twin", i))
    for e in (h, twin):
        e.flush_observations()
    _same_stats(h, twin, "stats")
    ob.check(twin, "end")
    _oracle_stats(twin, ob, "oracle stats")
    h.close()
    twin.close()


GROUP_MECHS = [
    dict(number_of_agents=2, tolls=0, max_timestep=8),
    dict(number_of_agents=5, tolls=2, max_timestep=20, agent_money=30),
    dict(number_of_agents=6, tolls=1, max_timestep=12, reveal_interval=3, reveal_skip_prob=0.5),
]


@pytest.mark.parametrize("stats_between", [False, True])
def test_rewind_with_mechanism_groups(torch_cuda, stats_between):
    """The rewind with mixed police counts, tolls and horizons: the per-group statistics count the rerun steps once and
    equal the twin's and the oracle's.  A new handle with the same groups accepts the dict but refuses to step before
    the full reset that set_mechanisms requires; after it the statistics carry over."""
    torch = torch_cuda
    sh = dict(SHAPES["c3"], N=60, E=130, B=230)
    pool = _pool(sh)
    h, twin = _env(sh, pool), _env(sh, pool)
    for e in (h, twin):
        e.set_mechanisms(GROUP_MECHS)
        e.reset()
    cfgs = [so.OracleConfig(num_police=m["number_of_agents"], agent_money=m["agent_money"], toll=m["tolls"],
                            reward_weights=dict(m["reward_weights"]), max_timestep=m["max_timestep"],
                            reveal_interval=m["reveal_interval"], reveal_skip_prob=m["reveal_skip_prob"], belief=True)
            for m in h.mechanisms]
    graphs = [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in pool]
    ob = so.OracleGroupBatch.from_seed(cfgs, h.group_id.cpu().numpy(), sh["P"], graphs, sh["B"], seed=S1)
    for s in range(6):
        a = h.sample_actions()
        assert np.array_equal(a.cpu().numpy(), ob.sample_actions(s)), s
        h.step(a)
        twin.step(twin.sample_actions())
        ob.step(a.cpu().numpy())
    sd = h.state_dict()
    first = []
    for s in range(6, 16):
        h.step(h.sample_actions())
        first.append(_snap(h))
    if stats_between:
        h.stats(by_group=True)
    h.load_state_dict(sd)
    for i, s in enumerate(range(6, 16)):
        a = h.sample_actions()
        h.step(a)
        _equal(_snap(h), first[i], ("second pass", s))
        twin.step(twin.sample_actions())
        _equal(_snap(twin), first[i], ("twin", s))
        ob.step(a.cpu().numpy())
    _same_stats(h, twin, "stats", groups=True)
    total, per = ob.expected_stats()
    names = _pkg()._cabi.STAT_NAMES
    for g, (got, want) in enumerate(zip(h.stats(by_group=True), per)):
        assert [got[k] for k in names[:14]] == want[:14], ("group", g)
    assert [h.stats()[k] for k in names[:14]] == total[:14]

    new = _env(sh, pool)
    new.set_mechanisms(GROUP_MECHS)
    new.load_state_dict(sd)
    with pytest.raises(_pkg().SyError):
        new.step(torch.full((sh["B"], sh["P"] + 1), -1, dtype=torch.int64, device=new.device))
    new.reset()
    assert new.stats(by_group=True) == [{k: int(v) for k, v in zip(names, row)} for row in sd["group_stats_vec"].tolist()]
    for e in (h, twin, new):
        e.close()


def _shard_state(sd, lo, hi, first):
    """the slice [lo, hi) of a state dict, as a handle with env_offset = lo would hold it; the statistics go to the
    first shard so that the shards' sum stays the whole batch's"""
    B = sd["pos"].shape[0]
    out = {}
    for k, v in sd.items():
        if k == "env_offset":
            out[k] = v.new_tensor(int(v) + lo)
        elif k == "stats_vec":
            out[k] = v.clone() if first else v.new_zeros(v.shape)
        elif v.dim() > 0 and v.shape[0] == B and k not in ("graph_pool_sha256",):
            out[k] = v[lo:hi].clone()
        else:
            out[k] = v.clone()
    return out


def test_resume_on_uneven_shards(torch_cuda):
    """A 4 099-env dict cut into shards of 1 000 / 1 900 / 1 199 envs, each loaded into a handle with env_offset = its
    start: every shard steps exactly as its slice of the whole handle, and the shards' statistics sum to the whole's."""
    sh = SHAPES["c3"]
    pool = _pool(sh)
    full = _env(sh, pool)
    full.reset()
    for s in range(8):
        full.step(full.sample_actions(step_counter=s))
    sd = full.state_dict()
    bounds = [(0, 1000), (1000, 2900), (2900, sh["B"])]
    shards = []
    for i, (lo, hi) in enumerate(bounds):
        e = _env(sh, pool, num_envs=hi - lo, env_offset=lo)
        e.load_state_dict(_shard_state(sd, lo, hi, i == 0))
        shards.append(e)
    for s in range(8, 20):
        full.step(full.sample_actions(step_counter=s))
        want = _snap(full)
        for e, (lo, hi) in zip(shards, bounds):
            e.step(e.sample_actions(step_counter=s))
            _equal(_snap(e), {k: v[lo:hi] for k, v in want.items()}, ("shard", lo, s))
    st = [e.stats() for e in shards]
    assert {k: sum(x[k] for x in st) for k in st[0]} == full.stats()
    for e in shards + [full]:
        e.close()


RESEED_CASES = [(p, SEEDS[i % len(SEEDS)]) for i, p in enumerate(PATHS)] + [("two_kernels", -1), ("lagged", U64)]


@pytest.mark.parametrize("path,s2", RESEED_CASES)
def test_reset_with_a_new_seed_equals_a_fresh_handle(torch_cuda, path, s2):
    """reset(seed=s2) on a handle that ran under S1 is byte-identical from then on to a handle built with s2 (-1 is
    2^64 - 1), on the 5-graph pool with graph resampling and reveal skips, and both follow the oracle keyed with s2."""
    sh = SHAPES["pool"]
    pool = _pool(sh)
    h, fresh = _env(sh, pool, seed=S1), _env(sh, pool, seed=s2 & U64)
    h.reset()
    for s in range(7):  # explicit counters: the default one stays at 0, as in the fresh handle
        h.step(h.sample_actions(step_counter=s))
    h.reset(seed=s2)
    fresh.reset()
    assert h.config.seed == fresh.config.seed == s2 & U64
    _equal(_snap(h, STATE + DENSE), _snap(fresh, STATE + DENSE), "reset")
    ob = _Follower(_oracle(sh, pool, s2))
    ob.check(h, "reset")
    for i, _ in zip(_run(h, path, 5), _run(fresh, path, 5)):
        _equal(_snap(h), _snap(fresh), (path, i))
        ob.check(h, (path, i))
    h.close()
    fresh.close()


@pytest.mark.parametrize("path", ["fused", "lagged", "per_step", "host"])
def test_set_seed_mid_episode_switches_every_later_draw(torch_cuda, path):
    """set_seed(s2) without a reset: the sampler, the same-step auto-reset start nodes and graph choice and the reveal
    skips of every later step use s2, exactly as the oracle whose seed switches at that step; one kept at S1 diverges."""
    sh = SHAPES["pool"]
    pool = _pool(sh)
    env = _env(sh, pool)
    ob = _Follower(_oracle(sh, pool))
    kept = _Follower(_oracle(sh, pool))
    env.reset()
    for i in _run(env, path, 4):
        ob.check(env, ("before", i))
    ob.to(env._sample_counter)
    s2 = 2 ** 32 + 7
    env.set_seed(s2)
    ob.ob.set_seed(s2)
    episodes = int(env.episode.sum())
    for i in _run(env, path, 8):
        ob.check(env, ("after", i))
    assert int(env.episode.sum()) > episodes  # auto-resets drew under s2
    kept.to(env._sample_counter)
    assert not np.array_equal(kept.ob.pos(), env.pos.cpu().numpy())
    env.close()


def test_policies_follow_the_new_key(torch_cuda):
    """HeuristicPolicy exploration and masked_sample_device with seed=env.seed draw with the key set by set_seed."""
    torch = torch_cuda
    from student_mechanism_design_b200.rollout import masked_sample_device

    sh = dict(SHAPES["pool"], B=192)
    pool = _pool(sh)
    env = _env(sh, pool, num_envs=sh["B"])
    graphs = [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in pool]
    cfg = so.OracleConfig(num_police=sh["P"], agent_money=sh["money"], toll=sh["toll"], belief=True,
                          reveal_interval=sh["reveal"], reveal_skip_prob=sh["skip"])
    ob = so.OracleBatch.from_seed(cfg, graphs, sh["B"], seed=S1, auto_reset=True, resample_graph=True)
    heur = _pkg().HeuristicPolicy(env, "evade", "chase", epsilon_mrx=0.4, epsilon_police=0.4)
    env.reset()
    ls = np.full(sh["B"], -1, dtype=np.int32)
    g = torch.Generator().manual_seed(0)
    N, A = sh["N"], sh["P"] + 1
    for s in range(12):
        if s == 5:
            env.set_seed(2 ** 64 - 3)
            ob.seed = 2 ** 64 - 3
        a = heur.act()
        want, ls = ho.batch_heuristic_actions(ob, s, ho.HEUR_EVADE, ho.HEUR_CHASE, heur._h.explore_mrx,
                                              heur._h.explore_police, last_seen=ls)
        assert np.array_equal(a.cpu().numpy(), want), s
        logits = (torch.randn(sh["B"], A, N, generator=g) * 2).to(env.device)
        got = masked_sample_device(logits, env.action_mask, seed=env.seed, step_counter=s).cpu().numpy()
        j = np.arange(N)
        r = po.philox4x32_batched(np.arange(sh["B"])[:, None, None], s, 5 + 16 * np.arange(A)[None, :, None],
                                  (j >> 2)[None, None, :], env.seed & U64)
        uu = ((np.choose(j & 3, r) >> 8).astype(np.float64) + 0.5) / 16777216.0
        mask = env.action_mask.cpu().numpy()
        keys = np.where(mask, logits.cpu().numpy().astype(np.float64) - np.log(-np.log(uu)), -np.inf)
        legal = mask.any(-1)
        assert (got[~legal] == -1).all()
        gk = np.take_along_axis(keys, np.clip(got, 0, N - 1)[..., None], -1)[..., 0]
        assert (gk[legal] >= keys.max(-1)[legal] - 1e-4).all(), s
        env.step(a)
        ob.step(want)
    env.close()


def test_torchrl_adapter_set_seed_rekeys_the_env(torch_cuda):
    """The torchrl adapter's set_seed re-keys the handle: its first reset and steps equal a handle built with that
    seed (tests/fake_torchrl.py stands in for torchrl)."""
    import fake_torchrl
    from student_mechanism_design_b200 import torchrl_env

    sh = SHAPES["pool"]
    pool = _pool(sh)
    env, fresh = _env(sh, pool), _env(sh, pool, seed=U64)
    adapter = torchrl_env.make_env_class(fake_torchrl.EnvBase, fake_torchrl.TensorDict, fake_torchrl.SPECS)(env)
    adapter.set_seed(-1)
    assert env.config.seed == U64
    adapter.reset()
    fresh.reset()
    _equal(_snap(env, STATE + DENSE), _snap(fresh, STATE + DENSE), "reset")
    for s in range(6):
        a = fresh.sample_actions(step_counter=s)
        assert torch_cuda.equal(env.sample_actions(step_counter=s), a)
        adapter.step(fake_torchrl.TensorDict({("agents", "action"): a}, batch_size=[sh["B"]]))
        fresh.step(a)
        _equal(_snap(env), _snap(fresh), ("step", s))
    env.close()
    fresh.close()


def test_refused_loads_change_nothing(torch_cuda):
    """load_state_dict raises ValueError, with the target untouched, for a dict of another env_offset, graph pool, B,
    N, A, node-feature type or key set (belief map, statistics, mechanism groups, a missing entry)."""
    sh = dict(SHAPES["pool"], N=30, E=60, B=64)
    pool = _pool(sh)
    src = _env(sh, pool)
    src.reset()
    src.step(src.sample_actions())
    sd = src.state_dict()
    other_n = dict(sh, N=31)
    targets = {
        "env_offset": lambda: _env(sh, pool, env_offset=64),
        "pool": lambda: _env(sh, _pool(sh, seed=1)),
        "B": lambda: _env(sh, pool, num_envs=65),
        "N": lambda: _env(other_n, _pool(other_n)),
        "A": lambda: _env(sh, pool, num_police=sh["P"] + 1),
        "nf_dtype": lambda: _env(dict(sh, nf="uint8"), pool),
        "belief_off": lambda: _env(sh, pool, belief=False, belief_ce=False),
        "stats_off": lambda: _env(sh, pool, collect_stats=False),
        "groups": lambda: _env(sh, pool),
        "missing_key": lambda: _env(sh, pool),
    }
    for name, make in targets.items():
        t = make()
        if name == "groups":
            t.set_mechanisms([GROUP_MECHS[0], dict(tolls=2)])
        t.reset(seed=123)
        t.step(t.sample_actions())
        bad = {k: v for k, v in sd.items() if k != "seed"} if name == "missing_key" else sd
        before, stats_before, counter = _snap(t), (t.stats_vec.clone() if t.stats_vec is not None else None), t._sample_counter
        with pytest.raises(ValueError):
            t.load_state_dict(bad)
        _equal(_snap(t), before, name)
        assert t.config.seed == 123 and t._sample_counter == counter, name
        if stats_before is not None:
            assert __import__("torch").equal(t.stats_vec, stats_before), name
        t.close()
    src.close()


def test_rollout_graph_refuses_replay_after_set_seed(torch_cuda):
    """A rollout graph keeps the key of its capture: after set_seed (or reset(seed=...)) replaying it raises SyError,
    and a graph captured again matches a handle built with the new seed."""
    sh = SHAPES["c2"]
    pool = _pool(sh)
    h, fresh = _env(sh, pool), _env(sh, pool, seed=2 ** 32 + 7)
    h.reset()
    graph, _ = h.capture_rollout(SEG)
    graph.replay()
    h.set_seed(S1)  # the same key: still replayable
    graph.replay()
    h.set_seed(2 ** 32 + 7)
    with pytest.raises(_pkg().SyError):
        graph.replay()
    h.reset(seed=2 ** 32 + 7)
    fresh.reset()
    with pytest.raises(_pkg().SyError):
        graph.replay()
    g2, c2 = h.capture_rollout(SEG)
    gf, cf = fresh.capture_rollout(SEG)
    for i in range(3):
        g2.replay()
        gf.replay()
        torch_cuda.cuda.synchronize()
        assert int(c2.item()) == int(cf.item())
        _equal(_snap(h), _snap(fresh), ("replay", i))
    h.close()
    fresh.close()
