"""Incremental node_features: which write path each call takes, and oracle parity of the in-place update at every
granule, alignment and agent count it accepts.

A plain two-kernel step into the float32 buffer the handle's previous call completed, for the same `pos` /
`mrx_revealed`, updates the one-hot in place (include/sy_env.h, SyObs): the dynamics kernel zeroes the granules --
32-byte sectors, or 16-byte chunks where the env rows are only 16-byte aligned -- that hold the entry state's ones, the
observation kernel stores only the granules of the new ones.  Every other call writes the whole one-hot.  Values alone
cannot tell the two paths apart, so the tests here watch the write path itself with a probe (`_Probe`): a float that
neither path's stores should touch on the fast path, set before a call and read after it.

1. `test_write_path_table`: sequences of calls, each call's path (full / fast at granule 8 / fast at granule 4) and the
   values after it.
2. `test_fast_path_matches_oracle` / `test_fast_path_through_c_abi_views` / `test_fast_path_groups_match_oracle`: the
   whole state, masks, node features and belief map against the C oracle (the group oracle for mechanism groups) after
   every step, at every agent count (logic kernel instantiations for up to 4, 8 and 16 agents, both reward modes),
   both granules and the full-write fallback, with the probe asserting that each row took the path it covers.
3. `test_package_consumers_leave_the_buffer_alone`: the torchrl adapter, RolloutCollector and a GNN policy on env
   features hand out the live buffer; since the in-place update, a stray write into it would persist."""
import ctypes as C

import numpy as np
import pytest

import sy_oracle as so
import sy_oracle_c as oc
from test_gpu_fullsize import _compare, _threads, torch_cuda  # noqa: F401
from test_gpu_mechanisms_oracle import _check as _check_groups
from test_gpu_mechanisms_oracle import _check_out as _check_groups_out
from test_gpu_mechanisms_oracle import _ocfg
from test_gpu_nf_incremental import _onehot

pytestmark = pytest.mark.gpu

FULL = "full"  # probe outcomes: the rows were rewritten whole | 8 / 4: updated in place with granules of that many floats


def _pkg():
    import student_mechanism_design_b200 as pkg

    return pkg


def _torch():
    return __import__("torch")


# ----------------------------------------------------------------------------------------------------------- the probe
class _Probe:
    """Tells the in-place update of node_features from a full write, and its granule, by watching floats the fast path
    leaves alone.

    `arm()` (before a call, the buffer an exact one-hot) picks, in each of a few envs spread over the tiles (the ragged
    last tile included), up to three "free" floats in 32-byte sectors that hold none of the env's ones, and up to two
    "half" floats in the other 16-byte half of a sector that holds an entry one in one half only; it sets them all to
    `value` (finite).  `read()` (after the call, no observations pending) looks at them again, ignores every probe
    whose sector now holds a new one, and sets the survivors back to 0, so that the buffer is again exactly the one-hot
    the library wrote.  The probes take the buffer outside the SyObs precondition for the duration of one call only,
    and only in granules the fast path does not touch: neither the entry ones' granules (zeroed by the dynamics kernel)
    nor the new ones' (stored by the writers).

    Per env: a free probe that survived = the row was not rewritten (fast path), one cleared = rewritten whole.  A half
    probe survives granule 4 (only the entry one's 16-byte chunk is zeroed) and is cleared by granule 8 (the whole
    sector) and by a full write.  Sectors are counted from 32-byte aligned addresses, so views at any 4-byte offset work.
    Float32 and uint8 buffers (32 / 16 elements per sector and half); only the free probes mean something for uint8."""

    def __init__(self, nf, value=None, n_envs=8):
        torch = _torch()
        self.nf = nf
        self.value = value if value is not None else (0.5 if nf.dtype == torch.float32 else 2)
        B, N, A = nf.shape
        self.B, self.NA = B, N * A
        es = nf.element_size()
        self.per = 32 // es  # elements per 32-byte sector
        self.shift = (nf.data_ptr() % 32) // es  # element index of the view's first element within its sector
        assert (nf.data_ptr() % es) == 0 and nf.is_contiguous()
        spread = [0, 1, 33, B // 3, B // 2 + 5, (2 * B) // 3 + 7, B - 40, B - 2, B - 1]
        self.envs = sorted({min(max(b, 0), B - 1) for b in spread})[:max(n_envs, 1)] if B > 1 else [0]
        self.rng = np.random.default_rng(1234)
        self.probes = None

    def _sector_range(self, s):
        lo = s * self.per - self.shift
        return lo, lo + self.per

    def arm(self, envs=None):
        torch = _torch()
        envs = self.envs if envs is None else envs
        rows = self.nf[envs].reshape(len(envs), -1).cpu().numpy()
        probes = []  # (env, kind, flat index, sector)
        for k, b in enumerate(envs):
            row = rows[k]
            ones = np.nonzero(row)[0]
            assert np.all(row[ones] == 1), ("the buffer is not a one-hot before the probed call", b)
            base = b * self.NA
            s_lo = -(-(base + self.shift) // self.per)  # sectors that lie wholly inside the row
            s_hi = (base + self.NA + self.shift) // self.per
            busy = set(((ones + base + self.shift) // self.per).tolist())
            free = [s for s in range(s_lo, s_hi) if s not in busy]
            for s in self.rng.permutation(free)[:3]:
                lo, _ = self._sector_range(int(s))
                probes.append((b, "free", lo + int(self.rng.integers(self.per)), int(s)))
            if self.nf.dtype != torch.float32:
                continue
            halves = {}
            for o in ones + base:
                s = (o + self.shift) // self.per
                halves.setdefault(int(s), set()).add(int((o + self.shift) % self.per) // (self.per // 2))
            cand = [(s, h.pop()) for s, h in halves.items() if len(h) == 1 and s_lo <= s < s_hi]
            for i in self.rng.permutation(len(cand))[:2]:
                s, h = cand[int(i)]
                lo, _ = self._sector_range(s)
                half = self.per // 2
                other = lo + (1 - h) * half
                probes.append((b, "half", other + int(self.rng.integers(half)), s))
        idx = torch.tensor([p[2] for p in probes], dtype=torch.int64, device=self.nf.device)
        self.nf.view(-1)[idx] = self.value
        self.probes = probes

    def read(self):
        """{env: (free probes kept, free probes cleared, half probes kept, half probes cleared)} over the conclusive
        probes; restores the buffer"""
        torch = _torch()
        probes, self.probes = self.probes, None
        assert probes is not None, "read() without arm()"
        flat = self.nf.view(-1)
        torch.cuda.synchronize()
        got = {}
        restore = []
        for b, kind, i, s in probes:
            lo, hi = self._sector_range(s)
            sector = flat[lo:hi].cpu().numpy()
            v = sector[i - lo]
            if v == self.value:
                restore.append(i)
            if np.any(sector == 1):  # a new one landed in the probe's sector: the probe says nothing
                continue
            assert v in (0, self.value), ("probe value neither kept nor cleared", b, kind, float(v))
            r = got.setdefault(b, [0, 0, 0, 0])
            r[(0 if kind == "free" else 2) + (0 if v == self.value else 1)] += 1
        if restore:
            flat[torch.tensor(restore, dtype=torch.int64, device=self.nf.device)] = 0
        return got

    @staticmethod
    def verdict(got, tag):
        """the path of the whole call: FULL, 8 or 4 -- or "fast" where no env showed its granule (which no expected
        outcome accepts); every probed env must agree"""
        kinds = set()
        for b, (fk, fc, hk, hc) in got.items():
            assert not (fk and fc), (tag, "env rewritten in part", b, got[b])
            if fc:
                assert hk == 0, (tag, "half probe survived a full write", b)
                kinds.add(FULL)
            elif fk:
                kinds.add("fast" if hk == hc == 0 else (4 if hk and not hc else 8 if hc and not hk else "mixed"))
        assert kinds, (tag, "no conclusive probe")
        assert "mixed" not in kinds, (tag, "half probes of one env disagree", got)
        granules = kinds - {"fast"}
        if FULL not in kinds and len(granules) <= 1:
            return granules.pop() if granules else "fast"
        assert len(kinds) == 1, (tag, "envs took different paths", got)
        return kinds.pop()


def _probed(nf, call, want, tag, probe=None):
    """run call() with the probe armed on nf; assert the path it took"""
    probe = probe or _Probe(nf)
    probe.arm()
    r = call()
    got = _Probe.verdict(probe.read(), tag)
    assert got == want, (tag, "write path", got, "expected", want)
    return r


# ---------------------------------------------------------------------------------------------------- 1: the path table
def _env(N=200, P=6, B=4099, *, E=None, money=12, reveal=3, step_kernel="two_kernels", **kw):
    pool = _pkg().generate_graph_pool(kw.pop("graphs", 2), N, E or 2 * N, seed=0)
    env = _pkg().BatchedScotlandYardEnv(B, P, money, graphs=pool, seed=kw.pop("seed", 5), tolls=1, belief=True,
                                        reveal_interval=reveal, auto_reset=True, **kw)
    env.set_option("step_kernel", step_kernel)
    return env


def _values(env, tag):
    torch = _torch()
    assert not env.observations_pending, tag
    assert torch.equal(env.node_features, _onehot(env).to(env.node_features.dtype)), (tag, "node_features")


def _step(env):
    return lambda: env.step(env.sample_actions())


def _cabi_step(env, nf, acts=None, no_out=False):
    """sy_step through the C ABI with `nf` as the float32 node_features (the env's other buffers; no_out: SyOut NULL)"""
    torch = _torch()
    from student_mechanism_design_b200 import _cabi

    acts = env.sample_actions() if acts is None else acts
    obs = _cabi.SyObs(env.action_mask.data_ptr(), nf.data_ptr(), env.agent_budget.data_ptr(), env.mrx_revealed.data_ptr(),
                      None)
    with torch.cuda.device(env.device):
        _cabi.check(env._lib.sy_step(env._handle, acts.data_ptr(), C.byref(env._state), C.byref(obs),
                                     None if no_out else C.byref(env._out), env._stream()))
    return acts


def _view(env, offset_bytes):
    """a float32 [B, N, A] view at `offset_bytes` (a multiple of 4) into a larger zeroed allocation"""
    torch = _torch()
    n = env.node_features.numel()
    raw = torch.zeros(n + 64, dtype=torch.float32, device=env.device)
    assert raw.data_ptr() % 256 == 0 and offset_bytes % 4 == 0
    k = offset_bytes // 4
    return raw, raw[k:k + n].view(env.node_features.shape)


def _seq_reset(env):
    _probed(env.node_features, env.reset, FULL, "full reset")
    _values(env, "reset")
    _probed(env.node_features, _step(env), 8, "step after reset")


def _seq_granule(want):
    def run(env):
        env.reset()
        for s in range(3):
            _probed(env.node_features, _step(env), want, ("plain step", s))
            _values(env, ("plain step", s))
    return run


def _seq_option(name, on, off):
    def run(env):
        env.reset()
        env.step(env.sample_actions())
        env.set_option(name, on)
        _probed(env.node_features, _step(env), FULL, (name, on))
        _values(env, (name, on))
        env.set_option(name, off)
        _probed(env.node_features, _step(env), 8, (name, off, "next"))
        _values(env, (name, off))
    return run


def _seq_fast_option(name, value):
    def run(env):
        env.set_option(name, value)
        env.reset()
        for s in range(3):
            _probed(env.node_features, _step(env), 8, (name, value, s))
            _values(env, (name, value, s))
    return run


def _seq_deferred(flush):
    def run(env):
        env.reset()
        env.step(env.sample_actions())
        env.step_deferred(env.sample_actions())
        assert env.observations_pending
        if flush:
            _probed(env.node_features, env.flush_observations, FULL, "flush")
        else:
            _probed(env.node_features, _step(env), FULL, "plain step after a deferred one")
        _values(env, "after deferred")
        _probed(env.node_features, _step(env), 8, "next plain step")
        _values(env, "next")
    return run


def _seq_rollout(env):
    env.reset()
    env.step(env.sample_actions())
    n0 = env._lib.sy_launch_count()
    _probed(env.node_features, lambda: env.rollout_random(4), FULL, "one-launch rollout")
    assert env._lib.sy_launch_count() - n0 == 2, "the rollout was not one launch (after the first draw)"
    _values(env, "rollout")
    _probed(env.node_features, _step(env), 8, "plain step after the rollout")
    _values(env, "after rollout")


def _seq_partial_reset(env):
    """the reset's observation kernel rewrites every env's row, the reset envs' and the others' (the observe kernel
    does not look at the mask); a valid record is kept"""
    torch = _torch()
    env.reset()
    env.step(env.sample_actions())
    mask = torch.arange(env.num_envs, device=env.device) % 3 == 0
    _probed(env.node_features, lambda: env.reset(reset_mask=mask), FULL, "partial reset")
    _values(env, "partial reset")
    _probed(env.node_features, _step(env), 8, "step after the partial reset")
    _values(env, "after partial reset")


def _seq_second_buffer(env):
    """a call into another buffer moves the record there: the own buffer (an older state's one-hot) is written whole,
    and a partial reset of the own buffer does not take the record back"""
    torch = _torch()
    env.reset()
    env.step(env.sample_actions())
    other = torch.zeros_like(env.node_features)
    _probed(other, lambda: _cabi_step(env, other), FULL, "first call into a second buffer")
    assert torch.equal(other, _onehot(env))
    _probed(other, lambda: _cabi_step(env, other), 8, "second call into the second buffer")
    assert torch.equal(other, _onehot(env))
    _probed(env.node_features, _step(env), FULL, "back to the own buffer")
    _values(env, "own buffer")
    _cabi_step(env, other)
    mask = torch.arange(env.num_envs, device=env.device) % 2 == 1
    _probed(env.node_features, lambda: env.reset(reset_mask=mask), FULL, "partial reset of the own buffer")
    _values(env, "partial reset")
    _probed(env.node_features, _step(env), FULL, "step after a partial reset that did not keep the record")
    _values(env, "step after partial reset")
    _probed(env.node_features, _step(env), 8, "next")
    _values(env, "next")


def _seq_load_state_dict(env):
    env.reset()
    for _ in range(2):
        env.step(env.sample_actions())
    sd = env.state_dict()
    for _ in range(3):
        env.step(env.sample_actions())
    env.load_state_dict(sd)
    _values(env, "rewound")
    _probed(env.node_features, _step(env), 8, "step after load_state_dict")
    _values(env, "after load")


def _seq_step_host(env):
    env.reset()
    env.step(env.sample_actions())
    _probed(env.node_features, lambda: env.step_host(env.sample_actions().cpu()), 8, "step_host")
    _values(env, "step_host")
    _probed(env.node_features, _step(env), 8, "plain step after step_host")
    _values(env, "after step_host")


def _seq_view(offset, want):
    def run(env):
        torch = _torch()
        env.reset()
        _raw, view = _view(env, offset)
        for s in range(3):
            _probed(view, lambda: _cabi_step(env, view), FULL if s == 0 else want, ("view", offset, s))
            assert torch.equal(view, _onehot(env)), ("view", offset, s)
    return run


def _seq_refused(env):
    """refused calls leave the record as it was: a step through the C ABI without SyOut, and steps while mechanism
    groups wait for their reset (the reset then covers every env through a mask, which keeps a valid record)"""
    torch = _torch()
    from student_mechanism_design_b200 import _cabi

    env.reset()
    env.step(env.sample_actions())
    with pytest.raises(_cabi.SyError):
        _cabi_step(env, env.node_features, no_out=True)
    _probed(env.node_features, _step(env), 8, "step after a refused step")
    _values(env, "after refusal")
    env.set_mechanisms([{}, {"agent_money": 9}])
    with pytest.raises(_cabi.SyError):
        env.step(torch.full((env.num_envs, env.num_agents), -1, dtype=torch.int64, device=env.device))
    everyone = torch.ones(env.num_envs, dtype=torch.bool, device=env.device)
    _probed(env.node_features, lambda: env.reset(reset_mask=everyone), FULL, "reset of every env through a mask")
    _values(env, "groups reset")
    _probed(env.node_features, _step(env), 8, "step after the groups' reset")
    _values(env, "groups step")


def _seq_u8(env):
    env.reset()
    for s in range(3):
        _probed(env.node_features, _step(env), FULL, ("uint8", s))
        _values(env, ("uint8", s))


PATH_ROWS = {  # name: (env kwargs, sequence)
    "reset": ({}, _seq_reset),
    "plain_granule8": ({}, _seq_granule(8)),
    "plain_granule4": (dict(N=201, P=3), _seq_granule(4)),
    "plain_full_odd": (dict(N=333, P=4), _seq_granule(FULL)),
    "plain_full_2mod4": (dict(N=202, P=8), _seq_granule(FULL)),
    "fused": ({}, _seq_option("step_kernel", "fused", "two_kernels")),
    "bulk_writer": ({}, _seq_option("writer_path", "bulk", "lsu")),
    "nf_fill": (dict(B=8192 + 37), _seq_fast_option("nf_fill", "on")),  # ignored: the fast path at the old split size
    "pdl": ({}, _seq_fast_option("pdl", "on")),
    "tail_split_off": ({}, _seq_fast_option("tail_split", "off")),
    "deferred_then_plain": ({}, _seq_deferred(False)),
    "deferred_then_flush": ({}, _seq_deferred(True)),
    "one_launch_rollout": (dict(B=2048 + 19), _seq_rollout),
    "partial_reset": ({}, _seq_partial_reset),
    "second_buffer": ({}, _seq_second_buffer),
    "load_state_dict": ({}, _seq_load_state_dict),
    "step_host": ({}, _seq_step_host),
    "view_plus16_granule8_shape": ({}, _seq_view(16, 4)),
    "view_plus16_granule4_shape": (dict(N=201, P=3), _seq_view(16, 4)),
    "view_plus4": ({}, _seq_view(4, FULL)),
    "refused_calls": ({}, _seq_refused),
    "uint8": ("u8", _seq_u8),
}


@pytest.mark.parametrize("row", list(PATH_ROWS))
def test_write_path_table(torch_cuda, row):
    """each call's write path (probe) and the one-hot after it, for the calls that keep, move or drop the handle's
    record of the buffer it last wrote"""
    kw, seq = PATH_ROWS[row]
    if kw == "u8":
        kw = dict(node_features_dtype=torch_cuda.uint8)
    env = _env(**kw)
    seq(env)
    env.close()


# ------------------------------------------------------------------------------------------ 2: oracle parity, fast path
def _pair(N, P, B, *, mode, belief, reveal, money, toll, seed, graphs=2):
    pkg = _pkg()
    torch = _torch()
    pool = pkg.generate_graph_pool(graphs, N, 2 * N, seed=0)
    w = {k: torch.tensor(v, dtype=torch.float32) for k, v in so.DEFAULT_REWARD_WEIGHTS.items()} if mode == "fp32" else None
    env = pkg.BatchedScotlandYardEnv(B, P, money, reward_weights=w, graphs=pool, seed=seed, auto_reset=True, tolls=toll,
                                     belief=belief, reveal_interval=reveal, keep_reward64=True, reward_mode=mode)
    cfg = so.OracleConfig(num_police=P, agent_money=money, toll=toll, belief=belief, reveal_interval=reveal,
                          reward_mode=mode)
    gid = ((np.arange(B) // 32) % graphs).astype(np.int32)
    ob = oc.CBatch(cfg, pool, B, seed=seed, auto_reset=True, threads=_threads(), graph_id=gid)
    return env, ob


# (N, police, B, reward mode, belief, reveal interval, budget, toll, step_kernel, extra option, expected path)
ORACLE_ROWS = {
    "c3_200x7": (200, 6, 4099, "fp64", True, 3, 12, 1, "two_kernels", None, 8),
    "c4_1000x7": (1000, 6, 4099, "fp32", False, 4, 12, 1, "two_kernels", None, 8),
    "201x4": (201, 3, 4099, "fp32", True, 2, 10, 1, "two_kernels", None, 4),
    "202x2": (202, 1, 4099, "fp64", False, 3, 10, 2, "two_kernels", None, 4),
    "200x2": (200, 1, 4099, "fp32", True, 2, 10, 1, "two_kernels", None, 8),
    "50x6_auto": (50, 5, 10539, "fp64", True, 3, 10, 1, "auto", None, 4),
    "199x8": (199, 7, 4099, "fp32", False, 3, 10, 1, "two_kernels", None, 8),
    "101x16": (101, 15, 4099, "fp64", True, 2, 10, 1, "two_kernels", None, 8),
    "501x12_auto": (501, 11, 10539, "fp32", True, 3, 12, 1, "auto", None, 4),
    "333x5_full": (333, 4, 4099, "fp64", True, 3, 10, 1, "two_kernels", None, FULL),
    "202x9_full": (202, 8, 4099, "fp32", False, 2, 10, 1, "two_kernels", None, FULL),
    "c3_65536_pdl": (200, 6, 65536, "fp64", True, 5, 12, 1, "auto", ("pdl", "on"), 8),
    "c3_65536_no_tail_split": (200, 6, 65536, "fp64", True, 5, 12, 1, "auto", ("tail_split", "off"), 8),
}


@pytest.mark.parametrize("row", list(ORACLE_ROWS))
def test_fast_path_matches_oracle(torch_cuda, row):
    """the whole state, action_mask, node_features (exact) and belief_map (1e-6) against the C oracle after every step;
    the probe on every step asserts the row's path; reveals switch MrX's column, small budgets and tolls end episodes
    (same-step auto-resets)"""
    N, P, B, mode, belief, reveal, money, toll, kernel, opt, want = ORACLE_ROWS[row]
    env, ob = _pair(N, P, B, mode=mode, belief=belief, reveal=reveal, money=money, toll=toll, seed=17)
    env.set_option("step_kernel", kernel)
    if opt:
        env.set_option(*opt)
    env.reset()
    _compare(env, ob, None, belief, "reset")
    probe = _Probe(env.node_features)
    steps = 6 if B > 20000 else 10
    ended, hidden, toggles = 0, int((env.mrx_revealed < 0).sum()), 0
    for s in range(steps):
        acts = env.sample_actions(step_counter=s)
        a_h = acts.cpu().numpy()
        assert np.array_equal(a_h, ob.sample_actions(s)), ("sampler", s)
        _probed(env.node_features, lambda: env.step(acts), want, (row, s), probe)
        want_out = ob.step(a_h)
        _compare(env, ob, want_out, belief, (row, s))
        ended += int(want_out["terminated"].sum() + want_out["truncated"].sum())
        now = int((env.mrx_revealed < 0).sum())
        toggles += int(now != hidden)
        hidden = now
    assert ended > 0 and toggles >= 2, (row, ended, toggles)
    env.close()


@pytest.mark.parametrize("offset", [16, 4])
@pytest.mark.parametrize("shape", [(200, 6), (201, 3)])
def test_fast_path_through_c_abi_views(torch_cuda, shape, offset):
    """sy_step through the C ABI into a float32 view at +16 B (16- but not 32-byte aligned: granule 4 after the first,
    full, call) and at +4 B (full writes) of a larger zeroed allocation, against the oracle after every step"""
    torch = torch_cuda
    N, P = shape
    env, ob = _pair(N, P, 4099, mode="fp64", belief=True, reveal=2, money=10, toll=1, seed=23)
    env.set_option("step_kernel", "two_kernels")
    env.reset()
    raw, view = _view(env, offset)
    want = 4 if offset == 16 else FULL
    for s in range(8):
        acts = env.sample_actions(step_counter=s)
        a_h = acts.cpu().numpy()
        assert np.array_equal(a_h, ob.sample_actions(s)), ("sampler", s)
        _probed(view, lambda: _cabi_step(env, view, acts), FULL if s == 0 else want, (shape, offset, s))
        want_out = ob.step(a_h)
        _compare(env, ob, want_out, True, (shape, offset, s), dense=False)
        assert np.array_equal(env.action_mask.cpu().numpy(), ob._mask), (shape, offset, s, "action_mask")
        assert np.array_equal(view.cpu().numpy(), ob._nf), (shape, offset, s, "node_features view")
    k = offset // 4
    assert not bool(raw[:k].any()) and not bool(raw[k + view.numel():].any()), "a store left the view"
    env.close()


GROUP_ROWS = {  # police of the handle, nodes (N * A = 0 mod 8), reward mode, number_of_agents of the groups
    "A4": (3, 40, "fp64", [1, 3, 2]),
    "A8": (7, 41, "fp32", [7, 4, 1]),
    "A16": (15, 40, "fp64", [15, 9, 2]),
}


@pytest.mark.parametrize("row", list(GROUP_ROWS))
def test_fast_path_groups_match_oracle(torch_cuda, row):
    """mechanism groups with fewer police (absent agents skipped by the zeroing loop) on the two-kernel fast path,
    against the group oracle after every step"""
    torch = torch_cuda
    P, N, mode, police = GROUP_ROWS[row]
    T, B = 12, 1100
    pkg = _pkg()
    mechs = [dict(number_of_agents=n, max_timestep=T - 3 * i, agent_money=8 + 4 * i, tolls=1 + (i == 1),
                  reveal_interval=2 + i, reveal_skip_prob=0.0, reward_weights=dict(so.DEFAULT_REWARD_WEIGHTS))
             for i, n in enumerate(police)]
    gid = np.random.default_rng(3).integers(0, len(mechs), B).astype(np.int32)
    pool = pkg.generate_graph_pool(3, N, 2 * N, seed=4)
    tables = pkg.env.numpy_reward_tables(T)
    env = pkg.BatchedScotlandYardEnv(B, P, 10, graphs=pool, seed=9, auto_reset=True, tolls=1, reveal_interval=5,
                                     max_timestep=T, belief=True, keep_reward64=True, reward_mode=mode,
                                     reward_tables=tables)
    env.set_option("step_kernel", "two_kernels")
    env.set_mechanisms(mechs, group_id=torch.as_tensor(gid))
    graphs = [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in pool]
    ob = so.OracleGroupBatch.from_seed([_ocfg(m, mode, tables) for m in mechs], gid, P, graphs, B, seed=9)
    env.reset()
    _check_groups(env, ob, mechs, gid, mode, "reset")
    assert bool((env.pos < 0).any())
    probe = _Probe(env.node_features)
    for s in range(12):
        acts = env.sample_actions(step_counter=s)
        a_h = acts.cpu().numpy()
        assert np.array_equal(a_h, ob.sample_actions(s)), ("sampler", s)
        _probed(env.node_features, lambda: env.step(acts), 8, (row, s), probe)
        want = ob.step(a_h)
        _check_groups_out(env, want, mode, (row, s))
        _check_groups(env, ob, mechs, gid, mode, (row, s))
    env.close()


# ------------------------------------------------------------------------------ 3: consumers of the live buffer
def test_package_consumers_leave_the_buffer_alone(torch_cuda):
    """10 steps each through the torchrl adapter, RolloutCollector with HeuristicPolicy and a GNN policy on env
    features, at 10 539 envs (two kernels, in place): after every step node_features equals the C oracle's, stepped
    with the same actions"""
    torch = torch_cuda
    import fake_torchrl
    from student_mechanism_design_b200 import torchrl_env

    pkg = _pkg()
    B = 10539

    def fresh(seed, reset=True):
        env, ob = _pair(200, 6, B, mode="fp64", belief=True, reveal=3, money=12, toll=1, seed=seed)
        if reset:
            env.reset()
        return env, ob

    def agree(env, ob, acts, tag):
        ob.step(acts.cpu().numpy())
        assert not env.observations_pending, tag
        assert np.array_equal(env.pos.cpu().numpy(), ob.pos()), (tag, "pos")
        assert np.array_equal(env.node_features.cpu().numpy(), ob._nf), (tag, "node_features")

    # the torchrl adapter
    env, ob = fresh(41, reset=False)
    adapter = torchrl_env.make_env_class(fake_torchrl.EnvBase, fake_torchrl.TensorDict, fake_torchrl.SPECS)(env)
    adapter.reset()
    assert np.array_equal(env.node_features.cpu().numpy(), ob._nf), "adapter reset"
    for s in range(10):
        a = env.sample_actions(step_counter=s)
        adapter.step(fake_torchrl.TensorDict({("agents", "action"): a}, batch_size=[B]))
        agree(env, ob, a, ("torchrl", s))
    env.close()

    # RolloutCollector with a heuristic policy that reads the belief map (plain steps, not deferred)
    env, ob = fresh(43)
    heur = pkg.HeuristicPolicy(env, "evade", "chase_belief", epsilon_mrx=0.3, epsilon_police=0.3)
    assert not heur.reads_state_only
    taken = []

    def policy(obs):
        if taken:
            agree(env, ob, taken[-1], ("collector", len(taken)))
        taken.append(heur(obs).clone())
        return taken[-1]
    policy.returns_actions = True
    pkg.RolloutCollector(env, policy, 10).collect()
    agree(env, ob, taken[-1], ("collector", len(taken)))
    env.close()

    # a GNN policy on the env's node_features, plain steps
    env, ob = fresh(47)
    pol = pkg.GNNPolicy(env, features="env", seed=3)
    for s in range(10):
        acts = pol.act(0.2, 0.2, step_counter=s)
        env.step(acts)
        agree(env, ob, acts, ("gnn", s))
    env.close()
