"""Incremental node_features: `node_features` (and `action_mask`) after EVERY call of step sequences that each hit one
way an in-place update of the float32 one-hot could go wrong.

A plain two-kernel step whose float32 `node_features` the library itself last wrote for the current state does not
rewrite the whole [B, N, A] one-hot: the dynamics kernel zeroes the granules that hold the entry state's ones and the
observation kernel stores only the granules of the new ones.  Every other call writes the whole one-hot.  The
sequences below switch between those paths and change the buffer or the state behind the library's back (rewinds,
deferred steps, partial resets, absent agents, a second buffer through the C ABI); the one-hot must be exact after
every call: against the C oracle where a twin batch is driven step by step, and otherwise against the one-hot built
from the env's own `pos` / `mrx_revealed` (which the other GPU tests hold against the oracle).  With a full write on
every step these sequences pass trivially; no other test checks `node_features` after every step of them."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_fullsize import _compare, _pair, torch_cuda  # noqa: F401

pytestmark = pytest.mark.gpu


def _pkg():
    import student_mechanism_design_b200 as pkg

    return pkg


def _onehot(env, pos=None, revealed=None):
    """float32 [B, N, A] one-hot of the env's state (yard.py:279-290): column 0 = MrX while revealed, absent agents blank"""
    torch = __import__("torch")
    pos = env.pos if pos is None else pos
    revealed = env.mrx_revealed if revealed is None else revealed
    B, A = pos.shape
    N = env.node_features.shape[1]
    want = torch.zeros(B, N, A, dtype=torch.float32, device=pos.device)
    on = pos >= 0
    on[:, 0] &= revealed >= 0
    b, a = torch.nonzero(on, as_tuple=True)
    want[b, pos[b, a].long(), a] = 1.0
    return want


def _check(env, tag):
    torch = __import__("torch")
    assert not env.observations_pending, tag
    want = _onehot(env)
    got = env.node_features
    if not torch.equal(got, want):
        bad = torch.nonzero(got != want)
        raise AssertionError(f"{tag}: node_features differ at {bad.shape[0]} entries, first {bad[0].tolist()}: "
                             f"got {got[tuple(bad[0])].item()} want {want[tuple(bad[0])].item()}")


def _oracle_step(env, ob, s, how):
    acts = env.sample_actions(step_counter=s)
    a_h = acts.cpu().numpy()
    assert np.array_equal(a_h, ob.sample_actions(s)), ("sampler", s)
    (env.step_deferred if how == "deferred" else env.step)(acts)
    return ob.step(a_h)


def test_config3_full_size_every_step_matches_oracle(torch_cuda):
    """c3 as benchmarked (65 536 envs, two kernels): same-step auto-resets and reveals turning MrX's column on and off;
    the whole state, the mask and the one-hot against the C oracle after every step."""
    env, ob = _pair(200, 400, 6, 20, 65536, 7, toll=1, belief=True, reveal=5, writer="lsu")
    env.reset()
    _compare(env, ob, None, True, "reset")
    resets = reveals = 0
    hidden = int((env.mrx_revealed < 0).sum())
    for s in range(14):
        want = _oracle_step(env, ob, s, "plain")
        _compare(env, ob, want, True, ("step", s))
        resets += int(want["terminated"].sum() + want["truncated"].sum())
        now_hidden = int((env.mrx_revealed < 0).sum())
        reveals += int(now_hidden < hidden)
        hidden = now_hidden
    assert resets > 1000 and reveals >= 2
    env.close()


@pytest.mark.parametrize("seq", ["deferred", "options"])
def test_ragged_pool_path_switches_match_oracle(torch_cuda, seq):
    """4 099 envs (a ragged last tile) on a 5-graph pool.  "deferred": sy_step_deferred followed by a plain step, and
    deferred -> flush -> plain, twice over.  "options": step_kernel / writer_path / lagged_kernel switched between steps."""
    env, ob = _pair(200, 400, 6, 20, 4099, 3, toll=1, belief=True, reveal=3, graphs=5, writer="lsu")
    env.reset()
    _compare(env, ob, None, True, "reset")
    if seq == "deferred":
        plan = ["plain", "deferred", "plain", "plain", "deferred", "flush", "plain", "deferred", "deferred", "plain",
                "plain", "deferred", "flush", "plain", "plain"]
    else:
        plan = [dict(step_kernel="two_kernels"), dict(step_kernel="fused"), dict(step_kernel="two_kernels"),
                dict(writer_path="bulk"), dict(writer_path="lsu"), dict(lagged_kernel="on"), dict(lagged_kernel="off"),
                dict(step_kernel="auto"), dict(step_kernel="two_kernels"), dict(nf_fill="on"), dict(nf_fill="off"), {}]
    s = 0
    for what in plan:
        if what == "flush":
            env.flush_observations()
            _compare(env, ob, None, True, ("flush", s))
            continue
        how = what if isinstance(what, str) else "plain"
        if isinstance(what, dict):
            for k, v in what.items():
                env.set_option(k, v)
        want = _oracle_step(env, ob, s, how)
        _compare(env, ob, want, how != "deferred", (what, s), dense=how != "deferred")  # (belief_map is pending too)
        if how != "deferred":
            _check(env, (what, s))
        s += 1
    env.close()


def _env(B=4099, P=6, N=200, E=400, **kw):
    pool = _pkg().generate_graph_pool(kw.pop("graphs", 1), N, E, seed=0)
    env = _pkg().BatchedScotlandYardEnv(B, P, kw.pop("money", 20), graphs=pool, seed=kw.pop("seed", 5), tolls=1,
                                        belief=True, reveal_interval=kw.pop("reveal", 3), **kw)
    env.set_option("step_kernel", "two_kernels")  # the path with the incremental write at every batch size
    return env


def test_freeze_then_partial_reset(torch_cuda):
    """auto_reset=False: finished envs freeze (their one-hot stays; the 6-step horizon ends every episode within the
    first 9 steps), then a partial reset of every other env, and steps in which only the reset envs move."""
    torch = __import__("torch")
    env = _env(auto_reset=False, max_timestep=6, money=8)
    env.reset()
    _check(env, "reset")
    for s in range(9):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("step", s))
    frozen = env.done_flags[:, 0].clone()
    assert bool(frozen.all())
    mask = torch.arange(env.num_envs, device=frozen.device) % 2 == 0
    t_frozen = env.timestep.clone()
    env.reset(reset_mask=mask)
    _check(env, "partial reset")
    for s in range(9, 13):  # fewer steps than the horizon: the reset envs are mid-episode
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("step", s))
    assert torch.equal(env.timestep[~mask], t_frozen[~mask])  # the frozen half stayed put
    assert bool((env.timestep[mask] != t_frozen[mask]).any())
    env.close()


def test_groups_with_absent_agents(torch_cuda):
    """mechanism groups with fewer police: absent agents (pos -1) have blank columns on every step"""
    env = _env(graphs=3)
    env.set_mechanisms([{"number_of_agents": 2}, {}, {"number_of_agents": 4, "max_timestep": 7}])
    env.reset()
    _check(env, "reset")
    assert bool((env.pos < 0).any())
    for s in range(12):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("step", s))
    env.close()


def test_load_state_dict_rewind(torch_cuda):
    """load_state_dict restores the buffer with the state: rewinding to an earlier dict and stepping on reproduces the
    observations of the first pass exactly"""
    torch = __import__("torch")
    env = _env()
    env.reset()
    for s in range(4):
        env.step(env.sample_actions(step_counter=s))
    sd = env.state_dict()
    first = []
    for s in range(4, 10):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("first", s))
        first.append((env.node_features.clone(), env.action_mask.clone()))
    env.load_state_dict(sd)
    _check(env, "rewound")
    for i, s in enumerate(range(4, 10)):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("again", s))
        assert torch.equal(env.node_features, first[i][0]) and torch.equal(env.action_mask, first[i][1]), s
    env.close()


def test_second_buffer_through_c_abi(torch_cuda):
    """a step through the C ABI into a second, freshly allocated node_features buffer writes it whole; the next step
    into the env's own buffer (which still holds an older state's one-hot) writes that one whole too"""
    torch = __import__("torch")
    from student_mechanism_design_b200 import _cabi

    env = _env()
    env.reset()
    for s in range(3):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("step", s))
    other = torch.full_like(env.node_features, 0.5)
    obs2 = _cabi.SyObs(env.action_mask.data_ptr(), other.data_ptr(), env.agent_budget.data_ptr(),
                       env.mrx_revealed.data_ptr(), None)
    for s in range(3, 6):
        acts = env.sample_actions(step_counter=s)
        with torch.cuda.device(env.device):
            _cabi.check(env._lib.sy_step(env._handle, acts.data_ptr(), C.byref(env._state), C.byref(obs2),
                                         C.byref(env._out), env._stream()))
        torch.cuda.synchronize()
        assert torch.equal(other, _onehot(env)), ("second buffer", s)
    for s in range(6, 9):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("own buffer", s))
    env.close()


def test_guard_bands_stay_intact(torch_cuda):
    """guard_bytes > 0: the granule stores of both kernels stay inside the buffer, at c3 size"""
    env = _env(B=65536, guard_bytes=64)
    env.reset()
    env.check_guards()
    for s in range(6):
        env.step(env.sample_actions(step_counter=s))
        _check(env, ("step", s))
        env.check_guards()
    env.close()
