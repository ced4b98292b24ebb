"""CPU: per-group police count and horizon (sy_set_group_rules) agree across the header, the ctypes binding and
INTEGRATION.md; the `number_of_agents` / `max_timestep` keys of a mechanism dict are validated (bounds, non-integral
values, bools); set_mechanisms makes the rules call only when some group differs from the handle; the mechanism dicts
carry both keys; and budget efficiency weighs each group by its own P_g x agent_money_g."""
import contextlib
import ctypes as C
import os
import re
import types

import numpy as np
import pytest

from conftest import ROOT


def _header():
    return open(os.path.join(ROOT, "include", "sy_env.h")).read()


def test_set_group_rules_header_binding_and_doc_agree():
    from student_mechanism_design_b200 import _cabi

    text = re.sub(r"/\*.*?\*/", "", _header(), flags=re.S)
    decl = re.search(r"int\s+sy_set_group_rules\s*\(([^)]*)\);", text).group(1)
    params = [" ".join(p.split()) for p in decl.split(",")]
    assert params == ["SyEnv* env", "int32_t num_groups", "const int32_t* num_police", "const int32_t* max_timestep",
                      "sy_stream_t stream"]
    restype, argtypes = _cabi.SIGNATURES["sy_set_group_rules"]
    assert restype is C.c_int
    assert argtypes == [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p]
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    sec3 = doc[doc.index("## 3. Binding the C ABI directly"):doc.index("## 3b.")]
    sec3b = doc[doc.index("## 3b."):doc.index("## 4.")]
    assert "sy_set_group_rules(env, C, num_police, max_timestep, stream)" in sec3
    assert '"number_of_agents"' in sec3b and "max_timestep" in sec3b
    for text in (doc, _header()):
        assert "stay one value per handle" not in text
    # the absent-agent values sit next to SyState.pos
    state = _header()[_header().index("Absent agents"):_header().index("} SyState;")]
    for v in ("pos -1", "money 0", "agent_budget 0.0f", "-1"):
        assert v in state


def _base(**kw):
    from student_mechanism_design_b200 import DEFAULT_REWARD_WEIGHTS

    d = dict(reward_weights=dict(DEFAULT_REWARD_WEIGHTS), agent_money=10, reveal_interval=5, tolls=1, number_of_agents=4,
             config=types.SimpleNamespace(reveal_skip_prob=0.25, max_timestep=100))
    d.update(kw)
    return types.SimpleNamespace(**d)


@pytest.mark.parametrize("mech, want", [({}, (4, 100)), ({"number_of_agents": 1}, (1, 100)),
                                        ({"number_of_agents": 4.0, "max_timestep": 0}, (4, 0)),
                                        ({"number_of_agents": np.int64(2), "max_timestep": np.int32(100)}, (2, 100)),
                                        ({"max_timestep": 37.0}, (4, 37))])
def test_rules_keys_accepted(mech, want):
    from student_mechanism_design_b200 import _cabi
    from student_mechanism_design_b200.env import mechanism_rules, pack_mechanism

    got = mechanism_rules(mech, _base())  # a missing key takes the constructor's value
    assert got == want and all(type(x) is int for x in got)
    assert C.sizeof(pack_mechanism(mech, _base())) == C.sizeof(_cabi.SyGroup)


@pytest.mark.parametrize("key, bad", [("number_of_agents", 0), ("number_of_agents", 5), ("number_of_agents", -1),
                                      ("number_of_agents", 1.5), ("number_of_agents", True), ("number_of_agents", "2"),
                                      ("number_of_agents", float("nan")), ("max_timestep", -1), ("max_timestep", 101),
                                      ("max_timestep", 2 ** 40), ("max_timestep", 10.5), ("max_timestep", False),
                                      ("max_timestep", float("inf")), ("max_timestep", None)])
def test_rules_keys_rejected(key, bad):
    from student_mechanism_design_b200.env import mechanism_rules, pack_mechanism

    with pytest.raises(ValueError, match=key):
        pack_mechanism({key: bad}, _base())
    with pytest.raises(ValueError, match=key):
        mechanism_rules({key: bad}, _base())


def test_mechanism_dicts_carry_the_rules():
    from student_mechanism_design_b200.env import MECHANISM_KEYS, mechanism_rules, pack_mechanism, unpack_mechanism

    assert "number_of_agents" in MECHANISM_KEYS and "max_timestep" in MECHANISM_KEYS
    base = _base()
    mechs = [{}, {"number_of_agents": 2}, {"max_timestep": 7, "agent_money": 3}]
    dicts = [unpack_mechanism(pack_mechanism(m, base), 1, mechanism_rules(m, base)) for m in mechs]
    assert [(d["number_of_agents"], d["max_timestep"]) for d in dicts] == [(4, 100), (2, 100), (4, 7)]
    assert dicts[2]["agent_money"] == 3
    m = unpack_mechanism(pack_mechanism({}, base))
    assert "number_of_agents" not in m and "max_timestep" not in m
    with pytest.raises(KeyError):  # the police count is `number_of_agents`, as in the constructor
        pack_mechanism({"num_police": 2}, base)


class _FakeLib:
    """records the mechanism-group calls of set_mechanisms (and their arguments) instead of launching anything"""

    def __init__(self):
        self.calls = []

    def sy_set_groups(self, handle, n, table, gid, stream):
        self.calls.append(("groups", n))
        return 0

    def sy_set_group_tolls(self, handle, n, tolls, stream):
        self.calls.append(("tolls", n, list(tolls)))
        return 0

    def sy_set_group_rules(self, handle, n, police, horizon, stream):
        self.calls.append(("rules", n, list(police), list(horizon)))
        return 0


def _fake_env(monkeypatch):
    import torch

    from student_mechanism_design_b200.env import BatchedScotlandYardEnv

    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    env = BatchedScotlandYardEnv.__new__(BatchedScotlandYardEnv)
    base = _base()
    env.__dict__.update(base.__dict__)
    env.__dict__.update(num_envs=10, env_offset=0, device=torch.device("cpu"), stats_vec=None, _groups_generation=0,
                        _handle=None, _lib=_FakeLib(), flush_observations=lambda: None, _stream=lambda: 0)
    return env


def test_rules_call_only_when_some_group_differs(monkeypatch):
    env = _fake_env(monkeypatch)
    env.set_mechanisms([{}, {"number_of_agents": 4, "max_timestep": 100.0}])
    assert env._lib.calls == [("groups", 2)] and env._env_police is None
    assert [(m["number_of_agents"], m["max_timestep"]) for m in env.mechanisms] == [(4, 100)] * 2
    env._lib.calls.clear()
    env.set_mechanisms([{}, {"max_timestep": 20}])  # a horizon alone: the call, but no per-env police table
    assert env._lib.calls == [("groups", 2), ("rules", 2, [4, 4], [100, 20])] and env._env_police is None
    env._lib.calls.clear()
    env.set_mechanisms([{"number_of_agents": 1}, {}, {"number_of_agents": 3, "tolls": 2}])
    assert env._lib.calls == [("groups", 3), ("tolls", 3, [1, 1, 2]), ("rules", 3, [1, 4, 3], [100, 100, 100])]
    assert env._env_police.view(-1).tolist() == [1, 4, 3, 1, 4, 3, 1, 4, 3, 1]
    env._lib.calls.clear()
    with pytest.raises(ValueError):  # rejected before any library call
        env.set_mechanisms([{}, {"number_of_agents": 5}])
    assert env._lib.calls == []
    env.set_mechanisms(None)
    assert env._lib.calls == [("groups", 0)] and env._env_police is None and env.mechanisms is None


def _stats_dicts(table):
    from student_mechanism_design_b200 import _cabi

    return [dict(zip(_cabi.STAT_NAMES, (int(x) for x in row))) for row in table]


def test_budget_efficiency_per_group_and_aggregate():
    from student_mechanism_design_b200 import _cabi
    from student_mechanism_design_b200.env import group_metrics, metrics_of

    rng = np.random.default_rng(5)
    C_ = 5
    table = rng.integers(0, 10 ** 6, size=(C_, _cabi.SY_NUM_STATS), dtype=np.int64)
    table[3] = 0  # a group without episodes
    i = _cabi.STAT_NAMES.index
    table[:, i("episodes")] = [17, 4, 250, 0, 1]
    table[:, i("mrx_wins")] = table[:, i("episodes")] // 2
    table[:, i("police_wins")] = table[:, i("episodes")] - table[:, i("mrx_wins")]
    per = _stats_dicts(table)
    total = _stats_dicts(table.sum(0, keepdims=True))[0]
    police, money = [1, 2, 3, 4, 2], [10, 7, 20, 5, 0]
    mechs = [dict(agent_money=m, tolls=1, number_of_agents=p) for p, m in zip(police, money)]
    eff, paid, by_group = group_metrics(per, mechs, number_of_agents=4)
    for g, st in enumerate(per):
        budget = max(police[g] * money[g], 1)
        want = st["sum_episode_budget_spent"] / st["episodes"] / budget if st["episodes"] else 0.0
        assert by_group[g]["mean_budget_efficiency"] == want, g
    assert eff == sum(st["sum_episode_budget_spent"] / max(p * m, 1) for st, p, m in zip(per, police, money))
    agg = metrics_of(total, initial=40, tolls_paid=paid, eff_sum=eff)
    assert agg["mean_budget_efficiency"] == eff / total["episodes"]
    # dicts without the key (older callers) take `number_of_agents`, as before
    eff4, _, _ = group_metrics(per, [dict(agent_money=m, tolls=1) for m in money], number_of_agents=4)
    assert eff4 == sum(st["sum_episode_budget_spent"] / max(4 * m, 1) for st, m in zip(per, money))
