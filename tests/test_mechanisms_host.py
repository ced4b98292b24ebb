"""CPU: the mechanism-group ABI (SyGroup, sy_set_groups, sy_group_stats) agrees across the header, the ctypes binding
and INTEGRATION.md, and env.pack_mechanism turns mechanism dicts into SyGroup rows or refuses them."""
import ctypes as C
import os
import re
import types

import pytest
import torch

from conftest import ROOT


def _header_members(name):
    """member names of `typedef struct <name> { ... } <name>;`, comma declarations expanded"""
    text = open(os.path.join(ROOT, "include", "sy_env.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for stmt in body.split(";"):
        stmt = stmt.strip()
        if not stmt:
            continue
        decl = stmt.split(None, 1)[1]
        names += [re.match(r"\s*(\w+)", d).group(1) for d in decl.split(",")]
    return names


def test_sygroup_header_binding_and_doc_agree():
    from student_mechanism_design_b200 import _cabi

    want = _header_members("SyGroup")
    assert want == ["struct_bytes", "reward_weights", "agent_money", "reveal_interval", "reveal_skip_prob", "reserved0"]
    assert [f[0] for f in _cabi.SyGroup._fields_] == want
    assert C.sizeof(_cabi.SyGroup) == 8 + 8 * _cabi.SY_NUM_REWARD_WEIGHTS + 16
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    stmt = re.search(r"class SyGroup\(C\.Structure\):(.*?)(?=\n\S)", doc, re.S).group(1)
    assert re.findall(r'"(\w+)"', stmt) == want
    header = open(os.path.join(ROOT, "include", "sy_env.h")).read()
    assert re.search(r"#define SY_MAX_GROUPS (\d+)", header).group(1) == str(_cabi.SY_MAX_GROUPS)
    for fn in ("sy_set_groups", "sy_group_stats"):
        assert fn in _cabi.SIGNATURES


def _base(**kw):
    from student_mechanism_design_b200 import DEFAULT_REWARD_WEIGHTS

    d = dict(reward_weights=dict(DEFAULT_REWARD_WEIGHTS), agent_money=10, reveal_interval=5,
             config=types.SimpleNamespace(reveal_skip_prob=0.25))
    d.update(kw)
    return types.SimpleNamespace(**d)


def test_pack_mechanism_fills_missing_keys_from_the_env():
    from student_mechanism_design_b200 import REWARD_WEIGHT_NAMES, _cabi
    from student_mechanism_design_b200.env import pack_mechanism, unpack_mechanism

    base = _base()
    g = pack_mechanism({}, base)
    assert g.struct_bytes == C.sizeof(_cabi.SyGroup)
    m = unpack_mechanism(g)
    assert m["agent_money"] == 10 and m["reveal_interval"] == 5 and m["reveal_skip_prob"] == 0.25
    assert m["reward_weights"] == base.reward_weights
    g = pack_mechanism({"agent_money": 4, "reveal_interval": 0, "reveal_skip_prob": 1.0,
                        "reward_weights": {"Mrx_time": 0.5, "Police_time": torch.tensor(0.1, dtype=torch.float32)}}, base)
    m = unpack_mechanism(g)
    assert (m["agent_money"], m["reveal_interval"], m["reveal_skip_prob"]) == (4, 0, 1.0)
    assert m["reward_weights"]["Mrx_time"] == 0.5
    # a 0-dim float32 tensor enters as its exact float32 value (what the fp32 reward mode computes with)
    assert m["reward_weights"]["Police_time"] == float(torch.tensor(0.1, dtype=torch.float32))
    assert m["reward_weights"]["Police_distance"] == base.reward_weights["Police_distance"]
    assert list(m["reward_weights"]) == REWARD_WEIGHT_NAMES


@pytest.mark.parametrize("mech, exc", [
    ({"agent_money": -1}, ValueError),
    ({"agent_money": 2.5}, ValueError),
    ({"reveal_interval": -3}, ValueError),
    ({"reveal_skip_prob": -0.1}, ValueError),
    ({"reveal_skip_prob": 1.01}, ValueError),
    ({"reward_weights": {"Mrx_time": float("nan")}}, ValueError),
    ({"reward_weights": {"Mrx_time": float("inf")}}, ValueError),
    ({"reward_weights": {"not_a_weight": 1.0}}, KeyError),
    ({"toll": 1}, KeyError),
    ([("agent_money", 3)], TypeError),
])
def test_pack_mechanism_rejects(mech, exc):
    from student_mechanism_design_b200.env import pack_mechanism

    with pytest.raises(exc):
        pack_mechanism(mech, _base())
