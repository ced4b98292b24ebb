"""CPU: per-group tolls (sy_set_group_tolls) agree across the header, the ctypes binding and INTEGRATION.md; the `tolls` key
of a mechanism dict is validated like the constructor's argument; the mechanism dicts carry it; and mean_tolls_paid is
computed per group and in aggregate from the per-group statistics."""
import ctypes as C
import os
import re
import types

import numpy as np
import pytest

from conftest import ROOT


def _header():
    return open(os.path.join(ROOT, "include", "sy_env.h")).read()


def test_set_group_tolls_header_binding_and_doc_agree():
    from student_mechanism_design_b200 import _cabi

    text = re.sub(r"/\*.*?\*/", "", _header(), flags=re.S)
    decl = re.search(r"int\s+sy_set_group_tolls\s*\(([^)]*)\);", text).group(1)
    params = [p.strip() for p in decl.split(",")]
    assert params == ["SyEnv* env", "int32_t num_groups", "const int32_t* tolls", "sy_stream_t stream"]
    restype, argtypes = _cabi.SIGNATURES["sy_set_group_tolls"]
    assert restype is C.c_int
    assert argtypes == [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p]
    assert re.search(r"#define SY_MAX_TOLL (\d+)", _header()).group(1) == str(_cabi.SY_MAX_TOLL)
    # w + toll (w <= 255) and a warp's sum of up to 32 x 15 police charges stay inside an int32
    assert 32 * 15 * (255 + _cabi.SY_MAX_TOLL) < 2 ** 31
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    sec3 = doc[doc.index("## 3. Binding the C ABI directly"):doc.index("## 3b.")]
    sec3b = doc[doc.index("## 3b."):doc.index("## 4.")]
    assert "sy_set_group_tolls(env, C, tolls, stream)" in sec3
    assert '"tolls"' in sec3b
    for text in (doc, _header()):
        assert "toll, the number of police" not in text and "Everything else stays one value per handle" not in text


def _base(**kw):
    from student_mechanism_design_b200 import DEFAULT_REWARD_WEIGHTS

    d = dict(reward_weights=dict(DEFAULT_REWARD_WEIGHTS), agent_money=10, reveal_interval=5, tolls=1,
             config=types.SimpleNamespace(reveal_skip_prob=0.25))
    d.update(kw)
    return types.SimpleNamespace(**d)


@pytest.mark.parametrize("toll, want", [(0, 0), (3, 3), (1.0, 1), (np.int64(2), 2), (None, 1)])
def test_tolls_key_accepted(toll, want):
    from student_mechanism_design_b200 import _cabi
    from student_mechanism_design_b200.env import mechanism_toll, pack_mechanism

    mech = {} if toll is None else {"tolls": toll}
    assert mechanism_toll(mech, _base()) == want  # a missing key takes the constructor's tolls
    assert C.sizeof(pack_mechanism(mech, _base())) == C.sizeof(_cabi.SyGroup)
    assert mechanism_toll({"tolls": _cabi.SY_MAX_TOLL}, _base()) == _cabi.SY_MAX_TOLL


def test_tolls_key_rejected():
    from student_mechanism_design_b200 import _cabi
    from student_mechanism_design_b200.env import mechanism_toll, pack_mechanism

    for bad in (-1, 1.5, _cabi.SY_MAX_TOLL + 1, 2 ** 40, float("nan"), float("inf"), "1", True):
        with pytest.raises(ValueError):
            pack_mechanism({"tolls": bad}, _base())
        with pytest.raises(ValueError):
            mechanism_toll({"tolls": bad}, _base())
    with pytest.raises(KeyError):  # the constructor's argument is `tolls`; `toll` stays an unknown key
        pack_mechanism({"toll": 1}, _base())


def test_pack_mechanism_without_tolls_on_the_base():
    from student_mechanism_design_b200.env import pack_mechanism

    base = _base()
    del base.tolls
    pack_mechanism({}, base)  # the toll travels separately: a base without `tolls` still packs
    pack_mechanism({"tolls": 2}, base)


def test_mechanism_dicts_carry_tolls():
    from student_mechanism_design_b200.env import MECHANISM_KEYS, mechanism_toll, pack_mechanism, unpack_mechanism

    assert "tolls" in MECHANISM_KEYS and "toll" not in MECHANISM_KEYS
    base = _base()
    mechs = [{}, {"tolls": 0}, {"tolls": 3.0, "agent_money": 4}]
    dicts = [unpack_mechanism(pack_mechanism(m, base), mechanism_toll(m, base)) for m in mechs]
    assert [d["tolls"] for d in dicts] == [1, 0, 3]
    assert all(type(d["tolls"]) is int for d in dicts)
    assert dicts[2]["agent_money"] == 4
    assert "tolls" not in unpack_mechanism(pack_mechanism({}, base))


def _stats_dicts(table):
    from student_mechanism_design_b200 import _cabi

    return [dict(zip(_cabi.STAT_NAMES, (int(x) for x in row))) for row in table]


def test_mean_tolls_paid_per_group_and_aggregate():
    from student_mechanism_design_b200 import _cabi
    from student_mechanism_design_b200.env import group_metrics, metrics_of

    rng = np.random.default_rng(7)
    C_ = 5
    table = rng.integers(0, 10 ** 6, size=(C_, _cabi.SY_NUM_STATS), dtype=np.int64)
    table[3] = 0  # a group without episodes
    i = _cabi.STAT_NAMES.index
    table[:, i("episodes")] = [17, 4, 250, 0, 1]
    table[:, i("police_moves")] = [1000, 33, 99999, 0, 7]
    table[:, i("mrx_wins")] = table[:, i("episodes")] // 2
    table[:, i("police_wins")] = table[:, i("episodes")] - table[:, i("mrx_wins")]
    per = _stats_dicts(table)
    total = _stats_dicts(table.sum(0, keepdims=True))[0]
    tolls = [0, 1, 2, 3, _cabi.SY_MAX_TOLL]
    mechs = [dict(agent_money=10 + g, tolls=t) for g, t in enumerate(tolls)]
    eff, paid, by_group = group_metrics(per, mechs, number_of_agents=4)
    assert paid == sum(t * int(g["police_moves"]) for t, g in zip(tolls, per))
    for g, (st, t) in enumerate(zip(per, tolls)):
        want = t * st["police_moves"] / st["episodes"] if st["episodes"] else 0.0
        assert by_group[g]["mean_tolls_paid"] == want
        assert by_group[g]["num_episodes"] == st["episodes"]
    agg = metrics_of(total, initial=40, tolls_paid=paid, eff_sum=eff)
    assert agg["mean_tolls_paid"] == paid / total["episodes"]
    # groups that all pay the constructor's toll give exactly the float of a handle without groups
    eff1, paid1, _ = group_metrics(per, [dict(agent_money=10, tolls=3)] * C_, number_of_agents=4)
    assert metrics_of(total, initial=40, tolls_paid=paid1, eff_sum=eff1)["mean_tolls_paid"] == \
        3 * total["police_moves"] / total["episodes"]
