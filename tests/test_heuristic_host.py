"""CPU: the heuristic opponents (sy_heuristic_actions) -- known answers of the oracle on hand-built graphs (evade
tie-breaks, chase towards a visible / last seen target, boxed-in and broke chasers, tolls, absent agents, NONE sides,
the belief argmax), the random and exploring kinds equal the random-valid sampler, and the header, the ctypes binding
and the host threshold agree."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT

import heuristic_oracle as ho
import sy_oracle as so

RAND, EVADE, CHASE, CHASE_B, NONE = ho.HEUR_RANDOM, ho.HEUR_EVADE, ho.HEUR_CHASE, ho.HEUR_CHASE_BELIEF, ho.HEUR_NONE


def _graph(n, edges):
    return so.Graph(n, [(u, v) for u, v, _ in edges], [w for _, _, w in edges])


PATH5 = _graph(5, [(0, 1, 1), (1, 2, 1), (2, 3, 1), (3, 4, 1)])
STAR = _graph(5, [(0, 1, 1), (0, 2, 1), (0, 3, 1), (0, 4, 1)])
CYCLE5 = _graph(5, [(0, 1, 1), (1, 2, 1), (2, 3, 1), (3, 4, 1), (4, 0, 1)])
CYCLE4_W = _graph(4, [(0, 1, 3), (1, 2, 1), (2, 3, 1), (3, 0, 1)])  # unequal weights


def _one(graph, pos, mrx_kind=EVADE, police_kind=CHASE, money=None, t=3, rev=None, toll=0, num_police=None,
         last_seen=None, belief=None, actions=None, seed=7, step=11):
    """heuristic_actions of a single env; rev None = MrX visible"""
    A = len(pos)
    money = [1000] + [50] * (A - 1) if money is None else money
    rev = pos[0] if rev is None else rev
    P = A - 1 if num_police is None else num_police
    acts, ls = ho.heuristic_actions(seed, [3], step, [pos], [money], [t], [rev], [0], [graph], [toll], [P], mrx_kind,
                                    police_kind, last_seen=None if last_seen is None else [last_seen],
                                    belief=None if belief is None else [belief],
                                    actions=None if actions is None else [actions])
    return acts[0].tolist(), None if ls is None else int(ls[0])


def test_evade_moves_away_from_the_nearest_police():
    assert _one(PATH5, [2, 0], police_kind=NONE)[0][0] == 3


def test_evade_ties_prefer_staying():
    # 5-cycle, police at 0: MrX at 2 scores 2, neighbour 3 scores 2 as well, neighbour 1 scores 1
    assert _one(CYCLE5, [2, 0], police_kind=NONE)[0][0] == 2


def test_evade_ties_between_neighbours_go_to_the_lowest_id():
    # star: MrX at the centre, police on leaf 1; leaves 2, 3, 4 all score 2
    assert _one(STAR, [0, 1], police_kind=NONE)[0][0] == 2


def test_evade_never_steps_onto_police_and_respects_budget():
    # MrX at 1 on the path, police at 0 and 3: neighbour 2 scores 1 = own score -> stay; with money 0 MrX can only stay
    assert _one(PATH5, [1, 0, 3], police_kind=NONE)[0][0] == 1
    assert _one(PATH5, [2, 0], police_kind=NONE, money=[0, 50])[0][0] == 2


def test_chase_towards_a_visible_target():
    acts, _ = _one(PATH5, [4, 0], mrx_kind=NONE)
    assert acts[1] == 1


def test_chase_uses_last_seen_while_hidden_and_forgets_it_at_t0():
    # hidden MrX, last seen at 4: the police heads there, last_seen kept
    acts, ls = _one(PATH5, [1, 2], mrx_kind=NONE, rev=-1, t=3, last_seen=4)
    assert acts[1] == 3 and ls == 4
    # a reveal updates the memory
    acts, ls = _one(PATH5, [1, 2], mrx_kind=NONE, rev=1, t=5, last_seen=4)
    assert acts[1] == 1 and ls == 1
    # t == 0 (a new episode): the memory is cleared; with no target the police takes the random draw
    acts, ls = _one(PATH5, [1, 2], mrx_kind=NONE, rev=-1, t=0, last_seen=4, seed=7, step=11)
    assert ls == -1
    assert acts[1] == so.philox_random_valid_action(7, 3, 11, 1, np.array([1, 3]))
    # no buffer: a hidden MrX is never remembered
    acts, ls = _one(PATH5, [1, 2], mrx_kind=NONE, rev=-1, t=3, last_seen=None)
    assert ls is None and acts[1] == so.philox_random_valid_action(7, 3, 11, 1, np.array([1, 3]))


def test_boxed_in_chaser_stays_but_a_broke_one_gets_minus_one():
    g = _graph(4, [(1, 0, 1), (0, 2, 1), (2, 3, 1)])  # path 1 - 0 - 2 - 3
    acts, _ = _one(g, [3, 0, 1, 2], mrx_kind=NONE)
    assert acts[1:] == [0, 1, 3]  # both neighbours of 0 occupied: own node; 1: own node; 2 -> MrX's node 3
    acts, _ = _one(g, [3, 0, 1, 2], mrx_kind=NONE, money=[1000, 0, 50, 50])
    assert acts[1] == -1


def test_tolls_make_the_nearest_neighbour_unaffordable():
    # police at 0 chases MrX at 1: the direct edge (weight 3) wins without toll; with toll 1 and budget 3 it costs 4
    acts, _ = _one(CYCLE4_W, [1, 0], mrx_kind=NONE, money=[1000, 3], toll=0)
    assert acts[1] == 1
    acts, _ = _one(CYCLE4_W, [1, 0], mrx_kind=NONE, money=[1000, 3], toll=1)
    assert acts[1] == 3


def test_absent_agents_and_none_sides():
    # num_police 1 in a 3-agent layout: agent 2 is absent (-1 whatever the buffer held)
    acts, _ = _one(PATH5, [4, 0, -1], money=[1000, 50, 0], num_police=1, actions=[77, 77, 77])
    assert acts == [4, 1, -1]
    acts, _ = _one(PATH5, [4, 0, -1], mrx_kind=NONE, money=[1000, 50, 0], num_police=1, actions=[77, 77, 77])
    assert acts == [77, 1, -1]
    acts, _ = _one(PATH5, [4, 0, -1], police_kind=NONE, money=[1000, 50, 0], num_police=1, actions=[77, 77, 77])
    assert acts == [4, 77, 77]


def test_belief_argmax_ties_go_to_the_lowest_node():
    belief = np.array([0.1, 0.3, 0.1, 0.3, 0.2], dtype=np.float32)
    acts, ls = _one(PATH5, [0, 4], mrx_kind=NONE, police_kind=CHASE_B, rev=-1, last_seen=0, belief=belief)
    assert acts[1] == 3 and ls == 0  # target 1 (first of the two maxima): from 4 the way is 3
    # a visible MrX overrides the belief
    acts, _ = _one(PATH5, [4, 2], mrx_kind=NONE, police_kind=CHASE_B, belief=belief)
    assert acts[1] == 3


def _batch(P=3, B=96, steps=6, toll=1):
    pool = so.philox_graph_pool(5, 3, 20, 40)
    cfg = so.OracleConfig(num_police=P, agent_money=12, reveal_interval=3, toll=toll)
    ob = so.OracleBatch.from_seed(cfg, pool, B, seed=5, env_offset=100)
    for s in range(steps):
        ob.step(ob.sample_actions(s))
    return ob


def test_random_and_full_exploration_equal_the_sampler():
    ob = _batch()
    for step in (6, 7):
        want = ob.sample_actions(step)
        got, _ = ho.batch_heuristic_actions(ob, step, RAND, RAND)
        np.testing.assert_array_equal(got, want)
        got, _ = ho.batch_heuristic_actions(ob, step, EVADE, CHASE, explore_mrx=2 ** 32, explore_police=2 ** 32)
        np.testing.assert_array_equal(got, want)
        # no exploration: the heuristics differ from the sampler somewhere
        got, _ = ho.batch_heuristic_actions(ob, step, EVADE, CHASE, last_seen=np.full(96, -1))
        assert (got != want).any()


def test_group_batch_random_kind_equals_the_sampler():
    pool = so.philox_graph_pool(5, 3, 20, 40)
    cfgs = [so.OracleConfig(num_police=p, agent_money=12, reveal_interval=3, toll=t) for p, t in ((3, 0), (2, 1), (1, 2))]
    gid = [b % 3 for b in range(64)]
    ob = so.OracleGroupBatch.from_seed(cfgs, gid, 3, pool, 64, seed=9)
    for s in range(4):
        ob.step(ob.sample_actions(s))
    got, _ = ho.batch_heuristic_actions(ob, 4, RAND, RAND)
    np.testing.assert_array_equal(got, ob.sample_actions(4))
    got, _ = ho.batch_heuristic_actions(ob, 4, EVADE, CHASE)
    pos = ob.pos()
    assert (got[pos < 0] == -1).all()  # absent agents


def test_partial_exploration_mixes_both():
    ob = _batch()
    thr = ho.heuristic_threshold(0.5)
    rnd = ob.sample_actions(6)
    det, _ = ho.batch_heuristic_actions(ob, 6, EVADE, CHASE, last_seen=ob.revealed())
    got, _ = ho.batch_heuristic_actions(ob, 6, EVADE, CHASE, explore_mrx=thr, explore_police=thr, last_seen=ob.revealed())
    key = (5, 0)
    for b in range(96):
        for a in range(4):
            explore = so.philox4x32((100 + b, 6, ho.RNG_HEURISTIC, a), key)[0] < thr
            assert got[b, a] == (rnd[b, a] if explore else det[b, a])


def _header_struct_fields(name):
    text = open(os.path.join(ROOT, "include", "sy_env.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.search(r"(\w+)(\[[^\]]*\])?\s*$", stmt.strip()).group(1) for stmt in body.split(";") if stmt.strip()]


def test_binding_matches_the_header():
    from student_mechanism_design_b200 import _cabi

    assert [f[0] for f in _cabi.SyHeuristic._fields_] == _header_struct_fields("SyHeuristic")
    assert C.sizeof(_cabi.SyHeuristic) == 40
    text = open(os.path.join(ROOT, "include", "sy_env.h")).read()
    enum = re.search(r"enum \{ (SY_HEUR_NONE[^}]*)\}", text).group(1)
    consts = dict(re.findall(r"(SY_HEUR_\w+) = (\d+)", enum))
    for k, v in consts.items():
        assert getattr(_cabi, k) == int(v)
        assert getattr(ho, k[3:]) == int(v)
    restype, argtypes = _cabi.SIGNATURES["sy_heuristic_actions"]
    assert restype is C.c_int and argtypes[1] == C.POINTER(_cabi.SyHeuristic) and argtypes[4] is C.c_uint32


@pytest.mark.parametrize("eps, want", [(0.0, 0), (2.0 ** -32, 1), (0.5, 2 ** 31), (1.0, 2 ** 32)])
def test_threshold_is_exact(eps, want):
    from student_mechanism_design_b200 import HeuristicPolicy

    assert HeuristicPolicy.explore_threshold(eps) == int(eps * 2 ** 32) == want == ho.heuristic_threshold(eps)


@pytest.mark.parametrize("eps", [float("nan"), -1e-9, 1.0 + 1e-9, True, "0.5", None])
def test_threshold_refuses_bad_epsilon(eps):
    from student_mechanism_design_b200 import HeuristicPolicy

    with pytest.raises(ValueError):
        HeuristicPolicy.explore_threshold(eps)
