"""CPU oracle of the heuristic opponents (`sy_heuristic_actions`, include/sy_env.h): an evading MrX and chasing police.

TEST INFRASTRUCTURE ONLY, like sy_oracle.py (whose Philox, graph tables and random-valid draw it reuses).

**parity unpinned**: the counterpart of the reference's src/eval/exploitability.py:122,188, whose source is not
available; the rules restated here are this project's own, as the header states them.
"""
from __future__ import annotations

from typing import List

import numpy as np

from sy_oracle import DEFAULT_ACTION, Graph, _M32, philox4x32, philox_random_valid_action

RNG_HEURISTIC = 4  # Philox purpose of the exploration draws (0..3 and 16..20 are taken)
HEUR_NONE, HEUR_RANDOM, HEUR_EVADE, HEUR_CHASE, HEUR_CHASE_BELIEF = 0, 1, 2, 3, 4


def heuristic_threshold(epsilon) -> int:
    """floor(epsilon * 2^32): an agent explores when its Philox word is below this (0 never, 2^32 always)"""
    return int(float(epsilon) * 2 ** 32)


def heuristic_actions(seed, env_ids, step, pos, money, timestep, revealed, graph_id, graphs: List[Graph], tolls, num_police,
                      mrx_kind, police_kind, explore_mrx=0, explore_police=0, last_seen=None, belief=None, actions=None):
    """The actions of sy_heuristic_actions for the rows given: env_ids [R] global env indices (env_offset + b), pos /
    money [R, A] (absent agents past num_police[r]: pos -1), timestep / revealed (mrx_revealed) / graph_id / tolls /
    num_police [R], last_seen [R] or None, belief [R, N] (CHASE_BELIEF), actions [R, A] whose HEUR_NONE columns are
    kept (None: -1).  Returns (actions int64 [R, A], the new last_seen int32 [R] or None)."""
    pos = np.asarray(pos, dtype=np.int64)
    money = np.asarray(money, dtype=np.int64)
    R, A = pos.shape
    key = (seed & _M32, (seed >> 32) & _M32)
    acts = np.full((R, A), DEFAULT_ACTION, dtype=np.int64) if actions is None else np.array(actions, dtype=np.int64)
    rev = np.asarray(revealed, dtype=np.int64)
    t = np.asarray(timestep, dtype=np.int64)
    # MrX's last revealed node: this step's reveal, else the memory (cleared when an episode starts, t == 0)
    ls = rev.copy()
    hidden = rev < 0
    if last_seen is None:
        ls[hidden] = -1
    else:
        ls[hidden] = np.where(t[hidden] == 0, -1, np.asarray(last_seen, dtype=np.int64)[hidden])
    target = ls.copy()
    if police_kind == HEUR_CHASE_BELIEF:
        target[hidden] = np.argmax(np.asarray(belief)[hidden], axis=1)  # first maximum
    W = np.stack([g.weight_matrix() for g in graphs])
    D = np.stack([g.apsp() for g in graphs])
    gid = np.asarray(graph_id, dtype=np.int64)
    toll = np.asarray(tolls, dtype=np.int64)
    npol = np.asarray(num_police, dtype=np.int64)
    N = W.shape[1]
    rows = np.arange(R)
    present = np.arange(A)[None, :] <= npol[:, None]  # [R, A]
    occ = np.zeros((R, N), dtype=bool)  # nodes of present police
    for i in range(1, A):
        live = present[:, i]
        occ[rows[live], pos[live, i]] = True
    for a in range(A):
        kind = mrx_kind if a == 0 else police_kind
        if kind == HEUR_NONE:
            continue
        thr = explore_mrx if a == 0 else explore_police
        live = present[:, a]
        acts[~live, a] = DEFAULT_ACTION
        u = np.where(live, pos[:, a], 0)
        wrow = W[gid, u]  # [R, N]
        afford = (wrow > 0) & (wrow + toll[:, None] <= money[:, a, None])
        free = afford & ~occ
        if a == 0:  # evade: score(c) = min over present police of D[c][pos_i]; ties: stay, then the lowest id
            score = np.full((R, N), np.iinfo(np.int64).max)
            for i in range(1, A):
                col = D[gid, :, np.where(present[:, i], pos[:, i], 0)]  # [R, N]: D[c][pos_i]
                score = np.where(present[:, i, None], np.minimum(score, col), score)
            own = score[rows, u]
            cand = np.where(free, score, -1)
            best = np.argmax(cand, axis=1)  # lowest id among equal scores
            choice = np.where(cand[rows, best] > own, best, u)
        else:  # chase: the free affordable neighbour with the smallest D[j][target]; boxed in: own node; broke: -1
            dj = D[gid, :, np.maximum(target, 0)]  # [R, N]
            cand = np.where(free, dj, np.iinfo(np.int64).max)
            best = np.argmin(cand, axis=1)
            choice = np.where(free.any(axis=1), best, np.where(afford.any(axis=1), u, DEFAULT_ACTION))
        rnd = np.full(R, kind == HEUR_RANDOM) | ((a > 0) & (target < 0))
        if thr:  # exploration draw of the agents that would play the heuristic
            for r in np.nonzero(live & ~rnd)[0]:
                rnd[r] = philox4x32((int(env_ids[r]), step, RNG_HEURISTIC, a), key)[0] < thr
        acts[live & ~rnd, a] = choice[live & ~rnd]
        for r in np.nonzero(live & rnd)[0]:
            acts[r, a] = philox_random_valid_action(seed, int(env_ids[r]), step, a, np.nonzero(afford[r])[0])
    return acts, None if last_seen is None else ls.astype(np.int32)


def batch_heuristic_actions(ob, step, mrx_kind, police_kind, explore_mrx=0, explore_police=0, last_seen=None,
                            belief=None, actions=None):
    """heuristic_actions on the state of an sy_oracle.OracleBatch or OracleGroupBatch `ob` (every env's own toll and
    police count), so that whole oracle rollouts can be driven by it; belief None = the batch's own belief maps.
    Returns (actions [B, A], new last_seen or None)."""
    B = len(ob.envs)
    if belief is None and police_kind == HEUR_CHASE_BELIEF:
        belief = ob.belief()
    return heuristic_actions(ob.seed, ob.env_offset + np.arange(B), step, ob.pos(), ob.money(), ob.timestep(),
                             ob.revealed(), ob.graph_id, ob.graphs, [e.cfg.toll for e in ob.envs],
                             [e.cfg.num_police for e in ob.envs], mrx_kind, police_kind, explore_mrx, explore_police,
                             last_seen, belief, actions)
