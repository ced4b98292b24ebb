"""Batched float64 restatement of one belief step (sy_oracle.belief_update / belief_cross_entropy, i.e.
src/environment/belief_module.py:69-111 in expectation and src/eval/belief_quality.py:8-11), for whole batches.

TEST INFRASTRUCTURE ONLY.  The scalar oracle loops over nodes and neighbours in Python; these functions gather with one
`scipy.sparse` matrix per graph and work graph by graph, so a step of config 4 (32 768 envs x 1000 nodes) fits in host
memory.  tests/test_belief_oracle.py pins them to the scalar oracle and to the C oracle's belief trajectory.

Per-env operations use the kernels' enum (sy_env.cu BEL_*): KEEP leaves the row, UNIFORM writes 1/N, DELTA writes the
one-hot of MrX's node, PROPAGATE spreads every node's mass over its neighbours (an isolated node keeps it), applies the
optional observation hint and normalises (an all-zero row becomes uniform).
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

import sy_oracle as so

KEEP, UNIFORM, DELTA, PROPAGATE = 0, 1, 2, 3


def _graph(g) -> so.Graph:
    return g if isinstance(g, so.Graph) else so.Graph(g.num_nodes, g.edge_links, g.edges)


def propagation_matrix(graph) -> sp.csr_matrix:
    """Gather matrix M [N, N]: M[j, i] = 1/deg(i) for every neighbour i of j, M[j, j] = 1 for an isolated j
    (belief_module.py:91-98).  Neighbours are the distinct ones of the weight matrix (parallel edges collapse)."""
    g = _graph(graph)
    n = g.num_nodes
    rp, col, _ = g.csr()
    deg = np.diff(rp).astype(np.int64)
    rows = np.repeat(np.arange(n), deg)
    vals = 1.0 / deg[col].astype(np.float64)
    iso = np.nonzero(deg == 0)[0]
    rows = np.concatenate([rows, iso])
    cols = np.concatenate([col.astype(np.int64), iso])
    vals = np.concatenate([vals, np.ones(len(iso))])
    return sp.csr_matrix((vals, (rows, cols)), shape=(n, n))


def max_degree(graph) -> int:
    rp = _graph(graph).csr()[0]
    return int(np.diff(rp).max()) if len(rp) > 1 else 0


def hub_graph(n, degrees, isolated=(), seed=0):
    """A GraphSpec-like graph for the belief kernels' edge cases: the nodes that are neither hubs nor `isolated` form a
    ring; hub k (the k-th node outside `isolated`) is joined to `degrees[k]` consecutive ring nodes (a hub of degree 0
    is isolated too).  Ring nodes next to several hubs get larger degrees as well.  Weights cycle through 1..4."""
    from student_mechanism_design_b200.graphs import GraphSpec

    isolated = set(int(i) for i in isolated)
    free = [j for j in range(n) if j not in isolated]
    hubs, ring = free[: len(degrees)], free[len(degrees):]
    links = [(ring[i], ring[(i + 1) % len(ring)]) for i in range(len(ring))]
    rng = np.random.default_rng(seed)
    for h, d in zip(hubs, degrees):
        assert d <= len(ring), "hub degree larger than the ring"
        start = int(rng.integers(len(ring)))
        links += [(h, ring[(start + i) % len(ring)]) for i in range(d)]
    links = np.asarray(links, dtype=np.int32).reshape(-1, 2)
    return GraphSpec(n, links, (np.arange(len(links)) % 4 + 1).astype(np.int64))


def _mats(graphs, mats):
    return mats if mats is not None else [propagation_matrix(g) for g in graphs]


def _propagate(prev, graphs, gid, rows, mats):
    """unnormalised M @ prev[b] for the envs `rows`, graph by graph"""
    out = np.zeros((len(rows), prev.shape[1]), dtype=np.float64)
    gr = np.asarray(gid)[rows]
    for g in np.unique(gr):
        sel = np.nonzero(gr == g)[0]
        out[sel] = (mats[int(g)] @ prev[rows[sel]].T).T
    return out


def _normalise(out):
    s = out.sum(axis=1)
    zero = s == 0
    res = np.empty_like(out)
    res[~zero] = out[~zero] / s[~zero, None]
    res[zero] = 1.0 / out.shape[1]
    return res


def belief_step_batched(prev, graphs, gid, op, x, hint=None, mats=None) -> np.ndarray:
    """One belief step for a batch.  prev float64 [B, N]; gid [B] graph of each env; op [B] (KEEP / UNIFORM / DELTA /
    PROPAGATE); x [B] MrX's node (read for DELTA rows); hint: optional [B, N], non-zero = candidate node, re-weights the
    propagated row by 0.1 + 0.9 * hint before the normalisation (a row without candidates is left as it is, like the
    reference's `if observation_hint:`).  `mats`: the graphs' propagation matrices, when the caller keeps them."""
    prev = np.asarray(prev, dtype=np.float64)
    B, N = prev.shape
    op = np.asarray(op)
    out = prev.copy()
    out[op == UNIFORM] = 1.0 / N
    d = np.nonzero(op == DELTA)[0]
    out[d] = 0.0
    out[d, np.asarray(x)[d]] = 1.0
    rows = np.nonzero(op == PROPAGATE)[0]
    if len(rows):
        a = _propagate(prev, graphs, gid, rows, _mats(graphs, mats))
        if hint is not None:
            h = np.asarray(hint)[rows] != 0
            has = h.any(axis=1)
            a[has] *= np.where(h[has], 1.0, 0.1)
        out[rows] = _normalise(a)
    return out


def belief_ce_batched(prev, graphs, gid, x, mats=None) -> np.ndarray:
    """Cross-entropy of the propagated row (no hint) at MrX's node x, per env [B] (belief_quality.py:8-11: clip to
    [1e-8, 1], renormalise, -log); what the kernels score before a reveal collapses the row."""
    prev = np.asarray(prev, dtype=np.float64)
    rows = np.arange(prev.shape[0])
    p = _normalise(_propagate(prev, graphs, gid, rows, _mats(graphs, mats)))
    c = np.clip(p, 1e-8, 1.0)
    c /= c.sum(axis=1, keepdims=True)
    return -np.log(c[rows, np.asarray(x)])


def op_from_transition(done_before, episode_before, episode_after, revealed_after, reveal_interval, auto_reset,
                       reset_mask=None) -> np.ndarray:
    """Each env's belief operation of one step, from its state before and after it: a frozen env (done, no auto-reset)
    keeps its row; a same-step auto-reset (episode counter moved) or an explicit reset (`reset_mask`) gives UNIFORM; a
    reveal that was scheduled and not skipped (reveal_interval > 0 and MrX revealed afterwards) gives DELTA at MrX's
    node; anything else propagates.  With reveal_interval == 0 MrX is always shown but the belief still propagates.
    `reveal_interval` is a scalar or per env [B] (mechanism groups)."""
    done_before = np.asarray(done_before).astype(bool)
    B = len(done_before)
    op = np.full(B, PROPAGATE, dtype=np.int64)
    ri = np.broadcast_to(np.asarray(reveal_interval), (B,))
    op[(ri > 0) & (np.asarray(revealed_after) >= 0)] = DELTA
    op[np.asarray(episode_after) != np.asarray(episode_before)] = UNIFORM
    if not auto_reset:
        op[done_before] = KEEP
    if reset_mask is not None:
        op[np.asarray(reset_mask).astype(bool)] = UNIFORM
    return op
