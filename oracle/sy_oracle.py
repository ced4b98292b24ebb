"""CPU oracle for the Scotland Yard hot path (numpy / pure Python).

TEST INFRASTRUCTURE ONLY -- this file is the *checker*, never the product.  Only
`tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of
`bench.py` may import it.  The product (`student_mechanism_design_b200`) never does and
fails loudly when its CUDA library is missing.

Parity status
-------------
* PINNED against the unmodified reference implementation (imported through
  `oracle/ref_loader.py` in the build container) for: graph sampling, reset state, step
  dynamics, budgets, action masks, capture / timeout / out-of-money endings, shaped rewards
  in both arithmetic modes, visit counts.  Evidence: `tests/golden/*.npz` written by
  `oracle/gen_golden.py` from the reference, replayed by `tests/test_oracle_golden.py`.
* PINNED against the reference's own known-answer tests for `compute_action_mask`
  (test/test_action_mask.py:9-124).
* **parity unpinned** (the reference env has no implementation, see SURVEY.md section 8(c)):
  `belief_map` (defined here as the exact expectation of `ParticleBeliefTracker`,
  src/environment/belief_module.py:41-111), the reveal schedule
  (src/eval/run_ablations.py:225-229) and tolls inside `step`
  (src/environment/action_mask.py:71-75 pins only the mask rule).  With these switched off
  the oracle is the reference, bit for bit.

Every function cites the reference lines it restates (paths relative to /root/reference).
"""
from __future__ import annotations

import heapq
import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

# src/reward_net.py:5-17 -- order of the 11 reward weights everywhere in this repo.
REWARD_WEIGHT_NAMES = [
    "Police_distance",
    "Police_group",
    "Police_position",
    "Police_time",
    "Mrx_closest",
    "Mrx_average",
    "Mrx_position",
    "Mrx_time",
    "Police_coverage",
    "Police_proximity",
    "Police_overlap_penalty",
]
# src/training/evaluator.py:59-71 -- the evaluation-path defaults (python floats -> fp64 mode)
DEFAULT_REWARD_WEIGHTS = {
    "Police_distance": 0.1,
    "Police_group": 0.1,
    "Police_position": 0.1,
    "Police_time": 0.0,
    "Mrx_closest": 0.3,
    "Mrx_average": 0.2,
    "Mrx_position": 0.1,
    "Mrx_time": 0.0,
    "Police_coverage": 0.05,
    "Police_proximity": 0.05,
    "Police_overlap_penalty": 0.0,
}
MAX_MONEY_LIMIT = 1000  # src/environment/yard.py:11
MAX_TIMESTEP = 250  # src/environment/reward_calculator.py:68
DEFAULT_ACTION = -1  # src/environment/yard.py:16
INF_U16 = 0xFFFF

WINNER_NONE, WINNER_MRX, WINNER_POLICE = 0, 1, 2


# --------------------------------------------------------------------------------------
# Graphs
# --------------------------------------------------------------------------------------
@dataclass
class Graph:
    """edge list exactly as the reference's GraphInstance holds it
    (graph_layout.py:53: nodes int64[N], edges int64[E], edge_links int32[E,2])."""

    num_nodes: int
    edge_links: np.ndarray  # int32 [E, 2]
    edges: np.ndarray  # int64 [E] weights

    def __post_init__(self):
        self.edge_links = np.asarray(self.edge_links, dtype=np.int32).reshape(-1, 2)
        self.edges = np.asarray(self.edges, dtype=np.int64).reshape(-1)
        self._W = None
        self._D = None
        self._csr = None

    # yard.py:404-418 (weight matrix) + yard.py:420-472 (min weight per neighbour)
    def weight_matrix(self) -> np.ndarray:
        """W[u, v] = weight of the (cheapest) undirected edge u-v, 0 if none."""
        if self._W is None:
            N = self.num_nodes
            W = np.zeros((N, N), dtype=np.int64)
            for (u, v), w in zip(self.edge_links.tolist(), self.edges.tolist()):
                for a, b in ((u, v), (v, u)):
                    if W[a, b] == 0 or w < W[a, b]:
                        W[a, b] = w
            self._W = W
        return self._W

    def csr(self):
        """(row_ptr int32[N+1], col int32[nnz], w int32[nnz]); neighbours ascending per row."""
        if self._csr is None:
            W = self.weight_matrix()
            N = self.num_nodes
            row_ptr = np.zeros(N + 1, dtype=np.int32)
            cols, ws = [], []
            for u in range(N):
                nz = np.nonzero(W[u])[0]
                cols.extend(nz.tolist())
                ws.extend(W[u, nz].tolist())
                row_ptr[u + 1] = len(cols)
            self._csr = (row_ptr, np.asarray(cols, dtype=np.int32), np.asarray(ws, dtype=np.int32))
        return self._csr

    # pathfinding.py:34-137 -- heap Dijkstra; the reference recomputes it per query, the
    # result equals this all-pairs table (unreachable -> inf there, INF_U16 here).
    def apsp(self) -> np.ndarray:
        if self._D is None:
            N = self.num_nodes
            row_ptr, col, w = self.csr()
            D = np.full((N, N), INF_U16, dtype=np.int64)
            for s in range(N):
                dist = {s: 0}
                done = set()
                pq = [(0, s)]
                while pq:
                    d, u = heapq.heappop(pq)
                    if u in done:
                        continue
                    done.add(u)
                    D[s, u] = d
                    for k in range(row_ptr[u], row_ptr[u + 1]):
                        v = int(col[k])
                        nd = d + int(w[k])
                        if v not in done and (v not in dist or nd < dist[v]):
                            dist[v] = nd
                            heapq.heappush(pq, (nd, v))
            self._D = D
        return self._D

    def adjacency(self) -> np.ndarray:
        """yard.py:390-402 -- float64 0/1 matrix."""
        return (self.weight_matrix() > 0).astype(np.float64)


def sample_connected_graph(num_nodes, num_edges, py_random, np_random, max_edges_per_node=4) -> Graph:
    """Draw-for-draw restatement of ConnectedGraph.sample (graph_layout.py:9-53) and
    _create_tree (graph_layout.py:55-80).

    `py_random` must offer `choice`/`shuffle` (the `random` module or a `random.Random`),
    `np_random` must offer `randint` (the `numpy.random` module or a `RandomState`); the
    reference consumes both *global* streams.  Python `set` iteration order matters for the
    draw sequence, so real sets are used, as in the reference.
    """
    # -- random-Prim tree (graph_layout.py:55-80)
    tree = []
    visited = set()
    unvisited = set(range(num_nodes))
    start = py_random.choice(list(unvisited))
    visited.add(start)
    unvisited.remove(start)
    while unvisited:
        candidates = [(a, b) for a in visited for b in unvisited]
        pick = py_random.choice(candidates)
        tree.append(pick)
        visited.add(pick[1])
        unvisited.remove(pick[1])
    links = list(tree)
    weights = [np_random.randint(1, 5) for _ in links]  # MAX_WEIGHT = 5 -> {1,2,3,4}
    if num_edges is None:
        num_edges = num_nodes - 1
    extra = num_edges - len(links)
    if extra > 0:
        tree_set = set(tree)
        cand = [
            (i, j)
            for i in range(num_nodes)
            for j in range(i + 1, num_nodes)
            if (i, j) not in tree_set and (j, i) not in tree_set
        ]
        py_random.shuffle(cand)
        degree = [0] * num_nodes
        for a, b in links:
            degree[a] += 1
            degree[b] += 1
        for a, b in cand:
            if extra <= 0:
                break
            if degree[a] < max_edges_per_node and degree[b] < max_edges_per_node:
                links.append((a, b))
                weights.append(np_random.randint(1, 5))
                degree[a] += 1
                degree[b] += 1
                extra -= 1
    return Graph(num_nodes, np.asarray(links, dtype=np.int32), np.asarray(weights, dtype=np.int64))


def reference_construct(seed, num_nodes, num_edges, num_agents):
    """Graph + start nodes the reference env holds after `random.seed(s); np.random.seed(s);
    CustomEnvironment(...)`: one probe sample fixes the edge count (yard.py:67-70), reset()
    resamples until the count matches (yard.py:89-101), then np.random.choice draws the A
    distinct start nodes (yard.py:112-116).  Returns (Graph, [mrx, police...])."""
    import random as _random

    py, npr = _random.Random(seed), np.random.RandomState(seed)
    probe = sample_connected_graph(num_nodes, num_edges, py, npr)
    want = probe.edge_links.shape[0]
    for attempt in range(100):
        g = sample_connected_graph(num_nodes, num_edges, py, npr)
        if g.edge_links.shape[0] == want:
            break
    else:
        raise RuntimeError(f"Failed to generate graph with {want} edges after 100 attempts.")
    start = npr.choice(num_nodes, size=num_agents, replace=False)
    return g, [int(x) for x in start]


# --------------------------------------------------------------------------------------
# Action mask (src/environment/action_mask.py:30-113)
# --------------------------------------------------------------------------------------
def action_mask_dense(adjacency, current_node, budget, tolls=None, edge_weights=None) -> np.ndarray:
    """mask[j] = j != cur and adj[cur, j] != 0 and w[cur, j] + toll[cur, j] <= budget, float64.
    tolls: None | scalar | per-destination vector | matrix (action_mask.py:86-96);
    edge_weights None -> adjacency as unit costs (action_mask.py:99-113)."""
    adjacency = np.asarray(adjacency)
    n = adjacency.shape[0]
    if tolls is None:
        toll_row = np.zeros(n)
    elif np.isscalar(tolls):
        toll_row = np.full(n, float(tolls))
    else:
        t = np.asarray(tolls, dtype=float)
        toll_row = t if t.ndim == 1 else t[current_node]
    w_row = (
        adjacency[current_node].astype(float)
        if edge_weights is None
        else np.asarray(edge_weights, dtype=float)[current_node]
    )
    mask = (adjacency[current_node] != 0) & ((w_row + toll_row) <= budget)
    mask[current_node] = False
    return mask


# --------------------------------------------------------------------------------------
# Belief (exact expectation of ParticleBeliefTracker, belief_module.py:21-111) -- parity unpinned
# --------------------------------------------------------------------------------------
def belief_uniform(n) -> np.ndarray:
    """belief_module.py:53-54,60 -- uniformly random particles => uniform expectation."""
    return np.full(n, 1.0 / n, dtype=np.float64)


def belief_update(belief, graph: Graph, reveal: Optional[int] = None, hint: Optional[Sequence[int]] = None):
    """belief_module.py:69-111 in expectation.  reveal -> delta (:86-88); else every node's mass
    is split uniformly over its neighbours, an isolated node keeps it (:91-98); optional hint
    re-weighting 0.1 + 0.9*[j in hint] (:102-106); normalise, all-zero -> uniform (:27-38)."""
    n = graph.num_nodes
    if reveal is not None:
        out = np.zeros(n, dtype=np.float64)
        out[int(reveal)] = 1.0
        return out
    row_ptr, col, _ = graph.csr()
    out = np.zeros(n, dtype=np.float64)
    for j in range(n):  # gather form (adjacency is symmetric): b'[j] = sum_{i in nbr(j)} b[i]/deg(i)
        acc = 0.0
        for k in range(row_ptr[j], row_ptr[j + 1]):
            i = int(col[k])
            acc += belief[i] / float(row_ptr[i + 1] - row_ptr[i])
        if row_ptr[j + 1] == row_ptr[j]:
            acc = belief[j]
        out[j] = acc
    if hint:
        like = np.full(n, 0.1)
        like[list(hint)] = 1.0
        out = out * like
    s = out.sum()
    if s == 0:
        return belief_uniform(n)
    return out / s


def belief_cross_entropy(belief, true_index) -> float:
    """src/eval/belief_quality.py:8-11: clip to [1e-8, 1], renormalise, -log at the true node."""
    b = np.clip(np.asarray(belief, dtype=np.float64), 1e-8, 1.0)
    b = b / b.sum()
    return float(-np.log(b[int(true_index)]))


def is_reveal(t, interval) -> bool:
    """src/eval/run_ablations.py:225-229."""
    return bool(interval and interval > 0 and t > 0 and t % interval == 0)


# --------------------------------------------------------------------------------------
# Philox4x32-10 (counter-based RNG shared, bit for bit, with the CUDA kernels)
# --------------------------------------------------------------------------------------
_PHILOX_M0, _PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
_PHILOX_W0, _PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
_M32 = 0xFFFFFFFF

RNG_RESET_POS, RNG_RESET_GRAPH, RNG_ACTION, RNG_REVEAL_SKIP = 0, 1, 2, 3


def philox4x32(ctr, key):
    c0, c1, c2, c3 = [int(x) & _M32 for x in ctr]
    k0, k1 = [int(x) & _M32 for x in key]
    for _ in range(10):
        p0 = _PHILOX_M0 * c0
        p1 = _PHILOX_M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & _M32, p1 & _M32, ((p0 >> 32) ^ c3 ^ k1) & _M32, p0 & _M32
        k0 = (k0 + _PHILOX_W0) & _M32
        k1 = (k1 + _PHILOX_W1) & _M32
    return c0, c1, c2, c3


def _rng_words(seed, env, episode_or_step, purpose, n):
    """n 32-bit words of the stream (seed; env, episode_or_step, purpose, block)."""
    key = (seed & _M32, (seed >> 32) & _M32)
    out = []
    blk = 0
    while len(out) < n:
        out.extend(philox4x32((env, episode_or_step, purpose, blk), key))
        blk += 1
    return out[:n]


def philox_start_positions(seed, env, episode, n_nodes, n_agents) -> List[int]:
    """A distinct uniform nodes: draw r_a in [0, N-a) and map it to the r_a-th unused node
    (same distribution as np.random.choice(N, A, replace=False), yard.py:112-116)."""
    words = _rng_words(seed, env, episode, RNG_RESET_POS, n_agents)
    chosen_sorted: List[int] = []
    out = []
    for a in range(n_agents):
        x = (words[a] * (n_nodes - a)) >> 32
        for c in chosen_sorted:
            if x >= c:
                x += 1
        out.append(x)
        chosen_sorted.append(x)
        chosen_sorted.sort()
    return out


def philox_graph_choice(seed, env, episode, n_graphs) -> int:
    return (_rng_words(seed, env, episode, RNG_RESET_GRAPH, 1)[0] * n_graphs) >> 32


# --------------------------------------------------------------------------------------
# Counter-based graph sampler (SURVEY 8(f) row f3): the SAME DISTRIBUTION as sample_connected_graph above
# (= ConnectedGraph.sample, graph_layout.py:9-80) from Philox streams keyed by (seed; graph index, generation /
# attempt), in a form a GPU warp can run per graph.  Why the distribution is the same:
#   * `_create_tree` (graph_layout.py:55-80) starts at a uniform node and always joins a uniform (visited, unvisited)
#     pair = a uniform unvisited node to a uniform visited node: a uniformly random insertion order whose k-th node
#     attaches to a uniform earlier one.
#   * the extra edges are a first-fit scan over a uniform shuffle of all non-tree pairs under the degree cap
#     (graph_layout.py:24-48).  A node only ever goes from "open" (degree < cap) to "closed", so a pair that was
#     scanned and skipped stays unacceptable for good, and a pair whose two ends are still open cannot have been
#     scanned without being accepted.  Hence the next accepted edge is uniform over the non-adjacent pairs of the
#     currently open nodes, and the scan ends early exactly when no such pair is left.  That is what is sampled here
#     (rejection over ordered pairs of open nodes, with the number V of acceptable pairs tracked exactly).
#   * weights are iid U{1..max_weight-1} (np.random.randint(1, MAX_WEIGHT), graph_layout.py:17,47).
# --------------------------------------------------------------------------------------
RNG_GEN_PERM, RNG_GEN_PARENT, RNG_GEN_TREE_W, RNG_GEN_PAIR, RNG_GEN_EXTRA_W = 16, 17, 18, 19, 20
GEN_MAX_ATTEMPTS = 100  # yard.py:89-101
GEN_MAX_DRAWS = 1 << 22


class _GenStream:
    """k-th 32-bit word of the stream (seed; graph, generation * 128 + attempt, purpose, k >> 2)."""

    def __init__(self, seed, graph, generation, attempt, purpose):
        self.key = (seed & _M32, (seed >> 32) & _M32)
        self.c0, self.c1, self.c2 = graph & _M32, (generation * 128 + attempt) & _M32, purpose
        self.blk, self.words = -1, None

    def word(self, k):
        if (k >> 2) != self.blk:
            self.blk = k >> 2
            self.words = philox4x32((self.c0, self.c1, self.c2, self.blk), self.key)
        return self.words[k & 3]


def philox_sample_graph_once(seed, graph, generation, attempt, num_nodes, num_edges, max_edges_per_node=4,
                             max_weight=5) -> Graph:
    N, cap, wr = int(num_nodes), int(max_edges_per_node), int(max_weight) - 1
    perm_s, par_s, tw_s, pair_s, xw_s = [_GenStream(seed, graph, generation, attempt, pu) for pu in
                                         (RNG_GEN_PERM, RNG_GEN_PARENT, RNG_GEN_TREE_W, RNG_GEN_PAIR, RNG_GEN_EXTRA_W)]
    order = list(range(N))
    for k in range(N - 1):  # Fisher-Yates
        j = k + ((perm_s.word(k) * (N - k)) >> 32)
        order[k], order[j] = order[j], order[k]
    adj = np.zeros((N, N), dtype=bool)
    deg = [0] * N
    links, weights = [], []
    for k in range(1, N):
        u, v = order[(par_s.word(k) * k) >> 32], order[k]
        links.append((u, v))
        weights.append(1 + ((tw_s.word(k) * wr) >> 32))
        adj[u, v] = adj[v, u] = True
        deg[u] += 1
        deg[v] += 1
    extra = (N - 1 if num_edges is None else int(num_edges)) - (N - 1)
    open_nodes = [u for u in range(N) if deg[u] < cap]  # ascending
    pos = {u: i for i, u in enumerate(open_nodes)}
    n_open = len(open_nodes)
    V = n_open * (n_open - 1) // 2 - sum(1 for u, v in links if deg[u] < cap and deg[v] < cap)
    draw = n_extra = 0
    while extra > 0 and V > 0:
        if draw >= GEN_MAX_DRAWS:
            raise RuntimeError("graph sampler: draw budget exhausted")
        a = (pair_s.word(draw) * n_open) >> 32
        b = (pair_s.word(draw + 1) * (n_open - 1)) >> 32
        draw += 2
        if b >= a:
            b += 1
        i, j = open_nodes[a], open_nodes[b]
        if adj[i, j]:
            continue
        links.append((i, j))
        weights.append(1 + ((xw_s.word(n_extra) * wr) >> 32))
        adj[i, j] = adj[j, i] = True
        deg[i] += 1
        deg[j] += 1
        V -= 1
        extra -= 1
        n_extra += 1
        for x in (i, j):
            if deg[x] >= cap:  # x closes: swap-with-last removal, its still-acceptable pairs disappear
                last = open_nodes[n_open - 1]
                open_nodes[pos[x]] = last
                pos[last] = pos[x]
                n_open -= 1
                open_nodes.pop()
                del pos[x]
                V -= sum(1 for k in open_nodes if not adj[x, k])
    return Graph(N, np.asarray(links, dtype=np.int32).reshape(-1, 2), np.asarray(weights, dtype=np.int64))


def philox_sample_graph(seed, graph, generation, num_nodes, num_edges, want_edges=0, max_edges_per_node=4, max_weight=5):
    """One pool slot: resample (attempt 0, 1, ...) until the edge count equals `want_edges` (0 = take the first), as
    CustomEnvironment.reset does against the count frozen at construction (yard.py:87-101).  Returns (Graph, attempt)."""
    for attempt in range(GEN_MAX_ATTEMPTS):
        g = philox_sample_graph_once(seed, graph, generation, attempt, num_nodes, num_edges, max_edges_per_node, max_weight)
        if want_edges <= 0 or len(g.edges) == want_edges:
            return g, attempt
    raise RuntimeError(f"Failed to generate graph with {want_edges} edges after {GEN_MAX_ATTEMPTS} attempts.")


def philox_graph_pool(seed, num_graphs, num_nodes, num_edges, generation=0, graph_offset=0, max_edges_per_node=4,
                      max_weight=5):
    """Slot `graph_offset` + 0 of generation `generation` fixes the edge count (the constructor's probe sample,
    yard.py:67-76); every other slot is resampled until it matches."""
    first, _ = philox_sample_graph(seed, 0, generation, num_nodes, num_edges, 0, max_edges_per_node, max_weight)
    want = len(first.edges)
    pool = []
    for g in range(num_graphs):
        gg = graph_offset + g
        pool.append(first if gg == 0 else philox_sample_graph(seed, gg, generation, num_nodes, num_edges, want,
                                                              max_edges_per_node, max_weight)[0])
    return pool


# --------------------------------------------------------------------------------------
# The environment
# --------------------------------------------------------------------------------------
@dataclass
class OracleConfig:
    num_police: int
    agent_money: int
    reward_weights: dict = field(default_factory=lambda: dict(DEFAULT_REWARD_WEIGHTS))
    reward_mode: str = "fp64"  # "fp64": python-float weights; "fp32": 0-dim fp32 torch weights
    max_timestep: int = MAX_TIMESTEP
    mrx_money: int = MAX_MONEY_LIMIT
    reveal_interval: int = 0  # 0 -> reference behaviour (MrX always visible)
    toll: int = 0  # 0 -> reference behaviour
    belief: bool = False
    # robustness hook of src/eval/ood_eval.py:227-229 (RobustnessWrapper): probability that a scheduled reveal is skipped
    reveal_skip_prob: float = 0.0
    # optional recorded float64 tables (tests/golden/tables.npz); None -> NumPy on this host
    exp_table: Optional[np.ndarray] = None
    cov_table: Optional[np.ndarray] = None


class OracleEnv:
    """One episode stream.  State and rule follow yard.py; see SURVEY.md Appendix B."""

    def __init__(self, cfg: OracleConfig, graph: Graph, start_positions: Sequence[int]):
        self.cfg = cfg
        self.P = cfg.num_police
        self.A = cfg.num_police + 1
        self.w64 = [float(cfg.reward_weights[k]) for k in REWARD_WEIGHT_NAMES]
        self.w32 = [np.float32(x) for x in self.w64]
        self.reset(graph, start_positions)

    # yard.py:80-142
    def reset(self, graph: Graph, start_positions: Sequence[int]):
        self.graph = graph
        self.N = graph.num_nodes
        self.W = graph.weight_matrix()
        self.D = graph.apsp()
        self.pos = [int(p) for p in start_positions]  # [MrX, Police0..]
        assert len(self.pos) == self.A
        self.money = [self.cfg.mrx_money] + [self.cfg.agent_money] * self.P  # yard.py:117-119
        self.t = 0
        self.visits = np.zeros(self.N, dtype=np.int64)  # node_visit_counts, yard.py:85
        self.winner = WINNER_NONE
        self.moves = getattr(self, "moves", 0)  # police moves over the env's lifetime (not reset)
        self.belief = belief_uniform(self.N) if self.cfg.belief else None
        self.revealed = -1 if self.cfg.reveal_interval > 0 else self.pos[0]

    # yard.py:420-472 with the toll extension (toll == 0 -> the reference rule)
    def legal(self, p, j, money) -> bool:
        if j < 0 or j >= self.N:
            return False
        w = int(self.W[p, j])
        return w > 0 and w + self.cfg.toll <= money

    def n_moves(self, p, money) -> int:
        row = self.W[p]
        return int(np.count_nonzero((row > 0) & (row + self.cfg.toll <= money)))

    def possible_moves(self, agent_idx) -> np.ndarray:
        """yard.py:474-480 -- sorted neighbour ids the agent can afford."""
        p, m = self.pos[agent_idx], self.money[agent_idx]
        row = self.W[p]
        return np.nonzero((row > 0) & (row + self.cfg.toll <= m))[0].astype(np.int32)

    # yard.py:144-269
    def step(self, actions: Sequence[Optional[int]], hint: Optional[Sequence[int]] = None, skip_reveal=None):
        """`hint`: candidate nodes of belief_module.py:102-106 for this step's belief update; `skip_reveal(t)`: the
        batch's Philox draw that decides whether the reveal scheduled at timestep t is skipped (ood_eval.py:227-229)"""
        P, A = self.P, self.A
        pos, money = self.pos, self.money
        # MrX (yard.py:155-188); None and any non-legal value both end in "stay"
        a0 = actions[0]
        if a0 is not None:
            tgt = int(a0) if self.legal(pos[0], int(a0), money[0]) else pos[0]
            if tgt not in pos[1:]:
                pos[0] = tgt
        # police, sequential (yard.py:190-243)
        no_money = True
        for i in range(1, A):
            act = actions[i]
            if act is None or int(money[i]) == 0 or int(act) == DEFAULT_ACTION:
                continue
            no_money = False
            act = int(act)
            tgt = act if self.legal(pos[i], act, money[i]) else pos[i]
            if tgt not in pos[1:] and tgt != pos[i]:
                money[i] -= int(self.W[pos[i], tgt]) + self.cfg.toll
                pos[i] = tgt
                self.moves += 1
        for i in range(1, A):  # yard.py:244-245
            self.visits[pos[i]] += 1
        rewards, terminated, truncated, winner = self._rewards_terminations(no_money)
        self.t += 1  # yard.py:355
        self.winner = winner
        # extensions (parity unpinned): reveal schedule + belief propagation on the new timestep
        rev = is_reveal(self.t, self.cfg.reveal_interval)
        if rev and skip_reveal is not None and skip_reveal(self.t):
            rev = False
        if self.cfg.reveal_interval > 0:
            self.revealed = pos[0] if rev else -1
        else:
            self.revealed = pos[0]
        self.last_ce = None
        if self.cfg.belief:
            if rev:  # score the prediction before the reveal collapses it (metrics.py:142-147)
                self.last_ce = belief_cross_entropy(belief_update(self.belief, self.graph), pos[0])
            self.belief = belief_update(self.belief, self.graph, reveal=pos[0] if rev else None, hint=None if rev else hint)
        return rewards, terminated, truncated, winner

    # reward_calculator.py:26-92
    def _rewards_terminations(self, no_money):
        mode32 = self.cfg.reward_mode == "fp32"
        if self.pos[0] in self.pos[1:]:
            r = [-1.0] + [1.0] * self.P
            return self._cast(r), True, False, WINNER_POLICE
        if self.t > self.cfg.max_timestep:
            r = [1.0] + [0.0] * self.P
            return self._cast(r), False, True, WINNER_MRX
        if no_money:
            r = [1.0] + [0.0] * self.P
            return self._cast(r), True, False, WINNER_MRX
        r = self._shaped_rewards_fp32() if mode32 else self._shaped_rewards_fp64()
        return r, False, False, WINNER_NONE

    def _cast(self, r):
        return [np.float32(x) for x in r] if self.cfg.reward_mode == "fp32" else [float(x) for x in r]

    def _dist(self, a, b) -> float:
        d = int(self.D[a, b])
        return math.inf if d >= INF_U16 else float(d)

    def _exp_neg(self, d: float):
        """np.exp(-d) (reward_calculator.py:186,199,214), optionally from the recorded table."""
        if self.cfg.exp_table is None or math.isinf(d):
            return np.exp(-d)
        return np.float64(self.cfg.exp_table[int(d)]) if int(d) < len(self.cfg.exp_table) else np.float64(0.0)

    def _coverage(self, c: int):
        """np.exp(-np.log1p(c)) (reward_calculator.py:204-205)."""
        if self.cfg.cov_table is None:
            return np.exp(-np.log1p(c))
        return np.float64(self.cfg.cov_table[min(c, len(self.cfg.cov_table) - 1)])

    def _terms(self):
        """The float64 quantities reward_calculator.py:126-205 computes before weighting."""
        P = self.P
        pos, t = self.pos, self.t
        d = [self._dist(pos[0], pos[1 + i]) for i in range(P)]
        closest = min(d)
        avg = float(np.mean(d))
        mrx = (
            -1 / (closest + 1),
            -1 / (avg + 1),
            self.n_moves(pos[0], self.money[0]),
            0.1 * t,
        )
        police = []
        for k in range(P):
            p = pos[1 + k]
            dx = self._exp_neg(self._dist(p, pos[0]))
            grp = 0
            ov = 0
            prox = 0
            for j in range(P):
                if j == k:
                    continue
                dj = self._dist(p, pos[1 + j])
                e = self._exp_neg(dj)
                grp = grp + e
                if dj <= 1:
                    ov = ov + 1.0
                else:
                    prox = prox + e
            mob = self.n_moves(p, self.money[k])  # QUIRK reward_calculator.py:190: agent index k, not k+1
            cov = self._coverage(int(self.visits[p]))
            police.append((dx, grp, mob, 0.05 * t, prox, ov, cov))
        return mrx, police

    # reward_calculator.py:139-147, 212-227 with python-float weights
    def _shaped_rewards_fp64(self):
        w = dict(zip(REWARD_WEIGHT_NAMES, self.w64))
        mrx, police = self._terms()
        out = [
            w["Mrx_closest"] * mrx[0]
            + w["Mrx_average"] * mrx[1]
            + w["Mrx_position"] * mrx[2]
            + (1 - w["Mrx_time"]) * mrx[3]
        ]
        for dx, grp, mob, tt, prox, ov, cov in police:
            out.append(
                w["Police_distance"] * dx
                + w["Police_group"] * grp
                + w["Police_position"] * mob
                + (1 - w["Police_time"]) * tt
                + w["Police_proximity"] * prox
                - w["Police_overlap_penalty"] * ov
                + w["Police_coverage"] * cov
            )
        return [float(x) for x in out]

    # same expressions when the weights are 0-dim fp32 torch tensors (gnn_trainer.py:98-110):
    # every scalar operand is rounded to fp32 first, every op rounds once, no FMA.
    def _shaped_rewards_fp32(self):
        f = np.float32
        w = dict(zip(REWARD_WEIGHT_NAMES, self.w32))
        one = f(1)
        mrx, police = self._terms()
        out = [
            w["Mrx_closest"] * f(mrx[0])
            + w["Mrx_average"] * f(mrx[1])
            + w["Mrx_position"] * f(mrx[2])
            + (one - w["Mrx_time"]) * f(mrx[3])
        ]
        for dx, grp, mob, tt, prox, ov, cov in police:
            out.append(
                w["Police_distance"] * f(dx)
                + w["Police_group"] * f(grp)
                + w["Police_position"] * f(mob)
                + (one - w["Police_time"]) * f(tt)
                + w["Police_proximity"] * f(prox)
                - w["Police_overlap_penalty"] * f(ov)
                + w["Police_coverage"] * f(cov)
            )
        return [f(x) for x in out]

    # yard.py:271-335 + action_mask.py:54-83
    def action_masks(self) -> np.ndarray:
        m = np.zeros((self.A, self.N), dtype=bool)
        for a in range(self.A):
            row = self.W[self.pos[a]]
            m[a] = (row > 0) & (row + self.cfg.toll <= self.money[a])
        return m

    def node_features(self) -> np.ndarray:
        """yard.py:279-290 (one-hot positions; column 0 = MrX, blank while hidden)."""
        nf = np.zeros((self.N, self.A), dtype=np.float32)
        if self.revealed >= 0:
            nf[self.pos[0], 0] = 1
        for i in range(1, self.A):
            nf[self.pos[i], i] = 1
        return nf


# --------------------------------------------------------------------------------------
# Random valid policy shared with the CUDA sampler (`sy_sample_actions`)
# --------------------------------------------------------------------------------------
def philox_random_valid_action(seed, env, step, agent, moves: np.ndarray) -> int:
    """uniform pick among the agent's affordable neighbours (ascending node order); -1 if none
    (mirrors the trainers: no valid move -> DEFAULT_ACTION, gnn_trainer.py:227-229)."""
    if len(moves) == 0:
        return DEFAULT_ACTION
    r = philox4x32((env, step, RNG_ACTION, agent), (seed & _M32, (seed >> 32) & _M32))[0]
    return int(moves[(r * len(moves)) >> 32])


SY_NUM_STATS = 16  # include/sy_env.h: the statistics vector of sy_stats / sy_group_stats
(STAT_ENV_STEPS, STAT_EPISODES, STAT_MRX_WINS, STAT_POLICE_WINS, STAT_TRUNCATIONS, STAT_OUT_OF_MONEY, STAT_SUM_LENGTH,
 STAT_SUM_BUDGET_SPENT, STAT_SUM_SQ_LENGTH, STAT_SUM_LENGTH_POLICE_WINS, STAT_SUM_LENGTH_MRX_WINS,
 STAT_SUM_EPISODE_BUDGET_SPENT, STAT_POLICE_MOVES, STAT_REVEALS) = range(14)


class OracleBatch:
    """B independent OracleEnv with the batched env's conventions: graph pool + graph_id,
    same-step auto-reset keyed by Philox(seed; global env index, episode)."""

    def __init__(self, cfg: OracleConfig, graphs: List[Graph], graph_id, start_positions, seed=0,
                 auto_reset=False, env_offset=0, resample_graph=False, groups=None):
        """groups: (cfgs, group_id) of an OracleGroupBatch; None = every env runs `cfg`"""
        self.cfg, self.graphs, self.seed = cfg, graphs, int(seed)
        self.auto_reset, self.env_offset, self.resample_graph = auto_reset, env_offset, resample_graph
        self.graph_id = [int(g) for g in graph_id]
        self.cfgs, self.group = (list(groups[0]), [int(g) for g in groups[1]]) if groups else ([cfg], [0] * len(self.graph_id))
        self.A = cfg.num_police + 1
        self.envs = [OracleEnv(self.cfgs[gr], graphs[g], list(sp)[: self.cfgs[gr].num_police + 1])
                     for g, gr, sp in zip(self.graph_id, self.group, start_positions)]
        self.episode = [0] * len(self.envs)
        self.done = [False] * len(self.envs)
        # (length, winner, budget spent, truncated, group) of every finished episode
        self.finished = []
        self.belief_ces = []  # cross-entropies at reveal steps (not scored when the same step auto-resets the env)
        self.ce_groups = []  # the group of each entry of belief_ces
        self.step_stats = [[0, 0, 0] for _ in self.cfgs]  # per group: env steps, budget spent, police moves

    @classmethod
    def from_seed(cls, cfg, graphs, num_envs, seed=0, env_offset=0, auto_reset=True, resample_graph=False):
        gid, sp = cls._seeded_starts(cfg.num_police + 1, graphs, num_envs, seed, env_offset, resample_graph)
        return cls(cfg, graphs, gid, sp, seed, auto_reset, env_offset, resample_graph)

    @staticmethod
    def _seeded_starts(A, graphs, num_envs, seed, env_offset, resample_graph):
        N = graphs[0].num_nodes
        gid, sp = [], []
        for b in range(num_envs):
            e = env_offset + b
            g = philox_graph_choice(seed, e, 0, len(graphs)) if resample_graph else (e // 32) % len(graphs)  # blocks of 32 envs
            gid.append(g)
            sp.append(philox_start_positions(seed, e, 0, N, A))
        return gid, sp

    def _skip_draw(self, b):
        """the device's draw: skip iff Philox(seed; global env, t, RNG_REVEAL_SKIP, episode)[0] < float32(p) * 2^32"""
        p = float(np.float32(self.envs[b].cfg.reveal_skip_prob))
        if p <= 0.0:
            return None
        thresh = int(min(p, 1.0) * 4294967296.0)
        key = (self.seed & _M32, (self.seed >> 32) & _M32)
        return lambda t: philox4x32((self.env_offset + b, t, RNG_REVEAL_SKIP, self.episode[b]), key)[0] < thresh

    def step(self, actions, hints=None):
        """actions int [B, A] (-1 == None); hints: optional bool/uint8 [B, N] observation hints (belief_module.py:
        102-106).  Returns dict of arrays for this step, then applies the same-step auto-reset (observations afterwards
        describe the fresh episode)."""
        B, A = len(self.envs), self.A
        f = np.float32 if self.cfg.reward_mode == "fp32" else np.float64
        out = dict(
            reward=np.zeros((B, A), dtype=f),
            terminated=np.zeros(B, dtype=bool),
            truncated=np.zeros(B, dtype=bool),
            winner=np.zeros(B, dtype=np.int8),
        )
        for b, env in enumerate(self.envs):
            if self.done[b]:  # frozen until reset (no auto-reset): zero reward, flags stay
                continue
            hint = None if hints is None else [int(j) for j in np.nonzero(np.asarray(hints[b]))[0]]
            money0, moves0 = sum(env.money[1:]), env.moves
            r, te, tr, win = env.step([int(x) for x in actions[b][: env.A]], hint=hint, skip_reveal=self._skip_draw(b))
            out["reward"][b, : env.A] = r
            out["terminated"][b], out["truncated"][b], out["winner"][b] = te, tr, win
            gs = self.step_stats[self.group[b]]
            gs[0] += 1
            gs[1] += money0 - sum(env.money[1:])
            gs[2] += env.moves - moves0
            if env.last_ce is not None and not ((te or tr) and self.auto_reset):
                self.belief_ces.append(env.last_ce)
                self.ce_groups.append(self.group[b])
            if te or tr:
                # (episode length, winner, budget spent) of the finished episode: what metrics.py:EpisodeMetrics records
                spent = env.cfg.num_police * env.cfg.agent_money - sum(env.money[1:])
                self.finished.append((env.t, int(win), spent, int(tr), self.group[b]))
                if self.auto_reset:
                    self.episode[b] += 1
                    e = self.env_offset + b
                    if self.resample_graph:
                        self.graph_id[b] = philox_graph_choice(self.seed, e, self.episode[b], len(self.graphs))
                    sp = philox_start_positions(self.seed, e, self.episode[b], env.N, env.A)
                    env.reset(self.graphs[self.graph_id[b]], sp)
                else:
                    self.done[b] = True
        return out

    def expected_stats(self):
        """(total, per_group): the statistics vectors of sy_stats and sy_group_stats (include/sy_env.h SY_STAT_*) as
        Python ints, from the finished episodes and the per-step counts.  Entries 0..12 are exact; entry 13 counts the
        scored reveals (what the device counts with belief scoring on); 14 and 15, the device's float32 cross-entropy
        sums, are left None (compare them with a tolerance against belief_ces)."""
        per = [[0] * SY_NUM_STATS for _ in self.cfgs]
        for g, (n, spent, moves) in enumerate(self.step_stats):
            per[g][STAT_ENV_STEPS], per[g][STAT_SUM_BUDGET_SPENT], per[g][STAT_POLICE_MOVES] = n, spent, moves
        for length, win, spent, trunc, g in self.finished:
            v = per[g]
            v[STAT_EPISODES] += 1
            v[STAT_SUM_LENGTH] += length
            v[STAT_SUM_SQ_LENGTH] += length * length
            v[STAT_SUM_EPISODE_BUDGET_SPENT] += spent
            if win == WINNER_POLICE:
                v[STAT_POLICE_WINS] += 1
                v[STAT_SUM_LENGTH_POLICE_WINS] += length
            else:
                v[STAT_MRX_WINS] += 1
                v[STAT_SUM_LENGTH_MRX_WINS] += length
                v[STAT_TRUNCATIONS if trunc else STAT_OUT_OF_MONEY] += 1
        for g in self.ce_groups:
            per[g][STAT_REVEALS] += 1
        for v in per:
            v[14] = v[15] = None
        total = [sum(v[k] for v in per) for k in range(14)] + [None, None]
        return total, per

    def sample_actions(self, step) -> np.ndarray:
        B, A = len(self.envs), self.A
        acts = np.full((B, A), DEFAULT_ACTION, dtype=np.int64)
        for b, env in enumerate(self.envs):
            for a in range(env.A):
                acts[b, a] = philox_random_valid_action(self.seed, self.env_offset + b, step, a, env.possible_moves(a))
        return acts

    # state views shaped like the device arrays (the agents past an env's police count carry the absent values of
    # include/sy_env.h: pos -1, money 0, all-zero mask rows and node_features columns)
    def _padded(self, rows, fill, dtype):
        out = np.full((len(self.envs), self.A) + np.shape(rows[0])[1:], fill, dtype=dtype)
        for b, r in enumerate(rows):
            out[b, : len(r)] = r
        return out

    def pos(self):
        return self._padded([e.pos for e in self.envs], -1, np.int32)

    def money(self):
        return self._padded([e.money for e in self.envs], 0, np.int32)

    def timestep(self):
        return np.asarray([e.t for e in self.envs], dtype=np.int32)

    def visits(self):
        return np.stack([e.visits for e in self.envs]).astype(np.uint16)

    def masks(self):
        return self._padded([e.action_masks() for e in self.envs], False, bool)

    def node_features(self):
        return self._padded([e.node_features().T for e in self.envs], 0, np.float32).transpose(0, 2, 1).copy()

    def belief(self):
        return np.stack([e.belief for e in self.envs])

    def revealed(self):
        return np.asarray([e.revealed for e in self.envs], dtype=np.int32)


class OracleGroupBatch(OracleBatch):
    """A batch of mechanism groups with the conventions of a handle with groups (include/sy_env.h, sy_set_groups,
    sy_set_group_tolls, sy_set_group_rules): env b runs OracleEnv(cfgs[group_id[b]]) -- that group's police count,
    horizon, police budget, toll, reveal schedule and reward weights -- inside the handle's layout of A = num_police + 1
    agents.  Its start nodes are the first P_g + 1 draws of philox_start_positions, its reveal-skip draw uses its
    group's probability, its absent agents carry the absent values in every view and -1 from sample_actions, and its
    finished episodes and statistics are recorded with its group.  The handle-wide settings (reward mode, MrX budget,
    belief) come from each cfg and must agree."""

    def __init__(self, cfgs: Sequence[OracleConfig], group_id, num_police: int, graphs: List[Graph], graph_id,
                 start_positions, seed=0, auto_reset=False, env_offset=0, resample_graph=False):
        for c in cfgs:
            assert 1 <= c.num_police <= num_police, "a group plays with 1 .. num_police police"
            assert (c.reward_mode, c.mrx_money, c.belief) == (cfgs[0].reward_mode, cfgs[0].mrx_money, cfgs[0].belief)
        handle = OracleConfig(num_police=num_police, agent_money=0, reward_mode=cfgs[0].reward_mode)
        super().__init__(handle, graphs, graph_id, start_positions, seed, auto_reset, env_offset, resample_graph,
                         groups=(cfgs, group_id))

    @classmethod
    def from_seed(cls, cfgs, group_id, num_police, graphs, num_envs, seed=0, env_offset=0, auto_reset=True,
                  resample_graph=False):
        gid, sp = cls._seeded_starts(num_police + 1, graphs, num_envs, seed, env_offset, resample_graph)
        return cls(cfgs, group_id, num_police, graphs, gid, sp, seed, auto_reset, env_offset, resample_graph)
