"""CPU restatement of the reference's policy forward (SURVEY.md 8(f) row f2).  TEST INFRASTRUCTURE ONLY: imported by
tests/, never by the product.

GNN  (src/agent/gnn_agent.py:45-82, 230-257; src/training/utils.py:151-211): torch_geometric is a requirements.txt
     dependency of the reference that is neither pinned nor present in this image, so `antisymmetric_conv` restates its
     PUBLISHED algorithm (torch_geometric.nn.AntiSymmetricConv with phi = GCNConv(K, K, bias=False), gcn_norm with
     self-loops, flow source_to_target) in float64 NumPy, dense and in PyG's own operation order -- **parity unpinned**
     for the GNN: there is no reference output to pin it to here.
MAPPO (src/agent/mappo_agent.py:6-44, 87-142): restated in NumPy and PINNED against the unmodified reference modules
     (importable: they only need torch) through tests/golden/mappo.npz, written by oracle/gen_policy_golden.py.
"""
from __future__ import annotations

import numpy as np

try:  # package import (tests) or flat import (oracle/ on sys.path)
    from .sy_oracle import _M32, philox4x32
except ImportError:  # pragma: no cover
    from sy_oracle import _M32, philox4x32

RNG_GNN_POLICY, RNG_MAPPO_POLICY = 3, 4
FEATURES_ENV, FEATURES_REFERENCE = 0, 1


def u01(word: int) -> float:
    return float(np.float32(word >> 8) * np.float32(1.0 / 16777216.0))


def philox4x32_batched(c0, c1, c2, c3, seed):
    """`sy_oracle.philox4x32` over arrays of counters (broadcast), one 64-bit key: four uint32 arrays."""
    m = np.uint64(_M32)
    c = [np.asarray(x, dtype=np.uint64) & m for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & _M32), np.uint64((seed >> 32) & _M32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]  # 32 x 32 bits: exact in uint64
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & m, p1 & m, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & m, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return [x.astype(np.uint32) for x in c]


def u01_batched(words) -> np.ndarray:
    """float32 [0, 1) of the kernels' u01, elementwise"""
    return (np.asarray(words, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


# ------------------------------------------------------------------------------------------ GNN
def graph_features(mode, pos, revealed, n_nodes, n_agents) -> np.ndarray:
    """x [N, K=A].  FEATURES_ENV: the env's node_features (yard.py:283-291, MrX column blank while hidden).
    FEATURES_REFERENCE: create_graph_data as written (utils.py:176-199): column 0 at MrX_pos (numpy index -1 while
    hidden), columns 1..P-1 all at Polices_pos[0], last column empty."""
    x = np.zeros((n_nodes, n_agents), dtype=np.float64)
    if mode == FEATURES_ENV:
        for k in range(n_agents):
            if k == 0 and revealed < 0:
                continue
            x[pos[k], k] = 1
    else:
        x[pos[0] if revealed >= 0 else -1, 0] = 1
        for i in range(n_agents - 2):  # range(env.number_of_agents - 1) with number_of_agents = police
            x[pos[1], i + 1] = 1
    return x


def antisymmetric_conv(x, src, dst, W, bias, lin_w, epsilon=0.1, gamma=0.1):
    n = x.shape[0]
    deg = 1.0 + np.bincount(dst, minlength=n)  # gcn_norm: self-loops, in-degree at the target
    dis = deg ** -0.5
    xl = x @ lin_w.T  # GCNConv.lin (no bias)
    agg = (dis * dis)[:, None] * xl
    np.add.at(agg, dst, (dis[src] * dis[dst])[:, None] * xl[src])
    h = x @ (W - W.T - gamma * np.eye(W.shape[0])).T + agg + bias
    return x + epsilon * np.tanh(h)


def gnn_forward(x, edge_links, sd, epsilon=0.1, gamma=0.1) -> np.ndarray:
    """GNNModel.forward (gnn_agent.py:249-257): q [N]."""
    f = lambda k: np.asarray(sd[k], dtype=np.float64)  # noqa: E731
    src, dst = edge_links[:, 0].astype(np.int64), edge_links[:, 1].astype(np.int64)
    x = np.maximum(antisymmetric_conv(x, src, dst, f("conv1.W"), f("conv1.bias"), f("conv1.phi.lin.weight"), epsilon, gamma), 0)
    x = np.maximum(antisymmetric_conv(x, src, dst, f("conv2.W"), f("conv2.bias"), f("conv2.phi.lin.weight"), epsilon, gamma), 0)
    return (x @ f("output_layer.weight").T).reshape(-1) + float(f("output_layer.bias").reshape(-1)[0])


def graph_features_batched(mode, pos, revealed, n_nodes, n_agents) -> np.ndarray:
    """`graph_features` of many envs at once: x [B, N, K=A] from pos [B, A] and revealed [B]."""
    pos, revealed = np.asarray(pos, dtype=np.int64), np.asarray(revealed)
    B = len(pos)
    b = np.arange(B)
    x = np.zeros((B, n_nodes, n_agents), dtype=np.float64)
    if mode == FEATURES_ENV:
        for k in range(n_agents):
            on = revealed >= 0 if k == 0 else np.ones(B, dtype=bool)
            x[b[on], pos[on, k], k] = 1
    else:
        x[b, np.where(revealed >= 0, pos[:, 0], n_nodes - 1), 0] = 1
        for i in range(n_agents - 2):
            x[b, pos[:, 1], i + 1] = 1
    return x


def gcn_matrix(edge_links, n_nodes):
    """GCNConv's normalised propagation as a sparse [N, N] matrix (row = target): one entry per stored edge u -> v with
    deg[u]^-1/2 deg[v]^-1/2 (parallel edges are separate messages, so their entries add up), self-loops 1/deg[v]."""
    import scipy.sparse as sp

    src, dst = np.asarray(edge_links)[:, 0].astype(np.int64), np.asarray(edge_links)[:, 1].astype(np.int64)
    dis = (1.0 + np.bincount(dst, minlength=n_nodes)) ** -0.5
    v = np.arange(n_nodes)
    return sp.csr_matrix((np.concatenate([dis[src] * dis[dst], dis * dis]), (np.concatenate([dst, v]), np.concatenate([src, v]))),
                         shape=(n_nodes, n_nodes))


def gnn_forward_batched(mode, pos, revealed, graph_id, edge_links, sds, n_nodes, epsilon=0.1, gamma=0.1,
                        chunk_floats=1 << 23) -> np.ndarray:
    """`gnn_forward` of every env and every model in `sds`: q [B, len(sds), N] float64.  Features follow
    `graph_features_batched`, env b aggregates over graph `edge_links[graph_id[b]]`; envs are processed in chunks of at
    most `chunk_floats` feature entries so that a full batch fits in host memory."""
    pos, revealed, graph_id = np.asarray(pos), np.asarray(revealed), np.asarray(graph_id)
    B, K = pos.shape
    mats = [gcn_matrix(el, n_nodes) for el in edge_links]
    f = [{k: np.asarray(sd[k], dtype=np.float64) for k in sd} for sd in sds]
    q = np.zeros((B, len(sds), n_nodes), dtype=np.float64)
    step = max(1, chunk_floats // (n_nodes * K))
    for g, Ahat in enumerate(mats):
        envs = np.nonzero(graph_id == g)[0]
        for c0 in range(0, len(envs), step):
            e = envs[c0: c0 + step]
            x0 = graph_features_batched(mode, pos[e], revealed[e], n_nodes, K)
            for m, w in enumerate(f):
                x = x0
                for c in ("conv1", "conv2"):
                    xl = x @ w[f"{c}.phi.lin.weight"].T
                    agg = (Ahat @ xl.transpose(1, 0, 2).reshape(n_nodes, -1)).reshape(n_nodes, len(e), K).transpose(1, 0, 2)
                    h = x @ (w[f"{c}.W"] - w[f"{c}.W"].T - gamma * np.eye(K)).T + agg + w[f"{c}.bias"]
                    x = np.maximum(x + epsilon * np.tanh(h), 0)
                q[e, m] = (x @ w["output_layer.weight"].T)[..., 0] + float(w["output_layer.bias"].reshape(-1)[0])
    return q


def gnn_select(q, valid_moves, eps, seed, env, step, agent, tie_tol=0.0):
    """GNNAgent.select_action (gnn_agent.py:62-82) with the kernel's Philox draws.  Returns (action or -1, explored,
    set of acceptable argmax nodes within tie_tol)."""
    if len(valid_moves) == 0:
        return -1, False, {-1}
    r = philox4x32((env & _M32, step & _M32, RNG_GNN_POLICY, agent), (seed & _M32, (seed >> 32) & _M32))
    if u01(r[0]) < eps:
        a = int(valid_moves[(r[1] * len(valid_moves)) >> 32])
        return a, True, {a}
    qv = q[valid_moves]
    a = int(valid_moves[int(np.argmax(qv))])
    return a, False, {int(m) for m, v in zip(valid_moves, qv) if v >= qv.max() - tie_tol}


def gnn_explore_batched(mask, eps_mrx, eps_police, seed, env_ids, step):
    """The exploration half of `gnn_select` for all envs and agents: (explored [B, A] bool, action [B, A] = the drawn
    valid move where explored, else -1).  Agents without a valid move never explore."""
    mask = np.asarray(mask, dtype=bool)
    B, A, N = mask.shape
    r = philox4x32_batched(np.asarray(env_ids)[:, None], step, RNG_GNN_POLICY, np.arange(A)[None, :], seed)
    eps = np.full(A, np.float32(eps_police), dtype=np.float32)
    eps[0] = np.float32(eps_mrx)
    n_valid = mask.sum(-1)
    explored = (u01_batched(r[0]) < eps[None, :]) & (n_valid > 0)
    target = (r[1].astype(np.uint64) * n_valid.astype(np.uint64)) >> np.uint64(32)  # index into the ascending valid moves
    rank = np.cumsum(mask, axis=-1, dtype=np.int16) - np.int16(1)
    hit = mask & (rank == target[..., None].astype(np.int16))
    return explored, np.where(explored, hit.argmax(-1), -1)


# ------------------------------------------------------------------------------------------ MAPPO
def mappo_probs(obs, sd, mask, dtype=np.float64):
    """AgentPolicy.forward + the masking of select_action (mappo_agent.py:18-29, 102-133): current_probs [N]."""
    f = lambda k: np.asarray(sd[k], dtype=dtype)  # noqa: E731
    h = np.maximum(f("actor.0.weight") @ np.asarray(obs, dtype=dtype) + f("actor.0.bias"), 0)
    logits = f("actor.2.weight") @ h + f("actor.2.bias")
    e = np.exp(logits - logits.max())
    p = e / e.sum()
    m = np.asarray(mask, dtype=dtype)
    p = p * m
    s = p.sum()
    if s <= 1e-8:
        return m / m.sum() if m.sum() > 1e-8 else np.ones_like(m) / len(m)
    return p / (s + dtype(1e-8))


MAPPO_SOFTMAX, MAPPO_UNIFORM_MASK, MAPPO_UNIFORM_ALL = 0, 1, 2


def mappo_forward_batched(obs, sd, mask, chunk=8192):
    """`mappo_probs` for many rows of ONE policy: obs [R, D], mask [R, N].  Returns a dict of float64 / int arrays:
    `probs` [R, N], `mode` [R] (MAPPO_SOFTMAX: softmax * mask / (Sv + 1e-8); MAPPO_UNIFORM_MASK; MAPPO_UNIFORM_ALL),
    `masked` [R, N] (the softmax branch's probabilities whichever branch the row takes), `Sv` [R] (the softmax mass on
    the mask) and `scale` [R] = max_n (|b2_n| + sum_k |W2_nk| (|b1_k| + sum_o |W1_ko x_o|)), the magnitude every
    rounding error of a float32 evaluation of the logits is proportional to."""
    f = lambda k: np.asarray(sd[k], dtype=np.float64)  # noqa: E731
    W1, b1, W2, b2 = f("actor.0.weight"), f("actor.0.bias"), f("actor.2.weight"), f("actor.2.bias")
    obs, mask = np.asarray(obs, dtype=np.float64), np.asarray(mask, dtype=bool)
    R, N = mask.shape
    out = dict(probs=np.zeros((R, N)), masked=np.zeros((R, N)), mode=np.zeros(R, dtype=np.int64), Sv=np.zeros(R), scale=np.zeros(R))
    aW1, ab1, aW2, ab2 = np.abs(W1), np.abs(b1), np.abs(W2), np.abs(b2)
    for r0 in range(0, R, chunk):
        x, m = obs[r0: r0 + chunk], mask[r0: r0 + chunk]
        h = np.maximum(x @ W1.T + b1, 0)
        logits = h @ W2.T + b2
        e = np.exp(logits - logits.max(-1, keepdims=True))
        p = e / e.sum(-1, keepdims=True)
        Sv = (p * m).sum(-1)
        nv = m.sum(-1)
        mode = np.where(Sv > 1e-8, MAPPO_SOFTMAX, np.where(nv > 0, MAPPO_UNIFORM_MASK, MAPPO_UNIFORM_ALL))
        masked = p * m / (Sv + 1e-8)[:, None]
        probs = np.where(mode[:, None] == MAPPO_SOFTMAX, masked,
                         np.where(mode[:, None] == MAPPO_UNIFORM_MASK, m / np.maximum(nv, 1)[:, None], 1.0 / N))
        s1 = ab1 + np.abs(x) @ aW1.T  # |b1_k| + sum_o |W1_ko| |x_o|: bounds the hidden unit's partial sums
        out["probs"][r0: r0 + chunk] = probs
        out["masked"][r0: r0 + chunk] = masked
        out["mode"][r0: r0 + chunk] = mode
        out["Sv"][r0: r0 + chunk] = Sv
        out["scale"][r0: r0 + chunk] = (ab2 + s1 @ aW2.T).max(-1)
    return out


def critic_value_batched(x, sd):
    """`critic_value` of every row of x [M, D]: (values [M], scale [M] as in `mappo_forward_batched`)."""
    f = lambda k: np.asarray(sd[k], dtype=np.float64)  # noqa: E731
    W1, b1, W2, b2 = f("critic.0.weight"), f("critic.0.bias"), f("critic.2.weight").reshape(-1), f("critic.2.bias").reshape(-1)
    x = np.asarray(x, dtype=np.float64)
    v = np.maximum(x @ W1.T + b1, 0) @ W2 + b2[0]
    scale = abs(b2[0]) + (np.abs(b1) + np.abs(x) @ np.abs(W1).T) @ np.abs(W2)
    return v, scale


def categorical_log_prob(probs, action, dtype=np.float64):
    """torch.distributions.Categorical(probs=p).log_prob(a): p is renormalised, clamped to [eps, 1-eps] (float32 eps)."""
    eps = float(np.finfo(np.float32).eps)
    p = np.asarray(probs, dtype=dtype)
    return float(np.log(np.clip(p[action] / p.sum(), eps, 1 - eps)))


def mappo_sample(probs, seed, env, step, agent) -> int:
    """the kernel's inverse-CDF draw over the support in ascending node order"""
    r = philox4x32((env & _M32, step & _M32, RNG_MAPPO_POLICY, agent), (seed & _M32, (seed >> 32) & _M32))
    u = np.float32(u01(r[0]))
    p = np.asarray(probs, dtype=np.float32)
    support = np.nonzero(p > 0)[0]
    if len(support) == len(p):  # uniform over all nodes (empty mask)
        return min(int(u * np.float32(len(p))), len(p) - 1)
    thr = u * p[support].sum(dtype=np.float32)
    cum = np.float32(0)
    for n in support:
        cum += p[n]
        if thr < cum:
            return int(n)
    return int(support[-1])


def critic_value(x, sd, dtype=np.float64) -> float:
    f = lambda k: np.asarray(sd[k], dtype=dtype)  # noqa: E731
    h = np.maximum(f("critic.0.weight") @ np.asarray(x, dtype=dtype) + f("critic.0.bias"), 0)
    return float((f("critic.2.weight") @ h + f("critic.2.bias")).reshape(-1)[0])


# ------------------------------------------------------------------------------------------ GNN, second restatement
def gnn_forward_message_passing(x, edge_links, sd, epsilon=0.1, gamma=0.1):
    """GNNModel.forward again, written INDEPENDENTLY of `gnn_forward` as literal message passing in Python floats (no
    matrix algebra, no NumPy scatter): the way torch_geometric.nn.MessagePassing executes GCNConv --
    add_remaining_self_loops, degree by counting incoming edges at the TARGET (flow = source_to_target), one message
    norm(e) * lin(x)[source] per edge summed at its target -- and AntiSymmetricConv.forward's update line by line.
    The two restatements must agree to 1e-12 (tests/test_policy_oracle.py); neither is pinned to the real module
    (torch_geometric is absent here: parity unpinned, see oracle/gen_gnn_golden.py)."""
    x = [[float(v) for v in row] for row in np.asarray(x, dtype=np.float64)]
    n, K = len(x), len(x[0])
    edges = [(int(s), int(d)) for s, d in np.asarray(edge_links)]
    edges += [(v, v) for v in range(n)]  # self-loops (create_graph_data's edge lists never contain one)

    def lin(mat, vec):  # nn.Linear without bias: y = W vec
        return [sum(float(mat[c][k]) * vec[k] for k in range(len(vec))) for c in range(len(mat))]

    def conv(x, W, bias, theta):
        deg = [0.0] * n
        for _, d in edges:
            deg[d] += 1.0
        xl = [lin(theta, row) for row in x]  # GCNConv: x = self.lin(x) first, then propagate
        agg = [[0.0] * K for _ in range(n)]
        for s, d in edges:
            norm = deg[s] ** -0.5 * deg[d] ** -0.5
            for c in range(K):
                agg[d][c] += norm * xl[s][c]
        anti = [[float(W[r][c]) - float(W[c][r]) - (gamma if r == c else 0.0) for c in range(K)] for r in range(K)]
        out = []
        for v in range(n):
            h = lin(anti, x[v])  # x @ antisymmetric_W.t()
            out.append([x[v][c] + epsilon * float(np.tanh(h[c] + agg[v][c] + float(bias[c]))) for c in range(K)])
        return out

    f = lambda k: np.asarray(sd[k], dtype=np.float64)  # noqa: E731
    for layer in ("conv1", "conv2"):
        x = conv(x, f(f"{layer}.W"), f(f"{layer}.bias"), f(f"{layer}.phi.lin.weight"))
        x = [[max(v, 0.0) for v in row] for row in x]
    ow, ob = f("output_layer.weight").reshape(-1), float(f("output_layer.bias").reshape(-1)[0])
    return np.asarray([sum(ow[c] * row[c] for c in range(K)) + ob for row in x], dtype=np.float64)
