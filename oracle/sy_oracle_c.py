"""ctypes wrapper of oracle/sy_oracle.c (the plain-C CPU restatement; OpenMP over envs).

TEST INFRASTRUCTURE ONLY -- imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs,
never by the product.  `CBatch` has the same surface as `sy_oracle.OracleBatch`.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import sy_oracle as so

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sy_oracle.c")
LIB = os.path.join(HERE, "_build", "libsy_oracle.so")
CFLAGS = ["-O2", "-fno-fast-math", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC"]


def build(force=False):
    if force or not os.path.isfile(LIB) or os.path.getmtime(LIB) < os.path.getmtime(SRC):
        os.makedirs(os.path.dirname(LIB), exist_ok=True)
        subprocess.check_call(["gcc", *CFLAGS, "-o", LIB, SRC, "-lm"])
    return LIB


def available() -> bool:
    try:
        _lib()
        return True
    except Exception:
        return False


class SyoConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "num_nodes", "num_police", "agent_money", "mrx_money", "max_timestep", "reveal_interval", "toll", "belief",
        "reward_mode", "auto_reset", "resample_graph", "num_graphs", "nnz_stride", "n_exp", "n_cov")] + [
        ("reveal_skip_prob", C.c_float), ("env_offset", C.c_int64), ("seed", C.c_uint64), ("w", C.c_double * 11),
        ("exp_neg", C.c_void_p), ("coverage", C.c_void_p), ("W", C.c_void_p), ("D", C.c_void_p),
        ("row_ptr", C.c_void_p), ("col", C.c_void_p)]


class SyoState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("pos", "money", "t", "gid", "episode", "done", "visits", "belief", "revealed")]


class SyoOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("reward", "terminated", "truncated", "winner", "mask", "node_features")]


_cdll = None


def _lib():
    global _cdll
    if _cdll is None:
        lib = C.CDLL(build())
        lib.syo_apsp.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.syo_reset_all.argtypes = [C.POINTER(SyoConfig), C.c_int32, C.POINTER(SyoState), C.c_void_p, C.c_void_p]
        lib.syo_observe.argtypes = [C.POINTER(SyoConfig), C.c_int32, C.POINTER(SyoState), C.POINTER(SyoOut)]
        lib.syo_step.argtypes = [C.POINTER(SyoConfig), C.c_int32, C.POINTER(SyoState), C.c_void_p, C.POINTER(SyoOut), C.c_int32]
        lib.syo_sample_actions.argtypes = [C.POINTER(SyoConfig), C.c_int32, C.POINTER(SyoState), C.c_uint32, C.c_void_p, C.c_int32]
        lib.syo_philox4x32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.syo_max_threads.restype = C.c_int32
        for f in (lib.syo_apsp, lib.syo_reset_all, lib.syo_observe, lib.syo_step, lib.syo_sample_actions, lib.syo_philox4x32):
            f.restype = None
        _cdll = lib
    return _cdll


def max_threads() -> int:
    return int(_lib().syo_max_threads())


def philox4x32(ctr, key):
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    _lib().syo_philox4x32(c.ctypes.data, k.ctypes.data, out.ctypes.data)
    return tuple(int(x) for x in out)


def apsp(num_nodes, row_ptr, col, w) -> np.ndarray:
    """pathfinding.py:34-137 as an all-pairs table (0xFFFF = unreachable)."""
    row_ptr = np.ascontiguousarray(row_ptr, dtype=np.int32)
    col = np.ascontiguousarray(col, dtype=np.int32)
    w = np.ascontiguousarray(w, dtype=np.int32)
    D = np.zeros((num_nodes, num_nodes), dtype=np.int32)
    _lib().syo_apsp(num_nodes, row_ptr.ctypes.data, col.ctypes.data, w.ctypes.data, D.ctypes.data)
    return D


def _tables(max_timestep):
    return (np.exp(-np.arange(1100, dtype=np.float64)),
            np.exp(-np.log1p(np.arange(max(max_timestep + 8, 16), dtype=np.float64))))


class CBatch:
    """B envs stepped by the C oracle.  `cfg` is a sy_oracle.OracleConfig; `graphs` a list of
    sy_oracle.Graph (or anything with num_nodes / edge_links / edges)."""

    def __init__(self, cfg: so.OracleConfig, graphs, num_envs, seed=0, auto_reset=True, env_offset=0,
                 resample_graph=False, start_positions=None, graph_id=None, threads=1, with_obs=True):
        lib = _lib()
        self.cfg, self.B, self.threads = cfg, int(num_envs), int(threads)
        graphs = [g if isinstance(g, so.Graph) else so.Graph(g.num_nodes, g.edge_links, g.edges) for g in graphs]
        self.graphs = graphs
        N, P = graphs[0].num_nodes, cfg.num_police
        A, B, G = P + 1, self.B, len(graphs)
        self.N, self.A = N, A
        csr = [g.csr() for g in graphs]
        stride = max(1, max(len(c[1]) for c in csr))
        self._row_ptr = np.zeros((G, N + 1), dtype=np.int32)
        self._col = np.zeros((G, stride), dtype=np.int32)
        self._W = np.zeros((G, N, N), dtype=np.int32)
        self._D = np.zeros((G, N, N), dtype=np.int32)
        for i, (g, (rp, col, w)) in enumerate(zip(graphs, csr)):
            self._row_ptr[i] = rp
            self._col[i, : len(col)] = col
            self._W[i] = g.weight_matrix()
            self._D[i] = apsp(N, rp, col, w)
        exp_t, cov_t = _tables(cfg.max_timestep)
        self._exp = np.ascontiguousarray(cfg.exp_table if cfg.exp_table is not None else exp_t, dtype=np.float64)
        self._cov = np.ascontiguousarray(cfg.cov_table if cfg.cov_table is not None else cov_t, dtype=np.float64)
        c = SyoConfig()
        c.num_nodes, c.num_police, c.agent_money, c.mrx_money = N, P, cfg.agent_money, cfg.mrx_money
        c.max_timestep, c.reveal_interval, c.toll, c.belief = cfg.max_timestep, cfg.reveal_interval, cfg.toll, int(cfg.belief)
        c.reward_mode, c.auto_reset, c.resample_graph = int(cfg.reward_mode == "fp32"), int(auto_reset), int(resample_graph)
        c.num_graphs, c.nnz_stride, c.n_exp, c.n_cov = G, stride, len(self._exp), len(self._cov)
        c.env_offset, c.seed = int(env_offset), int(seed) & 0xFFFFFFFFFFFFFFFF
        c.reveal_skip_prob = float(cfg.reveal_skip_prob)
        for i, k in enumerate(so.REWARD_WEIGHT_NAMES):
            c.w[i] = float(cfg.reward_weights[k])
        c.exp_neg, c.coverage = self._exp.ctypes.data, self._cov.ctypes.data
        c.W, c.D, c.row_ptr, c.col = self._W.ctypes.data, self._D.ctypes.data, self._row_ptr.ctypes.data, self._col.ctypes.data
        self._c = c
        self.seed, self.env_offset = int(seed), int(env_offset)
        z = np.zeros
        self._pos, self._money = z((B, A), np.int32), z((B, A), np.int32)
        self._t, self._gid, self._episode = z(B, np.int32), z(B, np.int32), z(B, np.int32)
        self._done, self._visits = z(B, np.uint8), z((B, N), np.int32)
        self._belief = z((B, N), np.float64) if cfg.belief else None
        self._revealed = z(B, np.int32)
        self._state = SyoState(*[None if a is None else a.ctypes.data for a in (
            self._pos, self._money, self._t, self._gid, self._episode, self._done, self._visits, self._belief, self._revealed)])
        self._reward = z((B, A), np.float64)
        self._term, self._trunc, self._winner = z(B, np.uint8), z(B, np.uint8), z(B, np.int8)
        self._mask = z((B, A, N), np.uint8) if with_obs else None
        self._nf = z((B, N, A), np.float32) if with_obs else None
        self._out = SyoOut(*[None if a is None else a.ctypes.data for a in (
            self._reward, self._term, self._trunc, self._winner, self._mask, self._nf)])
        self._actions = z((B, A), np.int64)
        self.reset(start_positions, graph_id)

    def set_seed(self, seed):
        """new Philox key for every later draw (the handle's sy_set_seed; the C oracle reads its config on every call)"""
        self._c.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.seed = int(seed)

    def reset(self, start_positions=None, graph_id=None):
        """every env restarts at episode 0 (start nodes Philox(seed; env, 0) unless given), then observes"""
        B, A = self.B, self.A
        ip = None if start_positions is None else np.ascontiguousarray(start_positions, dtype=np.int32).reshape(B, A)
        gi = None if graph_id is None else np.ascontiguousarray(graph_id, dtype=np.int32).reshape(B)
        _lib().syo_reset_all(C.byref(self._c), B, C.byref(self._state), None if ip is None else ip.ctypes.data,
                             None if gi is None else gi.ctypes.data)
        _lib().syo_observe(C.byref(self._c), B, C.byref(self._state), C.byref(self._out))

    # -- OracleBatch surface
    def step(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.int64).reshape(self.B, self.A)
        _lib().syo_step(C.byref(self._c), self.B, C.byref(self._state), a.ctypes.data, C.byref(self._out), self.threads)
        rew = self._reward.astype(np.float32) if self.cfg.reward_mode == "fp32" else self._reward.copy()
        return dict(reward=rew, terminated=self._term.astype(bool), truncated=self._trunc.astype(bool),
                    winner=self._winner.copy())

    def sample_actions(self, step) -> np.ndarray:
        _lib().syo_sample_actions(C.byref(self._c), self.B, C.byref(self._state), int(step) & 0xFFFFFFFF,
                                  self._actions.ctypes.data, self.threads)
        return self._actions.copy()

    def steps(self, n, first_step=0):
        """n self-driven steps (random valid policy + step), no copies: the CPU-baseline loop"""
        lib = _lib()
        for s in range(n):
            lib.syo_sample_actions(C.byref(self._c), self.B, C.byref(self._state), (first_step + s) & 0xFFFFFFFF,
                                   self._actions.ctypes.data, self.threads)
            lib.syo_step(C.byref(self._c), self.B, C.byref(self._state), self._actions.ctypes.data, C.byref(self._out),
                         self.threads)

    def pos(self):
        return self._pos.copy()

    def money(self):
        return self._money.copy()

    def timestep(self):
        return self._t.copy()

    def visits(self):
        return self._visits.astype(np.uint16)

    def masks(self):
        return self._mask.astype(bool)

    def node_features(self):
        return self._nf.copy()

    def belief(self):
        return self._belief.copy()

    def revealed(self):
        return self._revealed.copy()

    @property
    def graph_id(self):
        return self._gid.tolist()

    @property
    def episode(self):
        return self._episode.tolist()

    @property
    def done(self):
        return self._done.astype(bool).tolist()
