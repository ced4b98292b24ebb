"""Batched forward of the reference's two shipped agents on the env's device state (SURVEY.md 8(f) row f2).

`GNNPolicy`   = GNNAgent.select_action / GNNModel.forward (src/agent/gnn_agent.py:45-82, 230-257) for MrX's agent and
                the police agent (gnn_trainer.py:147-165), all envs and agents in one launch.
`MappoPolicy` = MappoAgent.select_action / AgentPolicy / CentralCritic (src/agent/mappo_agent.py:6-44, 87-142).
`HeuristicPolicy` = heuristic opponents (evading MrX, chasing police) of libsy_env.so's sy_heuristic_actions, the
                counterpart of src/eval/exploitability.py:122,188 (parity unpinned).

Parameters use the reference modules' own `state_dict` keys, so checkpoints written by the reference
(`GNNAgent.save`, `MappoAgent.save`) load unchanged.  The kernels live in libsy_policy.so (include/sy_policy.h);
there is no PyTorch or CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _cabi
from . import _policy_cabi as pc
from .graphs import GraphSpec, pack_csr

GNN_KEYS = ("conv1.W", "conv1.bias", "conv1.phi.lin.weight", "conv2.W", "conv2.bias", "conv2.phi.lin.weight",
            "output_layer.weight", "output_layer.bias")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def gcn_in_edges(graphs: Sequence[GraphSpec]):
    """The directed aggregation lists GCNConv builds from `edge_links.T` as create_graph_data passes it
    (utils.py:169: every stored edge (u, v) is a message u -> v only) with gcn_norm's coefficients:
    deg = 1 + in-degree, coef(u -> v) = deg[u]^-1/2 deg[v]^-1/2, self loop 1/deg[v]."""
    N, G = graphs[0].num_nodes, len(graphs)
    stride = max(1, max(len(g.edges) for g in graphs))
    in_ptr = np.zeros((G, N + 1), dtype=np.int32)
    in_src = np.zeros((G, stride), dtype=np.int32)
    in_coef = np.zeros((G, stride), dtype=np.float32)
    self_coef = np.zeros((G, N), dtype=np.float32)
    for i, g in enumerate(graphs):
        src, dst = g.edge_links[:, 0].astype(np.int64), g.edge_links[:, 1].astype(np.int64)
        deg = (1.0 + np.bincount(dst, minlength=N)).astype(np.float32)
        dis = (deg ** np.float32(-0.5)).astype(np.float32)
        order = np.argsort(dst, kind="stable")
        np.cumsum(np.bincount(dst, minlength=N), out=in_ptr[i, 1:])
        in_src[i, : len(order)] = src[order]
        in_coef[i, : len(order)] = dis[src[order]] * dis[dst[order]]
        self_coef[i] = dis * dis
    return in_ptr, in_src, in_coef, self_coef, stride


class _GraphTables:
    """Device copies of the pool's CSR + in-edge lists for the policy kernels (rebuilt when the pool changes)."""

    def __init__(self, env):
        dev = env.device
        row_ptr, col, wgt = env._csr
        in_ptr, in_src, in_coef, self_coef, in_stride = gcn_in_edges(env.graphs)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
        self.tensors = [t(row_ptr.astype(np.int32)), t(col.astype(np.int32)), t(wgt.astype(np.int32)), t(in_ptr), t(in_src),
                        t(in_coef), t(self_coef)]
        s = pc.SyPolicyGraphs()
        s.num_graphs, s.num_nodes, s.nnz_stride, s.in_stride = env.num_graphs, env.graph_nodes, col.shape[1], in_stride
        (s.row_ptr, s.col, s.w, s.in_ptr, s.in_src, s.in_coef, s.self_coef) = [x.data_ptr() for x in self.tensors]
        self.struct = s
        self.max_degree = int(np.diff(row_ptr, axis=1).max())
        self.generation = env._gen["generation"]
        self.graphs_id = id(env.graphs)


class _PolicyBase:
    def __init__(self, env):
        self._lib = pc.load_library()
        self.env = env
        self._tables: Optional[_GraphTables] = None
        self._headroom: Optional[torch.Tensor] = None  # int32 [B, A] money - toll of the env's mechanism group

    def _graphs(self) -> pc.SyPolicyGraphs:
        # a refreshed device pool (env.regenerate_graphs) bumps the generation; `id(list)` alone can be recycled by a
        # new list at the same address, so both are compared
        if self._tables is None or self._tables.graphs_id != id(self.env.graphs) or \
                self._tables.generation != self.env._gen["generation"]:
            self._tables = _GraphTables(self.env)
        return self._tables.struct

    def _refuse_mixed_police(self):
        """Raise ValueError (before anything is launched) while some mechanism group's police count differs from the
        env's: the GNN's feature width and MAPPO's per-agent actors depend on the police count, and the policy kernels
        index with every agent's pos, so mixed police counts need one handle (and model) per count, as the reference
        trainer builds them."""
        if self.env._env_police is not None:
            raise ValueError("mechanism groups with their own number_of_agents: the policies need one handle per police "
                             "count (set every group's number_of_agents to the env's)")

    def _state(self) -> pc.SyPolicyState:
        e = self.env
        s = pc.SyPolicyState()
        s.num_envs, s.num_agents, s.toll, s.env_offset = e.num_envs, e.num_agents, int(e.tolls), e.env_offset
        s.pos, s.money, s.graph_id = e.pos.data_ptr(), e.money.data_ptr(), e.graph_id.data_ptr()
        if e._env_toll is not None:
            # mechanism groups with their own tolls: the kernels read budgets only to test w + toll <= money, so they get
            # the headroom money - toll_b and toll 0 (the same test, in exact integers)
            if self._headroom is None or self._headroom.shape != e.money.shape or self._headroom.device != e.money.device:
                self._headroom = torch.empty_like(e.money)
            torch.sub(e.money, e._env_toll, out=self._headroom)
            s.money, s.toll = self._headroom.data_ptr(), 0
        s.mrx_revealed = e.mrx_revealed.data_ptr()
        return s


class GNNPolicy(_PolicyBase):
    """Both GNN agents of the reference trainer on the batched env.

    `mrx_state` / `police_state`: GNNModel state_dicts (keys GNN_KEYS; K = node_feature_size = agents) or None for the
    modules' default initialisation drawn from `seed`.  `features`: "env" (the env's node_features observation) or
    "reference" (create_graph_data exactly as written, utils.py:176-199 -- see include/sy_policy.h)."""

    def __init__(self, env, mrx_state: Optional[Dict] = None, police_state: Optional[Dict] = None, *, features: str = "env",
                 conv_epsilon: float = 0.1, gamma: float = 0.1, seed: int = 0):
        super().__init__(env)
        if features not in ("env", "reference"):
            raise ValueError("features must be 'env' or 'reference'")
        self.K = env.num_agents  # utils.py:176
        self.feature_mode = pc.SY_FEATURES_ENV if features == "env" else pc.SY_FEATURES_REFERENCE
        self.conv_epsilon, self.gamma = float(conv_epsilon), float(gamma)
        gen = torch.Generator().manual_seed(int(seed))
        self.state = [self.default_state(self.K, gen) if sd is None else {k: sd[k].detach().float().cpu() for k in GNN_KEYS}
                      for sd in (mrx_state, police_state)]
        self.step_counter = 0
        self._pack()

    @staticmethod
    def default_state(K: int, gen: torch.Generator) -> Dict[str, torch.Tensor]:
        """AntiSymmetricConv.reset_parameters (kaiming_uniform(a=sqrt(5)) on W, zeros bias; GCNConv lin glorot) and
        nn.Linear's default init, from a torch.Generator."""
        def uni(shape, bound):
            return (torch.rand(shape, generator=gen) * 2 - 1) * bound
        sd = {}
        for c in ("conv1", "conv2"):
            sd[f"{c}.W"] = uni((K, K), 1.0 / math.sqrt(K))            # kaiming_uniform_(a=sqrt(5)): bound = 1/sqrt(fan_in)
            sd[f"{c}.bias"] = torch.zeros(K)
            sd[f"{c}.phi.lin.weight"] = uni((K, K), math.sqrt(6.0 / (2 * K)))  # glorot
        sd["output_layer.weight"] = uni((1, K), 1.0 / math.sqrt(K))
        sd["output_layer.bias"] = uni((1,), 1.0 / math.sqrt(K))
        return sd

    def load_state_dicts(self, mrx_state: Dict, police_state: Dict):
        self.state = [{k: sd[k].detach().float().cpu() for k in GNN_KEYS} for sd in (mrx_state, police_state)]
        self._pack()

    def _pack(self):
        K = self.K
        n = self._lib.sy_gnn_param_count(K)
        KP = 4 if K <= 4 else (8 if K <= 8 else 16)
        buf = np.zeros((2, n), dtype=np.float32)
        for m, sd in enumerate(self.state):
            off = 0
            for c in ("conv1", "conv2"):
                W = sd[f"{c}.W"].float()
                if tuple(W.shape) != (K, K):
                    raise ValueError(f"{c}.W has shape {tuple(W.shape)}, expected {(K, K)} (node_feature_size = agents)")
                was = (W - W.t() - self.gamma * torch.eye(K)).numpy()  # AntiSymmetricConv.forward
                th = sd[f"{c}.phi.lin.weight"].float().numpy()
                wasT = np.zeros((KP, KP), dtype=np.float32)
                thT = np.zeros((KP, KP), dtype=np.float32)
                wasT[:K, :K] = was.T
                thT[:K, :K] = th.T
                bias = np.zeros(KP, dtype=np.float32)
                bias[:K] = sd[f"{c}.bias"].float().numpy()
                for a in (wasT.ravel(), thT.ravel(), bias):
                    buf[m, off: off + a.size] = a
                    off += a.size
            buf[m, off: off + K] = sd["output_layer.weight"].float().numpy().reshape(-1)
            buf[m, off + KP] = float(sd["output_layer.bias"].reshape(-1)[0])
        self.params = torch.from_numpy(buf).to(self.env.device)

    def q_values(self) -> torch.Tensor:
        """float32 [B, 2, N]: GNNModel.forward of MrX's model ([:, 0]) and the police model ([:, 1]) per env."""
        self._refuse_mixed_police()
        e = self.env
        q = torch.empty(e.num_envs, 2, e.graph_nodes, dtype=torch.float32, device=e.device)
        with torch.cuda.device(e.device):
            pc.check(self._lib.sy_gnn_q_values(C.byref(self._graphs()), C.byref(self._state()), self.params.data_ptr(), self.K,
                                               self.conv_epsilon, self.feature_mode, q.data_ptr(), e._stream()))
        return q

    def act(self, epsilon_mrx: float = 0.0, epsilon_police: Optional[float] = None, step_counter: Optional[int] = None,
            out: Optional[torch.Tensor] = None, return_q: bool = False):
        """int64 [B, A] actions (epsilon-greedy over the valid moves, -1 without one); optionally the chosen Q."""
        self._refuse_mixed_police()
        e = self.env
        if step_counter is None:
            step_counter = self.step_counter
            self.step_counter += 1
        eps_p = epsilon_mrx if epsilon_police is None else epsilon_police
        acts = out if out is not None else torch.empty(e.num_envs, e.num_agents, dtype=torch.int64, device=e.device)
        qt = torch.empty(e.num_envs, e.num_agents, dtype=torch.float32, device=e.device) if return_q else None
        with torch.cuda.device(e.device):
            pc.check(self._lib.sy_gnn_act(C.byref(self._graphs()), C.byref(self._state()), self.params.data_ptr(), self.K,
                                          self.conv_epsilon, self.feature_mode, float(epsilon_mrx), float(eps_p),
                                          e.seed & 0xFFFFFFFFFFFFFFFF, int(step_counter) & 0xFFFFFFFF, acts.data_ptr(), _ptr(qt),
                                          e._stream()))
        return (acts, qt) if return_q else acts

    returns_actions = True  # RolloutCollector: the kernel already does the masked epsilon-greedy selection
    reads_state_only = True  # ... from positions, budgets, reveal flags and the graph pool: no dense observation is read
    epsilon = (0.0, 0.0)    # (MrX, police) exploration rates used by __call__

    def __call__(self, obs=None):
        return self.act(self.epsilon[0], self.epsilon[1])


class HeuristicPolicy:
    """Heuristic opponents for every env in one launch (sy_heuristic_actions, include/sy_env.h): an evading MrX
    (`mrx="evade"`: stay or move to the affordable free neighbour farthest from the nearest police) and chasing police
    (`police="chase"`: step towards MrX's revealed or last revealed node; `"chase_belief"`: towards the belief map's mode
    while MrX is hidden), or the random-valid policy (`"random"`) per side.  `None` leaves that side's columns of `out`
    as they are, so a learned policy can be scored against heuristic opponents: `a = gnn.act(); heur.act(out=a)`.
    Each side explores (takes the random-valid action) with its own probability `epsilon_*`.  Works with every
    mechanism group field, mixed police counts included.  The counterpart of src/eval/exploitability.py:122,188
    (parity unpinned).

    The policy owns `last_seen` (int32 [B], MrX's last revealed node per env); it follows the episodes when `act` is
    called at every step, as RolloutCollector and a plain step loop do.  `reset_memory()` clears it."""

    MRX_KINDS = {None: _cabi.SY_HEUR_NONE, "random": _cabi.SY_HEUR_RANDOM, "evade": _cabi.SY_HEUR_EVADE}
    POLICE_KINDS = {None: _cabi.SY_HEUR_NONE, "random": _cabi.SY_HEUR_RANDOM, "chase": _cabi.SY_HEUR_CHASE,
                    "chase_belief": _cabi.SY_HEUR_CHASE_BELIEF}
    returns_actions = True  # RolloutCollector: act() returns actions

    def __init__(self, env, mrx: Optional[str] = "evade", police: Optional[str] = "chase", epsilon_mrx: float = 0.0,
                 epsilon_police: float = 0.0):
        if mrx not in self.MRX_KINDS:
            raise ValueError(f"mrx must be one of {list(self.MRX_KINDS)}, got {mrx!r}")
        if police not in self.POLICE_KINDS:
            raise ValueError(f"police must be one of {list(self.POLICE_KINDS)}, got {police!r}")
        if police == "chase_belief" and not env.belief_on:
            raise ValueError("police='chase_belief' needs an env built with belief=True")
        self._lib = _cabi.load_library()
        self.env, self.mrx, self.police = env, mrx, police
        self.epsilon_mrx, self.epsilon_police = float(epsilon_mrx), float(epsilon_police)
        self.last_seen = torch.full((env.num_envs,), -1, dtype=torch.int32, device=env.device)
        # the dense belief map lags the state after a deferred step; everything else the kernel reads is compact state
        self.reads_state_only = police != "chase_belief"
        self._h = _cabi.SyHeuristic(C.sizeof(_cabi.SyHeuristic), self.MRX_KINDS[mrx], self.POLICE_KINDS[police],
                                    self.explore_threshold(epsilon_mrx), self.explore_threshold(epsilon_police),
                                    self.last_seen.data_ptr())

    @staticmethod
    def explore_threshold(epsilon: float) -> int:
        """floor(epsilon * 2^32), exact for every double in [0, 1]: an agent explores when its Philox word is below it"""
        if isinstance(epsilon, bool) or not isinstance(epsilon, (int, float, np.integer, np.floating)):
            raise ValueError(f"epsilon must be a number in [0, 1], got {epsilon!r}")
        e = float(epsilon)
        if not 0.0 <= e <= 1.0:  # (NaN fails both comparisons)
            raise ValueError(f"epsilon must be in [0, 1], got {epsilon!r}")
        return int(e * 2 ** 32)

    def reset_memory(self):
        """forget MrX's last revealed node in every env"""
        self.last_seen.fill_(-1)

    def act(self, out: Optional[torch.Tensor] = None, step_counter: Optional[int] = None) -> torch.Tensor:
        """int64 [B, A] actions (-1 = none).  `out`: int64 [B, A] on the env's device, written in place (the columns of
        a `None` side keep their values); None allocates one filled with -1.  `step_counter` keys the random draws
        exactly as `env.sample_actions`; None takes the env's sampler counter and advances it."""
        e = self.env
        if not e._is_reset:
            raise _cabi.SyError("act() before reset()")
        shape = (e.num_envs, e.num_agents)
        if out is None:
            out = torch.full(shape, -1, dtype=torch.int64, device=e.device)
        elif not (isinstance(out, torch.Tensor) and out.dtype == torch.int64 and tuple(out.shape) == shape
                  and out.device == e.device and out.is_contiguous()):
            raise ValueError(f"out must be a contiguous int64 tensor of shape {shape} on {e.device}")
        if step_counter is None:
            step_counter = e._sample_counter
            e._sample_counter += 1
        with torch.cuda.device(e.device):
            _cabi.check(self._lib.sy_heuristic_actions(e._handle, C.byref(self._h), C.byref(e._state), C.byref(e._obs),
                                                       int(step_counter) & 0xFFFFFFFF, out.data_ptr(), e._stream()))
        return out

    def __call__(self, obs=None):
        return self.act()


class MappoPolicy(_PolicyBase):
    """MrX's MappoAgent (one AgentPolicy) and the police MappoAgent (one AgentPolicy per officer) of
    mappo_trainer.py:124-147 on the batched env.  `policies`: list of AgentPolicy state_dicts
    (`actor.0.weight` [H, obs], `actor.0.bias`, `actor.2.weight` [N, H], `actor.2.bias`), `policy_of_agent[a]` picks
    the one agent a uses; None = default nn.Linear initialisation from `seed`, one policy per agent."""

    def __init__(self, env, obs_size: int, hidden_size: int = 64, policies: Optional[Sequence[Dict]] = None,
                 policy_of_agent: Optional[Sequence[int]] = None, critic: Optional[Dict] = None,
                 global_obs_size: Optional[int] = None, seed: int = 0):
        super().__init__(env)
        self.obs_size, self.hidden, self.N = int(obs_size), int(hidden_size), env.graph_nodes
        gen = torch.Generator().manual_seed(int(seed))
        A = env.num_agents
        if policies is None:
            policies = [self.default_policy(self.obs_size, self.hidden, self.N, gen) for _ in range(A)]
            policy_of_agent = list(range(A))
        self.policy_of_agent = np.asarray(policy_of_agent if policy_of_agent is not None else range(A), dtype=np.int32)
        n = self._lib.sy_mappo_param_count(self.obs_size, self.hidden, self.N)
        buf = np.zeros((len(policies), n), dtype=np.float32)
        for i, sd in enumerate(policies):
            parts = [sd["actor.0.weight"], sd["actor.0.bias"], sd["actor.2.weight"], sd["actor.2.bias"]]
            flat = np.concatenate([p.detach().float().cpu().numpy().ravel() for p in parts])
            if flat.size != n:
                raise ValueError(f"policy {i}: {flat.size} parameters, expected {n}")
            buf[i] = flat
        self.policies = list(policies)
        self.params = torch.from_numpy(buf).to(env.device)
        self.global_obs_size = global_obs_size
        self.critic_params = None
        if global_obs_size is not None:
            critic = critic or self.default_critic(int(global_obs_size), self.hidden, gen)
            self.critic = critic
            flat = np.concatenate([critic[k].detach().float().cpu().numpy().ravel()
                                   for k in ("critic.0.weight", "critic.0.bias", "critic.2.weight", "critic.2.bias")])
            self.critic_params = torch.from_numpy(flat.astype(np.float32)).to(env.device)
        self.step_counter = 0
        self.tensor_cores = True  # let the library use the tcgen05 path when the shapes allow (include/sy_policy.h)

    def check(self):
        """synchronise and surface a (never expected) failure flag of the tensor-core kernel"""
        with torch.cuda.device(self.env.device):
            pc.check(self._lib.sy_policy_check(self.env._stream()))

    @staticmethod
    def _linear(out_f, in_f, gen):
        b = 1.0 / math.sqrt(in_f)
        return (torch.rand(out_f, in_f, generator=gen) * 2 - 1) * b, (torch.rand(out_f, generator=gen) * 2 - 1) * b

    @classmethod
    def default_policy(cls, obs, hidden, n, gen):
        w1, b1 = cls._linear(hidden, obs, gen)
        w2, b2 = cls._linear(n, hidden, gen)
        return {"actor.0.weight": w1, "actor.0.bias": b1, "actor.2.weight": w2, "actor.2.bias": b2}

    @classmethod
    def default_critic(cls, d, hidden, gen):
        w1, b1 = cls._linear(hidden, d, gen)
        w2, b2 = cls._linear(1, hidden, gen)
        return {"critic.0.weight": w1, "critic.0.bias": b1, "critic.2.weight": w2, "critic.2.bias": b2}

    def act(self, obs: Optional[torch.Tensor] = None, step_counter: Optional[int] = None, return_probs: bool = False,
            out: Optional[torch.Tensor] = None):
        """obs float32 [B, A, obs_size] -> (actions int64 [B, A], log_probs float32 [B, A][, probs [B, A, N]]).
        obs=None: the kernel builds MappoTrainer's own observations from the env state (mappo_trainer.py:171-199: MrX
        sees his node, every officer the officers' nodes; raw node ids, zero-padded to obs_size >= P) without any
        observation tensor being materialised."""
        self._refuse_mixed_police()
        e = self.env
        if obs is None:
            if self.obs_size < e.number_of_agents:
                raise ValueError("obs=None (trainer features) needs obs_size >= number of police")
        else:
            if tuple(obs.shape) != (e.num_envs, e.num_agents, self.obs_size) or obs.dtype != torch.float32:
                raise ValueError(f"obs must be float32 {(e.num_envs, e.num_agents, self.obs_size)}")  # mappo_agent.py:21-28
            obs = obs.contiguous()
        if step_counter is None:
            step_counter = self.step_counter
            self.step_counter += 1
        acts = out if out is not None else torch.empty(e.num_envs, e.num_agents, dtype=torch.int64, device=e.device)
        if getattr(self, "_lp", None) is None:
            self._lp = torch.empty(e.num_envs, e.num_agents, dtype=torch.float32, device=e.device)
        lp = self._lp if out is not None else torch.empty(e.num_envs, e.num_agents, dtype=torch.float32, device=e.device)
        pr = torch.empty(e.num_envs, e.num_agents, self.N, dtype=torch.float32, device=e.device) if return_probs else None
        with torch.cuda.device(e.device):
            graphs = self._graphs()
            pc.check(self._lib.sy_mappo_act(C.byref(graphs), C.byref(self._state()), _ptr(obs), self.obs_size,
                                            self.hidden, self.params.data_ptr(), self.policy_of_agent.ctypes.data,
                                            self._tables.max_degree if self.tensor_cores else 0,
                                            e.seed & 0xFFFFFFFFFFFFFFFF, int(step_counter) & 0xFFFFFFFF, acts.data_ptr(),
                                            lp.data_ptr(), _ptr(pr), e._stream()))
        return (acts, lp, pr) if return_probs else (acts, lp)

    def values(self, global_obs: torch.Tensor) -> torch.Tensor:
        """CentralCritic.forward: float32 [M, global_obs_size] -> [M]."""
        if self.critic_params is None:
            raise ValueError("constructed without global_obs_size")
        x = global_obs.reshape(-1, self.global_obs_size).float().contiguous()
        out = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
        with torch.cuda.device(self.env.device):
            pc.check(self._lib.sy_mappo_values(x.data_ptr(), x.shape[0], self.global_obs_size, self.hidden,
                                               self.critic_params.data_ptr(), out.data_ptr(), self.env._stream()))
        return out
