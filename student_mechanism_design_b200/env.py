"""Batched Scotland Yard environment on one B200: host-side mirror of the reference's
`CustomEnvironment` (/root/reference/src/environment/yard.py:14-607) over libsy_env.so.

Same constructor names (`number_of_agents`, `agent_money`, `reward_weights`, `logger`, `epoch`,
`graph_nodes`, `graph_edges`, `vis_configs`), same `reset` / `step` verbs, same observation keys
(yard.py:319-332 plus `belief_map` / `MrX_revealed`), but every tensor carries a leading batch
dimension B and lives on the GPU; all per-step work happens in the CUDA kernels of
csrc/sy_env.cu.  PyTorch is used only to own device memory and streams.
There is NO CPU fallback: constructing the env without the built library or without a CUDA
device raises.
"""
from __future__ import annotations

import ctypes as C
import hashlib
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _cabi
from .graphs import GraphSpec, generate_graph_pool, pack_csr

# /root/reference/src/reward_net.py:5-17
REWARD_WEIGHT_NAMES = [
    "Police_distance", "Police_group", "Police_position", "Police_time", "Mrx_closest", "Mrx_average",
    "Mrx_position", "Mrx_time", "Police_coverage", "Police_proximity", "Police_overlap_penalty",
]
# /root/reference/src/training/evaluator.py:59-71
DEFAULT_REWARD_WEIGHTS = {
    "Police_distance": 0.1, "Police_group": 0.1, "Police_position": 0.1, "Police_time": 0.0,
    "Mrx_closest": 0.3, "Mrx_average": 0.2, "Mrx_position": 0.1, "Mrx_time": 0.0,
    "Police_coverage": 0.05, "Police_proximity": 0.05, "Police_overlap_penalty": 0.0,
}
GRAPH_BLOCK = 32  # default graph assignment: env e plays on graph (e // 32) % G
MAX_MONEY_LIMIT = 1000  # yard.py:11
N_EXP_TABLE = 1100  # exp(-d) underflows to 0 beyond d = 745


MECHANISM_KEYS = ("reward_weights", "agent_money", "reveal_interval", "reveal_skip_prob", "tolls", "number_of_agents",
                  "max_timestep")


def _integral(name: str, v, lo: int, hi: int) -> int:
    """`v` as an int in [lo, hi]: integral numbers (2.0 too) and 0-dim tensors, never bools"""
    if isinstance(v, torch.Tensor):
        v = v.item()
    if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or not np.isfinite(v) \
            or int(v) != v or not lo <= int(v) <= hi:
        raise ValueError(f"{name} must be an integer in [{lo}, {hi}], got {v!r}")
    return int(v)


def mechanism_toll(mech: Dict, base) -> int:
    """The toll of one mechanism dict: its `tolls` (the constructor's rule: integral and >= 0, so 1.0 is accepted; at most
    SY_MAX_TOLL), else `base.tolls`.  Raises ValueError on what sy_set_group_tolls would refuse."""
    return _integral("tolls", mech["tolls"] if "tolls" in mech else base.tolls, 0, _cabi.SY_MAX_TOLL)


def mechanism_rules(mech: Dict, base) -> Tuple[int, int]:
    """(police count, episode horizon) of one mechanism dict: its `number_of_agents` (the number of POLICE, named as in
    the constructor; the reference trainer's `num_police_agents: k` is an env with k + 1 police) in
    [1, base.number_of_agents], and its `max_timestep` in [0, base.config.max_timestep]; a missing key takes `base`'s
    value.  Raises ValueError on what sy_set_group_rules would refuse."""
    top_p, top_t = base.number_of_agents, base.config.max_timestep
    police = _integral("number_of_agents", mech["number_of_agents"], 1, top_p) if "number_of_agents" in mech else top_p
    horizon = _integral("max_timestep", mech["max_timestep"], 0, top_t) if "max_timestep" in mech else top_t
    return police, horizon


def pack_mechanism(mech: Dict, base) -> "_cabi.SyGroup":
    """One mechanism dict (keys of MECHANISM_KEYS, all optional) as the SyGroup of sy_set_groups; missing keys and
    missing reward-weight names take `base`'s values (an env, or anything with `reward_weights`, `agent_money`,
    `reveal_interval` and `config.reveal_skip_prob`).  Raises ValueError / KeyError on what the library would refuse.
    `tolls`, `number_of_agents` and `max_timestep` keys are validated here (mechanism_toll, mechanism_rules) but travel
    separately, through sy_set_group_tolls / sy_set_group_rules."""
    if not isinstance(mech, dict):
        raise TypeError(f"a mechanism is a dict, got {type(mech).__name__}")
    unknown = set(mech) - set(MECHANISM_KEYS)
    if unknown:
        raise KeyError(f"unknown mechanism keys {sorted(unknown)}; expected {list(MECHANISM_KEYS)}")
    weights = dict(base.reward_weights)
    given = mech.get("reward_weights", {}) or {}
    bad = set(given) - set(REWARD_WEIGHT_NAMES)
    if bad:
        raise KeyError(f"unknown reward weights {sorted(bad)}")
    weights.update(given)
    w = [float(weights[k].detach()) if isinstance(weights[k], torch.Tensor) else float(weights[k]) for k in REWARD_WEIGHT_NAMES]
    if not all(np.isfinite(w)):
        raise ValueError("reward weights must be finite")
    money = _integral("agent_money", mech.get("agent_money", base.agent_money), 0, _cabi.INT32_MAX)
    reveal = _integral("reveal_interval", mech.get("reveal_interval", base.reveal_interval), 0, _cabi.INT32_MAX)
    skip = float(mech.get("reveal_skip_prob", base.config.reveal_skip_prob))
    if not 0.0 <= skip <= 1.0:
        raise ValueError(f"reveal_skip_prob must be in [0, 1], got {skip}")
    if "tolls" in mech:
        mechanism_toll(mech, base)
    if "number_of_agents" in mech or "max_timestep" in mech:
        mechanism_rules(mech, base)
    g = _cabi.SyGroup()
    g.struct_bytes = C.sizeof(_cabi.SyGroup)
    for i, v in enumerate(w):
        g.reward_weights[i] = v
    g.agent_money, g.reveal_interval, g.reveal_skip_prob = money, reveal, skip
    return g


def unpack_mechanism(g: "_cabi.SyGroup", tolls: Optional[int] = None, rules: Optional[Tuple[int, int]] = None) -> Dict:
    """The complete mechanism dict of a SyGroup (float weights), with `tolls` and (`rules` = (police, horizon))
    `number_of_agents` / `max_timestep` when given"""
    d = dict(reward_weights={k: float(g.reward_weights[i]) for i, k in enumerate(REWARD_WEIGHT_NAMES)},
             agent_money=int(g.agent_money), reveal_interval=int(g.reveal_interval),
             reveal_skip_prob=float(g.reveal_skip_prob))
    if tolls is not None:
        d["tolls"] = int(tolls)
    if rules is not None:
        d["number_of_agents"], d["max_timestep"] = int(rules[0]), int(rules[1])
    return d


def group_metrics(per: Sequence[Dict], mechanisms: Sequence[Dict], number_of_agents: int):
    """What metrics() needs while mechanism groups are set, from the per-group statistics `per` (stats(by_group=True))
    and the mechanism dicts: (efficiency sum, tolls paid, per-group metrics).  A group's budget efficiency uses its own
    police budget P_g * agent_money_g (P_g = its `number_of_agents`, else `number_of_agents`) and its mean_tolls_paid
    its own toll; the aggregate weighs every group against its own budget and sums the tolls paid as the integer sum
    over groups of toll * police_moves (divided once: groups with the constructor's toll give exactly the float of a
    handle without groups)."""
    budgets = [max(int(m.get("number_of_agents", number_of_agents)) * m["agent_money"], 1) for m in mechanisms]
    by_group = [metrics_of(g, initial=b, tolls_paid=m["tolls"] * g["police_moves"]) for g, m, b in zip(per, mechanisms, budgets)]
    eff = sum(g["sum_episode_budget_spent"] / b for g, b in zip(per, budgets))
    paid = sum(int(m["tolls"]) * int(g["police_moves"]) for g, m in zip(per, mechanisms))
    return eff, paid, by_group


def metrics_of(st: Dict, initial: int, tolls_paid: int, eff_sum=None) -> Dict[str, float]:
    """MetricsTracker.get_aggregated_metrics (src/eval/metrics.py:168-232) of one statistics dict; `initial` = the police
    budget of an episode, `tolls_paid` = the tolls paid over all episodes (an integer)"""
    n = st["episodes"]
    r = st["reveals"]
    mean_ce = st["sum_belief_ce_q24"] / _cabi.BELIEF_CE_SCALE / r if r else 0.0
    var_ce = max(st["sum_sq_belief_ce_q24"] / _cabi.BELIEF_CE_SCALE / r - mean_ce * mean_ce, 0.0) if r else 0.0
    if n == 0:  # metrics.py:170-186
        return dict(num_episodes=0, mrx_wins=0, police_wins=0, win_rate=0.5, win_rate_std=0.0, mean_episode_length=0.0,
                    episode_length_std=0.0, mean_belief_ce=mean_ce, belief_ce_std=float(np.sqrt(var_ce)),
                    mean_tolls_paid=0.0, mean_budget_spent=0.0, mean_budget_efficiency=0.0,
                    mean_time_to_catch=0.0, mean_survival_time=0.0)
    wr = st["mrx_wins"] / n
    ml = st["sum_episode_length"] / n
    var_l = max(st["sum_sq_episode_length"] / n - ml * ml, 0.0)
    spent = st["sum_episode_budget_spent"] / n
    return dict(
        num_episodes=n, mrx_wins=st["mrx_wins"], police_wins=st["police_wins"], win_rate=wr,
        win_rate_std=float(np.sqrt(wr * (1.0 - wr))), mean_episode_length=ml, episode_length_std=float(np.sqrt(var_l)),
        mean_belief_ce=mean_ce, belief_ce_std=float(np.sqrt(var_ce)),
        mean_tolls_paid=tolls_paid / n, mean_budget_spent=spent,
        mean_budget_efficiency=spent / initial if eff_sum is None else eff_sum / n,
        mean_time_to_catch=st["sum_length_police_wins"] / st["police_wins"] if st["police_wins"] else 0.0,
        mean_survival_time=st["sum_length_mrx_wins"] / st["mrx_wins"] if st["mrx_wins"] else 0.0,
    )


def numpy_reward_tables(max_timestep: int = 250):
    """The two float64 tables the kernels read instead of calling exp/log1p, computed by NumPy
    on this host so the rewards equal the reference's `np.exp` bit for bit
    (reward_calculator.py:186,199,204-205,214)."""
    exp_neg = np.exp(-np.arange(N_EXP_TABLE, dtype=np.float64))
    coverage = np.exp(-np.log1p(np.arange(max(max_timestep + 8, 16), dtype=np.float64)))
    return exp_neg, coverage


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class BatchedScotlandYardEnv:
    """B independent games stepped by one kernel launch.

    Parameters mirror yard.py:18-28; extras: `num_envs`, `graphs` (a pool of GraphSpec, None to
    generate `num_graphs` on the host, or "device" to sample them on the GPU -- both with the
    reference's distribution; `regenerate_graphs` then refreshes a device pool), `reveal_interval`,
    `tolls`, `belief`, `reward_mode` ("fp64" | "fp32" | None = infer from the weight types, as
    the reference's arithmetic follows them), `seed`, `auto_reset`, `resample_graph`,
    `env_offset` (global index of env 0 when the batch is sharded over GPUs).
    """

    DEFAULT_ACTION = -1  # yard.py:16
    metadata = {"name": "scotland_yard_env_b200"}

    def __init__(self, num_envs: int, number_of_agents: int, agent_money: int, reward_weights: Optional[Dict] = None,
                 logger=None, epoch: int = 0, graph_nodes: int = 50, graph_edges: Optional[int] = 110, vis_configs=None,
                 *, graphs: Optional[Sequence[GraphSpec]] = None, num_graphs: int = 1, reveal_interval: int = 0,
                 tolls: float = 0, belief: bool = False, belief_ce: bool = False, reward_mode: Optional[str] = None, seed: int = 0,
                 auto_reset: bool = False, resample_graph: bool = False, env_offset: int = 0, max_timestep: int = 250,
                 device="cuda:0", reward_tables=None, keep_reward64: bool = False, collect_stats: bool = True,
                 graph_offset: int = 0, max_edges_per_node: int = 4, max_weight: int = 5,
                 node_features_dtype: torch.dtype = torch.float32, reveal_skip_prob: float = 0.0, guard_bytes: int = 0):
        # the int32 fields of SyConfig, checked before ctypes would wrap them (2**32 + 5 reads back as 5); the library
        # refuses the rest (police count, node count)
        num_envs = _integral("num_envs", num_envs, 1, _cabi.INT32_MAX)
        agent_money = _integral("agent_money", agent_money, 0, _cabi.INT32_MAX)
        max_timestep = _integral("max_timestep", max_timestep, 0, _cabi.SY_MAX_TIMESTEP)
        reveal_interval = _integral("reveal_interval", reveal_interval or 0, 0, _cabi.INT32_MAX)
        tolls = _integral("tolls", tolls, 0, _cabi.SY_MAX_TOLL)
        if not torch.cuda.is_available():
            raise _cabi.SyError("BatchedScotlandYardEnv needs a CUDA device; there is no CPU fallback")
        self._lib = _cabi.load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _cabi.SyError(f"device must be a CUDA device, got {device}")
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)
        self.logger, self.epoch, self.vis_config = logger, epoch, vis_configs
        self.num_envs = int(num_envs)
        self.number_of_agents = int(number_of_agents)  # number of POLICE, yard.py:33
        self.num_agents = self.number_of_agents + 1
        self.agent_money = int(agent_money)
        self.possible_agents = ["MrX"] + [f"Police{i}" for i in range(self.number_of_agents)]  # yard.py:54-56
        self.agents = list(self.possible_agents)
        reward_weights = dict(DEFAULT_REWARD_WEIGHTS) if reward_weights is None else dict(reward_weights)
        missing = [k for k in REWARD_WEIGHT_NAMES if k not in reward_weights]
        if missing:
            raise KeyError(f"reward_weights lacks {missing}")
        if reward_mode is None:  # reference arithmetic follows the weight types (gnn_trainer.py:98-110)
            reward_mode = "fp32" if any(isinstance(v, torch.Tensor) for v in reward_weights.values()) else "fp64"
        if reward_mode not in ("fp64", "fp32"):
            raise ValueError("reward_mode must be 'fp64' or 'fp32'")
        self.reward_mode = reward_mode
        self.reward_weights = reward_weights
        wvals = [float(reward_weights[k].detach()) if isinstance(reward_weights[k], torch.Tensor) else float(reward_weights[k])
                 for k in REWARD_WEIGHT_NAMES]

        # ---- graph pool
        self._device_pool = isinstance(graphs, str)
        self._gen = dict(graph_offset=int(graph_offset), cap=int(max_edges_per_node), max_weight=int(max_weight), generation=0)
        if self._device_pool:
            if graphs != "device":
                raise ValueError("graphs must be a sequence of GraphSpec, None or 'device'")
            self.graphs: List[GraphSpec] = []
            self.graph_nodes, self.num_graphs, self.actual_num_edges = int(graph_nodes), int(num_graphs), 0
        else:
            if graphs is None:
                graphs = generate_graph_pool(num_graphs, graph_nodes, graph_edges, seed=seed)
            self.graphs = list(graphs)
            self.graph_nodes = self.graphs[0].num_nodes
            self.actual_num_edges = len(self.graphs[0].edges)  # yard.py:70
            self.num_graphs = len(self.graphs)
        self.graph_edges = graph_edges
        N, A, B = self.graph_nodes, self.num_agents, self.num_envs

        cfg = _cabi.SyConfig()
        cfg.struct_bytes = C.sizeof(_cabi.SyConfig)
        cfg.device, cfg.num_envs, cfg.num_nodes, cfg.num_police = dev_index, B, N, self.number_of_agents
        cfg.agent_money, cfg.mrx_money, cfg.max_timestep = self.agent_money, MAX_MONEY_LIMIT, int(max_timestep)
        cfg.reveal_interval, cfg.toll = int(reveal_interval or 0), int(tolls)
        # belief_ce: also score the predicted belief at reveal steps (stats "reveals" / "sum_belief_ce_q24", metrics())
        cfg.belief = 2 if (belief and belief_ce) else int(bool(belief))
        cfg.reward_mode = _cabi.SY_REWARD_FP32 if reward_mode == "fp32" else _cabi.SY_REWARD_FP64
        cfg.auto_reset, cfg.resample_graph = int(bool(auto_reset)), int(bool(resample_graph))
        cfg.env_offset, cfg.seed = int(env_offset), int(seed) & 0xFFFFFFFFFFFFFFFF
        # robustness hook of src/eval/ood_eval.py:191-234 (RobustnessWrapper.reveal_skip_prob; `reveal_probability` of
        # src/configs/ablation/belief.yaml is 1 - this): every scheduled reveal is skipped with this probability
        cfg.reveal_skip_prob = float(reveal_skip_prob)
        for i, v in enumerate(wvals):
            cfg.reward_weights[i] = v
        self.config = cfg
        self.reveal_interval, self.tolls, self.belief_on = cfg.reveal_interval, cfg.toll, bool(cfg.belief)
        self.auto_reset, self.seed, self.env_offset = bool(auto_reset), int(seed), int(env_offset)

        self._handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_create(C.byref(cfg), C.byref(self._handle)))
            stream = self._stream()
            exp_neg, coverage = reward_tables if reward_tables is not None else numpy_reward_tables(max_timestep)
            exp_neg = np.ascontiguousarray(exp_neg, dtype=np.float64)
            coverage = np.ascontiguousarray(coverage, dtype=np.float64)
            _cabi.check(self._lib.sy_set_reward_tables(self._handle, exp_neg.ctypes.data, len(exp_neg),
                                                       coverage.ctypes.data, len(coverage), stream))
            if self._device_pool:
                self._generate_on_device(0)
            else:
                row_ptr, col, wgt, stride = pack_csr(self.graphs)
                self._csr = (row_ptr, col, wgt)
                _cabi.check(self._lib.sy_load_graphs(self._handle, self.num_graphs, row_ptr.ctypes.data, col.ctypes.data,
                                                     wgt.ctypes.data, stride, stream))

            dev = self.device
            # guard_bytes > 0 (memory-safety tests; compute-sanitizer is not available on the GPU pool): every buffer the
            # kernels write sits between two canary bands inside its own allocation; check_guards() verifies them
            self._guards = []
            guard = (int(guard_bytes) + 255) & ~255

            def z(*shape, dtype):
                if not guard:
                    return torch.zeros(*shape, dtype=dtype, device=dev)
                n = 1
                for d in shape:
                    n *= int(d)
                nbytes = n * torch.empty((), dtype=dtype).element_size()
                raw = torch.full((2 * guard + ((nbytes + 255) & ~255),), 0xA5, dtype=torch.uint8, device=dev)
                raw[guard:guard + nbytes].zero_()
                self._guards.append((raw, guard, nbytes))
                return raw[guard:guard + nbytes].view(dtype).view(*shape)

            self.pos = z(B, A, dtype=torch.int32)
            self.money = z(B, A, dtype=torch.int32)
            self.timestep = z(B, dtype=torch.int32)
            self.graph_id = z(B, dtype=torch.int32)
            self.episode = z(B, dtype=torch.int32)
            self.done = z(B, dtype=torch.uint8)
            self.visits = z(B, N, dtype=torch.uint16)
            self.belief_map = z(B, N, dtype=torch.float32) if self.belief_on else None
            self.action_mask = z(B, A, N, dtype=torch.bool)
            if node_features_dtype not in (torch.float32, torch.uint8):
                raise ValueError("node_features_dtype must be torch.float32 or torch.uint8")
            # uint8: the one-hot is exact in a byte and the step writes 3 N A fewer bytes per env (opt-in)
            self.node_features = z(B, N, A, dtype=node_features_dtype)
            self.agent_budget = z(B, A, dtype=torch.float32)
            self.mrx_revealed = z(B, dtype=torch.int32)
            # step results live in ONE block (reward | terminated | truncated | done | winner) so that the host-buffer
            # path moves them with a single D2H copy
            self._result_block = z(self._result_bytes(), dtype=torch.uint8)
            (self.reward, self.terminated, self.truncated, self.done_flags, self.winner,
             self.status) = self._result_views(self._result_block)
            self.reward64 = z(B, A, dtype=torch.float64) if keep_reward64 else None
            self.stats_vec = z(_cabi.SY_NUM_STATS, dtype=torch.int64) if collect_stats else None
        self._state = _cabi.SyState(_ptr(self.pos), _ptr(self.money), _ptr(self.timestep), _ptr(self.graph_id),
                                    _ptr(self.episode), _ptr(self.done), _ptr(self.visits), _ptr(self.belief_map))
        nf_f32 = self.node_features.dtype == torch.float32
        self._obs = _cabi.SyObs(_ptr(self.action_mask), _ptr(self.node_features) if nf_f32 else None, _ptr(self.agent_budget),
                                _ptr(self.mrx_revealed), None if nf_f32 else _ptr(self.node_features))
        self._out = _cabi.SyOut(_ptr(self.reward), _ptr(self.reward64), _ptr(self.terminated), _ptr(self.truncated),
                                _ptr(self.done_flags), _ptr(self.winner), _ptr(self.stats_vec), _ptr(self.status))
        self._static = None
        self._sample_counter = 0
        self._is_reset = False
        self._need_full_reset = False
        self._mechanisms, self._group_id, self.group_stats_vec = None, None, None  # set_mechanisms
        self._env_toll = None  # int32 [B, 1] while some mechanism group's toll differs from `tolls`
        self._env_police = None  # int32 [B, 1] while some mechanism group's police count differs from number_of_agents
        self._groups_generation = 0  # set_mechanisms calls: captured rollout graphs check it

    # ------------------------------------------------------------------ plumbing
    def _result_bytes(self) -> int:
        n = self.num_envs * self.num_agents
        return 4 * n + 3 * n + 2 * self.num_envs

    def _result_views(self, block: torch.Tensor):
        B, A = self.num_envs, self.num_agents
        n = B * A
        reward = block[: 4 * n].view(torch.float32).view(B, A)
        flags = [block[4 * n + k * n: 4 * n + (k + 1) * n].view(torch.bool).view(B, A) for k in range(3)]
        winner = block[7 * n: 7 * n + B].view(torch.int8)
        status = block[7 * n + B: 7 * n + 2 * B]  # uint8 [B]: bit 0 terminated, 1 truncated, 2 frozen (done = any)
        return reward, flags[0], flags[1], flags[2], winner, status

    def check_guards(self):
        """(guard_bytes > 0) Raise if a kernel wrote outside any state / observation / result buffer."""
        for i, (raw, guard, nbytes) in enumerate(getattr(self, "_guards", [])):
            lo, hi = raw[:guard], raw[guard + nbytes:]
            if not (bool((lo == 0xA5).all()) and bool((hi == 0xA5).all())):
                bad_lo = int((lo != 0xA5).sum())
                bad_hi = int((hi != 0xA5).sum())
                raise _cabi.SyError(f"guard band of buffer {i} ({nbytes} bytes) overwritten: {bad_lo} bytes below, {bad_hi} above")

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def close(self):
        if getattr(self, "_handle", None) is not None and self._handle:
            self._lib.sy_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _dev(self, x, dtype, shape):
        t = torch.as_tensor(x)
        t = t.to(device=self.device, dtype=dtype).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    OPTIONS = {"writer_path": (0, {"bulk": 0, "lsu": 1}), "step_kernel": (1, {"fused": 0, "two_kernels": 1, "auto": 2}),
               "nf_fill": (2, {"off": 0, "on": 1}), "lagged_kernel": (3, {"off": 0, "on": 1, "auto": 2}),
               "tail_split": (4, {"off": 0, "on": 1}), "rollout_kernel": (5, {"off": 0, "on": 1}),
               "pdl": (6, {"off": 0, "on": 1})}  # include/sy_env.h SY_OPT_*

    def set_option(self, name: str, value):
        """Tuning knobs of the handle (results are identical for every setting; include/sy_env.h SY_OPT_*):
        `step_kernel` = "auto" (default: the fused persistent kernel for batches of up to ~9 500 envs, else two kernels)
        | "fused" | "two_kernels"; `writer_path` of the two-kernel path's observation kernel = "lsu" (default) | "bulk"
        (TMA bulk stores); `nf_fill` = "off" (default) | "on" (split step: TMA fill kernel next to the dynamics);
        `lagged_kernel` = "auto" (default: deferred steps and the random rollouts run observations of step k + dynamics of
        step k+1 as one launch when the batch is one wave of that kernel, <= ~9 500 envs) | "on" | "off"; `tail_split` =
        "on" (default) | "off" (the observation grid's partly filled last wave cut into parts); `rollout_kernel` = "on"
        (default) | "off" (random rollouts of single-wave batches as ONE launch for all steps)."""
        opt, values = self.OPTIONS[name]
        _cabi.check(self._lib.sy_set_option(self._handle, opt, values[value] if isinstance(value, str) else int(value)))
        self.options = dict(getattr(self, "options", {}), **{name: value})

    def set_belief_hint(self, hint: Optional[torch.Tensor]):
        """Observation hint of ParticleBeliefTracker.update (belief_module.py:102-106) for the following steps: uint8 /
        bool [B, N] on the device, non-zero = candidate node; after the propagation the belief of node j is multiplied by
        0.1 + 0.9 * hint[j] and renormalised (an all-zero row leaves the env's belief as it is).  None switches it off."""
        if hint is not None:
            if not self.belief_on:
                raise _cabi.SyError("belief hints need belief=True")
            hint = hint.to(device=self.device).contiguous()
            if hint.dtype == torch.bool:
                hint = hint.view(torch.uint8)
            if hint.dtype != torch.uint8 or tuple(hint.shape) != (self.num_envs, self.graph_nodes):
                raise ValueError(f"hint must be uint8/bool [{self.num_envs}, {self.graph_nodes}]")
        self._belief_hint = hint  # keeps the buffer alive
        self._state.belief_hint = _ptr(hint)

    def set_seed(self, seed: int):
        """New Philox key (its low 64 bits; -1 is 2^64 - 1) for every later draw: start nodes and graphs of (auto-)resets,
        reveal skips and the random actions.  Rollout graphs captured before refuse to replay."""
        self.seed = int(seed)
        self.config.seed = self.seed & 0xFFFFFFFFFFFFFFFF
        _cabi.check(self._lib.sy_set_seed(self._handle, self.config.seed))

    # ------------------------------------------------------------------ reference API, batched
    def reset(self, reset_mask=None, init_pos=None, graph_id=None, restart: Optional[bool] = None, episode=0,
              seed=None, options=None):
        """yard.py:80-142 for the envs selected by `reset_mask` ([B] bool; None = all).
        `init_pos` [B, A] / `graph_id` [B] hand over explicit start nodes / graphs (parity
        harness); otherwise Philox(seed; env, episode).  Returns the observation dict."""
        B, A = self.num_envs, self.num_agents
        if seed is not None:  # the reference ignores `seed` (yard.py:80); here it re-keys Philox
            self.set_seed(seed)
            restart = True if restart is None else restart
        m = None if reset_mask is None else self._dev(reset_mask, torch.uint8, (B,))
        ip = None if init_pos is None else self._dev(init_pos, torch.int32, (B, A))
        gi = None if graph_id is None else self._dev(graph_id, torch.int32, (B,))
        if gi is not None and (int(gi.min()) < 0 or int(gi.max()) >= self.num_graphs):
            raise ValueError("graph_id out of range")
        if ip is not None:
            # (agents beyond a mechanism group's police count are absent: their entries are ignored)
            live = ip if self._env_police is None else \
                ip[torch.arange(A, device=self.device).view(1, -1) <= self._env_police]
            if live.numel() and (int(live.min()) < 0 or int(live.max()) >= self.graph_nodes):
                raise ValueError("init_pos out of range")
        if restart is None:
            restart = not self._is_reset
        if not self._is_reset and m is not None:
            raise _cabi.SyError("the first reset must cover every env")
        if self._need_full_reset and m is not None and not bool(m.all()):
            raise _cabi.SyError("the first reset after set_mechanisms must cover every env")
        if gi is None and not self._is_reset and not self.config.resample_graph:
            # blocks of 32 consecutive envs share a graph: the kernels' 32-env tiles then stay on the single-graph fast
            # paths (shared-memory CSR, lane = env belief propagation) for pools of up to B / 32 graphs
            gi = (torch.arange(B, device=self.device, dtype=torch.int64) + self.env_offset).div(GRAPH_BLOCK, rounding_mode="floor") \
                .remainder(self.num_graphs).to(torch.int32)
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_reset(self._handle, _ptr(m), _ptr(ip), _ptr(gi), int(bool(restart)),
                                           C.byref(self._state), C.byref(self._obs), self._stream()))
        self._is_reset = True
        self._need_full_reset = False
        self._keep = (m, ip, gi)  # keep inputs alive until the stream has consumed them
        return self.observation()

    def step(self, actions):
        """yard.py:144-269 for the whole batch.  `actions`: int64 [B, A] (device tensor preferred),
        -1 = DEFAULT_ACTION/None.  Returns (obs, reward f32[B,A], terminated, truncated bool[B,A], info)."""
        if not self._is_reset:
            raise _cabi.SyError("step() before reset()")
        a = actions
        if not (isinstance(a, torch.Tensor) and a.device == self.device and a.dtype in (torch.int64, torch.int32, torch.int16)
                and a.is_contiguous() and tuple(a.shape) == (self.num_envs, self.num_agents)):
            a = self._dev(actions, torch.int64, (self.num_envs, self.num_agents))
        fn = {torch.int64: self._lib.sy_step, torch.int32: self._lib.sy_step_i32,
              torch.int16: self._lib.sy_step_i16}[a.dtype]  # int32 / int16: narrow wire formats
        with torch.cuda.device(self.device):
            _cabi.check(fn(self._handle, a.data_ptr(), C.byref(self._state), C.byref(self._obs), C.byref(self._out),
                           self._stream()))
        self._last_actions = a
        info = {"winner": self.winner, "done": self.done_flags}
        return self.observation(), self.reward, self.terminated, self.truncated, info

    def step_deferred(self, actions):
        """Software-pipelined `step` for policies that read only the compact state (`pos`, `money`, `agent_budget`,
        `mrx_revealed`): the dynamics of yard.py:144-269 exactly as `step` (state, reward, flags are those of the new
        state), while `action_mask` / `node_features` / `belief_map` of the new state are left pending and written by
        the NEXT `step_deferred` in the same launch as its dynamics (sy_step_deferred).  After the call the dense
        tensors describe the state before it; `flush_observations()` (or `step` / `reset`) brings them up to date.
        Returns (reward, terminated, truncated, info)."""
        if not self._is_reset:
            raise _cabi.SyError("step() before reset()")
        a = actions
        if not (isinstance(a, torch.Tensor) and a.device == self.device and a.dtype == torch.int64 and a.is_contiguous()
                and tuple(a.shape) == (self.num_envs, self.num_agents)):
            a = self._dev(actions, torch.int64, (self.num_envs, self.num_agents))
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_step_deferred(self._handle, a.data_ptr(), C.byref(self._state), C.byref(self._obs),
                                                   C.byref(self._out), self._stream()))
        self._last_actions = a
        return self.reward, self.terminated, self.truncated, {"winner": self.winner, "done": self.done_flags}

    def flush_observations(self):
        """Write the dense observations a `step_deferred` left pending (no-op when none are); returns the observation."""
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_flush_observations(self._handle, C.byref(self._state), C.byref(self._obs), self._stream()))
        return self.observation()

    @property
    def observations_pending(self) -> bool:
        return bool(self._lib.sy_observations_pending(self._handle))

    # ------------------------------------------------------------------ mechanism groups
    def set_mechanisms(self, mechanisms, group_id=None):
        """Evaluate several mechanisms in this one batch (sy_set_groups).  `mechanisms`: a sequence of dicts with the
        optional keys `reward_weights` (a dict keyed by REWARD_WEIGHT_NAMES, floats or 0-dim tensors; missing names keep
        the constructor's weight), `agent_money`, `reveal_interval`, `reveal_skip_prob`, `tolls`, `number_of_agents` and
        `max_timestep` (a missing key keeps the constructor's value).  `number_of_agents` is the group's number of POLICE
        in [1, number_of_agents] -- the reference trainer's `num_police_agents: k` (agent_configurations) plays k + 1
        police, so that entry is `number_of_agents=k + 1` -- and `max_timestep` its horizon in [0, max_timestep].  An env
        of a group with fewer police keeps the [B, A] layout; its agents past the group's police are absent (pos -1,
        budget 0, reward 0, all-zero mask row and node_features column, sampled action -1; include/sy_env.h, SyState).
        `group_id`: int tensor [B] (env -> index into `mechanisms`), or None for
        (env_offset + b) % len(mechanisms).  `mechanisms=None` clears the groups.  Pending observations are flushed
        first; the new mechanisms take effect at the next full `reset()`, which `step` and the rollouts require."""
        self.flush_observations()
        if mechanisms is None:
            table, tolls, rules, gid = [], [], [], None
        else:
            table = [pack_mechanism(m, self) for m in mechanisms]
            tolls = [mechanism_toll(m, self) for m in mechanisms]
            rules = [mechanism_rules(m, self) for m in mechanisms]
            if not 1 <= len(table) <= _cabi.SY_MAX_GROUPS:
                raise ValueError(f"between 1 and {_cabi.SY_MAX_GROUPS} mechanisms, got {len(table)}")
            gid = None if group_id is None else self._dev(group_id, torch.int32, (self.num_envs,))
        arr = (_cabi.SyGroup * max(len(table), 1))(*table)
        own_tolls = any(t != self.tolls for t in tolls)
        police, horizon = [r[0] for r in rules], [r[1] for r in rules]
        own_police = any(n != self.number_of_agents for n in police)
        own_rules = own_police or any(t != self.config.max_timestep for t in horizon)
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_set_groups(self._handle, len(table), arr, _ptr(gid), self._stream()))
            if own_tolls:  # (sy_set_groups gave every group the constructor's toll, police count and horizon)
                _cabi.check(self._lib.sy_set_group_tolls(self._handle, len(tolls), (C.c_int32 * len(tolls))(*tolls),
                                                         self._stream()))
            if own_rules:
                _cabi.check(self._lib.sy_set_group_rules(self._handle, len(rules), (C.c_int32 * len(rules))(*police),
                                                         (C.c_int32 * len(rules))(*horizon), self._stream()))
        self._mechanisms = None if mechanisms is None else tuple(
            unpack_mechanism(g, t, r) for g, t, r in zip(table, tolls, rules))
        self._group_id, self._env_toll, self._env_police = None, None, None
        if table:
            self._group_id = gid.clone() if gid is not None else (
                (torch.arange(self.num_envs, device=self.device, dtype=torch.int64) + self.env_offset) % len(table)).to(torch.int32)
            if own_tolls:  # int32 [B, 1] toll of each env (the policies' legality test, see policy._PolicyBase._state)
                self._env_toll = torch.tensor(tolls, dtype=torch.int32, device=self.device)[self._group_id.long()].view(-1, 1)
            if own_police:  # int32 [B, 1] police count of each env (init_pos checks, the policies' refusal)
                self._env_police = torch.tensor(police, dtype=torch.int32, device=self.device)[self._group_id.long()].view(-1, 1)
        self.group_stats_vec = torch.zeros(len(table), _cabi.SY_NUM_STATS, dtype=torch.int64, device=self.device) \
            if table and self.stats_vec is not None else None
        self._need_full_reset = True  # the next reset() covers every env
        self._groups_generation += 1

    @property
    def mechanisms(self):
        """The mechanism groups as set (tuple of complete dicts), or None"""
        return self._mechanisms

    @property
    def group_id(self) -> Optional[torch.Tensor]:
        """int32 [B] group of each env while mechanism groups are set (a copy), else None"""
        return None if self._group_id is None else self._group_id.clone()

    def sample_actions(self, out: Optional[torch.Tensor] = None, step_counter: Optional[int] = None) -> torch.Tensor:
        """Uniform random valid action per agent on the device (-1 when an agent cannot move)."""
        if out is None:
            out = torch.empty(self.num_envs, self.num_agents, dtype=torch.int64, device=self.device)
        if step_counter is None:
            step_counter = self._sample_counter
            self._sample_counter += 1
        fn = {torch.int64: self._lib.sy_sample_actions, torch.int32: self._lib.sy_sample_actions_i32,
              torch.int16: self._lib.sy_sample_actions_i16}[out.dtype]
        with torch.cuda.device(self.device):
            _cabi.check(fn(self._handle, C.byref(self._state), int(step_counter) & 0xFFFFFFFF, out.data_ptr(), self._stream()))
        return out

    def rollout_random(self, num_steps: int, actions: Optional[torch.Tensor] = None,
                       step_counter: Optional[int] = None) -> torch.Tensor:
        """`num_steps` steps of the on-device random-valid policy (the RandomAgent baseline of the reference,
        src/agent/random_agent.py:7), issued from C without returning to Python between steps.  Returns the
        actions of the last step; state / observations / results describe the last step."""
        if not self._is_reset:
            raise _cabi.SyError("step() before reset()")
        if actions is None:
            actions = torch.empty(self.num_envs, self.num_agents, dtype=torch.int64, device=self.device)
        if step_counter is None:
            step_counter = self._sample_counter
            self._sample_counter += int(num_steps)
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_rollout_random(self._handle, int(num_steps), int(step_counter) & 0xFFFFFFFF,
                                                    actions.data_ptr(), C.byref(self._state), C.byref(self._obs),
                                                    C.byref(self._out), self._stream()))
        return actions

    # ------------------------------------------------------------------ host-buffer API (the reference's call shape)
    def capture_rollout(self, num_steps: int, actions: Optional[torch.Tensor] = None):
        """A CUDA graph of `num_steps` random-policy steps whose step counter lives on the device, so every
        `graph.replay()` continues the rollout with fresh draws (sy_rollout_random_dev).  Small batches are
        launch-latency bound; replaying a graph removes most of that.  Returns (graph, counter tensor).  The captured
        launches assume that no observations are pending (what holds when this returns): call `flush_observations()`
        before a replay that follows `step_deferred`.  The graph keeps the Philox key and mechanism groups of its
        capture, so it refuses to replay after `set_seed` (a `reset(seed=...)` or a `load_state_dict` with another seed
        too) or `set_mechanisms`: capture it again."""
        if not self._is_reset:
            raise _cabi.SyError("step() before reset()")
        self.flush_observations()
        if actions is None:
            actions = torch.empty(self.num_envs, self.num_agents, dtype=torch.int64, device=self.device)
        counter = torch.tensor([self._sample_counter], dtype=torch.int32, device=self.device)  # read as uint32

        def issue():
            _cabi.check(self._lib.sy_rollout_random_dev(self._handle, int(num_steps), counter.data_ptr(), actions.data_ptr(),
                                                        C.byref(self._state), C.byref(self._obs), C.byref(self._out),
                                                        self._stream()))
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.device(self.device), torch.cuda.stream(side):
            issue()  # warm-up outside the capture (it advances the rollout like any other call)
        torch.cuda.current_stream(self.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.device(self.device), torch.cuda.graph(graph, stream=side):
            issue()
        self._rollout_graph_keepalive = (actions, counter)
        return _RolloutGraph(graph, self), counter

    def _host_buffers(self):
        if getattr(self, "_host", None) is None:
            B, A = self.num_envs, self.num_agents
            pin = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, pin_memory=True)  # noqa: E731
            self._host_block = pin(self._result_bytes(), dtype=torch.uint8)  # same layout as the device result block
            r, te, tr, dn, wn, st = self._result_views(self._host_block)
            self._host = dict(reward=r, terminated=te, truncated=tr, done=dn, winner=wn, status=st,
                              actions=pin(B, A, dtype=torch.int64), actions32=pin(B, A, dtype=torch.int32),
                              actions16=pin(B, A, dtype=torch.int16))
            self._actions_dev = torch.empty(B, A, dtype=torch.int64, device=self.device)
            self._actions_dev32 = torch.empty(B, A, dtype=torch.int32, device=self.device)
            self._actions_dev16 = torch.empty(B, A, dtype=torch.int16, device=self.device)
            self._host_out = _cabi.SyHostOut(*[self._host[k].data_ptr() for k in
                                               ("reward", "terminated", "truncated", "done", "winner", "status")])
            # compact form: the three [B, A] flag arrays stay on the device, one status byte per env travels instead
            self._host_out_compact = _cabi.SyHostOut(r.data_ptr(), None, None, None, wn.data_ptr(), st.data_ptr())
        return self._host

    def host_h2d_bytes_per_step(self, action_bytes: int = 8) -> int:
        return self.num_envs * self.num_agents * action_bytes

    def host_d2h_bytes_per_step(self, action_bytes: int = 8, flags: str = "per_agent") -> int:
        """step_host results (+ the sampled actions when sample_actions_host feeds it)"""
        B, A = self.num_envs, self.num_agents
        return B * A * 4 + (2 * B if flags == "compact" else 3 * B * A + 2 * B) + B * A * action_bytes

    def step_host(self, actions, flags: str = "per_agent") -> Dict[str, torch.Tensor]:
        """`step` with HOST buffers on both sides, as the reference's env is called (python ints in,
        numpy/python values out, yard.py:144,269): actions int64 / int32 / int16 [B, A] in host memory
        (pinned is fastest; the dtype is the wire format) -> H2D -> kernel -> D2H of reward / terminated /
        truncated / done / winner / status into pinned host tensors; synchronous.  Observations stay on the
        device (`observation()`).  flags="compact": only reward, winner and the status byte per env travel
        (bit 0 terminated, bit 1 truncated, bit 2 frozen; all agents of an env share them) -- 3A - 1 fewer
        bytes per env over PCIe; `expand_status` rebuilds the per-agent arrays on the host when needed."""
        if not self._is_reset:
            raise _cabi.SyError("step() before reset()")
        host = self._host_buffers()
        a = torch.as_tensor(actions)
        if a.is_cuda or a.dtype not in (torch.int64, torch.int32, torch.int16) or not a.is_contiguous() or \
                tuple(a.shape) != (self.num_envs, self.num_agents):
            a = torch.as_tensor(np.asarray(a.cpu() if a.is_cuda else a), dtype=torch.int64).contiguous()
            if tuple(a.shape) != (self.num_envs, self.num_agents):
                raise ValueError(f"expected shape {(self.num_envs, self.num_agents)}, got {tuple(a.shape)}")
        fn, stage = {torch.int64: (self._lib.sy_step_host, self._actions_dev),
                     torch.int32: (self._lib.sy_step_host_i32, self._actions_dev32),
                     torch.int16: (self._lib.sy_step_host_i16, self._actions_dev16)}[a.dtype]
        if flags not in ("per_agent", "compact"):
            raise ValueError("flags must be 'per_agent' or 'compact'")
        compact = flags == "compact"
        with torch.cuda.device(self.device):
            _cabi.check(fn(self._handle, a.data_ptr(), stage.data_ptr(), C.byref(self._state), C.byref(self._obs),
                           C.byref(self._out), C.byref(self._host_out_compact if compact else self._host_out), self._stream()))
        keys = ("reward", "winner", "status") if compact else ("reward", "terminated", "truncated", "done", "winner", "status")
        return {k: host[k] for k in keys}

    def host_rollout_random(self, num_steps: int, step_counter: Optional[int] = None, dtype=torch.int16,
                            flags: str = "compact") -> Dict[str, torch.Tensor]:
        """`num_steps` iterations of `step_host(sample_actions_host())` issued from C (sy_host_rollout_random): the
        host-buffer loop with all of its per-step copies and synchronisations, without the interpreter between the calls.
        Returns the pinned host results of the last step."""
        if not self._is_reset:
            raise _cabi.SyError("step() before reset()")
        host = self._host_buffers()
        key, stage = {torch.int64: ("actions", self._actions_dev), torch.int32: ("actions32", self._actions_dev32),
                      torch.int16: ("actions16", self._actions_dev16)}[dtype]
        if step_counter is None:
            step_counter = self._sample_counter
            self._sample_counter += int(num_steps)
        compact = flags == "compact"
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_host_rollout_random(
                self._handle, int(num_steps), int(step_counter) & 0xFFFFFFFF, stage.data_ptr(), host[key].data_ptr(),
                stage.element_size(), C.byref(self._state), C.byref(self._obs), C.byref(self._out),
                C.byref(self._host_out_compact if compact else self._host_out), self._stream()))
        keys = ("reward", "winner", "status") if compact else ("reward", "terminated", "truncated", "done", "winner", "status")
        return {k: host[k] for k in keys}

    def set_host_overlap(self, on: bool = True):
        """Host loops with overlap: `step_host` then returns as soon as the step's results are in the pinned host
        tensors -- the observation kernel of that step may still be running on the stream (any later stream work,
        incl. reading the observation tensors with torch on this stream, is ordered after it) -- and
        `sample_actions_host` runs on a library stream next to it.  Off by default (fully synchronous calls)."""
        _cabi.check(self._lib.sy_set_host_overlap(self._handle, int(bool(on))))

    def expand_status(self, status: torch.Tensor) -> Dict[str, torch.Tensor]:
        """per-agent bool [B, A] views of a status byte vector (what the reference's per-agent dicts hold)"""
        A = self.num_agents
        te, tr = (status & 1).bool(), (status & 2).bool()
        dn = status != 0
        return {"terminated": te[:, None].expand(-1, A), "truncated": tr[:, None].expand(-1, A), "done": dn[:, None].expand(-1, A)}

    def sample_actions_host(self, step_counter: Optional[int] = None, dtype=torch.int64) -> torch.Tensor:
        """random valid actions delivered in pinned HOST memory (stands in for a host-side policy)"""
        host = self._host_buffers()
        key, stage = {torch.int64: ("actions", self._actions_dev), torch.int32: ("actions32", self._actions_dev32),
                      torch.int16: ("actions16", self._actions_dev16)}[dtype]
        if step_counter is None:
            step_counter = self._sample_counter
            self._sample_counter += 1
        with torch.cuda.device(self.device):  # kernel + D2H + synchronise in one C call
            _cabi.check(self._lib.sy_sample_actions_host(self._handle, C.byref(self._state), int(step_counter) & 0xFFFFFFFF,
                                                         stage.data_ptr(), host[key].data_ptr(), stage.element_size(), self._stream()))
        return host[key]

    # ------------------------------------------------------------------ device graph pool (SURVEY 8(f) f3)
    def _generate_on_device(self, generation: int):
        """sy_generate_graphs + read the edge lists back (the host keeps GraphSpec views for the static observation
        tensors, exactly what the reference's `env.board` holds)."""
        N, G = self.graph_nodes, self.num_graphs
        want_e = N - 1 if self.graph_edges is None else int(self.graph_edges)
        max_e = min(max(want_e, N - 1), N * (N - 1) // 2)
        attempts = np.zeros(G, dtype=np.int32)
        _cabi.check(self._lib.sy_generate_graphs(self._handle, G, want_e, self._gen["cap"], self._gen["max_weight"],
                                                 self.seed & 0xFFFFFFFFFFFFFFFF, int(generation), self._gen["graph_offset"],
                                                 attempts.ctypes.data, self._stream()))
        links = np.zeros((G, max_e, 2), dtype=np.int32)
        weights = np.zeros((G, max_e), dtype=np.int32)
        counts = np.zeros(G, dtype=np.int32)
        _cabi.check(self._lib.sy_read_graph_edges(self._handle, links.ctypes.data, weights.ctypes.data, counts.ctypes.data,
                                                  max_e, self._stream()))
        self.graphs = [GraphSpec(N, links[g, : counts[g]], weights[g, : counts[g]]) for g in range(G)]
        self.actual_num_edges = int(counts[0])
        self.generation_attempts = attempts
        self._gen["generation"] = int(generation)
        row_ptr, col, wgt, _ = pack_csr(self.graphs)
        self._csr = (row_ptr, col, wgt)
        self._static = None

    def regenerate_graphs(self, generation: Optional[int] = None):
        """Refresh a device-sampled pool with a new generation of graphs (the reference draws a new graph on every
        reset, yard.py:87-101; here the whole pool is redrawn between rollouts).  Every env must be reset afterwards."""
        if not self._device_pool:
            raise _cabi.SyError("regenerate_graphs needs graphs='device'")
        with torch.cuda.device(self.device):
            self._generate_on_device(self._gen["generation"] + 1 if generation is None else int(generation))
        self._is_reset = False

    # ------------------------------------------------------------------ observations
    def _static_tensors(self):
        if self._static is None:
            N, G = self.graph_nodes, self.num_graphs
            row_ptr, col, wgt = self._csr
            adj = torch.zeros(G, N, N, dtype=torch.float32)
            for g in range(G):
                deg = np.diff(row_ptr[g])
                rows = np.repeat(np.arange(N), deg)
                adj[g, torch.from_numpy(rows), torch.from_numpy(col[g, : row_ptr[g, -1]].astype(np.int64))] = 1.0
            same_e = all(len(g.edges) == self.actual_num_edges for g in self.graphs)
            if same_e:
                ei = torch.from_numpy(np.stack([g.edge_links.T for g in self.graphs]).astype(np.int64))  # [G,2,E]
                ef = torch.from_numpy(np.stack([g.edges for g in self.graphs]).astype(np.int64))  # [G,E]
            else:
                ei = ef = None
            self._static = (adj.to(self.device), None if ei is None else ei.to(self.device),
                            None if ef is None else ef.to(self.device))
        return self._static

    def observation(self) -> Dict[str, torch.Tensor]:
        """yard.py:319-332 keys with a leading batch dim.  Static graph tensors are stride-0 /
        gathered views of one copy per graph; dynamic ones are the buffers the kernel wrote."""
        adj, ei, ef = self._static_tensors()
        B = self.num_envs
        if self.num_graphs == 1:
            adjacency = adj.expand(B, -1, -1)
            edge_index = None if ei is None else ei.expand(B, -1, -1)
            edge_features = None if ef is None else ef.expand(B, -1)
        else:
            gid = self.graph_id.long()
            adjacency = _LazyGather(adj, gid)
            edge_index = None if ei is None else _LazyGather(ei, gid)
            edge_features = None if ef is None else _LazyGather(ef, gid)
        obs = {
            "adjacency_matrix": adjacency,
            "node_features": self.node_features,
            "edge_index": edge_index,
            "edge_features": edge_features,
            "action_mask": self.action_mask,
            "agent_position": self.pos,
            "agent_budget": self.agent_budget.unsqueeze(-1),
            "MrX_pos": self.pos[:, 0],
            "Polices_pos": self.pos[:, 1:],
            "Currency": self.money[:, 1:],
            "MrX_revealed": self.mrx_revealed,
            "graph_id": self.graph_id,
        }
        if self.belief_on:
            obs["belief_map"] = self.belief_map
        return obs

    # ------------------------------------------------------------------ helpers callers use
    def action_space_n(self) -> int:
        return self.graph_nodes  # Discrete(num_nodes), yard.py:482-498

    def get_possible_moves(self, agent_idx: int, env_index: int = 0) -> np.ndarray:
        """yard.py:474-480 as a view of the action mask."""
        return torch.nonzero(self.action_mask[env_index, agent_idx]).flatten().to(torch.int32).cpu().numpy()

    def graph_tables(self, g: int = 0):
        """(weights u8[N,N], apsp u16[N,N]) of graph g copied to the host (get_distance parity)."""
        N = self.graph_nodes
        W = np.zeros((N, N), dtype=np.uint8)
        D = np.zeros((N, N), dtype=np.uint16)
        with torch.cuda.device(self.device):
            _cabi.check(self._lib.sy_read_graph_tables(self._handle, int(g), W.ctypes.data, D.ctypes.data, self._stream()))
        return W, D

    def get_distance(self, node1: int, node2: int, g: int = 0) -> float:
        """yard.py:375-388 / pathfinding.py:34-137 from the device-built table."""
        d = int(self.graph_tables(g)[1][node1, node2])
        return float("inf") if d == 0xFFFF else float(d)

    def stats(self, reduce_group=None, by_group: bool = False):
        """Episode statistics accumulated on the device; with `reduce_group` (or an initialised
        default process group and reduce_group=True) they are summed over ranks with one
        all-reduce (NCCL over NVLink on a GPU box).  by_group=True: one dict per mechanism group."""
        if self.stats_vec is None:
            raise _cabi.SyError("collect_stats=False")
        self._fold_stats()
        if by_group:
            if self.group_stats_vec is None:
                raise _cabi.SyError("no mechanism groups are set")
            t = self.group_stats_vec
            if reduce_group is not None:
                import torch.distributed as dist

                t = t.clone()
                dist.all_reduce(t, group=None if reduce_group is True else reduce_group)
            return [{k: int(row[i]) for i, k in enumerate(_cabi.STAT_NAMES)} for row in t.cpu().tolist()]
        if reduce_group is not None:
            from .sharding import allreduce_stats

            return allreduce_stats(self.stats_vec, None if reduce_group is True else reduce_group)
        h = self.stats_vec.cpu().tolist()
        return {k: int(h[i]) for i, k in enumerate(_cabi.STAT_NAMES)}

    def metrics(self, reduce_group=None, by_group: bool = False):
        """The aggregates of the reference's MetricsTracker.get_aggregated_metrics (src/eval/metrics.py:168-232) from
        the device statistics vector -- same keys.  `mean_belief_ce` / `belief_ce_std` (metrics.py:194-197,217-218):
        cross-entropy of the predicted belief at MrX's node over all reveal steps (belief_quality.py:8-11), scored
        inside the observe kernel before the reveal collapses the map.  by_group=True: one dict per mechanism group
        (its budget efficiency against its own agent_money).  While groups are set, the aggregate efficiency weighs
        every group's spending against that group's budget."""
        if by_group:
            return group_metrics(self.stats(reduce_group, by_group=True), self._mechanisms, self.number_of_agents)[2]
        st = self.stats(reduce_group)
        eff, paid = None, self.tolls * st["police_moves"]
        if self._mechanisms is not None and self.group_stats_vec is not None:
            eff, paid, _ = group_metrics(self.stats(reduce_group, by_group=True), self._mechanisms, self.number_of_agents)
        return metrics_of(st, initial=max(self.number_of_agents * self.agent_money, 1), tolls_paid=paid, eff_sum=eff)

    def _fold_stats(self):
        """sy_stats: add what the kernels accumulated since the last call to `stats_vec`"""
        if self.stats_vec is not None:
            with torch.cuda.device(self.device):
                _cabi.check(self._lib.sy_stats(self._handle, self.stats_vec.data_ptr(), self._stream()))
                if self.group_stats_vec is not None:
                    _cabi.check(self._lib.sy_group_stats(self._handle, self.group_stats_vec.shape[0],
                                                         self.group_stats_vec.data_ptr(), self._stream()))

    def reset_stats(self):
        if self.stats_vec is not None:
            self._fold_stats()
            self.stats_vec.zero_()
            if self.group_stats_vec is not None:
                self.group_stats_vec.zero_()

    _STATE_TENSORS = ("pos", "money", "timestep", "graph_id", "episode", "done", "visits", "belief_map", "action_mask",
                      "node_features", "agent_budget", "mrx_revealed", "stats_vec", "group_stats_vec")
    _STATE_SCALARS = ("seed", "sample_counter", "env_offset", "graph_pool_sha256")

    def _state_keys(self):
        keys = {k for k in self._STATE_TENSORS if getattr(self, k) is not None} | set(self._STATE_SCALARS)
        return keys | ({"group_id"} if self._group_id is not None else set())

    def _graph_pool_digest(self) -> torch.Tensor:
        """uint8 [32]: SHA-256 over every pool graph's node count, edge links and edge weights"""
        h = hashlib.sha256()
        for g in self.graphs:
            links, weights = np.asarray(g.edge_links, dtype=np.int64), np.asarray(g.edges, dtype=np.int64)
            h.update(np.asarray([g.num_nodes, len(weights)], dtype=np.int64).tobytes())
            h.update(np.ascontiguousarray(links).tobytes())
            h.update(np.ascontiguousarray(weights).tobytes())
        return torch.frombuffer(bytearray(h.digest()), dtype=torch.uint8)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """A checkpoint of the batch: clones of the state, the dense observations (the belief map included), the
        statistics (folded first; per group and the group assignment while mechanism groups are set), and as CPU int64
        tensors the Philox key (`seed`, the int64 view of its 64 bits), the sampler counter of `sample_actions` /
        `rollout_random` / `HeuristicPolicy.act`, `env_offset`, and `graph_pool_sha256` (uint8 [32], a digest of the
        pool).  Pending observations of `step_deferred` are flushed first, so the dict describes the current state.
        Callers' own counters (policy step counters, the counter tensor of `capture_rollout`, `HeuristicPolicy.last_seen`)
        are not in it.  `torch.save` / `torch.load` round-trip it."""
        self.flush_observations()
        self._fold_stats()
        sd = {k: getattr(self, k).clone() for k in self._STATE_TENSORS if getattr(self, k) is not None}
        if self._group_id is not None:  # mechanism groups: the assignment
            sd["group_id"] = self._group_id.clone()
        seed = self.config.seed
        sd["seed"] = torch.tensor(seed - (1 << 64) if seed >= 1 << 63 else seed, dtype=torch.int64)
        sd["sample_counter"] = torch.tensor(self._sample_counter, dtype=torch.int64)
        sd["env_offset"] = torch.tensor(self.env_offset, dtype=torch.int64)
        sd["graph_pool_sha256"] = self._graph_pool_digest()
        return sd

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        """Restore a `state_dict`: the state, observations and statistics, the Philox key (`set_seed`) and the sampler
        counter, so that the batch continues exactly as the one that was saved.  Raises ValueError, before anything is
        changed, when the dict comes from a handle with another `env_offset`, graph pool, batch size, node or agent
        count, node-feature type, or set of keys (belief map, statistics, mechanism groups on in one and off in the
        other).  Pending observations are flushed and the library's statistics accumulators folded and discarded first,
        so rewinding a handle to an earlier dict counts the replayed steps once.
        One taken while mechanism groups were set needs the same groups set first (with `set_mechanisms`).  In the same
        handle it then resumes mid-episode; in another handle, mechanism groups cannot be resumed mid-episode: after
        `set_mechanisms` the library requires a full `reset()` before the next step, which starts new episodes -- what
        carries over is the statistics, the per-group ones included."""
        want = self._state_keys()
        if set(sd) != want:
            raise ValueError(f"the state dict's keys differ from this env's: missing {sorted(want - set(sd))}, "
                             f"unexpected {sorted(set(sd) - want)}")
        if int(sd["env_offset"]) != self.env_offset:
            raise ValueError(f"the state dict was taken at env_offset {int(sd['env_offset'])}, this env has {self.env_offset}")
        if not torch.equal(sd["graph_pool_sha256"].cpu(), self._graph_pool_digest()):
            raise ValueError("the state dict was taken on another graph pool")
        if "group_id" in sd and not torch.equal(sd["group_id"].to(self._group_id.device), self._group_id):
            raise ValueError("the state dict's mechanism groups differ from this env's: set_mechanisms() first")
        for k in want & set(self._STATE_TENSORS):
            mine = getattr(self, k)
            if tuple(sd[k].shape) != tuple(mine.shape) or sd[k].dtype != mine.dtype:
                raise ValueError(f"state dict entry {k!r} is {sd[k].dtype} {tuple(sd[k].shape)}, this env has "
                                 f"{mine.dtype} {tuple(mine.shape)}")
        self.flush_observations()
        self._fold_stats()  # what the kernels accumulated since the last fold belongs to the state being replaced
        for k in want & set(self._STATE_TENSORS):
            getattr(self, k).copy_(sd[k])
        self.set_seed(int(sd["seed"]) & 0xFFFFFFFFFFFFFFFF)
        self._sample_counter = int(sd["sample_counter"])
        self._is_reset = True


class _RolloutGraph:
    """A captured rollout graph (torch.cuda.CUDAGraph) that refuses to replay once the env's mechanism groups or its
    seed changed: its launches carry the groups -- and the kernels chosen for them -- and the Philox key of the time it
    was captured."""

    def __init__(self, graph, env):
        self.graph, self._env, self._generation, self._seed = graph, env, env._groups_generation, env.config.seed

    def replay(self):
        if self._env._groups_generation != self._generation:
            raise _cabi.SyError("the mechanism groups changed since this rollout graph was captured: capture it again")
        if self._env.config.seed != self._seed:
            raise _cabi.SyError("the seed changed since this rollout graph was captured: capture it again")
        self.graph.replay()

    def __getattr__(self, name):
        return getattr(self.graph, name)


class _LazyGather:
    """Per-env view of a per-graph tensor, materialised only when a caller indexes it."""

    def __init__(self, table: torch.Tensor, gid: torch.Tensor):
        self.table, self.gid = table, gid
        self.shape = (gid.shape[0],) + tuple(table.shape[1:])

    def __getitem__(self, idx):
        if isinstance(idx, tuple):
            return self.table[self.gid[idx[0]]][(slice(None),) + idx[1:]] if not isinstance(idx[0], int) else \
                self.table[self.gid[idx[0]]][idx[1:]]
        return self.table[self.gid[idx]]

    def materialize(self) -> torch.Tensor:
        return self.table[self.gid]


def dense_action_mask(adjacency, current_node, budget, tolls=None, edge_weights=None, device="cuda:0") -> torch.Tensor:
    """Batched drop-in for compute_action_mask (action_mask.py:30-83) on dense float64 inputs.
    `current_node` [Q], `budget` [Q]; tolls: None | scalar | [N] per destination | [N,N]."""
    lib = _cabi.load_library()
    dev = torch.device(device)
    adj = torch.as_tensor(np.asarray(adjacency), dtype=torch.float64, device=dev).contiguous()
    N = adj.shape[0]
    w = None if edge_weights is None else torch.as_tensor(np.asarray(edge_weights, dtype=float), dtype=torch.float64, device=dev).contiguous()
    toll_s, toll_m = 0.0, None
    if tolls is not None:
        if np.isscalar(tolls):
            toll_s = float(tolls)
        else:
            t = np.asarray(tolls, dtype=float)
            if t.ndim == 1:
                t = np.tile(t.reshape(1, -1), (N, 1))  # action_mask.py:92-95
            toll_m = torch.as_tensor(t, dtype=torch.float64, device=dev).contiguous()
    cur = torch.as_tensor(np.atleast_1d(current_node), dtype=torch.int32, device=dev).contiguous()
    bud = torch.as_tensor(np.atleast_1d(budget), dtype=torch.float64, device=dev).contiguous()
    out = torch.zeros(cur.shape[0], N, dtype=torch.bool, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(lib.sy_action_mask_dense(cur.shape[0], N, adj.data_ptr(), _ptr(w), _ptr(toll_m), toll_s,
                                             cur.data_ptr(), bud.data_ptr(), out.data_ptr(),
                                             torch.cuda.current_stream(dev).cuda_stream))
    return out
