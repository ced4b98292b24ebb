#!/usr/bin/env python
"""Benchmark of the batched Scotland Yard env hot path (BASELINE.json metric: batched env-steps/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port on the host cores
    python bench.py ... --dump-outputs DIR                    # + what the last timed step computed, as DIR/*.npy

One "step" = one pass of the hot path over the rank's whole batch: the on-device random-valid
policy (`sy_sample_actions`) + `sy_step` (dynamics, budgets/tolls, capture/termination, rewards,
reveal schedule, belief propagation, observation assembly, same-step auto-reset).  Workload at
N=1 is BASELINE config 3 (200 nodes, 6 police, budgets+tolls, belief on, 65 536 envs); with N
GPUs every rank holds its own 65 536 envs (weak scaling, batch sharded by env index, no data-path
collective; one NCCL all-reduce of the statistics vector closes the timed region).

Keys of the JSON line (see DESIGN.md "Measurement"): `value` = device-resident throughput;
`e2e` = the same metric through the host-buffer API (`step_host`: pinned host actions -> H2D ->
kernel -> D2H of rewards/flags, every step, synchronised); `roofline` = algorithmic bytes of
`sy_step_kernel` (SURVEY.md 8(d): 8849 B/env-step at c3) / its CUDA-event duration / measured HBM
peak; `cpu_baseline` = the CPU oracle port timed on this box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: N, E, P, money, toll, belief, reveal, B per GPU
    "c2": dict(N=50, E=110, P=3, money=10, toll=0, belief=False, reveal=5, B=1024,
               desc="50-node graph, 3 police, reveal every 5 steps, 1024 envs, random policy"),
    "c3": dict(N=200, E=400, P=6, money=20, toll=1, belief=True, reveal=5, B=65536,
               desc="200-node graph, 6 police, budgets+tolls, 65536 envs per GPU, belief_map on, reveal every 5"),
    "c4": dict(N=1000, E=2000, P=6, money=20, toll=1, belief=True, reveal=5, B=32768,
               desc="1000-node synthetic random graph, 6 police, 32768 envs per GPU (262144 over 8)"),
    # BASELINE config 5: the policy forward of the reference's agents in the loop (--policy gnn | mappo, default gnn)
    "c5": dict(N=200, E=400, P=6, money=20, toll=1, belief=True, reveal=5, B=131072, policy="gnn",
               desc="GNN/MAPPO policy rollout, 200-node graph, 6 police, 131072 envs per GPU (1M over 8), belief_map on"),
}
METRIC, UNIT = "batched_env_steps_per_sec", "env-steps/s"


def algorithmic_bytes_per_env_step(N, P, belief, nf_bytes=4):
    """SURVEY.md section 8(d): actions R + pos/money/t R+W + visit RMW + belief R+W + reward/flags W
    + action_mask W + node_features W (static graph tables are L2-resident and excluded)."""
    A = P + 1
    return 8 * A + 2 * (4 * A + 4 * A + 4) + 2 * 2 * P + (2 * 4 * N if belief else 0) + 4 * A + 3 * A + A * N + nf_bytes * N * A


def kernel_source_hash():
    import hashlib

    with open(os.path.join(ROOT, "student_mechanism_design_b200", "csrc", "sy_env.cu"), "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi/NVML clocks + throttle reasons sampled DURING the timed regions."""

    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.reasons, self.active, self.stop = [], set(), False, False
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        while not self.stop:
            if self.nv is not None and self.active:
                try:
                    self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    get = getattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                        self.nv.nvmlDeviceGetCurrentClocksThrottleReasons
                    r = get(self.h)
                    for bit, name in self.BITS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.01)

    def summary(self):
        self.stop = True
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


DUMP_BYTES = 48 << 20  # per-env arrays of --dump-outputs: one sample of envs, sized to stay under 64 MB in all


def dump_outputs(out_dir, env, actions, stats):
    """`--dump-outputs DIR`: what the timed path hands its caller after its last step, as DIR/<name>.npy, so that two
    builds run with the same arguments can be compared output for output.  Per-env arrays (the policy's actions, the
    step's reward and flags, the dynamic observation entries) are float32 rows of a fixed, seeded sample of envs whose
    indices are `env_index`; `episode_stats` (float64, named by STAT_NAMES) covers the whole batch."""
    import numpy as np
    import torch

    from student_mechanism_design_b200._cabi import STAT_NAMES

    obs = env.observation()
    per_env = {"actions": actions, "reward": env.reward, "terminated": env.terminated, "truncated": env.truncated,
               "done": env.done_flags, "winner": env.winner}
    for k in ("agent_position", "Currency", "agent_budget", "MrX_revealed", "graph_id", "action_mask", "node_features",
              "belief_map"):
        if k in obs:
            per_env[k] = obs[k]
    B = env.num_envs
    n = min(B, DUMP_BYTES // sum(4 * t[0].numel() for t in per_env.values()))
    idx = np.sort(np.random.default_rng(0).choice(B, size=n, replace=False))
    sel = torch.from_numpy(idx).to(env.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in per_env.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.index_select(0, sel).float().cpu().numpy())
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "episode_stats.npy"), np.asarray([stats[k] for k in STAT_NAMES], dtype=np.float64))


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference itself is Python and does not travel to the GPU box)
# --------------------------------------------------------------------------------------------
class CpuRunner:
    """The CPU oracle on a bounded sample of the workload: the C restatement (oracle/sy_oracle.c,
    OpenMP over envs, all host threads) or, if gcc is unavailable, the numpy/Python one (1 core).
    One `step()` = random-valid policy + env step + masks + node features + belief for `B` envs."""

    def __init__(self, wl, all_cores=True, envs=None):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import sy_oracle as so

        from student_mechanism_design_b200.graphs import generate_graph_pool

        self.wl = wl
        pool = [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in generate_graph_pool(1, wl["N"], wl["E"], seed=0)]
        cfg = so.OracleConfig(num_police=wl["P"], agent_money=wl["money"], toll=wl["toll"], belief=wl["belief"],
                              reveal_interval=wl["reveal"])
        try:
            import sy_oracle_c as oc

            have_c = oc.available()
        except Exception:
            have_c = False
        self.n = 0
        if have_c:
            cores = (os.cpu_count() or 1) if all_cores else 1
            try:
                cores = min(cores, len(os.sched_getaffinity(0)))
            except Exception:
                pass
            # the workload's own batch (bounded at 65 536 envs: the large configs keep the host arrays to a few hundred MB)
            self.cores, self.B = cores, int(envs or min(wl["B"], 65536))
            self.run = oc.CBatch(cfg, pool, self.B, seed=0, threads=cores)
            self.what = f"C oracle (oracle/sy_oracle.c, OpenMP, {cores} threads)"
            self.step = self._step_c
        else:
            self.cores, self.B = 1, 64
            self.run = so.OracleBatch.from_seed(cfg, pool, self.B, seed=0)
            self.what = "numpy/Python oracle (oracle/sy_oracle.py)"
            self.step = self._step_py

    def _step_c(self):
        self.run.steps(1, first_step=self.n)
        self.n += 1

    def _step_py(self):
        self.run.step(self.run.sample_actions(self.n))
        self.run.masks(), self.run.node_features()
        self.n += 1

    def timed_passes(self, steps, warmup, min_seconds=2.0, max_seconds=150.0):
        """`warmup` untimed steps, then passes of exactly `steps` steps until `min_seconds` of timed work have been
        done (at most 5 passes, at most `max_seconds`); returns (median seconds per pass, passes)"""
        for _ in range(warmup):
            self.step()
        passes, total = [], 0.0
        while len(passes) < 5 and (not passes or total < min_seconds) and total < max_seconds:
            t0 = time.perf_counter()
            for _ in range(steps):
                self.step()
            passes.append(time.perf_counter() - t0)
            total += passes[-1]
        return statistics.median(passes), passes

    def timed(self, budget_s, max_steps=None):
        for _ in range(3):
            self.step()
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < budget_s and (max_steps is None or n < max_steps):
            self.step()
            n += 1
        dt = time.perf_counter() - t0
        return dict(value=self.B * n / dt, unit=UNIT, cores=self.cores, kind="port",
                    sample=f"{self.what}: {self.B} envs x {n} steps of {self.wl['name']} (random policy + step + masks + "
                           f"node features + belief), {dt:.1f} s"), dt, n


def run_reference_arm(args, wl):
    """`--impl reference`: the reference's CPU implementation of the path is Python and cannot travel
    to the GPU box, so this arm times its oracle port (bit-exact with it on the golden traces) on all
    host threads, on the SAME batch as the CUDA arm (`envs_per_gpu` envs; bounded at 65 536), with the same
    warm-up count; exactly `--steps` steps per timed pass, passes repeated until >= 2 s of timed work, median reported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = CpuRunner(wl, all_cores=True, envs=args.envs or None)
    sec, passes = r.timed_passes(args.steps, args.warmup)
    v = r.B * args.steps / sec
    base = dict(value=v, unit=UNIT, cores=r.cores, kind="port",
                sample=f"{r.what}: {r.B} envs x {args.steps} steps of {wl['name']} (random policy + step + masks + node "
                       f"features + belief) per pass, median of {len(passes)} passes, {sum(passes):.1f} s timed")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32/f64", "data": "synthetic",
        "config": {"workload": f"{wl['name']}: {wl['desc']}", "num_nodes": wl["N"], "num_police": wl["P"],
                   "envs_per_gpu": r.B, "passes_s": [round(x, 4) for x in passes],
                   "note": "CPU arm = oracle port of the reference env on all host threads (the reference is pure Python "
                           "and is not present on the GPU box; the unmodified reference timed in the build container: "
                           "profiles/r02_reference_python.json); one rank runs it, on one GPU's batch"},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# CUDA arm
# --------------------------------------------------------------------------------------------
def run_cuda_arm(args, wl):
    import torch

    import __graft_entry__ as ge

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    # one slice of the host cores per rank: the ranks' pinned copies, spin-waits and policy threads do not migrate onto
    # each other's cores (round 1 lost 13 % of the 8-GPU host-buffer throughput to that)
    affinity = None
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // max(world, 1)
        if world > 1 and per >= 2:
            affinity = cores[local * per:(local + 1) * per]
            os.sched_setaffinity(0, affinity)
    except Exception:
        affinity = None
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build()
    if dist is not None:
        dist.barrier()
    from student_mechanism_design_b200 import BatchedScotlandYardEnv, _cabi

    if os.environ.get("SY_LIB_PATH") and not args.allow_lib_override:
        raise SystemExit("bench.py: SY_LIB_PATH is set; the benchmark times the in-tree library (--allow-lib-override for experiments)")
    if os.environ.get("SY_DEBUG_SKIP"):
        raise SystemExit("bench.py: SY_DEBUG_SKIP is set; refusing to time a run with kernel parts switched off")
    lib = _cabi.load_library()
    N, P, B = wl["N"], wl["P"], args.envs or wl["B"]
    A = P + 1
    pool_kw = dict(num_graphs=1) if args.graphs <= 1 else dict(num_graphs=args.graphs, graphs="device")  # pool sampled on the device
    if args.nf_u8:
        pool_kw["node_features_dtype"] = torch.uint8
    env = BatchedScotlandYardEnv(B, P, wl["money"], graph_nodes=N, graph_edges=wl["E"], seed=0, **pool_kw,
                                 tolls=wl["toll"], belief=wl["belief"], reveal_interval=wl["reveal"], auto_reset=True,
                                 env_offset=rank * B, device=f"cuda:{local}")
    if args.writer:
        env.set_option("writer_path", args.writer)
    env.reset()
    dev = env.device
    actions = torch.empty(B, A, dtype=torch.int64, device=dev)
    K, W = args.steps, args.warmup
    sampler = ClockSampler(local)
    # the policy that picks the actions: the on-device random-valid sampler (configs 2-4) or the batched forward of
    # the reference's agents (config 5; random-init weights of the reference architectures, epsilon-greedy / sampling)
    policy = args.policy or wl.get("policy", "random")
    plib = None
    if policy == "gnn":
        from student_mechanism_design_b200 import GNNPolicy, _policy_cabi

        plib = _policy_cabi.load_library()
        gnn = GNNPolicy(env, seed=0)

        def choose(counter):
            gnn.act(args.epsilon, args.epsilon, step_counter=counter, out=actions)
        policy_desc = f"GNNAgent x2 (2 x AntiSymmetricConv + Linear, K={A}), epsilon-greedy eps={args.epsilon}, fused sy_gnn_act"
    elif policy == "mappo":
        from student_mechanism_design_b200 import MappoPolicy, _policy_cabi

        plib = _policy_cabi.load_library()
        mappo = MappoPolicy(env, obs_size=A, hidden_size=64, seed=0)

        def choose(counter):  # obs=None: MappoTrainer's observations (mappo_trainer.py:171-199) are built inside the kernel
            mappo.act(None, step_counter=counter, out=actions)
        policy_desc = (f"MappoAgent actors (Linear({A},64)-ReLU-Linear(64,{N})-softmax, one per agent) on the trainer's observations "
                       "(MrX_pos / Polices_pos, built in the kernel), masked sampling, fused sy_mappo_act")
    else:
        def choose(counter):
            env.sample_actions(out=actions, step_counter=counter)
        policy_desc = "on-device Philox random valid"
    py_loop = args.python_loop or policy != "random"

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput (`value`)
    counter = 0
    for _ in range(W):
        choose(counter)
        env.step(actions)
        counter += 1
    # --cuda-graph (random policy only): the K steps are replays of one captured sy_rollout_random_dev segment whose
    # step counter lives on the device (fresh draws on every replay)
    use_graph = not args.no_cuda_graph and not args.python_loop and policy == "random"
    seg = 0
    if use_graph:
        seg = next(s for s in (50, 25, 20, 10, 5, 4, 2, 1) if K % s == 0)
        env._sample_counter = counter
        rollout_graph, _ctr = env.capture_rollout(seg, actions=actions)
        counter += seg
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if use_graph:  # one more warm replay: the first launch of an instantiated graph uploads it
        rollout_graph.replay()
        counter += seg

    def timed_pass():
        """exactly K steps between two CUDA events, barrier + synchronise on both sides, max over ranks"""
        nonlocal counter
        barrier()
        ev0.record()
        if use_graph:  # replay the captured segment: launch latency is paid once per segment instead of three times per step
            for _ in range(K // seg):
                rollout_graph.replay()
            counter += K
        elif py_loop:
            for k in range(K):
                choose(counter)
                env.step(actions)
                counter += 1
        else:  # the K steps are issued by one C-ABI call (sy_rollout_random): no Python between steps
            env.rollout_random(K, actions=actions, step_counter=counter)
            counter += K
        ev1.record()
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1))

    sampler.active = True
    launches0 = lib.sy_launch_count() + (plib.sy_policy_launch_count() if plib else 0)
    pass_ms = [timed_pass() for _ in range(args.passes)]  # SURVEY 8(d): median of 5
    sampler.active = False
    launches = lib.sy_launch_count() + (plib.sy_policy_launch_count() if plib else 0) - launches0
    if use_graph:  # kernels inside a replayed graph do not pass through the library's host-side counter
        launches += args.passes * (K // seg) * (3 * seg + 1)
    launches //= args.passes  # per timed pass of K steps
    ms_total = statistics.median(pass_ms)
    value = world * B * K / (ms_total * 1e-3)
    # the one collective of the path (SURVEY 8(e)): the statistics vector, folded on the device and summed over the ranks
    # with one NCCL all-reduce per reporting interval -- here once, after the timed passes, timed on its own
    barrier()
    ev0.record()
    stats_total = env.stats(reduce_group=True if dist is not None else None)
    ev1.record()
    barrier()
    stats_ms = max_over_ranks(ev0.elapsed_time(ev1))
    if args.dump_outputs and rank == 0:  # before the roofline steps below move the env on
        dump_outputs(args.dump_outputs, env, actions, stats_total)

    # ---- duration of the sy_step call alone (its two kernels), CUDA events around every call, for the roofline
    Kk = min(K, 300)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(Kk)]
    barrier()
    sampler.active = True
    for k in range(Kk):
        kev[k][2].record()
        choose(counter)
        kev[k][0].record()
        env.step(actions)
        kev[k][1].record()
        counter += 1
    barrier()
    sampler.active = False
    # median: a host hiccup between the two launches of a call (this loop is driven from Python) must not read as kernel time
    step_kernel_ms = statistics.median(a.elapsed_time(b) for a, b, _ in kev)
    policy_ms = statistics.median(c.elapsed_time(a) for a, _, c in kev)

    # ---- end to end through the host-buffer API
    # The rank's batch is driven as `--e2e-halves` half-batch envs (own handle, own stream, own host thread; ctypes calls
    # release the GIL): while one half waits for its PCIe copies the other half's kernels run, so the host round trips of
    # the two halves hide behind each other's device work (ping-pong).  Every step of every half still moves its actions
    # host -> device and its results device -> host and synchronises before the next step of that half.
    Ke = max(3, args.e2e_steps)  # its own step count (reported): a 20-step region would be 3 ms, a third of it thread start-up
    H = max(1, args.e2e_halves)
    while B % H:
        H -= 1
    Bh = B // H
    e2e_envs, e2e_streams, e2e_policies = [], [], []
    for h in range(H):
        st = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(st):
            eh = BatchedScotlandYardEnv(Bh, P, wl["money"], graph_nodes=N, graph_edges=wl["E"], seed=0, **pool_kw,
                                        tolls=wl["toll"], belief=wl["belief"], reveal_interval=wl["reveal"], auto_reset=True,
                                        env_offset=rank * B + h * Bh, device=f"cuda:{local}")
            eh.reset()
            if policy == "gnn":
                e2e_policies.append(GNNPolicy(eh, seed=0))
            elif policy == "mappo":
                e2e_policies.append(MappoPolicy(eh, obs_size=A, hidden_size=64, seed=0))
            else:
                e2e_policies.append(None)
        e2e_envs.append(eh)
        e2e_streams.append(st)
    torch.cuda.synchronize(dev)

    def e2e_leg(wname, fl, passes=3):
        """Ke steps per half of: the policy's actions in pinned HOST memory -> H2D -> step -> D2H of the results ->
        synchronise; `passes` times, the median pass.  The policy (random sampler, or the GNN / MAPPO forward of config 5)
        runs on the device from the resident state and its actions travel to the host first, so a host-side consumer is
        emulated honestly (those D2H bytes are counted)."""
        wire, wb = {"int64": (torch.int64, 8), "int32": (torch.int32, 4), "int16": (torch.int16, 2)}[wname]
        errors, last = [], [None] * H

        def host_actions(h, eh, pol, c):
            if pol is None:
                return eh.sample_actions_host(step_counter=c, dtype=wire)  # kernel + D2H + synchronise in one C call
            buf = eh._host_buffers()["actions"]
            if policy == "gnn":
                acts = pol.act(args.epsilon, args.epsilon, step_counter=c)
            else:
                acts, _ = pol.act(None, step_counter=c)
            buf.copy_(acts, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            return buf

        def worker(h, steps, c0, gate):
            try:
                eh, pol = e2e_envs[h], e2e_policies[h]
                gate.wait()  # all host threads exist before the clock starts
                with torch.cuda.device(dev), torch.cuda.stream(e2e_streams[h]):
                    if pol is None and not args.e2e_python_loop:
                        # the same two C-ABI calls per step (sy_sample_actions_host, sy_step_host*), issued from C
                        last[h] = eh.host_rollout_random(steps, step_counter=c0, dtype=wire, flags=fl)
                    else:
                        for k in range(steps):
                            last[h] = eh.step_host(host_actions(h, eh, pol, c0 + k), flags=fl)
                    torch.cuda.current_stream(dev).synchronize()
            except Exception as exc:  # surfaced below: a dead worker must not look like a fast one
                errors.append(exc)

        def run(steps, c0):
            gate = threading.Barrier(H + 1)
            ts = [threading.Thread(target=worker, args=(h, steps, c0, gate)) for h in range(H)]
            for t in ts:
                t.start()
            barrier()
            t0 = time.perf_counter()
            gate.wait()
            for t in ts:
                t.join()
            if errors:
                raise errors[0]
            torch.cuda.synchronize(dev)
            return (time.perf_counter() - t0) * 1e3

        for eh in e2e_envs:
            eh.set_host_overlap(not args.e2e_no_overlap)  # results return while the observation kernel of the step still runs
        c = 1 << 20
        run(3, c)
        ms = []
        for _ in range(passes):
            c += Ke + 3
            ms.append(max_over_ranks(run(Ke, c)))
        for eh in e2e_envs:
            eh.set_host_overlap(False)
        assert all(r["reward"].shape == (Bh, A) and not r["reward"].is_cuda for r in last)
        e2e_ms = statistics.median(ms)
        pol_wb = wb if policy == "random" else 8  # the agents' kernels emit int64 actions
        return {"value": world * B * Ke / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": H * e2e_envs[0].host_h2d_bytes_per_step(wb if policy == "random" else 8),
                "d2h_bytes_per_step": H * e2e_envs[0].host_d2h_bytes_per_step(pol_wb, fl),
                "steps": Ke, "passes_ms": [round(x, 3) for x in ms], "half_batches": H, "policy": policy,
                "loop": "python" if (policy != "random" or args.e2e_python_loop) else "sy_host_rollout_random (C)",
                "note": f"{H} half-batch env(s) of {Bh} envs, one host thread and stream each (ping-pong); per step and half: "
                f"actions int{(wb if policy == 'random' else 8) * 8}[B,A] from pinned host memory in; reward f32 [B,A] + winner + "
                + ("one status byte per env (terminated/truncated/frozen bits; every agent of an env shares them)" if fl == "compact"
                   else "terminated/truncated/done u8 [B,A] + status") +
                " out to pinned host memory, synchronised; observations stay on the device for the GPU policy; the D2H count "
                "includes the policy's actions coming back to the host; wall clock with device synchronisation on both sides"}

    # wire format of the host actions: node ids fit 16 bits at every BASELINE config; --e2e-int64 = the reference's dtype
    wname = "int64" if args.e2e_int64 else (args.e2e_wire if N <= 32767 or args.e2e_wire != "int16" else "int32")
    sampler.active = True
    e2e = e2e_leg(wname, args.e2e_flags)
    # the reference's own call shape (yard.py:144,269): int64 actions in, per-agent [B, A] flag arrays out
    e2e_ref_shape = e2e if (wname, args.e2e_flags) == ("int64", "per_agent") else e2e_leg("int64", "per_agent")
    sampler.active = False
    for eh in e2e_envs:
        eh.close()

    clocks = sampler.summary()
    if rank == 0:
        bstep = algorithmic_bytes_per_env_step(N, P, wl["belief"], 1 if args.nf_u8 else 4)
        peak, peak_src = measured_hbm_peak()
        achieved = bstep * B / (step_kernel_ms * 1e-3) / 1e9
        traffic, traffic_note = None, None
        tp = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
        if os.path.isfile(tp) and not args.nf_u8:  # the ncu capture is of the float32 observation layout
            try:
                rec = json.load(open(tp))
                if rec.get("source_sha256") == kernel_source_hash():  # refuse a capture of other kernels
                    traffic = rec.get(wl["name"], {}).get("dram_bytes_per_launch")
                else:
                    traffic_note = "profiles/step_kernel_traffic.json was captured from a different csrc/sy_env.cu: ignored"
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32/f64", "data": "synthetic",
            "config": {"workload": f"{wl['name']}: {wl['desc']}", "num_nodes": N, "num_police": P,
                       "envs_per_gpu": B, "global_envs": world * B, "graph_pool": env.num_graphs, "node_features_dtype": "uint8 (opt-in)" if args.nf_u8 else "float32", "policy": policy_desc, "policy_ms_per_step": policy_ms, "loop": (f"CUDA graph replay of {seg}-step sy_rollout_random_dev segments" if use_graph else
                                "python" if py_loop else "sy_rollout_random (C)"),
                       "auto_reset": True, "parallelism": f"batch-sharded x{world}", "host_cores_per_rank": None if affinity is None else len(affinity),
                       "l2": f"per-step working set {bstep * B / 1e6:.0f} MB per GPU > 126 MB L2 (no flush needed)"},
            "clocks": clocks, "e2e": e2e, "e2e_reference_shape": e2e_ref_shape, "gpu_launches": int(launches),
            "passes_ms": [round(x, 4) for x in pass_ms], "stats_fold_allreduce_ms": stats_ms,
            "library": {"path": os.path.relpath(_cabi.LIB_PATH, ROOT), "override": bool(os.environ.get("SY_LIB_PATH")),
                        "options": getattr(env, "options", {})},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_note": traffic_note, "kernel": "sy_step = sy_logic_kernel + sy_observe_kernel", "kernel_ms": step_kernel_ms,
                         "algorithmic_bytes_per_env_step": bstep, "peak_source": peak_src},
            "episode_stats": stats_total,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = CpuRunner(wl, all_cores=True, envs=min(B, 65536)).timed(args.cpu_seconds)[0]
        print(json.dumps(line), flush=True)
    env.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="override envs per GPU")
    ap.add_argument("--nf-u8", action="store_true",
                    help="write node_features as uint8 instead of float32 (opt-in observation dtype; the roofline bytes follow)")
    ap.add_argument("--graphs", type=int, default=1, help="graph pool size (> 1: sampled on the device; envs in blocks of 32 per graph)")
    ap.add_argument("--passes", type=int, default=5, help="timed passes of --steps steps each; the median is reported")
    ap.add_argument("--writer", default=None, choices=["bulk", "lsu"], help="observation writer path (sy_set_option; default bulk)")
    ap.add_argument("--allow-lib-override", action="store_true", help="accept SY_LIB_PATH (kernel-variant experiments only)")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--e2e-python-loop", action="store_true",
                    help="host-buffer leg: call sample_actions_host / step_host from Python every step instead of sy_host_rollout_random")
    ap.add_argument("--e2e-halves", type=int, default=4,
                    help="host-buffer leg: number of half-batch envs (one host thread + stream each) the rank's batch is driven as")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-int64", action="store_true", help="host actions as int64 (the reference dtype)")
    ap.add_argument("--e2e-wire", default="int16", choices=["int16", "int32", "int64"], help="wire format of the host actions")
    ap.add_argument("--e2e-no-overlap", action="store_true",
                    help="fully synchronous host calls (default: step_host returns when the results are on the host, the next "
                         "host actions are produced while the observation kernel of the step still runs)")
    ap.add_argument("--e2e-flags", default="compact", choices=["compact", "per_agent"],
                    help="host results: one status byte per env, or the reference-shaped [B, A] flag arrays")
    ap.add_argument("--policy", default=None, choices=["random", "gnn", "mappo"],
                    help="who picks the actions (default: the workload's; c5 = gnn)")
    ap.add_argument("--epsilon", type=float, default=0.05, help="exploration rate of the GNN agents")
    ap.add_argument("--no-cuda-graph", action="store_true",
                    help="issue the timed steps with one sy_rollout_random call instead of replaying a captured CUDA graph of "
                         "50-step segments (the default for the random policy: no launch gaps between the kernels)")
    ap.add_argument("--python-loop", action="store_true", help="issue every step from Python instead of sy_rollout_random")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed passes, write what their last step computed as DIR/<name>.npy (CUDA arm, rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    wl = dict(WORKLOADS[args.workload], name=args.workload)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA arm")
        run_reference_arm(args, wl)
    else:
        run_cuda_arm(args, wl)


if __name__ == "__main__":
    main()
