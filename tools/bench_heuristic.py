"""Cost of the heuristic opponents (sy_heuristic_actions) at c2 and c3, in one process per workload.

Per-call time: K calls of the kernel between a CUDA event pair, for each heuristic kind and for the random sampler
(sy_sample_actions) on the same state, the variants alternated pass by pass, median of 5 passes.  c2 = 1 024 envs; c3 =
65 536 envs with belief on and toll 1, plus (c3) the same handle with 16 interleaved mechanism groups whose tolls cycle
0..3 and police counts P..1.  The state is 12 random steps into the episodes (some MrX revealed, some hidden, last_seen
filled), and the kernel does not change it, so every call times the same work.
Loop time: a 250-step mechanism-evaluation loop -- `HeuristicPolicy.act()` + `env.step` from Python -- against
`env.rollout_random(250)` (the random policy's loop issued from C), alternated, median of the passes.
Writes profiles/r06_heuristic_c{2,3}.json (or --out-dir) with the card's name and power limit read in the same run.

    python tools/bench_heuristic.py [--workloads c3,c2] [--calls 50] [--passes 5] [--loop-steps 250]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_mechanisms import WORKLOADS, card  # noqa: E402

KINDS = {  # variant -> (mrx, police)
    "evade_chase": ("evade", "chase"),
    "evade_chase_belief": ("evade", "chase_belief"),
    "evade_only": ("evade", None),
    "chase_only": (None, "chase"),
    "random_random": ("random", "random"),
}


def _env(wl, groups=False):
    from student_mechanism_design_b200 import BatchedScotlandYardEnv

    env = BatchedScotlandYardEnv(wl["B"], wl["P"], wl["money"], graph_nodes=wl["N"], graph_edges=wl["E"], seed=0,
                                 num_graphs=1, tolls=wl["toll"], belief=wl["belief"], reveal_interval=wl["reveal"],
                                 auto_reset=True, device="cuda:0")
    if groups:
        env.set_mechanisms([dict(tolls=g % 4, number_of_agents=wl["P"] - g % wl["P"]) for g in range(16)])
    env.reset()
    for s in range(12):
        env.step(env.sample_actions(step_counter=s))
    return env


def time_calls(env, calls, passes, belief):
    import torch

    from student_mechanism_design_b200 import HeuristicPolicy

    out = torch.empty(env.num_envs, env.num_agents, dtype=torch.int64, device=env.device)
    fns = {"sample_actions": lambda k: env.sample_actions(out=out, step_counter=k)}
    for name, (m, p) in KINDS.items():
        if p == "chase_belief" and not belief:
            continue
        h = HeuristicPolicy(env, m, p)
        for k in range(12):  # fill last_seen as a policy called at every step would have
            h.act(out=out, step_counter=k)
        fns[name] = (lambda h: lambda k: h.act(out=out, step_counter=k))(h)
    for f in fns.values():
        for k in range(3):
            f(k)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    names = list(fns)
    times = {n: [] for n in names}
    for p in range(passes):
        for n in (names if p % 2 == 0 else names[::-1]):
            ev0.record()
            for k in range(calls):
                fns[n](100 + k)
            ev1.record()
            torch.cuda.synchronize()
            times[n].append(ev0.elapsed_time(ev1) / calls)
    res = {}
    for n in names:
        res[n] = dict(ms=statistics.median(times[n]), ms_passes=[round(x, 5) for x in times[n]],
                      ms_spread=max(times[n]) - min(times[n]))
    for n in names[1:]:
        res[n]["vs_sample_actions"] = res[n]["ms"] / res["sample_actions"]["ms"]
    return res


def time_loops(wl, steps, passes):
    import torch

    from student_mechanism_design_b200 import HeuristicPolicy

    env_h, env_r = _env(wl), _env(wl)
    h = HeuristicPolicy(env_h, "evade", "chase")

    def heuristic_loop():
        for _ in range(steps):
            env_h.step(h.act())

    def random_loop():
        env_r.rollout_random(steps)

    loops = {"heuristic_act_plus_step": heuristic_loop, "rollout_random": random_loop}
    for f in loops.values():
        f()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {n: [] for n in loops}
    for p in range(passes):
        for n in (list(loops) if p % 2 == 0 else list(loops)[::-1]):
            ev0.record()
            loops[n]()
            ev1.record()
            torch.cuda.synchronize()
            times[n].append(ev0.elapsed_time(ev1))
    res = {n: dict(ms=statistics.median(xs), ms_passes=[round(x, 4) for x in xs], ms_spread=max(xs) - min(xs),
                   ms_per_step=statistics.median(xs) / steps) for n, xs in times.items()}
    res["heuristic_act_plus_step"]["vs_rollout_random"] = res["heuristic_act_plus_step"]["ms"] / res["rollout_random"]["ms"]
    env_h.close()
    env_r.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c2")
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--loop-steps", type=int, default=250)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_heuristic.py needs a CUDA device")
    info = card()
    os.makedirs(args.out_dir, exist_ok=True)
    for w in args.workloads.split(","):
        wl = WORKLOADS[w]
        env = _env(wl)
        calls = {"no_groups": time_calls(env, args.calls, args.passes, wl["belief"])}
        env.close()
        if w == "c3":
            env = _env(wl, groups=True)
            calls["groups_16_tolls_police"] = time_calls(env, args.calls, args.passes, wl["belief"])
            env.close()
        res = dict(workload=w, config=wl, calls_per_pass=args.calls, passes=args.passes, card=info,
                   note=("per-call times are CUDA-event means over `calls_per_pass` back-to-back calls on an unchanging "
                         "state; the graph tables stay in L2 between calls.  The loops include Python's per-step "
                         "launch overhead for the heuristic loop; rollout_random is issued from C"),
                   kernel_calls=calls, loops=time_loops(wl, args.loop_steps, args.passes))
        path = os.path.join(args.out_dir, f"r06_heuristic_{w}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res))


if __name__ == "__main__":
    main()
