"""Cost of mechanism groups (env.set_mechanisms) at c3 and c2: four variants of the same handle in one process,
timed alternately, median of 5 passes each -- no groups, one group equal to the config, 16 groups interleaved
(the default b % 16 assignment) and 1 024 groups, the groups differing in their reward weights only.  Two timings per variant: `sy_step` (K plain steps between a CUDA
event pair, actions drawn once beforehand) and the replayed `capture_rollout` graph (K steps of the random policy).
c3 runs with the belief scored at reveal steps (belief_ce), so the per-group cross-entropy atomics are included.
Writes profiles/r03_mechanisms_c{2,3}.json (or --out-dir) with the card's name and power limit.

--tolls (opt-in): no groups, the same 16 groups, and those 16 groups with their own tolls cycling 0..3 (group g pays
g % 4), timed the same way; writes profiles/r04_group_tolls_c{2,3}.json.  Other tolls change the games themselves (which
moves are legal, how long episodes last), so that variant does not do exactly the same game work.

--rules (opt-in): no groups, the same 16 groups, and those 16 groups with `number_of_agents` / `max_timestep` given
explicitly through sy_set_group_rules with the handle's own values (the same game work: any difference is the cost of
the per-env police count and horizon), timed the same way; plus, for information, the 16 groups with police counts
cycling P, P-1, ..., 1 (group g plays P - g % P police: less game work per env, different games).  Writes
profiles/r05_group_rules_c{2,3}.json.

    python tools/bench_mechanisms.py [--workloads c3,c2] [--steps 50] [--passes 5] [--tolls | --rules]
"""
import ctypes as C
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {  # bench.py's c2 / c3 (c3 with the belief scored at reveals)
    "c2": dict(N=50, E=110, P=3, money=10, toll=0, belief=False, reveal=5, B=1024),
    "c3": dict(N=200, E=400, P=6, money=20, toll=1, belief=True, reveal=5, B=65536),
}
VARIANTS = ["no_groups", "one_group_equal", "groups_16", "groups_1024"]
TOLL_VARIANTS = ["no_groups", "groups_16", "groups_16_tolls"]
RULE_VARIANTS = ["no_groups", "groups_16", "groups_16_rules", "groups_16_police"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, sm = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, sm_max_clock=sm)
    except Exception as exc:  # noqa: BLE001
        import torch

        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({exc.__class__.__name__})")


def run(wl_name, steps, passes, variants=VARIANTS):
    import torch

    from student_mechanism_design_b200 import BatchedScotlandYardEnv

    wl = WORKLOADS[wl_name]
    envs = {}
    for v in variants:
        env = BatchedScotlandYardEnv(wl["B"], wl["P"], wl["money"], graph_nodes=wl["N"], graph_edges=wl["E"], seed=0,
                                     num_graphs=1, tolls=wl["toll"], belief=wl["belief"], belief_ce=wl["belief"],
                                     reveal_interval=wl["reveal"], auto_reset=True, device="cuda:0")
        if v == "one_group_equal":
            env.set_mechanisms([{}])
        elif v in ("groups_16", "groups_1024", "groups_16_tolls", "groups_16_rules", "groups_16_police"):
            # distinct mechanisms with the config's budget and reveal schedule: only the reward weights differ, so
            # every variant does the same game work and the difference is the cost of the groups themselves
            n = 1024 if v == "groups_1024" else 16
            mechs = [dict(reward_weights={"Mrx_closest": 0.3 + 0.001 * g, "Police_distance": 0.1 + 0.001 * g})
                     for g in range(n)]
            if v == "groups_16_tolls":
                for g, m in enumerate(mechs):
                    m["tolls"] = g % 4
            if v == "groups_16_police":
                for g, m in enumerate(mechs):
                    m["number_of_agents"] = wl["P"] - g % wl["P"]
            env.set_mechanisms(mechs)
            if v == "groups_16_rules":  # the handle's values, explicitly (set_mechanisms only calls when one differs)
                arr = lambda x: (C.c_int32 * n)(*([x] * n))  # noqa: E731
                rc = env._lib.sy_set_group_rules(env._handle, n, arr(wl["P"]), arr(env.config.max_timestep), env._stream())
                assert rc == 0, rc
        env.reset()
        acts = env.sample_actions(step_counter=0)
        graph, _ = env.capture_rollout(steps)
        for _ in range(3):  # warm every shape of the timed window
            env.step(acts)
            graph.replay()
        envs[v] = (env, acts, graph)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {v: {"sy_step_ms": [], "graph_replay_ms": []} for v in variants}
    for p in range(passes):
        order = variants if p % 2 == 0 else variants[::-1]  # alternate, so drift does not favour one variant
        for v in order:
            env, acts, graph = envs[v]
            ev0.record()
            for _ in range(steps):
                env.step(acts)
            ev1.record()
            torch.cuda.synchronize()
            times[v]["sy_step_ms"].append(ev0.elapsed_time(ev1) / steps)
            ev0.record()
            graph.replay()
            ev1.record()
            torch.cuda.synchronize()
            times[v]["graph_replay_ms"].append(ev0.elapsed_time(ev1) / steps)
    out = {}
    for v in variants:
        env = envs[v][0]
        row = {}
        for k, xs in times[v].items():
            row[k] = statistics.median(xs)
            row[k + "_passes"] = [round(x, 5) for x in xs]
            row[k + "_spread"] = max(xs) - min(xs)
        row["groups"] = 0 if env.mechanisms is None else len(env.mechanisms)
        out[v] = row
    base = out["no_groups"]
    for v in variants[1:]:
        for k in ("sy_step_ms", "graph_replay_ms"):
            out[v][k + "_vs_no_groups"] = out[v][k] / base[k] - 1.0
            if v in ("groups_16_tolls", "groups_16_rules", "groups_16_police"):
                out[v][k + "_vs_groups_16"] = out[v][k] / out["groups_16"][k] - 1.0
    for env, _, _ in envs.values():
        env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c2")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--tolls", action="store_true", help="16 groups with and without their own tolls (r04 profiles)")
    ap.add_argument("--rules", action="store_true", help="16 groups with the police count / horizon machinery (r05 profiles)")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("bench_mechanisms.py needs a CUDA device")
    info = card()
    os.makedirs(args.out_dir, exist_ok=True)
    for w in args.workloads.split(","):
        note = ("every variant takes the handle's usual path (c3: dynamics + observation kernels, c2: fused "
                "step / one-launch rollout kernel), the grouped ones through its GROUPS instantiation; c3 scores "
                "the belief at reveal steps (about 4 us per step over bench.py's c3 line, which does not)")
        if args.tolls:
            note += (f"; groups_16_tolls: group g pays toll g % 4 (config toll {WORKLOADS[w]['toll']}), so its games "
                     "differ from the other variants'")
        if args.rules:
            note += (f"; groups_16_rules: the 16 groups with number_of_agents = {WORKLOADS[w]['P']} and max_timestep = 250 "
                     "given through sy_set_group_rules (same games as groups_16); groups_16_police (information only): "
                     f"group g plays {WORKLOADS[w]['P']} - g % {WORKLOADS[w]['P']} police, so its games differ")
        variants = TOLL_VARIANTS if args.tolls else (RULE_VARIANTS if args.rules else VARIANTS)
        res = dict(workload=w, config=WORKLOADS[w], steps_per_pass=args.steps, passes=args.passes, card=info, note=note,
                   variants=run(w, args.steps, args.passes, variants))
        name = "r04_group_tolls" if args.tolls else ("r05_group_rules" if args.rules else "r03_mechanisms")
        path = os.path.join(args.out_dir, f"{name}_{w}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res))


if __name__ == "__main__":
    main()
