"""Checks of bench.py: its accounting and the committed bench lines (the contract of its JSON line) on the CPU, the
outputs it dumps on the GPU."""
import importlib.util
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_bytes_match_the_survey_figure():
    """SURVEY.md 8(d): 8849 B per env-step at c3 (N = 200, P = 6, belief on)."""
    b = _bench()
    assert b.algorithmic_bytes_per_env_step(200, 6, True) == 8849
    assert b.algorithmic_bytes_per_env_step(200, 6, False) == 8849 - 8 * 200
    wl = b.WORKLOADS
    assert wl["c3"]["N"] == 200 and wl["c3"]["P"] == 6 and wl["c3"]["B"] == 65536 and wl["c3"]["belief"]
    assert wl["c2"]["B"] == 1024 and wl["c4"]["N"] == 1000 and wl["c5"]["B"] * 8 == 1 << 20


def test_committed_bench_lines_carry_the_contract_keys():
    need = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"}
    for name in ("r01_bench_c3_final.json", "r01_bench_c3_n8.json", "r01_bench_c5_gnn_n1.json", "r01_bench_c4_n1.json"):
        line = json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])
        assert need <= set(line), (name, need - set(line))
        assert line["metric"] == "batched_env_steps_per_sec" and line["higher_is_better"] is True and line["scaling"] == "weak"
        assert line["vs_baseline"] is None and "workload" in line["config"] and line["gpu_launches"] > 0
        r = line["roofline"]
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        e = line["e2e"]
        assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != line["value"]
        assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    final = json.loads(open(os.path.join(ROOT, "profiles", "r01_bench_c3_final.json")).read().strip().splitlines()[-1])
    assert final["n_gpus"] == 1 and {"value", "unit", "cores", "kind", "sample"} <= set(final["cpu_baseline"])
    ref = json.loads(open(os.path.join(ROOT, "profiles", "r01_bench_c3_reference_arm.json")).read().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["cpu_baseline"]["kind"] == "port"


def test_round2_bench_lines_carry_the_contract_keys():
    """The round-2 lines add: median-of-5 passes, the reference-shaped e2e, the library record, cpu_baseline on every
    N = 1 workload line, and a traffic figure that is either null or stamped for the build it ran on."""
    need = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "e2e_reference_shape", "gpu_launches", "roofline", "passes_ms", "library"}
    names = ["r02_bench_c3_n1.json", "r02_bench_c3_steps20.json", "r02_bench_c2_n1.json", "r02_bench_c4_n1.json",
             "r02_bench_c5_gnn_n1.json", "r02_bench_c5_mappo_n1.json", "r02_bench_c3_n2.json", "r02_bench_c3_n4.json",
             "r02_bench_c3_n8.json"]
    for name in names:
        line = json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])
        assert need <= set(line), (name, need - set(line))
        assert line["metric"] == "batched_env_steps_per_sec" and line["higher_is_better"] is True and line["scaling"] == "weak"
        assert line["vs_baseline"] is None and "workload" in line["config"] and line["gpu_launches"] > 0
        assert len(line["passes_ms"]) == 5 and line["library"]["override"] is False
        r = line["roofline"]
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert r["traffic"] is None or 0.5 < r["traffic"] / (r["algorithmic_bytes_per_env_step"] * line["config"]["envs_per_gpu"]) < 1.2
        for key in ("e2e", "e2e_reference_shape"):
            e = line[key]
            assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != line["value"]
        assert line["e2e_reference_shape"]["h2d_bytes_per_step"] >= line["e2e"]["h2d_bytes_per_step"]
        assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if line["n_gpus"] == 1:
            assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"]) and line["cpu_baseline"]["kind"] == "port"
    n1 = json.loads(open(os.path.join(ROOT, "profiles", "r02_bench_c3_steps20.json")).read().strip().splitlines()[-1])
    for n, name in ((2, "r02_bench_c3_n2.json"), (4, "r02_bench_c3_n4.json"), (8, "r02_bench_c3_n8.json")):
        line = json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])
        assert line["n_gpus"] == n and 0.95 < line["value"] / (n * n1["value"]) < 1.05  # weak scaling of the device path
    ref = json.loads(open(os.path.join(ROOT, "profiles", "r02_bench_c3_reference_arm.json")).read().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["cpu_baseline"]["kind"] == "port"
    assert ref["config"]["envs_per_gpu"] == n1["config"]["envs_per_gpu"]  # the CPU arm steps the same batch


@pytest.mark.gpu
def test_dump_outputs_are_those_of_the_last_timed_step(tmp_path):
    """--dump-outputs: the same arguments give the same inputs, so two runs write identical float32 / float64 arrays
    (under 64 MB in all); they equal the C oracle's after exactly the steps the benchmark has run at the end of its timed
    passes, and two more timed steps per pass add exactly that many steps."""
    import numpy as np

    import sy_oracle as so
    import sy_oracle_c as oc
    from student_mechanism_design_b200.graphs import generate_graph_pool

    B, warmup, passes = 1024, 3, 2  # c2: 50 nodes, 110 edges, 3 police, budget 10, no tolls, no belief, reveal every 5

    def run(tag, steps):
        out = tmp_path / tag
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "c2", "--steps", str(steps),
                            "--warmup", str(warmup), "--passes", str(passes), "--no-cpu-baseline", "--e2e-steps", "3",
                            "--dump-outputs", str(out)], capture_output=True, text=True, cwd=tmp_path)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == steps
        return {f.stem: np.load(f) for f in sorted(out.glob("*.npy"))}

    a, b, c = run("a", 7), run("b", 7), run("c", 9)
    assert set(a) == set(b) == set(c) >= {"actions", "reward", "terminated", "agent_position", "action_mask", "node_features",
                                          "env_index", "episode_stats"}
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    # 7 and 9 have no divisor among bench.py's segment lengths (50, 25, 20, 10, 5, 4, 2), so the timed passes replay a
    # 1-step graph, which also ran once when it was captured and once to upload it: at the dump the env has taken
    # warmup + 2 + passes * steps steps.  Other step counts change that count of untimed steps.
    T = warmup + 2 + passes * 7
    assert a["episode_stats"][0] == B * T and c["episode_stats"][0] == B * (T + passes * (9 - 7))  # STAT_NAMES[0] = env_steps
    pool = [so.Graph(g.num_nodes, g.edge_links, g.edges) for g in generate_graph_pool(1, 50, 110, seed=0)]
    ob = oc.CBatch(so.OracleConfig(num_police=3, agent_money=10, toll=0, belief=False, reveal_interval=5), pool, B, seed=0)
    ob.steps(T - 1)
    acts = ob.sample_actions(T - 1)
    want = ob.step(acts)
    idx = a["env_index"].astype(np.int64)
    assert np.array_equal(idx, np.arange(B))  # the whole c2 batch fits the sample
    expect = {"actions": acts, "agent_position": ob.pos(), "Currency": ob.money()[:, 1:], "MrX_revealed": ob.revealed(),
              "reward": want["reward"].astype(np.float32), "terminated": np.repeat(want["terminated"][:, None], 4, 1),
              "winner": want["winner"], "action_mask": ob.masks(), "node_features": ob.node_features()}
    for k, v in expect.items():
        np.testing.assert_array_equal(a[k], np.asarray(v, dtype=np.float32)[idx], err_msg=k)
