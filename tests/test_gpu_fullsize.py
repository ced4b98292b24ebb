"""Oracle parity at the BENCHMARKED sizes (BASELINE.json configs 2-4) and through the timed path.

The small-batch tests of test_gpu_parity.py never reach the kernels' grid tails, partially filled waves, the replicated
statistics lines or the fork/join ordering of the CUDA-graph rollout the benchmark replays; these do.  The CPU side is
the C oracle (oracle/sy_oracle.c, pinned bit-exact to the reference's golden traces in tests/test_oracle_c.py) on all
host threads with the same seed: positions, budgets, timesteps, episodes, visit counts, masks, node features, reveal
flags, rewards (float64 bits), flags and winners byte-equal; belief_map within 1e-6 abs (north_star).
Reference lines covered: yard.py:144-269 (step), reward_calculator.py:26-266, action_mask.py:54-83, yard.py:271-335."""
import os

import numpy as np
import pytest

import sy_oracle as so
import sy_oracle_c as oc

pytestmark = pytest.mark.gpu

BELIEF_TOL = 1e-6  # north_star: "belief_map must match within 1e-6 abs"


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _threads():
    try:
        return max(1, min(len(os.sched_getaffinity(0)), oc.max_threads()))
    except Exception:
        return 1


def _pair(N, E, P, money, B, seed, *, toll, belief, reveal, graphs=1, writer=None, **env_kw):
    import student_mechanism_design_b200 as pkg

    pool = pkg.generate_graph_pool(graphs, N, E, seed=0)
    env = pkg.BatchedScotlandYardEnv(B, P, money, graphs=pool, seed=seed, auto_reset=True, tolls=toll, belief=belief,
                                     reveal_interval=reveal, keep_reward64=True, **env_kw)
    # "fused": one persistent kernel | two kernels with: "lsu" = all observation stores through the LSU (the default for
    # large batches) | "bulk" = chunk images + bulk stores in the observation kernel
    if writer == "lsu_lagged":  # rollouts: software-pipelined deferred steps through the lagged kernel
        env.set_option("lagged_kernel", "on")
        writer = "lsu"
    if writer == "lsu_pdl":  # dynamics / observation kernels launched with programmatic stream serialisation
        env.set_option("pdl", "on")
        writer = "lsu"
    if writer is not None:
        env.set_option("step_kernel", "fused" if writer == "fused" else "two_kernels")
        if writer != "fused":
            env.set_option("writer_path", "bulk" if writer == "bulk" else "lsu")
    cfg = so.OracleConfig(num_police=P, agent_money=money, toll=toll, belief=belief, reveal_interval=reveal)
    # the env's default graph assignment: blocks of 32 consecutive envs share a graph
    gid = (np.arange(B) // 32) % graphs
    ob = oc.CBatch(cfg, pool, B, seed=seed, auto_reset=True, threads=_threads(), graph_id=gid.astype(np.int32))
    return env, ob


def _same(t, want, what):
    got = t.cpu().numpy()
    if got.dtype == np.bool_ and want.dtype != np.bool_:
        want = want.astype(bool)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError(f"{what}: {len(bad)} mismatches, first at {bad[0].tolist()}: got {got[tuple(bad[0])]} want {want[tuple(bad[0])]}")


def _compare(env, ob, want, belief, tag, dense=True):
    _same(env.pos, ob.pos(), (tag, "pos"))
    _same(env.money, ob.money(), (tag, "money"))
    _same(env.timestep, ob.timestep(), (tag, "timestep"))
    _same(env.episode, np.asarray(ob._episode), (tag, "episode"))
    _same(env.graph_id, np.asarray(ob._gid), (tag, "graph_id"))
    _same(env.visits, ob.visits(), (tag, "visits"))
    _same(env.mrx_revealed, ob.revealed(), (tag, "mrx_revealed"))
    _same(env.agent_budget, ob.money().astype(np.float32), (tag, "agent_budget"))
    if dense:
        _same(env.action_mask, ob._mask, (tag, "action_mask"))
        _same(env.node_features, ob._nf, (tag, "node_features"))
    if belief:
        err = np.abs(env.belief_map.cpu().numpy().astype(np.float64) - ob._belief).max()
        assert err <= BELIEF_TOL, (tag, "belief_map", err)
    if want is not None:
        if want["reward"].dtype == np.float64:  # fp32 reward mode: the oracle hands back the float32 values
            assert env.reward64.cpu().numpy().tobytes() == want["reward"].tobytes(), (tag, "reward64 bits")
        assert env.reward.cpu().numpy().tobytes() == want["reward"].astype(np.float32).tobytes(), (tag, "reward")
        A = env.num_agents
        _same(env.terminated, np.repeat(want["terminated"][:, None], A, 1), (tag, "terminated"))
        _same(env.truncated, np.repeat(want["truncated"][:, None], A, 1), (tag, "truncated"))
        _same(env.winner, want["winner"], (tag, "winner"))


def _rollout_against_oracle(env, ob, steps, belief, dense_every=1):
    env.reset()
    _compare(env, ob, None, belief, "reset")
    done = 0
    for s in range(steps):
        acts = env.sample_actions(step_counter=s)
        a_h = acts.cpu().numpy()
        assert np.array_equal(a_h, ob.sample_actions(s)), ("sampler", s)
        env.step(acts)
        want = ob.step(a_h)
        _compare(env, ob, want, belief, ("step", s), dense=(s % dense_every == 0 or s == steps - 1))
        done += int(want["terminated"].sum() + want["truncated"].sum())
    st = env.stats()
    assert st["env_steps"] == env.num_envs * steps and st["episodes"] == done
    return done


@pytest.mark.parametrize("writer", ["lsu", "lsu_pdl", "fused", "bulk"])
def test_config3_full_size_matches_oracle(torch_cuda, writer):
    """BASELINE config 3 exactly as benchmarked: 200 nodes / 400 edges / 6 police, budget 20, toll 1, belief on,
    reveal every 5, 65 536 envs, same-step auto-reset, 25 steps -- every tile of the 2 048-tile grid and all statistics
    replicas, through the fused persistent step kernel and through the two-kernel path with both writer paths (TMA bulk
    stores and LSU stores)."""
    env, ob = _pair(200, 400, 6, 20, 65536, 1, toll=1, belief=True, reveal=5, writer=writer)
    done = _rollout_against_oracle(env, ob, 25, True, dense_every=3)
    assert done > 1000  # captures / out-of-money endings + same-step auto-resets happened at scale
    env.close()


@pytest.mark.parametrize("writer", ["fused", "lsu"])
def test_config2_full_size_matches_oracle(torch_cuda, writer):
    """BASELINE config 2: 50 nodes, 3 police, reveal every 5, 1024 envs, 60 steps (reveals and all endings occur)."""
    env, ob = _pair(50, 110, 3, 10, 1024, 2, toll=0, belief=False, reveal=5, writer=writer)
    done = _rollout_against_oracle(env, ob, 60, False)
    assert done > 100
    env.close()


@pytest.mark.parametrize("writer", ["lsu", "bulk"])
def test_config4_full_size_matches_oracle(torch_cuda, writer):
    """BASELINE config 4's per-GPU shard: 1000 nodes / 2000 edges / 6 police, 32 768 envs, 10 steps (large-N belief path,
    staged-CSR writers, chunks that cut through envs on the bulk path)."""
    env, ob = _pair(1000, 2000, 6, 20, 32768, 3, toll=1, belief=True, reveal=5, writer=writer)
    _rollout_against_oracle(env, ob, 10, True, dense_every=3)
    env.close()


def test_config3_ragged_batch_graph_pool(torch_cuda):
    """c3 shape with B not a multiple of the 32-env tile and a pool of 5 graphs (blocks of 32 envs per graph): the ragged
    last tile takes the byte-tail of the bulk writers."""
    env, ob = _pair(200, 400, 6, 20, 4096 + 19, 5, toll=1, belief=True, reveal=5, graphs=5)
    _rollout_against_oracle(env, ob, 12, True)
    env.close()


@pytest.mark.parametrize("writer", ["lsu", "lsu_lagged", "lsu_pdl", "fused"])
def test_timed_path_graph_replay_matches_oracle(torch_cuda, writer):
    """The path bench.py times -- capture_rollout (sy_rollout_random_dev: device-resident step counter; "lsu", the
    default at this size: two launches per step, the sampler of step k+1 forked next to the observation kernel of step
    k; "lsu_lagged": software-pipelined deferred steps, one lagged launch per step that carries the observations of
    step k, the dynamics of step k+1 and the action draw of step k+2, one flush per segment; fused: one persistent
    kernel per step whose logic warps also draw the next step's actions) replayed from a CUDA graph -- against the
    oracle after K replays, at c3 with a ragged 65 523-env batch."""
    torch = torch_cuda
    B, seg, replays = 65536 - 13, 5, 6
    env, ob = _pair(200, 400, 6, 20, B, 7, toll=1, belief=True, reveal=5, writer=writer)
    env.reset()
    graph, counter = env.capture_rollout(seg)  # runs `seg` steps as warm-up, then captures
    for _ in range(replays):
        graph.replay()
    torch.cuda.synchronize()
    total = seg * (1 + replays)
    assert int(counter.item()) == total
    want = None
    for s in range(total):
        want = ob.step(ob.sample_actions(s))
    _compare(env, ob, want, True, "after graph replays")
    st = env.stats()
    assert st["env_steps"] == B * total and st["episodes"] == int(np.asarray(ob._episode).sum())
    env.close()


@pytest.mark.parametrize("case", ["generic_quarters", "fast_path", "no_belief", "off"])
def test_observation_grid_tail_split(torch_cuda, case):
    """The observation kernel cuts the tiles of a partly filled last wave into 2 or 4 parts (one CTA each): batches whose
    tile count leaves such a tail -- 296 resident CTAs on a B200: 330 tiles = 1 wave + 34 tiles (quarters on the
    warp-per-env belief path at N = 500 and without a belief map; the lane = env fast path at N = 200 keeps whole tiles), a
    ragged last part -- and the same inputs with the split switched off."""
    import student_mechanism_design_b200 as pkg

    N, E, belief = (500, 1000, True) if case in ("generic_quarters", "off") else (200, 400, case != "no_belief")
    B = 330 * 32 - 21  # last tile holds 11 envs: its second half and its last two quarters are empty
    pool = pkg.generate_graph_pool(2, N, E, seed=0)
    env = pkg.BatchedScotlandYardEnv(B, 4, 15, graphs=pool, seed=31, auto_reset=True, tolls=1, belief=belief, reveal_interval=4,
                                     keep_reward64=True)
    env.set_option("tail_split", "off" if case == "off" else "on")
    cfg = so.OracleConfig(num_police=4, agent_money=15, toll=1, belief=belief, reveal_interval=4)
    gid = ((np.arange(B) // 32) % 2).astype(np.int32)
    ob = oc.CBatch(cfg, pool, B, seed=31, auto_reset=True, threads=_threads(), graph_id=gid)
    _rollout_against_oracle(env, ob, 8, belief, dense_every=1)
    env.close()


def test_two_handles_of_different_shapes_coexist(torch_cuda):
    """A large belief env, then a small env created next to it, then the first one stepped again: the observe kernel's
    dynamic shared-memory attribute is per function, not per handle (round-1 advisor finding)."""
    big, ob = _pair(200, 400, 6, 20, 2048, 9, toll=1, belief=True, reveal=5)
    big.reset()
    import student_mechanism_design_b200 as pkg

    small = pkg.BatchedScotlandYardEnv(1, 2, 10, graph_nodes=15, graph_edges=20, seed=0)
    small.reset()
    small.step(small.sample_actions())
    for s in range(3):
        acts = big.sample_actions(step_counter=s)
        big.step(acts)
        want = ob.step(acts.cpu().numpy())
        _compare(big, ob, want, True, ("big after small", s))
    small.step(small.sample_actions())
    big.close()
    small.close()
