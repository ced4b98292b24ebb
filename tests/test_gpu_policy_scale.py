"""The policy kernels (include/sy_policy.h) against the batched float64 oracles of oracle/policy_oracle.py at the sizes
where they take their other branches: config 5 as bench.py builds it (131 072 envs, so the persistent GNN warps walk
many envs and every tensor-core MAPPO CTA many double-buffered tiles), both sides of every MAPPO dispatch boundary
(tensor cores / CUDA cores, the shared-memory edge, the valid-move limit of the tensor-core epilogue), the staged and
the recomputing dense GNN kernel, a second Philox block of the masked sampler, the critic at its sizes, canary bands
around every policy output, and shard invariance.

Probabilities are compared per row against a bound derived from that row's own magnitudes (see `LOGIT_C`); the few
cases accepted only by a rounding band are counted, must stay rare, and are printed with the largest error-to-bound
ratio (pytest -s)."""
import ctypes as C

import numpy as np
import pytest

from oracle import policy_oracle as po

pytestmark = pytest.mark.gpu
U = 2.0 ** -24            # float32 unit roundoff
Q_TOL = 2e-5              # dense GNN Q: fp32 kernel (fast tanh) vs float64 oracle, as in test_gpu_policy.py
BAND_RATE = 1e-4          # rows that only a rounding band accepts, at most this share of the rows checked
C5 = dict(N=200, E=400, P=6, money=20, toll=1, belief=True, reveal=5)  # bench.py's config 5


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return torch


def _pkg():
    import student_mechanism_design_b200 as pkg

    return pkg


def _sms(torch):
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _np(t):
    return t.detach().cpu().numpy()


class Bands:
    """bookkeeping of the cases only a rounding band accepted"""

    def __init__(self, label):
        self.label, self.rows, self.banded, self.ratio, self.ties = label, 0, 0, 0.0, 0

    def add(self, rows, banded, ratio=0.0):
        self.rows += int(rows)
        self.banded += int(banded)
        self.ratio = max(self.ratio, float(ratio))

    def finish(self):
        print(f"[{self.label}] rows {self.rows}, accepted by a band {self.banded}, exact ties {self.ties}, "
              f"max error / bound {self.ratio:.3g}")
        assert self.banded <= BAND_RATE * self.rows + 1, (self.label, self.banded, self.rows)
        assert self.ratio <= 1.0


def _c5_env(pkg, B, env_offset=0, rollout=6):
    env = pkg.BatchedScotlandYardEnv(B, C5["P"], C5["money"], graph_nodes=C5["N"], graph_edges=C5["E"], seed=0, tolls=C5["toll"],
                                     belief=C5["belief"], reveal_interval=C5["reveal"], auto_reset=True, env_offset=env_offset)
    env.reset()
    env.rollout_random(rollout)  # spread the agents, spend budgets, hide MrX in most envs
    if env.observations_pending:
        env.flush_observations()
    return env


def _trainer_obs(pos, D):
    """MappoTrainer's observation (mappo_trainer.py:171-199) as the kernel builds it for obs=None"""
    B, A = pos.shape
    obs = np.zeros((B, A, D))
    obs[:, 0, 0] = pos[:, 0]
    obs[:, 1:, : A - 1] = pos[:, None, 1:]
    return obs


# ----------------------------------------------------------------------------------------------- MAPPO checking
# c of the per-row logit error bound LOGIT_C * 2^-24 * scale (scale: po.mappo_forward_batched, the largest sum of
# magnitudes any logit of the row is computed from).  4 of it covers the exponent's argument: logit - max and its
# product with log2 e are rounded, |argument| <= 2 scale.  8 covers the two layers themselves.  Every fp32 FMA
# rounds by at most u of its partial sum, and 3xTF32 adds at most 2^-21 of each product (the dropped A_lo B_lo and
# the tf32 rounding of lo); those errors have independent signs, so they add up to a few u * sum|terms| however long
# the chains are (H, D), and sum|terms| <= scale.
LOGIT_C = 12.0


def _check_mappo(pol, obs, mask, runs, step, bands, label=""):
    """every (env, agent) row of MappoPolicy.act runs {name: (actions, log_probs, probs)} against
    po.mappo_forward_batched: probabilities within the row's bound (either mode where Sv is within its own error of
    1e-8), masked-out nodes exactly 0, the action drawn again from the kernel's own probabilities with a sequential
    float32 CDF, the log-probability of that action"""
    B, A, N = mask.shape
    e = pol.env
    env_ids = e.env_offset + np.arange(B)
    r = po.philox4x32_batched(env_ids[:, None], step, po.RNG_MAPPO_POLICY, np.arange(A)[None, :], e.seed)
    u = po.u01_batched(r[0])
    for a in range(A):
        sd = {k: _np(v) for k, v in pol.policies[pol.policy_of_agent[a]].items()}
        o = po.mappo_forward_batched(obs[:, a], sd, mask[:, a])
        for name, (acts, lp, probs) in runs.items():
            _check_mappo_agent(o, mask[:, a], u[:, a], acts[:, a], lp[:, a], probs[:, a], bands, f"{label} {name} agent {a}")


def _check_mappo_agent(o, m, u, ak, lp, got, bands, label):
    B, N = m.shape
    rows = np.arange(B)
    # softmax restricted to the mask, p_n = e_n / sum_mask e_m: twice the logit error, plus a few roundings of its own
    rel = 2.0 * LOGIT_C * U * o["scale"] + 16 * U
    bound = o["probs"] * rel[:, None] + 1e-9
    err = np.abs(got - o["probs"])
    row_ok = (err <= bound).all(1)
    nv = m.sum(1)
    # Sv within its own error of the 1e-8 threshold: the kernel may take the other branch (softmax <-> uniform)
    amb = np.nonzero((np.abs(o["Sv"] - 1e-8) <= o["Sv"] * rel) & (nv > 0))[0]
    alt_ok = np.zeros(B, dtype=bool)
    if len(amb):
        alt = np.where(o["mode"][amb, None] == po.MAPPO_SOFTMAX, m[amb] / nv[amb, None], o["masked"][amb])
        alt_ok[amb] = (np.abs(got[amb] - alt) <= alt * rel[amb, None] + 1e-9).all(1)
    bad = np.nonzero(~row_ok & ~alt_ok)[0]
    assert len(bad) == 0, (label, "probs", int(bad[0]), int(o["mode"][bad[0]]), float(o["scale"][bad[0]]),
                           float((err[bad[0]] / bound[bad[0]]).max()))
    bands.add(B, (~row_ok).sum(), (err / bound)[row_ok].max() if row_ok.any() else 0.0)
    assert (got[(o["mode"] != po.MAPPO_UNIFORM_ALL)[:, None] & ~m] == 0).all(), (label, "mass outside the mask")
    # the draw again, from the kernel's own probabilities: sequential float32 CDF in ascending node order (adding the
    # zeros of masked-out nodes leaves it unchanged), thr = u * total; either neighbour within 2 ulp of a boundary
    assert ((ak >= 0) & (ak < N)).all(), (label, "action range")
    cum = np.cumsum(got, axis=1, dtype=np.float32)
    total = cum[:, -1]
    thr = u * total
    pk = got[rows, ak]
    prev = np.where(ak > 0, cum[rows, np.maximum(ak - 1, 0)], np.float32(0))
    cur = cum[rows, ak]
    last = N - 1 - np.argmax(got[:, ::-1] > 0, axis=1)
    uniform_all = (got > 0).all(1)  # no node is its own neighbour: a full support is the uniform-over-all branch
    exact = np.where(uniform_all, ak == np.minimum((u * np.float32(N)).astype(np.int64), N - 1),
                     (pk > 0) & (((prev <= thr) & (thr < cur)) | ((thr >= total) & (ak == last))))
    slack = 2 * np.spacing(thr)
    near = ~uniform_all & (pk > 0) & (prev - slack <= thr) & (thr < cur + slack)
    bad = np.nonzero(~exact & ~near)[0]
    assert len(bad) == 0, (label, "sample", int(bad[0]), int(ak[bad[0]]), float(thr[bad[0]]))
    bands.add(0, (~exact).sum())
    want_lp = np.log(np.clip(pk.astype(np.float64) / got.sum(1, dtype=np.float64), np.finfo(np.float32).eps,
                             1 - np.finfo(np.float32).eps))
    np.testing.assert_allclose(lp, want_lp, rtol=1e-5, atol=2e-6, err_msg=f"{label} log-prob")


def _mappo_run(pol, obs_t, step, tc):
    pol.tensor_cores = tc
    acts, lp, probs = pol.act(obs_t, step_counter=step, return_probs=True)
    pol.check()
    return _np(acts), _np(lp), _np(probs)


def test_mappo_config5_both_kernels_match_the_oracle(torch_cuda):
    """config 5 exactly as bench.py runs MAPPO (obs=None: raw node ids, logits in the hundreds) at 131 072 envs, a ragged
    last tile, and the size at which exactly one CTA per agent takes a second, partial tile"""
    torch = torch_cuda
    pkg = _pkg()
    A = C5["P"] + 1
    sizes = [131072, 131072 - 77, 128 * (_sms(torch) // A + 1) - 5]
    for B in sizes:
        env = _c5_env(pkg, B)
        pol = pkg.MappoPolicy(env, obs_size=A, hidden_size=64, seed=0)
        mask = _np(env.action_mask)
        obs = _trainer_obs(_np(env.pos).astype(np.int64), A)
        bands = Bands(f"mappo c5 B={B}")
        runs = {f"tc={tc}": _mappo_run(pol, None, 21, tc) for tc in (True, False)}
        _check_mappo(pol, obs, mask, runs, 21, bands, f"B={B}")
        del runs
        bands.finish()
        env.close()


# ----------------------------------------------------------------------------------------------- GNN checking
def _gnn_with_biases(pkg, torch, env, features, seed=5):
    """non-zero conv biases: with the default zeros, the constant row of an untouched node is 0 for both models and a
    mix-up of the two models' rows goes unseen"""
    pol = pkg.GNNPolicy(env, features=features, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    for sd in pol.state:
        sd["conv1.bias"] = torch.randn(pol.K, generator=gen) * 0.3
        sd["conv2.bias"] = torch.randn(pol.K, generator=gen) * 0.3
    pol._pack()
    return pol


def _gnn_oracle(env, pol, mode):
    pos, rev, gid = _np(env.pos).astype(np.int64), _np(env.mrx_revealed), _np(env.graph_id)
    sds = [{k: _np(v) for k, v in s.items()} for s in pol.state]
    return po.gnn_forward_batched(mode, pos, rev, gid, [g.edge_links for g in env.graphs], sds, env.graph_nodes)


def _check_gnn_act(pol, want_q, mask, eps, step, bands, label):
    e = pol.env
    B, A, N = mask.shape
    acts, qt = pol.act(eps[0], eps[1], step_counter=step, return_q=True)
    acts, qt = _np(acts), _np(qt)
    explored, ex_act = po.gnn_explore_batched(mask, eps[0], eps[1], e.seed, e.env_offset + np.arange(B), step)
    rows = np.arange(B)
    for a in range(A):
        qa, m, ak = want_q[:, 0 if a == 0 else 1], mask[:, a], acts[:, a]
        nomove = ~m.any(1)
        assert (ak[nomove] == -1).all() and np.isnan(qt[nomove, a]).all(), (label, a)
        ex = explored[:, a]
        assert (ak[ex] == ex_act[ex, a]).all() and np.isnan(qt[ex, a]).all(), (label, "explore", a)
        gr = ~ex & ~nomove
        best = np.where(m, qa, -np.inf).max(1)
        akc = np.clip(ak, 0, N - 1)
        ok = m[rows, akc] & (qa[rows, akc] >= best - 2 * Q_TOL)
        bad = np.nonzero(gr & ~(ok & (ak >= 0)))[0]
        assert len(bad) == 0, (label, "greedy", a, int(bad[0]), int(ak[bad[0]]), float(best[bad[0]]))
        assert (np.abs(qt[gr, a] - qa[gr, akc[gr]]) <= Q_TOL).all(), (label, "q_taken", a)
        # a greedy choice other than the oracle's first argmax is accepted by the tie band; where the two Q values are
        # equal in float64 too (nodes whose 2-hop neighbourhoods look alike) it is a tie, not a rounding case
        other = gr & (ak != np.where(m, qa, -np.inf).argmax(1))
        tie = other & (best - qa[rows, akc] <= 1e-12 * np.maximum(1.0, np.abs(best)))
        bands.add(gr.sum(), (other & ~tie).sum())
        bands.ties += int(tie.sum())
    return explored


def test_gnn_config5_dense_q_and_actions_match_the_oracle(torch_cuda):
    """config 5 at 131 072 envs (every warp of the persistent kernels walks ~18 envs) and a ragged size, both feature
    modes: dense Q against the oracle, epsilon-greedy actions in the oracle's tie set, q_taken, exploration exact"""
    torch = torch_cuda
    pkg = _pkg()
    full = _c5_env(pkg, 131072)
    ragged = _c5_env(pkg, 131072 - 77)
    for k in ("pos", "money", "mrx_revealed", "graph_id"):  # the ragged handle is a prefix of the full one
        assert torch.equal(getattr(ragged, k), getattr(full, k)[: ragged.num_envs]), k
    # the oracle's env-mode features are the env's node_features
    rng = np.random.default_rng(0)
    sample = rng.choice(full.num_envs, 64, replace=False)
    x = po.graph_features_batched(po.FEATURES_ENV, _np(full.pos)[sample], _np(full.mrx_revealed)[sample], full.graph_nodes,
                                  full.num_agents)
    np.testing.assert_array_equal(x, _np(full.node_features[torch.from_numpy(sample).cuda()]).astype(np.float64))
    rev = _np(full.mrx_revealed)
    assert (rev < 0).any() and (rev >= 0).any()
    for features, mode in (("env", po.FEATURES_ENV), ("reference", po.FEATURES_REFERENCE)):
        want = _gnn_oracle(full, _gnn_with_biases(pkg, torch, full, features), mode)
        for env in (full, ragged):
            pol = _gnn_with_biases(pkg, torch, env, features)
            B = env.num_envs
            q = _np(pol.q_values())
            err = np.abs(q - want[:B]).max()
            print(f"[gnn c5 {features} B={B}] max |q - oracle| {err:.3g}")
            assert err <= Q_TOL, (features, B, err)
            mask = _np(env.action_mask)
            bands = Bands(f"gnn c5 {features} B={B}")
            for eps, step in (((0.0, 0.0), 3), ((0.05, 0.05), 4), ((1.0, 1.0), 5)):
                explored = _check_gnn_act(pol, want[:B], mask, eps, step, bands, f"{features} B={B} eps={eps}")
                has = mask.any(-1)
                assert (explored == has).all() if eps == (1.0, 1.0) else (not explored.any() if eps == (0.0, 0.0) else explored.any())
            bands.finish()
    full.close()
    ragged.close()


# ----------------------------------------------------------------------------------------------- MAPPO dispatch
def _tc_expected(N, H, D, max_degree):
    """sy_mappo_act's tensor-core envelope restated from include/sy_policy.h / tc_shape"""
    Kp, Np = (H + 7) & ~7, (N + 15) & ~15
    floats = 2 * 128 * Kp + 2 * Np * Kp + 2 * 128 * D + Np + 128 * 32 + 128 * 16 + 2 * 128 * 8 + 2 * 128 * 4 + Kp * (D + 1)
    return 1 <= max_degree <= 16 and 16 <= N <= 256 and H <= 64 and D <= 16 and floats * 4 + 64 <= 220 * 1024


def _hub_graph(pkg, N, hub_nbrs):
    """node 0 adjacent to exactly `hub_nbrs`; nodes 1..N-1 form a chain (degree <= 3)"""
    links = [(0, int(n)) for n in hub_nbrs] + [(i, i + 1) for i in range(1, N - 1)]
    return pkg.GraphSpec(N, np.asarray(links), np.ones(len(links), dtype=np.int64))


SWEEP = ([(n, 32, 7, None) for n in (15, 16, 17, 255, 256, 257, 300, 809)]
         + [(50, h, 7, None) for h in (1, 8, 9, 63, 64, 65, 96, 128, 512)]
         + [(50, 32, d, None) for d in (1, 16, 17, 40)]
         + [(208, 64, 7, None), (209, 64, 7, None), (256, 48, 16, None), (256, 56, 16, None)]
         + [(64, 32, 7, "hub16_low"), (64, 32, 7, "hub16_split"), (64, 32, 7, "hub17")])
HUBS = {"hub16_low": list(range(1, 17)), "hub16_split": list(range(1, 9)) + list(range(40, 48)), "hub17": list(range(1, 18))}


@pytest.mark.parametrize("N,H,D,hub", SWEEP)
def test_mappo_dispatch_sweep(torch_cuda, N, H, D, hub):
    """each shape on both settings at several tiles with a ragged tail: outside the tensor-core envelope both settings
    run the CUDA-core kernel (bit-identical); inside, both match the oracle and differ in some bits (3xTF32 vs FMA)"""
    torch = torch_cuda
    pkg = _pkg()
    P, B = 3, 4 * 128 + 37
    if hub is None:
        env = pkg.BatchedScotlandYardEnv(B, P, 20, graph_nodes=N, graph_edges=(3 * N) // 2, num_graphs=2, seed=3, tolls=1, auto_reset=True)
        env.reset()
        env.rollout_random(4)
        if env.observations_pending:
            env.flush_observations()
    else:
        env = pkg.BatchedScotlandYardEnv(B, P, 40, graphs=[_hub_graph(pkg, N, HUBS[hub])], seed=3)
        init = np.tile(np.asarray([[30, 0, 50, 60]], dtype=np.int32), (B, 1))
        init[::3, 0] = 0  # MrX on the hub too in a third of the envs
        env.reset(init_pos=init)
        assert int(env.action_mask[:, 1].sum(-1).min()) == len(HUBS[hub])
    pol = pkg.MappoPolicy(env, obs_size=D, hidden_size=H, seed=7)
    pol._graphs()
    tc = _tc_expected(N, H, D, pol._tables.max_degree)
    if hub is not None:
        assert tc == (hub != "hub17")
    obs_t = torch.randn(B, P + 1, D, generator=torch.Generator().manual_seed(N * 1000 + H * 10 + D)).cuda()
    obs, mask = _np(obs_t).astype(np.float64), _np(env.action_mask)
    bands = Bands(f"mappo N={N} H={H} D={D} {hub or ''}")
    runs = {use_tc: _mappo_run(pol, obs_t, 5, use_tc) for use_tc in (True, False)}
    _check_mappo(pol, obs, mask, runs, 5, bands)
    bands.finish()
    same = all(np.array_equal(x, y) for x, y in zip(runs[True], runs[False]))
    assert same != tc, f"tensor-core kernel expected: {tc}, outputs bit-identical: {same}"
    if H == 64 and D == 7 and hub is None:  # unit-scale observations at the shipped hidden size: no looser than 3e-5
        sd = {k: _np(v) for k, v in pol.policies[0].items()}
        scale = po.mappo_forward_batched(obs[:, 0], sd, mask[:, 0])["scale"]
        assert (2 * LOGIT_C * U * scale + 16 * U).max() <= 3e-5
    env.close()


def test_mappo_above_the_shared_memory_limit_fails_cleanly(torch_cuda):
    """H = 64, D = 7: N = 809 is the last node count the CUDA-core kernel holds; N = 810 is a clean SyError, after which
    the library and the env still work"""
    torch = torch_cuda
    pkg = _pkg()
    B, P, N = 300, 3, 810
    env = pkg.BatchedScotlandYardEnv(B, P, 20, graph_nodes=N, graph_edges=(3 * N) // 2, seed=3, tolls=1)
    env.reset()
    big = pkg.MappoPolicy(env, obs_size=7, hidden_size=64, seed=1)
    obs_t = torch.randn(B, P + 1, 7, generator=torch.Generator().manual_seed(0)).cuda()
    for tc in (True, False):
        big.tensor_cores = tc
        with pytest.raises(pkg.SyError, match="shared memory"):
            big.act(obs_t)
    small = pkg.MappoPolicy(env, obs_size=7, hidden_size=32, seed=1)
    bands = Bands("mappo after the error")
    _check_mappo(small, _np(obs_t).astype(np.float64), _np(env.action_mask), {"cuda cores": _mappo_run(small, obs_t, 2, False)}, 2,
                 bands)
    bands.finish()
    env.step(env.sample_actions())
    torch.cuda.synchronize()
    env.close()


# ----------------------------------------------------------------------------------------------- GNN shapes
@pytest.mark.parametrize("P,N", [(2, 960), (2, 961), (6, 533), (6, 534), (15, 282), (15, 283), (6, 1000)])
def test_gnn_staged_and_recompute_paths(torch_cuda, P, N):
    """K = 3 / 7 / 16 (KP 4 / 8 / 16) at the last node count whose layer-1 rows the dense kernel stages and one above
    (recompute per node), plus 1 000 nodes; a pool of 3 graphs, one with a parallel edge; enough envs that every warp
    of the persistent kernels takes more than one"""
    torch = torch_cuda
    pkg = _pkg()
    B = 8 * 6 * _sms(torch) + 99
    pool = pkg.generate_graph_pool(3, N, N + N // 4, seed=N)
    links = pool[2].edge_links.copy()
    links[-1] = links[0][::-1] if N % 2 else links[0]  # a parallel (or reversed) copy of an edge: two GCN messages
    pool[2] = pkg.GraphSpec(N, links, pool[2].edges)
    env = pkg.BatchedScotlandYardEnv(B, P, 20, graphs=pool, seed=4, tolls=1, reveal_interval=3, auto_reset=True)
    env.reset()
    env.rollout_random(5)
    if env.observations_pending:
        env.flush_observations()
    assert len(np.unique(_np(env.graph_id))) == 3
    features = "env" if N % 2 == 0 else "reference"
    mode = po.FEATURES_ENV if features == "env" else po.FEATURES_REFERENCE
    pol = _gnn_with_biases(pkg, torch, env, features)
    want = _gnn_oracle(env, pol, mode)
    q = _np(pol.q_values())
    err = np.abs(q - want).max()
    print(f"[gnn P={P} N={N}] max |q - oracle| {err:.3g}")
    assert err <= Q_TOL, err
    bands = Bands(f"gnn P={P} N={N}")
    _check_gnn_act(pol, want, _np(env.action_mask), (0.05, 0.1), 8, bands, f"N={N}")
    bands.finish()
    env.close()


# ----------------------------------------------------------------------------------------------- masked_sample, critic
@pytest.mark.parametrize("N", [129, 200, 1000])
def test_masked_sample_second_philox_block(torch_cuda, N):
    """N > 128: lanes take a second Philox block.  Greedy == first argmax over the legal nodes; sampling == Gumbel-max
    with the documented noise, recomputed on the CPU for every row"""
    torch = torch_cuda
    _pkg()
    from student_mechanism_design_b200.rollout import masked_sample, masked_sample_device

    g = torch.Generator().manual_seed(N)
    B, A = 64, 5
    logits = torch.randn(B, A, N, generator=g) * 2
    mask = torch.rand(B, A, N, generator=g) < 0.3
    mask[0, 1] = False
    mask[2, 3] = False
    mask[2, 3, N - 1] = True  # the only legal node in the last block
    greedy = masked_sample_device(logits.cuda(), mask.cuda(), greedy=True).cpu()
    assert torch.equal(greedy, masked_sample(logits, mask, greedy=True)) and greedy[0, 1] == -1 and greedy[2, 3] == N - 1
    seed, step, off = (3 << 32) | 77, 6, 50
    got = _np(masked_sample_device(logits.cuda(), mask.cuda(), seed=seed, step_counter=step, env_offset=off))
    j = np.arange(N)
    r = po.philox4x32_batched((off + np.arange(B))[:, None, None], step, 5 + 16 * np.arange(A)[None, :, None], (j >> 2)[None, None, :],
                              seed)
    words = np.choose(j & 3, r)
    uu = ((words >> 8).astype(np.float64) + 0.5) / 16777216.0
    keys = np.where(mask.numpy(), logits.numpy().astype(np.float64) - np.log(-np.log(uu)), -np.inf)
    legal = mask.numpy().any(-1)
    assert (got[~legal] == -1).all() and (got[legal] >= 0).all()
    gk = np.take_along_axis(keys, np.clip(got, 0, N - 1)[..., None], -1)[..., 0]
    assert (gk[legal] >= keys.max(-1)[legal] - 1e-4).all()
    assert (got[legal] >= 128).any()  # the second block does win rows


@pytest.mark.parametrize("M,D,H", [(131072 + 77, 49, 64), (1003, 797, 64)])
def test_critic_at_scale_and_at_its_shared_memory_limit(torch_cuda, M, D, H):
    torch = torch_cuda
    pkg = _pkg()
    env = pkg.BatchedScotlandYardEnv(8, 2, 10, graph_nodes=20, graph_edges=30, seed=1)
    env.reset()
    pol = pkg.MappoPolicy(env, obs_size=3, hidden_size=H, global_obs_size=D, seed=3)
    x = torch.randn(M, D, generator=torch.Generator().manual_seed(M)).cuda()
    v = _np(pol.values(x)).astype(np.float64)
    want, scale = po.critic_value_batched(_np(x), {k: _np(t) for k, t in pol.critic.items()})
    ratio = np.abs(v - want) / (LOGIT_C * U * scale)
    print(f"[critic M={M} D={D}] max error / bound {ratio.max():.3g}")
    assert ratio.max() <= 1.0
    if D == 797:  # one more input column no longer fits the kernel's shared memory
        big = pkg.MappoPolicy(env, obs_size=3, hidden_size=H, global_obs_size=D + 1, seed=3)
        with pytest.raises(pkg.SyError, match="shared memory"):
            big.values(torch.zeros(4, D + 1, device="cuda"))
        np.testing.assert_array_equal(_np(pol.values(x)), v.astype(np.float32))
    env.close()


# ----------------------------------------------------------------------------------------------- guard bands
GUARD = 4096


class Guarded:
    """an output tensor carved out of the middle of its own allocation, 4 KB canary bands on each side"""

    def __init__(self, torch, shape, dtype):
        self.nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        self.raw = torch.full((2 * GUARD + self.nbytes,), 0xA5, dtype=torch.uint8, device="cuda")
        self.t = self.raw[GUARD: GUARD + self.nbytes].view(dtype).view(*shape)

    @property
    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        import torch

        torch.cuda.synchronize()
        assert bool((self.raw[:GUARD] == 0xA5).all()) and bool((self.raw[GUARD + self.nbytes:] == 0xA5).all()), what


def test_policy_outputs_stay_inside_their_buffers(torch_cuda):
    """every policy kernel through the C ABI with each output between canary bands, at ragged sizes where the last tile,
    warp pass or block is partial; the guarded outputs equal the ones of the Python API bit for bit"""
    torch = torch_cuda
    pkg = _pkg()
    from student_mechanism_design_b200 import _policy_cabi as pc

    lib = pc.load_library()
    B = 8 * 6 * _sms(torch) + 99
    env = _c5_env(pkg, B)
    A, N, s = env.num_agents, env.graph_nodes, env._stream()
    gnn = _gnn_with_biases(pkg, torch, env, "env")
    q = Guarded(torch, (B, 2, N), torch.float32)
    pc.check(lib.sy_gnn_q_values(C.byref(gnn._graphs()), C.byref(gnn._state()), gnn.params.data_ptr(), gnn.K, gnn.conv_epsilon,
                                 gnn.feature_mode, q.ptr, s))
    q.check("sy_gnn_q_values")
    assert torch.equal(q.t, gnn.q_values())
    acts, qt = Guarded(torch, (B, A), torch.int64), Guarded(torch, (B, A), torch.float32)
    pc.check(lib.sy_gnn_act(C.byref(gnn._graphs()), C.byref(gnn._state()), gnn.params.data_ptr(), gnn.K, gnn.conv_epsilon,
                            gnn.feature_mode, 0.1, 0.1, env.seed, 3, acts.ptr, qt.ptr, s))
    acts.check("sy_gnn_act actions")
    qt.check("sy_gnn_act q_taken")
    a_ref, q_ref = gnn.act(0.1, 0.1, step_counter=3, return_q=True)
    assert torch.equal(acts.t, a_ref) and torch.equal(torch.nan_to_num(qt.t, 7.0), torch.nan_to_num(q_ref, 7.0))
    mp = pkg.MappoPolicy(env, obs_size=A, hidden_size=64, seed=0)
    for tc in (True, False):
        mp.tensor_cores = tc
        g = mp._graphs()
        acts, lp, pr = Guarded(torch, (B, A), torch.int64), Guarded(torch, (B, A), torch.float32), Guarded(torch, (B, A, N), torch.float32)
        pc.check(lib.sy_mappo_act(C.byref(g), C.byref(mp._state()), None, mp.obs_size, mp.hidden, mp.params.data_ptr(),
                                  mp.policy_of_agent.ctypes.data, mp._tables.max_degree if tc else 0, env.seed, 9, acts.ptr,
                                  lp.ptr, pr.ptr, s))
        mp.check()
        for t, what in ((acts, "actions"), (lp, "log_probs"), (pr, "probs")):
            t.check(f"sy_mappo_act tc={tc} {what}")
        ref = mp.act(None, step_counter=9, return_probs=True)
        assert all(torch.equal(x.t, y) for x, y in zip((acts, lp, pr), ref)), tc
    crit = pkg.MappoPolicy(env, obs_size=A, hidden_size=64, global_obs_size=49, seed=0)
    M = 131072 + 77
    x = torch.randn(M, 49, generator=torch.Generator().manual_seed(1)).cuda()
    v = Guarded(torch, (M,), torch.float32)
    pc.check(lib.sy_mappo_values(x.data_ptr(), M, 49, 64, crit.critic_params.data_ptr(), v.ptr, s))
    v.check("sy_mappo_values")
    assert torch.equal(v.t, crit.values(x))
    for n in (129, 1000):
        rows_b, rows_a = 37, 3
        logits = torch.randn(rows_b, rows_a, n, generator=torch.Generator().manual_seed(n)).cuda()
        mask = (torch.rand(rows_b, rows_a, n, generator=torch.Generator().manual_seed(n + 1)) < 0.2).cuda()
        for greedy in (1, 0):
            out = Guarded(torch, (rows_b, rows_a), torch.int64)
            pc.check(lib.sy_masked_sample(logits.data_ptr(), mask.data_ptr(), rows_b, rows_a, n, 0, 11, 2, greedy, out.ptr, s))
            out.check(f"sy_masked_sample N={n} greedy={greedy}")
    env.close()


# ----------------------------------------------------------------------------------------------- shard invariance
def test_policy_actions_are_shard_invariant(torch_cuda):
    """two handles at env_offset 0 and 1 237 (not a multiple of 8 or 128) pick exactly the actions of the matching rows
    of one handle over the whole batch: GNN with exploration, MAPPO on both kernels"""
    torch = torch_cuda
    pkg = _pkg()
    B, cut = 8 * 6 * _sms(torch) + 99, 1237
    full = _c5_env(pkg, B)
    shards = [_c5_env(pkg, cut), _c5_env(pkg, B - cut, env_offset=cut)]
    parts = [slice(0, cut), slice(cut, B)]
    for sh, sl in zip(shards, parts):
        assert torch.equal(sh.pos, full.pos[sl]) and torch.equal(sh.money, full.money[sl])
    for eps in ((0.2, 0.3), (0.0, 0.0)):
        ref = pkg.GNNPolicy(full, seed=9).act(*eps, step_counter=12)
        for sh, sl in zip(shards, parts):
            assert torch.equal(pkg.GNNPolicy(sh, seed=9).act(*eps, step_counter=12), ref[sl]), eps
    A = full.num_agents
    for tc in (True, False):
        mp = pkg.MappoPolicy(full, obs_size=A, hidden_size=64, seed=0)
        mp.tensor_cores = tc
        ref = mp.act(None, step_counter=13)[0]
        for sh, sl in zip(shards, parts):
            ms = pkg.MappoPolicy(sh, obs_size=A, hidden_size=64, seed=0)
            ms.tensor_cores = tc
            assert torch.equal(ms.act(None, step_counter=13)[0], ref[sl]), tc
    for e in [full, *shards]:
        e.close()
