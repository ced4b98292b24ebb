"""Belief map, one kernel step at a time, against the float64 batched oracle (oracle/belief_oracle.py).

Teacher forcing: before each step the device's own belief row is read (float32 -> float64); after it, every row is
compared with `belief_step_batched` applied to that row, with the operation each env took (derived from the device state
before and after the step, or from the C oracle stepping alongside where the device state is not observable):

* exact rows: KEEP rows are bit-identical to their input, DELTA rows are exactly 1.0 at MrX's node and 0 elsewhere,
  UNIFORM rows (and propagated all-zero rows) are exactly float32(1) / float32(N);
* exact support: a propagated entry is 0 iff the oracle's is (entries below 2^-100 are only held to that absolute bound);
* per-entry relative bound |got - want| <= rho * want, with rho from the rounding model (`rho` below), not fitted.

Coverage: the three propagation paths of sy_env.cu (the lane = env fast path `belief_role`, the warp-per-env gather over
the CSR the writer warps staged, and the warp-per-env gather over the padded global lists, on mixed-graph tiles and on
single-graph tiles above the staging limit), N on both sides of both dispatch boundaries of the host sizing rule
(restated in `belief_path`), hub graphs with degrees up to 255, isolated nodes 32-40 places into a fast-path warp's node
range, device-sampled pools, observation hints on every path, reveals, skipped reveals, auto-resets, frozen envs, rows
the caller wrote (zero, summing to 3.7, entries down to 1e-25), every launch form, c3 and c4 at full size, and the belief
cross-entropy per env through identity mechanism groups.  Where the C oracle runs alongside, the trajectory check of the
other GPU tests (1e-6 absolute, north_star) is kept as well."""
import math

import numpy as np
import pytest

import belief_oracle as bo
import sy_oracle as so
import sy_oracle_c as oc
from test_gpu_fullsize import BELIEF_TOL, _threads, torch_cuda  # noqa: F401

pytestmark = pytest.mark.gpu

U = 2.0 ** -24  # unit roundoff of float32 (round to nearest)
TINY = 2.0 ** -100  # oracle entries below this are held to an absolute bound of this size only
HUB_DEGREES = [0, 1, 3, 4, 5, 8, 9, 12, 13, 16, 17, 32, 33, 64, 255]
BEL_WARPS, GEN_BEL_WARPS = 8, 12  # belief warps of the fast / generic observe kernels (sy_env.cu SY_BEL_WARPS, GEN_BEL_WARPS)
WORST = {}  # case -> largest err / bound, printed at the end of each test


def belief_path(N, nnz_stride, A):
    """The host sizing rule of sy_env.cu (the belief / writer shared-memory plan after `sy_load_graphs`, "dynamic shared
    memory of the observe kernel's belief warps" through `bel_share_csr`), restated: which path a tile whose envs all
    share one graph takes.  "fast" (lane = env), "csr" (warp per env over the writers' staged CSR) or "global" (warp per
    env over the padded lists in global memory).  Tiles that mix graphs take "global" whatever this returns."""
    up16 = lambda x: (x + 15) & ~15  # noqa: E731
    TILE, BSTRIDE, BEL_JMAX, BULK_WARPS, MAXA, BUDGET = 32, 33, 128, 4, 16, 25344
    pack_stride = ((nnz_stride + 3 * N + 3) & ~3) + 4
    off_out = up16(N * BSTRIDE * 4)
    off_part = up16(2 * off_out)
    off_pack = up16(off_part + BEL_WARPS * 32 * 4)
    off_ptr = up16(off_pack + pack_stride * 8)
    fast = off_ptr + (N + 2) * 4
    bel_fast = fast <= 110 * 1024 and N <= BEL_WARPS * BEL_JMAX
    bw, wrw = (BEL_WARPS, 8) if bel_fast else (GEN_BEL_WARPS, 4)
    generic = bw * (N + 1) * 4
    bel_smem = fast if bel_fast and fast > generic else generic
    assert bel_smem <= 180 * 1024
    img_rows = 1 if A * N > 4096 else A
    img_stride = up16(img_rows * N + 16)
    base_lsu = (2 * TILE * A + 2 * TILE + wrw * MAXA) * 4 + wrw * img_stride
    nbw = min(wrw, BULK_WARPS)

    def plan_bulk_chunk(S, cap, w):
        g = 16
        while S % g:
            g >>= 1
        m = 16 // g
        group = S * m
        cap &= ~15
        if group <= cap:
            return group * min(cap // group, max(1, (TILE // m) // (2 * w)))
        for c in range(cap, max(cap // 2, 16) - 1, -16):
            if group % c == 0:
                return c
        return cap

    c_mask = plan_bulk_chunk(A * N, max(256, BUDGET // (2 * nbw + 1)), nbw)
    base = max(base_lsu, (2 * TILE * A + 2 * TILE) * 4 + (2 * nbw + 1) * c_mask)
    share = not bel_fast
    csr_core = ((((N + 1) * 4 + nnz_stride * 3) + 3) & ~3) + (N * 6 if share else 0)
    off_pad = up16(csr_core)
    csr = (off_pad + (((N + 1 + 3) & ~3) + pack_stride) * 2 if share else csr_core) + 16
    off_csr = up16(up16(bel_smem) + base)
    stage = csr <= 48 * 1024 and pack_stride < 65536 and off_csr + csr <= 200 * 1024
    return "fast" if bel_fast else ("csr" if stage else "global")


def _nnz_stride(pool):
    return max(1, max(int(so.Graph(g.num_nodes, g.edge_links, g.edges).csr()[0][-1]) for g in pool))


def _boundary(E_per_N, A, kind):
    """smallest N at which the rule leaves the fast path ("fast") / stops staging the CSR ("csr") for E = E_per_N * N"""
    want = {"fast": "fast", "csr": "csr"}[kind]
    N = 64 if kind == "fast" else 400
    while belief_path(N, 2 * int(E_per_N * N), A) == want:
        N += 1
    return N


def rho(N, dmax, k=1):
    """Relative error bound of one propagated entry after k kernel steps with no observation in between.

    One step, in units of u = 2^-24: an entry is a sum of deg(j) <= d_max nonnegative products b_i * fl(1/deg i) (fma
    chains: d_max roundings, plus 1 for the rounded 1/deg; on the staged-CSR path the row is pre-scaled by
    fl(1/deg * 1/tot), 2 more, and summed with d_max additions), then multiplied by 1/tot (2 roundings) and, with a hint,
    by fl(0.1) and 1/hs (3 more): |theta_j| <= (d_max + 4) u.  The normaliser is the kernel's own sum of such entries
    (fast path: its error is the entries' plus the summation; generic path: the input row's sum, whose error is common
    to every entry of the row) -- another (d_max + 4) u from the entries plus the summation, a nonnegative sum of at
    most ceil(N / BW) + BW terms on the fast path (per-warp node range, then the BW partial sums), ceil(N / 32) + 5 on
    the warp-per-env paths and for the hint sum (per-lane strided sums, then a 5-level butterfly), so at most
    ceil(N / BW) + BW + 32 for either BW the kernels use.  Together rho_1 = (2 (d_max + 4) + gamma_sum) u, with
    gamma_sum = max_BW (ceil(N / BW) + BW) + 32 (first order; the products n u are < 1e-4, the second-order terms are
    below the slack of the constants).

    k steps: every factor of a normalisation is common to a whole row, and nonnegative linear maps do not expand the
    Hilbert projective metric (normalisation leaves it unchanged), so the per-entry errors of the k propagations add up
    and only the last normaliser counts: k * 2 (d_max + 4) u + gamma_sum u."""
    gamma_sum = max(math.ceil(N / bw) + bw for bw in (BEL_WARPS, GEN_BEL_WARPS)) + 32
    return (k * 2 * (dmax + 4) + gamma_sum) * U


def ce_bound(N, dmax, ce):
    """|device CE - oracle CE| at a scored reveal: CE = log S - log v_x (S the sum of the clipped entries of the
    propagated row, v_x the clipped entry at MrX's node).  v_x carries rho; S carries rho plus its own summation
    (ceil(N/32) + 5 terms, inside gamma_sum); logf is good to 1 ulp of log S and of log v_x (|log v_x| <= |ce| + |log S|,
    |log S| < 1e-4), the subtraction adds u |ce|, and the Q24 fixed point rounds to 2^-25.  Clipping at 1e-8 is
    1-Lipschitz in relative terms and float(1e-8) differs from 1e-8 by less than u relative."""
    return 2 * rho(N, dmax) + 4 * U * (np.abs(ce) + 1) + 2.0 ** -25


class Teacher:
    """Per-step checks of one env handle against belief_step_batched on the device's previous row."""

    def __init__(self, env, pool, name, *, reveal, auto_reset, ob=None):
        self.env, self.pool, self.name, self.ob = env, list(pool), name, ob
        self.reveal, self.auto_reset = reveal, auto_reset
        self.mats = [bo.propagation_matrix(g) for g in self.pool]
        self.dmax = np.asarray([bo.max_degree(g) for g in self.pool])
        self.N = env.graph_nodes
        self.ops = np.zeros(4, dtype=np.int64)
        WORST.setdefault(name, 0.0)

    def snap(self):
        e = self.env
        return dict(bel=e.belief_map.cpu().numpy().copy(), done=e.done.cpu().numpy().copy(),
                    episode=e.episode.cpu().numpy().copy(), gid=e.graph_id.cpu().numpy().copy())

    def op_after(self, before, reset_mask=None):
        e = self.env
        ri = self.reveal
        if e.mechanisms is not None:  # mechanism groups: each env's own reveal schedule
            ri = np.asarray([m["reveal_interval"] for m in e.mechanisms])[e.group_id.cpu().numpy()]
        return bo.op_from_transition(before["done"], before["episode"], e.episode.cpu().numpy(), e.mrx_revealed.cpu().numpy(),
                                     ri, self.auto_reset, reset_mask), e.pos[:, 0].cpu().numpy()

    def check(self, before, op, x, tag, hint=None, k=1, got=None):
        """compare the device's row now with one (k > 1: k unobserved) step(s) from `before`"""
        got = self.env.belief_map.cpu().numpy() if got is None else got
        prev32 = before["bel"]
        N = self.N
        self.ops += np.bincount(op, minlength=4)
        want = bo.belief_step_batched(prev32.astype(np.float64), self.pool, before["gid"], op, x, hint, mats=self.mats)
        keep = op == bo.KEEP
        assert np.array_equal(got[keep].view(np.uint32), prev32[keep].view(np.uint32)), (self.name, tag, "KEEP rows changed")
        d = np.nonzero(op == bo.DELTA)[0]
        onehot = np.zeros((len(d), N), np.float32)
        onehot[np.arange(len(d)), x[d]] = 1.0
        assert np.array_equal(got[d], onehot), (self.name, tag, "DELTA rows")
        unif = np.float32(1) / np.float32(N)
        zero_in = (op == bo.PROPAGATE) & ~prev32.any(axis=1)
        u = (op == bo.UNIFORM) | zero_in
        assert (got[u] == unif).all(), (self.name, tag, "UNIFORM rows", np.nonzero(u)[0][:5])
        p = np.nonzero((op == bo.PROPAGATE) & ~zero_in)[0]
        if not len(p):
            return
        g, w = got[p].astype(np.float64), want[p]
        small = w < TINY
        assert (np.abs(g[small] - w[small]) <= TINY).all(), (self.name, tag, "tiny entries")
        supp = (g == 0) != (w == 0)
        supp &= ~small | (w == 0)
        if supp.any():
            r, c = np.argwhere(supp)[0]
            raise AssertionError((self.name, tag, "support", int(p[r]), int(c), g[r, c], w[r, c]))
        bound = np.asarray([rho(N, dm, k) for dm in self.dmax])[before["gid"][p]][:, None] * w
        ratio = np.where(small, 0.0, np.abs(g - w) / np.where(bound > 0, bound, 1.0))
        worst = float(ratio.max())
        WORST[self.name] = max(WORST[self.name], worst)
        if worst > 1.0:
            r, c = np.unravel_index(int(ratio.argmax()), ratio.shape)
            raise AssertionError((self.name, tag, "relative bound", f"env {p[r]} node {c}: got {g[r, c]!r} want {w[r, c]!r} "
                                  f"err/bound {worst:.3g} (deg_max {self.dmax[before['gid'][p[r]]]})"))

    def trajectory(self, tag):
        if self.ob is not None:
            err = np.abs(self.env.belief_map.cpu().numpy().astype(np.float64) - self.ob.belief()).max()
            assert err <= BELIEF_TOL, (self.name, tag, "trajectory", err)
            assert np.array_equal(self.env.pos.cpu().numpy(), self.ob.pos()), (self.name, tag, "positions")

    def report(self):
        print(f"\n[belief] {self.name}: ops keep/uniform/delta/propagate = {self.ops.tolist()}, "
              f"largest err/bound {WORST[self.name]:.3g}")


def _env(pool_or_none, B, P, money, *, reveal, auto_reset=True, seed=1, belief_ce=False, options=(), gid=None, **kw):
    import student_mechanism_design_b200 as pkg

    env = pkg.BatchedScotlandYardEnv(B, P, money, graphs=pool_or_none, seed=seed, auto_reset=auto_reset, tolls=1,
                                     belief=True, belief_ce=belief_ce, reveal_interval=reveal, **kw)
    for k, v in options:
        env.set_option(k, v)
    env.reset(graph_id=None if gid is None else gid)
    return env


def _hint(torch, B, N, rng):
    """rows alternate random (30 % candidates), empty and all-ones hints"""
    h = (rng.random((B, N)) < 0.3).astype(np.uint8)
    h[1::3] = 0
    h[2::3] = 1
    return torch.from_numpy(h).cuda()


def _write_rows(torch, env, rng):
    """caller-written input rows: zero, scaled to sum to 3.7, entries spanning 1e-25 .. 1 (a fifth of them 0)"""
    B, N = env.belief_map.shape
    bel = env.belief_map.cpu().numpy()
    bel[1::7] = 0.0
    bel[2::7] *= np.float32(3.7)
    n3 = len(bel[3::7])
    tiny = (10.0 ** rng.uniform(-25, 0, size=(n3, N))).astype(np.float32)
    tiny[rng.random((n3, N)) < 0.2] = 0.0
    bel[3::7] = tiny
    env.belief_map.copy_(torch.from_numpy(bel))


def _drive(torch, t, steps, *, hints=False, rows=False, resets=False, seed=0):
    """plain steps with the per-step check; optional hints (odd steps), caller-written rows (every third step) and a
    partial reset through the reset kernel (step 4)"""
    env = t.env
    rng = np.random.default_rng(seed)
    for s in range(steps):
        if rows and s % 3 == 1:
            _write_rows(torch, env, rng)
        if resets and s == 4:
            before = t.snap()
            mask = np.zeros(env.num_envs, bool)
            mask[::5] = True
            env.reset(reset_mask=torch.from_numpy(mask).cuda())
            t.check(before, np.where(mask, bo.UNIFORM, bo.KEEP), np.zeros(env.num_envs, np.int64), ("reset", s))
        hint = _hint(torch, env.num_envs, t.N, rng) if hints and s % 2 else None
        env.set_belief_hint(hint)
        before = t.snap()
        acts = env.sample_actions(step_counter=s)
        env.step(acts)
        op, x = t.op_after(before)
        t.check(before, op, x, ("step", s), hint=None if hint is None else hint.cpu().numpy())
        if t.ob is not None:
            t.ob.step(acts.cpu().numpy())
            t.trajectory(("step", s))
    env.set_belief_hint(None)


def _with_oracle(pool, B, P, money, reveal, seed, gid=None):
    cfg = so.OracleConfig(num_police=P, agent_money=money, toll=1, belief=True, reveal_interval=reveal)
    gid = ((np.arange(B) // 32) % len(pool)) if gid is None else np.asarray(gid)
    return oc.CBatch(cfg, pool, B, seed=seed, auto_reset=True, threads=_threads(), graph_id=gid.astype(np.int32))


# ---------------------------------------------------------------------------------------------------- launch forms
LAUNCH = {
    "two_kernels": [("step_kernel", "two_kernels")],
    "fused": [("step_kernel", "fused")],
    "pdl": [("step_kernel", "two_kernels"), ("pdl", "on")],
}


@pytest.mark.parametrize("form", list(LAUNCH))
def test_launch_forms_fast_path(torch_cuda, form):
    """c3 shape at 1000 envs on a 3-graph pool (fast path), each launch form, against the oracle step by step and the C
    oracle's trajectory; then hints, caller-written rows and a partial reset."""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    B, P, money, reveal = 1000, 6, 20, 3
    pool = pkg.generate_graph_pool(3, 200, 400, seed=0)
    assert belief_path(200, _nnz_stride(pool), P + 1) == "fast"
    env = _env(pool, B, P, money, reveal=reveal, options=LAUNCH[form])
    t = Teacher(env, pool, f"fast/{form}", reveal=reveal, auto_reset=True, ob=_with_oracle(pool, B, P, money, reveal, 1))
    t.trajectory("reset")
    _drive(torch, t, 12)
    t.ob = None
    _drive(torch, t, 9, hints=True, rows=True, resets=True, seed=1)
    assert (t.ops > 0).all(), t.ops
    t.report()
    env.close()


def test_step_deferred_lagged(torch_cuda):
    """step_deferred: the belief row of step k is written by the launch of step k + 1 (lagged kernel), so the row read
    after call k + 1 is checked against the row read after call k and the transition of call k."""
    import student_mechanism_design_b200 as pkg

    B, P, money, reveal = 1000, 6, 20, 3
    pool = pkg.generate_graph_pool(3, 200, 400, seed=0)
    env = _env(pool, B, P, money, reveal=reveal, options=[("lagged_kernel", "on")])
    t = Teacher(env, pool, "fast/deferred", reveal=reveal, auto_reset=True)
    state = t.snap()  # state after the reset, belief of it written
    pending = None  # (row before the pending step, its op, x)
    for s in range(12):
        acts = env.sample_actions(step_counter=s)
        env.step_deferred(acts)
        if pending is not None:
            t.check(*pending, ("deferred", s))
        op, x = t.op_after(state)
        bel_prev = env.belief_map.cpu().numpy().copy()  # the input row of the step this call left pending
        pending = (dict(state, bel=bel_prev), op, x)
        state = t.snap()
    env.flush_observations()
    t.check(*pending, "flush")
    assert t.ops[bo.DELTA] > 0 and t.ops[bo.UNIFORM] > 0
    t.report()
    env.close()


def test_rollout_random_one_launch_segments(torch_cuda):
    """rollout_random runs a segment of k steps as one launch with no observation in between: the ops of the k steps
    come from the C oracle stepping alongside, the row after the segment is checked with the k-step bound."""
    import student_mechanism_design_b200 as pkg

    B, P, money, reveal, k = 1000, 6, 20, 4, 5
    pool = pkg.generate_graph_pool(3, 200, 400, seed=0)
    env = _env(pool, B, P, money, reveal=reveal, options=[("rollout_kernel", "on")])
    ob = _with_oracle(pool, B, P, money, reveal, 1)
    t = Teacher(env, pool, "fast/rollout_k5", reveal=reveal, auto_reset=True, ob=ob)
    step = 0
    for seg in range(3):
        before = t.snap()
        row = before["bel"].astype(np.float64)
        nprop = np.zeros(B, np.int64)  # propagations since the last UNIFORM / DELTA (which leave an exact row)
        lastop = np.full(B, bo.PROPAGATE)
        for i in range(k):
            done, ep = np.asarray(ob.done), np.asarray(ob.episode)
            gid = np.asarray(ob.graph_id)
            ob.step(ob.sample_actions(step + i))
            op = bo.op_from_transition(done, ep, np.asarray(ob.episode), ob.revealed(), reveal, True)
            row = bo.belief_step_batched(row, pool, gid, op, ob.pos()[:, 0], mats=t.mats)
            nprop = np.where(op != bo.PROPAGATE, 0, nprop + 1)
            lastop = np.where(op != bo.PROPAGATE, op, lastop)
        env.rollout_random(k, step_counter=step)
        step += k
        got = env.belief_map.cpu().numpy()
        t.trajectory(("segment", seg))
        # exact rows: the last op of the segment decides; propagated rows get the bound of their propagations since then
        for n in np.unique(nprop[nprop > 0]):
            sel = nprop == n
            err = np.abs(got[sel].astype(np.float64) - row[sel])
            bound = np.asarray([rho(t.N, dm, int(n)) for dm in t.dmax])[before["gid"][sel]][:, None] * row[sel]
            ok = (row[sel] < TINY) & (err <= TINY) | (err <= bound)
            assert ok.all(), ("segment", seg, n)
            assert np.array_equal(got[sel] == 0, row[sel] == 0)
            WORST[t.name] = max(WORST[t.name], float((err / np.where(bound > 0, bound, 1))[row[sel] >= TINY].max()))
        last = nprop == 0
        want32 = row[last].astype(np.float32)
        want32[lastop[last] == bo.UNIFORM] = np.float32(1) / np.float32(t.N)
        assert np.array_equal(got[last], want32), ("segment", seg, "exact rows")
        assert nprop.max() > 1 and last.any()
    t.report()
    env.close()


@pytest.mark.parametrize("case", ["generic_quarters", "fast_whole_tiles"])
def test_tail_split_parts(torch_cuda, case):
    """The partly filled last wave cut into parts (330 tiles, ragged last tile) on the warp-per-env path at N = 500 and
    on the fast path at N = 200, with hints."""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    N = 500 if case == "generic_quarters" else 200
    B, P = 330 * 32 - 21, 4
    pool = pkg.generate_graph_pool(2, N, 2 * N, seed=0)
    env = _env(pool, B, P, 15, reveal=4, options=[("tail_split", "on"), ("step_kernel", "two_kernels")], seed=31)
    t = Teacher(env, pool, f"tail_split/{case}/{belief_path(N, _nnz_stride(pool), P + 1)}", reveal=4, auto_reset=True)
    _drive(torch, t, 6, hints=True, rows=True)
    t.report()
    env.close()


# ------------------------------------------------------------------------------------- dispatch boundaries
def _boundary_cases():
    out = []
    for epn in (2.0, 1.5):
        for kind in ("fast", "csr"):
            n = _boundary(epn, 7, kind)
            out += [(epn, n - 1), (epn, n)]
    return out


def test_boundaries_are_where_the_rule_says():
    """the restated rule's boundaries for 6 police: E = 2N -> 344 / 345 (fast / generic) and 1292 / 1293 (CSR staged
    or not); E = 1.5N -> 352 / 353 and 1488 / 1489"""
    assert [n for _, n in _boundary_cases()] == [344, 345, 1292, 1293, 352, 353, 1488, 1489]


@pytest.mark.parametrize("epn,N", _boundary_cases())
def test_dispatch_boundaries(torch_cuda, epn, N):
    """N on both sides of both boundaries, E = 2N and 1.5N, single-graph tiles and one tile-straddling mixed layout:
    propagation, reveals, auto-resets, hints on every path, caller-written rows."""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    P, B = 6, 160
    pool = pkg.generate_graph_pool(2, N, int(epn * N), seed=0)
    path = belief_path(N, _nnz_stride(pool), P + 1)
    gid = (np.arange(B) // 32) % 2
    gid[128:] = np.arange(32) % 2  # the last tile mixes the two graphs: global lists
    env = _env(pool, B, P, 20, reveal=3, gid=torch.from_numpy(gid.astype(np.int32)).cuda())
    t = Teacher(env, pool, f"boundary/E={epn}N/N={N}/{path}", reveal=3, auto_reset=True,
                ob=_with_oracle(pool, B, P, 20, 3, 1, gid=gid))
    _drive(torch, t, 6)
    t.ob = None
    _drive(torch, t, 6, hints=True, rows=True, seed=2)
    t.report()
    env.close()


# ------------------------------------------------------------------------------------------------ hub graphs
def _hub_pool(N):
    """a hub graph (degrees HUB_DEGREES, isolated nodes 32..37 places into fast-path warp ranges) and a sampled graph"""
    import student_mechanism_design_b200 as pkg

    jpw = -(-N // BEL_WARPS)
    iso = [w * jpw + o for w in (1, 3, 6) for o in (32, 35, min(40, jpw - 1)) if jpw > 32 and w * jpw + o < N]
    iso += [N - 1]
    ring = N - len(HUB_DEGREES) - len(iso)
    hub = bo.hub_graph(N, [d for d in HUB_DEGREES if d < ring], isolated=iso, seed=N)
    return [hub, pkg.generate_graph_pool(1, N, 2 * N, seed=1)[0]]


@pytest.mark.parametrize("N,layout", [(300, "single"), (300, "mixed"), (600, "single"), (1500, "single")])
def test_hub_graphs(torch_cuda, N, layout):
    """hub graphs on every path: N = 300 fast (isolated nodes in the second ballot word of three warps), N = 300 mixed
    tiles (global lists, 8 belief warps), N = 600 staged CSR, N = 1500 global lists on single-graph tiles"""
    torch = torch_cuda
    P, B = 3, 128
    pool = _hub_pool(N)
    path = belief_path(N, _nnz_stride(pool), P + 1) if layout == "single" else "global"
    assert path == {300: "fast", 600: "csr", 1500: "global"}[N] or layout == "mixed"
    gid = (np.arange(B) // 32) % 2 if layout == "single" else np.arange(B) % 2
    env = _env(pool, B, P, 30, reveal=4, gid=torch.from_numpy(gid.astype(np.int32)).cuda(), max_timestep=40)
    t = Teacher(env, pool, f"hub/N={N}/{layout}/{path}", reveal=4, auto_reset=True)
    _drive(torch, t, 8, hints=True, rows=True, seed=3)
    t.report()
    env.close()


# --------------------------------------------------------------------------------- reveals, skips, frozen envs
def test_skipped_reveals_and_frozen_envs(torch_cuda):
    """reveal_skip_prob = 0.5 (scheduled reveals that propagate instead) and auto_reset = False with a short horizon
    (envs that end stay frozen: their rows are KEEP)"""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    for N, E in ((200, 400), (700, 1400)):
        pool = pkg.generate_graph_pool(2, N, E, seed=0)
        env = _env(pool, 320, 4, 6, reveal=2, auto_reset=False, reveal_skip_prob=0.5, max_timestep=7)
        t = Teacher(env, pool, f"skip_frozen/N={N}/{belief_path(N, _nnz_stride(pool), 5)}", reveal=2, auto_reset=False)
        _drive(torch, t, 12, hints=True)
        assert t.ops[bo.KEEP] > 0 and t.ops[bo.DELTA] > 0
        t.report()
        env.close()


def test_device_sampled_pool_large_n(torch_cuda):
    """graphs="device" at N = 1000: the neighbour lists the device builds (sy_csr_from_dense_kernel) against the edge
    lists read back"""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    env = pkg.BatchedScotlandYardEnv(256, 4, 20, graph_nodes=1000, graph_edges=2000, graphs="device", num_graphs=3, seed=4,
                                     auto_reset=True, tolls=1, belief=True, reveal_interval=3)
    env.reset()
    t = Teacher(env, env.graphs, "device_pool/N=1000", reveal=3, auto_reset=True)
    _drive(torch, t, 6, hints=True, rows=True)
    t.report()
    env.close()


# -------------------------------------------------------------------------------------------------- full size
@pytest.mark.parametrize("cfg", ["c3", "c4"])
def test_full_size(torch_cuda, cfg):
    """BASELINE configs 3 (65 536 x 200, fast path) and 4 (32 768 x 1000, staged CSR) for a few steps"""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    N, B = (200, 65536) if cfg == "c3" else (1000, 32768)
    pool = pkg.generate_graph_pool(1, N, 2 * N, seed=0)
    env = _env(pool, B, 6, 20, reveal=5)
    t = Teacher(env, pool, f"full/{cfg}/{belief_path(N, _nnz_stride(pool), 7)}", reveal=5, auto_reset=True)
    _drive(torch, t, 6, hints=True)
    t.report()
    env.close()


# --------------------------------------------------------------------------------------- per-env cross-entropy
CE_CASES = {  # name: (N, layout, launch options)
    "fast": (200, "single", [("step_kernel", "two_kernels")]),
    "fast_fused": (200, "single", [("step_kernel", "fused")]),
    "csr": (600, "single", []),
    "global_mixed": (200, "mixed", []),
    "global_single": (1500, "single", []),
}


@pytest.mark.parametrize("groups", [True, False])
@pytest.mark.parametrize("case", list(CE_CASES))
def test_belief_cross_entropy_per_env(torch_cuda, case, groups):
    """Scored reveals: with one identity mechanism group per env (B = 1024 groups, so every warp holds 32 of them) the
    per-step change of stats(by_group=True) is each env's reveal count and Q24 cross-entropy, compared with
    belief_ce_batched on the device's previous row; without groups the handle-wide sums must match the sum of the per-env
    references within the sum of the per-env bounds.  The rows are checked step by step as well (GROUPS kernels)."""
    import student_mechanism_design_b200 as pkg

    torch = torch_cuda
    N, layout, options = CE_CASES[case]
    B, P, reveal = 1024, 3, 2
    pool = _hub_pool(N) if N != 200 else [*pkg.generate_graph_pool(1, N, 2 * N, seed=0), _hub_pool(N)[0]]
    gid = (np.arange(B) // 32) % 2 if layout == "single" else np.arange(B) % 2
    env = pkg.BatchedScotlandYardEnv(B, P, 30, graphs=pool, seed=9, auto_reset=True, tolls=1, belief=True, belief_ce=True,
                                     reveal_interval=reveal, max_timestep=30)
    for k, v in options:
        env.set_option(k, v)
    if groups:
        env.set_mechanisms([{}] * B)
    env.reset(graph_id=torch.from_numpy(gid.astype(np.int32)).cuda())
    t = Teacher(env, pool, f"ce/{case}/{'groups' if groups else 'handle'}", reveal=reveal, auto_reset=True)
    keys = ["reveals", "sum_belief_ce_q24", "sum_sq_belief_ce_q24"]

    def counters():
        if groups:
            return np.asarray([[d[k] for k in keys] for d in env.stats(by_group=True)], dtype=np.int64)
        st = env.stats()
        return np.asarray([[st[k] for k in keys]], dtype=np.int64)

    worst, scored = 0.0, 0
    for s in range(10):
        c0 = counters()
        before = t.snap()
        env.step(env.sample_actions(step_counter=s))
        op, x = t.op_after(before)
        t.check(before, op, x, ("step", s))
        dc = counters() - c0
        rev = op == bo.DELTA
        ce = bo.belief_ce_batched(before["bel"].astype(np.float64), pool, before["gid"], x, mats=t.mats)
        bound = np.asarray([ce_bound(N, t.dmax[g], c) for g, c in zip(before["gid"], ce)])
        if groups:
            assert np.array_equal(dc[:, 0], rev.astype(np.int64)), ("reveal counts", s, np.nonzero(dc[:, 0] != rev)[0][:8])
            got = dc[rev, 1] / 2.0 ** 24
            err = np.abs(got - ce[rev])
            assert (err <= bound[rev]).all(), ("CE", s, float((err / bound[rev]).max()))
            # the squared sum: Q24 of the float32 ce^2
            assert (np.abs(dc[rev, 2] / 2.0 ** 24 - ce[rev] ** 2) <= 2 * np.abs(ce[rev]) * bound[rev] + bound[rev] ** 2 + 4 * U * ce[rev] ** 2 + 2.0 ** -25).all()
            if rev.any():
                worst = max(worst, float((err / bound[rev]).max()))
        else:
            assert dc[0, 0] == int(rev.sum()), ("reveal count", s)
            err = abs(dc[0, 1] / 2.0 ** 24 - ce[rev].sum())
            assert err <= bound[rev].sum(), ("CE sum", s, err, bound[rev].sum())
            if rev.any():
                worst = max(worst, err / bound[rev].sum())
        scored += int(rev.sum())
    assert scored > 100
    print(f"\n[belief-ce] {case}/{'groups' if groups else 'handle'}: {scored} scored reveals, largest CE err/bound {worst:.3g}")
    t.report()
    env.close()
