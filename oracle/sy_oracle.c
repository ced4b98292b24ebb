/*
 * sy_oracle.c -- plain-C CPU restatement of the Scotland Yard env step (the checker and the CPU
 * baseline).  TEST INFRASTRUCTURE ONLY: only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load it; the product never does.
 *
 * It follows, line by line, the same reference code as oracle/sy_oracle.py (which is pinned
 * against golden vectors recorded from the unmodified reference); tests/test_oracle_c.py pins
 * this file against those golden vectors too and against the Python oracle.  Paths below are
 * relative to /root/reference.
 *
 *   src/environment/yard.py:144-269          step        -> syo_step (per env: step_one)
 *   src/environment/yard.py:420-472          legal moves -> legal() / n_moves()
 *   src/environment/reward_calculator.py:26-92   termination priority -> step_one
 *   src/environment/reward_calculator.py:94-266  shaped rewards       -> shaped_rewards
 *   src/environment/action_mask.py:54-83     mask        -> write_obs
 *   src/environment/pathfinding.py:34-137    distance    -> syo_apsp (Dijkstra from every source)
 *   src/environment/belief_module.py:69-111  belief (exact expectation; parity unpinned) -> belief_update
 *   src/eval/run_ablations.py:225-229        reveal predicate (parity unpinned)          -> is_reveal
 *
 * Arithmetic: float64 exactly in the reference's evaluation order (compile with
 * -ffp-contract=off -fno-fast-math); fp32 mode = every operand rounded to float first, one
 * rounding per operation (0-dim fp32 torch tensors, gnn_trainer.py:98-110).  exp(-d) and
 * exp(-log1p(c)) come from tables computed by NumPy (its SIMD exp is not libm's).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define SYO_MAX_AGENTS 16
#define SYO_INF 0xFFFF
enum { W_POLICE_DISTANCE, W_POLICE_GROUP, W_POLICE_POSITION, W_POLICE_TIME, W_MRX_CLOSEST, W_MRX_AVERAGE,
       W_MRX_POSITION, W_MRX_TIME, W_POLICE_COVERAGE, W_POLICE_PROXIMITY, W_POLICE_OVERLAP }; /* reward_net.py:5-17 */
enum { RNG_RESET_POS = 0, RNG_RESET_GRAPH = 1, RNG_ACTION = 2, RNG_REVEAL_SKIP = 3 };
enum { WIN_NONE = 0, WIN_MRX = 1, WIN_POLICE = 2 };

typedef struct SyoConfig {
  int32_t num_nodes, num_police, agent_money, mrx_money, max_timestep, reveal_interval, toll, belief;
  int32_t reward_mode, auto_reset, resample_graph, num_graphs, nnz_stride, n_exp, n_cov;
  float reveal_skip_prob; /* every scheduled reveal is skipped with this probability (the batched env's draw) */
  int64_t env_offset;
  uint64_t seed;
  double w[11];
  const double* exp_neg;  /* [n_exp]  np.exp(-d) */
  const double* coverage; /* [n_cov]  np.exp(-np.log1p(c)) */
  const int32_t* W;       /* [G, N, N] edge weight, 0 = no edge (yard.py:404-418) */
  const int32_t* D;       /* [G, N, N] all-pairs distance, 0xFFFF = unreachable */
  const int32_t* row_ptr; /* [G, N+1] */
  const int32_t* col;     /* [G, nnz_stride] neighbours ascending */
} SyoConfig;

typedef struct SyoState {
  int32_t* pos;      /* [B, A] */
  int32_t* money;    /* [B, A] */
  int32_t* t;        /* [B] */
  int32_t* gid;      /* [B] */
  int32_t* episode;  /* [B] */
  uint8_t* done;     /* [B] */
  int32_t* visits;   /* [B, N] */
  double* belief;    /* [B, N] or NULL */
  int32_t* revealed; /* [B] */
} SyoState;

typedef struct SyoOut {
  double* reward;      /* [B, A] (fp32 mode: the float value widened) */
  uint8_t* terminated; /* [B] */
  uint8_t* truncated;  /* [B] */
  int8_t* winner;      /* [B] */
  uint8_t* mask;       /* [B, A, N] or NULL */
  float* node_features; /* [B, N, A] or NULL */
} SyoOut;

/* ---------------------------------------------------------------- Philox4x32-10 (Random123) */
static void philox4x32(const uint32_t ctr[4], uint32_t k0, uint32_t k1, uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

void syo_philox4x32(const uint32_t* ctr, const uint32_t* key, uint32_t* out) { philox4x32(ctr, key[0], key[1], out); }

/* A distinct uniform nodes (distribution of np.random.choice(N, A, replace=False), yard.py:112-116) */
static void start_positions(const SyoConfig* c, uint32_t env, uint32_t episode, int32_t* out) {
  const int A = c->num_police + 1;
  int chosen[SYO_MAX_AGENTS];
  uint32_t r[4] = {0, 0, 0, 0};
  for (int a = 0; a < A; ++a) {
    if ((a & 3) == 0) {
      const uint32_t ctr[4] = {env, episode, RNG_RESET_POS, (uint32_t)(a >> 2)};
      philox4x32(ctr, (uint32_t)c->seed, (uint32_t)(c->seed >> 32), r);
    }
    int x = (int)(((uint64_t)r[a & 3] * (uint64_t)(c->num_nodes - a)) >> 32);
    for (int i = 0; i < a; ++i)
      if (x >= chosen[i]) ++x;
    int j = a;
    while (j > 0 && chosen[j - 1] > x) { chosen[j] = chosen[j - 1]; --j; }
    chosen[j] = x;
    out[a] = x;
  }
}

static int graph_choice(const SyoConfig* c, uint32_t env, uint32_t episode) {
  const uint32_t ctr[4] = {env, episode, RNG_RESET_GRAPH, 0};
  uint32_t r[4];
  philox4x32(ctr, (uint32_t)c->seed, (uint32_t)(c->seed >> 32), r);
  return (int)(((uint64_t)r[0] * (uint64_t)c->num_graphs) >> 32);
}

/* ---------------------------------------------------------------- graph helpers */
/* pathfinding.py:34-137: weighted shortest path; the reference re-runs a heap Dijkstra per query,
 * the result equals this table (array Dijkstra from every source; unreachable -> 0xFFFF). */
void syo_apsp(int32_t N, const int32_t* row_ptr, const int32_t* col, const int32_t* w, int32_t* D) {
  int64_t* dist = (int64_t*)malloc(sizeof(int64_t) * N);
  uint8_t* fin = (uint8_t*)malloc(N);
  for (int s = 0; s < N; ++s) {
    for (int v = 0; v < N; ++v) { dist[v] = INT64_MAX; fin[v] = 0; }
    dist[s] = 0;
    for (;;) {
      int u = -1;
      for (int v = 0; v < N; ++v)
        if (!fin[v] && dist[v] != INT64_MAX && (u < 0 || dist[v] < dist[u])) u = v;
      if (u < 0) break;
      fin[u] = 1;
      for (int k = row_ptr[u]; k < row_ptr[u + 1]; ++k)
        if (dist[u] + w[k] < dist[col[k]]) dist[col[k]] = dist[u] + w[k];
    }
    for (int v = 0; v < N; ++v) D[(size_t)s * N + v] = dist[v] == INT64_MAX ? SYO_INF : (int32_t)dist[v];
  }
  free(dist);
  free(fin);
}

/* yard.py:420-472 with the toll extension (toll == 0 -> the reference rule) */
static int legal(const SyoConfig* c, const int32_t* Wg, int p, int64_t j, int money) {
  if (j < 0 || j >= c->num_nodes) return 0;
  const int w = Wg[(size_t)p * c->num_nodes + j];
  return w > 0 && w + c->toll <= money;
}
static int n_moves(const SyoConfig* c, const int32_t* Wg, int p, int money) {
  int n = 0;
  const int32_t* row = Wg + (size_t)p * c->num_nodes;
  for (int j = 0; j < c->num_nodes; ++j) n += (row[j] > 0 && row[j] + c->toll <= money);
  return n;
}
static double distf(const SyoConfig* c, const int32_t* Dg, int a, int b) {
  const int d = Dg[(size_t)a * c->num_nodes + b];
  return d >= SYO_INF ? INFINITY : (double)d;
}
static double exp_neg(const SyoConfig* c, double d) {
  if (isinf(d)) return 0.0; /* np.exp(-inf) */
  const int i = (int)d;
  return i < c->n_exp ? c->exp_neg[i] : 0.0;
}
static int is_reveal(int t, int interval) { return interval > 0 && t > 0 && t % interval == 0; } /* run_ablations.py:225-229 */

/* ---------------------------------------------------------------- rewards (reward_calculator.py:94-266) */
static void shaped_rewards(const SyoConfig* c, const int32_t* Wg, const int32_t* Dg, const int32_t* pos,
                           const int32_t* money, int t, const int32_t* visits, double* out) {
  const int P = c->num_police;
  const double* w = c->w;
  /* MrX, :126-148 */
  double closest = INFINITY, sum = 0.0;
  for (int i = 0; i < P; ++i) {
    const double d = distf(c, Dg, pos[0], pos[1 + i]);
    if (d < closest) closest = d;
    sum += d;
  }
  const double avg = sum / (double)P; /* np.mean of exact small integers (inf stays inf) */
  const double m1 = -1.0 / (closest + 1.0), m2 = -1.0 / (avg + 1.0);
  const double m3 = (double)n_moves(c, Wg, pos[0], money[0]);
  const double m4 = 0.1 * (double)t;
  if (c->reward_mode == 0) {
    out[0] = w[W_MRX_CLOSEST] * m1 + w[W_MRX_AVERAGE] * m2 + w[W_MRX_POSITION] * m3 + (1.0 - w[W_MRX_TIME]) * m4;
  } else {
    const float a = (float)w[W_MRX_CLOSEST] * (float)m1, b = (float)w[W_MRX_AVERAGE] * (float)m2;
    const float cc = (float)w[W_MRX_POSITION] * (float)m3;
    const float one_minus = 1.0f - (float)w[W_MRX_TIME];
    const float d = one_minus * (float)m4;
    float r = a + b;
    r = r + cc;
    r = r + d;
    out[0] = (double)r;
  }
  /* police k, :182-227 */
  for (int k = 0; k < P; ++k) {
    const int p = pos[1 + k];
    const double dx = exp_neg(c, distf(c, Dg, p, pos[0]));
    double grp = 0.0, ov = 0.0, prox = 0.0;
    for (int j = 0; j < P; ++j) {
      if (j == k) continue;
      const double dj = distf(c, Dg, p, pos[1 + j]);
      const double e = exp_neg(c, dj);
      grp = grp + e;
      if (dj <= 1.0) ov = ov + 1.0;
      else prox = prox + e;
    }
    const double mob = (double)n_moves(c, Wg, p, money[k]); /* QUIRK :190 -- budget of agent index k, not k+1 */
    int vc = visits[p];
    if (vc > c->n_cov - 1) vc = c->n_cov - 1;
    const double cov = c->coverage[vc];
    const double tt = 0.05 * (double)t;
    if (c->reward_mode == 0) {
      out[1 + k] = w[W_POLICE_DISTANCE] * dx + w[W_POLICE_GROUP] * grp + w[W_POLICE_POSITION] * mob +
                   (1.0 - w[W_POLICE_TIME]) * tt + w[W_POLICE_PROXIMITY] * prox - w[W_POLICE_OVERLAP] * ov +
                   w[W_POLICE_COVERAGE] * cov;
    } else {
      const float u1 = (float)w[W_POLICE_DISTANCE] * (float)dx, u2 = (float)w[W_POLICE_GROUP] * (float)grp;
      const float u3 = (float)w[W_POLICE_POSITION] * (float)mob;
      const float om = 1.0f - (float)w[W_POLICE_TIME];
      const float u4 = om * (float)tt;
      const float u5 = (float)w[W_POLICE_PROXIMITY] * (float)prox, u6 = (float)w[W_POLICE_OVERLAP] * (float)ov;
      const float u7 = (float)w[W_POLICE_COVERAGE] * (float)cov;
      float r = u1 + u2;
      r = r + u3;
      r = r + u4;
      r = r + u5;
      r = r - u6;
      r = r + u7;
      out[1 + k] = (double)r;
    }
  }
}

/* belief_module.py:69-111 in expectation (see oracle/sy_oracle.py:belief_update) */
static void belief_update(const SyoConfig* c, const int32_t* rp, const int32_t* col, double* bel, double* tmp, int reveal) {
  const int N = c->num_nodes;
  if (reveal >= 0) {
    for (int j = 0; j < N; ++j) bel[j] = 0.0;
    bel[reveal] = 1.0;
    return;
  }
  double s = 0.0;
  for (int j = 0; j < N; ++j) {
    double acc = 0.0;
    for (int k = rp[j]; k < rp[j + 1]; ++k) {
      const int i = col[k];
      acc += bel[i] / (double)(rp[i + 1] - rp[i]);
    }
    if (rp[j + 1] == rp[j]) acc = bel[j];
    tmp[j] = acc;
    s += acc;
  }
  if (s == 0.0) {
    for (int j = 0; j < N; ++j) bel[j] = 1.0 / (double)N;
  } else {
    for (int j = 0; j < N; ++j) bel[j] = tmp[j] / s;
  }
}

static void reset_one(const SyoConfig* c, const SyoState* st, int b, const int32_t* start) {
  const int N = c->num_nodes, A = c->num_police + 1;
  for (int a = 0; a < A; ++a) {
    st->pos[(size_t)b * A + a] = start[a];
    st->money[(size_t)b * A + a] = a == 0 ? c->mrx_money : c->agent_money; /* yard.py:117-119 */
  }
  st->t[b] = 0;
  st->done[b] = 0;
  memset(st->visits + (size_t)b * N, 0, sizeof(int32_t) * N); /* yard.py:85 */
  if (st->belief)
    for (int j = 0; j < N; ++j) st->belief[(size_t)b * N + j] = 1.0 / (double)N;
  st->revealed[b] = c->reveal_interval > 0 ? -1 : start[0];
}

static void write_obs(const SyoConfig* c, const SyoState* st, const SyoOut* out, int b) {
  const int N = c->num_nodes, A = c->num_police + 1;
  const int32_t* Wg = c->W + (size_t)st->gid[b] * N * N;
  const int32_t* pos = st->pos + (size_t)b * A;
  const int32_t* money = st->money + (size_t)b * A;
  if (out->mask) { /* action_mask.py:65-76 */
    for (int a = 0; a < A; ++a) {
      const int32_t* row = Wg + (size_t)pos[a] * N;
      uint8_t* m = out->mask + ((size_t)b * A + a) * N;
      for (int j = 0; j < N; ++j) m[j] = (row[j] > 0 && row[j] + c->toll <= money[a]);
    }
  }
  if (out->node_features) { /* yard.py:279-290; MrX column blank while hidden */
    float* nf = out->node_features + (size_t)b * N * A;
    memset(nf, 0, sizeof(float) * N * A);
    if (st->revealed[b] >= 0) nf[(size_t)pos[0] * A] = 1.0f;
    for (int a = 1; a < A; ++a) nf[(size_t)pos[a] * A + a] = 1.0f;
  }
}

/* yard.py:144-269 for env b */
static void step_one(const SyoConfig* c, const SyoState* st, const SyoOut* out, const int64_t* actions, int b, double* tmp) {
  const int N = c->num_nodes, P = c->num_police, A = P + 1;
  const int g = st->gid[b];
  const int32_t* Wg = c->W + (size_t)g * N * N;
  const int32_t* Dg = c->D + (size_t)g * N * N;
  int32_t* pos = st->pos + (size_t)b * A;
  int32_t* money = st->money + (size_t)b * A;
  int32_t* visits = st->visits + (size_t)b * N;
  const int64_t* act = actions + (size_t)b * A;
  double* rew = out->reward + (size_t)b * A;
  if (st->done[b]) { /* frozen until reset */
    for (int a = 0; a < A; ++a) rew[a] = 0.0;
    out->terminated[b] = out->truncated[b] = 0;
    out->winner[b] = WIN_NONE;
    write_obs(c, st, out, b);
    return;
  }
  { /* MrX, yard.py:155-188 */
    const int tgt = legal(c, Wg, pos[0], act[0], money[0]) ? (int)act[0] : pos[0];
    int occupied = 0;
    for (int i = 1; i <= P; ++i) occupied |= (pos[i] == tgt);
    if (!occupied) pos[0] = tgt;
  }
  int no_money = 1;
  for (int i = 1; i <= P; ++i) { /* police in order, yard.py:190-243 */
    if (money[i] == 0 || act[i] == -1) continue;
    no_money = 0;
    const int tgt = legal(c, Wg, pos[i], act[i], money[i]) ? (int)act[i] : pos[i];
    int occupied = 0;
    for (int j = 1; j <= P; ++j) occupied |= (pos[j] == tgt);
    if (!occupied && tgt != pos[i]) {
      money[i] -= Wg[(size_t)pos[i] * N + tgt] + c->toll;
      pos[i] = tgt;
    }
  }
  for (int i = 1; i <= P; ++i) visits[pos[i]] += 1; /* yard.py:244-245 */
  /* reward_calculator.py:26-92 */
  int capture = 0;
  for (int i = 1; i <= P; ++i) capture |= (pos[i] == pos[0]);
  int term = 0, trunc = 0, win = WIN_NONE;
  if (capture) {
    rew[0] = -1.0;
    for (int i = 1; i <= P; ++i) rew[i] = 1.0;
    term = 1; win = WIN_POLICE;
  } else if (st->t[b] > c->max_timestep) {
    rew[0] = 1.0;
    for (int i = 1; i <= P; ++i) rew[i] = 0.0;
    trunc = 1; win = WIN_MRX;
  } else if (no_money) {
    rew[0] = 1.0;
    for (int i = 1; i <= P; ++i) rew[i] = 0.0;
    term = 1; win = WIN_MRX;
  } else {
    shaped_rewards(c, Wg, Dg, pos, money, st->t[b], visits, rew);
  }
  st->t[b] += 1; /* yard.py:355 */
  out->terminated[b] = (uint8_t)term;
  out->truncated[b] = (uint8_t)trunc;
  out->winner[b] = (int8_t)win;
  /* extensions (parity unpinned): reveal schedule + belief on the new timestep */
  int rev = is_reveal(st->t[b], c->reveal_interval);
  if (rev && c->reveal_skip_prob > 0.0f) { /* skip iff Philox(seed; env, t, RNG_REVEAL_SKIP, episode)[0] < p * 2^32 */
    const uint32_t ctr[4] = {(uint32_t)(c->env_offset + b), (uint32_t)st->t[b], RNG_REVEAL_SKIP, (uint32_t)st->episode[b]};
    uint32_t r[4];
    philox4x32(ctr, (uint32_t)c->seed, (uint32_t)(c->seed >> 32), r);
    if ((unsigned long long)r[0] < (unsigned long long)((double)fminf(c->reveal_skip_prob, 1.0f) * 4294967296.0)) rev = 0;
  }
  st->revealed[b] = (c->reveal_interval > 0) ? (rev ? pos[0] : -1) : pos[0];
  if (st->belief)
    belief_update(c, c->row_ptr + (size_t)g * (N + 1), c->col + (size_t)g * c->nnz_stride, st->belief + (size_t)b * N, tmp,
                  rev ? pos[0] : -1);
  if (term || trunc) {
    if (c->auto_reset) { /* same-step auto-reset, as the batched env */
      int32_t start[SYO_MAX_AGENTS];
      const uint32_t env = (uint32_t)(c->env_offset + b);
      st->episode[b] += 1;
      if (c->resample_graph) st->gid[b] = graph_choice(c, env, (uint32_t)st->episode[b]);
      start_positions(c, env, (uint32_t)st->episode[b], start);
      reset_one(c, st, b, start);
    } else {
      st->done[b] = 1;
    }
  }
  write_obs(c, st, out, b);
}

/* ---------------------------------------------------------------- exported batch entry points */
void syo_reset_all(const SyoConfig* c, int32_t B, const SyoState* st, const int32_t* init_pos, const int32_t* init_gid) {
  const int A = c->num_police + 1;
  for (int b = 0; b < B; ++b) {
    int32_t start[SYO_MAX_AGENTS];
    const uint32_t env = (uint32_t)(c->env_offset + b);
    st->episode[b] = 0;
    st->gid[b] = init_gid ? init_gid[b] : (c->resample_graph ? graph_choice(c, env, 0) : (int32_t)(((c->env_offset + b) / 32) % c->num_graphs));
    if (init_pos) memcpy(start, init_pos + (size_t)b * A, sizeof(int32_t) * A);
    else start_positions(c, env, 0, start);
    reset_one(c, st, b, start);
  }
}

void syo_observe(const SyoConfig* c, int32_t B, const SyoState* st, const SyoOut* out) {
  for (int b = 0; b < B; ++b) write_obs(c, st, out, b);
}

void syo_step(const SyoConfig* c, int32_t B, const SyoState* st, const int64_t* actions, const SyoOut* out, int32_t threads) {
  (void)threads;
#pragma omp parallel num_threads(threads > 0 ? threads : 1)
  {
    double* tmp = (double*)malloc(sizeof(double) * c->num_nodes);
#pragma omp for schedule(static)
    for (int b = 0; b < B; ++b) step_one(c, st, out, actions, b, tmp);
    free(tmp);
  }
}

/* uniform random valid action per agent, Philox(seed; env, step, RNG_ACTION, agent); -1 if none */
void syo_sample_actions(const SyoConfig* c, int32_t B, const SyoState* st, uint32_t step, int64_t* actions, int32_t threads) {
  const int N = c->num_nodes, A = c->num_police + 1;
  (void)threads;
#pragma omp parallel for schedule(static) num_threads(threads > 0 ? threads : 1)
  for (int b = 0; b < B; ++b) {
    const int32_t* Wg = c->W + (size_t)st->gid[b] * N * N;
    for (int a = 0; a < A; ++a) {
      const int p = st->pos[(size_t)b * A + a], m = st->money[(size_t)b * A + a];
      const int32_t* row = Wg + (size_t)p * N;
      int n = 0;
      for (int j = 0; j < N; ++j) n += (row[j] > 0 && row[j] + c->toll <= m);
      int64_t pick = -1;
      if (n > 0) {
        const uint32_t ctr[4] = {(uint32_t)(c->env_offset + b), step, RNG_ACTION, (uint32_t)a};
        uint32_t r[4];
        philox4x32(ctr, (uint32_t)c->seed, (uint32_t)(c->seed >> 32), r);
        int idx = (int)(((uint64_t)r[0] * (uint64_t)n) >> 32);
        for (int j = 0; j < N; ++j) {
          if (row[j] > 0 && row[j] + c->toll <= m) {
            if (idx == 0) { pick = j; break; }
            --idx;
          }
        }
      }
      actions[(size_t)b * A + a] = pick;
    }
  }
}

int32_t syo_max_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
