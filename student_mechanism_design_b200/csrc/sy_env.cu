// sy_env.cu -- B200 (sm_100a) kernels + C ABI of the batched Scotland Yard environment.
//
// Reference behaviour restated here (paths relative to /root/reference):
//   src/environment/yard.py:80-142   reset          -> sy_reset_kernel (+ sy_observe_kernel)
//   src/environment/yard.py:144-269  step           -> sy_logic_kernel
//   src/environment/yard.py:271-335  observations   -> sy_observe_kernel (writer warps)
//   src/environment/yard.py:420-472  possible moves -> dense weight table + move-count table
//   src/environment/action_mask.py:30-83            -> writer_role (mask rows), sy_mask_dense_kernel
//   src/environment/reward_calculator.py:26-266     -> move_phase (ending) and agent_reward
//   src/environment/pathfinding.py:34-137           -> sy_apsp_kernel (all-pairs table, built once per graph)
//   src/environment/belief_module.py:69-111         -> belief_role in sy_observe_kernel (expectation)
//
// Two launches per step (measured on B200: a fused per-tile kernel ran its phases in lockstep over the whole
// chip -- every phase added its full latency and HBM idled during the game logic; see DESIGN.md):
//   sy_logic_kernel    CTA of 4 warps per 32-env tile, lane = env, agents in a conflict-free smem row; the whole batch is
//                      resident in one wave.  Warp 0: order-dependent moves -> ending; all warps: visit counts + rewards
//                      (warp = agent; fp64 / no-FMA fp32); warp 0: timestep, reveal schedule, same-step auto-reset
//                      (Philox), statistics; coalesced state / result write-back.
//   sy_observe_kernel  CTA per 32-env tile, warp-specialised, no barrier between the roles: writer warps stream the
//                      dense observations (16-byte zero stores + the few ones while the lines sit in L2); belief
//                      warps run the belief propagation as a lane = env SpMM over a transposed smem tile (LDGSTS).
// The step is bound by the HBM writes of the observations (SURVEY.md section 8(d)); graph tables are a few hundred
// KB and are read through L1/L2 with ld.global.nc.
// Batches of at most one wave of tiles are latency bound instead, and take single-launch forms (DESIGN.md section 4,
// "Which kernels a call launches"):
//   sy_step_fused_kernel      sy_step as one persistent launch (dynamics -> TMA bulk-store writers + belief per CTA)
//   sy_step_lagged_kernel     sy_step_deferred: observation roles of step k + dynamics warps of step k+1 in one CTA
//   sy_rollout_lagged_kernel  sy_rollout_random*: all K steps in one launch, a CTA owns its tile throughout
#include "../../include/sy_env.h"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return fail(SY_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

constexpr int STAT_REPLICAS = 64;  // statistics accumulator lines (128 B each) the tiles are spread over
constexpr int GROUP_STAT_LINES = 4096;  // per-group statistics lines of a handle (replicas x groups)
constexpr int TILE = 32;       // envs per observe CTA / per logic warp (lane = env)
#ifndef SY_BEL_WARPS
#define SY_BEL_WARPS 8
#endif
#ifndef SY_WR_WARPS
#define SY_WR_WARPS 8
#endif
#ifndef SY_STORE_HINT
#define SY_STORE_HINT 0
#endif
#ifndef SY_NF_SCALAR_ONES
#define SY_NF_SCALAR_ONES 0  // 1: node_features ones as 4-byte stores after the zero fill instead of merged 16-byte chunks
#endif
#ifndef SY_BULK_HINT
#define SY_BULK_HINT 0  // 1: L2 evict_first policy on the bulk stores
#endif
#ifndef SY_BULK_IMG_BUDGET
#define SY_BULK_IMG_BUDGET 25344  // bytes of shared memory for the bulk writers' zero page and chunk images of a CTA
#endif
constexpr int BEL_WARPS = SY_BEL_WARPS;  // observe kernel: the first warps propagate the belief ...
constexpr int WR_WARPS = SY_WR_WARPS;    // ... the others stream the dense observations
constexpr int THREADS = (BEL_WARPS + WR_WARPS) * 32;
constexpr int EXP_SMEM = 96;   // logic kernel: exp(-d) entries staged in shared memory (larger d: global table)
constexpr int COV_SMEM = 64;   // logic kernel: coverage entries staged in shared memory
constexpr int HS = 18;         // row stride (halfwords) of the u16 smem rows: 9 words, conflict-free for lane = env
typedef unsigned short u16;
#ifndef SY_LOGIC_WARPS
#define SY_LOGIC_WARPS 4
#endif
constexpr int LOGIC_WARPS = SY_LOGIC_WARPS;  // logic kernel: warps per 32-env tile; reset kernel: warps x 32 envs
constexpr int LOGIC_THREADS = LOGIC_WARPS * 32;
constexpr int AS = SY_MAX_AGENTS + 1;  // odd smem row stride -> conflict-free lane = env access
constexpr unsigned FULL = 0xffffffffu;
enum { DIST_INF = 0xFFFF };

enum { RNG_RESET_POS = 0, RNG_RESET_GRAPH = 1, RNG_ACTION = 2, RNG_REVEAL_SKIP = 3 };
enum { ST_RUNNING = 0, ST_CAPTURE = 1, ST_TIMEOUT = 2, ST_NO_MONEY = 3 };
enum { BEL_KEEP = 0, BEL_UNIFORM = 1, BEL_DELTA = 2, BEL_PROPAGATE = 3 };

struct Tables {
  const uint8_t* W;      // [G, N, Ns] dense edge weight, 0 = no edge
  const uint16_t* D;     // [G, N, N]  all-pairs shortest path, 0xFFFF = unreachable
  const int32_t* row_ptr;  // [G, N+1]
  const uint16_t* col;   // [G, nnz_stride]
  const uint8_t* wgt;    // [G, nnz_stride]
  const uint8_t* cnt;    // [G, N, wcap+1] #neighbours with weight <= c
  const float* inv_deg;  // [G, N]
  const int2* nbr_pack;  // [G, pack_stride] belief fast path: per neighbour {byte offset of its tile row, bits of 1/deg(nbr)};
                         //  every node's list is padded to a multiple of 4 entries with {0, 0.0f}
  const int32_t* pack_ptr;  // [G, N+1] start of each node's list in nbr_pack (entries)
  const uint16_t* deg_perm; // [G, N] nodes ordered by degree: lanes of a warp that walk neighbour lists get equal lengths
  const double* exp_neg; // [n_exp]
  const double* coverage;  // [n_cov]
  int n_exp, n_cov, G, Ns, nnz_stride, wcap, pack_stride;
};

struct Params {
  int B, N, P, A;
  int inv_A;  // ceil(2^16 / A): (i * inv_A) >> 16 == i / A for i < 2^12
  int agent_money, mrx_money, max_t, reveal, toll, belief_on, belief_score, auto_reset, resample_graph, reward_mode;
  unsigned long long env_offset;
  unsigned long long reveal_skip_thresh;  // a scheduled reveal is skipped when its Philox word < this (reveal_skip_prob * 2^32)
  const uint8_t* belief_hint;             // [B, N] or NULL (SyState.belief_hint)
  unsigned seed_lo, seed_hi;
  double w64[SY_NUM_REWARD_WEIGHTS];
  float w32[SY_NUM_REWARD_WEIGHTS];
  Tables tb;
  SyState st;
  SyObs ob;
  SyOut out;
  const long long* actions;  // int64 [B, A] ...
  const int* actions32;      // ... or int32 [B, A] (narrow wire format of the host-buffer path), exactly one is set
  const short* actions16;    // ... or int16 [B, A]
  int bel_fast, bel_off_out, bel_off_part, bel_off_pack, bel_off_ptr;  // belief fast path: dynamic smem layout (bytes)
  int wr_off, wr_off_csr, wr_img_stride, wr_stage_csr;  // writer warps: smem staging layout (bytes) and path flag
  int bel_share_csr;  // generic belief path gathers over the writers' staged CSR (+ 1/deg) instead of the global lists
  int wr_img_rows;    // action_mask rows per writer image: A (a whole env) or 1 (large rows: saves shared memory)
  int wr_off_pad;     // shared-CSR belief path: byte offset (from wr_off_csr) of the padded neighbour lists
  // bulk (TMA) writers: the tile's action_mask / node_features regions are contiguous byte streams cut into chunks of
  // wr_c_mask / wr_c_nf bytes (multiples of 16); each chunk is assembled in a per-warp shared-memory image and leaves
  // the SM with one cp.async.bulk.  0 = the LSU writers (unaligned caller buffers, or selected with sy_set_option)
  int wr_bulk, wr_c_mask, wr_c_nf, wr_img_bytes;
  int nf_prefilled;  // float32 node_features were zero-filled by the logic kernel (bulk stores): the writers only store the ones
  int f_off_sbuf, f_sbuf_stride, f_off_zero, f_off_imgs;  // fused kernel: staged tile state (x2), zero page, chunk images
  int f_off_nbr4;  // fused kernel: packed neighbour table [N] uint4 + flag (after the staged CSR)
  int wr_epc;      // fused kernel fast geometry: whole envs per chunk (0: chunks cut through envs / more than 32 pairs)
  // observation kernel grid: CTAs [0, ob_full) take whole 32-env tiles; the tiles behind them -- the last, partly filled
  // wave of the grid -- are cut into ob_split parts of 32 / ob_split envs each, one CTA per part (0 / 1: no split)
  int ob_full, ob_split;
  int dbg_skip;  // profiling experiments only (SY_DEBUG_SKIP): 1 no observation writers, 4 no belief, 16 / 32 no observe / logic launch
  unsigned long long* stats_rep;  // [STAT_REPLICAS, SY_NUM_STATS] library-owned statistics accumulators
  uint8_t* bel_flags;  // [B] belief operation per env, logic/reset kernel -> observe kernel (library-owned)
  // fused rollout steps: the logic warps also draw the NEXT step's random valid actions (sy_sample_actions semantics)
  long long* next_actions;          // int64 [B, A] or NULL; may alias `actions` (a tile reads its actions before it writes them)
  unsigned next_counter;            // step counter of the draw (+ *next_counter_base when that is set)
  const unsigned* next_counter_base;
  // reset-only inputs
  const uint8_t* reset_mask;
  const int32_t* init_pos;
  const int32_t* init_gid;
  int restart;
  // mechanism groups (sy_set_groups; read only by the GROUPS instantiations): per-env reward weights, police budget,
  // reveal schedule and toll.  Appended so that the offsets of every field above stay where the default kernels expect them.
  const struct GroupRow* grp;        // [grp_n] library-owned table
  const int32_t* grp_id;             // [B] group of each env
  int grp_n, grp_rep;                // groups; replicas of the per-group statistics lines
  unsigned long long* grp_stats;     // [grp_rep, grp_n, SY_NUM_STATS] per-group statistics accumulators
};

// one mechanism group as the kernels read it (SyGroup prepared on the host: fp32 weights and the reveal-skip threshold
// precomputed exactly as fill_params does for the handle's config)
struct GroupRow {
  double w64[SY_NUM_REWARD_WEIGHTS];
  float w32[SY_NUM_REWARD_WEIGHTS];
  int agent_money, reveal;
  int toll;  // sy_set_group_tolls (sy_set_groups: the config's)
  int num_police, max_t;  // sy_set_group_rules (sy_set_groups: the config's), in [1, P] / [0, max_timestep]
  unsigned long long reveal_skip_thresh;
};

// the number of police an env plays with and its episode horizon: the handle's, or (GROUPS) those of the env's
// mechanism group `gr`.  Agents num_police + 1 .. A - 1 of an env are absent: pos -1, budget 0, reward 0, no action,
// and no kernel looks up a graph table at their node.
template <int GROUPS>
__device__ __forceinline__ int env_police(const Params& p, const GroupRow* gr) {
  if constexpr (GROUPS) return __ldg(&gr->num_police);
  else return p.P;
}
template <int GROUPS>
__device__ __forceinline__ int env_max_t(const Params& p, const GroupRow* gr) {
  if constexpr (GROUPS) return __ldg(&gr->max_t);
  else return p.max_t;
}
// ... whether agent a of env b is absent, when the env's group row is not at hand (false without groups)
template <int GROUPS>
__device__ __forceinline__ bool agent_absent(const Params& p, int b, int a) {
  if constexpr (GROUPS) return a > env_police<1>(p, p.grp + __ldg(p.grp_id + b));
  else return false;
}

// the toll an env pays per move (yard.py:223-229 and action_mask.py:65-76 with the toll extension: a move is legal iff
// weight + toll <= budget, and costs weight + toll): the handle's, or (GROUPS) that of the env's mechanism group `gr`
template <int GROUPS>
__device__ __forceinline__ int env_toll(const Params& p, const GroupRow* gr) {
  if constexpr (GROUPS) return __ldg(&gr->toll);
  else return p.toll;
}
// ... of env b, when its group row is not at hand
template <int GROUPS>
__device__ __forceinline__ int env_toll_of(const Params& p, int b) {
  if constexpr (GROUPS) return env_toll<1>(p, p.grp + __ldg(p.grp_id + b));
  else return p.toll;
}
// The observation writers stage one budget per (env, agent) and test `weight + wr_toll <= staged budget`.  Without
// groups that is the budget and the handle's toll.  With groups a tile mixes tolls, so they stage the headroom
// money - toll_b (at least -SY_MAX_TOLL: no overflow) and add nothing.
template <int GROUPS>
__device__ __forceinline__ int wr_toll(const Params& p) {
  if constexpr (GROUPS) return 0;
  else return p.toll;
}
template <int GROUPS>
__device__ __forceinline__ int wr_budget(const Params& p, int money, int b) {
  if constexpr (GROUPS) return money - env_toll_of<1>(p, b);
  else return money;
}


#ifdef SY_FUSED_CLOCKS  // profiling builds: per-role time inside the fused kernel, summed over CTAs (sy_debug_fused_clocks)
__device__ unsigned long long g_fused_clk[16];
#define FCLK_ADD(slot, v) do { if (lane == 0) atomicAdd(&g_fused_clk[slot], (unsigned long long)(v)); } while (0)
#define FCLK_NOW() clock64()
#else
#define FCLK_ADD(slot, v) do { } while (0)
#define FCLK_NOW() 0ll
#pragma nv_diag_suppress 177
#endif

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (same constants / counter layout as oracle/sy_oracle.py:philox4x32)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ unsigned word_of(const uint4& r, int i) {
  return i == 0 ? r.x : (i == 1 ? r.y : (i == 2 ? r.z : r.w));
}

// A distinct uniform nodes (distribution of np.random.choice(N, A, replace=False), yard.py:112-116).  Draw a depends
// only on draws 0..a-1, so the first n of them are the start nodes of a handle with n agents (an env whose mechanism
// group plays with fewer police uses the first num_police + 1 and ignores the rest).
template <typename T>
__device__ void philox_start_positions(const Params& p, unsigned env, unsigned episode, T* out, T* chosen /*A entries of scratch*/) {
  uint4 r = make_uint4(0, 0, 0, 0);
  const uint2 key = make_uint2(p.seed_lo, p.seed_hi);
  for (int a = 0; a < p.A; ++a) {
    if ((a & 3) == 0) r = philox4x32(make_uint4(env, episode, RNG_RESET_POS, (unsigned)(a >> 2)), key);
    int x = (int)__umulhi(word_of(r, a & 3), (unsigned)(p.N - a));
    for (int i = 0; i < a; ++i)
      if (x >= (int)chosen[i]) ++x;
    int j = a;
    while (j > 0 && (int)chosen[j - 1] > x) {
      chosen[j] = chosen[j - 1];
      --j;
    }
    chosen[j] = (T)x;
    out[a] = (T)x;
  }
}

// reveal schedule (src/eval/run_ablations.py:225-229) with the robustness hook of src/eval/ood_eval.py:227-229: a scheduled
// reveal is skipped with probability reveal_skip_prob, one Philox(seed; env, timestep, RNG_REVEAL_SKIP, episode) draw
// (GROUPS: the schedule of the env's mechanism group `gr` instead of the handle's)
template <int GROUPS = 0>
__device__ __forceinline__ bool reveal_now(const Params& p, unsigned env, int t, int episode, const GroupRow* gr = nullptr) {
  if constexpr (GROUPS) {
    const int reveal = __ldg(&gr->reveal);
    if (reveal <= 0 || t <= 0 || (t % reveal) != 0) return false;
    const unsigned long long thresh = __ldg(&gr->reveal_skip_thresh);
    if (thresh == 0) return true;
    const uint4 r = philox4x32(make_uint4(env, (unsigned)t, RNG_REVEAL_SKIP, (unsigned)episode), make_uint2(p.seed_lo, p.seed_hi));
    return (unsigned long long)r.x >= thresh;
  } else {
    if (p.reveal <= 0 || t <= 0 || (t % p.reveal) != 0) return false;
    if (p.reveal_skip_thresh == 0) return true;
    const uint4 r = philox4x32(make_uint4(env, (unsigned)t, RNG_REVEAL_SKIP, (unsigned)episode), make_uint2(p.seed_lo, p.seed_hi));
    return (unsigned long long)r.x >= p.reveal_skip_thresh;
  }
}

__device__ __forceinline__ int philox_graph_choice(const Params& p, unsigned env, unsigned episode) {
  uint4 r = philox4x32(make_uint4(env, episode, RNG_RESET_GRAPH, 0u), make_uint2(p.seed_lo, p.seed_hi));
  return (int)__umulhi(r.x, (unsigned)p.tb.G);
}

// ---------------------------------------------------------------------------------------------
// table lookups (read-only path; tables are tiny and L1/L2 resident)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int edge_weight(const Tables& tb, int N, int g, int u, int v) {
  return __ldg(tb.W + ((size_t)g * N + u) * tb.Ns + v);
}
// len(_get_possible_moves(pos, .)[0]) for a budget (yard.py:420-472), with the toll extension
__device__ __forceinline__ int move_count(const Tables& tb, int N, int g, int u, int money, int toll) {
  int c = money - toll;
  if (c <= 0) return 0;
  c = min(c, tb.wcap);
  return __ldg(tb.cnt + ((size_t)g * N + u) * (tb.wcap + 1) + c);
}
__device__ __forceinline__ double exp_neg(const Tables& tb, int d) {
  return (d < tb.n_exp) ? __ldg(tb.exp_neg + d) : 0.0;  // d == 0xFFFF (unreachable) -> exp(-inf) = 0
}

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
// streaming 16-byte store of the observation arrays (written once per step, read by the policy much later)
__device__ __forceinline__ void store_obs16(uint4* ptr, uint4 v) {
#if SY_STORE_HINT == 0
  __stcs(ptr, v);
#elif SY_STORE_HINT == 1
  *ptr = v;
#elif SY_STORE_HINT == 2
  __stcg(ptr, v);
#else
  __stwt(ptr, v);
#endif
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {  // LDGSTS: global -> shared, no staging register
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
// programmatic dependent launch (sm_90+): a kernel launched with the programmatic-serialisation attribute may start while
// its predecessor in the stream still runs; pdl_wait() blocks until that predecessor has completed and its writes are
// visible (a no-op for plainly launched kernels), pdl_launch_dependents() lets the successor's CTAs be scheduled early
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void named_barrier(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}
// sum of `v` over the lanes of `mask`, exact for values below 2^43 per lane: two 32-bit reductions, of the low 16 bits
// (sum < 2^21) and of the rest (sum < 2^32)
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned mask, unsigned long long v) {
  const unsigned lo = __reduce_add_sync(mask, (unsigned)(v & 0xFFFFu)), hi = __reduce_add_sync(mask, (unsigned)(v >> 16));
  return ((unsigned long long)hi << 16) + lo;
}

// bulk asynchronous copy shared -> global (TMA, SASS UBLKCP): one thread moves a whole image; the store stream never
// touches the LSU or a register.  Source / destination 16-byte aligned, size a multiple of 16.
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, unsigned bytes) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(ssrc);
#if SY_BULK_HINT == 1
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(pol));
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;\n" ::"l"(gdst), "r"(sa), "r"(bytes), "l"(pol)
               : "memory");
#else
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(sa), "r"(bytes) : "memory");
#endif
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void bulk_wait_read() {  // until at most PENDING of this thread's groups still read their source
  asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(PENDING) : "memory");
}

// warp-cooperative streaming zero-fill of n bytes at any alignment: byte head, 16-byte body, byte tail
__device__ __forceinline__ void warp_zero_bytes(uint8_t* ptr, int n, int lane) {
  const int head = min(n, (int)((16u - (unsigned)(reinterpret_cast<uintptr_t>(ptr) & 15u)) & 15u));
  if (lane < head) ptr[lane] = 0;
  uint4* v = reinterpret_cast<uint4*>(ptr + head);
  const int nvec = (n - head) >> 4;
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (int i = lane; i < nvec; i += 32) __stcs(v + i, z);
  const int done = head + (nvec << 4);
  if (lane < n - done) ptr[done + lane] = 0;
}

// ---------------------------------------------------------------------------------------------
// logic kernel pieces.  lane = env; the env's agents live in a shared-memory row (stride AS, conflict-free)
// ---------------------------------------------------------------------------------------------
struct WarpTile {
  int act[32 * AS];    // normalised actions, then visit counts / reward bits; reset kernel: Philox scratch
  int pos[32 * AS];
  int money[32 * AS];
};

// the order-dependent move rule (yard.py:155-243) and the ending (reward_calculator.py:63-79).  The env's agents are
// pulled into registers (loops fully unrolled over MAXA with predicates, so indexing is static and the rule runs on
// register compares instead of a chain of dependent shared-memory loads); an agent's own node does not change before
// its own move, so all A edge-weight lookups are issued up front (one round trip).
// the tile's graph as staged in shared memory by the observation writers of the same CTA (lagged kernel): row
// pointers, neighbours, weights.  Under a saturated store stream every global load of the dynamics queues behind the
// writers' stores in the SM's memory pipeline (~1 us per dependent round trip), so the edge-weight lookups of the
// moves and the neighbour walk of the action draw read this copy instead of the L1/L2-resident pool tables.
struct SharedGraph {
  const int* rp;
  const uint16_t* col;
  const uint8_t* wgt;
};
__device__ __forceinline__ int edge_weight_sg(const SharedGraph& sg, int u, int v) {
  int w = 0;
  for (int k = sg.rp[u], r1 = sg.rp[u + 1]; k < r1; ++k) w = (sg.col[k] == v) ? (int)sg.wgt[k] : w;
  return w;
}

// GROUPS: the toll, police count and horizon of the env's mechanism group `gr`
template <int MAXA, int GROUPS = 0, typename PosT>
__device__ __forceinline__ int move_phase(const Params& p, PosT* pos, int* money, const int* act, int g, int t, int& spent, int& moves,
                                          const SharedGraph* sg = nullptr, const GroupRow* gr = nullptr) {
  const Tables& tb = p.tb;
  const int N = p.N, P = env_police<GROUPS>(p, gr);
  int rp[MAXA], rm[MAXA], ra[MAXA], wpre[MAXA];
#pragma unroll
  for (int i = 0; i < MAXA; ++i) {
    const bool valid = i <= P;
    rp[i] = valid ? (int)pos[i] : -2 - i;  // unused slots: distinct negative values that never match a node
    rm[i] = valid ? money[i] : 0;
    ra[i] = valid ? act[i] : -1;
  }
#pragma unroll
  for (int i = 0; i < MAXA; ++i)
    wpre[i] = (i <= P && ra[i] >= 0) ? (sg ? edge_weight_sg(*sg, rp[i], ra[i]) : edge_weight(tb, N, g, rp[i], ra[i])) : 0;
  {  // MrX: legal target or stay; may not step onto a police node (yard.py:161-188)
    int tgt = rp[0];
    if (ra[0] >= 0 && wpre[0] > 0 && wpre[0] + env_toll<GROUPS>(p, gr) <= rm[0]) tgt = ra[0];
    bool occupied = false;
#pragma unroll
    for (int i = 1; i < MAXA; ++i) occupied |= (rp[i] == tgt);
    if (!occupied) rp[0] = tgt;
  }
  bool no_money = true;
#pragma unroll
  for (int i = 1; i < MAXA; ++i) {  // police in order; later police see earlier moves (yard.py:192-243)
    if (i <= P) {
      const int ai = ra[i], m = rm[i], w = wpre[i];
      const bool skipped = (ai == -1 || m == 0);  // None / DEFAULT_ACTION / broke: skipped (yard.py:210-215)
      no_money &= skipped;
      // a possible move: adjacent and affordable; otherwise the police stays (yard.py:223-229)
      const bool can = !skipped && ai >= 0 && ai != rp[i] && w != 0 && w + env_toll<GROUPS>(p, gr) <= m;
      bool occupied = false;  // may step onto MrX (capture) but not onto police (yard.py:231)
#pragma unroll
      for (int j = 1; j < MAXA; ++j) occupied |= (rp[j] == ai);
      if (can && !occupied) {
        rp[i] = ai;
        rm[i] = m - (w + env_toll<GROUPS>(p, gr));
        spent += w + env_toll<GROUPS>(p, gr);
        moves += 1;
      }
    }
  }
  bool capture = false;
#pragma unroll
  for (int i = 1; i < MAXA; ++i) capture |= (rp[i] == rp[0]);
#pragma unroll
  for (int i = 0; i < MAXA; ++i) {
    if (i <= P) {
      pos[i] = (PosT)rp[i];
      money[i] = rm[i];
    }
  }
  // reward_calculator.py:63-79; `timestep` is the pre-increment value (yard.py:345,355)
  return capture ? ST_CAPTURE : (t > env_max_t<GROUPS>(p, gr) ? ST_TIMEOUT : (no_money ? ST_NO_MONEY : ST_RUNNING));
}

struct RewardTables {  // shared-memory copies of the head of the two float64 tables (built by NumPy on the host)
  double exp_neg[EXP_SMEM];
  double coverage[COV_SMEM];
};
__device__ __forceinline__ double exp_neg_s(const Tables& tb, const RewardTables& rt, int d) {
  return d < EXP_SMEM ? rt.exp_neg[d] : exp_neg(tb, d);
}

// what an agent's reward needs from the graph tables
template <int MAXA>
struct RewardInputs {
  int dj[MAXA];  // d(u, pos[j]), j = 0 is MrX
  int mob;       // len(possible moves) with the budget the reference uses (see the quirk in the kernel)
};

// reward of agent a (reward_calculator.py:26-92 endings, :94-266 shaped), float64 value (fp32 mode: the float, widened)
// GROUPS: the weights and police count of the env's mechanism group `gr` instead of the handle's
template <int MODE, int MAXA, int GROUPS = 0>
__device__ __forceinline__ double agent_reward(const Params& p, const RewardTables& rt, const RewardInputs<MAXA>& in, int t, int status,
                                               int a, int visits_here, const GroupRow* gr = nullptr) {
  const Tables& tb = p.tb;
  auto w64 = [&](int k) { return GROUPS ? __ldg(&gr->w64[k]) : p.w64[k]; };
  auto w32 = [&](int k) { return GROUPS ? __ldg(&gr->w32[k]) : p.w32[k]; };
  const int P = env_police<GROUPS>(p, gr);
  if (status == ST_CAPTURE) return (a == 0) ? -1.0 : 1.0;
  if (status != ST_RUNNING) return (a == 0) ? 1.0 : 0.0;
  const double tt = (double)t;
  if (a == 0) {
    // reward_calculator.py:126-148
    int dmin = DIST_INF;
    long long dsum = 0;
    bool any_inf = false;
#pragma unroll
    for (int i = 1; i < MAXA; ++i) {
      if (i <= P) {
        dmin = min(dmin, in.dj[i]);
        any_inf |= (in.dj[i] == DIST_INF);
        dsum += in.dj[i];
      }
    }
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const double closest = (dmin == DIST_INF) ? inf : (double)dmin;
    const double avg = any_inf ? inf : __ddiv_rn((double)dsum, (double)P);  // np.mean: exact sum / P
    const double x1 = __ddiv_rn(-1.0, __dadd_rn(closest, 1.0));
    const double x2 = __ddiv_rn(-1.0, __dadd_rn(avg, 1.0));
    const double x3 = (double)in.mob;
    const double x4 = __dmul_rn(0.1, tt);
    if (MODE == SY_REWARD_FP64) {
      const double t1 = __dmul_rn(w64(4), x1), t2 = __dmul_rn(w64(5), x2), t3 = __dmul_rn(w64(6), x3);
      const double t4 = __dmul_rn(__dsub_rn(1.0, w64(7)), x4);
      return __dadd_rn(__dadd_rn(__dadd_rn(t1, t2), t3), t4);
    } else {
      const float t1 = __fmul_rn(w32(4), (float)x1), t2 = __fmul_rn(w32(5), (float)x2);
      const float t3 = __fmul_rn(w32(6), (float)x3);
      const float t4 = __fmul_rn(__fsub_rn(1.0f, w32(7)), (float)x4);
      return (double)__fadd_rn(__fadd_rn(__fadd_rn(t1, t2), t3), t4);
    }
  }
  // reward_calculator.py:182-227
  const int k = a - 1;
  const double mob = (double)in.mob;
  const int vc = min(visits_here, tb.n_cov - 1);
  const double cov = vc < COV_SMEM ? rt.coverage[vc] : __ldg(tb.coverage + vc);
  const double dx = exp_neg_s(tb, rt, in.dj[0]);
  double grp = 0.0, ov = 0.0, prox = 0.0;
#pragma unroll
  for (int j = 0; j < MAXA - 1; ++j) {
    if (j < P && j != k) {
      const int d = in.dj[1 + j];
      const double ex = exp_neg_s(tb, rt, d);
      grp = __dadd_rn(grp, ex);
      if (d <= 1)
        ov = __dadd_rn(ov, 1.0);
      else
        prox = __dadd_rn(prox, ex);
    }
  }
  const double x4 = __dmul_rn(0.05, tt);
  if (MODE == SY_REWARD_FP64) {
    const double u1 = __dmul_rn(w64(0), dx), u2 = __dmul_rn(w64(1), grp), u3 = __dmul_rn(w64(2), mob);
    const double u4 = __dmul_rn(__dsub_rn(1.0, w64(3)), x4);
    const double u5 = __dmul_rn(w64(9), prox), u6 = __dmul_rn(w64(10), ov), u7 = __dmul_rn(w64(8), cov);
    return __dadd_rn(__dsub_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dadd_rn(u1, u2), u3), u4), u5), u6), u7);
  } else {
    const float u1 = __fmul_rn(w32(0), (float)dx), u2 = __fmul_rn(w32(1), (float)grp);
    const float u3 = __fmul_rn(w32(2), (float)mob);
    const float u4 = __fmul_rn(__fsub_rn(1.0f, w32(3)), (float)x4);
    const float u5 = __fmul_rn(w32(9), (float)prox), u6 = __fmul_rn(w32(10), (float)ov);
    const float u7 = __fmul_rn(w32(8), (float)cov);
    return (double)__fadd_rn(__fsub_rn(__fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(u1, u2), u3), u4), u5), u6), u7);
  }
}

// state of the warp's envs back to HBM (coalesced from the smem rows), per-env scalars lane = env, visit rows of
// freshly reset envs cleared (yard.py:85), belief operation handed to the observe kernel
__device__ __forceinline__ void store_state(const Params& p, const WarpTile& wt, int b0, int nEnv, int lane, int t_new, int gid,
                                            int episode, int done, int bel_op, int revealed, bool clear_visits) {
  const int A = p.A, N = p.N;
  __syncwarp();
  for (int i = lane; i < nEnv * A; i += 32) {
    const int e = (i * p.inv_A) >> 16, a = i - e * A;  // i / A without a division (i < 512, A <= 16)
    const size_t o = (size_t)b0 * A + i;
    const int m = wt.money[e * AS + a];
    p.st.pos[o] = wt.pos[e * AS + a];
    p.st.money[o] = m;
    p.ob.agent_budget[o] = (float)m;  // yard.py:329-331
  }
  if (lane < nEnv) {
    const int b = b0 + lane;
    p.st.timestep[b] = t_new;
    p.st.graph_id[b] = gid;
    p.st.episode[b] = episode;
    p.st.done[b] = (uint8_t)done;
    p.ob.mrx_revealed[b] = revealed;
    p.bel_flags[b] = (uint8_t)bel_op;
  }
  unsigned clr = __ballot_sync(FULL, clear_visits && lane < nEnv);
  while (clr) {
    const int e = __ffs(clr) - 1;
    clr &= clr - 1;
    warp_zero_bytes(reinterpret_cast<uint8_t*>(p.st.visits + (size_t)(b0 + e) * N), N * (int)sizeof(uint16_t), lane);
  }
}

// ---------------------------------------------------------------------------------------------
// logic kernel: one CTA of 4 warps per 32-env tile, lane = env.  A warp executes a few thousand dependent
// instructions per tile, so the work is spread over the warps wherever the rule allows: warp 0 runs the
// order-dependent moves, all four warps the per-agent rewards (warp = agent), warp 0 the next-step state (Philox
// auto-reset) while warps 1..3 write the results; loads that do not depend on each other are issued together.
// MAXA (4 / 8 / 16 >= A) bounds the fully unrolled per-agent loops so that their values stay in registers.
// ---------------------------------------------------------------------------------------------
#ifdef SY_PHASE_CLOCKS
__device__ unsigned long long g_phase_clk[16];
#define PHASE_SPAN(k, t0) do { if (lane == 0) atomicAdd(&g_phase_clk[k], (unsigned long long)(clock64() - (t0))); } while (0)
#define PHASE_NOW() clock64()
#define PHASE_MARK(k) do { if (tid == 0) { const long long _c = clock64(); atomicAdd(&g_phase_clk[k], (unsigned long long)(_c - _t0)); _t0 = _c; } } while (0)
#else
#define PHASE_MARK(k) do { } while (0)
#define PHASE_SPAN(k, t0) do { } while (0)
#define PHASE_NOW() 0ll
#endif

constexpr int CNT_SMEM = 2048;  // bytes of the move-count table staged in shared memory (N * (wcap + 1) <= this); the
                                // tile smem is kept small: 9 CTAs per SM must leave room for an L1 that holds the graph tables
template <int MAXA>
struct LogicSmem {
  static constexpr int DS = MAXA * MAXA + 2;  // row stride (halfwords) of the pair-distance matrices: odd word count
  static constexpr int NPAIR = MAXA * (MAXA - 1) / 2;
  u16 pos[32 * HS];        // agents' nodes (post-move after P1, next-episode nodes after a same-step auto-reset)
  u16 reset_pos[32 * HS];  // start nodes of the next episode, drawn speculatively
  u16 dmat[32 * DS];       // all-pairs distances between the env's agents (P2); Philox scratch of warp 1 during P1
  u16 pair_ij[NPAIR];      // pair index -> (i << 8) | j, i < j
  int act[32 * AS];        // normalised actions (P0-P1); then visit counters at the police nodes (P2, as u16 rows)
  int money[32 * AS];
  RewardTables rt;
  alignas(16) uint8_t cnt[CNT_SMEM];   // move-count table of the tile's graph (when it fits and the tile sits on one graph)
  int reset_gid[32];
  int t[32], gid[32], episode[32], frozen[32], status[32];
  int t_new[32], done[32], bel[32], revealed[32], clear[32];
  long long ep_spent[32];  // statistics inputs handed from warp 0 to the statistics warp
  int spent[32], moves[32];
  int cnt_staged;
};

#ifndef SY_LOGIC_MIN_CTAS
#define SY_LOGIC_MIN_CTAS (LOGIC_WARPS == 2 ? 14 : 9)
#endif
#ifndef SY_VISIT_PREFETCH
#define SY_VISIT_PREFETCH 1
#endif
// one 32-env tile by LOGIC_THREADS threads (tid = 0 .. LOGIC_THREADS-1); BAR is the named barrier they share.
// LAGT > 0 (sy_step_lagged_kernel): the observation roles of the same CTA are still describing the tile's PREVIOUS
// state; the new state is only written back after all of them have taken their copy of the old one (named barrier
// LAG_BAR, LAGT threads: the observation warps arrive, the dynamics warps wait -- long after the arrival in practice).
constexpr int LAG_BAR = 4;
constexpr int LAG_CSR_BAR = 6;  // lagged kernel: the writers' staged graph is complete (writers arrive, dynamics warps wait)
// GROUPS: mechanism groups are set -- every env reads its group's row (reward weights, police budget, reveal schedule, toll,
// police count, horizon) once per step through the read-only path, and the statistics are also summed per group
template <int MODE, int MAXA, int BAR, int LAGT = 0, int CSRT = 0, int GROUPS = 0>
__device__ __forceinline__ void logic_tile(const Params& p, LogicSmem<MAXA>& sm, int b0, int tid, const SharedGraph* sgp = nullptr,
                                           const int* sg_valid = nullptr, unsigned extra_ctr = 0, bool draw_next = true) {
  constexpr int DS = LogicSmem<MAXA>::DS;
  const int lane = tid & 31, warp = tid >> 5;
  const int nEnv = min(32, p.B - b0);
  const int N = p.N, A = p.A;
  int P = p.P;  // (GROUPS: the env's police count, below; loaded here the instantiations without groups keep their code)
#ifdef SY_PHASE_CLOCKS
  long long _t0 = clock64();
#endif

  // ---- P0: stage the tile (coalesced) and the head of the two float64 tables
  for (int i = tid; i < EXP_SMEM; i += LOGIC_THREADS) sm.rt.exp_neg[i] = i < p.tb.n_exp ? __ldg(p.tb.exp_neg + i) : 0.0;
  for (int i = tid; i < COV_SMEM; i += LOGIC_THREADS) sm.rt.coverage[i] = __ldg(p.tb.coverage + min(i, p.tb.n_cov - 1));
  if constexpr (LAGT == 0) pdl_wait();  // everything above is independent of the state the previous kernel wrote
  for (int i = tid; i < nEnv * A; i += LOGIC_THREADS) {
    const int e = (i * p.inv_A) >> 16, a = i - e * A;  // i / A without a division (i < 512, A <= 16)
    const size_t o = (size_t)b0 * A + i;
    const long long a64 = p.actions ? p.actions[o] : (p.actions32 ? (long long)p.actions32[o] : (long long)p.actions16[o]);
    const int ps = p.st.pos[o];
    sm.act[e * AS + a] = (a64 >= 0 && a64 < N) ? (int)a64 : (a64 == -1 ? -1 : -2);
    sm.pos[e * HS + a] = (u16)ps;
    sm.money[e * AS + a] = p.st.money[o];
  }
  if (tid < 32) {
    const bool live = tid < nEnv;
    const int b = b0 + tid;
    sm.t[tid] = live ? p.st.timestep[b] : 0;
    sm.gid[tid] = live ? p.st.graph_id[b] : 0;
    sm.episode[tid] = live ? p.st.episode[b] : 0;
    sm.frozen[tid] = live ? (int)p.st.done[b] : 1;
    sm.status[tid] = ST_RUNNING;
  }
  for (int q = tid; q < A * (A - 1) / 2; q += LOGIC_THREADS) {  // pair index -> (i, j), i < j
    int i = 0, rem = q;
    while (rem >= A - 1 - i) {
      rem -= A - 1 - i;
      ++i;
    }
    sm.pair_ij[q] = (u16)((i << 8) | (i + 1 + rem));
  }
  {  // move-count table of the tile's graph (1 KB at c3): staged when every env of the tile sits on that graph
    const int g_first = p.st.graph_id[b0];
    const int gl = (lane < nEnv) ? p.st.graph_id[b0 + lane] : g_first;
    const int bytes = N * (p.tb.wcap + 1);
    const bool ok = bytes <= CNT_SMEM && __all_sync(FULL, gl == g_first);
    if (tid == 0) sm.cnt_staged = ok;
    if (ok) {
      const uint8_t* src = p.tb.cnt + (size_t)g_first * bytes;
      if ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) {  // 16-byte copies; the tail past `bytes` is never read
        for (int i = tid * 16; i < bytes; i += LOGIC_THREADS * 16)
          *reinterpret_cast<uint4*>(sm.cnt + i) = __ldg(reinterpret_cast<const uint4*>(src + i));
      } else {
        for (int i = tid; i < bytes; i += LOGIC_THREADS) sm.cnt[i] = __ldg(src + i);
      }
    }
  }
  named_barrier(BAR, LOGIC_THREADS);
  PHASE_MARK(0);
  const SharedGraph* sg = nullptr;
  if constexpr (CSRT > 0) {
    asm volatile("bar.sync %0, %1;\n" ::"n"(LAG_CSR_BAR), "n"(CSRT) : "memory");
    if (*sg_valid) sg = sgp;  // the tile sits on one graph and the writers staged it (CTA-uniform)
  }
  const bool live = lane < nEnv;
  const int b = b0 + lane;
  const int t = sm.t[lane], g = sm.gid[lane], frozen = sm.frozen[lane];
  const bool active = live && !frozen;
  u16* pos = sm.pos + lane * HS;
  int* money = sm.money + lane * AS;
  const int* act = sm.act + lane * AS;
  const GroupRow* gr = nullptr;  // this env's mechanism group (GROUPS only)
  int grp = -1;
  if constexpr (GROUPS) {
    grp = live ? __ldg(p.grp_id + b) : -1;
    gr = p.grp + max(grp, 0);
  }
  if constexpr (GROUPS) P = env_police<1>(p, gr);  // police of this env: agents P + 1 .. A - 1 are absent

  // ---- P1, four warps in parallel:
  //   warp 0    the order-dependent moves + ending
  //   warp 1    the start nodes (and graph) a same-step auto-reset WOULD draw: Philox(seed; env, episode + 1) does not
  //             depend on the outcome, so it is computed off the critical path
  //   warps 2,3 visit counters at both nodes each police can end on (its node or its action target): the HBM
  //             round trip of the read-modify-write overlaps the moves
  int spent = 0, moves = 0;
  [[maybe_unused]] const long long tp1 = PHASE_NOW();
  if (warp == 0) {
    if (active) sm.status[lane] = move_phase<MAXA, GROUPS>(p, pos, money, act, g, t, spent, moves, sg, gr);
    PHASE_SPAN(8, tp1);
  } else if (warp == 1 && p.auto_reset && active) {
    const unsigned env_id = (unsigned)(p.env_offset + (unsigned long long)b);
    const unsigned ep = (unsigned)(sm.episode[lane] + 1);
    sm.reset_gid[lane] = p.resample_graph ? philox_graph_choice(p, env_id, ep) : g;
    philox_start_positions(p, env_id, ep, sm.reset_pos + lane * HS, sm.dmat + lane * HS);  // (absent agents: unused)
    PHASE_SPAN(9, tp1);  // (lane-divergent branch: no warp-level synchronisation in here)
  }
  named_barrier(BAR, LOGIC_THREADS);
  PHASE_MARK(1);
  [[maybe_unused]] const long long tp2 = PHASE_NOW();

  // ---- P2a: every table lookup of the rewards, once: the A(A-1)/2 distinct distances between the env's agents (the
  // reference asks Pathfinder for each of them 2-4 times, reward_calculator.py:126-227) and the visit counters at the
  // police nodes, spread over the warps and all issued before any is consumed.  Divergent 2-byte gathers are the
  // scarce resource of this kernel (one L1 wavefront per lane), so each is loaded exactly once.
  const int status = sm.status[lane];
  const bool shaped = active && status == ST_RUNNING;
  {
    constexpr int NPQ = (LogicSmem<MAXA>::NPAIR + LOGIC_WARPS - 1) / LOGIC_WARPS;
    constexpr int NVQ = (MAXA + LOGIC_WARPS - 1) / LOGIC_WARPS;
    const int npairs = A * (A - 1) / 2;
    const uint16_t* Dg = p.tb.D + (size_t)g * N * N;
    const uint16_t* vrow = p.st.visits + (size_t)b * N;
    int dq[NPQ], vq[NVQ];
#pragma unroll
    for (int k = 0; k < NPQ; ++k) {
      const int q = warp + k * LOGIC_WARPS;
      dq[k] = 0;
      if (shaped && q < npairs) {
        const int ij = sm.pair_ij[q];
        if (!GROUPS || (ij & 0xff) <= P) dq[k] = __ldg(Dg + (size_t)pos[ij >> 8] * N + pos[ij & 0xff]);  // (i < j)
      }
    }
#pragma unroll
    for (int k = 0; k < NVQ; ++k) {
      const int i = 1 + warp + k * LOGIC_WARPS;
      vq[k] = (active && i <= P) ? (int)vrow[pos[i]] : 0;
    }
#pragma unroll
    for (int k = 0; k < NPQ; ++k) {
      const int q = warp + k * LOGIC_WARPS;
      if (shaped && q < npairs) {
        const int ij = sm.pair_ij[q], i = ij >> 8, j = ij & 0xff;
        sm.dmat[lane * DS + i * MAXA + j] = (u16)dq[k];
        sm.dmat[lane * DS + j * MAXA + i] = (u16)dq[k];
      }
    }
#pragma unroll
    for (int k = 0; k < NVQ; ++k) {
      const int i = 1 + warp + k * LOGIC_WARPS;
      if (active && i <= P) reinterpret_cast<u16*>(sm.act)[lane * HS + i] = (u16)vq[k];
    }
  }
  if (warp == 0) PHASE_MARK(1);
  if (warp == 0) PHASE_SPAN(10, tp2);
  if (warp == 3) PHASE_SPAN(11, tp2);
  named_barrier(BAR, LOGIC_THREADS);
  PHASE_MARK(2);

  // ---- P2b: visit counts (yard.py:244-245) and rewards, warp = agent (agents warp, warp + LOGIC_WARPS, ...)
  if (live) {
#pragma unroll 1
    for (int a = (warp + LOGIC_WARPS - 1) % LOGIC_WARPS; a < A; a += LOGIC_WARPS) {  // warp 0 (moves, next state) gets the fewest
      double r64 = 0.0;  // (absent agents: 0)
      if (active && (!GROUPS || a <= P)) {
        int visits_here = 0;
        const int u = pos[a];
        if (a > 0) {  // police never share a node (yard.py:231): the P counters of an env are distinct addresses
          visits_here = (int)reinterpret_cast<const u16*>(sm.act)[lane * HS + a] + 1;
          p.st.visits[(size_t)b * N + u] = (uint16_t)min(visits_here, 0xFFFF);
        }
        RewardInputs<MAXA> in;
        in.mob = 0;
        if (status == ST_RUNNING) {
#pragma unroll
          for (int j = 0; j < MAXA; ++j) in.dj[j] = (j <= P && j != a) ? (int)sm.dmat[lane * DS + a * MAXA + j] : 0;
          // QUIRK reward_calculator.py:190: the police mobility term uses the budget of agent index a-1 (not a)
          const int mny = money[a == 0 ? 0 : a - 1];
          const int c = min(mny - env_toll<GROUPS>(p, gr), p.tb.wcap);
          if (c > 0) in.mob = sm.cnt_staged ? (int)sm.cnt[u * (p.tb.wcap + 1) + c] : move_count(p.tb, N, g, u, mny, env_toll<GROUPS>(p, gr));
        }
        r64 = agent_reward<MODE, MAXA, GROUPS>(p, sm.rt, in, t, status, a, visits_here, gr);
      }
      p.out.reward[(size_t)b * A + a] = (float)r64;
      if (p.out.reward64) p.out.reward64[(size_t)b * A + a] = r64;
    }
  }
  if (warp == 0) PHASE_MARK(3);
  named_barrier(BAR, LOGIC_THREADS);
  PHASE_MARK(4);

  // ---- P3: warps 1..3 write the flags (coalesced)  ||  warp 0 computes the next-step state
  if (warp > 0) {
    for (int i = tid - 32; i < nEnv * A; i += LOGIC_THREADS - 32) {
      const int e = (i * p.inv_A) >> 16;
      const size_t o = (size_t)b0 * A + i;
      const int st = sm.status[e];
      const bool term = (st == ST_CAPTURE) || (st == ST_NO_MONEY), trunc = (st == ST_TIMEOUT);
      p.out.terminated[o] = term;
      p.out.truncated[o] = trunc;
      p.out.done[o] = term || trunc || sm.frozen[e];
      if (p.out.status && i - e * A == 0)  // one byte per env for host loops (SY_STATUS_*)
        p.out.status[b0 + e] = (uint8_t)((term ? SY_STATUS_TERMINATED : 0) | (trunc ? SY_STATUS_TRUNCATED : 0) | (sm.frozen[e] ? SY_STATUS_FROZEN : 0));
    }
  } else {
    // timestep, reveal schedule, same-step auto-reset, statistics
    long long ep_spent = 0;
    int t_new = t, done = frozen, bel = BEL_KEEP, revealed = -1, episode = sm.episode[lane], gnew = g;
    bool clear_visits = false;
    if (live) {
      if (active) {
        t_new = t + 1;  // yard.py:355
        p.out.winner[b] = (int8_t)(status == ST_CAPTURE ? SY_WINNER_POLICE : (status == ST_RUNNING ? SY_WINNER_NONE : SY_WINNER_MRX));
        bel = BEL_PROPAGATE;
        if (status != ST_RUNNING) {
          const int agent_money = GROUPS ? __ldg(&gr->agent_money) : p.agent_money;
          ep_spent = (long long)P * agent_money;  // every police starts an episode with agent_money (yard.py:117-119)
          for (int i = 1; i <= P; ++i) ep_spent -= money[i];
          if (p.auto_reset) {  // same-step auto-reset: the observation describes the fresh episode
            episode += 1;
            gnew = sm.reset_gid[lane];
            money[0] = p.mrx_money;
            pos[0] = sm.reset_pos[lane * HS];
            for (int i = 1; i <= P; ++i) {  // (absent agents keep pos / money: P4 stores their fixed values)
              money[i] = agent_money;
              pos[i] = sm.reset_pos[lane * HS + i];
            }
            t_new = 0;
            clear_visits = true;
            bel = BEL_UNIFORM;
          } else {
            done = 1;
          }
        }
      } else {
        p.out.winner[b] = SY_WINNER_NONE;
      }
      // reveal schedule (src/eval/run_ablations.py:225-229) on the new timestep
      const bool rev = reveal_now<GROUPS>(p, (unsigned)(p.env_offset + (unsigned long long)b), t_new, episode, gr);
      if (rev && bel == BEL_PROPAGATE) bel = BEL_DELTA;
      if constexpr (GROUPS) revealed = (__ldg(&gr->reveal) <= 0 || rev) ? (int)pos[0] : -1;
      else revealed = (p.reveal <= 0 || rev) ? (int)pos[0] : -1;
    }
    sm.t_new[lane] = t_new;
    sm.gid[lane] = gnew;
    sm.episode[lane] = episode;
    sm.done[lane] = done;
    sm.bel[lane] = bel;
    sm.revealed[lane] = revealed;
    sm.clear[lane] = clear_visits;
    sm.ep_spent[lane] = ep_spent;
    sm.spent[lane] = spent;
    sm.moves[lane] = moves;
    PHASE_MARK(5);
  }
  named_barrier(BAR, LOGIC_THREADS);
  PHASE_MARK(6);

  // ---- P4: new state back to HBM (coalesced), visit rows of freshly reset envs cleared (yard.py:85); the last warp
  // (lightest reward share) reduces the tile's episode statistics, off warp 0's critical path
  if constexpr (LAGT > 0) asm volatile("bar.sync %0, %1;\n" ::"n"(LAG_BAR), "n"(LAGT) : "memory");
  if (warp == LOGIC_WARPS - 1 && p.out.stats) {
    const int st = sm.status[lane];
    const bool fin = active && st != ST_RUNNING;
    // Sums over 32 lanes.  The squared length (< 2^32 with max_timestep <= SY_MAX_TIMESTEP) and the budget spent in the
    // episode (<= 15 x (2^31 - 1)) are summed in 64 bits; every other sum stays below 2^31 in int: counts <= 32,
    // lengths <= 32 x (SY_MAX_TIMESTEP + 2) < 2^22, a step's police charges <= 32 x 15 x (255 + SY_MAX_TOLL) < 2^29
    const int len = fin ? t + 1 : 0;  // episode length = timestep after the final step (yard.py:355)
    int n_step = active, n_ep = fin, n_pol = fin && st == ST_CAPTURE, n_mrx = fin && st != ST_CAPTURE;
    int n_trunc = fin && st == ST_TIMEOUT, n_broke = fin && st == ST_NO_MONEY;
    int len_sum = len, len_pol = n_pol ? len : 0, len_mrx = n_mrx ? len : 0;
    unsigned long long len_sq = (unsigned long long)len * len, ep_spent = (unsigned long long)sm.ep_spent[lane];
    int spent = sm.spent[lane], moves = sm.moves[lane];
    if constexpr (GROUPS) {
      // per-group sums: the lanes of each distinct group reduce together, one leader adds them to the group's line
      const int v[SY_STAT_POLICE_MOVES + 1] = {n_step, n_ep, n_mrx, n_pol, n_trunc, n_broke, len_sum, spent,
                                               0, len_pol, len_mrx, 0, moves};
      const unsigned same = __match_any_sync(FULL, grp);
      const bool leader = grp >= 0 && lane == __ffs(same) - 1;
      unsigned long long* line = p.grp_stats + ((size_t)(blockIdx.x % p.grp_rep) * p.grp_n + max(grp, 0)) * SY_NUM_STATS;
#pragma unroll
      for (int k = 0; k <= SY_STAT_POLICE_MOVES; ++k) {
        const unsigned long long sum = k == SY_STAT_SUM_SQ_EPISODE_LENGTH ? warp_sum_u64(same, len_sq)
                                       : k == SY_STAT_SUM_EPISODE_BUDGET_SPENT ? warp_sum_u64(same, ep_spent)
                                       : (unsigned long long)__reduce_add_sync(same, v[k]);
        if (leader && sum) atomicAdd(line + k, sum);
      }
    }
    // per-tile sums -> one of STAT_REPLICAS library-owned accumulator lines (sy_stats folds them into the caller's
    // vector): with a single shared line the 13 atomics of all 2048 tiles serialised in one L2 slice (8 us per step)
    n_step = __reduce_add_sync(FULL, n_step);
    n_ep = __reduce_add_sync(FULL, n_ep);
    spent = __reduce_add_sync(FULL, spent);
    moves = __reduce_add_sync(FULL, moves);
    if (n_ep) {  // warp-uniform
      n_mrx = __reduce_add_sync(FULL, n_mrx);
      n_pol = __reduce_add_sync(FULL, n_pol);
      n_trunc = __reduce_add_sync(FULL, n_trunc);
      n_broke = __reduce_add_sync(FULL, n_broke);
      len_sum = __reduce_add_sync(FULL, len_sum);
      len_sq = warp_sum_u64(FULL, len_sq);
      len_pol = __reduce_add_sync(FULL, len_pol);
      len_mrx = __reduce_add_sync(FULL, len_mrx);
      ep_spent = warp_sum_u64(FULL, ep_spent);
    }
    unsigned long long v = 0;  // every lane holds all sums: lane k adds statistic k (one atomic instruction for the warp)
    switch (lane) {
      case SY_STAT_ENV_STEPS: v = n_step; break;
      case SY_STAT_EPISODES: v = n_ep; break;
      case SY_STAT_MRX_WINS: v = n_mrx; break;
      case SY_STAT_POLICE_WINS: v = n_pol; break;
      case SY_STAT_TRUNCATIONS: v = n_trunc; break;
      case SY_STAT_OUT_OF_MONEY: v = n_broke; break;
      case SY_STAT_SUM_EPISODE_LENGTH: v = len_sum; break;
      case SY_STAT_SUM_BUDGET_SPENT: v = spent; break;
      case SY_STAT_SUM_SQ_EPISODE_LENGTH: v = len_sq; break;
      case SY_STAT_SUM_LENGTH_POLICE_WINS: v = len_pol; break;
      case SY_STAT_SUM_LENGTH_MRX_WINS: v = len_mrx; break;
      case SY_STAT_SUM_EPISODE_BUDGET_SPENT: v = ep_spent; break;
      case SY_STAT_POLICE_MOVES: v = moves; break;
      default: break;
    }
    if (v) atomicAdd(p.stats_rep + (size_t)(blockIdx.x % STAT_REPLICAS) * SY_NUM_STATS + lane, v);
  }
  for (int i = tid; i < nEnv * A; i += LOGIC_THREADS) {
    const int e = (i * p.inv_A) >> 16, a = i - e * A;  // i / A without a division (i < 512, A <= 16)
    const size_t o = (size_t)b0 * A + i;
    const bool absent = agent_absent<GROUPS>(p, b0 + e, a);
    const int m = absent ? 0 : sm.money[e * AS + a];
    p.st.pos[o] = absent ? -1 : (int)sm.pos[e * HS + a];
    p.st.money[o] = m;
    p.ob.agent_budget[o] = (float)m;  // yard.py:329-331
  }
  if (tid < nEnv) {
    const int bb = b0 + tid;
    p.st.timestep[bb] = sm.t_new[tid];
    p.st.graph_id[bb] = sm.gid[tid];
    p.st.episode[bb] = sm.episode[tid];
    p.st.done[bb] = (uint8_t)sm.done[tid];
    p.ob.mrx_revealed[bb] = sm.revealed[tid];
    p.bel_flags[bb] = (uint8_t)sm.bel[tid];
  }
  unsigned clr = __ballot_sync(FULL, live && sm.clear[lane]);
  for (int n = 0; clr; ++n) {
    const int e = __ffs(clr) - 1;
    clr &= clr - 1;
    if (n % LOGIC_WARPS == warp)
      warp_zero_bytes(reinterpret_cast<uint8_t*>(p.st.visits + (size_t)(b0 + e) * N), N * (int)sizeof(uint16_t), lane);
  }
  if (p.next_actions && draw_next) {
    // the next step's random valid actions from the NEW state still held in shared memory: the same draw as
    // sy_sample_actions_kernel (Philox(seed; env, step counter, agent) -> the pick-th affordable neighbour)
    const unsigned ctr = p.next_counter + (p.next_counter_base ? *p.next_counter_base : 0u) + extra_ctr;
    for (int i = tid; i < nEnv * A; i += LOGIC_THREADS) {
      const int e = (i * p.inv_A) >> 16, a = i - e * A;
      if (agent_absent<GROUPS>(p, b0 + e, a)) {  // no action, no table lookup
        p.next_actions[(size_t)b0 * A + i] = -1;
        continue;
      }
      const int gg = sm.gid[e], u = (int)sm.pos[e * HS + a], m = sm.money[e * AS + a];
      // a same-step auto-reset with resample_graph may have moved the env to another graph than the staged one
      const bool use_sg = sg != nullptr && !p.resample_graph;
      int nvalid;
      if (use_sg && sm.cnt_staged) {
        const int c = min(m - env_toll_of<GROUPS>(p, b0 + e), p.tb.wcap);
        nvalid = c > 0 ? (int)sm.cnt[u * (p.tb.wcap + 1) + c] : 0;
      } else {
        nvalid = move_count(p.tb, N, gg, u, m, env_toll_of<GROUPS>(p, b0 + e));
      }
      long long act = -1;
      if (nvalid > 0) {
        const unsigned env_id = (unsigned)(p.env_offset + (unsigned long long)(b0 + e));
        const uint4 r = philox4x32(make_uint4(env_id, ctr, RNG_ACTION, (unsigned)a), make_uint2(p.seed_lo, p.seed_hi));
        int pick = (int)__umulhi(r.x, (unsigned)nvalid);
        if (use_sg) {
          for (int k = sg->rp[u];; ++k) {  // the pick-th affordable neighbour exists
            if ((int)sg->wgt[k] + env_toll_of<GROUPS>(p, b0 + e) <= m) {
              if (pick == 0) {
                act = sg->col[k];
                break;
              }
              --pick;
            }
          }
        } else {
          const uint8_t* wg = p.tb.wgt + (size_t)gg * p.tb.nnz_stride;
          for (int k = __ldg(p.tb.row_ptr + (size_t)gg * (N + 1) + u);; ++k) {  // the pick-th affordable neighbour exists
            if (__ldg(wg + k) + env_toll_of<GROUPS>(p, b0 + e) <= m) {
              if (pick == 0) {
                act = __ldg(p.tb.col + (size_t)gg * p.tb.nnz_stride + k);
                break;
              }
              --pick;
            }
          }
        }
      }
      p.next_actions[(size_t)b0 * A + i] = act;
    }
  }
  PHASE_MARK(7);
}

template <int MODE, int MAXA, int GROUPS = 0>
__global__ void __launch_bounds__(LOGIC_THREADS, SY_LOGIC_MIN_CTAS) sy_logic_kernel(const Params p) {
  __shared__ LogicSmem<MAXA> sm;
  pdl_launch_dependents();  // the observation kernel's CTAs may take the slots the last wave of this grid leaves free
  logic_tile<MODE, MAXA, 3, 0, 0, GROUPS>(p, sm, blockIdx.x * 32, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------
// fill kernel: the zero fill of the float32 node_features array is 63 % of a step's bytes and does not depend on the
// state, while the dynamics and the belief propagation are latency / issue bound and leave HBM idle.  In the split step
// (step_impl) this kernel therefore runs from the first microsecond of the step NEXT TO the dynamics kernel: a handful
// of threads per SM hand the whole array to the TMA engine (cp.async.bulk from a shared-memory zero page: no LSU, no
// registers, ~2 % of the issue slots) and wait for completion; the observation writers later only store the 16-byte
// granules that hold a one (p.nf_prefilled).  Micro-benchmark (tools/exp/tma_fill.cu): 6.1-6.2 TB/s with 1 CTA per SM.
// ---------------------------------------------------------------------------------------------
#ifndef SY_FILL_PAGE
#define SY_FILL_PAGE 8192
#endif
constexpr int FILL_THREADS = 64;
#ifndef SY_SPLIT_MIN_ENVS
#define SY_SPLIT_MIN_ENVS 8192
#endif
constexpr int SPLIT_MIN_ENVS = SY_SPLIT_MIN_ENVS;  // smaller batches are launch-latency bound: two plain launches
__global__ void __launch_bounds__(FILL_THREADS) sy_fill_kernel(uint8_t* dst, size_t bytes) {
  __shared__ __align__(128) uint8_t zero_page[SY_FILL_PAGE];
  for (int i = threadIdx.x * 16; i < SY_FILL_PAGE; i += FILL_THREADS * 16) *reinterpret_cast<uint4*>(zero_page + i) = make_uint4(0, 0, 0, 0);
  fence_proxy_async_smem();
  __syncthreads();
  const size_t body = bytes & ~(size_t)15;
  const size_t stride = (size_t)gridDim.x * FILL_THREADS * SY_FILL_PAGE;
  for (size_t o = ((size_t)blockIdx.x * FILL_THREADS + threadIdx.x) * SY_FILL_PAGE; o < body; o += stride)
    bulk_store(dst + o, zero_page, (unsigned)min((size_t)SY_FILL_PAGE, body - o));
  bulk_commit();
  if (blockIdx.x == 0 && threadIdx.x < (int)(bytes - body)) dst[body + threadIdx.x] = 0;
  asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");  // complete before the kernel ends: the ones follow in stream order
}

// ---------------------------------------------------------------------------------------------
// reset kernel (yard.py:80-142): re-initialise the masked envs (same warp = 32 envs layout)
// ---------------------------------------------------------------------------------------------
// GROUPS: police budgets, police count and reveal schedule of each env's mechanism group
template <int GROUPS = 0>
__global__ void __launch_bounds__(LOGIC_THREADS) sy_reset_kernel(const Params p) {
  __shared__ WarpTile wts[LOGIC_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b0 = (blockIdx.x * (LOGIC_THREADS / 32) + warp) * 32;
  if (b0 >= p.B) return;
  WarpTile& wt = wts[warp];
  const int nEnv = min(32, p.B - b0);
  const int A = p.A;
  const bool live = lane < nEnv;
  const int b = b0 + lane;
  const bool rst = live && (p.reset_mask == nullptr || p.reset_mask[b] != 0);
  const unsigned rst_mask = __ballot_sync(FULL, rst);
  for (int i = lane; i < nEnv * A; i += 32) {
    const int e = (i * p.inv_A) >> 16, a = i - e * A;  // i / A without a division (i < 512, A <= 16)
    const size_t o = (size_t)b0 * A + i;
    if (agent_absent<GROUPS>(p, b0 + e, a)) {  // (init_pos entries of absent agents are ignored)
      wt.money[e * AS + a] = 0;
      wt.pos[e * AS + a] = -1;
    } else if ((rst_mask >> e) & 1u) {
      const int agent_money = GROUPS ? __ldg(&p.grp[__ldg(p.grp_id + b0 + e)].agent_money) : p.agent_money;
      wt.money[e * AS + a] = (a == 0) ? p.mrx_money : agent_money;  // yard.py:117-119
      wt.pos[e * AS + a] = p.init_pos ? p.init_pos[o] : 0;
    } else {
      wt.money[e * AS + a] = p.st.money[o];
      wt.pos[e * AS + a] = p.st.pos[o];
    }
  }
  __syncwarp();
  int t = 0, g = 0, episode = 0, done = 1, revealed = -1;
  if (live) {
    if (rst) {
      episode = p.restart ? 0 : p.st.episode[b] + 1;
      done = 0;
      g = p.init_gid ? p.init_gid[b] : p.st.graph_id[b];
      if (p.init_pos == nullptr) {
        const unsigned env_id = (unsigned)(p.env_offset + (unsigned long long)b);
        if (p.resample_graph && p.init_gid == nullptr) g = philox_graph_choice(p, env_id, (unsigned)episode);
        philox_start_positions(p, env_id, (unsigned)episode, wt.pos + lane * AS, wt.act + lane * AS);
        if constexpr (GROUPS)  // the draws past the env's police are not used
          for (int a = env_police<1>(p, p.grp + __ldg(p.grp_id + b)) + 1; a < A; ++a) wt.pos[lane * AS + a] = -1;
      }
    } else {
      t = p.st.timestep[b];
      episode = p.st.episode[b];
      done = p.st.done[b];
      g = p.st.graph_id[b];
    }
    const GroupRow* gr = GROUPS ? p.grp + __ldg(p.grp_id + b) : nullptr;
    const bool rev = reveal_now<GROUPS>(p, (unsigned)(p.env_offset + (unsigned long long)b), t, episode, gr);
    if constexpr (GROUPS) revealed = (__ldg(&gr->reveal) <= 0 || rev) ? wt.pos[lane * AS] : -1;
    else revealed = (p.reveal <= 0 || rev) ? wt.pos[lane * AS] : -1;
  }
  store_state(p, wt, b0, nEnv, lane, t, g, episode, done, rst ? BEL_UNIFORM : BEL_KEEP, revealed, rst);
}

// ---------------------------------------------------------------------------------------------
// observe kernel: everything that is a pure function of the new state (yard.py:271-335 observation assembly
// and the belief_map).  One CTA per 32-env tile, warp-specialised and barrier-free between the roles:
//   writer warps: stream the dense observations.  Per env: 16-byte zero stores over the env's contiguous
//                 action_mask [A,N] and node_features [N,A] regions, then -- while those lines are still in
//                 L2 -- the few ones (affordable neighbours, one-hot positions).  Pure HBM write stream.
//   belief warps: belief propagation (belief_module.py:69-111 in expectation) as a lane = env SpMM over the
//                 tile's rows held TRANSPOSED in shared memory; latency-bound, hidden under the write stream.
// ---------------------------------------------------------------------------------------------
constexpr int BSTRIDE = TILE + 1;
constexpr int BEL_JMAX = 128;  // nodes per belief warp on the fast path -> N <= BEL_WARPS * 128

// warp-cooperative copy of n bytes from shared memory to global memory; src and dst have the same 16-byte phase
__device__ __forceinline__ void warp_copy_bytes(uint8_t* dst, const uint8_t* src, int n, int lane) {
  const int head = min(n, (int)((16u - (unsigned)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u));
  if (lane < head) dst[lane] = src[lane];
  const int nvec = (n - head) >> 4;
  uint4* d = reinterpret_cast<uint4*>(dst + head);
  const uint4* sv = reinterpret_cast<const uint4*>(src + head);
#pragma unroll 2
  for (int i = lane; i < nvec; i += 32) store_obs16(d + i, sv[i]);
  const int done = head + (nvec << 4);
  if (lane < n - done) dst[done + lane] = src[done + lane];
}

// node_features of one env: n = N*A floats, all zero except the agents' one-hot entries at flat index fpos[a]
// (yard.py:279-290).  The region is zero-filled with 16-byte stores; lane a then overwrites, with one full 16-byte
// store, the chunk that holds agent a's one (assembled in registers from all agents that fall into it).  Measured:
// rewriting a handful of whole chunks costs nothing, whereas byte-sized ones after the fill cost 60 %.
// the same after a completed zero fill of the region (p.nf_prefilled): only the ones -- whole granules when the env rows
// are granule-aligned, single floats otherwise
__device__ __forceinline__ void warp_write_node_feature_ones(float* nf, int n, const int* fpos, int A, int lane) {
  if (lane >= A || fpos[lane] < 0) return;
  if ((n & 3) || (reinterpret_cast<uintptr_t>(nf) & 15u)) {
    nf[fpos[lane]] = 1.0f;
    return;
  }
  const int myc = fpos[lane] >> 2;
  uint4 v = make_uint4(0, 0, 0, 0);
  for (int a = 0; a < A; ++a) {
    const int f = fpos[a];
    if (f >= 0 && (f >> 2) == myc) {
      const unsigned one = 0x3f800000u;
      const int sub = f & 3;
      v.x = sub == 0 ? one : v.x;
      v.y = sub == 1 ? one : v.y;
      v.z = sub == 2 ? one : v.z;
      v.w = sub == 3 ? one : v.w;
    }
  }
  store_obs16(reinterpret_cast<uint4*>(nf) + myc, v);
}

__device__ __forceinline__ void warp_write_node_features(float* nf, int n, const int* fpos /*smem, A entries, -1 = none*/,
                                                          int A, int lane) {
  const int head = min(n, (int)(((16u - (unsigned)(reinterpret_cast<uintptr_t>(nf) & 15u)) & 15u) >> 2));
  const int nvec = (n - head) >> 2;
  const int tail0 = head + (nvec << 2);
  if (lane < head || (lane >= 32 - (n - tail0))) {  // the few floats before / after the aligned body
    const int f = lane < head ? lane : tail0 + (lane - (32 - (n - tail0)));
    float v = 0.0f;
    for (int a = 0; a < A; ++a) v = (fpos[a] == f) ? 1.0f : v;
    nf[f] = v;
  }
  uint4* body = reinterpret_cast<uint4*>(nf + head);
  const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll 4
  for (int i = lane; i < nvec; i += 32) store_obs16(body + i, z);
  __syncwarp();  // orders the zero stores before the chunks below (same warp, same addresses)
#if SY_NF_SCALAR_ONES
  // one 4-byte store per agent: no merging of ones that share a chunk (A x A loop) is needed; the lines are still in L2
  if (lane < A) {
    const int f0 = fpos[lane] - head;
    if (fpos[lane] >= 0 && f0 >= 0 && f0 < (nvec << 2)) __stcs(reinterpret_cast<float*>(body) + f0, 1.0f);
  }
#else
  if (lane < A) {
    const int f0 = fpos[lane] - head;
    if (fpos[lane] >= 0 && f0 >= 0 && f0 < (nvec << 2)) {
      const int myc = f0 >> 2;  // body chunk that holds this lane's agent
      uint4 v = z;
      for (int a = 0; a < A; ++a) {
        const int f = fpos[a] - head;
        if (fpos[a] >= 0 && (f >> 2) == myc) {
          const unsigned one = 0x3f800000u;
          const int sub = f & 3;
          v.x = sub == 0 ? one : v.x;
          v.y = sub == 1 ? one : v.y;
          v.z = sub == 2 ? one : v.z;
          v.w = sub == 3 ? one : v.w;
        }
      }
      store_obs16(body + myc, v);  // (match.any + redux instead of this loop was measured 18 % SLOWER per step: MATCH is slow)
    }
  }
#endif
}

// writer warps: stream the dense observations of the tile.  Everything the ones depend on is staged into shared
// memory first (one round trip for the whole tile): agents' nodes and budgets, reveal flags and -- when the tile sits
// on one graph and its CSR fits -- the graph's row pointers / neighbours / weights.  Each env's action_mask rows are
// assembled in a per-warp shared-memory image and copied out, node_features are zero-filled and the (at most A) chunks
// with a one rewritten whole: no byte-sized stores anywhere (they cost 60 % extra time when tried).  GROUPS: budgets are
// staged as headroom against each env's group toll (wr_budget).
template <int WRW, bool PREFILLED = false, int LAGT = 0, int CSRT = 0, int GROUPS = 0>
__device__ __forceinline__ void writer_role(const Params& p, unsigned char* dyn, int tile0, int nEnv, int w, int lane,
                                            int* lag_staged = nullptr) {
  const Tables& tb = p.tb;
  const int N = p.N, A = p.A;
  int* s_pos = reinterpret_cast<int*>(dyn + p.wr_off);  // [TILE * A]
  int* s_money = s_pos + TILE * A;                      // [TILE * A]
  int* s_rev = s_money + TILE * A;                      // [TILE]
  int* s_gid = s_rev + TILE;                            // [TILE]
  int* s_fpos = s_gid + TILE;                           // [WRW * SY_MAX_AGENTS] flat node_features index per agent
  uint8_t* s_img = reinterpret_cast<uint8_t*>(s_fpos + WRW * SY_MAX_AGENTS) + (size_t)w * p.wr_img_stride;  // mask image
  int* s_rp = reinterpret_cast<int*>(dyn + p.wr_off_csr);  // [N + 1]
  uint16_t* s_col = reinterpret_cast<uint16_t*>(s_rp + N + 1);
  uint8_t* s_wgt = reinterpret_cast<uint8_t*>(s_col + tb.nnz_stride);
  const int tw = w * 32 + lane;
  const int gl = (lane < nEnv) ? p.st.graph_id[tile0 + lane] : -1;
  const int g0 = __shfl_sync(FULL, gl, 0);
  const bool staged = p.wr_stage_csr && __all_sync(FULL, gl == g0 || gl < 0);
  for (int i = tw; i < nEnv * A; i += WRW * 32) {
    s_pos[i] = p.st.pos[(size_t)tile0 * A + i];
    s_money[i] = wr_budget<GROUPS>(p, p.st.money[(size_t)tile0 * A + i], tile0 + ((i * p.inv_A) >> 16));
  }
  if (tw < nEnv) {
    s_rev[tw] = p.ob.mrx_revealed[tile0 + tw];
    s_gid[tw] = gl;
  }
  if (staged) {
    const int32_t* grp = tb.row_ptr + (size_t)g0 * (N + 1);
    const int nnz = __ldg(grp + N);
    for (int i = tw; i <= N; i += WRW * 32) s_rp[i] = __ldg(grp + i);
    for (int k = tw; k < nnz; k += WRW * 32) {
      s_col[k] = __ldg(tb.col + (size_t)g0 * tb.nnz_stride + k);
      s_wgt[k] = __ldg(tb.wgt + (size_t)g0 * tb.nnz_stride + k);
    }
    if (p.bel_share_csr) {
      float* s_inv = reinterpret_cast<float*>(dyn + p.wr_off_csr + (((N + 1) * 4 + tb.nnz_stride * 3 + 3) & ~3));
      uint16_t* s_perm = reinterpret_cast<uint16_t*>(s_inv + N);
      for (int i = tw; i < N; i += WRW * 32) {
        s_inv[i] = __ldg(tb.inv_deg + (size_t)g0 * N + i);
        s_perm[i] = __ldg(tb.deg_perm + (size_t)g0 * N + i);
      }
      // padded neighbour lists for the belief gather: every node's list is a multiple of 4 node ids (pads point at the
      // zero slot N), so the gather reads 4 ids with one 8-byte load and has no per-neighbour loop control
      uint16_t* s_pptr = reinterpret_cast<uint16_t*>(dyn + p.wr_off_csr + p.wr_off_pad);  // [N + 1] list starts (entries)
      uint16_t* s_pcol = s_pptr + ((N + 1 + 3) & ~3);                                        // 8-byte aligned
      const int32_t* gpp = tb.pack_ptr + (size_t)g0 * (N + 1);
      const int2* gpk = tb.nbr_pack + (size_t)g0 * tb.pack_stride;
      const int npk = __ldg(gpp + N);
      for (int i = tw; i <= N; i += WRW * 32) s_pptr[i] = (uint16_t)__ldg(gpp + i);
      for (int k = tw; k < npk; k += WRW * 32) {
        const int2 en = __ldg(gpk + k);  // {byte offset of the neighbour's row in the transposed tile, bits of 1/deg}; pads are {0, 0}
        s_pcol[k] = en.y ? (uint16_t)((unsigned)en.x / (BSTRIDE * 4u)) : (uint16_t)N;
      }
    }
  }
  for (int i = lane * 16; i < p.wr_img_stride; i += 32 * 16) *reinterpret_cast<uint4*>(s_img + i) = make_uint4(0, 0, 0, 0);
  if constexpr (CSRT > 0) {
    if (tw == 0) *lag_staged = staged ? 1 : 0;
  }
  named_barrier(2, WRW * 32);
  // the staged CSR is complete: release the belief warps that gather over it (arrive only: the writers do not wait)
  if (p.bel_share_csr) asm volatile("bar.arrive 3, %0;\n" ::"r"(THREADS) : "memory");
  if constexpr (CSRT > 0) asm volatile("bar.arrive %0, %1;\n" ::"n"(LAG_CSR_BAR), "n"(CSRT) : "memory");  // ... and the dynamics warps
  // the tile's state is in shared memory: the dynamics warps of a lagged step may replace it
  if constexpr (LAGT > 0) asm volatile("bar.arrive %0, %1;\n" ::"n"(LAG_BAR), "n"(LAGT) : "memory");
  int* fpos = s_fpos + w * SY_MAX_AGENTS;
  const int R = p.wr_img_rows;       // mask rows per image: A (whole env) or 1 (large rows)
  const int lpa = R == 1 ? 32 : 32 / A;  // lanes that share one agent's neighbour list
  for (int e = w; e < nEnv; e += WRW) {
    const int b = tile0 + e;
    float* nf = p.ob.node_features + (size_t)b * N * A;
    // yard.py:279-290: one-hot positions; the MrX column stays blank while he is hidden
    if (lane < A) fpos[lane] = (lane > 0 || s_rev[e] >= 0) ? s_pos[e * A + lane] * A + lane : -1;
    for (int a0 = 0; a0 < A; a0 += R) {
      uint8_t* mask = p.ob.action_mask + ((size_t)b * A + a0) * N;
      const int phase = (int)(reinterpret_cast<uintptr_t>(mask) & 15u);
      uint8_t* img = s_img + phase;  // same 16-byte phase as the destination
      // ---- ones of these rows into the shared-memory image (action_mask.py:65-76: adjacent and weight + toll <= budget)
      const int ag = a0 + lane / lpa, sub = lane % lpa;
      if (ag < A && lane / lpa < R && !(p.dbg_skip & 2)) {
        const int u = s_pos[e * A + ag], m = s_money[e * A + ag], g = s_gid[e];
        uint8_t* row = img + (ag - a0) * N;
        if (GROUPS && u < 0) {
          // absent agent: an all-zero row
        } else if (staged) {
          const int r0 = s_rp[u], r1 = s_rp[u + 1];
          for (int k = r0 + sub; k < r1; k += lpa)
            if ((int)s_wgt[k] + wr_toll<GROUPS>(p) <= m) row[s_col[k]] = 1;
        } else {
          const int32_t* rp = tb.row_ptr + (size_t)g * (N + 1) + u;
          const int r0 = __ldg(rp), r1 = __ldg(rp + 1);
          const uint16_t* cl = tb.col + (size_t)g * tb.nnz_stride;
          const uint8_t* wg = tb.wgt + (size_t)g * tb.nnz_stride;
          for (int k = r0 + sub; k < r1; k += lpa)
            if ((int)__ldg(wg + k) + wr_toll<GROUPS>(p) <= m) row[__ldg(cl + k)] = 1;
        }
      }
      __syncwarp();
      warp_copy_bytes(mask, img, min(R, A - a0) * N, lane);
      if (a0 + R < A) {  // more rows of this env follow: clear the image for them
        __syncwarp();
        for (int i = lane * 16; i < p.wr_img_stride; i += 32 * 16) *reinterpret_cast<uint4*>(s_img + i) = make_uint4(0, 0, 0, 0);
        __syncwarp();
      }
    }
    __syncwarp();
    if (p.ob.node_features_u8 && R != A) {
      // large rows keep only one mask row in the image: the byte one-hot is zero-filled and its (at most A) ones stored as bytes
      uint8_t* nf8 = p.ob.node_features_u8 + (size_t)b * N * A;
      warp_zero_bytes(nf8, N * A, lane);
      __syncwarp();
      if (lane < A && fpos[lane] >= 0) nf8[fpos[lane]] = 1;
    } else if (p.ob.node_features_u8) {  // byte one-hot: same image-and-copy scheme as the mask (no byte-sized global stores)
      __syncwarp();
      for (int i = lane * 16; i < p.wr_img_stride; i += 32 * 16) *reinterpret_cast<uint4*>(s_img + i) = make_uint4(0, 0, 0, 0);
      __syncwarp();
      uint8_t* nf8 = p.ob.node_features_u8 + (size_t)b * N * A;
      uint8_t* img8 = s_img + (int)(reinterpret_cast<uintptr_t>(nf8) & 15u);
      if (lane < A && fpos[lane] >= 0) img8[fpos[lane]] = 1;
      __syncwarp();
      warp_copy_bytes(nf8, img8, N * A, lane);
    } else {
      if constexpr (PREFILLED) warp_write_node_feature_ones(nf, N * A, fpos, A, lane);
      else warp_write_node_features(nf, N * A, fpos, A, lane);
    }
    __syncwarp();
    for (int i = lane * 16; i < p.wr_img_stride; i += 32 * 16) *reinterpret_cast<uint4*>(s_img + i) = make_uint4(0, 0, 0, 0);
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// bulk (TMA) writers.  The tile's action_mask [nEnv, A, N] bytes and node_features [nEnv, N, A] elements are two
// contiguous byte streams that start 16-byte aligned (a tile is 32 envs).  Each stream is cut into chunks (multiples of
// 16 bytes, whole envs or whole fractions of an env where the sizes allow: plan_bulk_chunk on the host).  A writer warp
// owns two zeroed shared-memory images; per chunk it sets the few ones that fall into it (affordable
// neighbours, action_mask.py:65-76; one-hot positions, yard.py:279-290), hands the image to the TMA engine with ONE
// cp.async.bulk (SASS UBLKCP) and, once the engine has read it, clears the same ones again.  That is a few dozen
// shared-memory accesses per chunk instead of hundreds of STG.128: the store stream no longer passes through the LSU
// or the register file, which is what blocked every attempt to run the game logic next to the writers.
// ---------------------------------------------------------------------------------------------
struct BulkCtx {
  const int* s_pos;    // [TILE * A] staged state of the tile
  const int* s_money;  // [TILE * A]
  const int* s_rev;    // [TILE]
  const int* s_gid;    // [TILE]
  const int* rp;       // staged CSR of the tile's graph (STAGED) ...
  const uint16_t* col;
  const uint8_t* wgt;
};

// ones of the action_mask stream that fall into bytes [lo, lo + len): lane = (env, agent) pair (GROUPS: the staged
// budgets are headroom, see wr_budget)
template <bool STAGED, int GROUPS = 0>
__device__ __forceinline__ void bulk_mask_ones(const Params& p, const BulkCtx& c, uint8_t* img, int lo, int len, int lane, uint8_t v) {
  const int N = p.N, A = p.A, S = A * N;
  const int e_lo = lo / S, e_hi = (lo + len - 1) / S;
  const int npairs = (e_hi - e_lo + 1) * A;
  for (int q = lane; q < npairs; q += 32) {
    const int de = (q * p.inv_A) >> 16, a = q - de * A, e = e_lo + de;
    const int u = c.s_pos[e * A + a], m = c.s_money[e * A + a];
    const int base = e * S + a * N - lo;
    if (GROUPS && u < 0) continue;  // absent agent: an all-zero row
    if (STAGED) {
      const int r0 = c.rp[u], r1 = c.rp[u + 1];
      for (int k = r0; k < r1; ++k) {
        const int off = base + (int)c.col[k];
        if ((int)c.wgt[k] + wr_toll<GROUPS>(p) <= m && (unsigned)off < (unsigned)len) img[off] = v;
      }
    } else {
      const int g = c.s_gid[e];
      const int32_t* rp = p.tb.row_ptr + (size_t)g * (N + 1) + u;
      const int r0 = __ldg(rp), r1 = __ldg(rp + 1);
      const uint16_t* cl = p.tb.col + (size_t)g * p.tb.nnz_stride;
      const uint8_t* wg = p.tb.wgt + (size_t)g * p.tb.nnz_stride;
      for (int k = r0; k < r1; ++k) {
        const int off = base + (int)__ldg(cl + k);
        if ((int)__ldg(wg + k) + wr_toll<GROUPS>(p) <= m && (unsigned)off < (unsigned)len) img[off] = v;
      }
    }
  }
}

// ones of the node_features stream (ELEM = 4: float32 1.0f, 1: uint8 1) in bytes [lo, lo + len); the MrX column stays
// blank while he is hidden (yard.py:279-290 with the reveal schedule), and (GROUPS) an absent agent's column too
template <int ELEM, int GROUPS = 0>
__device__ __forceinline__ void bulk_nf_ones(const Params& p, const BulkCtx& c, uint8_t* img, int lo, int len, int lane, bool set) {
  const int N = p.N, A = p.A, S = N * A * ELEM;
  const int e_lo = lo / S, e_hi = (lo + len - 1) / S;
  const int npairs = (e_hi - e_lo + 1) * A;
  for (int q = lane; q < npairs; q += 32) {
    const int de = (q * p.inv_A) >> 16, a = q - de * A, e = e_lo + de;
    if (a == 0 && c.s_rev[e] < 0) continue;
    if (GROUPS && c.s_pos[e * A + a] < 0) continue;
    const int off = e * S + (c.s_pos[e * A + a] * A + a) * ELEM - lo;
    if ((unsigned)off < (unsigned)len) {
      if (ELEM == 4) *reinterpret_cast<unsigned*>(img + off) = set ? 0x3f800000u : 0u;
      else img[off] = set ? 1 : 0;
    }
  }
}

// ---- writer streams -----------------------------------------------------------------------------------------------
// float32 node_features: the region is filled with zeros by bulk copies from a read-only zero page (nothing to assemble,
// nothing to wait for before the page can be reused); once a piece's fill has COMPLETED, the few 16-byte granules that
// hold a one are stored whole from registers and merge with the zero lines still resident in L2.
// action_mask (and uint8 node_features): chunk images, two per warp, so the engine reads one while the next is built.
// A writer warp interleaves the two: per mask chunk it first issues the fill of the matching piece of the float32
// stream (4x the bytes), then the chunk's image, and D chunks later -- when that piece's fill has completed -- the
// piece's ones.  The interleaving keeps the SM's (in-order) bulk-copy queue short, so an image never waits behind more
// than a few KB of fill.  Micro-benchmark of exactly this schedule (tools/exp/tma_fill.cu, B200): the 458 MB of config 3
// leave the chip in 72 us with 2 warps on each of 2 CTAs per SM (cudaMemset: 66 us); issuing a whole tile's fill up
// front instead made every image wait behind ~180 KB of queued copies and doubled the kernel time.
struct ImageStreams {
  int ncf, ncm;  // chunks of the uint8 node_features stream (0 when float32), of the action_mask stream
  int Tf, Tm;    // stream lengths (bytes) of this tile
  uint8_t* gf;
  uint8_t* gm;
};

__device__ __forceinline__ ImageStreams image_streams(const Params& p, int tile0, int nEnv) {
  ImageStreams st;
  const int S = p.A * p.N;
  const bool nf8 = p.ob.node_features_u8 != nullptr;
  st.Tm = nEnv * S;
  st.Tf = nf8 ? nEnv * S : 0;
  st.ncm = (st.Tm + p.wr_c_mask - 1) / p.wr_c_mask;
  st.ncf = nf8 ? (st.Tf + p.wr_c_nf - 1) / p.wr_c_nf : 0;
  st.gm = p.ob.action_mask + (size_t)tile0 * S;
  st.gf = nf8 ? p.ob.node_features_u8 + (size_t)tile0 * S : nullptr;
  return st;
}

// zero fill of bytes [lo, hi) of the tile's float32 node_features stream (lo 16-byte aligned), issued by ONE lane
__device__ __forceinline__ void nf32_fill_piece(uint8_t* gnf, int lo, int hi, const uint8_t* zero_page, int Z) {
  const int body_hi = lo + ((hi - lo) & ~15);
  for (int o = lo; o < body_hi; o += Z) bulk_store(gnf + o, zero_page, (unsigned)min(Z, body_hi - o));
}

// ones of the float32 node_features stream that fall into bytes [lo, hi) (yard.py:279-290; the MrX column stays blank
// while he is hidden): lane = (env, agent) pair.  Env rows that are whole 16-byte granules get the granule rewritten
// (assembled from every agent of the env that falls into it), others a 4-byte store.  GROUPS: absent agents (pos -1)
// have no one (their negative flat index never shares a granule with a present agent's).
template <int GROUPS = 0>
__device__ __forceinline__ void nf32_ones_piece(const Params& p, const BulkCtx& c, uint8_t* gnf, int lo, int hi, int lane) {
  const int A = p.A, S = p.N * A * 4;
  const int e_lo = lo / S, e_hi = (hi - 1) / S;
  const int npairs = (e_hi - e_lo + 1) * A;
  const bool granules = (S & 15) == 0;
  for (int q = lane; q < npairs; q += 32) {
    const int de = (q * p.inv_A) >> 16, a = q - de * A, e = e_lo + de;
    const bool hidden = c.s_rev[e] < 0;
    if (a == 0 && hidden) continue;
    const int* pos = c.s_pos + e * A;
    if (GROUPS && pos[a] < 0) continue;
    const int f = pos[a] * A + a;  // element index inside the env's row
    const int off = e * S + f * 4;
    if (off < lo || off >= hi) continue;
    if (granules) {
      const int g = f >> 2;
      uint4 v = make_uint4(0, 0, 0, 0);
      for (int b2 = hidden ? 1 : 0; b2 < A; ++b2) {
        const int f2 = pos[b2] * A + b2;
        if ((f2 >> 2) == g) {
          const unsigned one = 0x3f800000u;
          const int sub = f2 & 3;
          v.x = sub == 0 ? one : v.x;
          v.y = sub == 1 ? one : v.y;
          v.z = sub == 2 ? one : v.z;
          v.w = sub == 3 ? one : v.w;
        }
      }
      store_obs16(reinterpret_cast<uint4*>(gnf + (size_t)e * S) + g, v);
    } else {
      *reinterpret_cast<float*>(gnf + off) = 1.0f;
    }
  }
}

// writer warp `iw` of `niw`: items iw, iw + niw, ... of [uint8 node_features chunks | action_mask chunks]; with float32
// node_features every mask chunk also carries the matching piece of that stream.  D = chunks between a piece's fill and
// its ones.  prefilled: the caller already issued (from this warp's lane 0) the fill of all of this warp's pieces.
template <int D, int GROUPS = 0>
__device__ __forceinline__ void writer_stream_warp(const Params& p, const BulkCtx& c, const ImageStreams& st, bool staged, uint8_t* my_img,
                                                   const uint8_t* zero_page, uint8_t* gnf32, int iw, int niw, int lane, bool prefilled) {
  const int Cm = p.wr_c_mask, Cf = p.wr_c_nf;
  const int Tf32 = 4 * st.Tm;  // float32 node_features stream: 4 bytes per mask byte
  auto ones = [&](int item, uint8_t* img, uint8_t v) {
    if (item < st.ncf) {
      const int lo = item * Cf;
      bulk_nf_ones<1, GROUPS>(p, c, img, lo, min(Cf, st.Tf - lo), lane, v != 0);
    } else {
      const int lo = (item - st.ncf) * Cm, len = min(Cm, st.Tm - lo);
      if (staged) bulk_mask_ones<true, GROUPS>(p, c, img, lo, len, lane, v);
      else bulk_mask_ones<false, GROUPS>(p, c, img, lo, len, lane, v);
    }
  };
  auto piece_ones = [&](int item) {
    if (gnf32 && item >= st.ncf) {
      const int lo = 4 * (item - st.ncf) * Cm;
      nf32_ones_piece<GROUPS>(p, c, gnf32, lo, min(Tf32, lo + 4 * Cm), lane);
    }
  };
  const int total = st.ncf + st.ncm;
  int it = 0;
  for (int item = iw; item < total; item += niw, ++it) {
    const bool is_nf8 = item < st.ncf;
    // ---- group F(it): zero fill of the float32 piece that belongs to this mask chunk
    if (gnf32 && !is_nf8) {
      const int lo = 4 * (item - st.ncf) * Cm, hi = min(Tf32, lo + 4 * Cm);
      if (lane == 0 && !prefilled) nf32_fill_piece(gnf32, lo, hi, zero_page, Cm);
      const int tail = (hi - lo) & 15;  // ragged end of the batch's last tile only
      if (!prefilled && lane < tail) gnf32[hi - tail + lane] = 0;
    }
    if (lane == 0) bulk_commit();
    // ---- group M(it): the chunk's image
    uint8_t* img = my_img + (size_t)(it & 1) * p.wr_img_bytes;
    if (it >= 2) {  // the image's previous chunk has left shared memory (younger groups: F(it-1), M(it-1), F(it)): take its ones out
      if (lane == 0) bulk_wait_read<3>();
      __syncwarp();
      ones(item - 2 * niw, img, 0);
      __syncwarp();
    }
    ones(item, img, 1);
    fence_proxy_async_smem();  // generic-proxy writes of every lane -> visible to the async proxy
    __syncwarp();
    const int lo = is_nf8 ? item * Cf : (item - st.ncf) * Cm;
    const int len = is_nf8 ? min(Cf, st.Tf - lo) : min(Cm, st.Tm - lo);
    uint8_t* dst = (is_nf8 ? st.gf : st.gm) + lo;
    const int body = len & ~15;
    if (lane == 0) {
      if (body) bulk_store(dst, img, (unsigned)body);
      bulk_commit();
    }
    if (lane < len - body) dst[body + lane] = img[body + lane];  // ragged end of the batch's last tile only
    // ---- ones of the piece filled D chunks ago: F(it-D) and everything older has completed
    if (gnf32 && it >= D) {
      if (lane == 0) asm volatile("cp.async.bulk.wait_group %0;\n" ::"n"(2 * D + 1) : "memory");
      __syncwarp();
      piece_ones(item - D * niw);
    }
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
  __syncwarp();
  for (int k = max(0, it - D); k < it; ++k) piece_ones(iw + k * niw);
  // leave both images zeroed (the next tile of a persistent CTA starts from clean images)
  for (int k = max(0, it - 2); k < it; ++k) ones(iw + k * niw, my_img + (size_t)(k & 1) * p.wr_img_bytes, 0);
  __syncwarp();
}

#ifndef SY_BULK_WARPS
#define SY_BULK_WARPS 4
#endif
#ifndef SY_BULK_DEPTH
#define SY_BULK_DEPTH 2
#endif
constexpr int BULK_WARPS = SY_BULK_WARPS;  // writer warps that stream on the bulk path (more only deepen the copy queue)
constexpr int BULK_DEPTH = SY_BULK_DEPTH;  // chunks between a float32 piece's fill and its ones

// stage the tile's post-step state (and, when the tile sits on one graph, its CSR) into shared memory: what every
// writer needs to place the ones (GROUPS: budgets as headroom, see wr_budget).  Returns whether the CSR was staged.
template <int NTHREADS, int GROUPS = 0>
__device__ __forceinline__ bool stage_tile_inputs(const Params& p, unsigned char* dyn, int tile0, int nEnv, int tw, int lane,
                                                  int* s_pos, int* s_money, int* s_rev, int* s_gid) {
  const Tables& tb = p.tb;
  const int N = p.N, A = p.A;
  int* s_rp = reinterpret_cast<int*>(dyn + p.wr_off_csr);  // [N + 1]
  uint16_t* s_col = reinterpret_cast<uint16_t*>(s_rp + N + 1);
  uint8_t* s_wgt = reinterpret_cast<uint8_t*>(s_col + tb.nnz_stride);
  const int gl = (lane < nEnv) ? p.st.graph_id[tile0 + lane] : -1;
  const int g0 = __shfl_sync(FULL, gl, 0);
  const bool staged = p.wr_stage_csr && __all_sync(FULL, gl == g0 || gl < 0);
  for (int i = tw; i < nEnv * A; i += NTHREADS) {
    s_pos[i] = p.st.pos[(size_t)tile0 * A + i];
    s_money[i] = wr_budget<GROUPS>(p, p.st.money[(size_t)tile0 * A + i], tile0 + ((i * p.inv_A) >> 16));
  }
  if (tw < nEnv) {
    s_rev[tw] = p.ob.mrx_revealed[tile0 + tw];
    s_gid[tw] = gl;
  }
  if (staged) {
    const int32_t* grp = tb.row_ptr + (size_t)g0 * (N + 1);
    const int nnz = __ldg(grp + N);
    for (int i = tw; i <= N; i += NTHREADS) s_rp[i] = __ldg(grp + i);
    for (int k = tw; k < nnz; k += NTHREADS) {
      s_col[k] = __ldg(tb.col + (size_t)g0 * tb.nnz_stride + k);
      s_wgt[k] = __ldg(tb.wgt + (size_t)g0 * tb.nnz_stride + k);
    }
    if (p.bel_share_csr) {
      float* s_inv = reinterpret_cast<float*>(dyn + p.wr_off_csr + (((N + 1) * 4 + tb.nnz_stride * 3 + 3) & ~3));
      uint16_t* s_perm = reinterpret_cast<uint16_t*>(s_inv + N);
      for (int i = tw; i < N; i += NTHREADS) {
        s_inv[i] = __ldg(tb.inv_deg + (size_t)g0 * N + i);
        s_perm[i] = __ldg(tb.deg_perm + (size_t)g0 * N + i);
      }
      // padded neighbour lists of the belief gather (see writer_role)
      uint16_t* s_pptr = reinterpret_cast<uint16_t*>(dyn + p.wr_off_csr + p.wr_off_pad);
      uint16_t* s_pcol = s_pptr + ((N + 1 + 3) & ~3);
      const int32_t* gpp = tb.pack_ptr + (size_t)g0 * (N + 1);
      const int2* gpk = tb.nbr_pack + (size_t)g0 * tb.pack_stride;
      const int npk = __ldg(gpp + N);
      for (int i = tw; i <= N; i += NTHREADS) s_pptr[i] = (uint16_t)__ldg(gpp + i);
      for (int k = tw; k < npk; k += NTHREADS) {
        const int2 en = __ldg(gpk + k);
        s_pcol[k] = en.y ? (uint16_t)((unsigned)en.x / (BSTRIDE * 4u)) : (uint16_t)N;
      }
    }
  }
  return staged;
}

template <int WRW, int GROUPS = 0>
__device__ __forceinline__ void writer_role_bulk(const Params& p, unsigned char* dyn, int tile0, int nEnv, int w, int lane) {
  constexpr int NW = WRW < BULK_WARPS ? WRW : BULK_WARPS;
  const int N = p.N, A = p.A;
  int* s_pos = reinterpret_cast<int*>(dyn + p.wr_off);  // [TILE * A]
  int* s_money = s_pos + TILE * A;                      // [TILE * A]
  int* s_rev = s_money + TILE * A;                      // [TILE]
  int* s_gid = s_rev + TILE;                            // [TILE]
  uint8_t* zero_page = reinterpret_cast<uint8_t*>(s_gid + TILE);  // [wr_img_bytes] read-only zeros, 16-byte aligned
  uint8_t* imgs = zero_page + p.wr_img_bytes;                     // [BULK_WARPS][2][wr_img_bytes]
  for (int i = (w * 32 + lane) * 16; i < (1 + 2 * NW) * p.wr_img_bytes; i += WRW * 32 * 16) *reinterpret_cast<uint4*>(zero_page + i) = make_uint4(0, 0, 0, 0);
  fence_proxy_async_smem();
  const bool staged = stage_tile_inputs<WRW * 32, GROUPS>(p, dyn, tile0, nEnv, w * 32 + lane, lane, s_pos, s_money, s_rev, s_gid);
  named_barrier(2, WRW * 32);
  if (p.bel_share_csr) asm volatile("bar.arrive 3, %0;\n" ::"r"(THREADS) : "memory");
  if (w >= NW) return;
  int* s_rp = reinterpret_cast<int*>(dyn + p.wr_off_csr);
  uint16_t* s_col = reinterpret_cast<uint16_t*>(s_rp + N + 1);
  const BulkCtx c{s_pos, s_money, s_rev, s_gid, s_rp, s_col, reinterpret_cast<uint8_t*>(s_col + p.tb.nnz_stride)};
  const ImageStreams st = image_streams(p, tile0, nEnv);
  uint8_t* gnf32 = p.ob.node_features_u8 ? nullptr : reinterpret_cast<uint8_t*>(p.ob.node_features) + (size_t)tile0 * N * A * 4;
  writer_stream_warp<BULK_DEPTH, GROUPS>(p, c, st, staged, imgs + (size_t)w * 2 * p.wr_img_bytes, zero_page, gnf32, w, NW, lane, false);
}

// generic belief path: one warp per env, lane = node; any N, any mix of graphs.  sb: N floats of this warp.
// The env's row is copied to shared memory (LDGSTS), every lane then gathers its nodes' padded neighbour lists
// {node, 1/deg} straight from the (L1-resident) pool tables.  The normaliser is the sum of the INPUT row: the
// propagation conserves mass exactly (sum_j sum_{i in nbr(j)} b_i/deg_i = sum_i b_i on an undirected graph, isolated
// nodes keep theirs), so it equals the reference's sum of the output up to fp32 rounding and needs no second buffer.
// Belief quality at reveal steps (src/eval/belief_quality.py:8-11 as fed by MetricsTracker.record_step,
// src/eval/metrics.py:127-147): cross-entropy of the PREDICTED belief (the propagated row, before the reveal collapses
// it) at MrX's true node.  Per-warp accumulator, flushed once per warp into the statistics lines as Q24 fixed point
// (integer sums: order-independent, so runs and shardings reproduce bit for bit).
struct CeAcc {
  int n = 0;
  long long sum_q = 0, sq_q = 0;
};
constexpr float CE_CLIP = 1e-8f;
constexpr float CE_Q = 16777216.0f;  // 2^24

__device__ __forceinline__ float ce_clip(float v) { return fminf(fmaxf(v, CE_CLIP), 1.0f); }

// lanes hold partial clipped sums `S` and (one lane) the clipped value at the true node `vx`.  GROUPS: the score of env
// b also goes straight into its mechanism group's line (reveals are a fraction of the steps: one atomic triple each)
template <int GROUPS = 0>
__device__ __forceinline__ void ce_record(CeAcc& acc, float S, float vx, const Params* p = nullptr, int b = 0, int lane = 0) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    S += __shfl_xor_sync(FULL, S, o);
    vx = fmaxf(vx, __shfl_xor_sync(FULL, vx, o));
  }
  const float ce = logf(S) - logf(vx);  // -log(vx / S); both logs are of normal floats (vx >= 1e-8)
  if constexpr (!GROUPS) {
    acc.n += 1;
    acc.sum_q += __float2ll_rn(ce * CE_Q);
    acc.sq_q += __float2ll_rn(ce * ce * CE_Q);
  } else {
    const long long q = __float2ll_rn(ce * CE_Q), sq = __float2ll_rn(ce * ce * CE_Q);
    acc.n += 1;
    acc.sum_q += q;
    acc.sq_q += sq;
    if (lane == 0) {
      unsigned long long* line = p->grp_stats + ((size_t)(blockIdx.x % p->grp_rep) * p->grp_n + __ldg(p->grp_id + b)) * SY_NUM_STATS;
      atomicAdd(line + SY_STAT_REVEALS, 1ull);
      atomicAdd(line + SY_STAT_SUM_BELIEF_CE_Q24, (unsigned long long)q);
      atomicAdd(line + SY_STAT_SUM_SQ_BELIEF_CE_Q24, (unsigned long long)sq);
    }
  }
}

__device__ __forceinline__ void ce_flush(const Params& p, const CeAcc& acc, int lane) {
  if (acc.n && lane == 0) {
    unsigned long long* line = p.stats_rep + (size_t)(blockIdx.x % STAT_REPLICAS) * SY_NUM_STATS;
    atomicAdd(line + SY_STAT_REVEALS, (unsigned long long)acc.n);
    atomicAdd(line + SY_STAT_SUM_BELIEF_CE_Q24, (unsigned long long)acc.sum_q);
    atomicAdd(line + SY_STAT_SUM_SQ_BELIEF_CE_Q24, (unsigned long long)acc.sq_q);
  }
}

struct SharedCsr {  // the writer warps' staged copy of the tile's graph (null rp: not available)
  const uint16_t* pptr;  // padded neighbour lists: starts [N + 1] (multiples of 4) ...
  const uint16_t* pcol;  // ... and node ids, pads = N (the zero slot of the row)
  const int* rp;
  const uint16_t* col;
  const float* inv;
  const uint16_t* perm;  // nodes by degree: the 32 lanes of a gather step walk lists of (nearly) equal length
};

template <int GROUPS>
__device__ __forceinline__ void belief_env_generic_t(const Params& p, float* sb, int b, int op, int g, int x, int lane, CeAcc& ce,
                                                     const SharedCsr sc) {
  const int N = p.N;
  const Tables& tb = p.tb;
  float* bel = p.st.belief + (size_t)b * N;
  const float unif = 1.0f / (float)N;
  const bool score = op == BEL_DELTA && p.belief_score && p.out.stats != nullptr;  // reveal: score the prediction, then collapse it
  if (op == BEL_UNIFORM) {
    _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = unif;
  } else if (op == BEL_DELTA && !score) {
    _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = (j == x) ? 1.0f : 0.0f;
  } else if (op == BEL_PROPAGATE || score) {
    float S = 0.0f, vx = 0.0f;
    const int32_t* gptr = tb.pack_ptr + (size_t)g * (N + 1);
    const int2* gpack = tb.nbr_pack + (size_t)g * tb.pack_stride;
    __syncwarp();
    for (int j = lane; j < N; j += 32) cp_async4(sb + j, bel + j);
    cp_async_wait_all();
    __syncwarp();
    float tot = 0.0f;
    for (int j = lane; j < N; j += 32) tot += sb[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(FULL, tot, o);
    if (tot == 0.0f) {  // belief_module.py:36-37
      if (score) {
        S = lane == 0 ? (float)N * ce_clip(unif) : 0.0f;
        vx = ce_clip(unif);
      } else {
        _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = unif;
      }
    } else if (sc.rp) {
      // gather over the staged CSR, every operand from shared memory.  The row is pre-scaled once, conflict-free, to
      // w[i] = b[i] / deg(i) / sum(b), so the random-access gather reads ONE value per neighbour (it was two: b[i] and
      // 1/deg(i)) and the result needs no further normalisation: a third fewer (bank-conflicted) shared-memory reads on
      // the path that bounds the large-N configurations.
      const float inv = 1.0f / tot;
      _Pragma("unroll 4") for (int j = lane; j < N; j += 32) sb[j] *= sc.inv[j] * inv;  // (isolated nodes: 1/deg = 0, handled below)
      if (lane == 0) sb[N] = 0.0f;  // what the pads of the neighbour lists read
      __syncwarp();
      _Pragma("unroll 1") for (int jj = lane; jj < N; jj += 32) {
        const int j = sc.perm[jj];  // degree order: the 32 lanes of a step walk lists of (nearly) equal length
        const int r0 = sc.pptr[j], r1 = sc.pptr[j + 1];
        float a = 0.0f;
        _Pragma("unroll 2") for (int k = r0; k < r1; k += 4) {  // 4 neighbour ids per 8-byte load, no per-neighbour control flow
          const uint2 c4 = *reinterpret_cast<const uint2*>(sc.pcol + k);
          a += (sb[c4.x & 0xffffu] + sb[c4.x >> 16]) + (sb[c4.y & 0xffffu] + sb[c4.y >> 16]);
        }
        if (r0 == r1) a = bel[j] * inv;  // isolated node keeps its mass (belief_module.py:93-97); bel[j] is still the input
        if (!score) {
          bel[j] = a;
        } else {
          const float c = ce_clip(a);
          S += c;
          if (j == x) vx = c;
        }
      }
    } else {
      const float inv = 1.0f / tot;
      constexpr int U = 2;  // nodes per lane in flight: their list bounds, then their first TWO blocks, are loaded together
      _Pragma("unroll 1") for (int j0 = lane; j0 < N; j0 += 32 * U) {
        int qa[U], qb[U];
        int4 e[U][4];
        float acc[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int j = j0 + 32 * u;
          qa[u] = qb[u] = 0;
          if (j < N) {
            qa[u] = __ldg(gptr + j);
            qb[u] = __ldg(gptr + j + 1);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {  // lists are padded to multiples of 4 entries ({0, 0.0f}); 2 entries per int4
            e[u][k] = make_int4(0, 0, 0, 0);
            if (qa[u] + 2 * k < qb[u]) e[u][k] = __ldg(reinterpret_cast<const int4*>(gpack + qa[u] + 2 * k));
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          // entries hold the byte offset of the neighbour's row in the fast path's transposed tile: node * BSTRIDE * 4
          float a = 0.0f;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            a = fmaf(sb[(unsigned)e[u][k].x / (BSTRIDE * 4u)], __int_as_float(e[u][k].y), a);
            a = fmaf(sb[(unsigned)e[u][k].z / (BSTRIDE * 4u)], __int_as_float(e[u][k].w), a);
          }
          acc[u] = a;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int j = j0 + 32 * u;
          _Pragma("unroll 1") for (int q = qa[u] + 8; q < qb[u]; q += 4) {  // nodes with more than 8 neighbours
            const int4 f0 = __ldg(reinterpret_cast<const int4*>(gpack + q)), f1 = __ldg(reinterpret_cast<const int4*>(gpack + q + 2));
            acc[u] = fmaf(sb[(unsigned)f0.x / (BSTRIDE * 4u)], __int_as_float(f0.y), acc[u]);
            acc[u] = fmaf(sb[(unsigned)f0.z / (BSTRIDE * 4u)], __int_as_float(f0.w), acc[u]);
            acc[u] = fmaf(sb[(unsigned)f1.x / (BSTRIDE * 4u)], __int_as_float(f1.y), acc[u]);
            acc[u] = fmaf(sb[(unsigned)f1.z / (BSTRIDE * 4u)], __int_as_float(f1.w), acc[u]);
          }
          if (j < N) {
            if (qa[u] == qb[u]) acc[u] = sb[j];  // isolated node keeps its mass (belief_module.py:93-97)
            const float v = acc[u] * inv;
            if (!score) {
              bel[j] = v;
            } else {
              const float c = ce_clip(v);
              S += c;
              if (j == x) vx = c;
            }
          }
        }
      }
    }
    if (score) {
      if constexpr (GROUPS) ce_record<1>(ce, S, vx, &p, b, lane);
      else ce_record(ce, S, vx);
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = (j == x) ? 1.0f : 0.0f;
    } else if (p.belief_hint && op == BEL_PROPAGATE && tot != 0.0f) {
      // observation hint (belief_module.py:102-106) on the row this warp just wrote.  Lane l re-reads the nodes
      // j = l (mod 32); the shared-CSR path wrote bel[perm[jj]] in degree order, so those values came from other lanes,
      // which may still be in the last trip of their gather loop when N % 32 != 0: wait for every lane's stores first
      // (here and not before the branch, so that the hint-free kernels keep their instruction stream)
      __syncwarp();
      const uint8_t* hint = p.belief_hint + (size_t)b * N;
      float hs = 0.0f;
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) hs += bel[j] * (hint[j] ? 1.0f : 0.1f);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) hs += __shfl_xor_sync(FULL, hs, o);
      const float inv = hs == 0.0f ? 0.0f : 1.0f / hs;
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = hs == 0.0f ? unif : bel[j] * (hint[j] ? 1.0f : 0.1f) * inv;
    }
  }
}

// one env's belief row, warp-wide (an out-of-line function, as the kernels were tuned with; GROUPS: its own copy)
__device__ void belief_env_generic(const Params& p, float* sb, int b, int op, int g, int x, int lane, CeAcc& ce, const SharedCsr sc) {
  belief_env_generic_t<0>(p, sb, b, op, g, x, lane, ce, sc);
}
__device__ void belief_env_generic_groups(const Params& p, float* sb, int b, int op, int g, int x, int lane, CeAcc& ce,
                                          const SharedCsr sc) {
  belief_env_generic_t<1>(p, sb, b, op, g, x, lane, ce, sc);
}

template <int BW, int LAGT = 0, int GROUPS = 0>
__device__ __forceinline__ void belief_role(const Params& p, unsigned char* dyn, int tile0, int nEnv, int w, int lane) {
  const int N = p.N;
  // every belief warp reads the same 32 flags / graph ids, so the branches below are uniform across the role
  int op = BEL_KEEP, g = -1, xm = -1;
  if (lane < nEnv) {
    op = __ldcg(p.bel_flags + tile0 + lane);
    g = __ldcg(p.st.graph_id + tile0 + lane);
    if (op == BEL_DELTA) xm = __ldcg(p.st.pos + (size_t)(tile0 + lane) * p.A);  // MrX's node (the reveal collapses the map onto it)
  }
  if constexpr (LAGT > 0) {
    // everything this role reads of the tile's state is in registers (the count operand makes the arrival wait for the
    // loads): the dynamics warps of the CTA may now replace the state
    int dep;
    asm volatile("and.b32 %0, %1, 0;\n" : "=r"(dep) : "r"(op | g | xm));
    asm volatile("bar.arrive %0, %1;\n" ::"n"(LAG_BAR), "r"(LAGT + dep) : "memory");
  }
  // rows that go through the propagation: moving envs, plus revealed ones while their prediction is being scored
  const bool score = p.belief_score && p.out.stats != nullptr;
  const unsigned prop = __ballot_sync(FULL, op == BEL_PROPAGATE || (score && op == BEL_DELTA));
  const unsigned any = __ballot_sync(FULL, op != BEL_KEEP);
  // the writers stage the tile's CSR (+ 1/deg) for the large-N path; every belief warp waits for it exactly once
  if (p.bel_share_csr) asm volatile("bar.sync 3, %0;\n" ::"r"(THREADS) : "memory");
  if (!any) return;
  CeAcc ce;
  const int g0 = __shfl_sync(FULL, g, prop ? __ffs(prop) - 1 : 0);
  const int gfirst = __shfl_sync(FULL, g, 0);
  const bool fast = p.bel_fast && prop && __all_sync(FULL, !((prop >> lane) & 1u) || g == g0);
  if (!fast) {
    float* sb = reinterpret_cast<float*>(dyn) + (size_t)w * (N + 1);  // + 1: the zero slot the padded lists point at
    SharedCsr sc{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    if (p.bel_share_csr && __all_sync(FULL, lane >= nEnv || g == gfirst)) {  // the writers' `staged` condition
      sc.rp = reinterpret_cast<const int*>(dyn + p.wr_off_csr);
      sc.col = reinterpret_cast<const uint16_t*>(sc.rp + N + 1);
      sc.inv = reinterpret_cast<const float*>(dyn + p.wr_off_csr + (((N + 1) * 4 + p.tb.nnz_stride * 3 + 3) & ~3));
      sc.perm = reinterpret_cast<const uint16_t*>(sc.inv + N);
      sc.pptr = reinterpret_cast<const uint16_t*>(dyn + p.wr_off_csr + p.wr_off_pad);
      sc.pcol = sc.pptr + ((N + 1 + 3) & ~3);
    }
    for (int e = w; e < nEnv; e += BW) {
      if constexpr (GROUPS)
        belief_env_generic_groups(p, sb, tile0 + e, __shfl_sync(FULL, op, e), __shfl_sync(FULL, g, e), __shfl_sync(FULL, xm, e), lane, ce, sc);
      else
        belief_env_generic(p, sb, tile0 + e, __shfl_sync(FULL, op, e), __shfl_sync(FULL, g, e), __shfl_sync(FULL, xm, e), lane, ce, sc);
    }
    ce_flush(p, ce, lane);
    return;
  }
  // fast path: tin[j * BSTRIDE + e] (transposed) so that lane = env: the CSR walk is warp-uniform (no divergence,
  // neighbour entries are one broadcast LDS), every smem access is conflict-free, the normaliser is lane-local.
  float* __restrict__ tin = reinterpret_cast<float*>(dyn);
  float* __restrict__ tout = reinterpret_cast<float*>(dyn + p.bel_off_out);
  float* __restrict__ part = reinterpret_cast<float*>(dyn + p.bel_off_part);
  int2* __restrict__ spack = reinterpret_cast<int2*>(dyn + p.bel_off_pack);
  int* __restrict__ sptr = reinterpret_cast<int*>(dyn + p.bel_off_ptr);
  const int32_t* gptr = p.tb.pack_ptr + (size_t)g0 * (N + 1);
  const int2* gpack = p.tb.nbr_pack + (size_t)g0 * p.tb.pack_stride;
  const int jpw = (N + BW - 1) / BW;  // warp w owns nodes [j0, j1) = list entries [q0, q1)
  const int j0 = min(N, w * jpw), j1 = min(N, j0 + jpw);
  const int q0 = __ldg(gptr + j0), q1 = __ldg(gptr + j1);
  for (int e = w; e < TILE; e += BW) {
    if ((prop >> e) & 1u) {
      const float* bel = p.st.belief + (size_t)(tile0 + e) * N;
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) cp_async4(tin + j * BSTRIDE + e, bel + j);
    } else {
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) tin[j * BSTRIDE + e] = 0.0f;
    }
  }
  for (int k = q0 + 2 * lane; k < q1; k += 64) cp_async16(spack + k, gpack + k);  // this warp's lists (2 entries / copy)
  // list bounds of this warp's nodes; isolated nodes keep their mass (belief_module.py:93-97)
  unsigned iso[(BEL_JMAX + 31) / 32];
#pragma unroll
  for (int r = 0; r < (BEL_JMAX + 31) / 32; ++r) {
    const int j = j0 + r * 32 + lane;
    int qa = 0, qb = 1;
    if (j < j1) {
      qa = __ldg(gptr + j);
      qb = __ldg(gptr + j + 1);
      sptr[j + 1] = qb;
    }
    iso[r] = __ballot_sync(FULL, qa == qb);
  }
  cp_async_wait_all();
  named_barrier(1, BW * 32);
  float sum = 0.0f;
  const unsigned char* tin_lane = reinterpret_cast<const unsigned char*>(tin + lane);
  float* tout_row = tout + j0 * BSTRIDE + lane;
  const int4* pp = reinterpret_cast<const int4*>(spack + q0);
  int qa = q0;
#pragma unroll 1
  for (int j = j0; j < j1; ++j, tout_row += BSTRIDE) {
    const int qb = sptr[j + 1];
    float a = 0.0f;
#pragma unroll 1
    for (; qa < qb; qa += 4, pp += 2) {  // 4 neighbours per trip (lists are padded); warp-uniform
      const int4 e0 = pp[0], e1 = pp[1];
      const float v0 = *reinterpret_cast<const float*>(tin_lane + e0.x), v1 = *reinterpret_cast<const float*>(tin_lane + e0.z);
      const float v2 = *reinterpret_cast<const float*>(tin_lane + e1.x), v3 = *reinterpret_cast<const float*>(tin_lane + e1.z);
      a = fmaf(v0, __int_as_float(e0.y), a);
      a = fmaf(v1, __int_as_float(e0.w), a);
      a = fmaf(v2, __int_as_float(e1.y), a);
      a = fmaf(v3, __int_as_float(e1.w), a);
    }
    *tout_row = a;
    sum += a;
  }
#pragma unroll
  for (int r = 0; r < (BEL_JMAX + 31) / 32; ++r) {
    unsigned m = iso[r];
    while (m) {
      const int j = j0 + r * 32 + __ffs(m) - 1;
      m &= m - 1;
      const float v = tin[j * BSTRIDE + lane];
      tout[j * BSTRIDE + lane] = v;
      sum += v;
    }
  }
  part[w * 32 + lane] = sum;
  named_barrier(1, BW * 32);
  // normalise + per-env operation, coalesced copy-out: warp per env, lane = node
  const float unif = 1.0f / (float)N;
  for (int e = w; e < nEnv; e += BW) {
    const int ope = __shfl_sync(FULL, op, e);
    if (ope == BEL_KEEP) continue;
    float* bel = p.st.belief + (size_t)(tile0 + e) * N;
    if (ope == BEL_PROPAGATE) {
      float tot = 0.0f;
#pragma unroll
      for (int ww = 0; ww < BW; ++ww) tot += part[ww * 32 + e];
      if (p.belief_hint && tot != 0.0f) {
        // observation hint (belief_module.py:102-106): likelihood 0.1 + 0.9 * [j is a candidate], then normalise.  An
        // all-zero hint row scales every node alike and normalises away, like the reference's `if observation_hint:`
        const uint8_t* hint = p.belief_hint + (size_t)(tile0 + e) * N;
        float hs = 0.0f;
        _Pragma("unroll 1") for (int j = lane; j < N; j += 32) hs += tout[j * BSTRIDE + e] * (hint[j] ? 1.0f : 0.1f);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) hs += __shfl_xor_sync(FULL, hs, o);
        if (hs == 0.0f) {
          _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = unif;
        } else {
          const float inv = 1.0f / hs;
          _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = tout[j * BSTRIDE + e] * (hint[j] ? 1.0f : 0.1f) * inv;
        }
      } else if (tot == 0.0f) {  // belief_module.py:29-38
        _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = unif;
      } else {
        const float inv = 1.0f / tot;
        _Pragma("unroll 4") for (int j = lane; j < N; j += 32) bel[j] = tout[j * BSTRIDE + e] * inv;
      }
    } else if (ope == BEL_UNIFORM) {
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = unif;
    } else {
      const int x = __shfl_sync(FULL, xm, e);
      if (score) {
        float tot = 0.0f, vx = 0.0f, S = 0.0f;
#pragma unroll
        for (int ww = 0; ww < BW; ++ww) tot += part[ww * 32 + e];
        if (tot == 0.0f) {
          S = lane == 0 ? (float)N * ce_clip(unif) : 0.0f;
          vx = ce_clip(unif);
        } else {
          const float inv = 1.0f / tot;
          _Pragma("unroll 1") for (int j = lane; j < N; j += 32) {
            const float c = ce_clip(tout[j * BSTRIDE + e] * inv);
            S += c;
            if (j == x) vx = c;
          }
        }
        if constexpr (GROUPS) ce_record<1>(ce, S, vx, &p, tile0 + e, lane);
        else ce_record(ce, S, vx);
      }
      _Pragma("unroll 1") for (int j = lane; j < N; j += 32) bel[j] = (j == x) ? 1.0f : 0.0f;
    }
  }
  ce_flush(p, ce, lane);
}

// BW belief warps + WRW writer warps.  <8, 8> everywhere the belief hides under the write stream (fast path); the
// large-N generic belief path is the critical role, there the split is <12, 4> (c4: 82 -> 91 M env-steps/s).
// WV selects the writers at compile time, so the default kernel carries none of the experimental paths' code or
// registers: WV_LSU = 16-byte streaming stores (default), WV_BULK = zero-page fill + chunk images through the TMA engine,
// WV_ONES = node_features were zero-filled by sy_fill_kernel, only the ones are stored (split step).
// <BW, 0> / <0, WRW>: one role per launch (the split step runs them as two concurrent kernels; the role hand-over
// barrier of the large-N belief path counts THREADS, so that path keeps both roles in one launch)
enum { WV_LSU = 0, WV_BULK = 1, WV_ONES = 2 };
// GROUPS (launched while mechanism groups are set): the writers test each env's moves against its group's toll, and the
// belief scores at reveal steps are also summed per group
template <int BW, int WRW, int WV = WV_LSU, int GROUPS = 0>
__global__ void __launch_bounds__((BW + WRW) * 32) sy_observe_kernel(const Params p) {
  static_assert((BW + WRW) * 32 == THREADS || BW == 0 || WRW == 0, "the role hand-over barrier counts THREADS");
  extern __shared__ __align__(16) unsigned char dyn[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int tile0 = blockIdx.x * TILE;
  int nEnv = min(TILE, p.B - tile0);
  if (p.ob_split > 1 && (int)blockIdx.x >= p.ob_full) {
    // tail of the grid: all CTAs last about equally long, so a last wave that fills only part of the chip costs a whole
    // CTA lifetime; its tiles are cut into parts so that the wave is full and short (c4: 3.46 waves -> 3 + 0.5)
    const int r = (int)blockIdx.x - p.ob_full, sub = TILE / p.ob_split;
    const int t = p.ob_full + r / p.ob_split, part = r % p.ob_split;
    tile0 = t * TILE + part * sub;
    nEnv = min(sub, p.B - tile0);
    if (nEnv <= 0) return;
  }
  const int nbw = BW;  // without a belief map the belief warps simply exit
  pdl_launch_dependents();
  pdl_wait();  // the dynamics kernel's state (CTAs of this grid may have been scheduled before it finished)
  if (warp < nbw && !p.belief_on) return;
  const long long t0 = FCLK_NOW();
  if (warp < nbw) {
    if constexpr (BW > 0) {
      if (!(p.dbg_skip & 4)) belief_role<BW, 0, GROUPS>(p, dyn, tile0, nEnv, warp, lane);
      if (warp == 0) FCLK_ADD(3, FCLK_NOW() - t0);
    }
  } else if (!(p.dbg_skip & 1)) {
    if constexpr (WRW > 0) {
      if constexpr (WV == WV_BULK) {
        if constexpr (WRW >= 2) writer_role_bulk<WRW, GROUPS>(p, dyn, tile0, nEnv, warp - nbw, lane);
      } else {
        writer_role<WRW, WV == WV_ONES, 0, 0, GROUPS>(p, dyn, tile0, nEnv, warp - nbw, lane);
      }
      if (warp == nbw) {
        FCLK_ADD(1, FCLK_NOW() - t0);
        FCLK_ADD(6, 1);
      }
    }
  }
}

constexpr int GEN_BEL_WARPS = THREADS / 32 >= 16 ? 12 : BEL_WARPS, GEN_WR_WARPS = THREADS / 32 - GEN_BEL_WARPS;  // split of the large-N configuration

// ---------------------------------------------------------------------------------------------
// lagged step kernel (software-pipelined rollouts): ONE launch = the dense observations of the CURRENT state (the
// roles of sy_observe_kernel, unchanged) and, on LOGIC_WARPS extra warps of the same CTA, the dynamics of the NEXT step
// for the same 32-env tile.  The two halves belong to different steps, so neither waits for the other: the
// latency-bound dynamics (a chain of dependent table lookups, ~13 us per tile) run in the shadow of the tile's
// HBM-bound observation stream (~15 us per tile) instead of in a kernel of their own in front of it.  The only
// ordering is write-after-read on the tile's state: the observation roles copy what they need first (registers /
// shared memory) and arrive on LAG_BAR; the dynamics warps wait on it right before their state write-back.
// A policy that needs only the compact state (positions, budgets, reveal flags: the random policy, both reference
// agents) sees the new state after every launch; action_mask / node_features / belief_map trail it by one step until
// sy_flush_observations (or any non-deferred call) brings them up to date.
// ---------------------------------------------------------------------------------------------
template <int MODE, int MAXA, int BW, int WRW, int GROUPS = 0>
__global__ void __launch_bounds__((BW + WRW + LOGIC_WARPS) * 32, 2) sy_step_lagged_kernel(const Params p) {
  constexpr int NT = (BW + WRW + LOGIC_WARPS) * 32;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ LogicSmem<MAXA> lsm;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile0 = blockIdx.x * TILE;
  const int nEnv = min(TILE, p.B - tile0);
  constexpr int CSRT = (WRW + LOGIC_WARPS) * 32;
  __shared__ int staged_flag;
  const long long t0 = FCLK_NOW();
  if (warp < BW) {
    if constexpr (BW > 0) belief_role<BW, NT, GROUPS>(p, dyn, tile0, nEnv, warp, lane);
    if (warp == 0) FCLK_ADD(3, FCLK_NOW() - t0);
  } else if (warp < BW + WRW) {
    writer_role<WRW, false, NT, CSRT, GROUPS>(p, dyn, tile0, nEnv, warp - BW, lane, &staged_flag);
    if (warp == BW) FCLK_ADD(1, FCLK_NOW() - t0);
  } else {
    const int* s_rp = reinterpret_cast<const int*>(dyn + p.wr_off_csr);
    const uint16_t* s_col = reinterpret_cast<const uint16_t*>(s_rp + p.N + 1);
    const SharedGraph sg{s_rp, s_col, reinterpret_cast<const uint8_t*>(s_col + p.tb.nnz_stride)};
    logic_tile<MODE, MAXA, 5, NT, CSRT, GROUPS>(p, lsm, tile0, threadIdx.x - (BW + WRW) * 32, &sg, &staged_flag);
    if (warp == BW + WRW) {
      FCLK_ADD(4, FCLK_NOW() - t0);
      FCLK_ADD(5, 1);
    }
  }
}

// K random-policy steps in ONE launch (sy_rollout_random* on batches of at most one wave): the lagged kernel's CTA in a
// loop.  Envs are independent and a CTA owns its 32-env tile for the whole rollout, so nothing is exchanged between CTAs
// and no grid-wide synchronisation exists: iteration `it` writes the observations of the state after `it` steps while
// the dynamics warps run step it + 1 (and draw the actions of step it + 2 from the new state); a CTA-wide barrier closes
// the iteration (the new state is visible to the CTA's own roles, shared memory may be reused).  K + 1 iterations: the
// first without observations (they are current on entry), the last without dynamics.
constexpr int ROLL_BAR = 7;
template <int MODE, int MAXA, int BW, int WRW, int GROUPS = 0>
__global__ void __launch_bounds__((BW + WRW + LOGIC_WARPS) * 32, 2) sy_rollout_lagged_kernel(const Params p, const int K) {
  constexpr int NT = (BW + WRW + LOGIC_WARPS) * 32;
  constexpr int CSRT = (WRW + LOGIC_WARPS) * 32;
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ LogicSmem<MAXA> lsm;
  __shared__ int staged_flag;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile0 = blockIdx.x * TILE;
  const int nEnv = min(TILE, p.B - tile0);
  for (int it = 0; it <= K; ++it) {
    const bool do_obs = it > 0, do_logic = it < K;
    if (warp < BW) {
      if constexpr (BW > 0) {
        if (do_obs) belief_role<BW, NT, GROUPS>(p, dyn, tile0, nEnv, warp, lane);
        else asm volatile("bar.arrive %0, %1;\n" ::"n"(LAG_BAR), "n"(NT) : "memory");
      }
    } else if (warp < BW + WRW) {
      if (do_obs) {
        writer_role<WRW, false, NT, CSRT, GROUPS>(p, dyn, tile0, nEnv, warp - BW, lane, &staged_flag);
      } else {
        if (threadIdx.x == BW * 32) staged_flag = 0;  // nothing staged: the dynamics read the pool tables
        asm volatile("bar.arrive %0, %1;\n" ::"n"(LAG_CSR_BAR), "n"(CSRT) : "memory");
        asm volatile("bar.arrive %0, %1;\n" ::"n"(LAG_BAR), "n"(NT) : "memory");
      }
    } else {
      if (do_logic) {
        const int* s_rp = reinterpret_cast<const int*>(dyn + p.wr_off_csr);
        const uint16_t* s_col = reinterpret_cast<const uint16_t*>(s_rp + p.N + 1);
        const SharedGraph sg{s_rp, s_col, reinterpret_cast<const uint8_t*>(s_col + p.tb.nnz_stride)};
        // (the last step draws nothing: `actions` keeps the actions of the last step, as sy_rollout_random documents)
        logic_tile<MODE, MAXA, 5, NT, CSRT, GROUPS>(p, lsm, tile0, threadIdx.x - (BW + WRW) * 32, &sg, &staged_flag, (unsigned)it, it + 1 < K);
      } else {  // complete the two hand-shakes of the observation roles
        asm volatile("bar.sync %0, %1;\n" ::"n"(LAG_CSR_BAR), "n"(CSRT) : "memory");
        asm volatile("bar.sync %0, %1;\n" ::"n"(LAG_BAR), "n"(NT) : "memory");
      }
    }
    asm volatile("bar.sync %0, %1;\n" ::"n"(ROLL_BAR), "n"(NT) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// fused persistent step kernel: ONE launch per sy_step.  Every CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...
// with three warp-specialised roles that run at their own pace:
//   logic warps   (LOGIC_WARPS)  the dynamics of tile k, k+1, ... back to back (logic_tile); after each tile they
//                                publish `tiles_done` (st.release).  Nothing they touch is shared with the other roles
//                                except through global memory, so they may run ahead freely.
//   writer warps  (FUSED_WR)     the dense observations of the tiles whose dynamics are done, as ONE continuous
//                                software pipeline over all of the CTA's chunks: zero fill of the NEXT chunk's float32
//                                piece (needs no state, so the store stream starts at cycle 0 and never stalls on the
//                                logic), image of this chunk, ones of the piece filled BULK_DEPTH chunks ago.
//   belief warps  (BW)           the belief propagation of the finished tiles (belief_role).
// The store stream goes through the TMA engine, so the logic's loads and shared-memory accesses no longer queue behind
// it in the LSU (what made the round-1 fused attempts slower than two kernels), and the latency-bound dynamics hide
// under a stream that is HBM-bound from the first microsecond.
// ---------------------------------------------------------------------------------------------
constexpr int FUSED_WR = 2;

__device__ __forceinline__ void publish_u32(unsigned* smem_word, unsigned v) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_word);
  asm volatile("st.release.cta.shared.u32 [%0], %1;\n" ::"r"(sa), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned acquire_u32(const unsigned* smem_word) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_word);
  unsigned v;
  asm volatile("ld.acquire.cta.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(sa) : "memory");
  return v;
}
// every lane of the warp continues only after the logic warps have finished tile index k of this CTA
__device__ __forceinline__ void wait_tiles_done(const unsigned* tiles_done, unsigned k, int lane, int clk_slot = -1) {
  const long long t0 = FCLK_NOW();
  if (lane == 0) {
    // the logic warps of this CTA never wait for anything, so the wait is bounded by their progress; the spin is
    // capped (~1 s) so that a can't-happen stall shows up as a wrong result in the parity tests, never as a hung GPU
    for (unsigned spins = 0; acquire_u32(tiles_done) <= k && spins < (1u << 24); ++spins) __nanosleep(64);
  }
  __syncwarp();
  if (clk_slot >= 0) FCLK_ADD(clk_slot, FCLK_NOW() - t0);
}

struct FusedSmemPlan {  // byte offsets into the dynamic shared memory of the fused kernel (Params carries them)
  int sbuf, sbuf_stride, zero, imgs, csr;
};

// One chunk of the writers' FAST geometry: a chunk is `epc` whole envs (epc * A <= 32), lane = (env, agent) pair, the
// tile sits on one staged graph whose nodes have at most 4 neighbours (s_nbr4: one LDS.128 per node holding 4 x
// {col | wgt << 16}, 0xFFFFFFFF = none).  Everything is straight-line code: no division, no loop.
struct PairView {
  bool valid;   // lane holds a live (env, agent) pair of the chunk
  int e, a;     // env inside the tile, agent
  int u, m;     // node, budget
};
// (GROUPS: an absent agent's pair is not valid: no mask ones, no node_features one)
template <int GROUPS = 0>
__device__ __forceinline__ PairView pair_of(const Params& p, const int* s_pos, const int* s_money, int cm, int epc, int nEnv, int lane) {
  PairView v;
  const int A = p.A;
  const int de = (lane * p.inv_A) >> 16;
  v.a = lane - de * A;
  v.e = cm * epc + de;
  v.valid = de < epc && v.e < nEnv;
  v.u = v.valid ? s_pos[v.e * A + v.a] : 0;
  if (GROUPS && v.u < 0) v.valid = false, v.u = 0;
  v.m = v.valid ? s_money[v.e * A + v.a] : 0;
  return v;
}
// affordable neighbours of the pair's node into (v = 1) or out of (v = 0) the chunk image (action_mask.py:65-76).
// s_nbr4[u] = the first four neighbours as {col | wgt << 16}, the degree in the top byte of .x; the rare nodes with
// more neighbours finish over the staged CSR.  GROUPS: the pair's budget is headroom (wr_budget).
template <int GROUPS = 0>
__device__ __forceinline__ void fast_mask_ones(const Params& p, const PairView& pv, const uint4* s_nbr4, const int* s_rp, const uint16_t* s_col,
                                               const uint8_t* s_wgt, uint8_t* img, int epc, int cm, uint8_t v) {
  if (!pv.valid) return;
  const uint4 nb = s_nbr4[pv.u];
  const int deg = (int)(nb.x >> 24);
  uint8_t* row = img + ((pv.e - cm * epc) * p.A + pv.a) * p.N;
  const int lim = pv.m - wr_toll<GROUPS>(p);  // wgt + toll <= m
  if (deg > 0 && (int)((nb.x >> 16) & 0xffu) <= lim) row[nb.x & 0xffffu] = v;
  if (deg > 1 && (int)(nb.y >> 16) <= lim) row[nb.y & 0xffffu] = v;
  if (deg > 2 && (int)(nb.z >> 16) <= lim) row[nb.z & 0xffffu] = v;
  if (deg > 3 && (int)(nb.w >> 16) <= lim) row[nb.w & 0xffffu] = v;
  if (deg > 4) {
    const int r0 = s_rp[pv.u];
    for (int k = r0 + 4; k < r0 + deg; ++k)
      if ((int)s_wgt[k] <= lim) row[s_col[k]] = v;
  }
}
// one-hot entries of the chunk's envs (float32 node_features): one 4-byte store per (env, agent) pair into the lines the
// zero fill has just completed (they are still in L2, the partial writes merge there).  Merging the ones that share a
// 16-byte granule with match.any + redux was measured far slower (MATCH is a slow instruction on this part).
__device__ __forceinline__ void fast_nf32_ones(const Params& p, const PairView& pv, const int* s_rev, uint8_t* gnf, int lane) {
  const int A = p.A;
  if (pv.valid && !(pv.a == 0 && s_rev[pv.e] < 0))  // the MrX column stays blank while he is hidden
    __stcs(reinterpret_cast<float*>(gnf + (size_t)pv.e * p.N * A * 4) + pv.u * A + pv.a, 1.0f);
}

template <int BW, int GROUPS = 0>
__device__ __forceinline__ void fused_writer_role(const Params& p, unsigned char* dyn, const unsigned* tiles_done, int w, int lane) {
  constexpr int D = BULK_DEPTH;
  const Tables& tb = p.tb;
  const int N = p.N, A = p.A;
  const int ntiles = (p.B + TILE - 1) / TILE;
  const int nk = ((int)blockIdx.x < ntiles) ? (ntiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  if (nk == 0) return;
  const int Cm = p.wr_c_mask;
  const bool nf8 = p.ob.node_features_u8 != nullptr;
  const size_t Sm = (size_t)A * N;
  uint8_t* zero_page = dyn + p.f_off_zero;
  uint8_t* my_img = dyn + p.f_off_imgs + (size_t)w * 2 * p.wr_img_bytes;
  int* s_rp = reinterpret_cast<int*>(dyn + p.wr_off_csr);
  uint16_t* s_col = reinterpret_cast<uint16_t*>(s_rp + N + 1);
  uint8_t* s_wgt = reinterpret_cast<uint8_t*>(s_col + tb.nnz_stride);
  uint4* s_nbr4 = reinterpret_cast<uint4*>(dyn + p.f_off_nbr4);  // [N] packed neighbour table of the staged graph (wr_epc only)
  const int tw = w * 32 + lane;
  for (int i = tw * 16; i < (1 + 2 * FUSED_WR) * p.wr_img_bytes; i += FUSED_WR * 32 * 16) *reinterpret_cast<uint4*>(zero_page + i) = make_uint4(0, 0, 0, 0);
  fence_proxy_async_smem();
  named_barrier(2, FUSED_WR * 32);
  auto tile_of = [&](int k) { return (int)blockIdx.x + k * (int)gridDim.x; };
  auto envs_of = [&](int k) { return min(TILE, p.B - tile_of(k) * TILE); };
  auto gnf_of = [&](int k) { return reinterpret_cast<uint8_t*>(p.ob.node_features) + (size_t)tile_of(k) * TILE * Sm * 4; };
  auto sbuf = [&](int k) { return reinterpret_cast<int*>(dyn + p.f_off_sbuf + (size_t)(k & 1) * p.f_sbuf_stride); };
  auto ctx_of = [&](int k) {
    int* b = sbuf(k);
    return BulkCtx{b, b + TILE * A, b + 2 * TILE * A, b + 2 * TILE * A + TILE, s_rp, s_col, s_wgt};
  };
  // zero fill of the float32 piece that belongs to mask chunk `cm` of a tile (lane 0 issues, the ragged tail is bytes)
  auto fill_piece = [&](uint8_t* g, int Tf32, int cm) {
    const int lo = 4 * cm * Cm, hi = min(Tf32, lo + 4 * Cm);
    if (lane == 0) nf32_fill_piece(g, lo, hi, zero_page, Cm);
    const int tail = (hi - lo) & 15;
    if (lane < tail) g[hi - tail + lane] = 0;
  };
  // ---- prologue: the whole float32 fill of this warp's share of the first tile -- it needs no state, so the store
  // stream runs while the logic warps are still busy with the tile
  if (!nf8) {
    const int Tm0 = envs_of(0) * (int)Sm;
    uint8_t* g0 = gnf_of(0);
    for (int cm = w; cm < (Tm0 + Cm - 1) / Cm; cm += FUSED_WR) fill_piece(g0, 4 * Tm0, cm);
  }
  if (lane == 0) bulk_commit();
  // chunks whose image ones / float32 ones are still owed, oldest first: (tile index k, item, fast geometry?)
  int ring_k[D], ring_item[D], ring_fast[D];
  int pending = 0, it = 0, last_g = -2;
  bool staged = false;
  // generic (any geometry) forms, used when a tile is not on the fast path
  auto generic_img = [&](int k, int item, const ImageStreams& st, uint8_t* img, uint8_t v) {
    const BulkCtx c = ctx_of(k);
    if (item < st.ncf) {
      const int lo = item * p.wr_c_nf;
      bulk_nf_ones<1, GROUPS>(p, c, img, lo, min(p.wr_c_nf, st.Tf - lo), lane, v != 0);
    } else {
      const int lo = (item - st.ncf) * Cm, len = min(Cm, st.Tm - lo);
      if (staged) bulk_mask_ones<true, GROUPS>(p, c, img, lo, len, lane, v);
      else bulk_mask_ones<false, GROUPS>(p, c, img, lo, len, lane, v);
    }
  };
  auto owed_ones = [&](int k, int item, int fast) {  // float32 ones of an older chunk, after its fill has completed
    if (nf8) return;
    int* b = sbuf(k);
    if (fast) {
      const PairView pv = pair_of<GROUPS>(p, b, b + TILE * A, item, p.wr_epc, envs_of(k), lane);
      fast_nf32_ones(p, pv, b + 2 * TILE * A, gnf_of(k), lane);
    } else {
      const ImageStreams so = image_streams(p, tile_of(k) * TILE, envs_of(k));
      if (item >= so.ncf) {
        const int lo = 4 * (item - so.ncf) * Cm;
        nf32_ones_piece<GROUPS>(p, ctx_of(k), gnf_of(k), lo, min(4 * so.Tm, lo + 4 * Cm), lane);
      }
    }
  };
  for (int k = 0; k < nk; ++k) {
    const int tile0 = tile_of(k) * TILE, nEnv = envs_of(k);
    const ImageStreams st = image_streams(p, tile0, nEnv);
    uint8_t* gnf = nf8 ? nullptr : gnf_of(k);
    // the state buffer of tile k is the one tile k-2 used: its owed ones (tiny tiles only) must be out first
    if (pending && ring_k[0] <= k - 2) {
      if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
      __syncwarp();
      for (int q = 0; q < pending; ++q) owed_ones(ring_k[q], ring_item[q], ring_fast[q]);
      pending = 0;
    }
    named_barrier(2, FUSED_WR * 32);  // every writer warp is done with the staged tables of the previous tile
    wait_tiles_done(tiles_done, (unsigned)k, lane, w == 0 ? 0 : -1);
    int* sb = sbuf(k);
    bool restage = false;
    {  // stage the tile's post-step state (and its graph's tables when the graph changed)
      const int gl = (lane < nEnv) ? __ldcg(p.st.graph_id + tile0 + lane) : -1;
      const int g0 = __shfl_sync(FULL, gl, 0);
      const bool one_graph = p.wr_stage_csr && __all_sync(FULL, gl == g0 || gl < 0);
      for (int i = tw; i < nEnv * A; i += FUSED_WR * 32) {
        sb[i] = __ldcg(p.st.pos + (size_t)tile0 * A + i);
        sb[TILE * A + i] = wr_budget<GROUPS>(p, __ldcg(p.st.money + (size_t)tile0 * A + i), tile0 + ((i * p.inv_A) >> 16));
      }
      if (tw < nEnv) {
        sb[2 * TILE * A + tw] = __ldcg(p.ob.mrx_revealed + tile0 + tw);
        sb[2 * TILE * A + TILE + tw] = gl;
      }
      if (one_graph && g0 != last_g) {
        restage = true;
        const int32_t* grp = tb.row_ptr + (size_t)g0 * (N + 1);
        const int nnz = __ldg(grp + N);
        for (int i = tw; i <= N; i += FUSED_WR * 32) s_rp[i] = __ldg(grp + i);
        for (int q = tw; q < nnz; q += FUSED_WR * 32) {
          s_col[q] = __ldg(tb.col + (size_t)g0 * tb.nnz_stride + q);
          s_wgt[q] = __ldg(tb.wgt + (size_t)g0 * tb.nnz_stride + q);
        }
      }
      staged = one_graph;
      last_g = one_graph ? g0 : -2;
    }
    named_barrier(2, FUSED_WR * 32);
    if (restage && p.wr_epc) {  // packed neighbour table of the newly staged graph
      for (int u = tw; u < N; u += FUSED_WR * 32) {
        const int r0 = s_rp[u], deg = s_rp[u + 1] - r0;  // deg <= 255 (sy_load_graphs)
        unsigned e4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) e4[q] = q < deg ? ((unsigned)s_col[r0 + q] | ((unsigned)s_wgt[r0 + q] << 16)) : 0u;
        s_nbr4[u] = make_uint4(e4[0] | ((unsigned)deg << 24), e4[1], e4[2], e4[3]);
      }
      named_barrier(2, FUSED_WR * 32);
    }
    const int fast = (p.wr_epc && staged && st.ncf == 0) ? 1 : 0;
    const int total = st.ncf + st.ncm;
    // next tile's geometry, for the look-ahead fill of its first chunk
    const bool have_next = !nf8 && k + 1 < nk;
    const int Tm_next = have_next ? envs_of(k + 1) * (int)Sm : 0;
    uint8_t* gnf_next = have_next ? gnf_of(k + 1) : nullptr;
    for (int item = w; item < total; item += FUSED_WR, ++it) {
      // ---- group F: zero fill for this warp's NEXT chunk (same tile, or the first chunk of the next tile)
      long long tc = FCLK_NOW();
      if (!nf8) {
        if (item + FUSED_WR < total) {
          if (k > 0) fill_piece(gnf, 4 * st.Tm, item + FUSED_WR);  // (tile 0 was filled by the prologue)
        } else if (have_next && w < (Tm_next + Cm - 1) / Cm) {
          fill_piece(gnf_next, 4 * Tm_next, w);
        }
      }
      if (lane == 0) bulk_commit();
      if (w == 0) { const long long t1 = FCLK_NOW(); FCLK_ADD(8, t1 - tc); tc = t1; }
      // ---- group M: the chunk's image
      uint8_t* img = my_img + (size_t)(it & 1) * p.wr_img_bytes;
      if (it >= 2) {  // the engine has read the image's previous chunk (younger groups: F, M of the last chunk and this F)
        const long long tw0 = FCLK_NOW();
        if (lane == 0) bulk_wait_read<3>();
        __syncwarp();
        if (w == 0) FCLK_ADD(6, FCLK_NOW() - tw0);
        // take that chunk's ones back out (it is the oldest entry of the ring: D == 2 chunks ago)
        static_assert(D == 2, "the image ring and the owed-ones ring are the same two chunks");
        if (pending == D && ring_fast[0]) {  // (after a tile-boundary flush the ring is short: clear the whole image)
          int* ob = sbuf(ring_k[0]);
          const PairView pv = pair_of<GROUPS>(p, ob, ob + TILE * A, ring_item[0], p.wr_epc, envs_of(ring_k[0]), lane);
          fast_mask_ones<GROUPS>(p, pv, s_nbr4, s_rp, s_col, s_wgt, img, p.wr_epc, ring_item[0], 0);
        } else {
          for (int i = lane * 16; i < p.wr_img_bytes; i += 32 * 16) *reinterpret_cast<uint4*>(img + i) = make_uint4(0, 0, 0, 0);
        }
        __syncwarp();
      }
      if (w == 0) { const long long t1 = FCLK_NOW(); FCLK_ADD(9, t1 - tc); tc = t1; }
      const bool is_nf8 = item < st.ncf;
      const int lo = is_nf8 ? item * p.wr_c_nf : (item - st.ncf) * Cm;
      const int len = is_nf8 ? min(p.wr_c_nf, st.Tf - lo) : min(Cm, st.Tm - lo);
      if (fast) {
        const PairView pv = pair_of<GROUPS>(p, sb, sb + TILE * A, item, p.wr_epc, nEnv, lane);
        fast_mask_ones<GROUPS>(p, pv, s_nbr4, s_rp, s_col, s_wgt, img, p.wr_epc, item, 1);
      } else {
        generic_img(k, item, st, img, 1);
      }
      if (w == 0) { const long long t1 = FCLK_NOW(); FCLK_ADD(10, t1 - tc); tc = t1; }
      fence_proxy_async_smem();
      __syncwarp();
      if (w == 0) { const long long t1 = FCLK_NOW(); FCLK_ADD(11, t1 - tc); tc = t1; }
      uint8_t* dst = (is_nf8 ? st.gf : st.gm) + lo;
      const int body = len & ~15;
      if (lane == 0) {
        if (body) bulk_store(dst, img, (unsigned)body);
        bulk_commit();
      }
      if (lane < len - body) dst[body + lane] = img[body + lane];  // ragged end of the batch's last tile only
      if (w == 0) { const long long t1 = FCLK_NOW(); FCLK_ADD(12, t1 - tc); tc = t1; }
      // ---- ones of the chunk whose piece was filled D + 1 chunks ago (younger groups: its own M, then F + M of D + 1 chunks)
      if (pending == D) {
        const long long tw0 = FCLK_NOW();
        if (lane == 0) asm volatile("cp.async.bulk.wait_group %0;\n" ::"n"(2 * D + 3) : "memory");
        __syncwarp();
        if (w == 0) FCLK_ADD(7, FCLK_NOW() - tw0);
        owed_ones(ring_k[0], ring_item[0], ring_fast[0]);
#pragma unroll
        for (int q = 0; q + 1 < D; ++q) {
          ring_k[q] = ring_k[q + 1];
          ring_item[q] = ring_item[q + 1];
          ring_fast[q] = ring_fast[q + 1];
        }
        pending = D - 1;
      }
      if (w == 0) { const long long t1 = FCLK_NOW(); FCLK_ADD(13, t1 - tc); tc = t1; }
      ring_k[pending] = k;
      ring_item[pending] = item;
      ring_fast[pending] = fast;
      ++pending;
    }
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");  // also: shared memory outlives the engine's reads
  __syncwarp();
  for (int q = 0; q < pending; ++q) owed_ones(ring_k[q], ring_item[q], ring_fast[q]);
}

template <int MODE, int MAXA, int BW, int GROUPS = 0>
__global__ void __launch_bounds__((BW + FUSED_WR + LOGIC_WARPS) * 32, 2) sy_step_fused_kernel(const Params p) {
  extern __shared__ __align__(16) unsigned char dyn[];
  __shared__ LogicSmem<MAXA> lsm;
  __shared__ unsigned tiles_done;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) tiles_done = 0;
  __syncthreads();
  const int ntiles = (p.B + TILE - 1) / TILE;
  if (warp < BW) {
    if constexpr (BW > 0) {
      if (!p.belief_on) return;
      const long long t0 = FCLK_NOW();
      for (int k = 0, t = blockIdx.x; t < ntiles; t += gridDim.x, ++k) {
        if (k) named_barrier(1, BW * 32);  // every belief warp has left the previous tile's scratch
        wait_tiles_done(&tiles_done, (unsigned)k, lane, warp == 0 ? 2 : -1);
        belief_role<BW, 0, GROUPS>(p, dyn, t * TILE, min(TILE, p.B - t * TILE), warp, lane);
      }
      if (warp == 0) FCLK_ADD(3, FCLK_NOW() - t0);
    }
  } else if (warp < BW + FUSED_WR) {
    const long long t0 = FCLK_NOW();
    fused_writer_role<BW, GROUPS>(p, dyn, &tiles_done, warp - BW, lane);
    if (warp == BW) FCLK_ADD(1, FCLK_NOW() - t0);
  } else {
    const int tid = threadIdx.x - (BW + FUSED_WR) * 32;
    unsigned k = 0;
    const long long t0 = FCLK_NOW();
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
      logic_tile<MODE, MAXA, 3, 0, 0, GROUPS>(p, lsm, t * TILE, tid);
      __threadfence_block();
      named_barrier(3, LOGIC_THREADS);  // every logic thread's stores of the tile are ordered; lsm may be reused
      ++k;
      if (tid == 0) publish_u32(&tiles_done, k);
    }
    if (tid == 0) {
      FCLK_ADD(4, FCLK_NOW() - t0);
      FCLK_ADD(5, 1);
    }
  }
}

// statistics: fold the replicated accumulators into the caller's vector and clear them
__global__ void sy_fold_stats_kernel(unsigned long long* rep, long long* out) {
  const int k = threadIdx.x;
  if (k >= SY_NUM_STATS) return;
  unsigned long long sum = 0;
  for (int r = 0; r < STAT_REPLICAS; ++r) {
    sum += rep[r * SY_NUM_STATS + k];
    rep[r * SY_NUM_STATS + k] = 0;
  }
  out[k] += (long long)sum;
}

// per-group statistics: fold the replicas of each group's line into the caller's [n, SY_NUM_STATS] table and clear them
__global__ void sy_fold_group_stats_kernel(unsigned long long* rep, int n, int reps, long long* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // = group * SY_NUM_STATS + statistic
  if (i >= n * SY_NUM_STATS) return;
  unsigned long long sum = 0;
  for (int r = 0; r < reps; ++r) {
    sum += rep[(size_t)r * n * SY_NUM_STATS + i];
    rep[(size_t)r * n * SY_NUM_STATS + i] = 0;
  }
  out[i] += (long long)sum;
}

// sy_set_groups: group ids in range ([B] -> count of ids outside [0, n)), or the default assignment (env_offset + b) % n
__global__ void sy_group_ids_kernel(const int32_t* in, int32_t* out, int B, int n, unsigned long long env_offset, int* bad) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (in) {
    const int g = in[b];
    if (g < 0 || g >= n) atomicAdd(bad, 1);
    out[b] = g;
  } else {
    out[b] = (int32_t)((env_offset + (unsigned long long)b) % (unsigned long long)n);
  }
}

// sy_reset after sy_set_groups: envs the mask leaves out
__global__ void sy_count_unset_kernel(const uint8_t* mask, int B, int* unset) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B && mask[b] == 0) atomicAdd(unset, 1);
}

// ---------------------------------------------------------------------------------------------
// random valid policy: thread per (env, agent)
// ---------------------------------------------------------------------------------------------
// GROUPS: each env's moves are tested against its mechanism group's toll; its absent agents get -1
template <typename ActT, int GROUPS = 0>
__global__ void __launch_bounds__(256) sy_sample_actions_kernel(const Params p, unsigned step_counter, ActT* actions,
                                                                const unsigned* __restrict__ step_base) {
  if (step_base) step_counter += *step_base;  // device-resident counter: a captured CUDA graph keeps advancing
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;  // B * A < 2^31 (checked at sy_create)
  if (i >= (unsigned)p.B * (unsigned)p.A) return;
  const unsigned b = i / (unsigned)p.A, a = i - b * (unsigned)p.A;
  if (agent_absent<GROUPS>(p, (int)b, (int)a)) {  // before any table lookup at its node (-1)
    actions[i] = (ActT)-1;
    return;
  }
  const Tables& tb = p.tb;
  const int N = p.N;
  const int g = p.st.graph_id[b], u = p.st.pos[i], m = p.st.money[i];
  const int toll = env_toll_of<GROUPS>(p, (int)b);
  const int nvalid = move_count(tb, N, g, u, m, toll);  // one table lookup instead of a pass over the row
  long long act = -1;
  if (nvalid > 0) {
    const unsigned env_id = (unsigned)(p.env_offset + (unsigned long long)b);
    const uint4 r = philox4x32(make_uint4(env_id, step_counter, RNG_ACTION, a), make_uint2(p.seed_lo, p.seed_hi));
    int pick = (int)__umulhi(r.x, (unsigned)nvalid);
    const uint8_t* wg = tb.wgt + (size_t)g * tb.nnz_stride;
    for (int k = __ldg(tb.row_ptr + (size_t)g * (N + 1) + u);; ++k) {  // the pick-th affordable neighbour exists
      if (__ldg(wg + k) + toll <= m) {
        if (pick == 0) {
          act = __ldg(tb.col + (size_t)g * tb.nnz_stride + k);
          break;
        }
        --pick;
      }
    }
  }
  actions[i] = (ActT)act;
}

__global__ void sy_advance_counter_kernel(unsigned* counter, unsigned by) { *counter += by; }

// trajectory recording (SURVEY 8(f) f1): up to SY_MAX_COPY_SEGMENTS device-to-device copies in ONE launch (blockIdx.y =
// segment) instead of one copy kernel per stored tensor and step
struct CopySegments {
  void* dst[SY_MAX_COPY_SEGMENTS];
  const void* src[SY_MAX_COPY_SEGMENTS];
  unsigned long long bytes[SY_MAX_COPY_SEGMENTS];
};
__global__ void __launch_bounds__(256) sy_copy_segments_kernel(const CopySegments c) {
  const int sgm = blockIdx.y;
  const unsigned long long n = c.bytes[sgm];
  uint8_t* d = static_cast<uint8_t*>(c.dst[sgm]);
  const uint8_t* sr = static_cast<const uint8_t*>(c.src[sgm]);
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (unsigned long long)gridDim.x * blockDim.x;
  if (((reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(sr)) & 15u) == 0) {
    const unsigned long long nv = n >> 4;
    for (unsigned long long i = tid; i < nv; i += nth) reinterpret_cast<uint4*>(d)[i] = reinterpret_cast<const uint4*>(sr)[i];
    for (unsigned long long i = (nv << 4) + tid; i < n; i += nth) d[i] = sr[i];
  } else {
    for (unsigned long long i = tid; i < n; i += nth) d[i] = sr[i];
  }
}

// ---------------------------------------------------------------------------------------------
// graph table construction
// ---------------------------------------------------------------------------------------------
// one CTA per (graph, node): dense weight row, move-count row, 1/deg
__global__ void sy_build_rows_kernel(int N, int Ns, int nnz_stride, int wcap, const int32_t* row_ptr,
                                     const uint16_t* col, const uint8_t* wgt, uint8_t* W, uint8_t* cnt,
                                     float* inv_deg) {
  const int g = blockIdx.y, u = blockIdx.x;
  const int r0 = row_ptr[(size_t)g * (N + 1) + u], r1 = row_ptr[(size_t)g * (N + 1) + u + 1];
  uint8_t* row = W + ((size_t)g * N + u) * Ns;
  for (int j = threadIdx.x; j < Ns; j += blockDim.x) row[j] = 0;
  __syncthreads();
  for (int k = r0 + threadIdx.x; k < r1; k += blockDim.x) row[col[(size_t)g * nnz_stride + k]] = wgt[(size_t)g * nnz_stride + k];
  for (int c = threadIdx.x; c <= wcap; c += blockDim.x) {
    int n = 0;
    for (int k = r0; k < r1; ++k) n += (wgt[(size_t)g * nnz_stride + k] <= c);
    cnt[((size_t)g * N + u) * (wcap + 1) + c] = (uint8_t)min(n, 255);
  }
  if (threadIdx.x == 0) inv_deg[(size_t)g * N + u] = (r1 > r0) ? 1.0f / (float)(r1 - r0) : 0.0f;
}

// nodes of every graph ordered by degree (stable counting sort, one thread per graph: setup path, N <= 65535)
__global__ void sy_degree_perm_kernel(int N, const int32_t* row_ptr, uint16_t* perm, int* scratch /*[G, 257]*/) {
  const int g = blockIdx.x;
  if (threadIdx.x != 0) return;
  const int32_t* rp = row_ptr + (size_t)g * (N + 1);
  int* cnt = scratch + (size_t)g * 257;
  for (int d = 0; d <= 256; ++d) cnt[d] = 0;
  for (int u = 0; u < N; ++u) cnt[min(rp[u + 1] - rp[u], 255) + 1] += 1;
  for (int d = 1; d <= 256; ++d) cnt[d] += cnt[d - 1];
  for (int u = 0; u < N; ++u) perm[(size_t)g * N + cnt[min(rp[u + 1] - rp[u], 255)]++] = (uint16_t)u;
}

// all-pairs shortest paths, one warp per (graph, source): in-place Bellman-Ford relaxation to a fixed point
// (replaces the per-query heap Dijkstra of pathfinding.py:34-137; weights are positive integers)
__global__ void sy_apsp_kernel(int G, int N, int nnz_stride, const int32_t* row_ptr, const uint16_t* col,
                               const uint8_t* wgt, uint16_t* D, int warps_per_block) {
  extern __shared__ int sdist_all[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long wg = (long long)blockIdx.x * warps_per_block + warp;
  if (wg >= (long long)G * N) return;
  const int g = (int)(wg / N), src = (int)(wg - (long long)g * N);
  volatile int* dist = sdist_all + (size_t)warp * N;
  const int32_t* rp = row_ptr + (size_t)g * (N + 1);
  const uint16_t* cl = col + (size_t)g * nnz_stride;
  const uint8_t* wt = wgt + (size_t)g * nnz_stride;
  const int BIG = 0x3fffffff;
  for (int v = lane; v < N; v += 32) dist[v] = (v == src) ? 0 : BIG;
  __syncwarp();
  bool changed = true;
  while (changed) {
    changed = false;
    for (int v = lane; v < N; v += 32) {
      int best = dist[v];
      for (int k = rp[v]; k < rp[v + 1]; ++k) best = min(best, dist[cl[k]] + (int)wt[k]);
      if (best < dist[v]) {
        dist[v] = best;
        changed = true;
      }
    }
    changed = __any_sync(FULL, changed);
    __syncwarp();
  }
  uint16_t* out = D + ((size_t)g * N + src) * N;
  for (int v = lane; v < N; v += 32) out[v] = (uint16_t)(dist[v] >= DIST_INF ? DIST_INF : dist[v]);
}

// ---------------------------------------------------------------------------------------------
// device-side graph sampler (SURVEY 8(f) row f3): ConnectedGraph.sample (graph_layout.py:9-80) plus the
// resample-until-the-edge-count-matches loop of CustomEnvironment.reset (yard.py:87-101), one warp per pool slot.
// Same distribution as the reference (argument in oracle/sy_oracle.py above philox_sample_graph_once, which restates
// this kernel draw for draw): uniform insertion order (Fisher-Yates), every node attaches to a uniform earlier one,
// then the extra edges one at a time, each uniform over the non-adjacent pairs of the nodes still under the degree
// cap (rejection sampling over ordered pairs of open nodes; the number V of acceptable pairs is tracked exactly, so
// the loop ends when the reference's scan would find nothing more).  Every lane carries the same scalars; lane 0
// writes, the warp shares the counting loops.  The adjacency being built is the pool's dense weight table itself.
// ---------------------------------------------------------------------------------------------
enum { RNG_GEN_PERM = 16, RNG_GEN_PARENT = 17, RNG_GEN_TREE_W = 18, RNG_GEN_PAIR = 19, RNG_GEN_EXTRA_W = 20 };
constexpr int GEN_MAX_ATTEMPTS = 100;  // yard.py:89
constexpr unsigned GEN_MAX_DRAWS = 1u << 22;
constexpr int GEN_MAX_NODES = 8192;

struct GenStream {  // k-th 32-bit word of Philox(seed; graph, generation * 128 + attempt, purpose, k >> 2)
  uint2 key;
  unsigned c0, c1, c2;
  int blk;
  uint4 w;
  __device__ GenStream(uint2 key_, unsigned graph, unsigned ga, unsigned purpose) : key(key_), c0(graph), c1(ga), c2(purpose), blk(-1), w(make_uint4(0, 0, 0, 0)) {}
  __device__ unsigned word(int k) {
    if ((k >> 2) != blk) {
      blk = k >> 2;
      w = philox4x32(make_uint4(c0, c1, c2, (unsigned)blk), key);
    }
    return word_of(w, k & 3);
  }
};

struct GenParams {
  int N, Ns, max_edges, num_edges, cap, wrange;
  unsigned seed_lo, seed_hi, generation, graph_offset;
  int probe;            // 1: sample GLOBAL graph 0 into slot 0 and publish its edge count (the constructor's probe, yard.py:67-76)
  int* want;            // device scalar: the edge count every slot must reach
  uint8_t* W;           // [G, N, Ns]
  ushort2* edges;       // [G, max_edges] in the reference's order: tree edges, then the extras
  uint8_t* edge_w;      // [G, max_edges]
  int* edge_count;      // [G]
  int* status;          // [G] attempts used (0-based), -1 = no sample with the wanted count, -2 = draw budget exhausted
};

__global__ void __launch_bounds__(32) sy_sample_graphs_kernel(const GenParams q) {
  extern __shared__ __align__(16) unsigned char gen_smem[];
  const int N = q.N, Ns = q.Ns, lane = threadIdx.x;
  int* deg = reinterpret_cast<int*>(gen_smem);
  uint16_t* order = reinterpret_cast<uint16_t*>(deg + N);
  uint16_t* open = order + N;
  uint16_t* opos = open + N;
  const int g = blockIdx.x;
  const unsigned gid = q.probe ? 0u : q.graph_offset + (unsigned)g;
  const int want = q.probe ? 0 : *q.want;
  const uint2 key = make_uint2(q.seed_lo, q.seed_hi);
  uint8_t* Wg = q.W + (size_t)g * N * Ns;
  volatile uint8_t* Wv = Wg;
  ushort2* edges = q.edges + (size_t)g * q.max_edges;
  uint8_t* ew = q.edge_w + (size_t)g * q.max_edges;
  int E = 0, attempt = 0, status = -1;
  for (; attempt < GEN_MAX_ATTEMPTS; ++attempt) {
    const unsigned ga = q.generation * 128u + (unsigned)attempt;
    uint4* W16 = reinterpret_cast<uint4*>(Wg);
    for (int i = lane; i < N * (Ns >> 4); i += 32) W16[i] = make_uint4(0, 0, 0, 0);
    for (int i = lane; i < N; i += 32) {
      order[i] = (uint16_t)i;
      deg[i] = 0;
    }
    __syncwarp();
    if (lane == 0) {  // uniform insertion order
      GenStream ps(key, gid, ga, RNG_GEN_PERM);
      for (int k = 0; k < N - 1; ++k) {
        const int j = k + (int)__umulhi(ps.word(k), (unsigned)(N - k));
        const uint16_t t = order[k];
        order[k] = order[j];
        order[j] = t;
      }
    }
    __syncwarp();
    for (int k = 1 + lane; k < N; k += 32) {  // tree: the k-th node joins a uniform earlier one
      const uint4 rp = philox4x32(make_uint4(gid, ga, RNG_GEN_PARENT, (unsigned)(k >> 2)), key);
      const uint4 rw = philox4x32(make_uint4(gid, ga, RNG_GEN_TREE_W, (unsigned)(k >> 2)), key);
      const int u = order[__umulhi(word_of(rp, k & 3), (unsigned)k)], v = order[k];
      const int wt = 1 + (int)__umulhi(word_of(rw, k & 3), (unsigned)q.wrange);
      Wv[(size_t)u * Ns + v] = (uint8_t)wt;
      Wv[(size_t)v * Ns + u] = (uint8_t)wt;
      edges[k - 1] = make_ushort2((unsigned short)u, (unsigned short)v);
      ew[k - 1] = (uint8_t)wt;
      atomicAdd(deg + u, 1);
      atomicAdd(deg + v, 1);
    }
    __threadfence_block();
    __syncwarp();
    int n_open = 0;  // nodes under the degree cap, ascending
    for (int base = 0; base < N; base += 32) {
      const int u = base + lane;
      const bool o = u < N && deg[u] < q.cap;
      const unsigned m = __ballot_sync(FULL, o);
      if (o) {
        const int idx = n_open + __popc(m & ((1u << lane) - 1u));
        open[idx] = (uint16_t)u;
        opos[u] = (uint16_t)idx;
      }
      n_open += __popc(m);
    }
    __syncwarp();
    int both = 0;
    for (int k = lane; k < N - 1; k += 32) {
      const ushort2 e = edges[k];
      both += (deg[e.x] < q.cap && deg[e.y] < q.cap);
    }
    both = __reduce_add_sync(FULL, both);
    long long V = (long long)n_open * (n_open - 1) / 2 - both;  // acceptable pairs
    int extra = q.num_edges - (N - 1), n_extra = 0;
    unsigned draw = 0;
    bool exhausted = false;
    GenStream pair_s(key, gid, ga, RNG_GEN_PAIR), xw_s(key, gid, ga, RNG_GEN_EXTRA_W);
    while (extra > 0 && V > 0) {
      if (draw >= GEN_MAX_DRAWS) {
        exhausted = true;
        break;
      }
      const int a = (int)__umulhi(pair_s.word((int)draw), (unsigned)n_open);
      int b = (int)__umulhi(pair_s.word((int)draw + 1), (unsigned)(n_open - 1));
      draw += 2;
      if (b >= a) ++b;
      const int i = open[a], j = open[b];
      if (Wv[(size_t)i * Ns + j]) continue;
      const int wt = 1 + (int)__umulhi(xw_s.word(n_extra), (unsigned)q.wrange);
      if (lane == 0) {
        Wv[(size_t)i * Ns + j] = (uint8_t)wt;
        Wv[(size_t)j * Ns + i] = (uint8_t)wt;
        edges[N - 1 + n_extra] = make_ushort2((unsigned short)i, (unsigned short)j);
        ew[N - 1 + n_extra] = (uint8_t)wt;
        deg[i] += 1;
        deg[j] += 1;
      }
      __threadfence_block();
      __syncwarp();
      --V;
      --extra;
      ++n_extra;
#pragma unroll
      for (int side = 0; side < 2; ++side) {
        const int x = side ? j : i;
        if (deg[x] >= q.cap) {  // x closes: swap-with-last removal; its still-acceptable pairs disappear
          __syncwarp();
          if (lane == 0) {
            const uint16_t last = open[n_open - 1], px = opos[x];
            open[px] = last;
            opos[last] = px;
          }
          --n_open;
          __syncwarp();
          int c = 0;
          for (int t = lane; t < n_open; t += 32) c += (Wv[(size_t)x * Ns + open[t]] == 0);
          V -= __reduce_add_sync(FULL, c);
        }
      }
    }
    E = N - 1 + n_extra;
    if (exhausted) {
      status = -2;
      break;
    }
    if (want <= 0 || E == want) {
      status = attempt;
      break;
    }
  }
  if (lane == 0) {
    q.edge_count[g] = E;
    q.status[g] = status;
    if (q.probe) *q.want = E;
  }
}

// CSR, padded neighbour lists and their offsets from the dense weight table; one CTA per graph
__global__ void __launch_bounds__(256) sy_csr_from_dense_kernel(int N, int Ns, int nnz_stride, int pack_stride, const uint8_t* W,
                                                                int32_t* row_ptr, uint16_t* col, uint8_t* wgt, int2* pack,
                                                                int32_t* pack_ptr, int* status) {
  extern __shared__ int csr_smem[];
  int* sdeg = csr_smem;            // [N]
  int* srow = csr_smem + N;        // [N + 1]
  int* spk = csr_smem + 2 * N + 1; // [N + 1]
  const int g = blockIdx.x, tid = threadIdx.x;
  const uint8_t* Wg = W + (size_t)g * N * Ns;
  for (int u = tid; u < N; u += blockDim.x) {
    const uint4* row = reinterpret_cast<const uint4*>(Wg + (size_t)u * Ns);
    int d = 0;
    for (int v = 0; v < (Ns >> 4); ++v) {
      const uint4 x = row[v];
      const unsigned wds[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int b = 0; b < 4; ++b) d += ((wds[q] >> (8 * b)) & 0xFFu) != 0;
    }
    sdeg[u] = d;
  }
  __syncthreads();
  if (tid == 0) {
    int a = 0, b = 0, bad = 0;
    for (int u = 0; u < N; ++u) {
      const int d = sdeg[u];
      srow[u] = a;
      spk[u] = b;
      a += d;
      b += (d + 3) & ~3;
      bad |= d > 255;
    }
    srow[N] = a;
    spk[N] = b;
    if (bad || a > nnz_stride || b > pack_stride) status[g] = -3;
  }
  __syncthreads();
  if (srow[N] > nnz_stride || spk[N] > pack_stride) return;
  for (int u = tid; u <= N; u += blockDim.x) {
    row_ptr[(size_t)g * (N + 1) + u] = srow[u];
    pack_ptr[(size_t)g * (N + 1) + u] = spk[u];
  }
  for (int u = tid; u < N; u += blockDim.x) {
    int k = srow[u], pk = spk[u];
    const uint8_t* row = Wg + (size_t)u * Ns;
    for (int v = 0; v < N; ++v) {
      const int w = row[v];
      if (w) {
        col[(size_t)g * nnz_stride + k] = (uint16_t)v;
        wgt[(size_t)g * nnz_stride + k] = (uint8_t)w;
        pack[(size_t)g * pack_stride + pk] = make_int2(v * BSTRIDE * (int)sizeof(float), __float_as_int(1.0f / (float)sdeg[v]));
        ++k;
        ++pk;
      }
    }
    for (; pk < spk[u + 1]; ++pk) pack[(size_t)g * pack_stride + pk] = make_int2(0, 0);
  }
}

// ---------------------------------------------------------------------------------------------
// dense float64 action mask == compute_action_mask (action_mask.py:30-83); one CTA per query
// ---------------------------------------------------------------------------------------------
__global__ void sy_mask_dense_kernel(int N, const double* adj, const double* w, const double* toll_m, double toll_s,
                                     const int32_t* cur, const double* budget, uint8_t* out) {
  const int q = blockIdx.x;
  const int u = cur[q];
  const double bud = budget[q];
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const double a = adj[(size_t)u * N + j];
    const double wt = w ? w[(size_t)u * N + j] : a;            // action_mask.py:110-112
    const double tl = toll_m ? toll_m[(size_t)u * N + j] : toll_s;
    const double cost = __dadd_rn(wt, tl);                     // action_mask.py:72
    out[(size_t)q * N + j] = (j != u) && (a != 0.0) && (cost <= bud);
  }
}

// ---------------------------------------------------------------------------------------------
// heuristic opponents (sy_heuristic_actions): an evading MrX and chasing police, the counterpart of the heuristics of
// src/eval/exploitability.py:122,188 (parity unpinned: the rules are those of include/sy_env.h, restated by
// oracle/heuristic_oracle.py).  CTA per 32-env tile: warp per env for the per-env part (MrX's last known node,
// the chase target, the belief argmax read as coalesced rows), then thread per (env, agent) for the actions.
// ---------------------------------------------------------------------------------------------
constexpr unsigned RNG_HEURISTIC = 4;  // Philox purpose of the exploration draws (0..3 and 16..20 are taken)
constexpr int HEUR_ENVS = 32, HEUR_THREADS = 256;

struct HeurArgs {
  int mrx_kind, police_kind;
  unsigned long long thr_mrx, thr_police;  // explore iff Philox word < threshold (epsilon * 2^32)
  int32_t* last_seen;                      // [B] or NULL
  long long* actions;                      // int64 [B, A]
  unsigned step_counter;
};

// the draw of sy_sample_actions_kernel for a present agent at node u with budget m
__device__ __forceinline__ int heur_random_action(const Params& p, unsigned b, unsigned a, int g, int u, int m, int toll,
                                                  unsigned step_counter) {
  const Tables& tb = p.tb;
  const int nvalid = move_count(tb, p.N, g, u, m, toll);
  if (nvalid <= 0) return -1;
  const unsigned env_id = (unsigned)(p.env_offset + (unsigned long long)b);
  const uint4 r = philox4x32(make_uint4(env_id, step_counter, RNG_ACTION, a), make_uint2(p.seed_lo, p.seed_hi));
  int pick = (int)__umulhi(r.x, (unsigned)nvalid);
  const uint8_t* wg = tb.wgt + (size_t)g * tb.nnz_stride;
  for (int k = __ldg(tb.row_ptr + (size_t)g * (p.N + 1) + u);; ++k) {  // the pick-th affordable neighbour exists
    if (__ldg(wg + k) + toll <= m) {
      if (pick == 0) return __ldg(tb.col + (size_t)g * tb.nnz_stride + k);
      --pick;
    }
  }
}

template <int GROUPS>
__global__ void __launch_bounds__(HEUR_THREADS) sy_heuristic_actions_kernel(const Params p, const HeurArgs h) {
  __shared__ int s_pos[HEUR_ENVS * AS];   // positions of the tile (row = env)
  __shared__ int s_target[HEUR_ENVS];     // chase target per env, -1 unknown
  const int b0 = blockIdx.x * HEUR_ENVS, ne = min(HEUR_ENVS, p.B - b0), A = p.A, N = p.N;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < ne * A; i += HEUR_THREADS) {
    const int e = i / A;
    s_pos[e * AS + (i - e * A)] = p.st.pos[(size_t)b0 * A + i];
  }
  for (int e = warp; e < ne; e += HEUR_THREADS / 32) {
    const int b = b0 + e;
    const int rev = p.ob.mrx_revealed[b];
    const int ls = rev >= 0 ? rev : ((h.last_seen && p.st.timestep[b] != 0) ? h.last_seen[b] : -1);
    int target = ls;
    if (h.police_kind == SY_HEUR_CHASE_BELIEF && rev < 0) {  // first argmax of the belief row
      const float* row = p.st.belief + (size_t)b * N;
      float best = -INFINITY;
      int bi = N;
      for (int j = lane; j < N; j += 32) {
        const float v = row[j];
        if (v > best) best = v, bi = j;
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const float ov = __shfl_xor_sync(FULL, best, off);
        const int oi = __shfl_xor_sync(FULL, bi, off);
        if (ov > best || (ov == best && oi < bi)) best = ov, bi = oi;
      }
      target = bi < N ? bi : 0;  // (a row without an ordered maximum, e.g. all NaN: node 0)
    }
    if (lane == 0) {
      s_target[e] = target;
      if (h.last_seen) h.last_seen[b] = ls;
    }
  }
  __syncthreads();
  const Tables& tb = p.tb;
  for (int i = tid; i < ne * A; i += HEUR_THREADS) {
    const int e = i / A, a = i - e * A, b = b0 + e;
    const int kind = a == 0 ? h.mrx_kind : h.police_kind;
    if (kind == SY_HEUR_NONE) continue;
    const GroupRow* gr = GROUPS ? p.grp + __ldg(p.grp_id + b) : nullptr;
    const int P = env_police<GROUPS>(p, gr);
    long long act = -1;
    if (a <= P) {  // absent agents: -1
      const int* sp = s_pos + e * AS;
      const int g = p.st.graph_id[b], u = sp[a], m = p.st.money[(size_t)b * A + a];
      const int toll = env_toll<GROUPS>(p, gr);
      const unsigned long long thr = a == 0 ? h.thr_mrx : h.thr_police;
      bool random = kind == SY_HEUR_RANDOM || (a > 0 && s_target[e] < 0);
      if (!random && thr) {
        const uint4 r = philox4x32(make_uint4((unsigned)(p.env_offset + (unsigned long long)b), h.step_counter, RNG_HEURISTIC,
                                              (unsigned)a), make_uint2(p.seed_lo, p.seed_hi));
        random = (unsigned long long)r.x < thr;
      }
      if (random) {
        act = heur_random_action(p, b, a, g, u, m, toll, h.step_counter);
      } else {
        const int k0 = __ldg(tb.row_ptr + (size_t)g * (N + 1) + u), k1 = __ldg(tb.row_ptr + (size_t)g * (N + 1) + u + 1);
        const uint16_t* col = tb.col + (size_t)g * tb.nnz_stride;
        const uint8_t* wg = tb.wgt + (size_t)g * tb.nnz_stride;
        const uint16_t* Dg = tb.D + (size_t)g * N * N;
        if (a == 0) {  // evade: the candidate farthest from the nearest police; ties: stay, then the lowest node
          int best = u, best_s = INT_MAX;
          for (int i2 = 1; i2 <= P; ++i2) best_s = min(best_s, (int)__ldg(Dg + (size_t)u * N + sp[i2]));
          for (int k = k0; k < k1; ++k) {
            const int c = __ldg(col + k);
            if (__ldg(wg + k) + toll > m) continue;
            bool occupied = false;
            for (int i2 = 1; i2 <= P; ++i2) occupied |= sp[i2] == c;
            if (occupied) continue;
            const uint16_t* row = Dg + (size_t)c * N;
            int s = INT_MAX;
            for (int i2 = 1; i2 <= P; ++i2) s = min(s, (int)__ldg(row + sp[i2]));
            if (s > best_s) best = c, best_s = s;
          }
          act = best;
        } else {  // chase: the free affordable neighbour nearest to the target (D symmetric: one row, D[target][.])
          const uint16_t* row = Dg + (size_t)s_target[e] * N;
          int best = -1, best_d = INT_MAX;
          bool affordable = false;
          for (int k = k0; k < k1; ++k) {
            const int c = __ldg(col + k);
            if (__ldg(wg + k) + toll > m) continue;
            affordable = true;
            bool occupied = false;
            for (int i2 = 1; i2 <= P; ++i2) occupied |= sp[i2] == c;
            if (occupied) continue;
            const int d = __ldg(row + c);
            if (d < best_d) best = c, best_d = d;
          }
          act = best >= 0 ? best : (affordable ? u : -1);  // boxed in by police: stays, but acts
        }
      }
    }
    h.actions[(size_t)b * A + a] = act;
  }
}

}  // namespace

// =============================================================================================
// host side
// =============================================================================================
struct SyEnv {
  SyConfig cfg;
  int A = 0;
  bool graphs_loaded = false;
  bool tables_set = false;
  Tables tb{};
  // device allocations owned by the handle
  void* d_W = nullptr;
  void* d_D = nullptr;
  void* d_row_ptr = nullptr;
  void* d_col = nullptr;
  void* d_wgt = nullptr;
  void* d_cnt = nullptr;
  void* d_inv_deg = nullptr;
  void* d_pack = nullptr;
  void* d_pack_ptr = nullptr;
  void* d_deg_perm = nullptr;
  // device graph sampler (sy_generate_graphs): edge lists in the reference's order, per-slot edge count / status
  void* d_edges = nullptr;
  void* d_edge_w = nullptr;
  void* d_edge_count = nullptr;
  void* d_gen_status = nullptr;
  void* d_gen_want = nullptr;
  int gen_max_edges = 0;  // > 0: the pool was sampled on the device
  int alloc_G = 0, alloc_nnz = 0, alloc_wcap = 0, alloc_pack = 0;  // shape of the current table allocations
  void* d_bel_flags = nullptr;  // [B] u8, logic/reset kernel -> observe kernel
  void* d_stats_rep = nullptr;  // [STAT_REPLICAS, SY_NUM_STATS] u64
  cudaStream_t aux_stream = nullptr;  // host-buffer path: result copies overlap the observe kernel
  int host_overlap = 0;               // sy_set_host_overlap
  bool aux_after_logic = false;       // the aux stream is ordered behind the last step's dynamics, nothing else touched the state since
  cudaEvent_t ev_main = nullptr;      // orders the aux stream behind the caller's stream when that is not known
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;  // sy_rollout_random_dev: sampler of the next step next to the observe kernel
  cudaEvent_t ev_logic = nullptr, ev_copied = nullptr;
  void* d_exp = nullptr;
  void* d_cov = nullptr;
  size_t bel_smem = 0;  // dynamic smem of the step / reset kernels (belief scratch)
  int bel_fast = 0, bel_off_out = 0, bel_off_part = 0, bel_off_pack = 0, bel_off_ptr = 0;
  int wr_off = 0, wr_off_csr = 0, wr_img_stride = 0, wr_stage_csr = 0, bel_share_csr = 0, wr_img_rows = 0, wr_off_pad = 0;
  int wr_c_mask = 0, wr_c_nf32 = 0, wr_c_nf8 = 0, wr_img_bytes = 0;  // bulk writers: chunk sizes per stream, image size
  // fused persistent step kernel (sy_step_fused_kernel): plan made with the graph tables
  bool fused_ok = false;
  int f_bw = 0, f_off_sbuf = 0, f_sbuf_stride = 0, f_off_zero = 0, f_off_imgs = 0, f_off_csr = 0, f_c_mask = 0, f_img_bytes = 0;
  int f_stage_csr = 0, f_grid = 0, f_epc = 0, f_off_nbr4 = 0;
  size_t f_smem = 0;
  // sy_set_option(SY_OPT_STEP_KERNEL): SY_STEP_AUTO = the fused persistent kernel for batches that fit its grid in one
  // wave (launch-latency bound: one launch instead of two, c2 runs 19 % faster), else the dynamics + observation kernels
  // (at 65 536 envs the fused kernel is slower: DESIGN.md section 4c)
  int opt_fused = SY_STEP_AUTO;
  int opt_fill = 0;   // sy_set_option(SY_OPT_NF_FILL): 1 = split step (fill kernel next to the dynamics, belief next to the writers)
  cudaStream_t split_stream = nullptr;  // split step: dynamics + belief run here, fill + writers on the caller's stream
  cudaEvent_t ev_split_start = nullptr, ev_split_logic = nullptr, ev_split_belief = nullptr;
  int fill_grid = 0;
  int opt_writer = SY_WRITER_LSU;  // sy_set_option(SY_OPT_WRITER_PATH) for the stand-alone observe kernel (sy_reset, two-kernel sy_step)
  int bel_warps = BEL_WARPS, wr_warps = WR_WARPS;  // role split of the observe kernel for this pool
  size_t obs_smem = 0;  // dynamic smem of the observe kernel: belief scratch + writer staging
  // software-pipelined steps (sy_step_deferred): the dense observations of the current state have not been written yet;
  // the next dynamics launch carries them (sy_step_lagged_kernel), sy_flush_observations / any plain call writes them
  int obs_slots = 0;        // resident CTAs of the observation kernel on this device (occupancy x SMs)
  int opt_tail_split = 1;   // sy_set_option(SY_OPT_TAIL_SPLIT)
  bool obs_pending = false;
  int64_t* pending_stats = nullptr;  // SyOut.stats of the step whose observations are pending (flush / reset have no SyOut)
  bool lag_ok = false;  // the lagged kernel fits this shape with two CTAs per SM
  // sy_set_option(SY_OPT_LAGGED_KERNEL): SY_LAGGED_AUTO = a deferred step with pending observations is ONE launch (and the
  // random rollouts step deferred) when the batch's tiles fit one wave of the lagged kernel, where a step costs
  // max(dynamics, observations) instead of their sum: c2 (1 024 envs) 11.8 -> 8.8 us per step, c3-shaped batches of 4 096 /
  // 9 472 envs 28.1 -> 17.0 / 33.8 -> 23.1 us.  Larger batches keep two launches: the dynamics warps take 21 us per tile next
  // to the store stream (13 us alone) and hold the CTA's slot after its observation roles are done, which every further
  // wave pays again (16 384 envs 44.4 vs 40.8 us, 65 536 envs 156 vs 129 us).
  int opt_lagged = SY_LAGGED_AUTO;
  int lag_slots = 0;  // resident CTAs of the lagged kernel (occupancy x SMs)
  int opt_pdl = 0;  // sy_set_option(SY_OPT_PDL): dynamics / observation kernels launched with programmatic stream serialisation
  int opt_rollout_kernel = 1;  // sy_set_option(SY_OPT_ROLLOUT_KERNEL): random rollouts of single-wave batches as ONE launch
  // mechanism groups (sy_set_groups).  While they are set, steps run the GROUPS instantiations of the dynamics kernel (and
  // of the observation kernel when belief scores are collected) as two launches: the fused / lagged / one-launch rollout
  // kernels and the split step are not instantiated for groups
  int grp_n = 0, grp_rep = 0;
  void* d_grp = nullptr;         // GroupRow [SY_MAX_GROUPS], rows [0, grp_n) in use
  void* d_grp_id = nullptr;      // int32 [B]
  void* d_grp_id_new = nullptr;  // int32 [B] staging of sy_set_groups (validated before it replaces d_grp_id)
  void* d_grp_bad = nullptr;     // int: ids out of range
  void* d_grp_stats = nullptr;   // u64 [GROUP_STAT_LINES, SY_NUM_STATS]: [grp_rep, grp_n] lines in use
  bool grp_need_reset = false;  // groups changed: steps are refused until a full sy_reset
  std::vector<GroupRow> grp_rows;  // host copy of the rows in use (sy_set_group_tolls rewrites their tolls)
};

namespace {

void free_graph_tables(SyEnv* e) {
  for (void** ptr : {&e->d_W, &e->d_D, &e->d_row_ptr, &e->d_col, &e->d_wgt, &e->d_cnt, &e->d_inv_deg, &e->d_pack, &e->d_pack_ptr, &e->d_deg_perm,
                     &e->d_edges, &e->d_edge_w, &e->d_edge_count, &e->d_gen_status, &e->d_gen_want}) {
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr;
  }
  e->graphs_loaded = false;
  e->gen_max_edges = 0;
  e->alloc_G = e->alloc_nnz = e->alloc_wcap = e->alloc_pack = 0;
}

int finish_graph_tables(SyEnv* e, int G, int nnz_stride, int wcap, int pack_stride, cudaStream_t s);

// (re)allocate the pool tables; an unchanged shape keeps the allocations, so pointers baked into captured CUDA
// graphs stay valid across pool refreshes
int alloc_graph_tables(SyEnv* e, int G, int nnz_stride, int wcap, int pack_stride) {
  const int N = e->cfg.num_nodes;
  if (e->d_W && e->alloc_G == G && e->alloc_nnz == nnz_stride && e->alloc_wcap == wcap && e->alloc_pack == pack_stride) return SY_OK;
  free_graph_tables(e);
  const int Ns = (N + 15) & ~15;
  CUDA_TRY(cudaMalloc(&e->d_W, (size_t)G * N * Ns));
  CUDA_TRY(cudaMalloc(&e->d_D, (size_t)G * N * N * sizeof(uint16_t)));
  CUDA_TRY(cudaMalloc(&e->d_row_ptr, (size_t)G * (N + 1) * sizeof(int32_t)));
  CUDA_TRY(cudaMalloc(&e->d_col, (size_t)G * nnz_stride * sizeof(uint16_t)));
  CUDA_TRY(cudaMalloc(&e->d_wgt, (size_t)G * nnz_stride));
  CUDA_TRY(cudaMalloc(&e->d_cnt, (size_t)G * N * (wcap + 1) + 16));  // + 16: vector loads of the last row's tail
  CUDA_TRY(cudaMalloc(&e->d_inv_deg, (size_t)G * N * sizeof(float)));
  CUDA_TRY(cudaMalloc(&e->d_pack, (size_t)G * pack_stride * sizeof(int2)));
  CUDA_TRY(cudaMalloc(&e->d_pack_ptr, (size_t)G * (N + 1) * sizeof(int32_t)));
  CUDA_TRY(cudaMalloc(&e->d_deg_perm, (size_t)G * N * sizeof(uint16_t)));
  e->alloc_G = G;
  e->alloc_nnz = nnz_stride;
  e->alloc_wcap = wcap;
  e->alloc_pack = pack_stride;
  return SY_OK;
}

// chunk size (bytes, multiple of 16, <= cap) of a bulk-writer stream whose envs are S bytes each: whole groups of envs
// when the smallest 16-byte sized group fits (leaving every writer warp a few chunks per tile), else a 16-byte
// multiple that divides the group evenly when there is one in [cap / 2, cap], else just cap (chunks may then straddle
// env boundaries, which the writers handle)
int plan_bulk_chunk(size_t S, int cap, int wr_warps) {
  size_t g = 16;
  while (S % g) g >>= 1;  // gcd(S, 16)
  const size_t m = 16 / g, group = S * m;
  cap &= ~15;
  if (group <= (size_t)cap) {
    size_t k = cap / group;
    const size_t kmax = std::max<size_t>(1, (TILE / m) / (2 * (size_t)wr_warps));
    k = std::min(k, kmax);
    return (int)(group * k);
  }
  for (int c = cap; c >= cap / 2 && c >= 16; c -= 16)
    if (group % (size_t)c == 0) return c;
  return cap;
}

using FusedFn = void (*)(const Params);
template <int BW, int GR>
FusedFn fused_fn_bw(int reward_mode, int A) {
  const bool f64 = reward_mode == SY_REWARD_FP64;
  if (A <= 4) return f64 ? sy_step_fused_kernel<SY_REWARD_FP64, 4, BW, GR> : sy_step_fused_kernel<SY_REWARD_FP32, 4, BW, GR>;
  if (A <= 8) return f64 ? sy_step_fused_kernel<SY_REWARD_FP64, 8, BW, GR> : sy_step_fused_kernel<SY_REWARD_FP32, 8, BW, GR>;
  return f64 ? sy_step_fused_kernel<SY_REWARD_FP64, 16, BW, GR> : sy_step_fused_kernel<SY_REWARD_FP32, 16, BW, GR>;
}
// groups: the GROUPS instantiation (mechanism groups are set)
FusedFn fused_fn(int bw, int reward_mode, int A, bool groups = false) {
  if (groups) return bw ? fused_fn_bw<BEL_WARPS, 1>(reward_mode, A) : fused_fn_bw<0, 1>(reward_mode, A);
  return bw ? fused_fn_bw<BEL_WARPS, 0>(reward_mode, A) : fused_fn_bw<0, 0>(reward_mode, A);
}

// shared-memory plan, grid and eligibility of the fused step kernel for this handle's shape (called with the tables)
int plan_fused(SyEnv* e, int nnz_stride) {
  const int N = e->cfg.num_nodes, A = e->A;
  e->fused_ok = false;
  if (e->cfg.belief && !e->bel_fast) return SY_OK;  // large-N belief path shares the writers' CSR: two-kernel path
  e->f_bw = e->cfg.belief ? BEL_WARPS : 0;
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const int cap = std::max(256, (int)(SY_BULK_IMG_BUDGET / (2 * FUSED_WR + 1)));
  e->f_c_mask = plan_bulk_chunk((size_t)A * N, cap, FUSED_WR);
  e->f_img_bytes = e->f_c_mask;
  const size_t csr = ((((size_t)(N + 1) * sizeof(int) + (size_t)nnz_stride * 3) + 3) & ~(size_t)3) + 16;
  e->f_stage_csr = csr <= 32 * 1024 ? 1 : 0;
  e->f_sbuf_stride = (int)up16(((size_t)2 * TILE * A + 2 * TILE) * sizeof(int));
  e->f_off_sbuf = (int)up16(e->cfg.belief ? e->bel_smem : 0);
  e->f_off_zero = e->f_off_sbuf + 2 * e->f_sbuf_stride;
  e->f_off_imgs = e->f_off_zero + e->f_img_bytes;
  e->f_off_csr = (int)up16((size_t)e->f_off_imgs + (size_t)2 * FUSED_WR * e->f_img_bytes);
  // fast geometry: a chunk is whole envs with at most 32 (env, agent) pairs, rows are whole granules, and the staged
  // graph gets a packed neighbour table (one uint4 per node)
  const size_t S = (size_t)A * N;
  e->f_epc = (e->f_stage_csr && e->f_c_mask % S == 0 && (e->f_c_mask / S) * A <= 32 && S % 4 == 0 && N <= 2048) ? (int)(e->f_c_mask / S) : 0;
  e->f_off_nbr4 = (int)up16((size_t)e->f_off_csr + (e->f_stage_csr ? csr : 0));
  e->f_smem = (size_t)e->f_off_nbr4 + (e->f_epc ? (size_t)N * 16 : 0);
  if (e->f_smem > 200 * 1024) return SY_OK;
  FusedFn fn = fused_fn(e->f_bw, e->cfg.reward_mode, A);
  if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess ||
      cudaFuncSetAttribute(fused_fn(e->f_bw, e->cfg.reward_mode, A, true), cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) {
    cudaGetLastError();
    return SY_OK;
  }
  int per_sm = 0, sms = 0;
  const int threads = (e->f_bw + FUSED_WR + LOGIC_WARPS) * 32;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, e->f_smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    return SY_OK;
  }
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
  const int ntiles = (e->cfg.num_envs + TILE - 1) / TILE;
  e->f_grid = std::min(ntiles, per_sm * sms);
  e->fused_ok = true;
  return SY_OK;
}

template <int BW, int GR>
FusedFn lagged_fn_bw(int reward_mode, int A) {
  const bool f64 = reward_mode == SY_REWARD_FP64;
  if (A <= 4) return f64 ? sy_step_lagged_kernel<SY_REWARD_FP64, 4, BW, WR_WARPS, GR> : sy_step_lagged_kernel<SY_REWARD_FP32, 4, BW, WR_WARPS, GR>;
  if (A <= 8) return f64 ? sy_step_lagged_kernel<SY_REWARD_FP64, 8, BW, WR_WARPS, GR> : sy_step_lagged_kernel<SY_REWARD_FP32, 8, BW, WR_WARPS, GR>;
  return f64 ? sy_step_lagged_kernel<SY_REWARD_FP64, 16, BW, WR_WARPS, GR> : sy_step_lagged_kernel<SY_REWARD_FP32, 16, BW, WR_WARPS, GR>;
}
using RolloutFn = void (*)(const Params, const int);
template <int BW, int GR>
RolloutFn rollout_fn_bw(int reward_mode, int A) {
  const bool f64 = reward_mode == SY_REWARD_FP64;
  if (A <= 4) return f64 ? sy_rollout_lagged_kernel<SY_REWARD_FP64, 4, BW, WR_WARPS, GR> : sy_rollout_lagged_kernel<SY_REWARD_FP32, 4, BW, WR_WARPS, GR>;
  if (A <= 8) return f64 ? sy_rollout_lagged_kernel<SY_REWARD_FP64, 8, BW, WR_WARPS, GR> : sy_rollout_lagged_kernel<SY_REWARD_FP32, 8, BW, WR_WARPS, GR>;
  return f64 ? sy_rollout_lagged_kernel<SY_REWARD_FP64, 16, BW, WR_WARPS, GR> : sy_rollout_lagged_kernel<SY_REWARD_FP32, 16, BW, WR_WARPS, GR>;
}
// groups: the GROUPS instantiation (mechanism groups are set)
RolloutFn rollout_fn(const SyEnv* e, bool groups = false) {
  if (groups) return e->cfg.belief ? rollout_fn_bw<BEL_WARPS, 1>(e->cfg.reward_mode, e->A) : rollout_fn_bw<0, 1>(e->cfg.reward_mode, e->A);
  return e->cfg.belief ? rollout_fn_bw<BEL_WARPS, 0>(e->cfg.reward_mode, e->A) : rollout_fn_bw<0, 0>(e->cfg.reward_mode, e->A);
}
FusedFn lagged_fn(const SyEnv* e, bool groups = false) {
  if (groups) return e->cfg.belief ? lagged_fn_bw<BEL_WARPS, 1>(e->cfg.reward_mode, e->A) : lagged_fn_bw<0, 1>(e->cfg.reward_mode, e->A);
  return e->cfg.belief ? lagged_fn_bw<BEL_WARPS, 0>(e->cfg.reward_mode, e->A) : lagged_fn_bw<0, 0>(e->cfg.reward_mode, e->A);
}
int lagged_threads(const SyEnv* e) { return ((e->cfg.belief ? BEL_WARPS : 0) + WR_WARPS + LOGIC_WARPS) * 32; }

// eligibility of the lagged step kernel for this handle's shape: the default role split, and two CTAs per SM (with one
// the observation stream loses more than the overlap gains: such shapes keep two launches)
int plan_lagged(SyEnv* e) {
  e->lag_ok = false;
  if (e->bel_warps != BEL_WARPS || e->wr_warps != WR_WARPS) return SY_OK;
  FusedFn fn = lagged_fn(e);
  static std::mutex mu;
  static size_t limit[64][12] = {};  // per device and instantiation: the attribute is only ever raised (see below)
  {
    std::lock_guard<std::mutex> lock(mu);
    const int slot = (e->cfg.belief ? 6 : 0) + (e->cfg.reward_mode == SY_REWARD_FP64 ? 3 : 0) + (e->A <= 4 ? 0 : (e->A <= 8 ? 1 : 2));
    size_t& cur = limit[e->cfg.device & 63][slot];
    if (e->obs_smem > cur) {
      if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->obs_smem) != cudaSuccess ||
          cudaFuncSetAttribute(rollout_fn(e), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->obs_smem) != cudaSuccess ||
          cudaFuncSetAttribute(lagged_fn(e, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->obs_smem) != cudaSuccess ||
          cudaFuncSetAttribute(rollout_fn(e, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->obs_smem) != cudaSuccess) {
        cudaGetLastError();
        return SY_OK;
      }
      cur = e->obs_smem;
    }
  }
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, lagged_threads(e), e->obs_smem) != cudaSuccess) {
    cudaGetLastError();
    return SY_OK;
  }
  e->lag_ok = per_sm >= 2;
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device) != cudaSuccess) {
    cudaGetLastError();
    sms = 0;
  }
  e->lag_slots = per_sm * sms;
  return SY_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the FUNCTION (per device), not to a handle: it is only ever
// raised, so a small env created next to a large one cannot pull the limit below what the large one launches with
int raise_observe_smem_limit(int device, size_t bytes) {
  static std::mutex mu;
  static size_t limit[64] = {};
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = limit[device & 63];
  if (bytes <= cur) return SY_OK;
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<BEL_WARPS, WR_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<BEL_WARPS, WR_WARPS, WV_BULK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS, WV_BULK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<BEL_WARPS, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<0, WR_WARPS, WV_ONES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<BEL_WARPS, WR_WARPS, WV_LSU, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS, WV_LSU, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<BEL_WARPS, WR_WARPS, WV_BULK, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  CUDA_TRY(cudaFuncSetAttribute(sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS, WV_BULK, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  cur = bytes;
  return SY_OK;
}

// <<<>>> with the programmatic-serialisation attribute (pdl): the kernel may be scheduled while its predecessor in the
// stream still runs; it calls pdl_wait() before it touches anything that predecessor writes
template <typename K>
void launch_ex(K kernel, unsigned grid, unsigned block, size_t smem, cudaStream_t s, bool pdl, const Params& p) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, p);
}

void launch_observe(const SyEnv* e, const Params& p0, unsigned grid, cudaStream_t s) {
  const bool gen = e->bel_warps == GEN_BEL_WARPS && GEN_BEL_WARPS != BEL_WARPS;
  Params p = p0;
  p.ob_full = (int)grid;
  p.ob_split = 1;
  if (e->obs_slots > 0 && e->opt_tail_split && !p.wr_bulk) {
    const int full = (int)(grid / (unsigned)e->obs_slots) * e->obs_slots, rest = (int)grid - full;
    // (fast belief path: lane = env, a part costs its belief warps what a whole tile costs: measured slower, no split)
    const int kmax = (p.belief_on && e->bel_fast) ? 1 : 4;
    int k = 1;
    while (rest > 0 && k < kmax && rest * (k * 2) <= e->obs_slots) k *= 2;  // parts per tile that still fit one wave
    // (measured at c4: the tail in halves 0.321 ms per step, no split 0.333, EVERY tile in halves 0.349, in quarters 0.384
    //  -- a part pays the tile's fixed staging again)
    if (k > 1) {
      p.ob_full = full;
      p.ob_split = k;
      grid = (unsigned)(full + rest * k);
    }
  }
  if (p.grp_n) {  // mechanism groups: every env's own toll, belief scores also summed per group
    if (p.wr_bulk) {
      if (gen) sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS, WV_BULK, 1><<<grid, THREADS, e->obs_smem, s>>>(p);
      else sy_observe_kernel<BEL_WARPS, WR_WARPS, WV_BULK, 1><<<grid, THREADS, e->obs_smem, s>>>(p);
    } else {
      if (gen) launch_ex(sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS, WV_LSU, 1>, grid, THREADS, e->obs_smem, s, e->opt_pdl != 0, p);
      else launch_ex(sy_observe_kernel<BEL_WARPS, WR_WARPS, WV_LSU, 1>, grid, THREADS, e->obs_smem, s, e->opt_pdl != 0, p);
    }
  } else if (p.wr_bulk) {
    if (gen) sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS, WV_BULK><<<grid, THREADS, e->obs_smem, s>>>(p);
    else sy_observe_kernel<BEL_WARPS, WR_WARPS, WV_BULK><<<grid, THREADS, e->obs_smem, s>>>(p);
  } else {
    if (gen) launch_ex(sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS>, grid, THREADS, e->obs_smem, s, e->opt_pdl != 0, p);
    else launch_ex(sy_observe_kernel<BEL_WARPS, WR_WARPS>, grid, THREADS, e->obs_smem, s, e->opt_pdl != 0, p);
  }
}

int fill_params(const SyEnv* env, const SyState* st, const SyObs* ob, const SyOut* out, Params& p) {
  const SyConfig& c = env->cfg;
  if (!env->graphs_loaded) return fail(SY_ERR_STATE, "sy_load_graphs must be called first");
  if (!env->tables_set) return fail(SY_ERR_STATE, "sy_set_reward_tables must be called first");
  // ABI guard of the pointer structs: a binding compiled against another header revision is refused before any of its
  // (mis-laid-out) pointers can reach a kernel
  if (!st) return fail(SY_ERR_INVALID_ARGUMENT, "SyState is NULL");
  if (st->struct_bytes != sizeof(SyState)) return fail(SY_ERR_INVALID_ARGUMENT, "SyState size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)st->struct_bytes, sizeof(SyState), SY_ABI_VERSION);
  if (ob && ob->struct_bytes != sizeof(SyObs)) return fail(SY_ERR_INVALID_ARGUMENT, "SyObs size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)ob->struct_bytes, sizeof(SyObs), SY_ABI_VERSION);
  if (out && out->struct_bytes != sizeof(SyOut)) return fail(SY_ERR_INVALID_ARGUMENT, "SyOut size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)out->struct_bytes, sizeof(SyOut), SY_ABI_VERSION);
  if (!st->pos || !st->money || !st->timestep || !st->graph_id || !st->episode || !st->done || !st->visits)
    return fail(SY_ERR_INVALID_ARGUMENT, "SyState has NULL members");
  if (c.belief && !st->belief) return fail(SY_ERR_INVALID_ARGUMENT, "SyState.belief is NULL but config.belief is on");
  std::memset(&p, 0, sizeof(p));
  p.B = c.num_envs;
  p.N = c.num_nodes;
  p.P = c.num_police;
  p.A = env->A;
  p.inv_A = (65536 + env->A - 1) / env->A;
  p.agent_money = c.agent_money;
  p.mrx_money = c.mrx_money;
  p.max_t = c.max_timestep;
  p.reveal = c.reveal_interval;
  p.toll = c.toll;
  p.belief_on = c.belief != 0;
  p.belief_score = c.belief == SY_BELIEF_SCORED;
  p.auto_reset = c.auto_reset;
  p.resample_graph = c.resample_graph;
  p.reward_mode = c.reward_mode;
  p.env_offset = (unsigned long long)c.env_offset;
  p.reveal_skip_thresh = c.reveal_skip_prob > 0.0f ? (unsigned long long)((double)fminf(c.reveal_skip_prob, 1.0f) * 4294967296.0) : 0ull;
  p.belief_hint = st->belief_hint;
  p.seed_lo = (unsigned)(c.seed & 0xffffffffu);
  p.seed_hi = (unsigned)(c.seed >> 32);
  for (int i = 0; i < SY_NUM_REWARD_WEIGHTS; ++i) {
    p.w64[i] = c.reward_weights[i];
    p.w32[i] = (float)c.reward_weights[i];
  }
  p.tb = env->tb;
#ifdef SY_PROFILING_BUILD  // kernel-part ablations for profiling variants only; the shipped library has no such switch
  {
    static const int dbg = [] { const char* v = getenv("SY_DEBUG_SKIP"); return v ? atoi(v) : 0; }();
    p.dbg_skip = dbg;
  }
#endif
  p.bel_flags = (uint8_t*)env->d_bel_flags;
  p.stats_rep = (unsigned long long*)env->d_stats_rep;
  p.bel_fast = env->bel_fast;
  p.bel_off_out = env->bel_off_out;
  p.bel_off_part = env->bel_off_part;
  p.bel_off_pack = env->bel_off_pack;
  p.bel_off_ptr = env->bel_off_ptr;
  p.wr_off = env->wr_off;
  p.wr_off_csr = env->wr_off_csr;
  p.wr_img_stride = env->wr_img_stride;
  p.wr_stage_csr = env->wr_stage_csr;
  p.wr_img_rows = env->wr_img_rows;
  p.wr_off_pad = env->wr_off_pad;
  p.bel_share_csr = (p.dbg_skip & 5) ? 0 : env->bel_share_csr;  // the hand-over barrier needs both roles
  p.st = *st;
  if (ob) p.ob = *ob;
  if (out) p.out = *out;
  if (ob) {  // bulk stores need 16-byte aligned streams (a tile is 32 envs, so aligned bases are enough)
    const uintptr_t bits = reinterpret_cast<uintptr_t>(ob->action_mask) | reinterpret_cast<uintptr_t>(ob->node_features_u8 ? (void*)ob->node_features_u8 : (void*)ob->node_features);
    p.wr_bulk = (env->opt_writer == SY_WRITER_BULK && (bits & 15u) == 0) ? 1 : 0;
    p.wr_c_mask = env->wr_c_mask;
    p.wr_c_nf = ob->node_features_u8 ? env->wr_c_nf8 : env->wr_c_nf32;
    p.wr_img_bytes = env->wr_img_bytes;
  }
  if (env->grp_n) {
    p.grp = (const GroupRow*)env->d_grp;
    p.grp_id = (const int32_t*)env->d_grp_id;
    p.grp_n = env->grp_n;
    p.grp_rep = env->grp_rep;
    p.grp_stats = (unsigned long long*)env->d_grp_stats;
  }
  return SY_OK;
}



int check_obs(const SyObs* ob) {
  if (ob && ob->struct_bytes != sizeof(SyObs)) return fail(SY_ERR_INVALID_ARGUMENT, "SyObs size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)ob->struct_bytes, sizeof(SyObs), SY_ABI_VERSION);
  if (!ob || !ob->action_mask || (!ob->node_features && !ob->node_features_u8) || !ob->agent_budget || !ob->mrx_revealed)
    return fail(SY_ERR_INVALID_ARGUMENT, "SyObs has NULL members");
  return SY_OK;
}

}  // namespace

extern "C" {

#ifdef SY_PHASE_CLOCKS
int sy_debug_phase_clocks(unsigned long long* out8, int reset) {  // profiling builds only, not declared in sy_env.h
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out8, g_phase_clk, sizeof(unsigned long long) * 16);
  if (reset) {
    unsigned long long z[16] = {};
    cudaMemcpyToSymbol(g_phase_clk, z, sizeof(z));
  }
  return 0;
}
#endif
#ifdef SY_FUSED_CLOCKS
int sy_debug_fused_clocks(unsigned long long* out16, int reset) {  // profiling builds only, not declared in sy_env.h
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out16, g_fused_clk, sizeof(unsigned long long) * 16);
  if (reset) {
    unsigned long long z[16] = {};
    cudaMemcpyToSymbol(g_fused_clk, z, sizeof(z));
  }
  return 0;
}
#endif
int sy_abi_version(void) { return SY_ABI_VERSION; }
const char* sy_last_error(void) { return g_err.c_str(); }
int64_t sy_launch_count(void) { return (int64_t)g_launches.load(); }

int sy_create(const SyConfig* c, SyEnv** out_env) {
  if (!c || !out_env) return fail(SY_ERR_INVALID_ARGUMENT, "NULL config / out_env");
  if (c->struct_bytes != (int32_t)sizeof(SyConfig))
    return fail(SY_ERR_INVALID_ARGUMENT, "SyConfig size mismatch: got %d, library expects %zu", c->struct_bytes, sizeof(SyConfig));
  if (c->num_envs <= 0) return fail(SY_ERR_INVALID_ARGUMENT, "num_envs must be positive");
  if ((long long)c->num_envs * (c->num_police + 1) >= (1LL << 31)) return fail(SY_ERR_INVALID_ARGUMENT, "num_envs x agents must stay below 2^31 per handle");
  if (c->num_police < 1 || c->num_police + 1 > SY_MAX_AGENTS)
    return fail(SY_ERR_INVALID_ARGUMENT, "num_police must be in [1, %d]", SY_MAX_AGENTS - 1);
  if (c->num_nodes < c->num_police + 1 || c->num_nodes > 65534)
    return fail(SY_ERR_INVALID_ARGUMENT, "num_nodes must be in [num_police + 1, 65534]");  // nodes are staged as u16
  if (c->agent_money < 0 || c->mrx_money < 0 || c->toll < 0 || c->reveal_interval < 0 || c->max_timestep < 0)
    return fail(SY_ERR_INVALID_ARGUMENT, "negative money / toll / reveal_interval / max_timestep");
  if (c->toll > SY_MAX_TOLL) return fail(SY_ERR_INVALID_ARGUMENT, "toll %d outside [0, %d]", c->toll, SY_MAX_TOLL);
  if (c->max_timestep > SY_MAX_TIMESTEP)  // longer episodes would saturate the u16 visit counters
    return fail(SY_ERR_INVALID_ARGUMENT, "max_timestep %d outside [0, %d]", c->max_timestep, SY_MAX_TIMESTEP);
  if (!(c->reveal_skip_prob >= 0.0f && c->reveal_skip_prob <= 1.0f)) return fail(SY_ERR_INVALID_ARGUMENT, "reveal_skip_prob must be in [0, 1]");
  if (c->reward_mode != SY_REWARD_FP64 && c->reward_mode != SY_REWARD_FP32)
    return fail(SY_ERR_INVALID_ARGUMENT, "unknown reward_mode %d", c->reward_mode);
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (c->device < 0 || c->device >= ndev) return fail(SY_ERR_INVALID_ARGUMENT, "device %d out of range (%d visible)", c->device, ndev);
  CUDA_TRY(cudaSetDevice(c->device));
  SyEnv* e = new SyEnv();
  e->cfg = *c;
  e->A = c->num_police + 1;
  if (cudaMalloc(&e->d_bel_flags, (size_t)c->num_envs) != cudaSuccess ||
      cudaMalloc(&e->d_stats_rep, (size_t)STAT_REPLICAS * SY_NUM_STATS * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(e->d_stats_rep, 0, (size_t)STAT_REPLICAS * SY_NUM_STATS * sizeof(unsigned long long)) != cudaSuccess) {
    sy_destroy(e);
    return fail(SY_ERR_CUDA, "cudaMalloc of the per-env flag / statistics buffers failed");
  }
  if (cudaStreamCreateWithFlags(&e->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_logic, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_copied, cudaEventDisableTiming) != cudaSuccess) {
    sy_destroy(e);
    return fail(SY_ERR_CUDA, "stream / event creation failed");
  }
  *out_env = e;
  return SY_OK;
}

void sy_destroy(SyEnv* e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  free_graph_tables(e);
  if (e->d_exp) cudaFree(e->d_exp);
  if (e->d_cov) cudaFree(e->d_cov);
  if (e->d_bel_flags) cudaFree(e->d_bel_flags);
  if (e->d_stats_rep) cudaFree(e->d_stats_rep);
  for (void* ptr : {e->d_grp, e->d_grp_id, e->d_grp_id_new, e->d_grp_bad, e->d_grp_stats})
    if (ptr) cudaFree(ptr);
  if (e->aux_stream) cudaStreamDestroy(e->aux_stream);
  if (e->split_stream) cudaStreamDestroy(e->split_stream);
  for (cudaEvent_t ev : {e->ev_split_start, e->ev_split_logic, e->ev_split_belief})
    if (ev) cudaEventDestroy(ev);
  if (e->ev_main) cudaEventDestroy(e->ev_main);
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->ev_logic) cudaEventDestroy(e->ev_logic);
  if (e->ev_copied) cudaEventDestroy(e->ev_copied);
  delete e;
}

int sy_set_option(SyEnv* e, int32_t option, int32_t value) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  switch (option) {
    case SY_OPT_STEP_KERNEL:
      if (value != SY_STEP_FUSED && value != SY_STEP_TWO_KERNELS && value != SY_STEP_AUTO)
        return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_STEP_KERNEL: 0 (fused), 1 (two kernels) or 2 (auto)");
      e->opt_fused = value;
      return SY_OK;
    case SY_OPT_NF_FILL:
      if (value != 0 && value != 1) return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_NF_FILL: 0 or 1");
      e->opt_fill = value;
      return SY_OK;
    case SY_OPT_WRITER_PATH:
      if (value != SY_WRITER_BULK && value != SY_WRITER_LSU) return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_WRITER_PATH: 0 (bulk) or 1 (LSU)");
      e->opt_writer = value;
      return SY_OK;
    case SY_OPT_PDL:
      if (value != 0 && value != 1) return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_PDL: 0 or 1");
      e->opt_pdl = value;
      return SY_OK;
    case SY_OPT_ROLLOUT_KERNEL:
      if (value != 0 && value != 1) return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_ROLLOUT_KERNEL: 0 or 1");
      e->opt_rollout_kernel = value;
      return SY_OK;
    case SY_OPT_TAIL_SPLIT:
      if (value != 0 && value != 1) return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_TAIL_SPLIT: 0 or 1");
      e->opt_tail_split = value;
      return SY_OK;
    case SY_OPT_LAGGED_KERNEL:
      if (value != SY_LAGGED_OFF && value != SY_LAGGED_ON && value != SY_LAGGED_AUTO)
        return fail(SY_ERR_INVALID_ARGUMENT, "SY_OPT_LAGGED_KERNEL: 0 (off), 1 (on) or 2 (auto)");
      e->opt_lagged = value;
      return SY_OK;
    default:
      return fail(SY_ERR_INVALID_ARGUMENT, "unknown option %d", option);
  }
}

int sy_set_seed(SyEnv* e, uint64_t seed) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  e->cfg.seed = seed;
  return SY_OK;
}

int sy_set_reward_tables(SyEnv* e, const double* exp_neg_h, int32_t n_exp, const double* cov_h, int32_t n_cov, sy_stream_t stream) {
  if (!e || !exp_neg_h || !cov_h || n_exp < 1 || n_cov < 2) return fail(SY_ERR_INVALID_ARGUMENT, "bad reward tables");
  if (n_exp > DIST_INF) n_exp = DIST_INF;  // index 0xFFFF must read as exp(-inf) = 0
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  if (e->d_exp) cudaFree(e->d_exp);
  if (e->d_cov) cudaFree(e->d_cov);
  e->d_exp = e->d_cov = nullptr;
  CUDA_TRY(cudaMalloc(&e->d_exp, (size_t)n_exp * sizeof(double)));
  CUDA_TRY(cudaMalloc(&e->d_cov, (size_t)n_cov * sizeof(double)));
  CUDA_TRY(cudaMemcpyAsync(e->d_exp, exp_neg_h, (size_t)n_exp * sizeof(double), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(e->d_cov, cov_h, (size_t)n_cov * sizeof(double), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  e->tb.exp_neg = (const double*)e->d_exp;
  e->tb.coverage = (const double*)e->d_cov;
  e->tb.n_exp = n_exp;
  e->tb.n_cov = n_cov;
  e->tables_set = true;
  return SY_OK;
}

int sy_load_graphs(SyEnv* e, int32_t G, const int32_t* row_ptr, const int32_t* col, const int32_t* w, int32_t nnz_stride, sy_stream_t stream) {
  if (G > 65535) return fail(SY_ERR_INVALID_ARGUMENT, "at most 65535 graphs in the pool");
  if (!e || G <= 0 || !row_ptr || !col || !w || nnz_stride <= 0) return fail(SY_ERR_INVALID_ARGUMENT, "bad graph arguments");
  const int N = e->cfg.num_nodes;
  // validate + narrow on the host (setup path)
  std::vector<uint16_t> col16((size_t)G * nnz_stride, 0);
  std::vector<uint8_t> w8((size_t)G * nnz_stride, 0);
  const int pack_stride = ((nnz_stride + 3 * N + 3) & ~3) + 4;  // every list padded to a multiple of 4 entries
  std::vector<int2> pack((size_t)G * pack_stride, make_int2(0, 0));
  std::vector<int32_t> pack_ptr((size_t)G * (N + 1), 0);
  int wcap = 1;
  for (int g = 0; g < G; ++g) {
    const int32_t* rp = row_ptr + (size_t)g * (N + 1);
    if (rp[0] != 0) return fail(SY_ERR_INVALID_ARGUMENT, "graph %d: row_ptr[0] != 0", g);
    for (int u = 0; u < N; ++u) {
      if (rp[u + 1] < rp[u] || rp[u + 1] > nnz_stride) return fail(SY_ERR_INVALID_ARGUMENT, "graph %d: bad row_ptr at node %d", g, u);
      if (rp[u + 1] - rp[u] > 255) return fail(SY_ERR_INVALID_ARGUMENT, "graph %d: node %d has more than 255 neighbours", g, u);
      pack_ptr[(size_t)g * (N + 1) + u + 1] = pack_ptr[(size_t)g * (N + 1) + u] + ((rp[u + 1] - rp[u] + 3) & ~3);
      for (int k = rp[u]; k < rp[u + 1]; ++k) {
        const int v = col[(size_t)g * nnz_stride + k], wt = w[(size_t)g * nnz_stride + k];
        if (v < 0 || v >= N || v == u) return fail(SY_ERR_INVALID_ARGUMENT, "graph %d: bad neighbour %d of node %d", g, v, u);
        if (k > rp[u] && v <= col[(size_t)g * nnz_stride + k - 1]) return fail(SY_ERR_INVALID_ARGUMENT, "graph %d: neighbours of node %d not strictly ascending", g, u);
        if (wt < 1 || wt > 255) return fail(SY_ERR_INVALID_ARGUMENT, "graph %d: edge weight %d outside 1..255", g, wt);
        col16[(size_t)g * nnz_stride + k] = (uint16_t)v;
        w8[(size_t)g * nnz_stride + k] = (uint8_t)wt;
        const float inv_deg_v = 1.0f / (float)(rp[v + 1] - rp[v]);  // v has at least the edge back to u
        int bits;
        std::memcpy(&bits, &inv_deg_v, sizeof(bits));
        pack[(size_t)g * pack_stride + pack_ptr[(size_t)g * (N + 1) + u] + (k - rp[u])] = make_int2(v * BSTRIDE * (int)sizeof(float), bits);
        if (wt > wcap) wcap = wt;
      }
    }
  }
  if ((long long)wcap * (N - 1) >= DIST_INF) return fail(SY_ERR_INVALID_ARGUMENT, "max path length does not fit u16");
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  e->graphs_loaded = false;
  e->gen_max_edges = 0;
  if (int rc = alloc_graph_tables(e, G, nnz_stride, wcap, pack_stride)) return rc;
  CUDA_TRY(cudaMemcpyAsync(e->d_pack, pack.data(), pack.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(e->d_pack_ptr, pack_ptr.data(), pack_ptr.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(e->d_row_ptr, row_ptr, (size_t)G * (N + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(e->d_col, col16.data(), col16.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaMemcpyAsync(e->d_wgt, w8.data(), w8.size(), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));  // the staging vectors die at return
  return finish_graph_tables(e, G, nnz_stride, wcap, pack_stride, s);
}

}  // extern "C"

namespace {
// everything derived from the CSR (dense weights, move counts, 1/deg, all-pairs distances) + the kernels' smem plans
int finish_graph_tables(SyEnv* e, int G, int nnz_stride, int wcap, int pack_stride, cudaStream_t s) {
  const int N = e->cfg.num_nodes;
  const int Ns = (N + 15) & ~15;
  sy_build_rows_kernel<<<dim3(N, G), 64, 0, s>>>(N, Ns, nnz_stride, wcap, (const int32_t*)e->d_row_ptr, (const uint16_t*)e->d_col,
                                                 (const uint8_t*)e->d_wgt, (uint8_t*)e->d_W, (uint8_t*)e->d_cnt, (float*)e->d_inv_deg);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  int wpb = (int)((96 * 1024) / ((size_t)N * sizeof(int)));
  if (wpb < 1) wpb = 1;
  if (wpb > 8) wpb = 8;
  const size_t smem = (size_t)wpb * N * sizeof(int);
  if (smem > 200 * 1024) return fail(SY_ERR_INVALID_ARGUMENT, "num_nodes too large for the APSP kernel");
  if (smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(sy_apsp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long nwarps = (long long)G * N;
  const unsigned nblocks = (unsigned)((nwarps + wpb - 1) / wpb);
  sy_apsp_kernel<<<nblocks, wpb * 32, smem, s>>>(G, N, nnz_stride, (const int32_t*)e->d_row_ptr, (const uint16_t*)e->d_col,
                                                 (const uint8_t*)e->d_wgt, (uint16_t*)e->d_D, wpb);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  e->tb.W = (const uint8_t*)e->d_W;
  e->tb.D = (const uint16_t*)e->d_D;
  e->tb.row_ptr = (const int32_t*)e->d_row_ptr;
  e->tb.col = (const uint16_t*)e->d_col;
  e->tb.wgt = (const uint8_t*)e->d_wgt;
  e->tb.cnt = (const uint8_t*)e->d_cnt;
  e->tb.inv_deg = (const float*)e->d_inv_deg;
  e->tb.nbr_pack = (const int2*)e->d_pack;
  e->tb.pack_ptr = (const int32_t*)e->d_pack_ptr;
  e->tb.pack_stride = pack_stride;
  {
    int* scratch = nullptr;
    CUDA_TRY(cudaMalloc(&scratch, (size_t)G * 257 * sizeof(int)));
    sy_degree_perm_kernel<<<G, 32, 0, s>>>(N, (const int32_t*)e->d_row_ptr, (uint16_t*)e->d_deg_perm, scratch);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s));
    cudaFree(scratch);
    e->tb.deg_perm = (const uint16_t*)e->d_deg_perm;
  }
  // dynamic shared memory of the observe kernel's belief warps (generic: BEL_WARPS x N floats; fast path: two
  // transposed tiles [N][BSTRIDE] + per-warp partial sums)
  e->bel_smem = 0;
  e->bel_fast = 0;
  if (e->cfg.belief) {
    size_t generic = (size_t)BEL_WARPS * (N + 1) * sizeof(float);
    auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
    const size_t off_out = up16((size_t)N * BSTRIDE * sizeof(float));
    const size_t off_part = up16(2 * off_out);
    const size_t off_pack = up16(off_part + (size_t)BEL_WARPS * 32 * sizeof(float));
    const size_t off_ptr = up16(off_pack + (size_t)pack_stride * sizeof(int2));
    const size_t fast = off_ptr + (size_t)(N + 2) * sizeof(int);
    if (fast <= 110 * 1024 && N <= BEL_WARPS * BEL_JMAX) {
      e->bel_fast = 1;  // N <= ~400 (2 CTAs per SM); N <= ~250 keeps 3 CTAs per SM
      e->bel_off_out = (int)off_out;
      e->bel_off_part = (int)off_part;
      e->bel_off_pack = (int)off_pack;
      e->bel_off_ptr = (int)off_ptr;
    }
    e->bel_warps = BEL_WARPS;
    e->wr_warps = WR_WARPS;
    if (!e->bel_fast && THREADS / 32 > GEN_BEL_WARPS) {  // the generic path is the critical role: give it more warps
      e->bel_warps = GEN_BEL_WARPS;
      e->wr_warps = GEN_WR_WARPS;
      generic = (size_t)e->bel_warps * (N + 1) * sizeof(float);
    }
    e->bel_smem = e->bel_fast && fast > generic ? fast : generic;
    if (e->bel_smem > 180 * 1024) return fail(SY_ERR_INVALID_ARGUMENT, "num_nodes too large for the belief kernel's shared memory");
  }
  {  // writer staging area: pos, money [TILE, A], revealed, graph id [TILE], per-warp flat one-hot indices and
     // action_mask images, then (optionally) the graph's CSR
    // mask image of a writer warp: a whole env (A rows) or, for large rows, ONE row at a time -- the shared memory that
    // saves pays for the padded neighbour lists of the large-N belief path
    e->wr_img_rows = (size_t)e->A * N > 4096 ? 1 : e->A;
    const size_t img_stride = (((size_t)e->wr_img_rows * N + 16) + 15) & ~(size_t)15;
    const size_t base_lsu = ((size_t)2 * TILE * e->A + 2 * TILE + e->wr_warps * SY_MAX_AGENTS) * sizeof(int) + e->wr_warps * img_stride;
    // bulk writers: one zero page + two chunk images for each of the (at most BULK_WARPS) streaming warps
    const int nbw = std::min(e->wr_warps, BULK_WARPS);
    const int cap = std::max(256, (int)(SY_BULK_IMG_BUDGET / (2 * nbw + 1)));
    e->wr_c_mask = plan_bulk_chunk((size_t)e->A * N, cap, nbw);
    e->wr_c_nf32 = e->wr_c_nf8 = e->wr_c_mask;  // the uint8 node_features stream has the mask's geometry
    e->wr_img_bytes = e->wr_c_mask;
    const size_t base_bulk = ((size_t)2 * TILE * e->A + 2 * TILE) * sizeof(int) + (size_t)(2 * nbw + 1) * e->wr_img_bytes;
    const size_t base = std::max(base_lsu, base_bulk);  // either writer path can be selected at run time
    // generic (large-N) belief path: it gathers over the same staged CSR, plus the 1/deg row, instead of walking the
    // neighbour lists in global memory (at N = 1000 they no longer fit the L1 left over by the shared-memory carve-out)
    const bool share = e->cfg.belief && !e->bel_fast;
    const size_t csr_core = ((((size_t)(N + 1) * sizeof(int) + (size_t)nnz_stride * 3) + 3) & ~(size_t)3) + (share ? (size_t)N * (sizeof(float) + sizeof(uint16_t)) : 0);
    e->wr_off_pad = (int)((csr_core + 15) & ~(size_t)15);
    const size_t csr = (share ? (size_t)e->wr_off_pad + ((size_t)((N + 1 + 3) & ~3) + pack_stride) * sizeof(uint16_t) : csr_core) + 16;
    e->wr_off = (int)((e->bel_smem + 15) & ~(size_t)15);
    e->wr_img_stride = (int)img_stride;
    e->wr_off_csr = (int)(((size_t)e->wr_off + base + 15) & ~(size_t)15);
    e->wr_stage_csr = (csr <= 48 * 1024 && pack_stride < 65536 && (size_t)e->wr_off_csr + csr <= 200 * 1024) ? 1 : 0;
    e->bel_share_csr = (share && e->wr_stage_csr) ? 1 : 0;
    e->obs_smem = (size_t)e->wr_off_csr + (e->wr_stage_csr ? csr : 0);
    if (e->obs_smem > 220 * 1024) return fail(SY_ERR_INVALID_ARGUMENT, "num_nodes x agents too large for the observe kernel's shared memory");
    if (int rc = raise_observe_smem_limit(e->cfg.device, e->obs_smem)) return rc;
    int per_sm = 0, sms = 0;
    const bool gen = e->bel_warps == GEN_BEL_WARPS && GEN_BEL_WARPS != BEL_WARPS;
    cudaError_t oe = gen ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sy_observe_kernel<GEN_BEL_WARPS, GEN_WR_WARPS>, THREADS, e->obs_smem)
                         : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sy_observe_kernel<BEL_WARPS, WR_WARPS>, THREADS, e->obs_smem);
    if (oe != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device) != cudaSuccess) {
      cudaGetLastError();
      per_sm = 0;
    }
    e->obs_slots = per_sm * sms;
  }
  e->tb.G = G;
  e->tb.Ns = Ns;
  e->tb.nnz_stride = nnz_stride;
  e->tb.wcap = wcap;
  if (int rc = plan_fused(e, nnz_stride)) return rc;
  if (int rc = plan_lagged(e)) return rc;
  e->graphs_loaded = true;
  return SY_OK;
}
}  // namespace

extern "C" {

// Replaces ConnectedGraph.sample (graph_layout.py:9-80) + the resample loop of yard.py:67-101 for a whole pool, on the
// device.  Slot g of this handle is global graph `graph_offset + g`; global graph 0 of the generation fixes the edge
// count (it is sampled first, as a probe, into slot 0).
int sy_generate_graphs(SyEnv* e, int32_t G, int32_t num_edges, int32_t max_edges_per_node, int32_t max_weight, uint64_t seed,
                       uint32_t generation, uint32_t graph_offset, int32_t* attempts_host, sy_stream_t stream) {
  if (!e || G <= 0 || G > 65535) return fail(SY_ERR_INVALID_ARGUMENT, "1..65535 graphs in the pool");
  const int N = e->cfg.num_nodes;
  if (N > GEN_MAX_NODES) return fail(SY_ERR_INVALID_ARGUMENT, "device graph sampler: at most %d nodes", GEN_MAX_NODES);
  if (max_edges_per_node < 1 || max_weight < 2 || max_weight > 256) return fail(SY_ERR_INVALID_ARGUMENT, "bad degree cap / max_weight");
  if (generation >= (1u << 25)) return fail(SY_ERR_INVALID_ARGUMENT, "generation must be below 2^25");
  if ((long long)(max_weight - 1) * (N - 1) >= DIST_INF) return fail(SY_ERR_INVALID_ARGUMENT, "max path length does not fit u16");
  const long long all_pairs = (long long)N * (N - 1) / 2;
  if (num_edges < N - 1) num_edges = N - 1;  // graph_layout.py:20-21: the tree is the minimum
  if (num_edges > all_pairs) num_edges = (int32_t)all_pairs;
  const int max_edges = num_edges, nnz_stride = 2 * max_edges > 0 ? 2 * max_edges : 1, wcap = max_weight - 1;
  const int pack_stride = ((nnz_stride + 3 * N + 3) & ~3) + 4;
  const int Ns = (N + 15) & ~15;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  e->graphs_loaded = false;
  if (int rc = alloc_graph_tables(e, G, nnz_stride, wcap, pack_stride)) return rc;
  if (!e->d_edges || e->gen_max_edges != max_edges) {
    for (void** ptr : {&e->d_edges, &e->d_edge_w, &e->d_edge_count, &e->d_gen_status, &e->d_gen_want}) {
      if (*ptr) cudaFree(*ptr);
      *ptr = nullptr;
    }
    CUDA_TRY(cudaMalloc(&e->d_edges, (size_t)G * max_edges * sizeof(ushort2)));
    CUDA_TRY(cudaMalloc(&e->d_edge_w, (size_t)G * max_edges));
    CUDA_TRY(cudaMalloc(&e->d_edge_count, (size_t)G * sizeof(int)));
    CUDA_TRY(cudaMalloc(&e->d_gen_status, (size_t)G * sizeof(int)));
    CUDA_TRY(cudaMalloc(&e->d_gen_want, sizeof(int)));
  }
  e->gen_max_edges = max_edges;
  CUDA_TRY(cudaMemsetAsync(e->d_col, 0, (size_t)G * nnz_stride * sizeof(uint16_t), s));
  CUDA_TRY(cudaMemsetAsync(e->d_wgt, 0, (size_t)G * nnz_stride, s));
  GenParams q{};
  q.N = N;
  q.Ns = Ns;
  q.max_edges = max_edges;
  q.num_edges = num_edges;
  q.cap = max_edges_per_node;
  q.wrange = max_weight - 1;
  q.seed_lo = (unsigned)(seed & 0xFFFFFFFFu);
  q.seed_hi = (unsigned)(seed >> 32);
  q.generation = generation;
  q.graph_offset = graph_offset;
  q.want = (int*)e->d_gen_want;
  q.W = (uint8_t*)e->d_W;
  q.edges = (ushort2*)e->d_edges;
  q.edge_w = (uint8_t*)e->d_edge_w;
  q.edge_count = (int*)e->d_edge_count;
  q.status = (int*)e->d_gen_status;
  const size_t gen_smem = (size_t)N * (sizeof(int) + 3 * sizeof(uint16_t));
  if (gen_smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(sy_sample_graphs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gen_smem));
  q.probe = 1;
  sy_sample_graphs_kernel<<<1, 32, gen_smem, s>>>(q);
  q.probe = 0;
  sy_sample_graphs_kernel<<<G, 32, gen_smem, s>>>(q);
  g_launches += 2;
  CUDA_TRY(cudaGetLastError());
  const size_t csr_smem = (size_t)(3 * N + 2) * sizeof(int);
  if (csr_smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(sy_csr_from_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)csr_smem));
  sy_csr_from_dense_kernel<<<G, 256, csr_smem, s>>>(N, Ns, nnz_stride, pack_stride, (const uint8_t*)e->d_W, (int32_t*)e->d_row_ptr,
                                                    (uint16_t*)e->d_col, (uint8_t*)e->d_wgt, (int2*)e->d_pack, (int32_t*)e->d_pack_ptr,
                                                    (int*)e->d_gen_status);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  std::vector<int> status((size_t)G);
  int want = 0;
  CUDA_TRY(cudaMemcpyAsync(status.data(), e->d_gen_status, (size_t)G * sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaMemcpyAsync(&want, e->d_gen_want, sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  for (int g = 0; g < G; ++g) {
    if (attempts_host) attempts_host[g] = status[g];
    if (status[g] == -1)  // the reference's RuntimeError, yard.py:96-101
      return fail(SY_ERR_STATE, "Failed to generate graph with %d edges after %d attempts (pool slot %d).", want, GEN_MAX_ATTEMPTS, g);
    if (status[g] < 0) return fail(SY_ERR_STATE, "device graph sampler failed for pool slot %d (status %d)", g, status[g]);
  }
  return finish_graph_tables(e, G, nnz_stride, wcap, pack_stride, s);
}

// edge lists of a device-sampled pool in the reference's order (tree edges, then the extras): what GraphInstance
// holds as edge_links / edges (graph_layout.py:53).  HOST buffers: edge_links int32 [G, max_edges, 2], weights
// int32 [G, max_edges], counts int32 [G]; rows are valid up to counts[g].
int sy_read_graph_edges(SyEnv* e, int32_t* edge_links, int32_t* weights, int32_t* counts, int32_t max_edges, sy_stream_t stream) {
  if (!e || !e->graphs_loaded || e->gen_max_edges <= 0) return fail(SY_ERR_STATE, "the pool was not sampled on the device");
  if (!edge_links || !weights || !counts || max_edges < e->gen_max_edges) return fail(SY_ERR_INVALID_ARGUMENT, "bad edge buffers (need max_edges >= %d)", e->gen_max_edges);
  const int G = e->tb.G, M = e->gen_max_edges;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  std::vector<ushort2> ed((size_t)G * M);
  std::vector<uint8_t> ew((size_t)G * M);
  CUDA_TRY(cudaMemcpyAsync(ed.data(), e->d_edges, ed.size() * sizeof(ushort2), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaMemcpyAsync(ew.data(), e->d_edge_w, ew.size(), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaMemcpyAsync(counts, e->d_edge_count, (size_t)G * sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  for (int g = 0; g < G; ++g)
    for (int k = 0; k < max_edges; ++k) {
      const bool live = k < M && k < counts[g];
      edge_links[((size_t)g * max_edges + k) * 2] = live ? ed[(size_t)g * M + k].x : 0;
      edge_links[((size_t)g * max_edges + k) * 2 + 1] = live ? ed[(size_t)g * M + k].y : 0;
      weights[(size_t)g * max_edges + k] = live ? ew[(size_t)g * M + k] : 0;
    }
  return SY_OK;
}

int sy_read_graph_tables(SyEnv* e, int32_t g, uint8_t* weights, uint16_t* apsp, sy_stream_t stream) {
  if (!e || !e->graphs_loaded) return fail(SY_ERR_STATE, "graphs not loaded");
  if (g < 0 || g >= e->tb.G) return fail(SY_ERR_INVALID_ARGUMENT, "graph index out of range");
  const int N = e->cfg.num_nodes;
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  if (weights)
    CUDA_TRY(cudaMemcpy2DAsync(weights, N, e->tb.W + (size_t)g * N * e->tb.Ns, e->tb.Ns, N, N, cudaMemcpyDeviceToHost, s));
  if (apsp) CUDA_TRY(cudaMemcpyAsync(apsp, e->tb.D + (size_t)g * N * N, (size_t)N * N * sizeof(uint16_t), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  return SY_OK;
}

int sy_reset(SyEnv* e, const uint8_t* reset_mask, const int32_t* init_pos, const int32_t* init_gid, int32_t restart,
             const SyState* st, const SyObs* ob, sy_stream_t stream) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  e->aux_after_logic = false;
  Params p;
  int rc = fill_params(e, st, ob, nullptr, p);
  if (rc) return rc;
  if ((rc = check_obs(ob))) return rc;
  p.reset_mask = reset_mask;
  p.init_pos = init_pos;
  p.init_gid = init_gid;
  p.restart = restart;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  if (e->obs_pending) {  // deferred observations (belief propagation of the last step) first: a partial reset keeps the other envs
    Params pf = p;
    pf.out.stats = e->pending_stats;
    launch_observe(e, pf, (unsigned)((p.B + TILE - 1) / TILE), s);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    e->obs_pending = false;
  }
  const unsigned rgrid = (unsigned)((p.B + LOGIC_THREADS - 1) / LOGIC_THREADS);
  if (p.grp_n) sy_reset_kernel<1><<<rgrid, LOGIC_THREADS, 0, s>>>(p);
  else sy_reset_kernel<<<rgrid, LOGIC_THREADS, 0, s>>>(p);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  if (e->grp_need_reset && reset_mask) {  // does the mask cover every env?  (once after sy_set_groups: one synchronise)
    int unset = 0;
    CUDA_TRY(cudaMemsetAsync(e->d_grp_bad, 0, sizeof(int), s));
    sy_count_unset_kernel<<<(unsigned)((p.B + 255) / 256), 256, 0, s>>>(reset_mask, p.B, (int*)e->d_grp_bad);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(&unset, e->d_grp_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (unset == 0) e->grp_need_reset = false;
  }
  if (!reset_mask) e->grp_need_reset = false;  // every env starts an episode under its (new) group
  launch_observe(e, p, (unsigned)((p.B + TILE - 1) / TILE), s);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

}  // extern "C"

namespace {
// after_logic (optional): recorded between the two kernels -- rewards / flags are final once the logic kernel is done
bool fused_eligible(const SyEnv* e, const SyObs* ob) {
  if (!e->fused_ok || e->opt_fused == SY_STEP_TWO_KERNELS || !ob) return false;
  if (e->opt_fused == SY_STEP_AUTO && (e->cfg.num_envs + TILE - 1) / TILE > e->f_grid) return false;  // more than one wave of tiles
  const uintptr_t bits = reinterpret_cast<uintptr_t>(ob->action_mask) | reinterpret_cast<uintptr_t>(ob->node_features_u8 ? (void*)ob->node_features_u8 : (void*)ob->node_features);
  return (bits & 15u) == 0;  // bulk stores need 16-byte aligned streams
}

// next_actions (+ counter): a fused launch also draws the next step's random actions; *fused_sampled reports whether it did
void launch_logic(const SyEnv* e, const Params& p, unsigned grid, cudaStream_t ls) {
  const bool f64 = e->cfg.reward_mode == SY_REWARD_FP64, pdl = e->opt_pdl != 0;
  if (p.grp_n) {  // mechanism groups
    if (p.A <= 4) launch_ex(f64 ? sy_logic_kernel<SY_REWARD_FP64, 4, 1> : sy_logic_kernel<SY_REWARD_FP32, 4, 1>, grid, LOGIC_THREADS, 0, ls, pdl, p);
    else if (p.A <= 8) launch_ex(f64 ? sy_logic_kernel<SY_REWARD_FP64, 8, 1> : sy_logic_kernel<SY_REWARD_FP32, 8, 1>, grid, LOGIC_THREADS, 0, ls, pdl, p);
    else launch_ex(f64 ? sy_logic_kernel<SY_REWARD_FP64, 16, 1> : sy_logic_kernel<SY_REWARD_FP32, 16, 1>, grid, LOGIC_THREADS, 0, ls, pdl, p);
    return;
  }
  if (p.A <= 4) {
    if (f64) launch_ex(sy_logic_kernel<SY_REWARD_FP64, 4>, grid, LOGIC_THREADS, 0, ls, pdl, p);
    else launch_ex(sy_logic_kernel<SY_REWARD_FP32, 4>, grid, LOGIC_THREADS, 0, ls, pdl, p);
  } else if (p.A <= 8) {
    if (f64) launch_ex(sy_logic_kernel<SY_REWARD_FP64, 8>, grid, LOGIC_THREADS, 0, ls, pdl, p);
    else launch_ex(sy_logic_kernel<SY_REWARD_FP32, 8>, grid, LOGIC_THREADS, 0, ls, pdl, p);
  } else {
    if (f64) launch_ex(sy_logic_kernel<SY_REWARD_FP64, 16>, grid, LOGIC_THREADS, 0, ls, pdl, p);
    else launch_ex(sy_logic_kernel<SY_REWARD_FP32, 16>, grid, LOGIC_THREADS, 0, ls, pdl, p);
  }
}

// the lagged kernel carries pending observations: always (option on), or when the batch is one wave of it (auto)
bool use_lagged(const SyEnv* e) {
  if (!e->lag_ok || e->opt_lagged == SY_LAGGED_OFF) return false;
  if (e->opt_lagged == SY_LAGGED_ON) return true;
  return (e->cfg.num_envs + TILE - 1) / TILE <= e->lag_slots;
}

// defer: leave the dense observations of the new state pending (sy_step_deferred); the next call writes them
int step_impl(SyEnv* e, const int64_t* actions, const int32_t* actions32, const SyState* st, const SyObs* ob, const SyOut* out,
              sy_stream_t stream, cudaEvent_t after_logic = nullptr, const int16_t* actions16 = nullptr,
              int64_t* next_actions = nullptr, uint32_t next_counter = 0, const uint32_t* next_counter_base = nullptr,
              bool* fused_sampled = nullptr, bool defer = false) {
  if (!e || (!actions && !actions32 && !actions16)) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions");
  if (actions16 && e->cfg.num_nodes > 32767) return fail(SY_ERR_INVALID_ARGUMENT, "int16 actions need num_nodes <= 32767");
  e->aux_after_logic = false;
  if (e->grp_need_reset) return fail(SY_ERR_STATE, "mechanism groups changed: a sy_reset of every env (NULL or all-set mask) must come before the next step");
  if (!out) return fail(SY_ERR_INVALID_ARGUMENT, "SyOut is NULL");
  if (out->struct_bytes != sizeof(SyOut)) return fail(SY_ERR_INVALID_ARGUMENT, "SyOut size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)out->struct_bytes, sizeof(SyOut), SY_ABI_VERSION);
  if (!out->reward || !out->terminated || !out->truncated || !out->done || !out->winner)
    return fail(SY_ERR_INVALID_ARGUMENT, "SyOut has NULL members");
  Params p;
  int rc = fill_params(e, st, ob, out, p);
  if (rc) return rc;
  if ((rc = check_obs(ob))) return rc;
  p.actions = reinterpret_cast<const long long*>(actions);
  p.actions32 = actions32;
  p.actions16 = actions16;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned grid = (unsigned)((p.B + TILE - 1) / TILE);
  // Two plain launches.  Measured alternatives that did NOT pay on B200: issuing the step in chunks on two streams or a
  // persistent observe grid (the block scheduler drains the older grid first: no overlap), and one persistent kernel
  // whose logic warps run one tile ahead of the observe warps (the logic's loads and shared-memory accesses queue
  // behind the writers' store stream in the SM's in-order LSU: the times added up, 159 vs 136 us).
  // A persistent single-launch kernel that dedicates every k-th SM to the logic (SM roles elected at run time, tiles
  // handed over through epoch flags) was correct but slower for every k (159 us at k = 4, 241 us at k = 8): both kernels
  // are bound by SM issue/latency throughput as much as by HBM, so taking SMs away from either one loses more than the
  // overlap gains.
  // Also measured: an L2 persisting access-policy window on the belief map (52 MB at c3) slowed the step to 166-255 us
  // (the carve-out starves the write stream of L2), so no residency hints are set.
  if (defer || e->obs_pending) {
    // Software-pipelined step.  Pending observations (of the state BEFORE this step) and this step's dynamics are
    // independent pieces of work on the same tiles: one launch carries both (sy_step_lagged_kernel), the dynamics in the
    // shadow of the observation stream.  Without pending observations (first deferred step) the dynamics run alone;
    // a plain call (defer == false) then brings the observations up to date with the stand-alone kernel.
    p.next_actions = reinterpret_cast<long long*>(next_actions);
    p.next_counter = next_counter;
    p.next_counter_base = next_counter_base;
    if (e->obs_pending && use_lagged(e) && !p.wr_bulk && !p.dbg_skip) {
      lagged_fn(e, p.grp_n > 0)<<<grid, lagged_threads(e), e->obs_smem, s>>>(p);
    } else {
      if (e->obs_pending) {
        launch_observe(e, p, grid, s);
        g_launches++;
        CUDA_TRY(cudaGetLastError());
      }
      launch_logic(e, p, grid, s);
    }
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    e->obs_pending = true;
    e->pending_stats = p.out.stats;  // the observation kernel that follows scores the belief at reveals iff this step collected statistics
    if (after_logic) CUDA_TRY(cudaEventRecord(after_logic, s));
    if (fused_sampled) *fused_sampled = next_actions != nullptr;
    if (!defer) {
      launch_observe(e, p, grid, s);
      g_launches++;
      CUDA_TRY(cudaGetLastError());
      e->obs_pending = false;
    }
    return SY_OK;
  }
  if (fused_eligible(e, ob) && !p.dbg_skip) {
    // ONE persistent launch: dynamics, belief and the bulk-store observation stream of all tiles, software-pipelined
    p.next_actions = reinterpret_cast<long long*>(next_actions);
    p.next_counter = next_counter;
    p.next_counter_base = next_counter_base;
    p.bel_share_csr = 0;
    p.wr_bulk = 1;
    p.wr_c_mask = p.wr_c_nf = e->f_c_mask;
    p.wr_img_bytes = e->f_img_bytes;
    p.wr_stage_csr = e->f_stage_csr;
    p.wr_off_csr = e->f_off_csr;
    p.f_off_sbuf = e->f_off_sbuf;
    p.f_sbuf_stride = e->f_sbuf_stride;
    p.f_off_zero = e->f_off_zero;
    p.f_off_imgs = e->f_off_imgs;
    p.f_off_nbr4 = e->f_off_nbr4;
    p.wr_epc = e->f_epc;
    const int threads = (e->f_bw + FUSED_WR + LOGIC_WARPS) * 32;
    fused_fn(e->f_bw, e->cfg.reward_mode, p.A, p.grp_n > 0)<<<(unsigned)e->f_grid, threads, e->f_smem, s>>>(p);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    if (after_logic) CUDA_TRY(cudaEventRecord(after_logic, s));
    if (fused_sampled) *fused_sampled = true;
    return SY_OK;
  }
  // Split step: the state-independent zero fill of float32 node_features (63 % of the bytes) goes to the TMA engine in
  // its own tiny kernel on the caller's stream while the dynamics kernel runs on the handle's split stream; afterwards
  // the belief propagation (split stream) and the writers of the ones (caller's stream) run next to each other.  Both
  // join on the caller's stream before step_impl returns (events; capturable in a CUDA graph as a DAG).
  const bool split = e->opt_fill && !ob->node_features_u8 && !p.wr_bulk && (reinterpret_cast<uintptr_t>(ob->node_features) & 15u) == 0 &&
                     !p.dbg_skip && !e->bel_share_csr && e->cfg.num_envs >= SPLIT_MIN_ENVS && !e->grp_n;
  cudaStream_t ls = s;  // stream of the dynamics kernel
  if (split) {
    if (!e->split_stream) {
      CUDA_TRY(cudaStreamCreateWithFlags(&e->split_stream, cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&e->ev_split_start, cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&e->ev_split_logic, cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&e->ev_split_belief, cudaEventDisableTiming));
      int sms = 0;
      CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
      e->fill_grid = sms;
    }
    CUDA_TRY(cudaEventRecord(e->ev_split_start, s));
    CUDA_TRY(cudaStreamWaitEvent(e->split_stream, e->ev_split_start, 0));
    sy_fill_kernel<<<(unsigned)e->fill_grid, FILL_THREADS, 0, s>>>(reinterpret_cast<uint8_t*>(ob->node_features),
                                                                  (size_t)p.B * p.N * p.A * sizeof(float));
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    p.nf_prefilled = 1;
    ls = e->split_stream;
  }
  if (!(p.dbg_skip & 32)) launch_logic(e, p, grid, ls);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  if (after_logic) CUDA_TRY(cudaEventRecord(after_logic, ls));
  if (split) {
    CUDA_TRY(cudaEventRecord(e->ev_split_logic, ls));
    if (p.belief_on) {  // belief propagation: one role per launch, next to the writers
      sy_observe_kernel<BEL_WARPS, 0><<<grid, BEL_WARPS * 32, e->bel_smem, ls>>>(p);
      g_launches++;
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaEventRecord(e->ev_split_belief, ls));
    }
    CUDA_TRY(cudaStreamWaitEvent(s, e->ev_split_logic, 0));
    Params pw = p;  // writers only: their staging area starts at the beginning of the dynamic shared memory
    pw.wr_off = 0;
    pw.wr_off_csr = e->wr_off_csr - e->wr_off;
    sy_observe_kernel<0, WR_WARPS, WV_ONES><<<grid, WR_WARPS * 32, e->obs_smem - (size_t)e->wr_off, s>>>(pw);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    if (p.belief_on) CUDA_TRY(cudaStreamWaitEvent(s, e->ev_split_belief, 0));
    return SY_OK;
  }
  if (!(p.dbg_skip & 16)) launch_observe(e, p, grid, s);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

// D2H of the step results, overlapped with the observe kernel: the rewards / flags are final after the logic kernel, so
// they are copied on the handle's auxiliary stream while the (much longer) observation stream still runs on the
// caller's stream; both are joined before returning.  Members that are adjacent in both device and host memory (the
// host mirror allocates each side as one block) are merged into a single copy.
int copy_results_and_sync(SyEnv* e, const SyOut* out, const SyHostOut* ho, cudaStream_t s) {
  const size_t n = (size_t)e->cfg.num_envs * e->A;
  struct Seg { char* dst; const char* src; size_t bytes; };
  Seg segs[6] = {};
  int m = 0;
  auto add = [&](void* dst, const void* src, size_t bytes) {
    if (!dst) return;
    if (m > 0 && segs[m - 1].dst + segs[m - 1].bytes == (char*)dst && segs[m - 1].src + segs[m - 1].bytes == (const char*)src)
      segs[m - 1].bytes += bytes;
    else
      segs[m++] = Seg{(char*)dst, (const char*)src, bytes};
  };
  add(ho->reward, out->reward, n * sizeof(float));
  add(ho->terminated, out->terminated, n);
  add(ho->truncated, out->truncated, n);
  add(ho->done, out->done, n);
  add(ho->winner, out->winner, (size_t)e->cfg.num_envs);
  if (ho->status && !out->status) return fail(SY_ERR_INVALID_ARGUMENT, "SyHostOut.status needs SyOut.status");
  add(ho->status, out->status, (size_t)e->cfg.num_envs);
  CUDA_TRY(cudaStreamWaitEvent(e->aux_stream, e->ev_logic, 0));
  for (int i = 0; i < m; ++i) CUDA_TRY(cudaMemcpyAsync(segs[i].dst, segs[i].src, segs[i].bytes, cudaMemcpyDeviceToHost, e->aux_stream));
  CUDA_TRY(cudaEventRecord(e->ev_copied, e->aux_stream));
  CUDA_TRY(cudaStreamWaitEvent(s, e->ev_copied, 0));  // later work on the caller's stream is ordered after the copy
  if (e->host_overlap) {  // the results are on the host; the observe kernel keeps running on the caller's stream
    CUDA_TRY(cudaEventSynchronize(e->ev_copied));
    e->aux_after_logic = true;
  } else {
    CUDA_TRY(cudaStreamSynchronize(s));
  }
  return SY_OK;
}

template <typename ActT>
int sample_impl(SyEnv* e, const SyState* st, uint32_t step_counter, ActT* actions, sy_stream_t stream,
                const uint32_t* step_base = nullptr) {
  if (!e || !actions) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions");
  Params p;
  int rc = fill_params(e, st, nullptr, nullptr, p);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  const size_t n = (size_t)p.B * p.A;
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (p.grp_n) sy_sample_actions_kernel<ActT, 1><<<grid, 256, 0, (cudaStream_t)stream>>>(p, step_counter, actions, step_base);
  else sy_sample_actions_kernel<ActT><<<grid, 256, 0, (cudaStream_t)stream>>>(p, step_counter, actions, step_base);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}
}  // namespace

extern "C" {

int sy_step(SyEnv* e, const int64_t* actions, const SyState* st, const SyObs* ob, const SyOut* out, sy_stream_t stream) {
  return step_impl(e, actions, nullptr, st, ob, out, stream);
}

int sy_step_deferred(SyEnv* e, const int64_t* actions, const SyState* st, const SyObs* ob, const SyOut* out, sy_stream_t stream) {
  return step_impl(e, actions, nullptr, st, ob, out, stream, nullptr, nullptr, nullptr, 0, nullptr, nullptr, true);
}

int sy_flush_observations(SyEnv* e, const SyState* st, const SyObs* ob, sy_stream_t stream) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  if (!e->obs_pending) return SY_OK;
  Params p;
  int rc = fill_params(e, st, ob, nullptr, p);
  if (rc) return rc;
  if ((rc = check_obs(ob))) return rc;
  p.out.stats = e->pending_stats;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  launch_observe(e, p, (unsigned)((p.B + TILE - 1) / TILE), (cudaStream_t)stream);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  e->obs_pending = false;
  return SY_OK;
}

int sy_observations_pending(SyEnv* e) { return e && e->obs_pending ? 1 : 0; }

int sy_step_i32(SyEnv* e, const int32_t* actions, const SyState* st, const SyObs* ob, const SyOut* out, sy_stream_t stream) {
  return step_impl(e, nullptr, actions, st, ob, out, stream);
}

int sy_step_host(SyEnv* e, const int64_t* actions_host, int64_t* actions_dev, const SyState* st, const SyObs* ob,
                 const SyOut* out, const SyHostOut* ho, sy_stream_t stream) {
  if (!e || !actions_host || !actions_dev || !ho) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions / host_out");
  if (ho->struct_bytes != sizeof(SyHostOut)) return fail(SY_ERR_INVALID_ARGUMENT, "SyHostOut size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)ho->struct_bytes, sizeof(SyHostOut), SY_ABI_VERSION);
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)e->cfg.num_envs * e->A;
  CUDA_TRY(cudaMemcpyAsync(actions_dev, actions_host, n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
  const int rc = step_impl(e, actions_dev, nullptr, st, ob, out, stream, e->ev_logic);
  if (rc) return rc;
  return copy_results_and_sync(e, out, ho, s);
}

int sy_step_host_i32(SyEnv* e, const int32_t* actions_host, int32_t* actions_dev, const SyState* st, const SyObs* ob,
                     const SyOut* out, const SyHostOut* ho, sy_stream_t stream) {
  if (!e || !actions_host || !actions_dev || !ho) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions / host_out");
  if (ho->struct_bytes != sizeof(SyHostOut)) return fail(SY_ERR_INVALID_ARGUMENT, "SyHostOut size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)ho->struct_bytes, sizeof(SyHostOut), SY_ABI_VERSION);
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)e->cfg.num_envs * e->A;
  CUDA_TRY(cudaMemcpyAsync(actions_dev, actions_host, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  const int rc = step_impl(e, nullptr, actions_dev, st, ob, out, stream, e->ev_logic);
  if (rc) return rc;
  return copy_results_and_sync(e, out, ho, s);
}

int sy_step_i16(SyEnv* e, const int16_t* actions, const SyState* st, const SyObs* ob, const SyOut* out, sy_stream_t stream) {
  return step_impl(e, nullptr, nullptr, st, ob, out, stream, nullptr, actions);
}

int sy_step_host_i16(SyEnv* e, const int16_t* actions_host, int16_t* actions_dev, const SyState* st, const SyObs* ob,
                     const SyOut* out, const SyHostOut* ho, sy_stream_t stream) {
  if (!e || !actions_host || !actions_dev || !ho) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions / host_out");
  if (ho->struct_bytes != sizeof(SyHostOut)) return fail(SY_ERR_INVALID_ARGUMENT, "SyHostOut size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)ho->struct_bytes, sizeof(SyHostOut), SY_ABI_VERSION);
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)e->cfg.num_envs * e->A;
  CUDA_TRY(cudaMemcpyAsync(actions_dev, actions_host, n * sizeof(int16_t), cudaMemcpyHostToDevice, s));
  const int rc = step_impl(e, nullptr, nullptr, st, ob, out, stream, e->ev_logic, actions_dev);
  if (rc) return rc;
  return copy_results_and_sync(e, out, ho, s);
}

int sy_sample_actions_i16(SyEnv* e, const SyState* st, uint32_t step_counter, int16_t* actions, sy_stream_t stream) {
  if (e && e->cfg.num_nodes > 32767) return fail(SY_ERR_INVALID_ARGUMENT, "int16 actions need num_nodes <= 32767");
  return sample_impl<short>(e, st, step_counter, reinterpret_cast<short*>(actions), stream);
}

int sy_sample_actions_host(SyEnv* e, const SyState* st, uint32_t step_counter, void* actions_dev, void* actions_host,
                           int32_t bytes_per_action, sy_stream_t stream) {
  if (!e || !actions_dev || !actions_host) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions");
  // overlap mode: sample on the library stream, which sits right behind the last step's dynamics (the observe kernel of
  // that step only READS the state the sampler reads); otherwise, or when anything else touched the state since, in
  // order on the caller's stream
  cudaStream_t s = (cudaStream_t)stream;
  if (e->host_overlap) {
    if (!e->aux_after_logic) {
      CUDA_TRY(cudaEventRecord(e->ev_main, s));
      CUDA_TRY(cudaStreamWaitEvent(e->aux_stream, e->ev_main, 0));
    }
    s = e->aux_stream;
    stream = (sy_stream_t)s;
  }
  int rc;
  if (bytes_per_action == 8) rc = sample_impl<long long>(e, st, step_counter, reinterpret_cast<long long*>(actions_dev), stream);
  else if (bytes_per_action == 4) rc = sample_impl<int>(e, st, step_counter, reinterpret_cast<int*>(actions_dev), stream);
  else if (bytes_per_action == 2) rc = sy_sample_actions_i16(e, st, step_counter, reinterpret_cast<int16_t*>(actions_dev), stream);
  else return fail(SY_ERR_INVALID_ARGUMENT, "bytes_per_action must be 8, 4 or 2");
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(actions_host, actions_dev, (size_t)e->cfg.num_envs * e->A * bytes_per_action, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  return SY_OK;
}

// K steps of the host-buffer loop driven from C: per step sy_sample_actions_host (the random policy's actions arrive in
// HOST memory) followed by sy_step_host* with those host actions -- the same two calls, copies and synchronisations a
// host-side policy loop makes, without an interpreter between them
int sy_host_rollout_random(SyEnv* e, int32_t num_steps, uint32_t step_counter0, void* actions_dev, void* actions_host,
                           int32_t bytes_per_action, const SyState* st, const SyObs* ob, const SyOut* out,
                           const SyHostOut* ho, sy_stream_t stream) {
  if (!e || num_steps < 0) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env or negative num_steps");
  if (e->grp_need_reset) return fail(SY_ERR_STATE, "mechanism groups changed: a sy_reset of every env (NULL or all-set mask) must come before the next step");
  for (int32_t k = 0; k < num_steps; ++k) {
    int rc = sy_sample_actions_host(e, st, step_counter0 + (uint32_t)k, actions_dev, actions_host, bytes_per_action, stream);
    if (rc) return rc;
    if (bytes_per_action == 8) rc = sy_step_host(e, (const int64_t*)actions_host, (int64_t*)actions_dev, st, ob, out, ho, stream);
    else if (bytes_per_action == 4) rc = sy_step_host_i32(e, (const int32_t*)actions_host, (int32_t*)actions_dev, st, ob, out, ho, stream);
    else rc = sy_step_host_i16(e, (const int16_t*)actions_host, (int16_t*)actions_dev, st, ob, out, ho, stream);
    if (rc) return rc;
  }
  return SY_OK;
}

int sy_set_host_overlap(SyEnv* e, int32_t on) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  if (on && !e->ev_main) CUDA_TRY(cudaEventCreateWithFlags(&e->ev_main, cudaEventDisableTiming));
  e->host_overlap = on ? 1 : 0;
  e->aux_after_logic = false;
  return SY_OK;
}

int sy_sample_actions(SyEnv* e, const SyState* st, uint32_t step_counter, int64_t* actions, sy_stream_t stream) {
  return sample_impl<long long>(e, st, step_counter, reinterpret_cast<long long*>(actions), stream);
}

int sy_sample_actions_i32(SyEnv* e, const SyState* st, uint32_t step_counter, int32_t* actions, sy_stream_t stream) {
  return sample_impl<int>(e, st, step_counter, actions, stream);
}

int sy_heuristic_actions(SyEnv* e, const SyHeuristic* h, const SyState* st, const SyObs* ob, uint32_t step_counter,
                         int64_t* actions, sy_stream_t stream) {
  if (!e || !h || !actions) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / heuristic / actions");
  if (h->struct_bytes != sizeof(SyHeuristic)) return fail(SY_ERR_INVALID_ARGUMENT, "SyHeuristic size mismatch: got %llu, library expects %zu (ABI %d)", (unsigned long long)h->struct_bytes, sizeof(SyHeuristic), SY_ABI_VERSION);
  if (h->mrx_kind != SY_HEUR_NONE && h->mrx_kind != SY_HEUR_RANDOM && h->mrx_kind != SY_HEUR_EVADE)
    return fail(SY_ERR_INVALID_ARGUMENT, "SyHeuristic.mrx_kind must be SY_HEUR_NONE, SY_HEUR_RANDOM or SY_HEUR_EVADE, got %d", h->mrx_kind);
  if (h->police_kind != SY_HEUR_NONE && h->police_kind != SY_HEUR_RANDOM && h->police_kind != SY_HEUR_CHASE && h->police_kind != SY_HEUR_CHASE_BELIEF)
    return fail(SY_ERR_INVALID_ARGUMENT, "SyHeuristic.police_kind must be SY_HEUR_NONE, SY_HEUR_RANDOM, SY_HEUR_CHASE or SY_HEUR_CHASE_BELIEF, got %d", h->police_kind);
  if (h->explore_mrx > (1ull << 32) || h->explore_police > (1ull << 32))
    return fail(SY_ERR_INVALID_ARGUMENT, "SyHeuristic exploration thresholds must be at most 2^32");
  Params p;
  int rc = fill_params(e, st, ob, nullptr, p);
  if (rc) return rc;
  if (!ob || !ob->mrx_revealed) return fail(SY_ERR_INVALID_ARGUMENT, "SyObs.mrx_revealed is NULL");
  const bool belief = h->police_kind == SY_HEUR_CHASE_BELIEF;
  if (belief && (!e->cfg.belief || !st->belief)) return fail(SY_ERR_INVALID_ARGUMENT, "SY_HEUR_CHASE_BELIEF needs config.belief and SyState.belief");
  if (e->grp_need_reset) return fail(SY_ERR_STATE, "mechanism groups changed: a sy_reset of every env (NULL or all-set mask) must come before the next step");
  if (belief && e->obs_pending) return fail(SY_ERR_STATE, "SY_HEUR_CHASE_BELIEF reads the belief map: observations are pending (sy_flush_observations first)");
  const HeurArgs a{h->mrx_kind, h->police_kind, h->explore_mrx, h->explore_police, h->last_seen,
                   reinterpret_cast<long long*>(actions), step_counter};
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  const unsigned grid = (unsigned)((p.B + HEUR_ENVS - 1) / HEUR_ENVS);
  if (p.grp_n) sy_heuristic_actions_kernel<1><<<grid, HEUR_THREADS, 0, (cudaStream_t)stream>>>(p, a);
  else sy_heuristic_actions_kernel<0><<<grid, HEUR_THREADS, 0, (cudaStream_t)stream>>>(p, a);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

int sy_stats(SyEnv* e, int64_t* stats, sy_stream_t stream) {
  if (!e || !stats) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / stats");
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  sy_fold_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((unsigned long long*)e->d_stats_rep, reinterpret_cast<long long*>(stats));
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

int sy_set_groups(SyEnv* e, int32_t n, const SyGroup* groups, const int32_t* group_id, sy_stream_t stream) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  if (e->obs_pending) return fail(SY_ERR_STATE, "sy_set_groups: observations are pending (sy_flush_observations first)");
  if (n < 0 || n > SY_MAX_GROUPS) return fail(SY_ERR_INVALID_ARGUMENT, "num_groups must be in [0, %d], got %d", SY_MAX_GROUPS, n);
  if (n > 0 && !groups) return fail(SY_ERR_INVALID_ARGUMENT, "SyGroup table is NULL");
  std::vector<GroupRow> rows((size_t)n);
  for (int g = 0; g < n; ++g) {
    const SyGroup& q = groups[g];
    if (q.struct_bytes != sizeof(SyGroup))
      return fail(SY_ERR_INVALID_ARGUMENT, "SyGroup size mismatch in group %d: got %llu, library expects %zu (ABI %d)", g, (unsigned long long)q.struct_bytes, sizeof(SyGroup), SY_ABI_VERSION);
    if (q.agent_money < 0 || q.reveal_interval < 0) return fail(SY_ERR_INVALID_ARGUMENT, "group %d: negative agent_money / reveal_interval", g);
    if (!(q.reveal_skip_prob >= 0.0f && q.reveal_skip_prob <= 1.0f)) return fail(SY_ERR_INVALID_ARGUMENT, "group %d: reveal_skip_prob must be in [0, 1]", g);
    for (int i = 0; i < SY_NUM_REWARD_WEIGHTS; ++i) {
      if (!std::isfinite(q.reward_weights[i])) return fail(SY_ERR_INVALID_ARGUMENT, "group %d: reward weight %d is not finite", g, i);
      rows[g].w64[i] = q.reward_weights[i];
      rows[g].w32[i] = (float)q.reward_weights[i];
    }
    rows[g].agent_money = q.agent_money;
    rows[g].reveal = q.reveal_interval;
    rows[g].reveal_skip_thresh = q.reveal_skip_prob > 0.0f ? (unsigned long long)((double)fminf(q.reveal_skip_prob, 1.0f) * 4294967296.0) : 0ull;
    rows[g].toll = e->cfg.toll;  // every group starts with the config's toll (sy_set_group_tolls changes it) ...
    rows[g].num_police = e->cfg.num_police;  // ... police count and horizon (sy_set_group_rules)
    rows[g].max_t = e->cfg.max_timestep;
  }
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const int B = e->cfg.num_envs;
  // The buffers are allocated once, at their largest, and updated in place: kernels in flight, and CUDA graphs captured
  // earlier, never see a freed address (a graph captured under other groups still has to be recaptured -- its launches
  // carry the old group count and kernel choice)
  if (!e->d_grp) {
    if (cudaMalloc(&e->d_grp, (size_t)SY_MAX_GROUPS * sizeof(GroupRow)) != cudaSuccess ||
        cudaMalloc(&e->d_grp_id, (size_t)B * sizeof(int32_t)) != cudaSuccess ||
        cudaMalloc(&e->d_grp_id_new, (size_t)B * sizeof(int32_t)) != cudaSuccess ||
        cudaMalloc(&e->d_grp_stats, (size_t)GROUP_STAT_LINES * SY_NUM_STATS * sizeof(unsigned long long)) != cudaSuccess ||
        cudaMalloc(&e->d_grp_bad, sizeof(int)) != cudaSuccess) {
      for (void** ptr : {&e->d_grp, &e->d_grp_id, &e->d_grp_id_new, &e->d_grp_stats, &e->d_grp_bad}) {
        if (*ptr) cudaFree(*ptr);
        *ptr = nullptr;
      }
      return fail(SY_ERR_CUDA, "cudaMalloc of the mechanism group buffers failed");
    }
  }
  if (n > 0) {
    // ids into the staging buffer first: a rejected call leaves the handle's groups as they were
    int bad = 0;
    CUDA_TRY(cudaMemsetAsync(e->d_grp_bad, 0, sizeof(int), s));
    sy_group_ids_kernel<<<(unsigned)((B + 255) / 256), 256, 0, s>>>(group_id, (int32_t*)e->d_grp_id_new, B, n,
                                                                    (unsigned long long)e->cfg.env_offset, (int*)e->d_grp_bad);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(&bad, e->d_grp_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (bad) return fail(SY_ERR_INVALID_ARGUMENT, "%d group ids outside [0, %d)", bad, n);
    CUDA_TRY(cudaMemcpyAsync(e->d_grp_id, e->d_grp_id_new, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(e->d_grp, rows.data(), (size_t)n * sizeof(GroupRow), cudaMemcpyHostToDevice, s));
  }
  CUDA_TRY(cudaMemsetAsync(e->d_grp_stats, 0, (size_t)GROUP_STAT_LINES * SY_NUM_STATS * sizeof(unsigned long long), s));
  CUDA_TRY(cudaStreamSynchronize(s));  // (the host table is a local)
  e->grp_n = n;
  e->grp_rows = std::move(rows);
  // per-group lines spread like the handle-wide replicas: rep * n <= GROUP_STAT_LINES for every n <= SY_MAX_GROUPS
  e->grp_rep = n ? std::max(1, std::min(STAT_REPLICAS, GROUP_STAT_LINES / n)) : 0;
  e->grp_need_reset = true;
  return SY_OK;
}

int sy_set_group_tolls(SyEnv* e, int32_t n, const int32_t* tolls, sy_stream_t stream) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  if (e->obs_pending) return fail(SY_ERR_STATE, "sy_set_group_tolls: observations are pending (sy_flush_observations first)");
  if (e->grp_n == 0) return fail(SY_ERR_STATE, "sy_set_group_tolls: no mechanism groups are set (sy_set_groups first)");
  if (n != e->grp_n) return fail(SY_ERR_INVALID_ARGUMENT, "sy_set_group_tolls: num_groups %d, but the handle holds %d groups", n, e->grp_n);
  if (!tolls) return fail(SY_ERR_INVALID_ARGUMENT, "tolls is NULL");
  for (int g = 0; g < n; ++g)
    if (tolls[g] < 0 || tolls[g] > SY_MAX_TOLL) return fail(SY_ERR_INVALID_ARGUMENT, "group %d: toll %d outside [0, %d]", g, tolls[g], SY_MAX_TOLL);
  std::vector<GroupRow> rows = e->grp_rows;
  for (int g = 0; g < n; ++g) rows[g].toll = tolls[g];
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaMemcpyAsync(e->d_grp, rows.data(), (size_t)n * sizeof(GroupRow), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));  // (the host table is a local)
  e->grp_rows = std::move(rows);
  e->grp_need_reset = true;
  return SY_OK;
}

int sy_set_group_rules(SyEnv* e, int32_t n, const int32_t* num_police, const int32_t* max_timestep, sy_stream_t stream) {
  if (!e) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env");
  if (e->obs_pending) return fail(SY_ERR_STATE, "sy_set_group_rules: observations are pending (sy_flush_observations first)");
  if (e->grp_n == 0) return fail(SY_ERR_STATE, "sy_set_group_rules: no mechanism groups are set (sy_set_groups first)");
  if (n != e->grp_n) return fail(SY_ERR_INVALID_ARGUMENT, "sy_set_group_rules: num_groups %d, but the handle holds %d groups", n, e->grp_n);
  const int P = e->cfg.num_police, T = e->cfg.max_timestep;
  for (int g = 0; g < n; ++g) {
    if (num_police && (num_police[g] < 1 || num_police[g] > P))
      return fail(SY_ERR_INVALID_ARGUMENT, "group %d: num_police %d outside [1, %d]", g, num_police[g], P);
    if (max_timestep && (max_timestep[g] < 0 || max_timestep[g] > T))
      return fail(SY_ERR_INVALID_ARGUMENT, "group %d: max_timestep %d outside [0, %d]", g, max_timestep[g], T);
  }
  std::vector<GroupRow> rows = e->grp_rows;
  for (int g = 0; g < n; ++g) {
    rows[g].num_police = num_police ? num_police[g] : P;
    rows[g].max_t = max_timestep ? max_timestep[g] : T;
  }
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  CUDA_TRY(cudaMemcpyAsync(e->d_grp, rows.data(), (size_t)n * sizeof(GroupRow), cudaMemcpyHostToDevice, s));
  CUDA_TRY(cudaStreamSynchronize(s));  // (the host table is a local)
  e->grp_rows = std::move(rows);
  e->grp_need_reset = true;
  return SY_OK;
}

int sy_group_stats(SyEnv* e, int32_t n, int64_t* stats, sy_stream_t stream) {
  if (!e || !stats) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / stats");
  if (n != e->grp_n || n == 0) return fail(SY_ERR_INVALID_ARGUMENT, "sy_group_stats: num_groups %d, but the handle holds %d groups", n, e->grp_n);
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  const int total = n * SY_NUM_STATS;
  sy_fold_group_stats_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>((unsigned long long*)e->d_grp_stats, n, e->grp_rep, reinterpret_cast<long long*>(stats));
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

// SURVEY 8(b)/(e): the one collective of the path.  NCCL is resolved at run time (dlopen of the libnccl the host process
// already uses, e.g. the one bundled with PyTorch), so the library has no link-time dependency on it and a host that is
// not PyTorch (a C++ / Go / Rust learner with its own ncclComm_t) gets the multi-GPU reduction too.
namespace {
typedef int (*NcclAllReduceFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*NcclGetErrorStringFn)(int);
NcclAllReduceFn g_nccl_allreduce = nullptr;
NcclGetErrorStringFn g_nccl_errstr = nullptr;
int resolve_nccl() {
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (g_nccl_allreduce) return SY_OK;
  void* h = nullptr;
  const char* override_path = getenv("SY_NCCL_LIB");
  const char* names[] = {override_path, "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (!n) continue;
    if ((h = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
  }
  void* sym = h ? dlsym(h, "ncclAllReduce") : dlsym(RTLD_DEFAULT, "ncclAllReduce");  // already loaded by the host process?
  if (!sym) return fail(SY_ERR_STATE, "sy_allreduce_stats: libnccl.so.2 not found (load NCCL in the host process or set SY_NCCL_LIB)");
  g_nccl_allreduce = reinterpret_cast<NcclAllReduceFn>(sym);
  g_nccl_errstr = reinterpret_cast<NcclGetErrorStringFn>(h ? dlsym(h, "ncclGetErrorString") : dlsym(RTLD_DEFAULT, "ncclGetErrorString"));
  return SY_OK;
}
}  // namespace

int sy_allreduce_stats(SyEnv* e, void* nccl_comm, int64_t* stats_local, int64_t* stats_global, sy_stream_t stream) {
  if (!e || !nccl_comm || !stats_local || !stats_global) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / communicator / statistics vectors");
  if (int rc = resolve_nccl()) return rc;
  if (int rc = sy_stats(e, stats_local, stream)) return rc;  // fold the library's accumulators into the rank's cumulative vector
  enum { NCCL_INT64 = 4, NCCL_SUM = 0 };  // nccl.h: ncclInt64, ncclSum
  const int nrc = g_nccl_allreduce(stats_local, stats_global, SY_NUM_STATS, NCCL_INT64, NCCL_SUM, nccl_comm, (cudaStream_t)stream);
  if (nrc != 0) return fail(SY_ERR_CUDA, "ncclAllReduce failed: %s", g_nccl_errstr ? g_nccl_errstr(nrc) : "unknown NCCL error");
  return SY_OK;
}

int sy_copy_segments(int32_t num_segments, void* const* dst, const void* const* src, const uint64_t* bytes, sy_stream_t stream) {
  if (num_segments < 0 || num_segments > SY_MAX_COPY_SEGMENTS || (num_segments && (!dst || !src || !bytes)))
    return fail(SY_ERR_INVALID_ARGUMENT, "0..%d segments with non-NULL pointer tables", SY_MAX_COPY_SEGMENTS);
  if (num_segments == 0) return SY_OK;
  CopySegments c{};
  unsigned long long longest = 0;
  for (int i = 0; i < num_segments; ++i) {
    if (bytes[i] && (!dst[i] || !src[i])) return fail(SY_ERR_INVALID_ARGUMENT, "segment %d has a NULL pointer", i);
    c.dst[i] = dst[i];
    c.src[i] = src[i];
    c.bytes[i] = bytes[i];
    longest = std::max<unsigned long long>(longest, bytes[i]);
  }
  const unsigned gx = (unsigned)std::min<unsigned long long>(std::max<unsigned long long>((longest / 16 + 255) / 256, 1), 148 * 8);
  sy_copy_segments_kernel<<<dim3(gx, (unsigned)num_segments), 256, 0, (cudaStream_t)stream>>>(c);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

}  // extern "C"

namespace {
// the whole rollout as ONE launch of sy_rollout_lagged_kernel (batches of at most one wave, observations current on entry;
// `actions` holds the first step's draw).  The draw of step k + 1 uses counter next_counter + k (+ *base).
int rollout_one_launch(SyEnv* e, int32_t num_steps, int64_t* actions, uint32_t next_counter, const uint32_t* next_counter_base,
                       const SyState* st, const SyObs* ob, const SyOut* out, cudaStream_t s) {
  if (!out) return fail(SY_ERR_INVALID_ARGUMENT, "SyOut is NULL");
  if (out->struct_bytes != sizeof(SyOut)) return fail(SY_ERR_INVALID_ARGUMENT, "SyOut size mismatch");
  if (!out->reward || !out->terminated || !out->truncated || !out->done || !out->winner)
    return fail(SY_ERR_INVALID_ARGUMENT, "SyOut has NULL members");
  Params p;
  int rc = fill_params(e, st, ob, out, p);
  if (rc) return rc;
  if ((rc = check_obs(ob))) return rc;
  p.actions = reinterpret_cast<const long long*>(actions);
  p.next_actions = reinterpret_cast<long long*>(actions);
  p.next_counter = next_counter;
  p.next_counter_base = next_counter_base;
  CUDA_TRY(cudaSetDevice(e->cfg.device));
  e->aux_after_logic = false;
  rollout_fn(e, p.grp_n > 0)<<<(unsigned)((p.B + TILE - 1) / TILE), lagged_threads(e), e->obs_smem, s>>>(p, (int)num_steps);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}
bool one_launch_rollout(const SyEnv* e, const SyObs* ob) {
  // at most one CTA per SM: there the launches it saves outweigh the CTA-wide barrier per step (c2, 32 tiles: 8.8 -> 6.8 us
  // per step; c3-shaped 148 tiles 17.3 -> 16.4 us; 192 tiles 22.0 -> 22.4 us, 296 tiles 23.2 -> 24.8 us)
  return use_lagged(e) && e->opt_writer != SY_WRITER_BULK && e->opt_fused != SY_STEP_FUSED && e->opt_rollout_kernel &&
         2 * ((e->cfg.num_envs + TILE - 1) / TILE) <= e->lag_slots && ob != nullptr;
}
}  // namespace

extern "C" {

int sy_rollout_random(SyEnv* e, int32_t num_steps, uint32_t step_counter0, int64_t* actions, const SyState* st, const SyObs* ob,
                      const SyOut* out, sy_stream_t stream) {
  if (!e || !actions || num_steps < 0) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions or negative num_steps");
  if (e->grp_need_reset) return fail(SY_ERR_STATE, "mechanism groups changed: a sy_reset of every env (NULL or all-set mask) must come before the next step");
  if (num_steps >= 2 && one_launch_rollout(e, ob)) {
    int rc = sy_flush_observations(e, st, ob, stream);
    if (!rc) rc = sy_sample_actions(e, st, step_counter0, actions, stream);
    if (!rc) rc = rollout_one_launch(e, num_steps, actions, step_counter0 + 1u, nullptr, st, ob, out, (cudaStream_t)stream);
    return rc;
  }
  bool have_actions = false;  // the fused / lagged step kernels draw the next step's actions themselves
  const bool pipelined = use_lagged(e) && e->opt_writer != SY_WRITER_BULK && e->opt_fused != SY_STEP_FUSED;  // deferred steps, one flush at the end
  for (int32_t k = 0; k < num_steps; ++k) {
    int rc;
    if (!have_actions && (rc = sy_sample_actions(e, st, step_counter0 + (uint32_t)k, actions, stream))) return rc;
    have_actions = false;
    const bool more = k + 1 < num_steps;
    if ((rc = step_impl(e, actions, nullptr, st, ob, out, stream, nullptr, nullptr, more ? actions : nullptr,
                        step_counter0 + (uint32_t)k + 1u, nullptr, &have_actions, pipelined)))
      return rc;
    have_actions = have_actions && more;
  }
  return sy_flush_observations(e, st, ob, stream);
}

int sy_rollout_random_dev(SyEnv* e, int32_t num_steps, uint32_t* step_counter_dev, int64_t* actions, const SyState* st,
                          const SyObs* ob, const SyOut* out, sy_stream_t stream) {
  if (!e || !actions || !step_counter_dev || num_steps < 0) return fail(SY_ERR_INVALID_ARGUMENT, "NULL env / actions / counter or negative num_steps");
  if (e->grp_need_reset) return fail(SY_ERR_STATE, "mechanism groups changed: a sy_reset of every env (NULL or all-set mask) must come before the next step");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = SY_OK;
  if (num_steps >= 2 && one_launch_rollout(e, ob)) {
    rc = sy_flush_observations(e, st, ob, stream);
    if (!rc) rc = sample_impl<long long>(e, st, 0u, reinterpret_cast<long long*>(actions), stream, step_counter_dev);
    if (!rc) rc = rollout_one_launch(e, num_steps, actions, 1u, step_counter_dev, st, ob, out, s);
    if (rc) return rc;
    sy_advance_counter_kernel<<<1, 1, 0, s>>>(step_counter_dev, (unsigned)num_steps);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return SY_OK;
  }
  rc = num_steps > 0 ? sample_impl<long long>(e, st, 0u, reinterpret_cast<long long*>(actions), stream, step_counter_dev) : SY_OK;
  if (rc) return rc;
  const bool pipelined = use_lagged(e) && e->opt_writer != SY_WRITER_BULK && e->opt_fused != SY_STEP_FUSED;
  if (fused_eligible(e, ob) || pipelined) {
    // one launch per step: the dynamics warps of the fused / lagged kernel draw the next step's actions from the new
    // state.  Pipelined: step k's launch also writes the observations of step k - 1; one flush closes the segment.
    for (int32_t k = 0; k < num_steps; ++k) {
      const bool more = k + 1 < num_steps;
      if ((rc = step_impl(e, actions, nullptr, st, ob, out, stream, nullptr, nullptr, more ? actions : nullptr, (uint32_t)(k + 1), step_counter_dev,
                          nullptr, pipelined)))
        return rc;
    }
    if ((rc = sy_flush_observations(e, st, ob, stream))) return rc;
  } else {
    // The sampler of step k + 1 only needs the state the dynamics of step k wrote, not its observations: it is forked
    // onto the library stream right behind the logic kernel (fork / join with events, capturable), so it runs next to
    // the observation kernel of step k instead of after it.  (Drawing the actions at the end of the dynamics kernel
    // instead, as the single-launch kernels do, was measured slower here: c3 0.1319 vs 0.1294 ms per step, c4 0.3175 vs
    // 0.3145 -- it lengthens the latency-bound kernel, while the forked sampler hides under the store stream.)
    if (!e->ev_fork) CUDA_TRY(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    if (!e->ev_join) CUDA_TRY(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    for (int32_t k = 0; k < num_steps; ++k) {
      const bool more = k + 1 < num_steps;
      if ((rc = step_impl(e, actions, nullptr, st, ob, out, stream, more ? e->ev_fork : nullptr))) return rc;
      if (more) {
        CUDA_TRY(cudaStreamWaitEvent(e->aux_stream, e->ev_fork, 0));
        if ((rc = sample_impl<long long>(e, st, (uint32_t)(k + 1), reinterpret_cast<long long*>(actions), (sy_stream_t)e->aux_stream, step_counter_dev)))
          return rc;
        CUDA_TRY(cudaEventRecord(e->ev_join, e->aux_stream));
        CUDA_TRY(cudaStreamWaitEvent(s, e->ev_join, 0));
      }
    }
  }
  sy_advance_counter_kernel<<<1, 1, 0, s>>>(step_counter_dev, (unsigned)num_steps);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

int sy_action_mask_dense(int32_t Q, int32_t N, const double* adj, const double* w, const double* toll_m, double toll_s,
                         const int32_t* cur, const double* budget, uint8_t* out, sy_stream_t stream) {
  if (Q < 0 || N <= 0 || !adj || !cur || !budget || !out) return fail(SY_ERR_INVALID_ARGUMENT, "bad dense mask arguments");
  if (Q == 0) return SY_OK;
  sy_mask_dense_kernel<<<(unsigned)Q, 128, 0, (cudaStream_t)stream>>>(N, adj, w, toll_m, toll_s, cur, budget, out);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return SY_OK;
}

}  // extern "C"
