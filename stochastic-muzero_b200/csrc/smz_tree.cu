// smz_tree.cu — tree kernels of the batched Stochastic-MuZero search (sm_100a).
//
// G threads ("lanes") of a warp cooperate on one tree, one lane per child / per path node; G is a
// template parameter (2..32, 32 = warp per tree).  All arithmetic that decides a visit order follows
// the reference's numpy semantics exactly (SURVEY.md §8a T3-T9): explicit round-to-nearest
// intrinsics (no FMA contraction), float64 pUCT prior term, float32 value term, numpy's pairwise
// float32 summation order, RandomState.choice's cdf/searchsorted algorithm.
//
//   k_root_expand    monte_carlo_tree_search.py:203-225  root children + Dirichlet mixing
//   k_select         :235-267   pUCT argmax / chance sampling descent, leaf record, branch compaction
//   k_expand_backup  :289-308   children of the leaf + min-max discounted backup
//   k_read_roots     game.py:179-204 consumer view (child visits, priors, rewards, root value)
#include <stdlib.h>

#include "smz_common.cuh"
#include "smz_kernels.h"
#include "smz_tree_dev.cuh"

namespace {

using namespace smz_tree_dev;

// ------------------------------------------------------------------------------------------------
// Legal set of a tree's root: bit a = action a may be played.  No mask means every action.  A mask that is empty or
// names an action >= A is `bad`: the tree is then searched with every action legal (k_root_expand raises flag 3).
__device__ __forceinline__ unsigned root_legal_set(const uint32_t* __restrict__ legal, int tree, int A, bool& bad) {
  const unsigned all = A >= 32 ? 0xffffffffu : (1u << A) - 1u;
  const unsigned m = legal ? legal[tree] : all;
  bad = m == 0u || (m & ~all) != 0u;
  return bad ? all : m;
}

// Simulation budget of a tree at the root step: given (smz_set_root_budgets) or N.  A budget outside [0, N] is `bad`: the
// tree is then searched with N (k_root_expand raises flag 4).
__device__ __forceinline__ int root_budget(const int* __restrict__ budget, int tree, int N, bool& bad) {
  const int b = budget ? budget[tree] : N;
  bad = b < 0 || b > N;
  return bad ? N : b;
}
// Root noise of a tree (Dirichlet in pUCT mode, Gumbels in Gumbel mode): its exploration flag, or the call's `train`.
__device__ __forceinline__ bool root_explores(const unsigned char* __restrict__ explore, int tree, int train) {
  return explore ? explore[tree] != 0 : train != 0;
}

template <int G>
__global__ void k_root_expand(SmzArena a, int n_trees, const float* __restrict__ policy, int pstride,
                              const int* __restrict__ root_to_play, int train,
                              const double* __restrict__ dirichlet, const uint32_t* __restrict__ legal,
                              const int* budget, const unsigned char* __restrict__ explore) {   // budget may be a.budget
  Group<G> g;
  int tree = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const bool alive = tree < n_trees;
  if (!alive) tree = n_trees - 1;
  const size_t tb = (size_t)tree * a.M;
  bool bad;
  const unsigned lm = root_legal_set(legal, tree, a.A, bad);
  bool bad_budget;
  const int bud = root_budget(budget, tree, a.N, bad_budget);
  // Dirichlet noise (pUCT only: `train` is 0 in Gumbel mode) iff the tree explores and has a simulation (mcts.py:215-216)
  const bool noise = (explore ? explore[tree] != 0 && !a.gumbel : train != 0) && bud > 0;
  // the root's action space is the legal set L: lane i works on its i-th action, so the policy is compacted before
  // it is normalised and drawn from (with every action legal, lane i is action i)
  const int n = __popc(lm);
  const int act = g.gl < n ? (int)__fns(lm, 0, g.gl + 1) : 0;
  int cursor = 0;
  const float pol = (g.gl < n) ? policy[(size_t)tree * pstride + act] : 0.f;
  const float p = normalise_policy(g, pol, n);
  // all legal actions become children (ascending); the call still consumes its draws (T5)
  const SmzRng rng = smz_make_rng(a);
  choice_without_replacement(g, a, rng, alive, tree, p, n, n, cursor);
  if (!alive) return;
  if (g.gl < n) {
    double prior = (double)p;
    if (noise) {
      const double nz = dirichlet[(size_t)tree * a.A + act];
      prior = __dadd_rn((double)__fmul_rn(p, a.one_minus_frac_f32), __dmul_rn(nz, a.frac));
    }
    a.root_prior[(size_t)tree * a.A + act] = prior;
    a.stat[tb + 1 + act] = make_int4(0, 0, 0, __float_as_int(p));
    a.link[tb + 1 + act] = make_int2(0, act);
  }
  // root-child slots stay indexed by action: the slot of an illegal action holds the sentinel key -1, prior 0, and
  // is never expanded; its recorded noise reads 0
  if (g.gl < a.A && !((lm >> g.gl) & 1u)) {
    a.root_prior[(size_t)tree * a.A + g.gl] = 0.0;
    a.stat[tb + 1 + g.gl] = make_int4(0, 0, 0, 0);
    a.link[tb + 1 + g.gl] = make_int2(0, -1);
    if (noise) a.dirichlet[(size_t)tree * a.A + g.gl] = 0.0;
  }
  if (g.gl == 0) {
    if (bad) *a.error_flag = 3;
    if (bad_budget) *a.error_flag = 4;
    a.budget[tree] = bud;
    a.stat[tb] = make_int4(0, 0, 0, 0);
    a.link[tb] = make_int2(1, -1);
    a.minmax[tree] = make_float2(__int_as_float(0x7f800000), __int_as_float(0xff800000));
    a.ucursor[tree] = cursor;
    // wrapped into [0, n_phases) like Player_cycle.global_step() (mcts.py:55-58): the backup indexes the sign table with it
    const int rtp = root_to_play ? root_to_play[tree] % a.n_phases : 0;
    a.root_to_play[tree] = rtp < 0 ? rtp + a.n_phases : rtp;
    a.path_len[tree] = 0;
    if (a.rec_root_policy)
      for (int i = 0; i < a.W; ++i) a.rec_root_policy[(size_t)tree * a.W + i] = i < a.A ? policy[(size_t)tree * pstride + i] : 0.f;
  }
}

// BUDGET (compile time, like GUMBEL): the search was given per-tree budgets (smz_set_root_budgets), so a tree takes part
// in simulation `sim` iff sim < a.budget[tree].  Without budgets every tree has N simulations: the default instantiations
// do not read the column and keep their registers.
template <int G, bool GUMBEL, bool BUDGET>
__global__ void k_select(SmzArena a, int n_trees, int sim, int* __restrict__ o_slot, int* __restrict__ o_action,
                         int* __restrict__ o_branch) {
  Group<G> g;
  int tree = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const bool exists = tree < n_trees;
  if (!exists) tree = n_trees - 1;
  const int bud = BUDGET ? a.budget[tree] : a.N;
  const bool alive = exists && (!BUDGET || sim < bud);
  const SmzRng rng = smz_make_rng(a);
  TreeState ts;
  ts.cursor = a.ucursor[tree];
  ts.mm = a.minmax[tree];
  const int4 rs = a.stat[(size_t)tree * a.M];
  ts.root = make_int2(rs.x, rs.y);
  select_phase<G, false, GUMBEL>(g, a, rng, tree, alive, BUDGET ? bud : -1, sim, ts, o_slot, o_action, o_branch);
  if (BUDGET && exists && !alive && g.gl == 0 && o_slot) o_slot[tree] = -1;     // no simulation `sim` for this tree
}

template <int G, bool GUMBEL, bool BUDGET>
__global__ void k_expand_backup(SmzArena a, int n_trees, int sim, const float* __restrict__ policy, int pstride,
                                const float* __restrict__ value, const float* __restrict__ reward) {
  Group<G> g;
  int tree = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const bool exists = tree < n_trees;
  if (!exists) tree = n_trees - 1;
  const bool alive = exists && (!BUDGET || sim < a.budget[tree]);
  const SmzRng rng = smz_make_rng(a);
  expand_backup_phase<G, false, GUMBEL>(g, a, rng, tree, alive, sim, policy, pstride, value, reward);
}

// expansion + backup of simulation `sim` followed by the descent of simulation `sim + 1` for the same
// tree by the same lanes: one launch per simulation instead of two, the path nodes just updated are
// re-read from L1/L2.
template <int G, bool GUMBEL, bool BUDGET>
__global__ void k_backup_select(SmzArena a, int n_trees, int sim) {
  Group<G> g;
  int tree = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const bool exists = tree < n_trees;
  if (!exists) tree = n_trees - 1;
  const int bud = BUDGET ? a.budget[tree] : a.N;     // written by the root step: requested before the wait
  smz_pdl_wait();                 // the network step of `sim` must have landed
  smz_pdl_launch_dependents();    // the next network step may set itself up (barriers, TMEM, weights)
  // a tree whose budget is used up takes no part in either phase (its TreeState is then never read)
  const bool alive = exists && (!BUDGET || sim < bud), alive_next = exists && (!BUDGET || sim + 1 < bud);
  const bool stamp = a.dbg && blockIdx.x == 0 && threadIdx.x == 0;
  if (stamp) a.dbg[0] = clock64();
  const SmzRng rng = smz_make_rng(a);
  const TreeState ts = expand_backup_phase<G, false, GUMBEL>(g, a, rng, tree, alive, sim, a.out_policy, a.W, a.out_value,
                                                             a.out_reward);
  __syncwarp();
  if (stamp) a.dbg[1] = clock64();
  select_phase<G, false, GUMBEL>(g, a, rng, tree, alive_next, BUDGET ? bud : -1, sim + 1, ts, nullptr, nullptr, nullptr);
  if (stamp) { a.dbg[2] = clock64(); a.dbg[3] = a.path_len[tree]; }
}

// Same step with every tree's node records mirrored in shared memory.  The tree arena is written by tree kernels
// only, so the mirror is filled BEFORE griddepcontrol.wait — while the network step is still running (the network
// kernels signal their dependents only after their own wait, so the previous tree kernel has completed).  After
// the wait the phases touch L2 for the network outputs alone: expansion and backup update mirror + arena, the
// descent reads the mirror (shared-memory latency per level instead of an L2 round trip).
constexpr int SMZ_UWIN = 32;     // uniforms generated ahead per tree (Philox mode): expansion draws + ~12 levels of descent

// dynamic shared memory of k_backup_select_sm for `tpb` trees per block (must match the kernel's carve-up)
__host__ __device__ inline size_t smz_mirror_bytes(int tpb, int M, int A, int n_tab, int n_pbc) {
  size_t b = (size_t)tpb * M * (sizeof(int4) + sizeof(int2));          // node records
  b += (size_t)tpb * (A + SMZ_UWIN) * sizeof(double);                    // root priors, uniform window
  b += (size_t)(n_pbc + n_tab) * sizeof(double) + (size_t)n_tab * sizeof(float);   // pbc, rcp64, rcp32
  return b + 16;
}

template <int G, bool GUMBEL, bool BUDGET>
__global__ void k_backup_select_sm(SmzArena a, int n_trees, int sim, int n_tab) {
  extern __shared__ int4 smz_sm_nodes[];
  Group<G> g;
  int tree = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const bool exists = tree < n_trees;
  if (!exists) tree = n_trees - 1;
  const int bud = BUDGET ? a.budget[tree] : a.N;
  const bool alive = exists && (!BUDGET || sim < bud), alive_next = exists && (!BUDGET || sim + 1 < bud);
  const int tpb = blockDim.x / G, lt = threadIdx.x / G;           // trees per block, local tree
  // ---- carve-up: [stat][link][root priors][uniform window][pbc][rcp64][rcp32]
  int4* sst = smz_sm_nodes + (size_t)lt * a.M;
  int2* slk_all = reinterpret_cast<int2*>(smz_sm_nodes + (size_t)tpb * a.M);
  int2* slk = slk_all + (size_t)lt * a.M;
  double* dbl = reinterpret_cast<double*>(slk_all + (size_t)tpb * a.M + ((size_t)tpb * a.M & 1));
  double* srp = dbl + (size_t)lt * a.A;
  double* swin = dbl + (size_t)tpb * a.A + (size_t)lt * SMZ_UWIN;
  double* spbc = dbl + (size_t)tpb * (a.A + SMZ_UWIN);
  double* sr64 = spbc + (a.N + 2);
  float* sr32 = reinterpret_cast<float*>(sr64 + n_tab);

  // ---- prologue: everything here was written by tree kernels / the host, not by the running network step
  SmzRng rng = smz_make_rng(a);
  const int cursor0 = a.ucursor[tree];
  {
    const size_t tb = (size_t)tree * a.M;
    // nodes allocated before this expansion (a tree whose budget is used up never reads its mirror)
    const int used = (BUDGET && !alive) ? 0 : 1 + a.A + sim * a.Kmax;
    for (int i = g.gl; i < used; i += G) {
      sst[i] = a.stat[tb + i];
      slk[i] = a.link[tb + i];
    }
    for (int i = g.gl; i < a.A; i += G) srp[i] = a.root_prior[(size_t)tree * a.A + i];
    for (int i = threadIdx.x; i < a.N + 2; i += blockDim.x) spbc[i] = a.pbc[i];
    for (int i = threadIdx.x; i < n_tab; i += blockDim.x) { sr64[i] = a.rcp64[i]; sr32[i] = a.rcp32[i]; }
    if (rng.mode == 0)                                            // device Philox: the draws depend on the cursor only
      for (int i = g.gl; i < SMZ_UWIN; i += G) swin[i] = smz_rng_uniform(rng, tree, cursor0 + i);
  }
  SmzArena al = a;                                                // same arena, tables served from shared memory
  al.pbc = spbc; al.rcp64 = sr64; al.rcp32 = sr32;
  if (rng.mode == 0) { rng.win = swin; rng.win_base = cursor0; rng.win_len = SMZ_UWIN; }
  smz_pdl_wait();                 // the network step of `sim` must have landed
  smz_pdl_launch_dependents();    // the next network step may set itself up (barriers, TMEM, weights)
  smz_stamp_min(a.dbg, sim, 0);
  __syncthreads();
  const bool stamp = a.dbg && blockIdx.x == 0 && threadIdx.x == 0;
  if (stamp) a.dbg[0] = clock64();
  const TreeState ts = expand_backup_phase<G, true, GUMBEL>(g, al, rng, tree, alive, sim, a.out_policy, a.W, a.out_value,
                                                            a.out_reward, sst, slk);
  __syncwarp();
  if (stamp) a.dbg[1] = clock64();
  select_phase<G, true, GUMBEL>(g, al, rng, tree, alive_next, BUDGET ? bud : -1, sim + 1, ts, nullptr, nullptr, nullptr, sst, slk, srp);
  if (stamp) { a.dbg[2] = clock64(); a.dbg[3] = a.path_len[tree]; }
  if (a.dbg) {
    __syncthreads();
    smz_stamp_max(a.dbg, sim, 1);
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void k_read_roots(SmzArena a, int n_trees, int* __restrict__ visits, float* __restrict__ values,
                             double* __restrict__ priors, float* __restrict__ rewards, int* __restrict__ error_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && error_out) *error_out = *a.error_flag;
  if (i >= n_trees * a.A) return;
  const int tree = i / a.A, c = i % a.A;
  const size_t tb = (size_t)tree * a.M;
  const int4 st = a.stat[tb + 1 + c];
  if (visits) visits[i] = st.x;
  if (rewards) rewards[i] = __int_as_float(st.z);
  if (priors) priors[i] = a.root_prior[i];
  if (values && c == 0) {
    const int4 r = a.stat[tb];
    values[tree] = r.x == 0 ? 0.f : __fdiv_rn(__int_as_float(r.y), (float)r.x);
  }
}

// numpy float64 add.reduce order over a small local array (same pairwise scheme as np_sum_f32)
__device__ double np_sum_f64(const double* x, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r = __dadd_rn(r, x[i]);
    return r;
  }
  double r[8];
  for (int j = 0; j < 8; ++j) r[j] = x[j];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], x[i + j]);
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, x[i]);
  return res;
}

// The step after the search, one thread per tree (game.py:179-216): the policy stored as training target
// (`store_search_statistics`), the temperature-scaled acting policy (`policy_action_reward_from_tree` +
// `softmax_stable`) and the action (`select_action`: sample when T > 0.1 or the policy is flat, else argmax).
__global__ void k_select_actions(SmzArena a, int n_trees, double temperature, const double* __restrict__ u_in,
                                 int* __restrict__ action_out, double* __restrict__ policy_out,
                                 double* __restrict__ stored_out) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= n_trees) return;
  const size_t tb = (size_t)tree * a.M;
  const int A = a.A;
  // the reference's rule over the legal children only (key -1 marks an illegal action's slot): compacted vectors,
  // results scattered back with 0 for illegal actions
  double v[SMZ_MAX_POLICY], pr[SMZ_MAX_POLICY], p[SMZ_MAX_POLICY];
  int act[SMZ_MAX_POLICY];
  int n = 0;
  for (int i = 0; i < A; ++i) {
    if (a.link[tb + 1 + i].y < 0) {
      if (stored_out) stored_out[(size_t)tree * A + i] = 0.0;
      if (policy_out) policy_out[(size_t)tree * A + i] = 0.0;
      continue;
    }
    act[n] = i;
    v[n] = (double)a.stat[tb + 1 + i].x;
    pr[n] = a.root_prior[(size_t)tree * A + i];
    ++n;
  }
  const double sv = np_sum_f64(v, n);
  if (stored_out) {
    const double sp = np_sum_f64(pr, n);
    for (int i = 0; i < n; ++i) stored_out[(size_t)tree * A + act[i]] = sv >= 3.0 ? __ddiv_rn(v[i], sv) : __ddiv_rn(pr[i], sp);
  }
  const double e = 1.0 / temperature;
  for (int i = 0; i < n; ++i) {
    double x = sv <= 1.0 ? pr[i] : v[i];
    if (temperature >= 0.3) x = e == 1.0 ? x : (e == 2.0 ? __dmul_rn(x, x) : (e == 0.5 ? sqrt(x) : pow(x, e)));
    p[i] = x;
  }
  const double s = np_sum_f64(p, n);
  bool flat = true;
  for (int i = 0; i < n; ++i) {
    p[i] = __ddiv_rn(p[i], s);
    flat = flat && p[i] == p[0];
    if (policy_out) policy_out[(size_t)tree * A + act[i]] = p[i];
  }
  int pick = 0;
  if (temperature > 0.1 || flat) {
    const double u = u_in ? u_in[tree] : smz_philox_uniform(a.seed_state[0], a.seed_state[1] + (unsigned long long)tree, 0u, 2u);
    double acc = 0.0;
    for (int i = 0; i < n; ++i) { acc = __dadd_rn(acc, p[i]); v[i] = acc; }
    for (int i = 0; i < n; ++i) pick += __ddiv_rn(v[i], acc) <= u;
    pick = pick < n ? pick : n - 1;
  } else {
    for (int i = 1; i < n; ++i) if (p[i] > p[pick]) pick = i;
  }
  if (action_out) action_out[tree] = act[pick];
}

// Dirichlet(alpha) per tree on the device: Gamma(alpha) by Marsaglia-Tsang (alpha+1 boost), Philox
// stream 1.  Production mode only; parity runs pass recorded noise (np.random.dirichlet, mcts.py:220).
// Draws are taken for the legal actions of the root only, in ascending order; an illegal action's noise is 0.
__global__ void k_dirichlet(SmzArena a, int n_trees, const uint32_t* __restrict__ legal, int train,
                            const int* __restrict__ budget, const unsigned char* __restrict__ explore) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= n_trees) return;
  bool bad;
  unsigned lm = root_legal_set(legal, tree, a.A, bad);
  if (!root_explores(explore, tree, train) || root_budget(budget, tree, a.N, bad) == 0) return;   // no noise: as train = 0
  unsigned ctr = 0;
  const unsigned long long seed = a.seed_state[0], tid = a.seed_state[1] + (unsigned long long)tree;
  auto U = [&]() { double u = smz_philox_uniform(seed, tid, ctr++, 1u); return u > 0.0 ? u : 1.0 / 9007199254740992.0; };
  double sum = 0.0;
  for (int i = 0; i < a.A; ++i) {
    if (!((lm >> i) & 1u)) {
      a.dirichlet[(size_t)tree * a.A + i] = 0.0;
      continue;
    }
    const double al = a.alpha;
    const double d = (al < 1.0 ? al + 1.0 : al) - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    double gsample = d;
    for (int it = 0; it < 256; ++it) {
      const double u1 = U(), u2 = U();
      const double x = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
      const double t = 1.0 + c * x;
      if (t <= 0.0) continue;
      const double v3 = t * t * t, u = U();
      if (log(u) < 0.5 * x * x + d - d * v3 + d * log(v3)) { gsample = d * v3; break; }
    }
    if (al < 1.0) gsample *= pow(U(), 1.0 / al);
    a.dirichlet[(size_t)tree * a.A + i] = gsample;
    sum += gsample;
  }
  for (int i = 0; i < a.A; ++i) a.dirichlet[(size_t)tree * a.A + i] /= (sum > 0.0 ? sum : 1.0);
}

// Root of a Gumbel search, one thread per tree, after k_root_expand: the root's network value into raw_value slot 0, the
// root logits log(p_a) - max_b log(p_b) over the legal actions (float64 root priors), and one Gumbel per legal action in
// ascending order (train): given by the caller, or -log(-log u) of the uniform #rank of Philox stream 3; eval: 0.
__global__ void k_gumbel_root(SmzArena a, int n_trees, const float* __restrict__ root_value, int train_call,
                              const double* __restrict__ given, const unsigned char* __restrict__ explore) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= n_trees) return;
  const bool train = root_explores(explore, tree, train_call);     // a budget-0 tree draws its Gumbels too
  const size_t tb = (size_t)tree * a.M, ro = (size_t)tree * a.A;
  a.raw_value[(size_t)tree * (a.N + 1)] = root_value[tree];
  double mx = -__longlong_as_double(0x7ff0000000000000LL);
  for (int i = 0; i < a.A; ++i)
    if (a.link[tb + 1 + i].y >= 0) mx = fmax(mx, log(a.root_prior[ro + i]));
  const unsigned long long seed = a.seed_state[0], tid = a.seed_state[1] + (unsigned long long)tree;
  unsigned rank = 0;
  for (int i = 0; i < a.A; ++i) {
    double gv = 0.0, lg = 0.0;
    if (a.link[tb + 1 + i].y >= 0) {
      lg = __dsub_rn(log(a.root_prior[ro + i]), mx);
      if (train && given) {
        gv = given[ro + i];
      } else if (train) {
        double u = smz_philox_uniform(seed, tid, rank, 3u);
        u = u > 0.0 ? u : 1.0 / 9007199254740992.0;         // (0, 1): u = 0 would give an infinite Gumbel
        gv = -log(-log(u));
      }
      ++rank;
    }
    a.gumbel_g[ro + i] = gv;
    a.root_logit[ro + i] = lg;
  }
}

// Read-out of a Gumbel search, one thread per tree: action = argmax over the legal actions with the most visits of
// g + logit + sigma (ties: the smaller action); improved policy = softmax over the legal actions of logit + sigma
// (0 for illegal actions); sigma from the completed Q-values of the root as the descent forms them.
__global__ void k_read_gumbel(SmzArena a, int n_trees, int* __restrict__ actions, double* __restrict__ improved,
                              double* __restrict__ gumbels) {
  const int tree = blockIdx.x * blockDim.x + threadIdx.x;
  if (tree >= n_trees) return;
  const size_t tb = (size_t)tree * a.M, ro = (size_t)tree * a.A;
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  int nv[SMZ_MAX_POLICY];
  double cq[SMZ_MAX_POLICY];
  bool legal[SMZ_MAX_POLICY];
  int sn = 0, mn = 0;
  double spq = 0.0, sp = 0.0;
  for (int i = 0; i < a.A; ++i) {
    const int4 st = a.stat[tb + 1 + i];
    legal[i] = a.link[tb + 1 + i].y >= 0;
    nv[i] = legal[i] ? st.x : 0;
    cq[i] = 0.0;
    if (!legal[i]) continue;
    sn += st.x;
    mn = max(mn, st.x);
    if (st.x > 0) {
      const float q = __fadd_rn(__int_as_float(st.z), __fmul_rn(a.discount, __fdiv_rn(__int_as_float(st.y), (float)st.x)));
      const double p = a.root_prior[ro + i];
      cq[i] = (double)q;
      spq = __dadd_rn(spq, __dmul_rn(p, (double)q));
      sp = __dadd_rn(sp, p);
    }
  }
  const double vhat = (double)a.raw_value[(size_t)tree * (a.N + 1)];
  const double vmix = sn == 0 ? vhat
                              : __ddiv_rn(__dadd_rn(vhat, __ddiv_rn(__dmul_rn((double)sn, spq), sp)), (double)(sn + 1));
  double lo = inf, hi = -inf;
  for (int i = 0; i < a.A; ++i) {
    if (!legal[i]) continue;
    if (nv[i] == 0) cq[i] = vmix;
    lo = fmin(lo, cq[i]);
    hi = fmax(hi, cq[i]);
  }
  const double scale = __dmul_rn(__dadd_rn(a.c_visit, (double)mn), a.c_scale), range = fmax(__dsub_rn(hi, lo), 1e-8);
  int best = -1;
  double bs = -inf, zmax = -inf;
  for (int i = 0; i < a.A; ++i) {
    if (!legal[i]) continue;
    const double sigma = __dmul_rn(scale, __ddiv_rn(__dsub_rn(cq[i], lo), range));
    const double z = __dadd_rn(a.root_logit[ro + i], sigma);
    cq[i] = z;                                             // from here on: logit + sigma
    zmax = fmax(zmax, z);
    const double s = __dadd_rn(__dadd_rn(a.gumbel_g[ro + i], a.root_logit[ro + i]), sigma);
    if (nv[i] == mn && (best < 0 || s > bs)) { best = i; bs = s; }
  }
  if (actions) actions[tree] = best;
  if (gumbels)
    for (int i = 0; i < a.A; ++i) gumbels[ro + i] = a.gumbel_g[ro + i];
  if (!improved) return;
  double se = 0.0;
  for (int i = 0; i < a.A; ++i)
    if (legal[i]) { cq[i] = exp(__dsub_rn(cq[i], zmax)); se = __dadd_rn(se, cq[i]); }
  for (int i = 0; i < a.A; ++i) improved[ro + i] = legal[i] ? __ddiv_rn(cq[i], se) : 0.0;
}

template <int G>
int grid_for(int n_trees, int threads) { return (int)(((long long)n_trees * G + threads - 1) / threads); }

}  // namespace

#define SMZ_DISPATCH_G(G_, CALL)        \
  switch (G_) {                         \
    case 2: { constexpr int G = 2; CALL; } break;   \
    case 4: { constexpr int G = 4; CALL; } break;   \
    case 8: { constexpr int G = 8; CALL; } break;   \
    case 16: { constexpr int G = 16; CALL; } break; \
    default: { constexpr int G = 32; CALL; } break; \
  }
// lane width and search rule (V = a.gumbel) of the per-simulation tree kernels
#define SMZ_DISPATCH_GV(G_, V_, CALL)                                        \
  if (V_) { constexpr bool V = true; SMZ_DISPATCH_G(G_, CALL); }             \
  else { constexpr bool V = false; SMZ_DISPATCH_G(G_, CALL); }
// ... and per-tree budgets (U = a.budgeted)
#define SMZ_DISPATCH_GVU(G_, V_, U_, CALL)                                   \
  if (U_) { constexpr bool U = true; SMZ_DISPATCH_GV(G_, V_, CALL); }        \
  else { constexpr bool U = false; SMZ_DISPATCH_GV(G_, V_, CALL); }

static const int kThreads = 128;

void smz_launch_root_expand(const SmzArena& a, int lanes, int n_trees, const float* policy, int pstride,
                            const int* root_to_play, int train, const double* dirichlet, const uint32_t* legal,
                            const int* budget, const unsigned char* explore, cudaStream_t s) {
  SMZ_DISPATCH_G(lanes, (k_root_expand<G><<<grid_for<G>(n_trees, kThreads), kThreads, 0, s>>>(
                            a, n_trees, policy, pstride, root_to_play, train, dirichlet, legal, budget, explore)));
}

void smz_launch_select(const SmzArena& a, int lanes, int n_trees, int sim, int* o_slot, int* o_action, int* o_branch,
                       cudaStream_t s) {
  SMZ_DISPATCH_GVU(lanes, a.gumbel, a.budgeted, (k_select<G, V, U><<<grid_for<G>(n_trees, kThreads), kThreads, 0, s>>>(
                                       a, n_trees, sim, o_slot, o_action, o_branch)));
}

void smz_launch_expand_backup(const SmzArena& a, int lanes, int n_trees, int sim, const float* policy, int pstride,
                              const float* value, const float* reward, cudaStream_t s) {
  SMZ_DISPATCH_GVU(lanes, a.gumbel, a.budgeted, (k_expand_backup<G, V, U><<<grid_for<G>(n_trees, kThreads), kThreads, 0, s>>>(
                                       a, n_trees, sim, policy, pstride, value, reward)));
}

// shared-memory mirror: node records of (trees per block) trees + tables must fit; SMZ_NO_TREE_SMEM=1 keeps the
// arena-only kernel
static int rcp_entries(const SmzArena& a) { return a.N + 3 > SMZ_MAX_POLICY + 1 ? a.N + 3 : SMZ_MAX_POLICY + 1; }
static size_t mirror_bytes(const SmzArena& a, int lanes) {
  return smz_mirror_bytes(kThreads / lanes, a.M, a.A, rcp_entries(a), a.N + 2);
}

bool smz_tree_mirror_fits(const SmzArena& a, int lanes) {
  const bool off = getenv("SMZ_NO_TREE_SMEM") != nullptr;     // read per launch (launches are graph-captured): tests toggle it
  return !off && mirror_bytes(a, lanes) <= 96 * 1024;
}

// The mirror kernel is the low-latency variant (one block of 128 threads per SM or two); with more blocks per SM the
// arena-only kernel wins on occupancy (measured on B200, cfg-2 shapes, round 2: 8192 trees = 256 blocks 1.53 ms with the
// mirror vs 1.78 ms without; 12288 trees = 384 blocks 2.07 vs 1.84 ms; 16384 trees 2.30 vs 1.85 ms).
static bool mirror_pays(int blocks) {
  static int sms_of[64] = {0};      // per device: engines of one process may live on different GPUs
  int dev = 0;
  cudaGetDevice(&dev);
  int& sms = sms_of[dev & 63];
  if (!sms && (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)) sms = 148;
  static const int per_sm = getenv("SMZ_MIRROR_BLOCKS_PER_SM") ? atoi(getenv("SMZ_MIRROR_BLOCKS_PER_SM")) : 2;   // tuning switch
  return blocks <= per_sm * sms;
}

void smz_launch_backup_select(const SmzArena& a, int lanes, int n_trees, int sim, bool pdl, cudaStream_t s) {
  if (smz_tree_mirror_fits(a, lanes) && mirror_pays((n_trees * lanes + kThreads - 1) / kThreads)) {
    const size_t smem = mirror_bytes(a, lanes);
    SMZ_DISPATCH_GVU(lanes, a.gumbel, a.budgeted,
                    (cudaFuncSetAttribute((const void*)k_backup_select_sm<G, V, U>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem),
                     getenv("SMZ_NO_CARVEOUT") ? cudaSuccess :
                     cudaFuncSetAttribute((const void*)k_backup_select_sm<G, V, U>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                          cudaSharedmemCarveoutMaxShared),
                     smz_launch(k_backup_select_sm<G, V, U>, dim3(grid_for<G>(n_trees, kThreads)), dim3(kThreads), smem, s, pdl,
                                a, n_trees, sim, rcp_entries(a))));
    return;
  }
  SMZ_DISPATCH_GVU(lanes, a.gumbel, a.budgeted, (smz_launch(k_backup_select<G, V, U>, dim3(grid_for<G>(n_trees, kThreads)), dim3(kThreads), 0,
                                               s, pdl, a, n_trees, sim)));
}

void smz_launch_read_roots(const SmzArena& a, int n_trees, int* visits, float* values, double* priors, float* rewards,
                           int* error_out, cudaStream_t s) {
  const int n = n_trees * a.A;
  k_read_roots<<<(n + 255) / 256, 256, 0, s>>>(a, n_trees, visits, values, priors, rewards, error_out);
}

void smz_launch_select_actions(const SmzArena& a, int n_trees, double temperature, const double* u, int* actions,
                               double* policy, double* stored, cudaStream_t s) {
  k_select_actions<<<(n_trees + 127) / 128, 128, 0, s>>>(a, n_trees, temperature, u, actions, policy, stored);
}

// start of a search: the per-simulation row counters, the error flag and the depth statistic in ONE launch (three
// memsets cost three host enqueues before the first real kernel of a move)
__global__ void k_begin_search(SmzArena a) {
  for (int i = threadIdx.x; i < (a.N + 1) * 2; i += blockDim.x) a.branch_count[i] = 0;
  if (threadIdx.x == 0) { *a.error_flag = 0; *a.depth_sum = 0ull; }
}
void smz_launch_begin_search(const SmzArena& a, cudaStream_t s) { k_begin_search<<<1, 128, 0, s>>>(a); }

__global__ void k_set_seed(unsigned long long* dst, unsigned long long seed, unsigned long long tree_id_offset) {
  dst[0] = seed;
  dst[1] = tree_id_offset;
}
// stream-ordered update of the device-resident Philox key: the values travel as kernel arguments (no host buffer
// whose lifetime would need a synchronisation)
void smz_launch_set_seed(unsigned long long* dst, unsigned long long seed, unsigned long long tree_id_offset, cudaStream_t s) {
  k_set_seed<<<1, 1, 0, s>>>(dst, seed, tree_id_offset);
}

void smz_launch_dirichlet(const SmzArena& a, int n_trees, const uint32_t* legal, int train, const int* budget,
                          const unsigned char* explore, cudaStream_t s) {
  k_dirichlet<<<(n_trees + 127) / 128, 128, 0, s>>>(a, n_trees, legal, train, budget, explore);
}

void smz_launch_gumbel_root(const SmzArena& a, int n_trees, const float* root_value, int train, const double* given,
                            const unsigned char* explore, cudaStream_t s) {
  k_gumbel_root<<<(n_trees + 127) / 128, 128, 0, s>>>(a, n_trees, root_value, train, given, explore);
}

void smz_launch_read_gumbel(const SmzArena& a, int n_trees, int* actions, double* improved, double* gumbels,
                            cudaStream_t s) {
  k_read_gumbel<<<(n_trees + 127) / 128, 128, 0, s>>>(a, n_trees, actions, improved, gumbels);
}
