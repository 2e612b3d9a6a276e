// smz_tree_dev.cuh — device-side tree phases of the tree kernels (smz_tree.cu).  Everything that decides a visit order uses
// explicit round-to-nearest intrinsics, so the translation unit's -fmad setting does not matter here.
#pragma once
#include "smz_common.cuh"

namespace smz_tree_dev {

#define FULL 0xffffffffu

// Every kernel below keeps all 32 lanes of a warp converged: loops run for the warp-wide maximum trip
// count and per-group work is predicated, so every shuffle / ballot is a full-mask, constant-mask
// instruction on sub-warp segments of width G (no mask matching, no dependence on independent
// thread scheduling).  Trees beyond n_trees keep their lanes alive with `alive == false`.
template <int G>
struct Group {
  int lane, gl, gbase;
  __device__ Group() {
    lane = threadIdx.x & 31;
    gl = lane & (G - 1);
    gbase = lane & ~(G - 1);
  }
  template <typename T>
  __device__ T bcast(T v, int src) const { return __shfl_sync(FULL, v, src, G); }
  __device__ unsigned ballot(bool p) const {
    unsigned b = __ballot_sync(FULL, p);
    return (G == 32) ? b : ((b >> gbase) & ((1u << G) - 1u));
  }
};

// numpy float32 add.reduce over n values held one per lane (n may differ between the groups of a
// warp): pairwise summation with an 8-way unrolled block (n >= 8) or a plain loop from 0.f (n < 8)
// — numpy/_core/src/umath/loops_utils.h.src.  Trip counts are compile-time (G), adds are predicated.
template <int G>
__device__ float np_sum_f32(const Group<G>& g, float a, int n) {
  float seq = 0.f;
#pragma unroll
  for (int i = 0; i < (G < 7 ? G : 7); ++i) {
    const float v = g.bcast(a, i);
    if (i < n) seq = __fadd_rn(seq, v);
  }
  if (G < 8) return seq;
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = g.bcast(a, j & (G - 1));
  const int nb = n - (n % 8);
#pragma unroll
  for (int i = 8; i + 8 <= G; i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = g.bcast(a, (i + j) & (G - 1));
      if (i < nb) r[j] = __fadd_rn(r[j], v);
    }
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
#pragma unroll
  for (int t = 0; t < 7; ++t) {
    const float v = g.bcast(a, (nb + t) & (G - 1));
    if (nb + t < n) res = __fadd_rn(res, v);
  }
  return n < 8 ? seq : res;
}

// cdf of RandomState.choice: float64 cumsum of p (sequential), divided by the last entry.  The DIVISION is what costs
// (a float64 IEEE division is a ~40-instruction dependent chain) and its result is only ever COMPARED with a uniform
// draw, so the phases keep every entry as numerator / total and decide `RN(num / total) <= u` in float32 whenever that
// is safe: cf = num / total in float32 is within 3e-7 of the float64 quotient, so |cf - u| > 2e-6 settles the comparison;
// a closer call (probability ~4e-6 per comparison) takes the exact division.
// choice_cdf_raw: every lane i < n returns cumsum[i] (lanes >= n: 0) and `total` = cumsum[n-1] for the whole group.
template <int G>
__device__ double choice_cdf_raw(const Group<G>& g, double p, int n, double& total) {
  double acc = 0.0, mine = 0.0;
  if constexpr (G >= 16) {
    // Wide groups: inclusive scan by doubling (log2 G steps instead of G).  A sum of float32-born values is usually
    // EXACT in float64 (24-bit significands, 53 available), and exact partial sums do not depend on the order of the
    // additions — so whenever every addition of the scan is exact (TwoSum error term zero), the scan equals numpy's
    // sequential cumsum bit for bit.  Any inexact addition anywhere in the warp -> the sequential loop below.
    double sc = p;
    bool inexact = false;
#pragma unroll
    for (int off = 1; off < G; off <<= 1) {
      const double o = __shfl_up_sync(FULL, sc, off, G);
      if (g.gl >= off) {
        const double t = __dadd_rn(sc, o);
        const double bv = __dsub_rn(t, sc);
        const double err = __dadd_rn(__dsub_rn(sc, __dsub_rn(t, bv)), __dsub_rn(o, bv));
        inexact |= err != 0.0;
        sc = t;
      }
    }
    if (!__any_sync(FULL, inexact)) {
      total = g.bcast(sc, G - 1);            // lanes >= n hold p = 0: the last lane carries the total
      return sc;
    }
  }
#pragma unroll
  for (int i = 0; i < G; ++i) {
    acc = __dadd_rn(acc, g.bcast(p, i));     // + 0.0 beyond n leaves acc unchanged
    if (g.gl == i) mine = acc;
  }
  total = acc;
  return mine;
}
constexpr float SMZ_CDF_MARGIN = 2e-6f;
// this lane's cdf entry in float32 (lanes >= n: 3.0 — above every uniform and every "no draw" marker)
__device__ __forceinline__ float cdf_f32(double num, double total, bool in_range) {
  return in_range ? __fdividef((float)num, (float)total) : 3.f;
}
__device__ __forceinline__ double cdf_exact(double num, double total, bool in_range) {
  return in_range ? __ddiv_rn(num, total) : 2.0;
}

// searchsorted(cdf, u, side='right') = #{i : cdf[i] <= u} for the non-decreasing cdf held one entry per lane
// (num / total, lanes >= n never count); u may differ per lane.  The count never reaches G (cdf[n-1] = 1 > u).
template <int G>
__device__ int searchsorted_right(const Group<G>& g, double num, double total, int n, double u) {
  const float cf = cdf_f32(num, total, g.gl < n), uf = (float)u;
  int cnt = 0;
  bool close = false;
  if constexpr (G >= 16) {
#pragma unroll
    for (int step = G / 2; step >= 1; step >>= 1) {
      const float cv = g.bcast(cf, cnt + step - 1);
      close |= fabsf(cv - uf) <= SMZ_CDF_MARGIN;
      if (cv < uf) cnt += step;
    }
  } else {
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const float cv = g.bcast(cf, i);
      close |= fabsf(cv - uf) <= SMZ_CDF_MARGIN;
      cnt += cv < uf;
    }
  }
  if (__any_sync(FULL, close)) {             // rare: some comparison of the warp is too close for float32
    const double c = cdf_exact(num, total, g.gl < n);
    cnt = 0;
    if constexpr (G >= 16) {
#pragma unroll
      for (int step = G / 2; step >= 1; step >>= 1) {
        const double cv = g.bcast(c, cnt + step - 1);
        if (cv <= u) cnt += step;
      }
    } else {
#pragma unroll
      for (int i = 0; i < G; ++i) cnt += g.bcast(c, i) <= u;
    }
  }
  return cnt;
}

// (policy + 1e-12) / sum in float32 (mcts.py:205-206, :291-292); lanes >= n hold 0.
template <int G>
__device__ float normalise_policy(const Group<G>& g, float pol, int n) {
  const float p = (g.gl < n) ? __fadd_rn(pol, 1e-12f) : 0.f;
  const float s = np_sum_f32(g, p, n);
  return (g.gl < n) ? __fdiv_rn(p, s) : 0.f;
}

// np.random.choice(n, bound, p=p, replace=False): returns the bit set of chosen indices and advances
// the tree's uniform cursor by the number of draws numpy would have consumed.
// numpy (mtrand.pyx, the replace=False branch) loops: draw m = bound - found uniforms, zero the found entries of p,
// cdf = cumsum(p) / cumsum(p)[-1], new = searchsorted(cdf, x, 'right'), keep the not-yet-found values.  Which values a
// round adds does not depend on the order of its draws (the result is sorted afterwards, mcts.py:208/:294), so the m
// draws of a round are handled by m lanes at once: lane j generates uniform `cursor + j`, counts the cdf entries <= u
// (searchsorted), and the new indices are OR-reduced over the group.  The cdf itself keeps numpy's sequential order of
// additions.
template <int G>
__device__ unsigned choice_without_replacement(const Group<G>& g, const SmzArena& a, const SmzRng& rng, bool alive, int tree,
                                               float p32, int n, int bound, int& cursor) {
  unsigned found = 0;
  int nf = alive ? 0 : bound;
  // np.random.choice validates p first ("probabilities contain NaN" / "are not non-negative"): ValueError in the reference
  if (g.ballot(alive && g.gl < n && !(p32 >= 0.f))) {
    if (alive) *a.error_flag = 2;
    found = bound >= 32 ? 0xffffffffu : ((1u << bound) - 1u);
    nf = bound;
  }
  const double pd = (g.gl < n) ? (double)p32 : 0.0;
  for (int round = 0; __any_sync(FULL, nf < bound); ++round) {
    if (round > 2 * SMZ_MAX_POLICY) {   // degenerate policy: do not hang
      if (nf < bound) {
        *a.error_flag = 2;
        for (int i = 0; i < n && nf < bound; ++i)
          if (!((found >> i) & 1u)) { found |= 1u << i; ++nf; }
      }
      break;
    }
    const int m = bound - nf;                    // 0 for groups that are done; m <= bound <= n <= G
    double total;
    const double num = choice_cdf_raw(g, ((found >> g.gl) & 1u) ? 0.0 : pd, n, total);
    const bool on = g.gl < m;
    double u = 2.0;                              // lanes without a draw never match
    if (__any_sync(FULL, on)) {
      if (on) u = smz_rng_uniform(rng, tree, cursor + g.gl);
    }
    const int cnt = searchsorted_right(g, num, total, n, u);   // entries of lanes >= n never count
    const int idx = cnt < n ? cnt : n - 1;
    unsigned bits = on ? (1u << idx) : 0u;
#pragma unroll
    for (int off = G / 2; off > 0; off >>= 1) bits |= __shfl_xor_sync(FULL, bits, off, G);
    found |= bits;
    nf = alive ? __popc(found) : bound;
    cursor += m;
  }
  return found;
}


// uniform #uidx of the tree for the lanes that `want` one; the draw only depends on the index, and a window of draws may
// have been generated ahead (SmzRng::win)
__device__ __forceinline__ double draw_uniform(const SmzRng& rng, int tree, int uidx, bool want) {
  const unsigned wofs = (unsigned)(uidx - rng.win_base);
  const bool hit = rng.win != nullptr && wofs < (unsigned)rng.win_len;
  double u = hit ? rng.win[wofs] : 0.0;
  if (__any_sync(FULL, want && !hit)) {
    if (want && !hit) u = smz_rng_uniform(rng, tree, uidx);
  }
  return u;
}

// ------------------------------------------------------------------------------------------------
// Gumbel MuZero decision rule (Danihelka et al., ICLR 2022; smz_set_search in include/smz.h), one lane per child.
// float64 sum over the lanes in ascending order, as a sequential loop adds; lanes that take no part hold +0.0, which
// leaves the sum unchanged (a sum that starts at +0.0 never becomes -0.0 under round-to-nearest).
template <int G>
__device__ __forceinline__ double seq_sum_f64(const Group<G>& g, double x) {
  double acc = 0.0;
#pragma unroll
  for (int i = 0; i < G; ++i) acc = __dadd_rn(acc, g.bcast(x, i));
  return acc;
}

// sigma_i = (c_visit + max N) * c_scale * r_i of the completed Q-values, for the lanes `on` (the node's existing
// children: visit count n, prior p, q = reward + discount * value() in float32); the node's own network value is vhat.
template <int G>
__device__ __forceinline__ double gumbel_sigma(const Group<G>& g, const SmzArena& a, bool on, int n, double p, float q,
                                               double vhat, int& sum_n) {
  int sn = on ? n : 0, mn = sn;
#pragma unroll
  for (int off = G / 2; off > 0; off >>= 1) {
    sn += __shfl_xor_sync(FULL, sn, off, G);
    mn = max(mn, __shfl_xor_sync(FULL, mn, off, G));
  }
  const bool vis = on && n > 0;
  const double qd = (double)q;
  const double spq = seq_sum_f64(g, vis ? __dmul_rn(p, qd) : 0.0);
  const double sp = seq_sum_f64(g, vis ? p : 0.0);
  // v_mix = (vhat + sum N * (sum p q) / (sum p)) / (sum N + 1), left to right
  const double vmix = sn == 0 ? vhat
                              : __ddiv_rn(__dadd_rn(vhat, __ddiv_rn(__dmul_rn((double)sn, spq), sp)), (double)(sn + 1));
  const double cq = vis ? qd : vmix;
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double lo = on ? cq : inf, hi = on ? cq : -inf;
#pragma unroll
  for (int off = G / 2; off > 0; off >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(FULL, lo, off, G));
    hi = fmax(hi, __shfl_xor_sync(FULL, hi, off, G));
  }
  const double r = __ddiv_rn(__dsub_rn(cq, lo), fmax(__dsub_rn(hi, lo), 1e-8));
  sum_n = sn;
  return on ? __dmul_rn(__dmul_rn(__dadd_rn(a.c_visit, (double)mn), a.c_scale), r) : 0.0;
}

// The child a decision node descends to under the Gumbel rule; no uniform is drawn.  Root (lanes = actions, `act` = a
// legal child): argmax over the children whose visit count is the considered count T[min(m, |L|)][sum N] of
// max(-1e9, g + logit + sigma).  Elsewhere: argmax of pi'_i - N_i / (1 + sum N), pi' = softmax-weighted priors
// p_i exp(sigma_i - max sigma) / sum.  Ties go to the smaller action; a root with no child at the considered count
// (the schedule rules it out) takes its first legal child.  T is the schedule of the tree's budget `bud` (-1: a search
// without budgets, T_N).
template <int G>
__device__ __forceinline__ int gumbel_pick(const Group<G>& g, const SmzArena& a, int tree, bool going, bool act, bool root,
                                           int4 st, double prior_root, double gum, double lgt, int cbase, int width, int bud) {
  const int slot = (root || !going) ? 0 : (cbase - 1 - a.A) / a.Kmax + 1;     // a group that stopped reads slot 0
  const double vhat = (double)a.raw_value[(size_t)tree * (a.N + 1) + slot];
  const double p = root ? prior_root : (double)__int_as_float(st.w);
  float q = 0.f;
  if (act && st.x > 0) {
    const float val = smz_div_r32(__int_as_float(st.y), (float)st.x, a.rcp32[st.x]);
    q = __fadd_rn(__int_as_float(st.z), __fmul_rn(a.discount, val));
  }
  int sum_n;
  const double sigma = gumbel_sigma(g, a, act, st.x, p, q, vhat, sum_n);
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double score = -inf;
  int best = act ? g.gl : 64;
  if (root) {
    const int n_cons = min(a.gumbel_m, width);
    const int* T = bud < 0 ? a.cv_table_n : a.cv_table + (size_t)bud * (SMZ_MAX_POLICY + 1) * a.N;
    const int considered = T[n_cons * a.N + min(sum_n, a.N - 1)];
    if (act && st.x == considered) score = fmax(-1e9, __dadd_rn(__dadd_rn(gum, lgt), sigma));
  } else {
    double ms = act ? sigma : -inf;
#pragma unroll
    for (int off = G / 2; off > 0; off >>= 1) ms = fmax(ms, __shfl_xor_sync(FULL, ms, off, G));
    const double w = act ? __dmul_rn(p, exp(__dsub_rn(sigma, ms))) : 0.0;
    const double sw = seq_sum_f64(g, w);
    if (act) score = __dsub_rn(__ddiv_rn(w, sw), __ddiv_rn((double)st.x, (double)(1 + sum_n)));
  }
#pragma unroll
  for (int off = G / 2; off > 0; off >>= 1) {
    const double os = __shfl_xor_sync(FULL, score, off, G);
    const int ob = __shfl_xor_sync(FULL, best, off, G);
    if (os > score || (os == score && ob < best)) { score = os; best = ob; }
  }
  return best < G ? best : 0;
}

// ------------------------------------------------------------------------------------------------
// Per-tree state that flows from the backup of one simulation into the descent of the next.  The fused
// kernel keeps it in registers; the stand-alone kernels load / store it.
struct TreeState {
  int cursor;      // uniform draws consumed so far
  float2 mm;       // MinMaxStats
  int2 root;       // root {visit_count, value_sum bits}
};

// The search path is kept as one int4 record per level {node, visit_count, value_sum, reward} captured
// while descending, so the backup needs ONE round trip (the record) instead of two (index -> stat).
// The tree is appended to the per-branch row list of the simulation, from which the network step tiles its leaves.
// Called by every thread of the block: the row reservation below synchronises the block.
// `alive`: the tree takes part in simulation `sim` (it exists and sim < its budget); `bud` = its budget, or -1 in a search
// without budgets (the Gumbel root's schedule).
template <int G, bool MIRROR = false, bool GUMBEL = false>
__device__ __forceinline__ void select_phase(const Group<G>& g, const SmzArena& a, const SmzRng& rng, int tree, bool alive,
                                             int bud, int sim, TreeState ts, int* __restrict__ o_slot, int* __restrict__ o_action,
                                             int* __restrict__ o_branch, const int4* __restrict__ sst = nullptr,
                                             const int2* __restrict__ slk = nullptr, const double* __restrict__ srp = nullptr) {
  const size_t tb = (size_t)tree * a.M;
  int cursor = ts.cursor;
  const float vmin = ts.mm.x, vmax = ts.mm.y;
  int4* path = a.path + (size_t)tree * a.path_stride;

  int depth = 0, cbase = 1, nch = a.A;
  int parent_visit = ts.root.x;
  // min-max normalisation divides by the same range at every level: one correctly rounded reciprocal, then
  // Markstein's exact division (smz_common.cuh); a range whose significand is all ones keeps the plain division
  const float range = __fsub_rn(vmax, vmin);
  const float rrange = vmax > vmin ? __frcp_rn(range) : 0.f;
  const bool range_plain = (__float_as_int(range) & 0x7FFFFF) == 0x7FFFFF || range < 1e-30f;
  if (alive && g.gl == 0) path[0] = make_int4(0, ts.root.x, ts.root.y, 0);
  int L = 1, child = 0, child_key = 0;
  bool going = alive;
  // the Dirichlet-mixed root priors are f64 and only used at depth 0: one load, before the loop
  const double prior0 = (alive && g.gl < a.A) ? (srp ? srp[g.gl] : a.root_prior[(size_t)tree * a.A + g.gl]) : 0.0;
  // Gumbel rule: the root's Gumbels and logits, read from the arena (L2) by both kernels
  double gum0 = 0.0, lgt0 = 0.0;
  if constexpr (GUMBEL) {
    if (alive && g.gl < a.A) {
      gum0 = a.gumbel_g[(size_t)tree * a.A + g.gl];
      lgt0 = a.root_logit[(size_t)tree * a.A + g.gl];
    }
  }
  // Every group that is still descending is at depth == level, so the node kind (and the child count) is uniform
  // across the warp: plain uniform branches instead of votes, loads and draws without divergent regions.
  int level = 0;
  while (__any_sync(FULL, going)) {
    bool act = going && g.gl < nch;
    const bool chance = (level >> a.kind_shift) & 1;
    const int ci = act ? cbase + g.gl : 0;                     // idle lanes read node 0 and discard it
    int4 st;
    int2 lk;
    if constexpr (MIRROR) {      // the tree's node records live in shared memory (k_backup_select_sm)
      st = sst[ci];
      lk = slk[ci];
    } else {
      st = a.stat[tb + ci];
      lk = a.link[tb + ci];
    }
    // The root (a decision node in both patterns) scores its legal children only: an illegal action's slot holds key -1.
    // Child j takes draw `cursor + rank of j among the legal children`, and the root consumes |L| draws.
    const bool root = level == 0;
    int width = nch;
    double pbc, u;
    if constexpr (MIRROR) {      // the node records are at hand: the draw is indexed by legal rank
      int rank = g.gl;
      if (root) {
        act = act && lk.y >= 0;
        const unsigned lm = g.ballot(act);
        rank = __popc(lm & ((1u << g.gl) - 1u));
        width = __popc(lm);
      }
      if (!act) { st = make_int4(0, 0, 0, 0); lk = make_int2(0, 0); }
      pbc = (GUMBEL || chance) ? 0.0 : a.pbc[going ? parent_visit : 0];     // plain load: the table lives in shared memory
      u = draw_uniform(rng, tree, chance ? cursor : cursor + rank, going && (chance || (!GUMBEL && act)));
    } else {
      // the node records are still in flight: the draws are taken by lane index without waiting for them, and child
      // j gets the draw of lane `rank` by a shuffle.  With a tape only lanes 0..|L|-1 draw, so the tape is read
      // exactly where the search reads it.
      pbc = (GUMBEL || chance) ? 0.0 : a.pbc[going ? parent_visit : 0];
      bool want = going && (chance || (!GUMBEL && act));     // a Gumbel decision node draws nothing
      if (!GUMBEL && root && rng.mode) {    // every lane takes part in the ballot (no short-circuit around it)
        const int n_legal = __popc(g.ballot(act && lk.y >= 0));
        want = want && g.gl < n_legal;
      }
      u = draw_uniform(rng, tree, chance ? cursor : cursor + g.gl, want);
      if (root) {
        act = act && lk.y >= 0;
        const unsigned lm = g.ballot(act);
        width = __popc(lm);
        u = g.bcast(u, __popc(lm & ((1u << g.gl) - 1u)));
      }
      if (!act) { st = make_int4(0, 0, 0, 0); lk = make_int2(0, 0); }
    }
    int pick = 0;
    if (chance) {
      // chance node: sample a child from the smoothed priors (mcts.py:249-255, T9)
      const float p = __int_as_float(st.w);
      const float om = act ? __fadd_rn(__fsub_rn(1.f, p), 1e-12f) : 0.f;
      const float rem = fabsf(smz_div_r32(np_sum_f32(g, om, nch), (float)nch, a.rcp32[nch]));
      const float sh = act ? __fadd_rn(p, rem) : 0.f;
      const float tot = np_sum_f32(g, sh, nch);
      const float q = act ? __fdiv_rn(sh, tot) : 0.f;
      double total;
      const double num = choice_cdf_raw(g, (double)q, nch, total);
      const float cf = cdf_f32(num, total, act), uf = (float)u;
      bool le = cf < uf;
      const bool close = act && fabsf(cf - uf) <= SMZ_CDF_MARGIN;
      if (__any_sync(FULL, close)) {         // rare: float32 cannot decide RN(num / total) <= u
        if (close) le = __ddiv_rn(num, total) <= u;
      }
      int pk = __popc(g.ballot(act && le));
      pk = pk < nch ? pk : nch - 1;
      if (chance) { pick = pk; cursor += going ? 1 : 0; }
    }
    if (GUMBEL && !chance) {
      pick = gumbel_pick(g, a, tree, going, act, root, st, prior0, gum0, lgt0, cbase, width, bud);
    } else if (!chance) {
      // decision node: argmax of ucb_score, one fresh uniform per child (mcts.py:235-243, T3/T5/T6)
      double score = -__longlong_as_double(0x7ff0000000000000LL);
      int best = -1;
      if (act && !chance) {
        const double prior = (level == 0) ? prior0 : (double)__int_as_float(st.w);
        // pbc = sqrt(n) * pb_c(n), the left-associated head of mcts.py:237, tabulated by the host
        const double ps = smz_div_r64(__dmul_rn(pbc, prior), (double)(st.x + 1), a.rcp64[st.x + 1]);
        double vs = 0.0;
        if (st.x > 0) {
          const float val = smz_div_r32(__int_as_float(st.y), (float)st.x, a.rcp32[st.x]);
          float v = __fadd_rn(__int_as_float(st.z), __fmul_rn(a.discount, val));
          if (vmax > vmin) v = range_plain ? __fdiv_rn(__fsub_rn(v, vmin), range) : smz_div_r32(__fsub_rn(v, vmin), range, rrange);
          vs = (double)v;
        }
        const double noise = __dadd_rn(1e-7, __dmul_rn(2e-7 - 1e-7, u));
        score = __dadd_rn(__dadd_rn(ps, vs), noise);
        best = g.gl;
      }
#pragma unroll
      for (int off = G / 2; off > 0; off >>= 1) {
        const double os = __shfl_xor_sync(FULL, score, off, G);
        const int ob = __shfl_xor_sync(FULL, best, off, G);
        if (os > score || (os == score && ob > best)) { score = os; best = ob; }
      }
      if (!chance) { pick = best < 0 ? 0 : best; cursor += going ? width : 0; }
    }
    const int4 cst = make_int4(g.bcast(st.x, pick), g.bcast(st.y, pick), g.bcast(st.z, pick), 0);
    const int child_cb = g.bcast(lk.x, pick);
    const int key = g.bcast(lk.y, pick);
    if (going) {
      child = cbase + pick;
      child_key = key;
      if (g.gl == 0) path[L] = make_int4(child, cst.x, cst.y, cst.z);
      ++L;
      if (child_cb == 0 || L >= a.path_stride) {
        going = false;
      } else {
        // the child (depth+1) was expanded through the dynamics pair iff this node is a chance node (T2)
        nch = chance ? a.Kd : a.Kc;
        parent_visit = cst.x;
        cbase = child_cb;
        ++depth;
      }
    }
    ++level;
  }
  if (a.dbg && blockIdx.x == 0 && threadIdx.x == 0) { a.dbg[4] = clock64(); a.dbg[5] = level; }
  // ---- leaf record.  The row compaction is aggregated per block (one global atomic per branch per block) and the
  //      depth statistic per warp, instead of one atomic per tree — thousands of same-address atomics per
  //      simulation serialise in the L2 and their return value is on the critical path of the kernel.
  const bool lead = alive && g.gl == 0;
  const int branch = ((depth >> a.kind_shift) & 1) ? SMZ_BRANCH_DYNAMICS : SMZ_BRANCH_AFTERSTATE;   // the leaf's parent's kind
  const int slot = (cbase == 1) ? 0 : (cbase - 1 - a.A) / a.Kmax + 1;
  // the parent's hidden row is requested now and stored once the row index is known (bf16 network: a.xin)
  uint4 hcopy[(G < 8) ? 8 / G : 1], hcopy2[(G < 8) ? 8 / G : 1];
  const bool copy_row = a.xin != nullptr && alive;
  const bool wide_row = a.xin_q > 8;          // fp16 hi + lo rows (SMZ_NET_TC32): a second batch of 8 pieces
  if (copy_row) {
    const uint4* src = reinterpret_cast<const uint4*>(a.hidden) + ((size_t)slot * a.B + tree) * a.xin_q;
#pragma unroll
    for (int j = 0; j < ((G < 8) ? 8 / G : 1); ++j) {
      const int idx = g.gl + j * G;
      hcopy[j] = idx < 8 ? src[idx] : make_uint4(0, 0, 0, 0);
      if (wide_row) hcopy2[j] = idx < 8 ? src[8 + idx] : make_uint4(0, 0, 0, 0);
    }
  }
  // warps reserve ranks in shared memory, two threads reserve the block's rows globally
  int r = 0;
  {
    const unsigned lane = threadIdx.x & 31u;
    __shared__ int s_cnt[2], s_base[2];
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const unsigned m = __ballot_sync(FULL, lead && branch == b);
      if (m) {
        const int leader = __ffs(m) - 1;
        int base = 0;
        if ((int)lane == leader) base = atomicAdd(&s_cnt[b], __popc(m));
        base = __shfl_sync(FULL, base, leader);
        if (lead && branch == b) r = base + __popc(m & ((1u << lane) - 1u));
      }
    }
    __syncthreads();
    if (threadIdx.x < 2) s_base[threadIdx.x] = s_cnt[threadIdx.x] ? atomicAdd(&a.branch_count[sim * 2 + threadIdx.x], s_cnt[threadIdx.x]) : 0;
    __syncthreads();
    r += s_base[branch];
  }
  const int rg = g.bcast(r, 0);
  if (copy_row) {
    uint4* dst = a.xin + smz_row_index(a, sim, branch, rg) * a.xin_q;
#pragma unroll
    for (int j = 0; j < ((G < 8) ? 8 / G : 1); ++j) {
      const int idx = g.gl + j * G;
      if (idx < 8) dst[idx] = hcopy[j];
      if (wide_row && idx < 8) dst[8 + idx] = hcopy2[j];
    }
  }
  {
    int dsum = lead ? depth + 1 : 0;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dsum += __shfl_xor_sync(FULL, dsum, off);
    if ((threadIdx.x & 31u) == 0 && dsum) atomicAdd(a.depth_sum, (unsigned long long)dsum);
  }
  if (lead) {
    a.leaf_node[tree] = child;
    a.leaf_slot[tree] = slot;
    a.leaf_action[tree] = child_key;
    a.leaf_branch[tree] = branch;
    a.path_len[tree] = L;
    a.ucursor[tree] = cursor;
    if (o_slot) o_slot[tree] = slot;
    if (o_action) o_action[tree] = child_key;
    if (o_branch) o_branch[tree] = branch;
    a.rows[smz_row_index(a, sim, branch, r)] = tree;
    a.rows4[smz_row_index(a, sim, branch, r)] = make_int4(tree, slot, child_key, 0);
  }
}

// ------------------------------------------------------------------------------------------------
template <int G, bool MIRROR = false, bool GUMBEL = false>
__device__ __forceinline__ TreeState expand_backup_phase(const Group<G>& g, const SmzArena& a, const SmzRng& rng, int tree,
                                                         bool alive, int sim, const float* __restrict__ policy,
                                                         int pstride, const float* __restrict__ value,
                                                         const float* __restrict__ reward, int4* __restrict__ sst = nullptr,
                                                         int2* __restrict__ slk = nullptr) {
  const size_t tb = (size_t)tree * a.M;
  // everything this phase needs from memory is requested up front (one round trip): the leaf record,
  // the network outputs, the tree state and — speculatively — the first two chunks of path records
  const int4* path = a.path + (size_t)tree * a.path_stride;
  const int4 rec0 = (g.gl < a.path_stride) ? path[g.gl] : make_int4(0, 0, 0, 0);
  const int4 rec1 = (G + g.gl < a.path_stride) ? path[G + g.gl] : make_int4(0, 0, 0, 0);
  const int leaf = a.leaf_node[tree];
  const int branch = a.leaf_branch[tree];
  const int L = alive ? a.path_len[tree] : 0;
  int cursor = a.ucursor[tree];
  float2 mm = a.minmax[tree];
  float v = value[tree];
  const float rew_in = reward[tree];
  const signed char* sign = a.sign + (size_t)a.root_to_play[tree] * (a.N + 2);

  // children of the leaf (mcts.py:289-297): width C after the afterstate pair, A after dynamics
  const int n = branch ? a.A : a.C;
  const int bound = min(a.K, n);
  const float pol = (g.gl < n) ? policy[(size_t)tree * pstride + g.gl] : 0.f;
  const float p = normalise_policy(g, pol, n);
  const unsigned found = choice_without_replacement(g, a, rng, alive, tree, p, n, bound, cursor);
  const int cb = 1 + a.A + sim * a.Kmax;
  if (alive && g.gl < n && ((found >> g.gl) & 1u)) {
    const int r = __popc(found & ((1u << g.gl) - 1u));
    a.stat[tb + cb + r] = make_int4(0, 0, 0, __float_as_int(p));
    a.link[tb + cb + r] = make_int2(0, g.gl);
    if constexpr (MIRROR) {
      sst[cb + r] = make_int4(0, 0, 0, __float_as_int(p));
      slk[cb + r] = make_int2(0, g.gl);
    }
  }
  const float rew = branch ? rew_in : 0.f;
  if (alive && g.gl == 0) {
    a.link[tb + leaf].x = cb;
    a.ucursor[tree] = cursor;
    if (branch) reinterpret_cast<int*>(a.stat + tb + leaf)[2] = __float_as_int(rew);     // Node.reward of the leaf
    if constexpr (GUMBEL) a.raw_value[(size_t)tree * (a.N + 1) + sim + 1] = v;        // the leaf's slot is sim + 1
    if constexpr (MIRROR) {
      slk[leaf].x = cb;
      if (branch) sst[leaf].z = __float_as_int(rew);
    }
    if (a.rec_policy) {
      const size_t ro = ((size_t)tree * a.N + sim);
      for (int i = 0; i < a.W; ++i) a.rec_policy[ro * a.W + i] = i < n ? policy[(size_t)tree * pstride + i] : 0.f;
      a.rec_value[ro] = v;
      a.rec_reward[ro] = rew;
      a.rec_branch[ro] = (signed char)branch;
    }
  }

  // backup leaf -> root (mcts.py:299-308): lanes own path levels, the discounted return is a serial
  // float32 recurrence (mul then add, two roundings) carried through shuffles
  int2 root = make_int2(0, 0);
  int l_max = L;                                     // longest path in the warp
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) l_max = max(l_max, __shfl_xor_sync(FULL, l_max, off));
  const int n_chunks = (l_max + G - 1) / G;
  for (int chunk = n_chunks - 1; chunk >= 0; --chunk) {
    const int l = chunk * G + g.gl;
    const bool valid = l < L;
    int4 rec = chunk == 0 ? rec0 : rec1;
    if (chunk > 1 && valid) rec = path[l];
    if (!valid) rec = make_int4(0, 0, 0, 0);
    if (valid && l == L - 1 && branch) rec.w = __float_as_int(rew);
    const float r = __int_as_float(rec.w);
    float myv = 0.f;
    if constexpr (G >= 16) {
      // wide groups: paths are much shorter than G — walk only the levels some group of the warp has
      for (int t = min(G, l_max - chunk * G) - 1; t >= 0; --t) {
        const float ri = g.bcast(r, t);
        if (chunk * G + t < L) {
          if (g.gl == t) myv = v;
          v = __fadd_rn(ri, __fmul_rn(a.discount, v));
        }
      }
    } else {
#pragma unroll
      for (int t = G - 1; t >= 0; --t) {
        const float ri = g.bcast(r, t);
        if (chunk * G + t < L) {
          if (g.gl == t) myv = v;
          v = __fadd_rn(ri, __fmul_rn(a.discount, v));
        }
      }
    }
    if (valid) {
      const float vs = __fadd_rn(__int_as_float(rec.z), (signed char)__ldg(sign + l) > 0 ? myv : -myv);
      const int2 upd = make_int2(rec.y + 1, __float_as_int(vs));
      *reinterpret_cast<int2*>(a.stat + tb + rec.x) = upd;          // {visit_count, value_sum}
      if constexpr (MIRROR) *reinterpret_cast<int2*>(sst + rec.x) = upd;
      if (l == 0) root = upd;
      const float nv = smz_div_r32(vs, (float)upd.x, a.rcp32[upd.x]);
      mm.x = fminf(mm.x, nv);
      mm.y = fmaxf(mm.y, nv);
    }
  }
#pragma unroll
  for (int off = G / 2; off > 0; off >>= 1) {
    mm.x = fminf(mm.x, __shfl_xor_sync(FULL, mm.x, off, G));
    mm.y = fmaxf(mm.y, __shfl_xor_sync(FULL, mm.y, off, G));
  }
  if (alive && g.gl == 0) a.minmax[tree] = mm;
  TreeState ts;
  ts.cursor = cursor;
  ts.mm = mm;
  ts.root = make_int2(g.bcast(root.x, 0), g.bcast(root.y, 0));   // level 0 lives in lane 0 of chunk 0
  return ts;
}


}  // namespace smz_tree_dev
