// smz_common.cuh — shared device/host definitions of the search engine (sm_100a).
//
// Arena ("structure of arrays" of vectorised columns, one slice per tree):
//   stat [B][M] int4   {visit_count i32, value_sum f32, reward f32, prior f32}   Node, mcts.py:6-21
//   link [B][M] int2   {child_base i32 (0 = not expanded), key i32}
//   root_prior [B][A] f64   priors of the root children after Dirichlet mixing (f64 in the reference)
//   minmax [B] float2  MinMaxStats, mcts.py:24-36
//   budget [B] int     simulations of each tree, in [0, N] (N unless the root step was given budgets)
//   hidden [N+1][B][Sp] f32  hidden state of every expanded node: slot 0 = root, slot s+1 = sim s
//   raw_value [B][N+1] f32   network value of every expanded node by the same slot (Gumbel searches only)
// Node 0 is the root, 1..A its children, simulation s allocates its children at 1 + A + s*Kmax, so a
// node's child_base also names the hidden slot of the node (no allocator, no counters).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define SMZ_BRANCH_AFTERSTATE 0
#define SMZ_BRANCH_DYNAMICS 1
#define SMZ_MAX_POLICY 32   // widest policy head handled by the lane-per-entry tree kernels
#define SMZ_HP 128          // padded hidden width of the MLP tiles
#define SMZ_SP 64           // padded state width
#define SMZ_MAX_OBS 8192    // widest observation of the MLP family (an 84 x 84 frame flattened is 7056)
#define SMZ_VISION_SP 160   // hidden-row stride of the vision family: 3*7*7 = 147 floats padded to 160

struct SmzArena {
  // shape
  int B, N, A, C, K, Kd, Kc, Kmax, M, W, Sp, path_stride, n_phases;
  int row_cap, row_top;   // compacted-row arrays: row_cap positions per parity; the current search uses [0, row_top)
  int kind_shift;         // node kind at depth d = (d >> kind_shift) & 1 (1 = chance): 1 = reference F,F,T,T,...  0 = paper F,T,F,T,...
  // tree columns
  int4* stat;
  int2* link;
  double* root_prior;
  float2* minmax;
  int* ucursor;
  int* root_to_play;
  int budgeted;     // 1: the current search was given budgets; selects the BUDGET instantiations of the tree kernels
  int* budget;      // [B] simulations of each tree (smz_set_root_budgets; N without): tree b takes part in simulation s
                    // iff s < budget[b].  Written by the root step only, so the captured simulation graph stays valid.
  unsigned char* explore_in;  // [B] staging of the next root step's exploration flags (smz_set_root_budgets)
  // per-simulation scratch
  int4* path;       // [B][path_stride] per level {node, visit_count, value_sum, reward} captured by the descent
  int* path_len;    // [B]
  int* leaf_node;   // [B]
  int* leaf_slot;   // [B] hidden slot of search_path[-2]
  int* leaf_action; // [B] history[-1]
  int* leaf_branch; // [B]
  int* branch_count; // [N+1][2] rows per branch of each simulation
  // compacted rows of a simulation, double-buffered by simulation parity (the descent of sim s+1 may run in
  // the tail of the kernel that still gathers sim s in another CTA): index smz_row_index(a, sim, branch, row).
  // ONE array of row_top positions per parity: afterstate rows grow upward from 0, dynamics rows downward from
  // row_top - 1.  row_top = (ceil(trees / 512) + 1) * 512, so a tile of 32 / 64 / 128 positions or a group of 2 / 4 tiles never
  // holds rows of both branches and a network CTA can request its positions before the branch counts are known.
  int* rows;        // [2 parities][row_cap] tree ids
  int4* rows4;      // same order: {tree, parent hidden slot, action, 0} — one load per gathered row
  uint4* xin;       // same order, tensor-core networks only (else null): the parent's hidden row (xin_q x 16 B), copied by
                    // the descent so that the network step gathers with ONE dependent load instead of two
  int xin_q;        // 16-byte pieces per hidden row: 8 (64 bf16) or 16 (64 fp16 hi + 64 fp16 lo, SMZ_NET_TC32)
  int* error_flag;  // [1]
  unsigned long long* depth_sum;  // [1] sum of leaf depths (bench bookkeeping)
  long long* dbg;   // debug clock stamps (null unless SMZ_TREE_TIMELINE is set)
  // network I/O
  float* out_policy;  // [B][W]
  float* out_value;   // [B]
  float* out_reward;  // [B]
  float* hidden;      // [N+1][B][Sp]
  double* dirichlet;  // [B][A]
  // record
  float* rec_policy;  // [B][N][W] or null
  float* rec_value;   // [B][N]
  float* rec_reward;  // [B][N]
  signed char* rec_branch;  // [B][N]
  float* rec_root_policy;   // [B][W]
  // rng
  int rng_mode;
  const double* tape_u;
  int tape_stride;
  const unsigned long long* seed_state;  // device [2]: {Philox key, global id of local tree 0}
  // constants
  const double* pbc;         // [N+2]: sqrt(n) * (log((n + base + 1)/base) + init)
  const double* rcp64;       // [N+3]: correctly rounded 1/n (n >= 1): exact small-integer divisions without DDIV
  const float* rcp32;        // [N+3]: the same in float32
  const signed char* sign;   // [n_phases][N+2]
  float discount;
  float one_minus_frac_f32;  // f32(1 - frac), the weak-scalar cast the reference performs
  double frac;
  double alpha;
  // Gumbel MuZero search (smz_set_search): null / 0 unless a Gumbel search has been rooted on this engine.  The tree
  // kernels take the mode as a template argument; these columns are only read or written by the Gumbel instantiations.
  int gumbel;                // 1: the current search uses the Gumbel rule at decision nodes
  int gumbel_m;              // max_considered_actions
  double c_visit, c_scale;
  float* raw_value;          // [B][N+1] the network value of every expanded node, by hidden slot (slot 0 = root)
  double* gumbel_g;          // [B][A] the root's Gumbels (0 for illegal actions)
  double* root_logit;        // [B][A] log(prior) - max over legal log(prior) at the root (0 for illegal actions)
  const int* cv_table;       // [N + 1][SMZ_MAX_POLICY + 1][max(N, 1)] considered visits of Sequential Halving,
                             // T_budget[n][sum of N]: each tree follows the schedule of its own budget
  const int* cv_table_n;     // cv_table's slice of budget N: the schedule of every tree of a search without budgets
};

#ifdef __CUDACC__
// debug (SMZ_TREE_TIMELINE=1): wall-clock stamps per simulation in a.dbg[8 + 4 sim + k]: k = 0 / 2 first wait-return of
// the tree / network step, k = 1 / 3 last block end of the tree / network step (atomicMin / atomicMax over the blocks)
__device__ __forceinline__ unsigned long long smz_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void smz_stamp_min(long long* dbg, int sim, int k) {
  if (dbg && threadIdx.x == 0) atomicMin(reinterpret_cast<unsigned long long*>(dbg) + 8 + 4 * sim + k, smz_globaltimer());
}
__device__ __forceinline__ void smz_stamp_max(long long* dbg, int sim, int k) {
  if (dbg && threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned long long*>(dbg) + 8 + 4 * sim + k, smz_globaltimer());
}
__device__ __forceinline__ size_t smz_row_index(const SmzArena& a, int sim, int branch, int row) {
  return (size_t)(sim & 1) * a.row_cap + (branch ? a.row_top - 1 - row : row);
}
// Programmatic dependent launch (PDL): `smz_pdl_wait` blocks until the preceding kernel of the stream has
// completed and its writes are visible (no-op when the launch carries no programmatic dependency);
// `smz_pdl_launch_dependents` lets the next kernel's CTAs become resident and run their prologue.
__device__ __forceinline__ void smz_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void smz_pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t smz_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
                              Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
// ---------------------------------------------------------------------------------------------
// Philox4x32-10, counter = (index>>1, stream, tree_lo, tree_hi), key = (seed_lo, seed_hi)
// (restated on the CPU in oracle/mcts_oracle.py::philox_uniform)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 smz_philox(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ double smz_philox_uniform(unsigned long long seed, unsigned long long tree,
                                                     unsigned index, unsigned stream) {
  uint4 r = smz_philox(make_uint4(index >> 1, stream, (unsigned)tree, (unsigned)(tree >> 32)),
                       make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
  unsigned a = (index & 1) ? r.z : r.x, b = (index & 1) ? r.w : r.y;
  // numpy random_sample: ((a>>5)*2^26 + (b>>6)) / 2^53 — exact in double
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// per-thread view of the uniform source: the Philox key is read from device memory ONCE per kernel
struct SmzRng {
  int mode, stride;
  const double* tape;
  unsigned long long seed, tree0;
  int* err;
  // optional window of uniforms [win_base, win_base + win_len) of THIS thread's tree, generated ahead of time
  // (k_backup_select_sm fills it while the network step is still running)
  const double* win;
  int win_base, win_len;
};
__device__ __forceinline__ SmzRng smz_make_rng(const SmzArena& a) {
  SmzRng r;
  r.mode = a.rng_mode; r.stride = a.tape_stride; r.tape = a.tape_u; r.err = a.error_flag;
  r.seed = a.rng_mode ? 0ull : a.seed_state[0];
  r.tree0 = a.rng_mode ? 0ull : a.seed_state[1];
  r.win = nullptr; r.win_base = 0; r.win_len = 0;
  return r;
}
__device__ __forceinline__ double smz_rng_uniform(const SmzRng& r, int tree, int idx) {
  if (r.mode) {
    if (idx >= r.stride) { *r.err = 1; return 0.5; }
    return r.tape[(size_t)tree * r.stride + idx];
  }
  if (r.win && (unsigned)(idx - r.win_base) < (unsigned)r.win_len) return r.win[idx - r.win_base];
  return smz_philox_uniform(r.seed, r.tree0 + (unsigned long long)tree, (unsigned)idx, 0u);
}

// Exact division through a correctly rounded reciprocal (Markstein): q = RN(x*r), rem = x - q*d (exact, one FMA),
// RN(q + rem*r) == RN(x/d) whenever r == RN(1/d), q is faithful and d's significand is not all ones — true for
// the small integers (visit counts, child counts) tabulated in rcp64 / rcp32.  Three dependent instructions
// instead of the ~40 of a software DDIV; checked against IEEE division in tests/test_host_logic.py.
__device__ __forceinline__ double smz_div_r64(double x, double d, double r) {
  const double q = __dmul_rn(x, r);
  return __fma_rn(__fma_rn(-q, d, x), r, q);
}
__device__ __forceinline__ float smz_div_r32(float x, float d, float r) {
  const float q = __fmul_rn(x, r);
  return __fmaf_rn(__fmaf_rn(-q, d, x), r, q);
}
#endif
