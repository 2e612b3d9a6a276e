// smz_api.cu — the C ABI of libsmz.so (include/smz.h): engine life-cycle, arena allocation in HBM,
// the search loop (root step + N x {select, network step, expand+backup}) enqueued on the caller's
// stream, and the read-out calls.  No torch types, no exceptions across the boundary.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/smz.h"
#include "smz_kernels.h"
#include "smz_net_bf16.h"
#include "smz_net_tc32.h"
#include "smz_net_vision.h"

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// Every entry point works on the engine's device and leaves the caller's current device as it found it
// (torch allocations and launches of the calling thread follow the current device).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev); else if (err == cudaSuccess) prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ON_DEVICE(e_)                                                                                    \
  DeviceGuard guard_((e_)->cfg.device);                                                                 \
  if (guard_.err != cudaSuccess) return fail(SMZ_E_CUDA, "cudaSetDevice(%d) failed: %s", (e_)->cfg.device, cudaGetErrorString(guard_.err))

#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) return fail(SMZ_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

struct smz_engine {
  smz_config cfg;
  smz_dims dims;
  SmzArena a;            // device pointers + shape, passed by value to every kernel
  SmzNetShape shape;
  SmzNetImageF32 img32;
  float* img32_buf;
  float* blob_buf;
  SmzBf16Image* bf16;    // tcgen05 path state (null unless net_mode == SMZ_NET_BF16)
  SmzTc32Image* tc32;    // fp16-operand tcgen05 path state (null unless net_mode == SMZ_NET_TC32 / SMZ_NET_F16)
  SmzVisionImage* vision;  // vision family state (null unless net_mode == SMZ_NET_VISION)
  double* pbc_dev;
  double* rcp64_dev;
  float* rcp32_dev;
  unsigned long long* seed_dev;
  signed char* sign_dev;
  std::vector<int32_t> to_play_tab;   // [n_phases][N+2], host copy for export
  std::vector<void*> allocs;
  int n_trees;           // trees of the current search
  int sims_done;
  int have_weights;
  int64_t launches;        // kernels of the last smz_root + smz_simulate
  int64_t launches_total;  // kernels since smz_create
  cudaGraphExec_t graph_exec;
  int graph_trees, graph_sims, graph_first, graph_launches;
  cudaStream_t capture_stream;
  int use_pdl;
  int32_t node_pattern;  // SMZ_PATTERN_*, copied into the arena (a.kind_shift) by the next smz_root
};

const char* smz_last_error(void) { return g_err; }

static void count_launches(smz_engine* e, int64_t n) { e->launches += n; e->launches_total += n; }

static int pow2ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }

template <typename T>
static cudaError_t dev_alloc(smz_engine* e, T** p, size_t n) {
  void* q = nullptr;
  cudaError_t r = cudaMalloc(&q, (n ? n : 1) * sizeof(T));
  if (r == cudaSuccess) { e->allocs.push_back(q); *p = (T*)q; e->dims.arena_bytes += n * sizeof(T); }
  return r;
}

static int rcp_entries(int n_sims) { return n_sims + 3 > SMZ_MAX_POLICY + 1 ? n_sims + 3 : SMZ_MAX_POLICY + 1; }

static int fill_default_tables(smz_engine* e) {
  const smz_config& c = e->cfg;
  const int n = c.num_simulations + 2;
  std::vector<double> pbc(n);
  for (int i = 0; i < n; ++i)
    pbc[i] = sqrt((double)i) * (log(((double)i + (double)c.pb_c_base + 1.0) / (double)c.pb_c_base) + c.pb_c_init);
  CU(cudaMemcpy(e->pbc_dev, pbc.data(), n * sizeof(double), cudaMemcpyHostToDevice));
  const int nt = rcp_entries(c.num_simulations);     // divisors: visit counts <= N + 2 and child counts <= 32
  std::vector<double> r64(nt, 0.0);
  std::vector<float> r32(nt, 0.f);
  for (int i = 1; i < nt; ++i) { r64[i] = 1.0 / (double)i; r32[i] = 1.0f / (float)i; }   // IEEE: correctly rounded
  CU(cudaMemcpy(e->rcp64_dev, r64.data(), nt * sizeof(double), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(e->rcp32_dev, r32.data(), nt * sizeof(float), cudaMemcpyHostToDevice));
  std::vector<signed char> sign(n, 1);
  CU(cudaMemcpy(e->sign_dev, sign.data(), n, cudaMemcpyHostToDevice));
  e->to_play_tab.assign(n, 0);
  e->a.n_phases = 1;
  return SMZ_OK;
}

int smz_create(const smz_config* cfg, smz_engine** out) {
  if (!cfg || !out) return fail(SMZ_E_INVALID_ARG, "smz_create: null argument");
  if (cfg->abi_version != SMZ_ABI_VERSION)
    return fail(SMZ_E_INVALID_ARG, "smz_create: abi_version %d, library is %d", cfg->abi_version, SMZ_ABI_VERSION);
  const smz_config& c = *cfg;
  if (c.max_trees < 1 || c.num_simulations < 0 || c.action_dim < 1 || c.chance_dim < 1 || c.max_action_sample < 1 ||
      c.pb_c_base < 1 || c.pb_c_init < 0 || c.discount < 0)
    return fail(SMZ_E_INVALID_ARG, "smz_create: search parameter out of range");
  if (c.action_dim > SMZ_MAX_POLICY || c.chance_dim > SMZ_MAX_POLICY)
    return fail(SMZ_E_CAPACITY, "smz_create: policy width %d/%d exceeds %d (one lane per policy entry)",
                c.action_dim, c.chance_dim, SMZ_MAX_POLICY);
  if (c.net_mode < SMZ_NET_EXTERNAL || c.net_mode > SMZ_NET_F16) return fail(SMZ_E_INVALID_ARG, "bad net_mode");
  if (c.net_mode == SMZ_NET_VISION) {
    if (c.obs_dim != 3 * 98 * 98) return fail(SMZ_E_INVALID_ARG, "smz_create: vision models take 3x98x98 observations (obs_dim %d)", c.obs_dim);
    if (c.action_dim != c.chance_dim) return fail(SMZ_E_INVALID_ARG, "smz_create: vision family needs chance_dim == action_dim");
  } else if (c.net_mode != SMZ_NET_EXTERNAL) {
    if (c.obs_dim < 1 || c.state_dim < 2 || c.hidden_dim < 1 || c.num_hidden_layers < 0)
      return fail(SMZ_E_INVALID_ARG, "smz_create: model shape out of range");
    if (c.hidden_dim > SMZ_HP || c.state_dim > SMZ_SP)
      return fail(SMZ_E_CAPACITY, "smz_create: fused MLP tiles hold H<=%d, S<=%d (got %d, %d)",
                  SMZ_HP, SMZ_SP, c.hidden_dim, c.state_dim);
    if (c.obs_dim > SMZ_MAX_OBS)
      return fail(SMZ_E_CAPACITY, "smz_create: observations of the MLP family are limited to obs_dim<=%d (got %d)",
                  SMZ_MAX_OBS, c.obs_dim);
  }
  int need = pow2ceil(c.action_dim > c.chance_dim ? c.action_dim : c.chance_dim);
  if (need < 2) need = 2;
  int lanes = c.lanes_per_tree;
  if (lanes == 0) lanes = need < 4 ? 4 : need;
  if ((lanes & (lanes - 1)) || lanes < need || lanes > 32)
    return fail(SMZ_E_INVALID_ARG, "smz_create: lanes_per_tree must be a power of two in [%d, 32]", need);

  DeviceGuard guard_(c.device);
  if (guard_.err != cudaSuccess) return fail(SMZ_E_CUDA, "cudaSetDevice(%d) failed: %s", c.device, cudaGetErrorString(guard_.err));
  smz_engine* e = new smz_engine();
  e->cfg = c;
  memset(&e->dims, 0, sizeof(e->dims));
  memset(&e->a, 0, sizeof(e->a));
  e->img32_buf = nullptr; e->blob_buf = nullptr; e->bf16 = nullptr; e->tc32 = nullptr; e->vision = nullptr;
  e->n_trees = 0; e->sims_done = 0; e->have_weights = 0; e->launches = 0; e->launches_total = 0;
  e->use_pdl = getenv("SMZ_NO_PDL") ? 0 : 1;
  e->graph_exec = nullptr; e->graph_trees = e->graph_sims = e->graph_first = -1; e->capture_stream = nullptr;

  SmzArena& a = e->a;
  a.B = c.max_trees; a.N = c.num_simulations; a.A = c.action_dim; a.C = c.chance_dim; a.K = c.max_action_sample;
  a.Kd = a.K < a.A ? a.K : a.A;
  a.Kc = a.K < a.C ? a.K : a.C;
  a.Kmax = a.Kd > a.Kc ? a.Kd : a.Kc;
  a.M = 1 + a.A + a.N * a.Kmax;
  a.W = a.A > a.C ? a.A : a.C;
  a.Sp = c.net_mode == SMZ_NET_VISION ? SMZ_VISION_SP : SMZ_SP;
  a.path_stride = a.N + 2;
  a.n_phases = 1;
  a.kind_shift = 1;
  e->node_pattern = SMZ_PATTERN_REFERENCE;
  a.rng_mode = c.rng_mode;
  a.discount = (float)c.discount;
  a.one_minus_frac_f32 = (float)(1.0 - c.root_exploration_fraction);
  a.frac = c.root_exploration_fraction;
  a.alpha = c.root_dirichlet_alpha;

  e->dims.nodes_per_tree = a.M; e->dims.max_children = a.Kmax; e->dims.policy_stride = a.W;
  e->dims.hidden_stride = a.Sp; e->dims.hidden_slots = a.N + 1; e->dims.path_stride = a.path_stride;
  e->dims.lanes_per_tree = lanes;
  e->cfg.lanes_per_tree = lanes;

  const size_t B = a.B, M = a.M;
  a.row_cap = (a.B + 511) / 512 * 512 + 512;
  a.row_top = a.row_cap;
  const size_t RC = a.row_cap;
  cudaError_t r = cudaSuccess;
#define ALLOC(ptr, n) if (r == cudaSuccess) r = dev_alloc(e, &(ptr), (n))
  ALLOC(a.stat, B * M); ALLOC(a.link, B * M); ALLOC(a.root_prior, B * a.A); ALLOC(a.minmax, B);
  ALLOC(a.ucursor, B); ALLOC(a.root_to_play, B); ALLOC(a.path, B * a.path_stride); ALLOC(a.path_len, B);
  ALLOC(a.leaf_node, B); ALLOC(a.leaf_slot, B); ALLOC(a.leaf_action, B); ALLOC(a.leaf_branch, B);
  ALLOC(a.branch_count, (size_t)(a.N + 1) * 2); ALLOC(a.rows, 2 * RC); ALLOC(a.rows4, 2 * RC); ALLOC(a.error_flag, 1);
  ALLOC(a.depth_sum, 1);
  a.xin_q = c.net_mode == SMZ_NET_TC32 ? 16 : 8;
  if (c.net_mode == SMZ_NET_BF16 || c.net_mode == SMZ_NET_TC32 || c.net_mode == SMZ_NET_F16) { ALLOC(a.xin, 2 * RC * a.xin_q); }
  if (getenv("SMZ_TREE_TIMELINE")) { ALLOC(a.dbg, 8 + 4 * ((size_t)a.N + 2)); }
  ALLOC(a.out_policy, B * a.W); ALLOC(a.out_value, B); ALLOC(a.out_reward, B); ALLOC(a.dirichlet, B * a.A);
  if (c.record) {
    ALLOC(a.rec_policy, B * a.N * a.W); ALLOC(a.rec_value, B * a.N); ALLOC(a.rec_reward, B * a.N);
    ALLOC(a.rec_branch, B * a.N); ALLOC(a.rec_root_policy, B * a.W);
  }
  ALLOC(e->pbc_dev, (size_t)a.N + 2);
  ALLOC(e->rcp64_dev, (size_t)rcp_entries(a.N));
  ALLOC(e->rcp32_dev, (size_t)rcp_entries(a.N));
  ALLOC(e->seed_dev, 2);
  ALLOC(e->sign_dev, (size_t)a.N + 2);
  if (c.net_mode == SMZ_NET_VISION) {
    ALLOC(a.hidden, (size_t)(a.N + 1) * B * a.Sp);
    e->dims.weight_blob_floats = smz_vision_blob_floats(a.A, c.state_dim, c.hidden_dim, c.num_hidden_layers);
    ALLOC(e->blob_buf, e->dims.weight_blob_floats);
  } else if (c.net_mode != SMZ_NET_EXTERNAL) {
    SmzNetShape& sh = e->shape;
    sh.obs = c.obs_dim; sh.A = a.A; sh.C = a.C; sh.S = c.state_dim; sh.H = c.hidden_dim; sh.L = c.num_hidden_layers;
    sh.OH = a.W; sh.obs_pad = (c.obs_dim + 31) / 32 * 32;
    ALLOC(a.hidden, (size_t)(a.N + 1) * B * SMZ_SP);
    ALLOC(e->img32_buf, smz_net_f32_image_floats(sh));
    e->dims.weight_blob_floats = smz_blob_floats(sh);
    ALLOC(e->blob_buf, e->dims.weight_blob_floats);
  }
#undef ALLOC
  if (r != cudaSuccess) {
    for (void* p : e->allocs) cudaFree(p);
    delete e;
    return fail(SMZ_E_CUDA, "smz_create: cudaMalloc failed: %s", cudaGetErrorString(r));
  }
  a.pbc = e->pbc_dev;
  a.rcp64 = e->rcp64_dev;
  a.rcp32 = e->rcp32_dev;
  a.seed_state = e->seed_dev;
  a.sign = e->sign_dev;
  int rc = fill_default_tables(e);
  if (rc == SMZ_OK) {
    const unsigned long long st[2] = {c.seed, c.tree_id_offset};
    if (cudaMemcpy(e->seed_dev, st, sizeof(st), cudaMemcpyHostToDevice) != cudaSuccess) rc = fail(SMZ_E_CUDA, "seed upload failed");
  }
  if (rc == SMZ_OK && a.hidden) {
    cudaMemset(a.rows, 0, 2 * RC * sizeof(int));          // speculative gathers read rows beyond the live count
    cudaMemset(a.rows4, 0, 2 * RC * sizeof(int4));
    if (a.xin) cudaMemset(a.xin, 0, 2 * RC * a.xin_q * sizeof(uint4));
    cudaError_t m = cudaMemset(a.hidden, 0, (size_t)(a.N + 1) * B * a.Sp * sizeof(float));
    if (m != cudaSuccess) rc = fail(SMZ_E_CUDA, "memset: %s", cudaGetErrorString(m));
  }
  if (rc == SMZ_OK && c.net_mode == SMZ_NET_BF16) rc = smz_bf16_create(e->shape, a, &e->bf16, g_err, sizeof(g_err));
  if (rc == SMZ_OK && (c.net_mode == SMZ_NET_TC32 || c.net_mode == SMZ_NET_F16))
    rc = smz_tc32_create(e->shape, c.net_mode == SMZ_NET_F16 ? 1 : 3, &e->tc32, g_err, sizeof(g_err));
  if (rc == SMZ_OK && c.net_mode == SMZ_NET_VISION)
    rc = smz_vision_create(a.A, c.state_dim, c.hidden_dim, c.num_hidden_layers, c.max_trees, &e->vision, g_err, sizeof(g_err));
  if (rc == SMZ_OK && cudaStreamCreateWithFlags(&e->capture_stream, cudaStreamNonBlocking) != cudaSuccess)
    rc = fail(SMZ_E_CUDA, "cudaStreamCreate failed");
  if (rc != SMZ_OK) { smz_destroy(e); return rc; }
  *out = e;
  return SMZ_OK;
}

int smz_destroy(smz_engine* e) {
  if (!e) return SMZ_OK;
  DeviceGuard guard_(e->cfg.device);
  if (e->a.dbg) {
    long long t[8];
    std::vector<unsigned long long> w(4 * ((size_t)e->a.N + 2));
    if (cudaMemcpy(w.data(), e->a.dbg + 8, w.size() * sizeof(w[0]), cudaMemcpyDeviceToHost) == cudaSuccess && e->a.N >= 12) {
      // wall clock (ns) of the last search, averaged over simulations N-11 .. N-2
      double tree = 0, net = 0, g1 = 0, g2 = 0;
      int n = 0;
      for (int s = e->a.N - 11; s <= e->a.N - 2; ++s, ++n) {
        const unsigned long long *c = &w[4 * s], *nx = &w[4 * (s + 1)];
        net += (double)(c[3] - c[2]);            // network step of s: first wait-return -> last CTA end
        g1 += (double)((long long)c[0] - (long long)c[3]);   // -> first wait-return of the tree step of s
        tree += (double)(c[1] - c[0]);           // tree step of s (+ descent of s+1)
        g2 += (double)((long long)nx[2] - (long long)c[1]);  // -> first wait-return of the network step of s+1
      }
      fprintf(stderr, "smz step timeline (%%globaltimer, mean of %d simulations): network step %.2f us | -> tree step %.2f us | tree step %.2f us | -> network step %.2f us\n",
              n, net / n / 1e3, g1 / n / 1e3, tree / n / 1e3, g2 / n / 1e3);
    }
    if (cudaMemcpy(t, e->a.dbg, sizeof(t), cudaMemcpyDeviceToHost) == cudaSuccess)
      fprintf(stderr, "smz tree timeline (block 0, last fused launch): expand+backup %lld cycles | descent %lld cycles = %lld levels walked by warp 0 in %lld + leaf record / row reservation %lld (path length of tree 0: %lld)\n",
              t[1] - t[0], t[2] - t[1], t[5], t[4] - t[1], t[2] - t[4], t[3]);
  }
  if (e->graph_exec) cudaGraphExecDestroy(e->graph_exec);
  if (e->capture_stream) cudaStreamDestroy(e->capture_stream);
  if (e->bf16) smz_bf16_destroy(e->bf16);
  if (e->tc32) smz_tc32_destroy(e->tc32);
  if (e->vision) smz_vision_destroy(e->vision);
  for (void* p : e->allocs) cudaFree(p);
  delete e;
  return SMZ_OK;
}

int smz_get_dims(const smz_engine* e, smz_dims* out) {
  if (!e || !out) return fail(SMZ_E_INVALID_ARG, "smz_get_dims: null argument");
  *out = e->dims;
  return SMZ_OK;
}

static void drop_graph(smz_engine* e) {
  if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
  e->graph_trees = e->graph_sims = e->graph_first = -1;
}

int smz_set_pbc_table(smz_engine* e, const double* t, int32_t n) {
  if (!e || !t) return fail(SMZ_E_INVALID_ARG, "smz_set_pbc_table: null argument");
  if (n != e->a.N + 2) return fail(SMZ_E_INVALID_ARG, "smz_set_pbc_table: need %d entries, got %d", e->a.N + 2, n);
  ON_DEVICE(e);
  CU(cudaMemcpy(e->pbc_dev, t, (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
  return SMZ_OK;
}

int smz_set_player_tables(smz_engine* e, const int8_t* sign, const int32_t* to_play, int32_t n_phases) {
  if (!e || !sign || !to_play || n_phases < 1) return fail(SMZ_E_INVALID_ARG, "smz_set_player_tables: bad argument");
  ON_DEVICE(e);
  const size_t n = (size_t)n_phases * (e->a.N + 2);
  signed char* d = nullptr;
  CU(dev_alloc(e, &d, n));
  CU(cudaMemcpy(d, sign, n, cudaMemcpyHostToDevice));
  e->sign_dev = d;
  e->a.sign = d;
  e->a.n_phases = n_phases;
  e->to_play_tab.assign(to_play, to_play + n);
  drop_graph(e);
  return SMZ_OK;
}

int smz_set_weights(smz_engine* e, const float* blob, uint64_t n_floats, int32_t on_device, void* stream) {
  if (!e || !blob) return fail(SMZ_E_INVALID_ARG, "smz_set_weights: null argument");
  if (e->cfg.net_mode == SMZ_NET_EXTERNAL) return fail(SMZ_E_STATE, "smz_set_weights: engine has no internal network");
  if (n_floats != e->dims.weight_blob_floats)
    return fail(SMZ_E_INVALID_ARG, "smz_set_weights: blob has %llu floats, model shape needs %llu",
                (unsigned long long)n_floats, (unsigned long long)e->dims.weight_blob_floats);
  cudaStream_t s = (cudaStream_t)stream;
  ON_DEVICE(e);
  CU(cudaMemcpyAsync(e->blob_buf, blob, n_floats * sizeof(float),
                     on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  if (e->vision) {
    int rc = smz_vision_pack(e->vision, e->blob_buf, s, g_err, sizeof(g_err));
    if (rc != SMZ_OK) return rc;
    e->have_weights = 1;
    return SMZ_OK;
  }
  smz_net_f32_pack(e->shape, e->blob_buf, e->img32_buf, &e->img32, s);
  if (e->bf16) {
    int rc = smz_bf16_pack(e->bf16, e->shape, e->blob_buf, s, g_err, sizeof(g_err));
    if (rc != SMZ_OK) return rc;
  }
  if (e->tc32) {
    int rc = smz_tc32_pack(e->tc32, e->shape, e->blob_buf, s, g_err, sizeof(g_err));
    if (rc != SMZ_OK) return rc;
  }
  CU(cudaGetLastError());
  e->have_weights = 1;
  return SMZ_OK;
}

int smz_set_seed(smz_engine* e, uint64_t seed, uint64_t tree_id_offset, void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_set_seed: null engine");
  ON_DEVICE(e);
  // stream-ordered update by a one-thread kernel: the values travel as launch arguments, nothing to synchronise on
  smz_launch_set_seed(e->seed_dev, seed, tree_id_offset, (cudaStream_t)stream);
  CU(cudaGetLastError());
  e->cfg.seed = seed;
  e->cfg.tree_id_offset = tree_id_offset;
  return SMZ_OK;
}

int smz_set_uniform_tape(smz_engine* e, const double* u, int32_t stride) {
  if (!e || !u || stride < 1) return fail(SMZ_E_INVALID_ARG, "smz_set_uniform_tape: bad argument");
  if (e->cfg.rng_mode != SMZ_RNG_TAPE) return fail(SMZ_E_STATE, "smz_set_uniform_tape: engine rng_mode is not TAPE");
  e->a.tape_u = u;
  e->a.tape_stride = stride;
  drop_graph(e);
  return SMZ_OK;
}

int smz_set_node_pattern(smz_engine* e, int32_t pattern) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_set_node_pattern: null engine");
  if (pattern != SMZ_PATTERN_REFERENCE && pattern != SMZ_PATTERN_PAPER)
    return fail(SMZ_E_INVALID_ARG, "smz_set_node_pattern: pattern %d is neither SMZ_PATTERN_REFERENCE (0) nor SMZ_PATTERN_PAPER (1)",
                pattern);
  e->node_pattern = pattern;
  return SMZ_OK;
}

int smz_root(smz_engine* e, int32_t n_trees, const float* obs, const float* root_policy, const int32_t* root_to_play,
             int32_t train, const double* dirichlet, void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_root: null engine");
  if (n_trees < 1 || n_trees > e->a.B) return fail(SMZ_E_CAPACITY, "smz_root: n_trees %d not in [1, %d]", n_trees, e->a.B);
  if ((obs == nullptr) == (root_policy == nullptr))
    return fail(SMZ_E_INVALID_ARG, "smz_root: give exactly one of obs_dev / root_policy_dev");
  if (obs && e->cfg.net_mode == SMZ_NET_EXTERNAL) return fail(SMZ_E_STATE, "smz_root: obs given but engine has no network");
  if (obs && !e->have_weights) return fail(SMZ_E_STATE, "smz_root: smz_set_weights has not been called");
  if (e->cfg.rng_mode == SMZ_RNG_TAPE && !e->a.tape_u) return fail(SMZ_E_STATE, "smz_root: no uniform tape set");
  cudaStream_t s = (cudaStream_t)stream;
  ON_DEVICE(e);
  SmzArena& a = e->a;
  const int kind_shift = e->node_pattern == SMZ_PATTERN_PAPER ? 0 : 1;
  if (a.kind_shift != kind_shift) {   // the captured simulation graph holds the arena by value
    a.kind_shift = kind_shift;
    drop_graph(e);
  }
  smz_launch_begin_search(a, s);       // row counters, error flag, depth statistic
  if (a.dbg) {      // wall-clock stamps: "first" slots start at all-ones (atomicMin), "last" slots at zero (atomicMax)
    std::vector<unsigned long long> init(4 * ((size_t)a.N + 2));
    for (size_t i = 0; i < init.size(); ++i) init[i] = (i & 1) ? 0ull : ~0ull;
    CU(cudaMemcpyAsync(a.dbg + 8, init.data(), init.size() * sizeof(init[0]), cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));
  }
  e->launches = 0;
  if (e->cfg.num_simulations == 0) train = 0;   // mcts.py:215-216
  const float* policy = root_policy;
  if (obs) {
    if (e->vision) { smz_vision_root(e->vision, a, n_trees, obs, s); count_launches(e, 1); }
    else if (e->bf16) smz_bf16_root(e->bf16, a, e->shape, n_trees, obs, s);
    else if (e->tc32) smz_tc32_root(e->tc32, a, e->shape, n_trees, obs, s);
    else smz_net_f32_root(a, e->shape, e->img32, n_trees, obs, s);
    count_launches(e, 1);
    policy = a.out_policy;
  }
  if (train) {
    if (dirichlet) {
      CU(cudaMemcpyAsync(a.dirichlet, dirichlet, (size_t)n_trees * a.A * sizeof(double), cudaMemcpyDeviceToDevice, s));
    } else {
      smz_launch_dirichlet(a, n_trees, s);
      count_launches(e, 1);
    }
  }
  smz_launch_root_expand(a, e->cfg.lanes_per_tree, n_trees, policy, a.W, root_to_play, train, a.dirichlet, s);
  count_launches(e, 1);
  CU(cudaGetLastError());
  e->n_trees = n_trees;
  a.row_top = (n_trees + 511) / 512 * 512 + 512;    // see smz_common.cuh: rows of the two branches never share a tile (group of 4)
  e->sims_done = 0;
  return SMZ_OK;
}

static int check_sim(smz_engine* e, int sim, const char* who) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "%s: null engine", who);
  if (e->n_trees < 1) return fail(SMZ_E_STATE, "%s: smz_root has not been called", who);
  if (sim < 0 || sim >= e->a.N) return fail(SMZ_E_CAPACITY, "%s: simulation %d not in [0, %d)", who, sim, e->a.N);
  return SMZ_OK;
}

int smz_select(smz_engine* e, int32_t sim, int32_t* slot, int32_t* action, int32_t* branch, void* stream) {
  int rc = check_sim(e, sim, "smz_select");
  if (rc) return rc;
  ON_DEVICE(e);
  smz_launch_select(e->a, e->cfg.lanes_per_tree, e->n_trees, sim, slot, action, branch, (cudaStream_t)stream);
  count_launches(e, 1);
  CU(cudaGetLastError());
  return SMZ_OK;
}

// returns the number of kernels launched
static int enqueue_net(smz_engine* e, int sim, cudaStream_t s, bool pdl = false) {
  if (e->vision) return smz_vision_sim(e->vision, e->a, e->n_trees, sim, pdl, s);
  if (e->bf16) smz_bf16_sim(e->bf16, e->a, e->shape, e->n_trees, sim, pdl, s);
  else if (e->tc32) smz_tc32_sim(e->tc32, e->a, e->shape, e->n_trees, sim, pdl, s);
  else smz_net_f32_sim(e->a, e->shape, e->img32, e->n_trees, sim, s);
  return 1;
}

int smz_net_step(smz_engine* e, int32_t sim, void* stream) {
  int rc = check_sim(e, sim, "smz_net_step");
  if (rc) return rc;
  if (e->cfg.net_mode == SMZ_NET_EXTERNAL) return fail(SMZ_E_STATE, "smz_net_step: engine has no internal network");
  if (!e->have_weights) return fail(SMZ_E_STATE, "smz_net_step: smz_set_weights has not been called");
  ON_DEVICE(e);
  count_launches(e, enqueue_net(e, sim, (cudaStream_t)stream));
  CU(cudaGetLastError());
  return SMZ_OK;
}

int smz_expand_backup(smz_engine* e, int32_t sim, const float* policy, const float* value, const float* reward,
                      void* stream) {
  int rc = check_sim(e, sim, "smz_expand_backup");
  if (rc) return rc;
  if (policy && (!value || !reward)) return fail(SMZ_E_INVALID_ARG, "smz_expand_backup: value/reward missing");
  ON_DEVICE(e);
  const SmzArena& a = e->a;
  smz_launch_expand_backup(a, e->cfg.lanes_per_tree, e->n_trees, sim, policy ? policy : a.out_policy, a.W,
                           policy ? value : a.out_value, policy ? reward : a.out_reward, (cudaStream_t)stream);
  count_launches(e, 1);
  if (sim + 1 > e->sims_done) e->sims_done = sim + 1;
  CU(cudaGetLastError());
  return SMZ_OK;
}

int smz_backup_select(smz_engine* e, int32_t sim, void* stream) {
  int rc = check_sim(e, sim, "smz_backup_select");
  if (rc) return rc;
  if (sim + 1 >= e->a.N) return fail(SMZ_E_CAPACITY, "smz_backup_select: simulation %d has no successor (N = %d)", sim, e->a.N);
  if (e->cfg.net_mode == SMZ_NET_EXTERNAL) return fail(SMZ_E_STATE, "smz_backup_select: engine has no internal network");
  ON_DEVICE(e);
  smz_launch_backup_select(e->a, e->cfg.lanes_per_tree, e->n_trees, sim, false, (cudaStream_t)stream);
  count_launches(e, 1);
  if (sim + 1 > e->sims_done) e->sims_done = sim + 1;
  CU(cudaGetLastError());
  return SMZ_OK;
}

// returns the number of kernels enqueued
static int enqueue_sims(smz_engine* e, int first, int n_sims, cudaStream_t s) {
  const SmzArena& a = e->a;
  const int G = e->cfg.lanes_per_tree;
  // select(first); then per simulation: network step, then [expand+backup(sim) fused with select(sim+1)]
  // With the tensor-core network both hot kernels are chained by programmatic dependent launch: the
  // next kernel's CTAs become resident and run their prologue while the previous one drains.
  const bool pdl = (e->bf16 != nullptr || e->tc32 != nullptr || smz_vision_has_tc(e->vision)) && e->use_pdl;
  smz_launch_select(a, G, e->n_trees, first, nullptr, nullptr, nullptr, s);
  int launched = 1;
  for (int sim = first; sim < first + n_sims; ++sim) {
    const bool last = sim + 1 >= first + n_sims;
    launched += enqueue_net(e, sim, s, pdl) + 1;
    if (!last) smz_launch_backup_select(a, G, e->n_trees, sim, pdl, s);
    else smz_launch_expand_backup(a, G, e->n_trees, sim, a.out_policy, a.W, a.out_value, a.out_reward, s);
  }
  return launched;
}

int smz_simulate(smz_engine* e, int32_t n_sims, void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_simulate: null engine");
  if (e->n_trees < 1) return fail(SMZ_E_STATE, "smz_simulate: smz_root has not been called");
  if (e->cfg.net_mode == SMZ_NET_EXTERNAL) return fail(SMZ_E_STATE, "smz_simulate: engine has no internal network");
  if (!e->have_weights) return fail(SMZ_E_STATE, "smz_simulate: smz_set_weights has not been called");
  if (n_sims < 0 || e->sims_done + n_sims > e->a.N)
    return fail(SMZ_E_CAPACITY, "smz_simulate: %d + %d simulations exceed num_simulations %d", e->sims_done, n_sims, e->a.N);
  if (n_sims == 0) return SMZ_OK;
  cudaStream_t s = (cudaStream_t)stream;
  ON_DEVICE(e);
  const int first = e->sims_done;
  // The N-step loop is launch-bound: capture it once per (trees, first, count) into a CUDA graph and
  // replay it on the caller's stream.
  if (!e->graph_exec || e->graph_trees != e->n_trees || e->graph_sims != n_sims || e->graph_first != first) {
    drop_graph(e);
    cudaGraph_t graph = nullptr;
    CU(cudaStreamBeginCapture(e->capture_stream, cudaStreamCaptureModeThreadLocal));
    e->graph_launches = enqueue_sims(e, first, n_sims, e->capture_stream);
    cudaError_t ce = cudaStreamEndCapture(e->capture_stream, &graph);
    if (ce == cudaSuccess) {
      ce = cudaGraphInstantiate(&e->graph_exec, graph, 0);
      cudaGraphDestroy(graph);
    }
    if (ce != cudaSuccess && e->use_pdl && (e->bf16 || e->tc32 || e->vision)) {
      // programmatic edges not capturable on this driver: fall back to plain stream order, once
      cudaGetLastError();
      e->graph_exec = nullptr;
      e->use_pdl = 0;
      return smz_simulate(e, n_sims, stream);
    }
    if (ce != cudaSuccess) { e->graph_exec = nullptr; return fail(SMZ_E_CUDA, "graph capture/instantiate failed: %s", cudaGetErrorString(ce)); }
    e->graph_trees = e->n_trees; e->graph_sims = n_sims; e->graph_first = first;
  }
  CU(cudaGraphLaunch(e->graph_exec, s));
  count_launches(e, e->graph_launches);
  e->sims_done += n_sims;
  return SMZ_OK;
}

int smz_net_eval(smz_engine* e, int32_t which, int32_t n_rows, const float* in, const int32_t* idx, float* hidden_out,
                 float* policy_out, float* value_out, float* reward_out, int32_t* code_out, void* stream) {
  if (!e || !in) return fail(SMZ_E_INVALID_ARG, "smz_net_eval: null argument");
  if (e->cfg.net_mode == SMZ_NET_EXTERNAL) return fail(SMZ_E_STATE, "smz_net_eval: engine has no internal network");
  if (!e->have_weights) return fail(SMZ_E_STATE, "smz_net_eval: smz_set_weights has not been called");
  if (which < 0 || which > 5 || n_rows < 1) return fail(SMZ_E_INVALID_ARG, "smz_net_eval: bad which / n_rows");
  if ((which == 2 || which == 4) && !idx) return fail(SMZ_E_INVALID_ARG, "smz_net_eval: idx_dev required");
  ON_DEVICE(e);
  if (e->vision) {
    if (smz_vision_eval(e->vision, which, n_rows, in, idx, hidden_out, policy_out, value_out, reward_out, e->a.W,
                        (cudaStream_t)stream) != SMZ_OK)
      return fail(SMZ_E_INVALID_ARG, "smz_net_eval: the vision family has no stand-alone network %d", which);
    CU(cudaGetLastError());
    return SMZ_OK;
  }
  if (e->bf16)
    smz_bf16_eval(e->bf16, e->shape, which, n_rows, in, idx, hidden_out, policy_out, value_out, reward_out, code_out,
                  e->a.W, (cudaStream_t)stream);
  else if (e->tc32)
    smz_tc32_eval(e->tc32, e->shape, which, n_rows, in, idx, hidden_out, policy_out, value_out, reward_out, code_out,
                  e->a.W, (cudaStream_t)stream);
  else
    smz_net_f32_eval(e->shape, e->img32, which, n_rows, in, idx, hidden_out, policy_out, value_out, reward_out,
                     code_out, e->a.W, (cudaStream_t)stream);
  CU(cudaGetLastError());
  return SMZ_OK;
}

int smz_read_roots(smz_engine* e, int32_t* visits, float* values, double* priors, float* rewards, int32_t* error_out,
                   void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_read_roots: null engine");
  if (e->n_trees < 1) return fail(SMZ_E_STATE, "smz_read_roots: smz_root has not been called");
  ON_DEVICE(e);
  smz_launch_read_roots(e->a, e->n_trees, visits, values, priors, rewards, error_out, (cudaStream_t)stream);
  count_launches(e, 1);
  CU(cudaGetLastError());
  return SMZ_OK;
}

int smz_select_actions(smz_engine* e, double temperature, const double* uniforms, int32_t* actions, double* policy,
                       double* stored_policy, void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_select_actions: null engine");
  if (e->n_trees < 1) return fail(SMZ_E_STATE, "smz_select_actions: smz_root has not been called");
  if (!(temperature >= 0.0)) return fail(SMZ_E_INVALID_ARG, "smz_select_actions: temperature must be >= 0");
  ON_DEVICE(e);
  smz_launch_select_actions(e->a, e->n_trees, temperature, uniforms, actions, policy, stored_policy, (cudaStream_t)stream);
  count_launches(e, 1);
  CU(cudaGetLastError());
  return SMZ_OK;
}

int smz_export_tree(smz_engine* e, int32_t tree, smz_tree_host* out, void* stream) {
  if (!e || !out) return fail(SMZ_E_INVALID_ARG, "smz_export_tree: null argument");
  if (tree < 0 || tree >= e->n_trees) return fail(SMZ_E_INVALID_ARG, "smz_export_tree: tree %d not in [0, %d)", tree, e->n_trees);
  ON_DEVICE(e);
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  const SmzArena& a = e->a;
  const size_t M = a.M;
  std::vector<int4> stat(M);
  std::vector<int2> link(M);
  CU(cudaMemcpy(stat.data(), a.stat + (size_t)tree * M, M * sizeof(int4), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(link.data(), a.link + (size_t)tree * M, M * sizeof(int2), cudaMemcpyDeviceToHost));
  for (size_t n = 0; n < M; ++n) {
    if (out->visit) out->visit[n] = stat[n].x;
    if (out->value_sum) memcpy(&out->value_sum[n], &stat[n].y, 4);
    if (out->reward) memcpy(&out->reward[n], &stat[n].z, 4);
    if (out->prior) memcpy(&out->prior[n], &stat[n].w, 4);
    if (out->child_base) out->child_base[n] = link[n].x;
    if (out->key) out->key[n] = link[n].y;
  }
  if (out->root_prior)
    CU(cudaMemcpy(out->root_prior, a.root_prior + (size_t)tree * a.A, a.A * sizeof(double), cudaMemcpyDeviceToHost));
  float2 mm;
  CU(cudaMemcpy(&mm, a.minmax + tree, sizeof(mm), cudaMemcpyDeviceToHost));
  out->minmax[0] = mm.x; out->minmax[1] = mm.y;
  CU(cudaMemcpy(&out->n_uniforms, a.ucursor + tree, sizeof(int), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(&out->root_to_play, a.root_to_play + tree, sizeof(int), cudaMemcpyDeviceToHost));
  return SMZ_OK;
}

int smz_read_hidden(smz_engine* e, int32_t slot, float* out, void* stream) {
  if (!e || !out) return fail(SMZ_E_INVALID_ARG, "smz_read_hidden: null argument");
  if (!e->a.hidden) return fail(SMZ_E_STATE, "smz_read_hidden: engine has no internal network");
  if (slot < 0 || slot > e->a.N || e->n_trees < 1) return fail(SMZ_E_INVALID_ARG, "smz_read_hidden: bad slot");
  ON_DEVICE(e);
  if (e->bf16 || e->tc32) {
    if (e->bf16) smz_bf16_read_hidden(e->a, slot, e->n_trees, out, (cudaStream_t)stream);
    else smz_tc32_read_hidden(e->a, slot, e->n_trees, out, (cudaStream_t)stream);
    CU(cudaGetLastError());
    return SMZ_OK;
  }
  CU(cudaMemcpyAsync(out, e->a.hidden + (size_t)slot * e->a.B * e->a.Sp, (size_t)e->n_trees * e->a.Sp * sizeof(float),
                     cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return SMZ_OK;
}

int smz_read_record(smz_engine* e, float* policy, float* value, float* reward, int8_t* branch, double* dirichlet,
                    float* root_policy, void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_read_record: null engine");
  if (!e->a.rec_policy) return fail(SMZ_E_STATE, "smz_read_record: engine was created with record = 0");
  if (e->n_trees < 1) return fail(SMZ_E_STATE, "smz_read_record: smz_root has not been called");
  cudaStream_t s = (cudaStream_t)stream;
  ON_DEVICE(e);
  const SmzArena& a = e->a;
  const size_t n = e->n_trees, N = a.N;
  if (policy) CU(cudaMemcpyAsync(policy, a.rec_policy, n * N * a.W * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (value) CU(cudaMemcpyAsync(value, a.rec_value, n * N * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (reward) CU(cudaMemcpyAsync(reward, a.rec_reward, n * N * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (branch) CU(cudaMemcpyAsync(branch, a.rec_branch, n * N, cudaMemcpyDeviceToDevice, s));
  if (dirichlet) CU(cudaMemcpyAsync(dirichlet, a.dirichlet, n * a.A * sizeof(double), cudaMemcpyDeviceToDevice, s));
  if (root_policy) CU(cudaMemcpyAsync(root_policy, a.rec_root_policy, n * a.W * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return SMZ_OK;
}

int smz_stats(smz_engine* e, double* mean_leaf_depth, int64_t* launches, int64_t* launches_total, void* stream) {
  if (!e) return fail(SMZ_E_INVALID_ARG, "smz_stats: null engine");
  ON_DEVICE(e);
  CU(cudaStreamSynchronize((cudaStream_t)stream));
  unsigned long long ds = 0;
  int err = 0;
  CU(cudaMemcpy(&ds, e->a.depth_sum, sizeof(ds), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(&err, e->a.error_flag, sizeof(err), cudaMemcpyDeviceToHost));
  if (mean_leaf_depth) {
    const double n = (double)e->n_trees * (double)e->sims_done;
    *mean_leaf_depth = n > 0 ? (double)ds / n : 0.0;
  }
  if (launches) *launches = e->launches;
  if (launches_total) *launches_total = e->launches_total;
  if (err == 1) return fail(SMZ_E_CAPACITY, "uniform tape exhausted during the search");
  if (err == 2) return fail(SMZ_E_STATE, "degenerate (NaN / all-zero) policy met during expansion");
  return SMZ_OK;
}
