// smz_net_f32.cu — fp32 CUDA-core network step (parity mode: 1e-5 against the reference's torch fp32).
//
// One CTA evaluates a tile of 32 leaves through a whole network pair without leaving the SM:
//   afterstate leaves: Afterstate_dynamics (mlp:85-124) -> scale_to_bound_action (mlp:349-357)
//                      -> Afterstate_prediction (mlp:127-163) -> softmax / support expectation
//   dynamics leaves:   Dynamics (mlp:167-206, trunk evaluated ONCE, reward + state heads together)
//                      -> Prediction (mlp:47-83)
//   root:              Representation (mlp:5-42) -> Prediction
// plus the inference facade of muzero_model.py: one-hot action folded in as an embedding-row add
// (:496-509), softmax on the policy head (:837), inverse_transform_with_support (:575-591).
// Activations stay in shared memory between layers; weights stream through a double-buffered
// cp.async ring of 32-row k-slabs of the transposed, padded image (coalesced 512-byte rows).
#include <cuda_runtime.h>

#include "smz_common.cuh"
#include "smz_kernels.h"

namespace {

constexpr int R = 32;              // leaves per CTA
constexpr int NT = 256;            // threads per CTA
constexpr int LD = SMZ_HP + 4;     // activation row stride in shared memory
constexpr int KC = 32;             // k-slab rows per cp.async stage
constexpr int POL_OFF = 64;        // column of the second head inside the concatenated head tile

struct Smem {
  float x[R][LD];
  float y[R][LD];
  float w[2][KC][SMZ_HP];
  int tree[R];
  int idx[R];
  int slot[R];
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ float elu(float v) { return v > 0.f ? v : expm1f(v); }

// out[r][c] = act( sum_k in[r][k] * Wt[k][c] + b[c] (+ emb[idx[r]][c]) ),  r < 32, c < 128
__device__ void dense(const float* __restrict__ wt, int K, const float* __restrict__ bias,
                      const float* __restrict__ emb, const int* idx_s, const float (*in)[LD], float (*out)[LD],
                      bool act, float (*wbuf)[KC][SMZ_HP]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[2][8];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  const int nchunks = K / KC;
  auto issue = [&](int c) {
    const float* src = wt + (size_t)c * KC * SMZ_HP;
    float* dst = &wbuf[c & 1][0][0];
#pragma unroll
    for (int i = 0; i < (KC * SMZ_HP / 4) / NT; ++i) {
      const int e = (i * NT + tid) * 4;
      cp_async16(dst + e, src + e);
    }
    cp_async_commit();
  };
  issue(0);
  for (int c = 0; c < nchunks; ++c) {
    if (c + 1 < nchunks) { issue(c + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const float(*w)[SMZ_HP] = wbuf[c & 1];
#pragma unroll
    for (int kk = 0; kk < KC; kk += 4) {
      const float4 a0 = *reinterpret_cast<const float4*>(&in[ty * 2][c * KC + kk]);
      const float4 a1 = *reinterpret_cast<const float4*>(&in[ty * 2 + 1][c * KC + kk]);
      const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b0 = *reinterpret_cast<const float4*>(&w[kk + q][tx * 8]);
        const float4 b1 = *reinterpret_cast<const float4*>(&w[kk + q][tx * 8 + 4]);
        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[0][j] = fmaf(av0[q], bv[j], acc[0][j]);
          acc[1][j] = fmaf(av1[q], bv[j], acc[1][j]);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int r = ty * 2 + i;
    const float* e = (emb && idx_s[r] >= 0) ? emb + (size_t)idx_s[r] * SMZ_HP : nullptr;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = tx * 8 + j;
      float v = acc[i][j] + bias[c];
      if (e) v += e[c];
      out[r][c] = act ? elu(v) : v;
    }
  }
  __syncthreads();
}

// First layer of a network that reads caller rows of any width (the observation of repr / enc):
// out[r][c] = elu( sum_k in[row0 + r][k] * Wt[k][c] + b[c] ).  The input streams through xs in slices of SMZ_HP
// columns, re-staged whenever the k-slab ring crosses into the next slice, and the products are accumulated in the
// same order as dense() does over a staged row — so for in_w <= SMZ_HP the result is bit-identical to staging the
// whole row and calling dense().
__device__ void dense_wide_in(const SmzNetF32& net, const float* __restrict__ in, int in_w, int row0, int n_rows,
                              float (*xs)[LD], float (*out)[LD], float (*wbuf)[KC][SMZ_HP]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[2][8];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  const int nchunks = net.kin_pad / KC;
  auto issue = [&](int c) {
    const float* src = net.in_wt + (size_t)c * KC * SMZ_HP;
    float* dst = &wbuf[c & 1][0][0];
#pragma unroll
    for (int i = 0; i < (KC * SMZ_HP / 4) / NT; ++i) {
      const int e = (i * NT + tid) * 4;
      cp_async16(dst + e, src + e);
    }
    cp_async_commit();
  };
  issue(0);
  for (int c = 0; c < nchunks; ++c) {
    const int kc = (c * KC) % SMZ_HP;          // column of this k-slab inside the staged slice
    if (kc == 0) {                             // every thread is past the previous slice (barrier ending the last slab)
      const int k0 = c * KC, w = min(SMZ_HP, net.kin_pad - k0);
      for (int e = tid; e < R * w; e += NT) {
        const int r = e / w, k = e % w;
        xs[r][k] = (row0 + r < n_rows && k0 + k < in_w) ? in[(size_t)(row0 + r) * in_w + k0 + k] : 0.f;
      }
    }
    if (c + 1 < nchunks) { issue(c + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const float(*w)[SMZ_HP] = wbuf[c & 1];
#pragma unroll
    for (int kk = 0; kk < KC; kk += 4) {
      const float4 a0 = *reinterpret_cast<const float4*>(&xs[ty * 2][kc + kk]);
      const float4 a1 = *reinterpret_cast<const float4*>(&xs[ty * 2 + 1][kc + kk]);
      const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b0 = *reinterpret_cast<const float4*>(&w[kk + q][tx * 8]);
        const float4 b1 = *reinterpret_cast<const float4*>(&w[kk + q][tx * 8 + 4]);
        const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[0][j] = fmaf(av0[q], bv[j], acc[0][j]);
          acc[1][j] = fmaf(av1[q], bv[j], acc[1][j]);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int r = ty * 2 + i;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = tx * 8 + j;
      out[r][c] = elu(acc[i][j] + net.in_b[c]);
    }
  }
  __syncthreads();
}

// in-layer + L tied hidden layers + concatenated heads.  Returns the buffer holding the head tile;
// *free_buf receives the other one.
__device__ float (*run_net(const SmzNetF32& net, int L, float (*in)[LD], float (*other)[LD], const int* idx_s,
                           float (*wbuf)[KC][SMZ_HP], float (**free_buf)[LD]))[LD] {
  float(*cur)[LD] = in;
  float(*nxt)[LD] = other;
  dense(net.in_wt, net.kin_pad, net.in_b, net.emb, idx_s, cur, nxt, true, wbuf);
  { auto t = cur; cur = nxt; nxt = t; }
  for (int l = 0; l < L; ++l) {
    dense(net.mid_wt, SMZ_HP, net.mid_b, nullptr, nullptr, cur, nxt, true, wbuf);
    auto t = cur; cur = nxt; nxt = t;
  }
  dense(net.head_wt, SMZ_HP, net.head_b, nullptr, nullptr, cur, nxt, false, wbuf);
  *free_buf = cur;
  return nxt;
}

// run_net for a network whose input is caller rows [n_rows][in_w] in global memory (the observation):
// the first layer streams them through x, the result lands in y.
__device__ float (*run_net_wide_in(const SmzNetF32& net, int L, const float* in, int in_w, int row0, int n_rows,
                                   float (*x)[LD], float (*y)[LD], float (*wbuf)[KC][SMZ_HP], float (**free_buf)[LD]))[LD] {
  dense_wide_in(net, in, in_w, row0, n_rows, x, y, wbuf);
  float(*cur)[LD] = y;
  float(*nxt)[LD] = x;
  for (int l = 0; l < L; ++l) {
    dense(net.mid_wt, SMZ_HP, net.mid_b, nullptr, nullptr, cur, nxt, true, wbuf);
    auto t = cur; cur = nxt; nxt = t;
  }
  dense(net.head_wt, SMZ_HP, net.head_b, nullptr, nullptr, cur, nxt, false, wbuf);
  *free_buf = cur;
  return nxt;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// scale_to_bound_action (mlp:349-357) of head columns [0,S) of row r -> next[r][0..63] (zero padded)
// and, when dst != null, the same 64 floats to global memory.  One warp per row.
__device__ void state_epilogue(const float* head_row, int S, float* next_row, float* dst) {
  const int lane = threadIdx.x & 31;
  const float v0 = lane < S ? head_row[lane] : 0.f, v1 = lane + 32 < S ? head_row[lane + 32] : 0.f;
  const float lo = warp_min(fminf(lane < S ? v0 : INFINITY, lane + 32 < S ? v1 : INFINITY));
  const float hi = warp_max(fmaxf(lane < S ? v0 : -INFINITY, lane + 32 < S ? v1 : -INFINITY));
  float scale = hi - lo;
  if (scale < 1e-5f) scale += 1e-5f;
  const float s0 = lane < S ? (v0 - lo) / scale : 0.f, s1 = lane + 32 < S ? (v1 - lo) / scale : 0.f;
  next_row[lane] = s0;
  next_row[lane + 32] = s1;
  if (dst) { dst[lane] = s0; dst[lane + 32] = s1; }
}

// inverse_transform_with_support (muzero_model.py:575-591) of S logits at logits[0..S)
__device__ float support_scalar(const float* logits, int S) {
  const int lane = threadIdx.x & 31;
  const float v0 = lane < S ? logits[lane] : -INFINITY, v1 = lane + 32 < S ? logits[lane + 32] : -INFINITY;
  const float m = warp_max(fmaxf(v0, v1));
  const float e0 = lane < S ? expf(v0 - m) : 0.f, e1 = lane + 32 < S ? expf(v1 - m) : 0.f;
  const float z = warp_sum(e0 + e1);
  const int half = S / 2;
  const float y = warp_sum((float)(lane - half) * (e0 / z) + (float)(lane + 32 - half) * (e1 / z));
  // same operation order as the torch expression (muzero_model.py:589-590), one rounding per op:
  // the sqrt(1 + small) - 1 cancellation amplifies a 1-ulp change ~1e-5 relative, so do not fuse.
  const float inner = __fadd_rn(1.f, __fmul_rn(0.004f, __fadd_rn(__fadd_rn(fabsf(y), 1.f), 0.001f)));
  const float t = __fdiv_rn(__fsub_rn(__fsqrt_rn(inner), 1.f), 0.002f);
  const float mag = __fsub_rn(__fmul_rn(t, t), 1.f);
  return y > 0.f ? mag : (y < 0.f ? -mag : 0.f);
}

// softmax of n <= 32 logits -> dst[0..n)
__device__ void policy_softmax(const float* logits, int n, float* dst) {
  const int lane = threadIdx.x & 31;
  const float v = lane < n ? logits[lane] : -INFINITY;
  const float m = warp_max(v);
  const float e = lane < n ? expf(v - m) : 0.f;
  const float z = warp_sum(e);
  if (lane < n) dst[lane] = e / z;
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT) k_net_sim(SmzArena a, SmzNetShape sh, SmzNetImageF32 img, int sim) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int n0 = a.branch_count[sim * 2 + 0], n1 = a.branch_count[sim * 2 + 1];
  const int t0 = (n0 + R - 1) / R, t1 = (n1 + R - 1) / R;
  int tile = blockIdx.x, branch, count;
  if (tile < t0) { branch = SMZ_BRANCH_AFTERSTATE; count = n0; }
  else if (tile < t0 + t1) { branch = SMZ_BRANCH_DYNAMICS; count = n1; tile -= t0; }
  else return;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid < R) {
    const int row = tile * R + tid;
    const int tree = row < count ? a.rows[smz_row_index(a, sim, branch, row)] : -1;
    sm.tree[tid] = tree;
    sm.idx[tid] = tree >= 0 ? a.leaf_action[tree] : -1;
    sm.slot[tid] = tree >= 0 ? a.leaf_slot[tree] : 0;
  }
  __syncthreads();
  // gather parent hidden rows (64 floats each) with 128-bit loads
  for (int e = tid; e < R * (SMZ_SP / 4); e += NT) {
    const int r = e / (SMZ_SP / 4), c4 = e % (SMZ_SP / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (sm.tree[r] >= 0)
      v = *reinterpret_cast<const float4*>(a.hidden + ((size_t)sm.slot[r] * a.B + sm.tree[r]) * SMZ_SP + c4 * 4);
    *reinterpret_cast<float4*>(&sm.x[r][c4 * 4]) = v;
  }
  __syncthreads();
  float(*fre)[LD];
  const SmzNetF32& dynnet = branch ? img.dyn : img.adyn;
  float(*head)[LD] = run_net(dynnet, sh.L, sm.x, sm.y, sm.idx, sm.w, &fre);
  for (int r = warp; r < R; r += NT / 32) {
    const int tree = sm.tree[r];
    float* dst = tree >= 0 ? a.hidden + ((size_t)(sim + 1) * a.B + tree) * SMZ_SP : nullptr;
    state_epilogue(head[r], sh.S, fre[r], dst);
    if (branch) {
      const float rew = support_scalar(&head[r][POL_OFF], sh.S);
      if (tree >= 0 && (tid & 31) == 0) a.out_reward[tree] = rew;
    }
  }
  __syncthreads();
  float(*fre2)[LD];
  const SmzNetF32& prednet = branch ? img.pred : img.apred;
  float(*head2)[LD] = run_net(prednet, sh.L, fre, head, nullptr, sm.w, &fre2);
  const int n = branch ? sh.A : sh.C;
  for (int r = warp; r < R; r += NT / 32) {
    const int tree = sm.tree[r];
    const float val = support_scalar(&head2[r][0], sh.S);
    if (tree < 0) continue;
    policy_softmax(&head2[r][POL_OFF], n, a.out_policy + (size_t)tree * a.W);
    if ((tid & 31) == 0) a.out_value[tree] = val;
  }
}

__global__ void __launch_bounds__(NT) k_net_root(SmzArena a, SmzNetShape sh, SmzNetImageF32 img, int n_trees,
                                                 const float* __restrict__ obs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, row0 = blockIdx.x * R;
  float(*fre)[LD];
  float(*head)[LD] = run_net_wide_in(img.repr, sh.L, obs, sh.obs, row0, n_trees, sm.x, sm.y, sm.w, &fre);
  for (int r = warp; r < R; r += NT / 32) {
    const int tree = row0 + r;
    state_epilogue(head[r], sh.S, fre[r], tree < n_trees ? a.hidden + (size_t)tree * SMZ_SP : nullptr);
  }
  __syncthreads();
  float(*fre2)[LD];
  float(*head2)[LD] = run_net(img.pred, sh.L, fre, head, nullptr, sm.w, &fre2);
  for (int r = warp; r < R; r += NT / 32) {
    const int tree = row0 + r;
    const float val = support_scalar(&head2[r][0], sh.S);
    if (tree >= n_trees) continue;
    policy_softmax(&head2[r][POL_OFF], sh.A, a.out_policy + (size_t)tree * a.W);
    if ((tid & 31) == 0) a.out_value[tree] = val;
  }
}

// stand-alone evaluation of one network on caller rows (smz_net_eval)
__global__ void __launch_bounds__(NT) k_net_eval(SmzNetShape sh, SmzNetImageF32 img, int which, int n_rows,
                                                 const float* __restrict__ in, const int* __restrict__ idx,
                                                 float* hidden_out, float* policy_out, float* value_out,
                                                 float* reward_out, int* code_out, int pstride) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, row0 = blockIdx.x * R;
  const bool from_obs = (which == 0 || which == 5);
  if (!from_obs) {
    for (int e = tid; e < R * SMZ_SP; e += NT) {
      const int r = e / SMZ_SP, c = e % SMZ_SP;
      sm.x[r][c] = row0 + r < n_rows ? in[(size_t)(row0 + r) * SMZ_SP + c] : 0.f;
    }
  }
  if (tid < R) sm.idx[tid] = (idx && row0 + tid < n_rows) ? idx[row0 + tid] : -1;
  __syncthreads();
  const SmzNetF32* nets[6] = {&img.repr, &img.pred, &img.adyn, &img.apred, &img.dyn, &img.enc};
  float(*fre)[LD];
  float(*head)[LD] = from_obs ? run_net_wide_in(*nets[which], sh.L, in, sh.obs, row0, n_rows, sm.x, sm.y, sm.w, &fre)
                              : run_net(*nets[which], sh.L, sm.x, sm.y, (which == 2 || which == 4) ? sm.idx : nullptr, sm.w, &fre);
  for (int r = warp; r < R; r += NT / 32) {
    const int row = row0 + r;
    const bool ok = row < n_rows;
    if (which == 0 || which == 2 || which == 4) {
      state_epilogue(head[r], sh.S, fre[r], (ok && hidden_out) ? hidden_out + (size_t)row * SMZ_SP : nullptr);
      if (which == 4) {
        const float rew = support_scalar(&head[r][POL_OFF], sh.S);
        if (ok && reward_out && lane == 0) reward_out[row] = rew;
      }
    } else if (which == 1 || which == 3) {
      const float val = support_scalar(&head[r][0], sh.S);
      if (ok && value_out && lane == 0) value_out[row] = val;
      if (ok && policy_out) policy_softmax(&head[r][POL_OFF], which == 1 ? sh.A : sh.C, policy_out + (size_t)row * pstride);
    } else {
      // Encoder (mlp:209-250): softmax over C code logits, one-hot argmax -> code index
      float* dst = fre[r];
      policy_softmax(&head[r][0], sh.C, dst);
      __syncwarp();
      float best = lane < sh.C ? dst[lane] : -1.f;
      int bi = lane < sh.C ? lane : 0x7fffffff;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
      }
      if (ok && policy_out && lane < sh.C) policy_out[(size_t)row * pstride + lane] = dst[lane];
      if (ok && code_out && lane == 0) code_out[row] = bi;
    }
  }
}

// ---- weight repacking: torch Linear W[out][in] -> transposed, padded Wt[k][128] ------------------
__global__ void k_pack_wt(float* __restrict__ dst, const float* __restrict__ src, int n_out, int in_stride, int col0,
                          int n_in, int dst_col) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out * n_in) return;
  const int o = i / n_in, k = i % n_in;
  dst[(size_t)k * SMZ_HP + dst_col + o] = src[(size_t)o * in_stride + col0 + k];
}
__global__ void k_pack_vec(float* __restrict__ dst, const float* __restrict__ src, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

struct Packer {
  const SmzNetShape& sh;
  const float* blob;
  float* image;
  size_t blob_off = 0, img_off = 0;
  cudaStream_t s;
  bool dry;
  float* alloc(size_t n) { float* p = image + img_off; img_off += n; return p; }
  void wt(float* dst, int n_out, int n_in_total, int col0, int n_in, int dst_col) {
    if (dry) return;
    const int n = n_out * n_in;
    k_pack_wt<<<(n + 255) / 256, 256, 0, s>>>(dst, blob + blob_off, n_out, n_in_total, col0, n_in, dst_col);
  }
  void vec(float* dst, size_t src_off, int n) {
    if (dry) return;
    k_pack_vec<<<(n + 255) / 256, 256, 0, s>>>(dst, blob + src_off, n);
  }
  // heads: list of (width, dst_col)
  SmzNetF32 net(int in_dim, int in_live, int kin_pad, bool has_emb, int n_heads, const int* widths, const int* cols) {
    SmzNetF32 o{};
    const int H = sh.H;
    float* in_wt = alloc((size_t)kin_pad * SMZ_HP);
    float* in_b = alloc(SMZ_HP);
    float* emb = has_emb ? alloc((size_t)sh.OH * SMZ_HP) : nullptr;
    wt(in_wt, H, in_dim, 0, in_live, 0);
    if (has_emb) wt(emb, H, in_dim, in_live, sh.OH, 0);
    blob_off += (size_t)H * in_dim;
    vec(in_b, blob_off, H);
    blob_off += H;
    float* mid_wt = alloc((size_t)SMZ_HP * SMZ_HP);
    float* mid_b = alloc(SMZ_HP);
    if (sh.L > 0) {
      wt(mid_wt, H, H, 0, H, 0);
      blob_off += (size_t)H * H;
      vec(mid_b, blob_off, H);
      blob_off += H;
    }
    float* head_wt = alloc((size_t)SMZ_HP * SMZ_HP);
    float* head_b = alloc(SMZ_HP);
    for (int h = 0; h < n_heads; ++h) {
      wt(head_wt, widths[h], H, 0, H, cols[h]);
      blob_off += (size_t)widths[h] * H;
      vec(head_b + cols[h], blob_off, widths[h]);
      blob_off += widths[h];
    }
    o.in_wt = in_wt; o.in_b = in_b; o.emb = emb; o.mid_wt = mid_wt; o.mid_b = mid_b;
    o.head_wt = head_wt; o.head_b = head_b; o.kin_pad = kin_pad;
    return o;
  }
  void all(SmzNetImageF32* out) {
    const int S = sh.S, A = sh.A, C = sh.C, OH = sh.OH;
    SmzNetImageF32 im{};
    { int w[1] = {S}, c[1] = {0}; im.repr = net(sh.obs, sh.obs, sh.obs_pad, false, 1, w, c); }
    { int w[2] = {A, S}, c[2] = {POL_OFF, 0}; im.pred = net(S, S, SMZ_SP, false, 2, w, c); }
    { int w[1] = {S}, c[1] = {0}; im.adyn = net(S + OH, S, SMZ_SP, true, 1, w, c); }
    { int w[2] = {C, S}, c[2] = {POL_OFF, 0}; im.apred = net(S, S, SMZ_SP, false, 2, w, c); }
    { int w[2] = {S, S}, c[2] = {POL_OFF, 0}; im.dyn = net(S + OH, S, SMZ_SP, true, 2, w, c); }
    { int w[1] = {C}, c[1] = {0}; im.enc = net(sh.obs, sh.obs, sh.obs_pad, false, 1, w, c); }
    if (out) *out = im;
  }
};

}  // namespace

size_t smz_net_f32_image_floats(const SmzNetShape& sh) {
  Packer p{sh, nullptr, nullptr, 0, 0, nullptr, true};
  p.all(nullptr);
  return p.img_off;
}

uint64_t smz_blob_floats(const SmzNetShape& sh) {
  Packer p{sh, nullptr, nullptr, 0, 0, nullptr, true};
  p.all(nullptr);
  return p.blob_off;
}

void smz_net_f32_pack(const SmzNetShape& sh, const float* blob_dev, float* image_dev, SmzNetImageF32* out,
                      cudaStream_t s) {
  cudaMemsetAsync(image_dev, 0, smz_net_f32_image_floats(sh) * sizeof(float), s);
  Packer p{sh, blob_dev, image_dev, 0, 0, s, false};
  p.all(out);
}

static void set_smem(const void* fn) {
  cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
}

void smz_net_f32_root(const SmzArena& a, const SmzNetShape& sh, const SmzNetImageF32& img, int n_trees,
                      const float* obs, cudaStream_t s) {
  set_smem((const void*)k_net_root);
  k_net_root<<<(n_trees + R - 1) / R, NT, sizeof(Smem), s>>>(a, sh, img, n_trees, obs);
}

void smz_net_f32_sim(const SmzArena& a, const SmzNetShape& sh, const SmzNetImageF32& img, int n_trees, int sim,
                     cudaStream_t s) {
  set_smem((const void*)k_net_sim);
  k_net_sim<<<(n_trees + R - 1) / R + 1, NT, sizeof(Smem), s>>>(a, sh, img, sim);
}

void smz_net_f32_eval(const SmzNetShape& sh, const SmzNetImageF32& img, int which, int n_rows, const float* in,
                      const int* idx, float* hidden_out, float* policy_out, float* value_out, float* reward_out,
                      int* code_out, int policy_stride, cudaStream_t s) {
  set_smem((const void*)k_net_eval);
  k_net_eval<<<(n_rows + R - 1) / R, NT, sizeof(Smem), s>>>(sh, img, which, n_rows, in, idx, hidden_out, policy_out,
                                                             value_out, reward_out, code_out, policy_stride);
}
