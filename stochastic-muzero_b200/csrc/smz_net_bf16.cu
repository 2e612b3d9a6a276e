// smz_net_bf16.cu — the per-simulation network step on the 5th-generation tensor cores (sm_100a).
//
// One CTA (128 threads = 128 TMEM lanes = 128 leaves) pushes a tile of leaves through a whole
// network pair — e.g. Dynamics (mlp:167-206) then Prediction (mlp:47-83): 2*(L+2) dependent GEMM
// layers — without leaving the SM:
//   * the layer's weight tile (B operand, bf16, <= 32 KB, pre-laid-out in the UMMA canonical K-major
//     no-swizzle form by k_pack_bf16) streams global -> shared with cp.async.bulk (TMA bulk copy,
//     SASS UBLKCP) into a 2-deep ring, completion on an mbarrier, two layers ahead of the math;
//   * one thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=128, K=16 per instruction),
//     A = the activations in shared memory (bf16, written by the previous epilogue in canonical
//     layout), D = fp32 accumulators in TMEM; tcgen05.commit signals an mbarrier;
//   * the epilogue is row-per-thread: tcgen05.ld 32 lanes x 32 columns per warp, bias + ELU in fp32,
//     pack to bf16 and store straight into the next layer's A operand (conflict-free 16-byte stores);
//     the head layers finish scale_to_bound_action (mlp:349-357), softmax on the policy (:837) and
//     inverse_transform_with_support (muzero_model.py:575-591) thread-locally — no shuffles.
// The one-hot action / chance code (muzero_model.py:496-509) is folded into the first GEMM as 16 or
// 32 extra K columns holding a single 1.0.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/smz.h"
#include "smz_net_bf16.h"
#include "smz_common.cuh"
#include "smz_tc_ptx.cuh"

namespace {

using namespace smz_tc;

constexpr int TM = 128;                 // rows (leaves) per CTA == MMA M
constexpr int NTHREADS = 512;           // 16 warps: 4 TMEM lane quarters x 4 column blocks
constexpr int TN = 128;                 // MMA N (all layers padded to 128 output channels)
constexpr int KMAX = 128;               // widest K
constexpr int MAXL = 24;                // layers per chain: 2 * (L + 2), L <= 10
constexpr int A_BYTES = TM * KMAX * 2;  // 32 KB activation operand
constexpr int W_BYTES = TN * KMAX * 2;  // 32 KB weight operand (one ring slot)
constexpr int CHUNK_A = TM * 16;        // bytes between K-chunks (8 bf16) of the A operand: LBO
constexpr int CHUNK_W = TN * 16;        // same for the B operand
constexpr int POL_OFF = 64;             // column of the second head inside a head tile

enum LayerKind { LK_HIDDEN = 0, LK_STATE = 1, LK_STATE_REWARD = 2, LK_PRED = 3, LK_CODE = 4 };
enum InputKind { IN_GATHER = 0, IN_OBS = 1, IN_ROWS = 2 };

struct LayerRef {
  const __nv_bfloat16* w;   // [K/8][128][8] canonical image
  int K;                    // multiple of 16
  int kind;
};

struct Chain {
  LayerRef layer[MAXL];
  const float* bias;        // [n_layers][128]
  int n_layers;
  int n_policy;             // width of the policy / code head of this chain
  int kin;                  // K of the first layer
  int onehot_pad;           // 0, 16 or 32 one-hot columns after the 64 state columns
};

struct Job {
  int input_kind;
  int n_rows;               // rows when not compacted
  const float* in;          // IN_OBS: [n][obs]; IN_ROWS: [n][64]
  const int* idx;           // IN_ROWS: action / code per row (or null)
  int obs;                  // IN_OBS width
  float* hidden_dst;        // fp32 rows [index][64] (stand-alone evaluation) or null
  __nv_bfloat16* hidden16_dst;  // bf16 rows [index][64] in the arena's hidden store, or null
  float* policy_dst;        // [index][pstride] or null
  float* value_dst;
  float* reward_dst;
  int* code_dst;
  int pstride;
  int S;
  long long* timeline;      // debug: clock64 stamps of CTA 0 (null = off)
  int stream_all;           // debug (SMZ_STREAM_ALL=1): stream every layer's weight tile even when it is already resident
};

struct Smem {
  alignas(1024) unsigned char a[A_BYTES];
  alignas(1024) unsigned char w[2][W_BYTES];
  float bias[MAXL][TN];
  unsigned long long wbar[2];
  unsigned long long mbar;
  unsigned long long bbar;
  unsigned int tmem_base;
  float4 part[4][TM];       // per-row partial reductions of the head epilogues, one slot per column block
};

// InstrDescriptor: D=f32 (bit 4), A=B=bf16 (bits 7, 10), both K-major, N>>3 at [17,23), M>>4 at [24,29)
constexpr unsigned IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(TN >> 3) << 17) | ((unsigned)(TM >> 4) << 24);

__device__ __forceinline__ void umma(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc, unsigned accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accum)
      : "memory");
}

// store 8 consecutive K values of row r (already bf16-packed) into the canonical A operand
__device__ __forceinline__ void a_store(unsigned char* a, int r, int kchunk, uint4 v) {
  // explicit st.shared (not a generic store): the .shared::cta proxy fence that follows must cover it
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(s32(a + kchunk * CHUNK_A + r * 16)), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}

// ELU with the exponential on the MUFU pipe: exp(x) - 1 = 2^(x*log2e) - 1 (abs error ~1e-7, far below
// the bf16 rounding the result gets next)
__device__ __forceinline__ float elu_fast(float x) { return x > 0.f ? x : ex2f(x * 1.4426950408889634f) - 1.f; }

// bulk copy of the weight tile of layer l of chain c into ring slot `slot` (w[slot]), completion on wbar[slot]
__device__ __forceinline__ void load_weight_tile(const Chain& c, int l, unsigned long long* wbar, unsigned char (*w)[W_BYTES], int slot) {
  const unsigned bytes = (unsigned)c.layer[l].K * TN * 2;
  mbar_expect_tx(&wbar[slot], bytes);
  bulk_g2s(w[slot], c.layer[l].w, bytes, &wbar[slot]);
}

// k_bf16_chain streams the K of a first layer wider than KMAX (an observation of more than 128 features) in slices of
// KMAX through the same ring: ring tile t < ns is slice t of layer 0, tile ns - 1 + l is layer l >= 1.  The image is
// K-major, so a slice is one contiguous piece of it.
__device__ __forceinline__ void load_ring_tile(const Chain& c, int t, int ns, unsigned long long* wbar, unsigned char (*w)[W_BYTES],
                                               int slot) {
  if (t >= ns) { load_weight_tile(c, t - ns + 1, wbar, w, slot); return; }
  const unsigned bytes = (unsigned)min(KMAX, c.layer[0].K - t * KMAX) * TN * 2;
  mbar_expect_tx(&wbar[slot], bytes);
  bulk_g2s(w[slot], c.layer[0].w + (size_t)t * KMAX * TN, bytes, &wbar[slot]);
}

// K-chunk kc (8 columns) of the one-hot block of a row whose action / code is act (-1 = none)
__device__ __forceinline__ uint4 onehot_chunk(int act, int kc) {
  unsigned w4[4] = {0, 0, 0, 0};
  if (act >= kc * 8 && act < kc * 8 + 8) {
    const int j = act - kc * 8;
    w4[j >> 1] = (j & 1) ? 0x3F800000u : 0x00003F80u;   // bf16 1.0 in the high / low half
  }
  return make_uint4(w4[0], w4[1], w4[2], w4[3]);
}

// A CTA with nothing to do: it must not exit while a bulk copy into its shared memory is still in flight, so thread 0
// waits for every copy it has issued (bbar: the bias table, or null; wbar[0] and, if wbar1, wbar[1]: the first weight
// tiles); then the TMEM allocation is given back.
__device__ __forceinline__ void idle_cta_exit(unsigned long long* bbar, unsigned long long* wbar, bool wbar1,
                                              const unsigned& tmem_base, unsigned ncols) {
  if (threadIdx.x == 0) {
    if (bbar) mbar_wait(bbar, 0);
    mbar_wait(&wbar[0], 0);
    if (wbar1) mbar_wait(&wbar[1], 0);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (threadIdx.x < 32) tmem_dealloc(tmem_base, ncols);
}

// ---- the head layer of a 128-row tile: thread (row r, column block cb) holds the 32 biased logits x of columns
//      32cb .. 32cb+31.  Columns [0,64) = state or value logits, [64,128) = reward or policy logits.  Row-wise
//      reductions span two column blocks: head_partials leaves this thread's partials in part[cb][r], the caller
//      synchronises, head_finish combines them.
__device__ __forceinline__ bool head_state_seg(int kind, int cb) { return (kind == LK_STATE || kind == LK_STATE_REWARD) && cb < 2; }
__device__ __forceinline__ bool head_soft_seg(int kind, int cb) {
  return (kind == LK_STATE_REWARD && cb >= 2) || (kind == LK_PRED && cb < 2);
}

__device__ __forceinline__ SoftPart head_partials(const float* x, int kind, int cb, int r, int S, float4 (*part)[TM]) {
  SoftPart sp{-1e30f, 0.f, 0.f};
  if (head_state_seg(kind, cb)) {
    float lo = INFINITY, hi = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      { lo = fminf(lo, x[j]); hi = fmaxf(hi, x[j]); }   // padded columns replicate column 0 (weight image)
    part[cb][r] = make_float4(lo, hi, 0.f, 0.f);
  } else if (head_soft_seg(kind, cb)) {
    sp = soft_part(x, (cb * 32) & 63, S);
    part[cb][r] = make_float4(sp.m, sp.z, sp.y, 0.f);
  }
  return sp;
}

// the bf16 state row piece of a head layer, whose global store the caller defers past its barrier (the proxy fence
// before it would otherwise wait for the store to land)
struct HeadStores {
  uint4 v[4];
  uint4* dst;               // -> the arena's bf16 hidden store, or null
  __device__ __forceinline__ void flush() const {
    if (dst) {             // the arena keeps hidden states in bf16: exactly what the next gather needs
#pragma unroll
      for (int q = 0; q < 4; ++q) dst[q] = v[q];
    }
  }
};

// second half: the state head becomes the next network's A operand (A: the tile's shared-memory operand) and leaves
// the normalised state in x, the value / reward head its scalar, the policy / code head its softmax (+ argmax for
// LK_CODE); index = output row (-1 = none)
__device__ __forceinline__ HeadStores head_finish(float* x, int kind, int cb, int r, SoftPart sp, const float4 (*part)[TM],
                                                  unsigned char* A, int index, const Job& job, int n_policy) {
  HeadStores st;
  st.dst = nullptr;
  const int c0 = cb * 32;
  if (head_state_seg(kind, cb)) {
    // scale_to_bound_action (mlp:349-357): bf16 copy to HBM and into the next network's A operand
    const float4 o = part[cb ^ 1][r];
    const float lo = fminf(part[cb][r].x, o.x), hi = fmaxf(part[cb][r].y, o.y);
    float scale = hi - lo;
    if (scale < 1e-5f) scale += 1e-5f;
    const float inv = 1.f / scale;
#pragma unroll
    for (int j = 0; j < 32; ++j) x[j] = (x[j] - lo) * inv;   // padded columns: finite copies, zero weights next
    if (index >= 0 && job.hidden16_dst) st.dst = reinterpret_cast<uint4*>(job.hidden16_dst + (size_t)index * SMZ_SP + c0);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      st.v[q] = make_uint4(pack_bf16(x[q * 8 + 0], x[q * 8 + 1]), pack_bf16(x[q * 8 + 2], x[q * 8 + 3]),
                           pack_bf16(x[q * 8 + 4], x[q * 8 + 5]), pack_bf16(x[q * 8 + 6], x[q * 8 + 7]));
      a_store(A, r, cb * 4 + q, st.v[q]);
    }
  } else if (head_soft_seg(kind, cb) && (cb & 1) == 0) {
    const float4 o = part[cb + 1][r];
    const float v = support_scalar(sp, SoftPart{o.x, o.y, o.z});
    float* dst = (kind == LK_PRED) ? job.value_dst : job.reward_dst;
    if (index >= 0 && dst) dst[index] = v;
  } else if ((kind == LK_PRED && cb == 2) || (kind == LK_CODE && cb == 0)) {
    // policy softmax (muzero_model.py:837) / Encoder code distribution + argmax (mlp:209-250)
    float m = -1e30f, z = 0.f;
    int best = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (x[i] > m) { m = x[i]; best = i; }             // padded logits sit at -1e30 (bias)
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      x[i] = ex2f((x[i] - m) * 1.4426950408889634f);
      z += x[i];
    }
    if (index >= 0) {
      if (job.policy_dst) {
        float* dst = job.policy_dst + (size_t)index * job.pstride;
        const float inv = 1.f / z;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < n_policy) dst[i] = x[i] * inv;
      }
      if (kind == LK_CODE && job.code_dst) job.code_dst[index] = best;
    }
  }
  return st;
}


// ---------------------------------------------------------------------------------------------
// the fused chain kernel: 512 threads = 16 warps; warp w owns TMEM lanes 32*(w%4).. (rows) and the
// 32 accumulator columns 32*(w/4).. of every layer, so each SM sub-partition always has 4 warps to
// interleave around the TMEM-load / MUFU latencies.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NTHREADS, 1)
k_bf16_chain(SmzArena a, Chain chain0, Chain chain1, Job job, int sim) {
  extern __shared__ unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool stamp = job.timeline && blockIdx.x == 0 && tid == 0;
  if (stamp) job.timeline[0] = clock64();
  const int r = (warp & 3) * 32 + lane;   // row of the tile == TMEM lane
  const int cb = warp >> 2;               // column block: accumulator columns 32*cb .. 32*cb+31

  // ---- which rows does this CTA own?  Gather launches use a static split: CTAs [0, T) serve the
  //      afterstate rows, [T, 2T) the dynamics rows (T = tiles of the whole batch), so the branch —
  //      and with it the weight chain — is known before the previous kernel has finished. -------------
  int tile = blockIdx.x, branch = 0;
  if (job.input_kind == IN_GATHER) {
    const int T = (job.n_rows + TM - 1) / TM;
    branch = tile >= T;
    tile -= branch * T;
  }
  const Chain& ch = branch ? chain1 : chain0;
  // K slices of the first layer (1 unless an observation is wider than KMAX); see load_ring_tile.  Ring tile and
  // accumulator-barrier phase of layer l: t = l + ns - 1.
  const int ns = (ch.kin + KMAX - 1) / KMAX;
  const int n_tiles = ch.n_layers + ns - 1;

  // ---- barriers + first weight tiles (one thread), TMEM allocation (warp 0): all of it overlaps the
  //      dependent global loads of the gather below; one barrier publishes everything ----------------
  if (tid == 0) {
    mbar_init(&sm.wbar[0], 1);
    mbar_init(&sm.wbar[1], 1);
    mbar_init(&sm.mbar, 1);
    mbar_init(&sm.bbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned bbytes = (unsigned)ch.n_layers * TN * 4;
    mbar_expect_tx(&sm.bbar, bbytes);
    bulk_g2s(sm.bias, ch.bias, bbytes, &sm.bbar);
    load_ring_tile(ch, 0, ns, sm.wbar, sm.w, 0);
    if (n_tiles > 1) load_ring_tile(ch, 1, ns, sm.wbar, sm.w, 1);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&sm.tmem_base, TN);

  // ---- everything above is independent of the previous kernel; from here on we read its results ---
  smz_pdl_wait();
  // only now may the tree kernel of this simulation start: its prologue mirrors the tree arena into shared memory,
  // which the PREVIOUS tree kernel (complete once the wait above returns) was still writing
  smz_pdl_launch_dependents();
  int count = job.n_rows;
  if (job.input_kind == IN_GATHER) count = a.branch_count[sim * 2 + branch];
  const int row = tile * TM + r;
  const bool valid = row < count;
  if (tile * TM >= count) {
    idle_cta_exit(&sm.bbar, sm.wbar, n_tiles > 1, sm.tmem_base, TN);
    return;
  }

  // K slice s of this thread's observation row, K-chunks cb, cb + 4, cb + 8, cb + 12 (8 columns each), packed to bf16;
  // loaded into registers first, so that the next slice's loads are in flight while the tensor core works on this one
  auto load_obs_slice = [&](int s, uint4 (&o)[4]) {
    const int k0 = s * KMAX;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = k0 + (cb + 4 * i) * 8 + j;
        v[j] = (valid && c < job.obs) ? job.in[(size_t)row * job.obs + c] : 0.f;
      }
      o[i] = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    }
  };
  auto store_obs_slice = [&](int s, const uint4 (&o)[4]) {
    const int kw = min(KMAX, ch.kin - s * KMAX);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if ((cb + 4 * i) * 8 < kw) a_store(sm.a, r, cb + 4 * i, o[i]);
  };

  // ---- stage the first A operand: bf16, canonical K-major layout; thread (r, cb) fills its K-chunks ---
  int index = -1;      // tree id (gather) or caller row: where this row's outputs go
  {
    if (job.input_kind == IN_OBS) {
      index = valid ? row : -1;
      uint4 o[4];
      load_obs_slice(0, o);
      store_obs_slice(0, o);
    } else {
      const float* src = nullptr;
      const __nv_bfloat16* src16 = nullptr;   // arena rows are already bf16: copied straight into the operand
      int act = -1;
      if (valid) {
        if (job.input_kind == IN_GATHER) {
          const int4 rec = a.rows4[smz_row_index(a, sim, branch, row)];     // {tree, parent slot, action, -}
          index = rec.x;
          src16 = reinterpret_cast<const __nv_bfloat16*>(a.hidden) + ((size_t)rec.y * a.B + index) * SMZ_SP;
          act = rec.z;
        } else {
          index = row;
          src = job.in + (size_t)row * SMZ_SP;
          act = job.idx ? job.idx[row] : -1;
        }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int kc = cb * 2 + q;
        uint4 o = make_uint4(0, 0, 0, 0);
        if (valid && src16) {
          o = *reinterpret_cast<const uint4*>(src16 + kc * 8);
        } else if (valid) {
          const float4 lo = *reinterpret_cast<const float4*>(src + kc * 8);
          const float4 hi = *reinterpret_cast<const float4*>(src + kc * 8 + 4);
          o = make_uint4(pack_bf16(lo.x, lo.y), pack_bf16(lo.z, lo.w), pack_bf16(hi.x, hi.y), pack_bf16(hi.z, hi.w));
        }
        a_store(sm.a, r, kc, o);
      }
      for (int kc = cb; kc < ch.onehot_pad / 8; kc += 4) a_store(sm.a, r, 8 + kc, onehot_chunk(act, kc));   // columns 64 + act
    }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = sm.tmem_base;

  // ---- a first layer wider than KMAX: every K slice but the last accumulates into the layer-0 accumulator; the
  //      last one is layer 0 of the loop below -------------------------------------------------------------------
  if (tid == 0) mbar_wait(&sm.wbar[0], 0);
  for (int s = 0; s + 1 < ns; ++s) {
    if (tid == 0) {
      tc_fence_after();
      const unsigned long long ad = umma_desc(s32(sm.a), CHUNK_A, 128), bd = umma_desc(s32(sm.w[s & 1]), CHUNK_W, 128);
#pragma unroll
      for (int k = 0; k < 8; ++k)
        umma(tmem, ad + (unsigned long long)(k * ((2 * CHUNK_A) >> 4)), bd + (unsigned long long)(k * ((2 * CHUNK_W) >> 4)),
             (s > 0 || k > 0) ? 1u : 0u);
      umma_commit(&sm.mbar);
      mbar_wait(&sm.wbar[(s + 1) & 1], ((s + 1) >> 1) & 1);
    }
    uint4 o[4];
    load_obs_slice(s + 1, o);
    mbar_wait(&sm.mbar, s & 1);
    __syncwarp();
    tc_fence_after();
    if (tid == 0 && s + 2 < n_tiles) load_ring_tile(ch, s + 2, ns, sm.wbar, sm.w, s & 1);   // ring slot s&1 is free again
    store_obs_slice(s + 1, o);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  mbar_wait(&sm.bbar, 0);

  const unsigned taddr = tmem + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)(cb * 32);
  const int S = job.S;
  const int c0 = cb * 32;

  // ---- the layer loop ---------------------------------------------------------------------------------
  for (int l = 0; l < ch.n_layers; ++l) {
    const int K = l ? ch.layer[l].K : ch.kin - (ns - 1) * KMAX, kind = ch.layer[l].kind;
    const int t = l + ns - 1;          // ring tile of this layer (= completed accumulator phases before it)
    if (tid == 0) {
      if (stamp) job.timeline[1 + l * 4 + 0] = clock64();
      tc_fence_after();
      // descriptors advance by two K-chunks per MMA: only the 14-bit start-address field changes
      const unsigned long long ad = umma_desc(s32(sm.a), CHUNK_A, 128), bd = umma_desc(s32(sm.w[t & 1]), CHUNK_W, 128);
      const int nk = K / 16;
      umma(tmem, ad, bd, (l == 0 && ns > 1) ? 1u : 0u);
#pragma unroll
      for (int k = 1; k < 8; ++k)
        if (k < nk) umma(tmem, ad + (unsigned long long)(k * ((2 * CHUNK_A) >> 4)), bd + (unsigned long long)(k * ((2 * CHUNK_W) >> 4)), 1u);
      umma_commit(&sm.mbar);
      if (stamp) job.timeline[1 + l * 4 + 1] = clock64();
      // the next layer's weights were requested two layers ago: absorb that wait while the MMAs run
      if (l + 1 < ch.n_layers) mbar_wait(&sm.wbar[(t + 1) & 1], ((t + 1) >> 1) & 1);
    }
    mbar_wait(&sm.mbar, t & 1);
    __syncwarp();       // tcgen05.ld below is .sync.aligned: reconverge after the spin loop
    if (stamp) job.timeline[1 + l * 4 + 2] = clock64();
    tc_fence_after();
    if (tid == 0 && l + 2 < ch.n_layers) load_weight_tile(ch, l + 2, sm.wbar, sm.w, t & 1);   // ring slot t&1 is free again
    __syncwarp();
    const float* bias = sm.bias[l] + c0;

    HeadStores pend;              // global stores deferred past the barrier
    pend.dst = nullptr;
    float4* pend32_dst = nullptr;
    float x[32];
    {
      unsigned raw[32];
      tmem_ld16_nowait(taddr, raw);
      tmem_wait_ld();
      tmem_ld16_nowait(taddr + 16, raw + 16);      // in flight while the first half is processed
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        x[j] = __uint_as_float(raw[j]) + bias[j];
        if (kind == LK_HIDDEN) x[j] = elu_fast(x[j]);
      }
      tmem_wait_ld();
#pragma unroll
      for (int j = 16; j < 32; ++j) {
        x[j] = __uint_as_float(raw[j]) + bias[j];
        if (kind == LK_HIDDEN) x[j] = elu_fast(x[j]);
      }
    }

    long long* hs = (stamp && kind != LK_HIDDEN) ? job.timeline + 1 + 4 * MAXL + (kind == LK_PRED ? 8 : 0) : nullptr;
    if (hs) hs[0] = clock64();
    if (kind == LK_HIDDEN) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        a_store(sm.a, r, cb * 4 + q,
                make_uint4(pack_bf16(x[q * 8 + 0], x[q * 8 + 1]), pack_bf16(x[q * 8 + 2], x[q * 8 + 3]),
                           pack_bf16(x[q * 8 + 4], x[q * 8 + 5]), pack_bf16(x[q * 8 + 6], x[q * 8 + 7])));
    } else {
      const SoftPart sp = head_partials(x, kind, cb, r, S, sm.part);
      if (hs) hs[1] = clock64();
      __syncthreads();
      if (hs) hs[2] = clock64();
      pend = head_finish(x, kind, cb, r, sp, sm.part, sm.a, index, job, ch.n_policy);
      // stand-alone evaluation (only this kernel serves it) also returns the normalised state in fp32
      if (head_state_seg(kind, cb) && index >= 0 && job.hidden_dst)
        pend32_dst = reinterpret_cast<float4*>(job.hidden_dst + (size_t)index * SMZ_SP + cb * 32);
    }
    if (hs) hs[3] = clock64();
    // make the new A operand visible to the tensor core (async proxy) and retire the TMEM reads.
    // Global stores come AFTER the barrier: the proxy fence would otherwise wait for them to land.
    if (l + 1 < ch.n_layers) {
      fence_async_smem();
      tc_fence_before();
      __syncthreads();
    }
    if (hs) hs[4] = clock64();
    pend.flush();
    if (pend32_dst) {
#pragma unroll
      for (int q = 0; q < 8; ++q) pend32_dst[q] = make_float4(x[q * 4], x[q * 4 + 1], x[q * 4 + 2], x[q * 4 + 3]);
    }
    if (stamp) job.timeline[1 + l * 4 + 3] = clock64();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, TN);
}

// ---------------------------------------------------------------------------------------------
// K-pipelined chain (simulation step only).  A dedicated issuer warp feeds the tensor core; the 16 epilogue warps
// walk each hidden layer in ROUNDS of 64 (or 32) output columns (every warp takes a 16- (8-) column slice of the
// round for its 32 rows).  When a round's columns of layer l are in the A operand, the issuer launches the two K-steps of
// layer l+1 that consume exactly those columns — the MMA issue (~76 cycles per instruction) and most of the
// commit -> wake-up latency disappear under the epilogue instead of following it.  Accumulators are
// double-buffered in TMEM (columns [0,128) / [128,256) for even / odd layers); there is no CTA-wide barrier on
// the hidden-layer path:
//   named barrier 2+c  "columns 32c..32c+31 of the next layer's A operand are written": the 512 epilogue threads
//                      bar.arrive (non-blocking), the issuer warp bar.sync's
//   dbar[b]            "accumulator buffer b holds a finished layer"  (tcgen05.commit -> mbarrier)
// Two things learnt the hard way (profiles/r1_bf16_ncu_summary.md): (1) the issuer loop must be walked by the
// WHOLE warp with one lane issuing — a loop run by a single lane lets ptxas move loop-carried operands to uniform
// registers with plain R2UR; (2) handing the A operand over through an mbarrier (arrive by the writers, try_wait
// by the issuer) gave stale / garbage operand rows on B200 no matter which proxy fences were added on either
// side, while the same hand-off through a named barrier is correct — so named barriers it is.
// ---------------------------------------------------------------------------------------------
constexpr int NEPI = NTHREADS;            // 512 epilogue threads
constexpr int NPIPE = NTHREADS + 32;      // + issuer warp

struct SmemPipe {
  alignas(1024) unsigned char a[A_BYTES];
  alignas(1024) unsigned char w[2][W_BYTES];
  float bias[2][MAXL][TN];   // both chains: the branch of a tile is known only after the dependency wait
  unsigned long long wbar[2];
  unsigned long long dbar[2];
  unsigned long long bbar;
  unsigned int tmem_base;
  float4 part[4][TM];
};

__device__ __forceinline__ void epi_sync() { __syncwarp(); asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory"); }
// producer / consumer split of a named barrier: the 512 epilogue threads arrive (non-blocking), the issuer warp waits
__device__ __forceinline__ void nb_arrive(int id) { __syncwarp(); asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(NPIPE) : "memory"); }
__device__ __forceinline__ void nb_sync(int id) { __syncwarp(); asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NPIPE) : "memory"); }

// Row record {tree, parent slot, action, -} of position pos of the simulation's row array, and the NC 16-byte chunks
// kc0 .. kc0+NC-1 of the parent's bf16 hidden row: copied next to the record by the descent (a.xin: one dependent load
// less), else gathered from the arena.  Positions beyond the live rows hold stale but in-range records (zeroed at create).
template <int NC>
__device__ __forceinline__ int4 load_row(const SmzArena& a, int sim, int pos, int kc0, uint4* hrow) {
  const size_t ri = (size_t)(sim & 1) * a.row_cap + pos;
  int4 rec = a.rows4[ri];
  if (a.xin) {
#pragma unroll
    for (int q = 0; q < NC; ++q) hrow[q] = a.xin[ri * 8 + kc0 + q];
  } else {
    rec.x = min(max(rec.x, 0), a.B - 1);
    rec.y = min(max(rec.y, 0), a.N);
    const __nv_bfloat16* src16 = reinterpret_cast<const __nv_bfloat16*>(a.hidden) + ((size_t)rec.y * a.B + rec.x) * SMZ_SP;
#pragma unroll
    for (int q = 0; q < NC; ++q) hrow[q] = *reinterpret_cast<const uint4*>(src16 + (kc0 + q) * 8);
  }
  return rec;
}

// The issuer warp's weight ring: layer l of the CTA's chain lives in slot (l + branch) & 1 (layer 0 of chain b was
// prefetched into slot b before the branch was known).  The hidden layers of a network share ONE weight tile (the
// reference ties them, mlp:31-37): a tile that is already resident in its slot is not streamed again — 6 bulk copies
// per chain instead of 12.  nfill / nseen = fills issued to / waited for on each slot.  Every counter and resident-tile
// pointer is a scalar member, kept in registers (an indexed array would not be).  The whole warp calls every method;
// lane 0 issues the copies.
struct WeightRing {
  const Chain& ch;
  unsigned long long* wbar;       // [2]
  unsigned char (*w)[W_BYTES];    // [2]
  int branch, lane;
  unsigned nfill0, nfill1, nseen0, nseen1;
  const __nv_bfloat16 *res0, *res1;

  __device__ __forceinline__ WeightRing(const Chain& c, unsigned long long* bars, unsigned char (*slots)[W_BYTES], int lane_)
      : ch(c), wbar(bars), w(slots), branch(0), lane(lane_), nfill0(1u), nfill1(1u), nseen0(0u), nseen1(0u),
        res0(nullptr), res1(nullptr) {}
  // slot `branch` holds layer 0 (fill 0); the other slot's fill 0 was the unused chain's layer 0: layer 1 replaces it
  // as soon as it has landed
  __device__ __forceinline__ void start(int branch_, int nl) {
    branch = branch_;
    if (branch) res1 = ch.layer[0].w; else res0 = ch.layer[0].w;
    if (nl > 1) {
      const int s1 = branch ^ 1;
      mbar_wait(&wbar[s1], 0);
      if (lane == 0) load_weight_tile(ch, 1, wbar, w, s1);
      if (s1) { nseen1 = 1u; nfill1 = 2u; res1 = ch.layer[1].w; } else { nseen0 = 1u; nfill0 = 2u; res0 = ch.layer[1].w; }
      __syncwarp();
    }
  }
  // the slot of layer l, once its tile has landed
  __device__ __forceinline__ int wait(int l) {
    const int slot = (l + branch) & 1;
    const unsigned seen = slot ? nseen1 : nseen0;
    if (seen < (slot ? nfill1 : nfill0)) {
      mbar_wait(&wbar[slot], seen & 1u);
      if (slot) ++nseen1; else ++nseen0;
    }
    return slot;
  }
  // layer l + 2 goes into the slot of layer l — unless it is resident there already (stream_all: always) — once the
  // MMAs that read that slot have completed: mbarrier `done`, phase `parity`
  __device__ __forceinline__ void refill(int l, int nl, bool stream_all, unsigned long long* done, unsigned parity) {
    const int slot = (l + branch) & 1;
    if (l + 2 < nl && ((slot ? res1 : res0) != ch.layer[l + 2].w || stream_all)) {
      mbar_wait(done, parity);
      if (lane == 0) load_weight_tile(ch, l + 2, wbar, w, slot);
      if (slot) { ++nfill1; res1 = ch.layer[l + 2].w; } else { ++nfill0; res0 = ch.layer[l + 2].w; }
      __syncwarp();
    }
  }
};

// Hidden layer of a 128-row tile in NR = 2 rounds of 64 columns (every round costs a proxy fence; two rounds measured
// best): this warp owns a 16-column slice of every round for its 32 rows.  All slices are requested at once (one exposed
// TMEM latency per layer); each round then goes bias + ELU -> bf16 -> A operand and is handed to the issuer through
// named barrier bar0 + round.  taddr: TMEM lane address of the tile's accumulator; bias: the layer's bias row.
constexpr int NR = 2;
__device__ __forceinline__ void hidden_rounds(unsigned char* A, unsigned taddr, const float* bias, int bar0, int r, int cb) {
  constexpr int SL = 32 / NR;              // slice width: 16 columns
  constexpr int RC = TN / NR;              // columns per round
  const int j0 = cb * SL;
  unsigned raw[NR][SL];
#pragma unroll
  for (int c = 0; c < NR; ++c) tmem_ld16_nowait(taddr + c * RC + j0, raw[c]);
  tmem_wait_ld();
#pragma unroll
  for (int c = 0; c < NR; ++c) {
    const float* b = bias + c * RC + j0;
    float x[SL];
#pragma unroll
    for (int i = 0; i < SL; ++i) x[i] = elu_fast(__uint_as_float(raw[c][i]) + b[i]);
#pragma unroll
    for (int q = 0; q < SL / 8; ++q)
      a_store(A, r, (c * RC + j0) / 8 + q,
              make_uint4(pack_bf16(x[q * 8 + 0], x[q * 8 + 1]), pack_bf16(x[q * 8 + 2], x[q * 8 + 3]),
                         pack_bf16(x[q * 8 + 4], x[q * 8 + 5]), pack_bf16(x[q * 8 + 6], x[q * 8 + 7])));
    fence_async_smem();
    if (c == NR - 1) tc_fence_before();
    nb_arrive(bar0 + c);
  }
}

__global__ void __launch_bounds__(NPIPE, 1)
k_bf16_chain_pipe(SmzArena a, Chain chain0, Chain chain1, Job job, int sim) {
  extern __shared__ unsigned char smem_raw[];
  SmemPipe& sm = *reinterpret_cast<SmemPipe*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_issuer_warp = warp == NEPI / 32;
  const int r = (warp & 3) * 32 + lane;   // epilogue role: row of the tile == TMEM lane
  const int cb = (warp >> 2) & 3;         // head layers: 32-column block; hidden layers: 16-column slice of a round

  // CTA i owns positions [i * 128, (i + 1) * 128) of the simulation's row array (smz_common.cuh): afterstate rows from the
  // bottom, dynamics rows from the top, never both in one tile — no CTA is launched for an empty tile of the other branch
  const int tile = blockIdx.x;
  const int nl = chain0.n_layers;          // == chain1.n_layers
  long long* tl = (job.timeline && blockIdx.x == 0 && lane == 0) ? job.timeline : nullptr;   // debug stamps
  if (tl && tid == 0) tl[0] = clock64();

  if (tid == 0) {
    mbar_init(&sm.wbar[0], 1); mbar_init(&sm.wbar[1], 1);
    mbar_init(&sm.dbar[0], 1); mbar_init(&sm.dbar[1], 1);
    mbar_init(&sm.bbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned bbytes = (unsigned)nl * TN * 4;
    mbar_expect_tx(&sm.bbar, 2 * bbytes);
    bulk_g2s(sm.bias[0], chain0.bias, bbytes, &sm.bbar);
    bulk_g2s(sm.bias[1], chain1.bias, bbytes, &sm.bbar);
    load_weight_tile(chain0, 0, sm.wbar, sm.w, 0);   // the first weight tile of BOTH chains: the branch is not known yet
    load_weight_tile(chain1, 0, sm.wbar, sm.w, 1);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&sm.tmem_base, 2 * TN);
  smz_pdl_wait();
  // only now may the tree kernel of this simulation start: its prologue mirrors the tree arena into shared memory,
  // which the PREVIOUS tree kernel (complete once the wait above returns) was still writing
  smz_pdl_launch_dependents();
  // The row record and the parent's hidden row are requested together with the branch counts (one L2 round trip).
  int4 rec = make_int4(0, 0, 0, 0);
  uint4 hrow[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
  const int pos = tile * TM + r;
  if (!is_issuer_warp) rec = load_row<2>(a, sim, pos, cb * 2, hrow);
  const int count0 = a.branch_count[sim * 2], count1 = a.branch_count[sim * 2 + 1];
  const int top1 = a.row_top - count1;      // dynamics rows occupy [top1, row_top)
  const int branch = tile * TM < count0 ? 0 : ((tile + 1) * TM > top1 ? 1 : -1);
  if (branch < 0) {
    idle_cta_exit(&sm.bbar, sm.wbar, true, sm.tmem_base, 2 * TN);
    return;
  }
  const Chain& ch = branch ? chain1 : chain0;
  // TMEM address + barrier inits become visible to everybody here
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = sm.tmem_base;

  if (is_issuer_warp) {
    // =========================== issuer warp: weights ring + tcgen05.mma =======================================
    const unsigned long long ad = umma_desc(s32(sm.a), CHUNK_A, 128);
    WeightRing ring(ch, sm.wbar, sm.w, lane);
    ring.start(branch, nl);
    for (int l = 0; l < nl; ++l) {
      const int nk = ch.layer[l].K / 16;
      const int slot = ring.wait(l);
      const unsigned long long bd = umma_desc(s32(sm.w[slot]), CHUNK_W, 128);
      const unsigned d = tmem + (unsigned)((l & 1) * TN);
      for (int c = 0; c < NR; ++c) {
        // the A columns of round c of this layer are in shared memory.  Every barrier is consumed for every layer
        // (also for column blocks a short-K layer does not read): arrivals and waits stay paired.
        nb_sync(2 + c);
        if (tl && c == NR - 1) tl[1 + l * 4 + 0] = clock64();   // last round of the layer is in the A operand
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = (8 / NR) * c; k < (8 / NR) * (c + 1); ++k)
            if (k < nk)
              umma(d, ad + (unsigned long long)(k * ((2 * CHUNK_A) >> 4)), bd + (unsigned long long)(k * ((2 * CHUNK_W) >> 4)),
                   k > 0 ? 1u : 0u);
        }
        __syncwarp();
      }
      if (lane == 0) umma_commit(&sm.dbar[l & 1]);
      if (tl) tl[1 + l * 4 + 1] = clock64();
      __syncwarp();
      ring.refill(l, nl, job.stream_all, &sm.dbar[l & 1], (l >> 1) & 1);   // the slot is reusable once these MMAs have completed
    }
  } else {
    // =========================== epilogue warps =================================================================
    const bool valid = branch ? pos >= top1 : pos < count0;
    const int index = valid ? rec.x : -1;
    const float (*cbias)[TN] = sm.bias[branch];
    {   // stage the first A operand: thread (r, cb) fills K-chunks 2cb, 2cb+1 (+ its share of the one-hot chunks)
      const int act = valid ? rec.z : -1;
#pragma unroll
      for (int q = 0; q < 2; ++q) a_store(sm.a, r, cb * 2 + q, valid ? hrow[q] : make_uint4(0, 0, 0, 0));
      for (int kc = cb; kc < ch.onehot_pad / 8; kc += 4) a_store(sm.a, r, 8 + kc, onehot_chunk(act, kc));
    }
    fence_async_smem();
    for (int c = 0; c < NR; ++c) nb_arrive(2 + c);
    mbar_wait(&sm.bbar, 0);
    const unsigned lane_t = tmem + ((unsigned)((warp & 3) * 32) << 16);
    const int S = job.S;

    for (int l = 0; l < nl; ++l) {
      const int kind = ch.layer[l].kind;
      const unsigned dcol = (unsigned)((l & 1) * TN);
      mbar_wait(&sm.dbar[l & 1], (l >> 1) & 1);
      if (tl && warp == 0) tl[1 + l * 4 + 2] = clock64();
      __syncwarp();
      tc_fence_after();
      if (kind == LK_HIDDEN) {
        hidden_rounds(sm.a, lane_t + dcol, cbias[l], 2, r, cb);
      } else {
        // head layers are not pipelined: row-wise reductions need all columns.  Warp (quarter, cb) owns the 32-column
        // block cb of its rows; barriers among the epilogue warps only.
        const int c0 = cb * 32;
        const float* bias = cbias[l] + c0;
        float x[32];
        tmem_ld32(lane_t + dcol + c0, x);
#pragma unroll
        for (int i = 0; i < 32; ++i) x[i] += bias[i];
        const SoftPart sp = head_partials(x, kind, cb, r, S, sm.part);
        epi_sync();
        const HeadStores pend = head_finish(x, kind, cb, r, sp, sm.part, sm.a, index, job, ch.n_policy);
        if (l + 1 < nl) {
          // the next network's A operand (K = 64: column blocks 0, 1); the other two barriers are consumed as well
          fence_async_smem();
          tc_fence_before();
          for (int c = 0; c < NR; ++c) nb_arrive(2 + c);
        }
        pend.flush();
      }
      if (tl && warp == 0) tl[1 + l * 4 + 3] = clock64();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 2 * TN);
}

// ---------------------------------------------------------------------------------------------
// Two tiles per CTA for batches of more than one wave (k_bf16_chain_pipeN<2>).  With one 128-leaf tile per SM the tensor
// pipe idles while the 16 epilogue warps work through a layer (~1800 cycles, MUFU / issue bound) and the epilogue warps
// idle while the layer's last K-steps complete (~600 cycles).  A CTA that owns TWO adjacent tiles of the row array (256
// positions: never both branches, see smz_common.cuh) alternates them: the epilogue warps do (tile 0, layer l), (tile 1,
// layer l), (tile 0, layer l + 1) ... and the issuer feeds tile 0's layer l + 1 while tile 1's layer l is in the
// epilogue — the contraction disappears behind the activation function.  Both tiles read the SAME weight tile
// (one ring, one stream of bulk copies per group); accumulators: one per tile, NT x 128 TMEM columns.
// ---------------------------------------------------------------------------------------------
// NT = tiles per CTA (2).  One accumulator per tile is enough (NT x 128 TMEM columns): an epilogue loads all of
// its tile's accumulator before it hands the first round of columns to the issuer, so the next layer's K-steps never
// overwrite values that are still to be read.
template <int NT>
struct SmemPipeN {
  alignas(1024) unsigned char a[NT][A_BYTES];
  alignas(1024) unsigned char w[2][W_BYTES];
  float bias[MAXL][TN];            // this CTA's chain, fetched once the branch is known
  unsigned long long wbar[2];
  unsigned long long dbar[NT];     // accumulator of tile t complete
  unsigned long long bbar;
  unsigned int tmem_base;
  float4 part[2][4][TM];           // head-layer exchange, alternating between consecutive tiles (no barrier between their head layers)
  int rowidx[NT][TM];              // tree id of every row of every tile (-1 = none)
};

template <int NT>
__global__ void __launch_bounds__(NPIPE, 1)
k_bf16_chain_pipeN(SmzArena a, Chain chain0, Chain chain1, Job job, int sim) {
  extern __shared__ unsigned char smem_raw[];
  SmemPipeN<NT>& sm = *reinterpret_cast<SmemPipeN<NT>*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_issuer_warp = warp == NEPI / 32;
  const int r = (warp & 3) * 32 + lane;   // epilogue role: row of a tile == TMEM lane
  const int cb = (warp >> 2) & 3;         // head layers: 32-column block; hidden layers: 16-column slice of a round
  const int group = blockIdx.x;           // positions [NT * 128 * group, NT * 128 * (group + 1)) of the row array
  const int nl = chain0.n_layers;

  if (tid == 0) {
    mbar_init(&sm.wbar[0], 1); mbar_init(&sm.wbar[1], 1);
#pragma unroll
    for (int t = 0; t < NT; ++t) mbar_init(&sm.dbar[t], 1);
    mbar_init(&sm.bbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    load_weight_tile(chain0, 0, sm.wbar, sm.w, 0);   // the first weight tile of BOTH chains: the branch is not known yet
    load_weight_tile(chain1, 0, sm.wbar, sm.w, 1);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&sm.tmem_base, NT * TN);
  smz_pdl_wait();
  smz_pdl_launch_dependents();
  // row records + parent hidden rows of both tiles, requested together with the branch counts
  int4 rec[NT];
  uint4 hrow[NT][2];
#pragma unroll
  for (int t = 0; t < NT; ++t) { rec[t] = make_int4(0, 0, 0, 0); hrow[t][0] = hrow[t][1] = make_uint4(0, 0, 0, 0); }
  if (!is_issuer_warp) {
#pragma unroll
    for (int t = 0; t < NT; ++t) rec[t] = load_row<2>(a, sim, (NT * group + t) * TM + r, cb * 2, hrow[t]);
  }
  const int count0 = a.branch_count[sim * 2], count1 = a.branch_count[sim * 2 + 1];
  const int top1 = a.row_top - count1;      // dynamics rows occupy [top1, row_top)
  const int lo = NT * group * TM;
  const int branch = lo < count0 ? 0 : (lo + NT * TM > top1 ? 1 : -1);
  if (branch < 0) {                // the bias table has not been requested yet
    idle_cta_exit(nullptr, sm.wbar, true, sm.tmem_base, NT * TN);
    return;
  }
  // which tiles carry rows (CTA-uniform bit mask): afterstate rows fill the group from below, dynamics rows from above
  unsigned actm = 0;
#pragma unroll
  for (int t = 0; t < NT; ++t)
    if (branch ? lo + (t + 1) * TM > top1 : lo + t * TM < count0) actm |= 1u << t;
  const int t_last = 31 - __clz(actm);      // the tile whose MMAs are issued last in every layer
  const Chain& ch = branch ? chain1 : chain0;
  if (tid == 0) {                           // this chain's bias table (12 KB), needed by the first epilogue
    const unsigned bbytes = (unsigned)nl * TN * 4;
    mbar_expect_tx(&sm.bbar, bbytes);
    bulk_g2s(sm.bias, ch.bias, bbytes, &sm.bbar);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = sm.tmem_base;

  if (is_issuer_warp) {
    // =========================== issuer warp: one weight ring, two tiles ======================================
    WeightRing ring(ch, sm.wbar, sm.w, lane);
    ring.start(branch, nl);
    for (int l = 0; l < nl; ++l) {
      const int nk = ch.layer[l].K / 16;
      const int slot = ring.wait(l);
      const unsigned long long bd = umma_desc(s32(sm.w[slot]), CHUNK_W, 128);
#pragma unroll 1
      for (int t = 0; t < NT; ++t) {
        if (!((actm >> t) & 1u)) continue;
        const unsigned long long ad = umma_desc(s32(sm.a[t]), CHUNK_A, 128);
        const unsigned d = tmem + (unsigned)(t * TN);
        for (int c = 0; c < NR; ++c) {
          nb_sync(2 + 2 * t + c);               // the A columns of round c of tile t are in shared memory
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
              if (k >= 4 * c && k < 4 * (c + 1) && k < nk)
                umma(d, ad + (unsigned long long)(k * ((2 * CHUNK_A) >> 4)), bd + (unsigned long long)(k * ((2 * CHUNK_W) >> 4)),
                     k > 0 ? 1u : 0u);
          }
          __syncwarp();
        }
        if (lane == 0) umma_commit(&sm.dbar[t]);
        __syncwarp();
      }
      // the slot is reusable once the MMAs of ALL tiles have completed (commits complete in issue order)
      ring.refill(l, nl, job.stream_all, &sm.dbar[t_last], l & 1);
    }
  } else {
    // =========================== epilogue warps: (tile 0, l), (tile 1, l), (tile 0, l + 1), ... =====================
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const int pos = lo + t * TM + r;
      const bool tact = (actm >> t) & 1u;
      const bool valid = tact && (branch ? pos >= top1 : pos < count0);
      if (cb == 0) sm.rowidx[t][r] = valid ? rec[t].x : -1;
      if (tact) {              // stage the first A operand of tile t
        const int act = valid ? rec[t].z : -1;
#pragma unroll
        for (int q = 0; q < 2; ++q) a_store(sm.a[t], r, cb * 2 + q, valid ? hrow[t][q] : make_uint4(0, 0, 0, 0));
        for (int kc = cb; kc < ch.onehot_pad / 8; kc += 4) a_store(sm.a[t], r, 8 + kc, onehot_chunk(act, kc));
      }
    }
    fence_async_smem();
#pragma unroll
    for (int t = 0; t < NT; ++t)
      if ((actm >> t) & 1u)
        for (int c = 0; c < NR; ++c) nb_arrive(2 + 2 * t + c);
    mbar_wait(&sm.bbar, 0);
    epi_sync();                              // rowidx is read by other threads from here on
    const float (*cbias)[TN] = sm.bias;
    const int S = job.S;

    for (int l = 0; l < nl; ++l) {
      const int kind = ch.layer[l].kind;
#pragma unroll 1
      for (int t = 0; t < NT; ++t) {
        if (!((actm >> t) & 1u)) continue;
        const int index_t = sm.rowidx[t][r];
        unsigned char* const A = sm.a[t];
        const unsigned lane_t = tmem + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)(t * TN);
        mbar_wait(&sm.dbar[t], l & 1);
        __syncwarp();
        tc_fence_after();
        if (kind == LK_HIDDEN) {
          hidden_rounds(A, lane_t, cbias[l], 2 + 2 * t, r, cb);
        } else {
          // head layers: row-wise reductions need all columns; warp (quarter, cb) owns the 32-column block cb of its rows
          const int c0 = cb * 32;
          const float* bias = cbias[l] + c0;
          float4 (*part)[TM] = sm.part[t & 1];
          float x[32];
          tmem_ld32(lane_t + c0, x);
#pragma unroll
          for (int i = 0; i < 32; ++i) x[i] += bias[i];
          const SoftPart sp = head_partials(x, kind, cb, r, S, part);
          epi_sync();
          const HeadStores pend = head_finish(x, kind, cb, r, sp, part, A, index_t, job, ch.n_policy);
          if (l + 1 < nl) {
            fence_async_smem();
            tc_fence_before();
            for (int c = 0; c < NR; ++c) nb_arrive(2 + 2 * t + c);
          }
          pend.flush();
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, NT * TN);
}

// ---------------------------------------------------------------------------------------------
// 64-row tiles (chosen automatically for small batches, SMZ_M64=0/1 forces): the hidden-layer epilogue is bound by the MUFU pipe of the SM (128 x 128
// exponentials per layer at 16 per clock), so a tile of 64 leaves per CTA on twice as many SMs halves it.
// tcgen05.mma M = 64 puts accumulator row m in TMEM lane (m % 16) + 32 * (m / 16): every warp quarter owns 16 rows,
// read with tcgen05.ld.16x256b so that all 32 lanes carry data (thread t: row t/4 and row t/4 + 8, two consecutive
// columns per 8-column group — the m16n8 accumulator fragment).  Same issuer warp / rounds / named-barrier
// structure as k_bf16_chain_pipe.
// Only layer 0 (gathered rows + one-hot columns) reads A from shared memory.  The MMAs of every later layer read it from
// tensor memory (umma_ts): A row m sits in the lane of accumulator row m, so each epilogue thread writes its packed bf16
// results with tcgen05.st.16x128b into the very lanes it loaded them from, and the hand-off to the issuer is
// tcgen05.wait::st + tcgen05 fence + named barrier — no st.shared, no generic -> async proxy fence.
// TMEM: one 128-column accumulator (every epilogue thread has loaded all of it before its first arrive, so the next
// layer may overwrite it) + the 64-column A operand (K = 128 bf16) = the same 256-column allocation as two accumulators.
// ---------------------------------------------------------------------------------------------
constexpr int TM64 = 64;
constexpr int A64_BYTES = TM64 * KMAX * 2;       // 16 KB (layer 0 only)
constexpr int CHUNK_A64 = TM64 * 16;             // LBO of the 64-row A operand
constexpr unsigned A64_TCOL = TN;                // TMEM column of the A operand of layers 1 .. nl-1
constexpr unsigned IDESC64 = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(TN >> 3) << 17) | ((unsigned)(TM64 >> 4) << 24);

struct Smem64 {
  alignas(1024) unsigned char a[A64_BYTES];
  alignas(1024) unsigned char w[2][W_BYTES];
  float bias[2][MAXL][TN];   // both chains: the branch of a tile is known only after the dependency wait
  unsigned long long wbar[2];
  unsigned long long dbar[2];
  unsigned long long bbar;
  unsigned int tmem_base;
  int rowidx[TM64];          // tree id of every tile row (-1 = none)
  float4 part[4][TM64];
};

__device__ __forceinline__ void umma64(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc, unsigned accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(IDESC64), "r"(accum)
      : "memory");
}
// N consecutive 8-column accumulator groups of this thread (pa: row t/4, pb: row t/4 + 8, packed bf16 pairs) -> the 4N
// TMEM columns of the A operand that hold the same K range, starting at taddr (lane quarter base + A64_TCOL + group * 4)
template <int N>
__device__ __forceinline__ void a64_tstore(unsigned taddr, const unsigned* pa, const unsigned* pb) {
  unsigned r[2 * N];
#pragma unroll
  for (int i = 0; i < N; ++i) { r[2 * i] = pa[i]; r[2 * i + 1] = pb[i]; }
  if constexpr (N == 1) {
    tmem_st16x128_x1(taddr, r[0], r[1]);
  } else if constexpr (N == 3) {
    tmem_st16x128_x2(taddr, r);
    tmem_st16x128_x1(taddr + 8, r[4], r[5]);
  } else {
    static_assert(N == 4, "a64_tstore: 1, 3 or 4 groups");
    tmem_st16x128_x4(taddr, r);
  }
}

// HALF = 32 leaves per tile instead of 64: the leaves sit in the accumulator rows m with m % 16 < 8, i.e. in the FIRST
// row of every thread's 16x256b fragment (thread t: rows t/4 and t/4 + 8), so the epilogue — bound by the MUFU pipe and
// by instruction issue, not by the contraction — does half the work per SM with all 32 lanes of every warp busy, on
// twice as many SMs.  Chosen while the tiles of the batch fit one wave of SMs.
// Tile -> rows: CTA i owns positions [i * TV, (i + 1) * TV) of the simulation's row array (smz_common.cuh: afterstate rows
// from the bottom, dynamics rows from the top, never both in one tile), so the row records are requested together with
// the branch counts — one L2 round trip after the dependency wait — and no CTA is launched for an empty tile of
// the "other" branch.  The first weight tile of BOTH chains is prefetched before the wait.
template <bool HALF>
__device__ __forceinline__ void chain_m64_body(const SmzArena& a, const Chain& chain0, const Chain& chain1, const Job& job, int sim) {
  extern __shared__ unsigned char smem_raw[];
  Smem64& sm = *reinterpret_cast<Smem64*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int R0 = 96;                   // hidden layers: rounds of 96 + 32 columns (two K-steps left for the tail)
  constexpr int TV = HALF ? 32 : 64;       // leaves per tile
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_issuer_warp = warp == NEPI / 32;
  const int q = warp & 3;                  // TMEM lane quarter: tile rows 16q .. 16q+15
  const int cb = (warp >> 2) & 3;          // head layers: 32-column block; hidden layers: 16-column slice of a round
  const int rA = 16 * q + (lane >> 2), rB = rA + 8;     // the two tile rows of this thread's fragment (HALF: rB is empty)
  const int cq = 2 * (lane & 3);           // column offset inside an 8-column group

  const int tile = blockIdx.x;
  const int nl = chain0.n_layers;          // == chain1.n_layers (both pairs are 2 (L + 2) layers)
  long long* tl = (job.timeline && blockIdx.x == 0 && lane == 0) ? job.timeline : nullptr;   // debug stamps
  if (tl && tid == 0) tl[0] = clock64();

  if (tid == 0) {
    mbar_init(&sm.wbar[0], 1); mbar_init(&sm.wbar[1], 1);
    mbar_init(&sm.dbar[0], 1); mbar_init(&sm.dbar[1], 1);
    mbar_init(&sm.bbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned bbytes = (unsigned)nl * TN * 4;
    mbar_expect_tx(&sm.bbar, 2 * bbytes);
    bulk_g2s(sm.bias[0], chain0.bias, bbytes, &sm.bbar);
    bulk_g2s(sm.bias[1], chain1.bias, bbytes, &sm.bbar);
    load_weight_tile(chain0, 0, sm.wbar, sm.w, 0);
    load_weight_tile(chain1, 0, sm.wbar, sm.w, 1);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&sm.tmem_base, 2 * TN);
  smz_pdl_wait();
  smz_pdl_launch_dependents();
  smz_stamp_min(a.dbg, sim, 2);
  if (tl && tid == 0) tl[1 + 4 * MAXL] = clock64();
  // gather: a staging thread owns the 16-byte K-chunk skc of leaf srow of the tile; requested before the counts are known
  const bool stager = HALF ? tid < 256 : !is_issuer_warp;
  const int srow = HALF ? (tid & 31) : (tid & 63), skc = HALF ? ((tid >> 5) & 7) : ((tid >> 6) & 7);
  const int mrow = HALF ? 16 * (srow >> 3) + (srow & 7) : srow;     // accumulator row of that leaf
  const int pos = tile * TV + srow;
  int4 rec = make_int4(0, 0, 0, 0);
  uint4 hrow = make_uint4(0, 0, 0, 0);
  if (stager) rec = load_row<1>(a, sim, pos, skc, &hrow);
  const int count0 = a.branch_count[sim * 2], count1 = a.branch_count[sim * 2 + 1];
  const int top1 = a.row_top - count1;      // dynamics rows occupy [top1, row_top)
  const int branch = tile * TV < count0 ? 0 : ((tile + 1) * TV > top1 ? 1 : -1);
  if (branch < 0) {
    idle_cta_exit(&sm.bbar, sm.wbar, true, sm.tmem_base, 2 * TN);
    return;
  }
  const Chain& ch = branch ? chain1 : chain0;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = sm.tmem_base;

  if (is_issuer_warp) {
    const unsigned long long ad = umma_desc(s32(sm.a), CHUNK_A64, 128);
    WeightRing ring(ch, sm.wbar, sm.w, lane);
    ring.start(branch, nl);
    for (int l = 0; l < nl; ++l) {
      const int nk = ch.layer[l].K / 16;
      const int slot = ring.wait(l);
      const unsigned long long bd = umma_desc(s32(sm.w[slot]), CHUNK_W, 128);
      for (int c = 0; c < 2; ++c) {
        nb_sync(2 + c);
        if (tl && c == 1) tl[1 + l * 4 + 0] = clock64();       // last round of the layer is in the A operand
        if (tl && c == 0 && l == 3) tl[1 + 4 * MAXL + 10] = clock64();
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            if (k >= (c ? R0 / 16 : 0) && k < (c ? 8 : R0 / 16) && k < nk) {
              const unsigned long long bk = bd + (unsigned long long)(k * ((2 * CHUNK_W) >> 4));
              if (l == 0)
                umma64(tmem, ad + (unsigned long long)(k * ((2 * CHUNK_A64) >> 4)), bk, k > 0 ? 1u : 0u);
              else
                umma_ts(tmem, tmem + A64_TCOL + 8 * k, bk, IDESC64, k > 0 ? 1u : 0u);
            }
        }
        __syncwarp();
        if (tl && c == 0 && l == 3) tl[1 + 4 * MAXL + 11] = clock64();
      }
      if (lane == 0) umma_commit(&sm.dbar[l & 1]);
      if (tl) tl[1 + l * 4 + 1] = clock64();
      __syncwarp();
      ring.refill(l, nl, job.stream_all, &sm.dbar[l & 1], (l >> 1) & 1);   // the slot is free once these MMAs have completed
    }
  } else {
    {   // stage the first A operand
      if (stager) {
        const bool valid = branch ? pos >= top1 : pos < count0;
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(s32(sm.a + skc * CHUNK_A64 + mrow * 16)), "r"(valid ? hrow.x : 0u),
                     "r"(valid ? hrow.y : 0u), "r"(valid ? hrow.z : 0u), "r"(valid ? hrow.w : 0u)
                     : "memory");
        if (skc < ch.onehot_pad / 8) {
          const uint4 oh = onehot_chunk(valid ? rec.z : -1, skc);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(s32(sm.a + (8 + skc) * CHUNK_A64 + mrow * 16)), "r"(oh.x),
                       "r"(oh.y), "r"(oh.z), "r"(oh.w)
                       : "memory");
        }
        if (skc == 0) sm.rowidx[mrow] = valid ? rec.x : -1;
      } else {
        // HALF: the accumulator rows m % 16 >= 8 carry no leaf — zero operand rows (nothing ever reads their results)
        const int j = tid - 256;
        const int zrow = 16 * ((j >> 3) & 3) + 8 + (j & 7), zc = j >> 5;
#pragma unroll
        for (int h = 0; h < 2; ++h)
          asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(s32(sm.a + (zc + 8 * h) * CHUNK_A64 + zrow * 16)), "r"(0u)
                       : "memory");
        if (zc == 0) sm.rowidx[zrow] = -1;
      }
    }
    fence_async_smem();
    for (int c = 0; c < 2; ++c) nb_arrive(2 + c);
    mbar_wait(&sm.bbar, 0);
    epi_sync();                              // rowidx is read by other threads from here on
    const unsigned lane_t = tmem + ((unsigned)(q * 32) << 16), a_t = lane_t + A64_TCOL;
    const int S = job.S;
    const int idxA = sm.rowidx[rA], idxB = HALF ? -1 : sm.rowidx[rB];
    const float (*bias)[TN] = sm.bias[branch];

    for (int l = 0; l < nl; ++l) {
      const int kind = ch.layer[l].kind;
      // hidden layers: this warp's bias pairs are fetched before the accumulator wait (the asm volatile stores below
      // are compiler barriers: a load placed after one of them waits for it)
      constexpr int G0 = R0 / 32, G1 = (TN - R0) / 32;          // 8-column groups per warp in round 0 / 1
      float2 bi[G0 + G1];
      if (kind == LK_HIDDEN) {
#pragma unroll
        for (int g = 0; g < G0 + G1; ++g)
          bi[g] = *reinterpret_cast<const float2*>(bias[l] + (g < G0 ? cb * 8 * G0 + g * 8 : R0 + cb * 8 * G1 + (g - G0) * 8) + cq);
      }
      mbar_wait(&sm.dbar[l & 1], (l >> 1) & 1);
      if (tl && warp == 0) tl[1 + l * 4 + 2] = clock64();
      __syncwarp();
      tc_fence_after();
      if (kind == LK_HIDDEN) {
        // two rounds: columns [0, R0) and [R0, 128); this warp owns a quarter of each round for its 16 rows.  All the
        // arithmetic of both rounds first (independent chains: the MUFU latencies overlap), then stores + hand-off per round.
        unsigned raw[4 * (G0 + G1)];
        tmem_ld16x256_x2(lane_t + cb * 24, raw);
        tmem_ld16x256_x1(lane_t + cb * 24 + 16, raw + 8);
        tmem_ld16x256_x1(lane_t + R0 + cb * 8, raw + 12);
        tmem_wait_ld();
        const bool fine = tl && warp == 0 && l == 2;
        if (fine) tl[1 + 4 * MAXL + 2] = clock64();
        // 32-leaf tiles: the arithmetic of both rounds first (8 values per thread), then stores + hand-off per round;
        // 64-leaf tiles (16 values per thread): round by round, or the packed results spill.
        // HALF: the rows without a leaf (rB) get zeros, so that the A operand holds finite values in every lane
        unsigned pa[G0 + G1], pb[G0 + G1];
        auto math = [&](int g) {
          const unsigned* rr = raw + 4 * g;
          pa[g] = pack_bf16(elu_fast(__uint_as_float(rr[0]) + bi[g].x), elu_fast(__uint_as_float(rr[1]) + bi[g].y));
          if constexpr (!HALF) pb[g] = pack_bf16(elu_fast(__uint_as_float(rr[2]) + bi[g].x), elu_fast(__uint_as_float(rr[3]) + bi[g].y));
          else pb[g] = 0u;
        };
        if constexpr (HALF) {
#pragma unroll
          for (int g = 0; g < G0 + G1; ++g) math(g);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          if constexpr (!HALF) {
#pragma unroll
            for (int g = 0; g < (c ? G1 : G0); ++g) math((c ? G0 : 0) + g);
          }
          if (c == 0)
            a64_tstore<G0>(a_t + cb * 4 * G0, pa, pb);
          else
            a64_tstore<G1>(a_t + R0 / 2 + cb * 4 * G1, pa + G0, pb + G0);
          if (fine) tl[1 + 4 * MAXL + 3 + 3 * c] = clock64();
          tmem_wait_st();
          tc_fence_before();
          if (fine) tl[1 + 4 * MAXL + 4 + 3 * c] = clock64();
          nb_arrive(2 + c);
          if (fine) tl[1 + 4 * MAXL + 5 + 3 * c] = clock64();
        }
      } else {
        // head layer: this warp owns the 32-column block cb of its 16 rows (fragment: 4 groups x {rowA, rowB} x 2 columns)
        const int c0 = cb * 32;
        unsigned raw[16];
        tmem_ld16x256_x4(lane_t + c0, raw);
        tmem_wait_ld();
        float xa[8], xb[8];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float2 bi = *reinterpret_cast<const float2*>(bias[l] + c0 + g * 8 + cq);
          xa[2 * g] = __uint_as_float(raw[4 * g + 0]) + bi.x; xa[2 * g + 1] = __uint_as_float(raw[4 * g + 1]) + bi.y;
          if constexpr (!HALF) {
            xb[2 * g] = __uint_as_float(raw[4 * g + 2]) + bi.x; xb[2 * g + 1] = __uint_as_float(raw[4 * g + 3]) + bi.y;
          } else {
            xb[2 * g] = 0.f; xb[2 * g + 1] = 0.f;
          }
        }
        const bool state_seg = (kind == LK_STATE || kind == LK_STATE_REWARD) && cb < 2;
        const bool soft_seg = (kind == LK_STATE_REWARD && cb >= 2) || (kind == LK_PRED && cb < 2);
        SoftPart spa{-1e30f, 0.f, 0.f}, spb{-1e30f, 0.f, 0.f};
        if (state_seg) {
          float loa = INFINITY, hia = -INFINITY, lob = INFINITY, hib = -INFINITY;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            loa = fminf(loa, xa[i]); hia = fmaxf(hia, xa[i]);
            if constexpr (!HALF) { lob = fminf(lob, xb[i]); hib = fmaxf(hib, xb[i]); }
          }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            loa = fminf(loa, __shfl_xor_sync(0xffffffffu, loa, off)); hia = fmaxf(hia, __shfl_xor_sync(0xffffffffu, hia, off));
            if constexpr (!HALF) {
              lob = fminf(lob, __shfl_xor_sync(0xffffffffu, lob, off)); hib = fmaxf(hib, __shfl_xor_sync(0xffffffffu, hib, off));
            }
          }
          if ((lane & 3) == 0) {
            sm.part[cb][rA] = make_float4(loa, hia, 0.f, 0.f);
            if constexpr (!HALF) sm.part[cb][rB] = make_float4(lob, hib, 0.f, 0.f);
          }
        } else if (soft_seg) {
          float ma = -1e30f, mb = -1e30f;
#pragma unroll
          for (int i = 0; i < 8; ++i) { ma = fmaxf(ma, xa[i]); if constexpr (!HALF) mb = fmaxf(mb, xb[i]); }
          spa.m = ma; spb.m = mb;
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const float pos_c = (float)(((c0 + g * 8 + cq + j) & 63) - S / 2);
              const float ea = ex2f((xa[2 * g + j] - ma) * 1.4426950408889634f);
              spa.z += ea; spa.y = fmaf(pos_c, ea, spa.y);
              if constexpr (!HALF) {
                const float eb = ex2f((xb[2 * g + j] - mb) * 1.4426950408889634f);
                spb.z += eb; spb.y = fmaf(pos_c, eb, spb.y);
              }
            }
          spa = soft_quad(spa);
          if constexpr (!HALF) spb = soft_quad(spb);
          if ((lane & 3) == 0) {
            sm.part[cb][rA] = make_float4(spa.m, spa.z, spa.y, 0.f);
            if constexpr (!HALF) sm.part[cb][rB] = make_float4(spb.m, spb.z, spb.y, 0.f);
          }
        }
        epi_sync();
        unsigned pend_a[4], pend_b[4];
        bool have_pend = false;
        if (state_seg) {
          const float4 oa = sm.part[cb ^ 1][rA], ma4 = sm.part[cb][rA];
          const float loa = fminf(ma4.x, oa.x), hia = fmaxf(ma4.y, oa.y);
          float sa = hia - loa;
          if (sa < 1e-5f) sa += 1e-5f;
          const float ia = 1.f / sa;
          float lob = 0.f, ib = 0.f;
          if constexpr (!HALF) {
            const float4 ob = sm.part[cb ^ 1][rB], mb4 = sm.part[cb][rB];
            lob = fminf(mb4.x, ob.x);
            float sb = fmaxf(mb4.y, ob.y) - lob;
            if (sb < 1e-5f) sb += 1e-5f;
            ib = 1.f / sb;
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            pend_a[g] = pack_bf16((xa[2 * g] - loa) * ia, (xa[2 * g + 1] - loa) * ia);
            if constexpr (!HALF) pend_b[g] = pack_bf16((xb[2 * g] - lob) * ib, (xb[2 * g + 1] - lob) * ib);
            else pend_b[g] = 0u;
          }
          a64_tstore<4>(a_t + c0 / 2, pend_a, pend_b);
          have_pend = job.hidden16_dst != nullptr;
        } else if (soft_seg && (cb & 1) == 0) {
          if ((lane & 3) == 0) {
            float* dst = (kind == LK_PRED) ? job.value_dst : job.reward_dst;
            if (dst) {
              const float4 oa = sm.part[cb + 1][rA];
              if (idxA >= 0) dst[idxA] = support_scalar(spa, SoftPart{oa.x, oa.y, oa.z});
              if constexpr (!HALF) {
                const float4 ob = sm.part[cb + 1][rB];
                if (idxB >= 0) dst[idxB] = support_scalar(spb, SoftPart{ob.x, ob.y, ob.z});
              }
            }
          }
        } else if (kind == LK_PRED && cb == 2) {
          const int n = ch.n_policy;
          float ma = -1e30f, mb = -1e30f;
#pragma unroll
          for (int i = 0; i < 8; ++i) { ma = fmaxf(ma, xa[i]); if constexpr (!HALF) mb = fmaxf(mb, xb[i]); }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, off));
            if constexpr (!HALF) mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, off));
          }
          float za = 0.f, zb = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            xa[i] = ex2f((xa[i] - ma) * 1.4426950408889634f); za += xa[i];
            if constexpr (!HALF) { xb[i] = ex2f((xb[i] - mb) * 1.4426950408889634f); zb += xb[i]; }
          }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            za += __shfl_xor_sync(0xffffffffu, za, off);
            if constexpr (!HALF) zb += __shfl_xor_sync(0xffffffffu, zb, off);
          }
          if (job.policy_dst) {
            const float ia = 1.f / za, ib = HALF ? 0.f : 1.f / zb;
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const int i = g * 8 + cq + j;
                if (i < n) {
                  if (idxA >= 0) job.policy_dst[(size_t)idxA * job.pstride + i] = xa[2 * g + j] * ia;
                  if constexpr (!HALF) {
                    if (idxB >= 0) job.policy_dst[(size_t)idxB * job.pstride + i] = xb[2 * g + j] * ib;
                  }
                }
              }
          }
        }
        if (l + 1 < nl) {
          tmem_wait_st();
          tc_fence_before();
          for (int c = 0; c < 2; ++c) nb_arrive(2 + c);
        }
        if (have_pend) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            if (idxA >= 0) *reinterpret_cast<unsigned*>(job.hidden16_dst + (size_t)idxA * SMZ_SP + c0 + g * 8 + cq) = pend_a[g];
            if constexpr (!HALF) {
              if (idxB >= 0) *reinterpret_cast<unsigned*>(job.hidden16_dst + (size_t)idxB * SMZ_SP + c0 + g * 8 + cq) = pend_b[g];
            }
          }
        }
      }
      if (tl && warp == 0) tl[1 + l * 4 + 3] = clock64();
    }
  }
  tc_fence_before();
  __syncthreads();
  smz_stamp_max(a.dbg, sim, 3);
  if (warp == 0) tmem_dealloc(tmem, 2 * TN);
}

__global__ void __maxnreg__(80)      // see k_bf16_chain_m32: measured 1.33 vs 1.50 ms per search at 6144 trees (98 CTAs)
k_bf16_chain_m64(SmzArena a, Chain chain0, Chain chain1, Job job, int sim) {
  chain_m64_body<false>(a, chain0, chain1, job, sim);
}
// 32-leaf tiles: 80 registers per thread, so that a block of the tree step (4 warps x 88 registers) still fits next to
// the 17 warps of this CTA in every SM sub-partition (16 K registers each; sub-partition 0 holds 5 of the 17 warps) —
// with one network CTA on nearly every SM the tree step launched under it (PDL) has nowhere else to go
__global__ void __maxnreg__(80)
k_bf16_chain_m32(SmzArena a, Chain chain0, Chain chain1, Job job, int sim) {
  chain_m64_body<true>(a, chain0, chain1, job, sim);
}

// ---------------------------------------------------------------------------------------------
// weight image: torch Linear W[out][in] (fp32 blob) -> bf16 canonical B operand [K/8][128][8]
// ---------------------------------------------------------------------------------------------
__global__ void k_pack_bf16(__nv_bfloat16* __restrict__ dst, const float* __restrict__ src, int n_rows, int in_stride,
                            int seg0, int seg1_dst, int seg1_src, int seg1_n, int dst_n0) {
  // dst k in [0, seg0) <- src column k;  dst k in [seg1_dst, seg1_dst + seg1_n) <- src column seg1_src + (k - seg1_dst)
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per_row = seg0 + seg1_n;
  if (i >= n_rows * per_row) return;
  const int n = i / per_row, j = i % per_row;
  const int k = j < seg0 ? j : seg1_dst + (j - seg0);
  const int c = j < seg0 ? j : seg1_src + (j - seg0);
  dst[((size_t)(k >> 3) * TN + dst_n0 + n) * 8 + (k & 7)] = __float2bfloat16_rn(src[(size_t)n * in_stride + c]);
}
__global__ void k_bf16_to_f32(float* __restrict__ dst, const __nv_bfloat16* __restrict__ src, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __bfloat162float(src[i]);
}
// state head: columns [S, 64) replicate column 0 so that they never move the row min / max
__global__ void k_replicate_col0(__nv_bfloat16* __restrict__ w, float* __restrict__ b, int S, int K) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;      // over (64 - S) * K
  const int npad = 64 - S;
  if (i >= npad * K) return;
  const int n = S + i / K, k = i % K;
  w[((size_t)(k >> 3) * TN + n) * 8 + (k & 7)] = w[((size_t)(k >> 3) * TN + 0) * 8 + (k & 7)];
  if (k == 0) b[n] = b[0];
}
// softmax heads: padded logits get bias -1e30 (weights stay zero) => probability exactly 0
__global__ void k_fill_f32(float* __restrict__ dst, float v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = v;
}
__global__ void k_copy_f32(float* __restrict__ dst, const float* __restrict__ src, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct NetImg {
  __nv_bfloat16 *in_w, *mid_w, *head_w;
  float *in_b, *mid_b, *head_b;   // 128 floats each
  int kin, head_kind, n_policy, onehot_pad;
};

struct SmzBf16Image {
  SmzNetShape sh;
  NetImg net[6];          // repr, pred, adyn, apred, dyn, enc
  Chain chain_after, chain_dyn, chain_root, chain_single[6];
  float* bias_pool;       // device: per chain [n_layers][128]
  unsigned char* pool;    // device: all images
  size_t pool_bytes;
  int smem_bytes;
  long long* timeline;    // device debug buffer or null (SMZ_BF16_TIMELINE=1)
  int use_m64;            // 64-row tiles: -1 = by batch size (busy CTAs fit one wave of SMs), SMZ_M64=0/1 forces
  int use_m32;            // 32 leaves per 64-row tile: -1 = while those tiles fit one wave of SMs, SMZ_M32=0/1 forces
  int n_sms;
  int use_pipe;           // K-pipelined chain for the simulation step (SMZ_NO_PIPE=1 turns it off)
  int use_pipe2;          // 128-leaf tiles per CTA: -1 = by batch size (1 / 2), SMZ_PIPE2 = 0 / 1 forces one / two
};

static int round16(int v) { return (v + 15) / 16 * 16; }

int smz_bf16_create(const SmzNetShape& sh, const SmzArena&, SmzBf16Image** out, char* err, size_t err_len) {
  if (2 * (sh.L + 2) > MAXL) {
    snprintf(err, err_len, "SMZ_NET_BF16: number_of_hidden_layer %d exceeds %d", sh.L, MAXL / 2 - 2);
    return SMZ_E_CAPACITY;
  }
  if (sh.OH > 32) {
    snprintf(err, err_len, "SMZ_NET_BF16: one-hot width %d exceeds 32", sh.OH);
    return SMZ_E_CAPACITY;
  }
  SmzBf16Image* im = new SmzBf16Image();
  memset(im, 0, sizeof(*im));
  im->sh = sh;
  const int ohp = round16(sh.OH);
  const int kin[6] = {round16(sh.obs), 64, 64 + ohp, 64, 64 + ohp, round16(sh.obs)};
  const int kind[6] = {LK_STATE, LK_PRED, LK_STATE, LK_PRED, LK_STATE_REWARD, LK_CODE};
  const int npol[6] = {0, sh.A, 0, sh.C, 0, sh.C};
  // pool: per net in (kin x 128) + mid (128 x 128) + head (128 x 128) bf16, + 3 x 128 fp32 biases; then chain biases
  size_t bytes = 0;
  for (int i = 0; i < 6; ++i) bytes += (size_t)(kin[i] + 2 * KMAX) * TN * 2 + 3 * TN * 4;
  const size_t chain_bias_floats = (size_t)(3 + 6) * MAXL * TN;
  bytes += chain_bias_floats * 4;
  if (cudaMalloc(&im->pool, bytes) != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_BF16: cudaMalloc of the weight image failed");
    delete im;
    return SMZ_E_CUDA;
  }
  im->pool_bytes = bytes;
  unsigned char* p = im->pool;
  for (int i = 0; i < 6; ++i) {
    NetImg& n = im->net[i];
    n.kin = kin[i]; n.head_kind = kind[i]; n.n_policy = npol[i]; n.onehot_pad = (i == 2 || i == 4) ? ohp : 0;
    n.in_w = (__nv_bfloat16*)p; p += (size_t)kin[i] * TN * 2;
    n.mid_w = (__nv_bfloat16*)p; p += (size_t)KMAX * TN * 2;
    n.head_w = (__nv_bfloat16*)p; p += (size_t)KMAX * TN * 2;
    n.in_b = (float*)p; p += TN * 4;
    n.mid_b = (float*)p; p += TN * 4;
    n.head_b = (float*)p; p += TN * 4;
  }
  im->bias_pool = (float*)p;
  im->smem_bytes = (int)sizeof(Smem) + 1024;
  cudaFuncSetAttribute((const void*)k_bf16_chain_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemPipe) + 1024);
  im->use_pipe = getenv("SMZ_NO_PIPE") ? 0 : 1;
  cudaFuncSetAttribute((const void*)k_bf16_chain_pipeN<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SmemPipeN<2>) + 1024);
  im->use_pipe2 = getenv("SMZ_PIPE2") ? atoi(getenv("SMZ_PIPE2")) : -1;
  im->use_m64 = getenv("SMZ_M64") ? atoi(getenv("SMZ_M64")) : -1;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&im->n_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || im->n_sms <= 0) im->n_sms = 148;
  }
  cudaFuncSetAttribute((const void*)k_bf16_chain_m64, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem64) + 1024);
  cudaFuncSetAttribute((const void*)k_bf16_chain_m32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem64) + 1024);
  im->use_m32 = getenv("SMZ_M32") ? atoi(getenv("SMZ_M32")) : -1;
  // The small-batch network CTAs share their SMs with the blocks of the shared-memory tree step that is launched while
  // they run (PDL): both kernels ask for the largest shared-memory carve-out, otherwise an SM is configured for the first
  // of them alone and the other's blocks wait for it to drain (measured: 156 vs 176 M sims/s on cfg2).  NOT set on the
  // arena-only tree kernels of the large batches — they live on the L1 (cfg4: 534 -> 480 M sims/s with it).
  if (!getenv("SMZ_NO_CARVEOUT"))
    for (const void* f : {(const void*)k_bf16_chain_m64, (const void*)k_bf16_chain_m32})
      cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (getenv("SMZ_BF16_TIMELINE")) {
    cudaMalloc(&im->timeline, (1 + 4 * MAXL + 32) * sizeof(long long));
    cudaMemset(im->timeline, 0, (1 + 4 * MAXL + 32) * sizeof(long long));
  }
  cudaFuncSetAttribute((const void*)k_bf16_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, im->smem_bytes);
  *out = im;
  return SMZ_OK;
}

void smz_bf16_destroy(SmzBf16Image* im) {
  if (!im) return;
  if (im->timeline) {
    long long t[1 + 4 * MAXL + 32];
    if (cudaMemcpy(t, im->timeline, sizeof(t), cudaMemcpyDeviceToHost) == cudaSuccess) {
      fprintf(stderr, "smz bf16 timeline (cycles, CTA 0 of the last simulation step):\n");
      for (int l = 0; l < MAXL && t[1 + l * 4 + 3]; ++l)
        fprintf(stderr, "  layer %2d: A operand complete +%6lld | mma issue -> commit %5lld | commit -> accumulator seen %5lld | epilogue %5lld\n", l,
                t[1 + l * 4] - t[0], t[1 + l * 4 + 1] - t[1 + l * 4], t[1 + l * 4 + 2] - t[1 + l * 4 + 1],
                t[1 + l * 4 + 3] - t[1 + l * 4 + 2]);
      const long long* h = t + 1 + 4 * MAXL;
      if (h[0] && !h[1]) {
        fprintf(stderr, "  pipelined kernel: dependency wait returned at +%lld (A operand of layer 0 complete %lld cycles later)\n",
                h[0] - t[0], t[1] - h[0]);
        if (h[2])
          fprintf(stderr, "  layer 2, epilogue warp 0: accumulator seen -> loaded %lld | round 0: math+stores %lld, fence %lld, arrive %lld | "
                  "round 1: math+stores %lld, fence %lld, arrive %lld\n  layer 3, issuer: round 0 in operand +%lld after the layer-2 epilogue "
                  "started; its K-steps issued in %lld; round 1 seen %lld later\n",
                  h[2] - t[1 + 2 * 4 + 2], h[3] - h[2], h[4] - h[3], h[5] - h[4], h[6] - h[5], h[7] - h[6], h[8] - h[7],
                  h[10] - t[1 + 2 * 4 + 2], h[11] - h[10], t[1 + 3 * 4] - h[11]);
      }
      else
      for (int k = 0; k < 2; ++k, h += 8)
        fprintf(stderr, "  %s head (thread 0): load+bias -> partials %lld | barrier %lld | finish %lld | fence+barrier %lld\n",
                k ? "pred " : "state", h[1] - h[0], h[2] - h[1], h[3] - h[2], h[4] - h[3]);
    }
    cudaFree(im->timeline);
  }
  cudaFree(im->pool);
  delete im;
}

static void build_chain(SmzBf16Image* im, Chain* ch, const int* nets, int n_nets, float* bias_dst, cudaStream_t s) {
  memset(ch, 0, sizeof(*ch));
  int l = 0;
  for (int t = 0; t < n_nets; ++t) {
    const NetImg& n = im->net[nets[t]];
    auto add = [&](const __nv_bfloat16* w, const float* b, int K, int kind) {
      ch->layer[l].w = w; ch->layer[l].K = K; ch->layer[l].kind = kind;
      k_copy_f32<<<1, TN, 0, s>>>(bias_dst + (size_t)l * TN, b, TN);
      ++l;
    };
    add(n.in_w, n.in_b, n.kin, LK_HIDDEN);
    for (int i = 0; i < im->sh.L; ++i) add(n.mid_w, n.mid_b, KMAX, LK_HIDDEN);
    add(n.head_w, n.head_b, KMAX, n.head_kind);
    if (n.n_policy) ch->n_policy = n.n_policy;
  }
  ch->n_layers = l;
  ch->bias = bias_dst;
  ch->kin = im->net[nets[0]].kin;
  ch->onehot_pad = im->net[nets[0]].onehot_pad;
}

int smz_bf16_pack(SmzBf16Image* im, const SmzNetShape& sh, const float* blob, cudaStream_t s, char* err, size_t err_len) {
  if (cudaMemsetAsync(im->pool, 0, im->pool_bytes, s) != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_BF16: memset failed");
    return SMZ_E_CUDA;
  }
  const int S = sh.S, H = sh.H, A = sh.A, C = sh.C, OH = sh.OH;
  size_t off = 0;
  auto pack = [&](__nv_bfloat16* dst, int n_rows, int in_stride, int seg0, int seg1_dst, int seg1_src, int seg1_n, int dst_n0) {
    const int n = n_rows * (seg0 + seg1_n);
    k_pack_bf16<<<(n + 255) / 256, 256, 0, s>>>(dst, blob + off, n_rows, in_stride, seg0, seg1_dst, seg1_src, seg1_n, dst_n0);
    off += (size_t)n_rows * in_stride;
  };
  auto vec = [&](float* dst, int n) {
    k_copy_f32<<<1, 128, 0, s>>>(dst, blob + off, n);
    off += n;
  };
  // blob order: repr, pred, adyn, apred, dyn, enc (stochastic-muzero_b200/weights.py)
  const int in_dim[6] = {sh.obs, S, S + OH, S, S + OH, sh.obs};
  const int order[6] = {0, 1, 2, 3, 4, 5};
  for (int t = 0; t < 6; ++t) {
    NetImg& n = im->net[order[t]];
    const bool oh = (t == 2 || t == 4);
    const int live = oh ? S : in_dim[t];
    pack(n.in_w, H, in_dim[t], live, 64, S, oh ? OH : 0, 0);
    vec(n.in_b, H);
    if (sh.L > 0) { pack(n.mid_w, H, H, H, 0, 0, 0, 0); vec(n.mid_b, H); }
    auto neg = [&](float* dst, int cnt) { if (cnt > 0) k_fill_f32<<<1, 128, 0, s>>>(dst, -1e30f, cnt); };
    auto rep = [&](NetImg& m) { const int c = (64 - S) * KMAX; if (c > 0) k_replicate_col0<<<(c + 255) / 256, 256, 0, s>>>(m.head_w, m.head_b, S, KMAX); };
    switch (t) {
      case 0: pack(n.head_w, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); rep(n); break;                          // repr: state
      case 1: neg(n.head_b + S, 64 - S); neg(n.head_b + POL_OFF + A, 64 - A);
              pack(n.head_w, A, H, H, 0, 0, 0, POL_OFF); vec(n.head_b + POL_OFF, A);                          // pred: policy,
              pack(n.head_w, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); break;                                  //       value
      case 2: pack(n.head_w, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); rep(n); break;                          // adyn: state
      case 3: neg(n.head_b + S, 64 - S); neg(n.head_b + POL_OFF + C, 64 - C);
              pack(n.head_w, C, H, H, 0, 0, 0, POL_OFF); vec(n.head_b + POL_OFF, C);
              pack(n.head_w, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); break;
      case 4: neg(n.head_b + POL_OFF + S, 64 - S);
              pack(n.head_w, S, H, H, 0, 0, 0, POL_OFF); vec(n.head_b + POL_OFF, S);                          // dyn: reward,
              pack(n.head_w, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); rep(n); break;                          //      state
      case 5: neg(n.head_b + C, 128 - C);
              pack(n.head_w, C, H, H, 0, 0, 0, 0); vec(n.head_b, C); break;                                  // enc: code
    }
  }
  float* bp = im->bias_pool;
  { const int nets[2] = {2, 3}; build_chain(im, &im->chain_after, nets, 2, bp, s); bp += MAXL * TN; }
  { const int nets[2] = {4, 1}; build_chain(im, &im->chain_dyn, nets, 2, bp, s); bp += MAXL * TN; }
  { const int nets[2] = {0, 1}; build_chain(im, &im->chain_root, nets, 2, bp, s); bp += MAXL * TN; }
  for (int i = 0; i < 6; ++i) { const int nets[1] = {i}; build_chain(im, &im->chain_single[i], nets, 1, bp, s); bp += MAXL * TN; }
  if (cudaGetLastError() != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_BF16: weight packing launch failed");
    return SMZ_E_CUDA;
  }
  return SMZ_OK;
}

void smz_bf16_read_hidden(const SmzArena& a, int slot, int n_trees, float* out, cudaStream_t s) {
  const size_t n = (size_t)n_trees * SMZ_SP;
  k_bf16_to_f32<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(
      out, reinterpret_cast<const __nv_bfloat16*>(a.hidden) + (size_t)slot * a.B * SMZ_SP, n);
}

void smz_bf16_root(SmzBf16Image* im, const SmzArena& a, const SmzNetShape& sh, int n_trees, const float* obs, cudaStream_t s) {
  Job job{};
  job.input_kind = IN_OBS; job.n_rows = n_trees; job.in = obs; job.obs = sh.obs; job.S = sh.S;
  job.hidden16_dst = reinterpret_cast<__nv_bfloat16*>(a.hidden);
  job.policy_dst = a.out_policy; job.value_dst = a.out_value; job.pstride = a.W;
  k_bf16_chain<<<(n_trees + TM - 1) / TM, NTHREADS, im->smem_bytes, s>>>(a, im->chain_root, im->chain_root, job, 0);
}

void smz_bf16_sim(SmzBf16Image* im, const SmzArena& a, const SmzNetShape& sh, int n_trees, int sim, bool pdl,
                  cudaStream_t s) {
  Job job{};
  job.input_kind = IN_GATHER; job.n_rows = n_trees; job.S = sh.S;
  job.hidden16_dst = reinterpret_cast<__nv_bfloat16*>(a.hidden) + (size_t)(sim + 1) * a.B * SMZ_SP;
  job.policy_dst = a.out_policy; job.value_dst = a.out_value; job.reward_dst = a.out_reward; job.pstride = a.W;
  job.timeline = im->timeline;
  job.stream_all = getenv("SMZ_STREAM_ALL") != nullptr;
  const dim3 grid(2 * ((n_trees + TM - 1) / TM)), block(NTHREADS);
  // 64-row tiles halve the MUFU-bound epilogue per SM as long as the busy CTAs (~trees / 64 + 2) fit one wave
  // (measured on B200, cfg-2 shapes: 8192 trees 267 vs 240 M sims/s, 16384 trees 288 vs 350)
  // one CTA per tile of the simulation's row array (a.row_top positions, both branches): no idle CTAs of the
  // "other" branch, so the one-wave condition is on row_top / tile
  const bool m64 = im->use_m64 < 0 ? a.row_top / TM64 <= im->n_sms : im->use_m64 != 0;
  const bool m32 = m64 && (im->use_m32 < 0 ? a.row_top / 32 <= im->n_sms : im->use_m32 != 0);
  if (im->use_pipe && m64) {
    auto* k64 = m32 ? k_bf16_chain_m32 : k_bf16_chain_m64;
    smz_launch(k64, dim3(a.row_top / (m32 ? 32 : TM64)), dim3(NPIPE), sizeof(Smem64) + 1024, s, pdl, a, im->chain_after,
               im->chain_dyn, job, sim);
    return;
  }
  // tiles per CTA: 1 while the tiles fit one wave of SMs, else 2 (SMZ_PIPE2 = 0 / 1 forces one / two)
  const int tiles = a.row_top / TM;
  const bool two = im->use_pipe2 < 0 ? tiles > im->n_sms : im->use_pipe2 == 1;
  if (im->use_pipe && two && a.row_top % (2 * TM) == 0) {
    smz_launch(k_bf16_chain_pipeN<2>, dim3(tiles / 2), dim3(NPIPE), sizeof(SmemPipeN<2>) + 1024, s, pdl, a, im->chain_after, im->chain_dyn, job, sim);
    return;
  }
  if (im->use_pipe) {
    smz_launch(k_bf16_chain_pipe, dim3(a.row_top / TM), dim3(NPIPE), sizeof(SmemPipe) + 1024, s, pdl, a, im->chain_after, im->chain_dyn, job, sim);
    return;
  }
  smz_launch(k_bf16_chain, grid, block, (size_t)im->smem_bytes, s, pdl, a, im->chain_after, im->chain_dyn, job, sim);
}

void smz_bf16_eval(SmzBf16Image* im, const SmzNetShape& sh, int which, int n_rows, const float* in, const int* idx,
                   float* hidden_out, float* policy_out, float* value_out, float* reward_out, int* code_out,
                   int policy_stride, cudaStream_t s) {
  Job job{};
  job.input_kind = (which == 0 || which == 5) ? IN_OBS : IN_ROWS;
  job.n_rows = n_rows; job.in = in; job.idx = idx; job.obs = sh.obs; job.S = sh.S;
  job.hidden_dst = hidden_out; job.policy_dst = policy_out; job.value_dst = value_out; job.reward_dst = reward_out;
  job.code_dst = code_out; job.pstride = policy_stride;
  SmzArena dummy{};
  k_bf16_chain<<<(n_rows + TM - 1) / TM, NTHREADS, im->smem_bytes, s>>>(dummy, im->chain_single[which], im->chain_single[which], job, 0);
}
