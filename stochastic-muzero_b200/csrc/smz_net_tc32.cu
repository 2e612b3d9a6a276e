// smz_net_tc32.cu — the network step at the REFERENCE'S precision on the 5th-generation tensor cores (sm_100a).
//
// The reference computes the five inference functions in fp32 (muzero_model.py:802-909, use_amp=False;
// neural_network_mlp_model.py:5-250).  tcgen05.mma has no fp32 operand type, so every fp32 operand is split into
// two fp16 numbers, x = hi + lo with hi = RN16(x), lo = RN16(x - hi) (22 significand bits; the weights are first
// scaled by a power of two per layer so that their lo parts stay normal).  The hi and lo parts of the ACTIVATIONS are
// stacked along M (one 128-row A operand: tcgen05.mma costs the same for M = 64 and M = 128), so every K-step issues
// TWO tcgen05.mma.kind::f16 into one fp32 TMEM accumulator of 128 lanes:
//       D[hi rows] += A_hi * W_hi + A_hi * W_lo          D[lo rows] += A_lo * W_hi + A_lo * W_lo
// and the epilogue adds the two halves in registers — all four partial products (see IDESC_S below).
// fp16 x fp16 products are exact in the fp32 accumulator, so a layer's pre-activations carry ~2^-22 relative error —
// the same order as the fp32 reference's own summation error (a numpy emulation of exactly this scheme reproduces the
// reference's outputs on tests/golden/net_*.npz to 2.4e-7; the CUDA-core fp32 kernel is at 2.9e-7).  Bias, ELU, the
// head epilogues (scale_to_bound, softmax, inverse_transform_with_support) run in fp32 on the accumulator.
//
// Structure = the 64-row pipelined chain of smz_net_bf16.cu (one CTA per 64-leaf tile runs the whole 2(L+2)-layer
// chain on the SM; issuer warp + 16 epilogue warps; A operand and accumulators double-buffered; weights streamed by
// cp.async.bulk two layers ahead; named-barrier hand-off of the A operand in two rounds of 96 + 32 columns), with
// a 128-row stacked A operand (32 KB) and a weight ring of 2 x (hi, lo) x 32 KB.  One kernel serves the simulation
// step (rows gathered through the descent's row records), the root step (observations) and stand-alone evaluation.
// Hidden states live in the arena as [hi[64] fp16 | lo[64] fp16] = 256 B per row.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/smz.h"
#include "smz_net_tc32.h"
#include "smz_tc_ptx.cuh"

namespace {

using namespace smz_tc;

constexpr int TM = 64;                  // rows (leaves) per CTA == MMA M
constexpr int TN = 128;                 // MMA N (all layers padded to 128 output channels)
constexpr int KMAX = 128;               // widest K
constexpr int MAXL = 24;                // layers per chain: 2 * (L + 2), L <= 10
constexpr int NEPI = 512;               // 16 epilogue warps: 4 TMEM lane quarters x 4 column blocks
constexpr int NTHR = NEPI + 32;         // + issuer warp
constexpr int KVIS = 160;               // widest first layer: the 147 features of a vision head, padded
constexpr int A_BYTES = TM * KMAX * 2;  // 16 KB per operand part (MLP family)
constexpr int W_BYTES = TN * KMAX * 2;  // 32 KB per operand part
constexpr int CHUNK_A = TM * 16;        // bytes between K-chunks (8 halves) of the A operand: LBO
constexpr int CHUNK_W = TN * 16;
constexpr int POL_OFF = 64;             // column of the second head inside a head tile
constexpr int R0 = 96;                  // columns of the first hidden-layer round (96 + 32: two K-steps left for the tail)
// InstrDescriptor: D = f32 (bit 4), A = B = f16 (format 0 at bits 7, 10), both K-major, N>>3 at [17,23), M>>4 at [24,29)
constexpr unsigned IDESC = (1u << 4) | ((unsigned)(TN >> 3) << 17) | ((unsigned)(TM >> 4) << 24);
// Split (fp32-grade) mode: the hi and lo parts of the activations are STACKED along M — one 128-row A operand whose rows
// 32q + i hold the hi part and rows 32q + 16 + i the lo part of leaf 16q + i.  tcgen05.mma costs the same for M = 64 and
// M = 128 (max(M, 128) N / 256 cycles), so (hi; lo) x W_hi and (hi; lo) x W_lo — all FOUR partial products, lo x lo
// included — take two instructions per K-step instead of three.  The accumulator of M = 128 keeps row r in TMEM lane r:
// a warp reads the hi rows of its leaves with one 16x256b load (lanes 32q ..) and the lo rows with a second one
// (lanes 32q + 16 ..), same fragment positions, and adds them in registers.
constexpr int TMS = 128;                // A rows of the stacked operand
constexpr int CHUNK_AS = TMS * 16;      // its LBO
constexpr unsigned IDESC_S = (1u << 4) | ((unsigned)(TN >> 3) << 17) | ((unsigned)(TMS >> 4) << 24);

enum LayerKind { LK_HIDDEN = 0, LK_STATE = 1, LK_STATE_REWARD = 2, LK_PRED = 3, LK_CODE = 4 };
// IN_FEAT: the MLP heads of the vision family (neural_network_vision_model.py: 147 -> H -> .. -> S / A after the 1x1
// convolutions).  Rows = the compacted leaves of a simulation, features written by k_vision_step's convolution stage.
enum InputKind { IN_GATHER = 0, IN_OBS = 1, IN_ROWS = 2, IN_FEAT = 3 };

struct LayerRef {
  const __half* w;          // [hi | lo], each [K/8][128][8] canonical K-major image of W * 2^s
  int K;                    // multiple of 16
  int kind;
};

struct Chain {
  LayerRef layer[MAXL];
  float inv_scale[MAXL];    // 2^-s of every layer: accumulator -> pre-activation
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
  __half* hidden_split_dst; // arena rows [index][hi 64 | lo 64] or null
  float* policy_dst;        // [index][pstride] or null
  float* value_dst;
  float* reward_dst;
  int* code_dst;
  int pstride;
  int S;
  int exact_elu;            // 1: polynomial expm1 for small |x| next to ex2.approx (SMZ_TC32_POLY=1)
  // IN_FEAT: CTAs [c*T, (c+1)*T) serve combination c of (branch, head): 0 afterstate value, 1 afterstate policy,
  // 2 dynamics reward, 3 dynamics value, 4 dynamics policy — chain `vchains[c]` (device memory)
  const float* feat;        // [3 heads: reward, value, policy][2 branches][B rows][KVIS] fp32
  const Chain* vchains;
};

template <int KA>           // widest K of the chain: 128 (MLP family) or 160 (vision heads)
struct SmemT {
  alignas(1024) unsigned char a[2][TM * KA * 2];    // activations: hi, lo
  alignas(1024) unsigned char w[2][2][TN * KA * 2]; // weights: [ring slot][hi, lo]
  float bias[MAXL][TN];
  unsigned long long wbar[2];
  unsigned long long dbar[2];
  unsigned long long bbar;
  unsigned int tmem_base;
  int rowidx[TM];           // output index (tree id / caller row) of every tile row, -1 = none
  float4 part[4][TM];       // head layers, first exchange: row min / max (state) or row max (softmax) per column block
  float4 part2[4][TM];      // second exchange: softmax sums.  A later head layer reuses both only after every warp has
                            // passed the named-barrier arrivals that follow its reads (the accumulator wait implies them)
  unsigned long long sbar;  // WIDE: "the MMAs of a K slice of the first layer have completed"
};

template <bool STACKED>
__device__ __forceinline__ void umma(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc, unsigned accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(STACKED ? IDESC_S : IDESC), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void epi_sync() { __syncwarp(); asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id) { __syncwarp(); asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(NTHR) : "memory"); }
__device__ __forceinline__ void nb_sync(int id) { __syncwarp(); asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NTHR) : "memory"); }

// x = hi + lo with hi = RN16(x), lo = RN16(x - hi): the subtraction is exact in fp32
__device__ __forceinline__ void split2(float x0, float x1, unsigned& hi, unsigned& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
  hi = *reinterpret_cast<const unsigned*>(&h);
  lo = *reinterpret_cast<const unsigned*>(&l);
}
__device__ __forceinline__ void split8(const float* v, uint4& hi, uint4& lo) {
  split2(v[0], v[1], hi.x, lo.x);
  split2(v[2], v[3], hi.y, lo.y);
  split2(v[4], v[5], hi.z, lo.z);
  split2(v[6], v[7], hi.w, lo.w);
}
__device__ __forceinline__ void sts16(unsigned char* p, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(s32(p)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts4(unsigned char* p, unsigned v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(s32(p)), "r"(v) : "memory"); }
// two halves at (operand row, col), col even; CH = bytes between K-chunks (CHUNK_A, or CHUNK_AS for the stacked operand)
template <int CH>
__device__ __forceinline__ unsigned char* a_at(unsigned char* part, int row, int col) {
  return part + (col >> 3) * CH + row * 16 + (col & 7) * 2;
}

__device__ __forceinline__ unsigned pack_f16(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&h);
}
// head-layer exponential: expf where the result feeds inverse_transform_with_support at reference precision, ex2.approx
// in the plain-fp16 throughput mode
template <bool PRECISE>
__device__ __forceinline__ float exp_head(float x) { return PRECISE ? expf(x) : ex2f(x * 1.4426950408889634f); }

// ELU (neural_network_mlp_model.py: nn.ELU).  exp through ex2.approx (relative error 2^-22: absolute error of
// exp(x) - 1 below 2.4e-7); EXACT adds the degree-5 Taylor form of expm1 for -1/16 < x < 0, where the subtraction
// would otherwise cancel.
template <bool EXACT>
__device__ __forceinline__ float elu32(float x) {
  const float e = ex2f(x * 1.4426950408889634f) - 1.f;
  float r = e;
  if (EXACT) {
    float p = fmaf(x, 1.f / 120.f, 1.f / 24.f);
    p = fmaf(x, p, 1.f / 6.f);
    p = fmaf(x, p, 0.5f);
    p = fmaf(x, p, 1.f);
    r = x > -0.0625f ? x * p : e;
  }
  return x > 0.f ? x : r;
}

template <bool EXACT, bool RELU>
__device__ __forceinline__ float act32(float x) { return RELU ? fmaxf(x, 0.f) : elu32<EXACT>(x); }

// ---------------------------------------------------------------------------------------------
// NPROD = 3: fp32-grade (hi/lo split operands, three products).  NPROD = 1: plain fp16 operands (the hi parts only,
// one product; "f16" throughput mode: 11-bit significands instead of bf16's 8, same speed class as the bf16 chain;
// arena rows are then 64 fp16 = 128 B and the head exponentials use ex2.approx).
// RELU: the vision heads use nn.ReLU between their Linear layers (the MLP family nn.ELU).
// WIDE: the observation of an IN_OBS job is wider than KMAX.  The first layer's K then streams in ns slices of KMAX
// through the same weight ring and A operand, all accumulated into the layer-0 accumulator: ring tile t < ns is slice t,
// tile ns - 1 + l is layer l >= 1.  The epilogue stages slice s + 1 once the MMAs of slice s have completed (sbar); the
// last slice is issued as layer 0 of the ordinary loop.  A separate instantiation, so the simulation step's code is
// untouched by it.
template <int NPROD, bool EXACT, bool RELU, int KA, bool WIDE>
__global__ void __launch_bounds__(NTHR, 1)
k_tc32_chain_m64(SmzArena a, Chain chain0, Chain chain1, Job job, int sim) {
  constexpr bool SPLIT = NPROD == 3;
  constexpr int ROWQ = SPLIT ? 16 : 8;            // 16-byte pieces per arena row
  constexpr int CH = SPLIT ? CHUNK_AS : CHUNK_A;  // bytes between K-chunks of the A operand (SPLIT: 128 stacked rows)
  extern __shared__ unsigned char smem_raw[];
  SmemT<KA>& sm = *reinterpret_cast<SmemT<KA>*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_issuer_warp = warp == NEPI / 32;
  const int q = warp & 3;                  // TMEM lane quarter: tile rows 16q .. 16q+15
  const int cb = (warp >> 2) & 3;          // head layers: 32-column block; hidden layers: slice of a round
  const int rA = 16 * q + (lane >> 2), rB = rA + 8;     // the two tile rows (leaves) of this thread's accumulator fragment
  // operand rows of those leaves: SPLIT stacks hi rows at 32q + i and lo rows at 32q + 16 + i (see IDESC_S)
  const int oA = SPLIT ? 32 * q + (lane >> 2) : rA, oB = oA + 8;
  const int cq = 2 * (lane & 3);           // column offset inside an 8-column group

  // gather launches use a static split: CTAs [0, T) serve the afterstate rows, [T, 2T) the dynamics rows, so the
  // weight chain is known before the previous kernel has finished
  int tile = blockIdx.x, branch = 0, head = 1;
  const Chain* chp = &chain0;
  float *value_dst = job.value_dst, *policy_dst = job.policy_dst;
  if (job.input_kind == IN_GATHER) {
    const int T = (job.n_rows + TM - 1) / TM;
    branch = tile >= T;
    tile -= branch * T;
    if (branch) chp = &chain1;
  } else if (job.input_kind == IN_FEAT) {
    const int T = (job.n_rows + TM - 1) / TM;
    const int combo = tile / T;
    tile -= combo * T;
    branch = combo >= 2;
    head = combo == 2 ? 0 : (combo == 0 || combo == 3 ? 1 : 2);      // 0 reward, 1 value, 2 policy
    chp = job.vchains + combo;
    if (head == 0) value_dst = job.reward_dst;                        // the reward head is a value-shaped head
    if (head != 2) policy_dst = nullptr;
  }
  const Chain& ch = *chp;
  const int nl = ch.n_layers;
  const int ns = WIDE ? (ch.kin + KMAX - 1) / KMAX : 1;     // K slices of the first layer (>= 2 when WIDE)

  auto load_weights = [&](int l) {
    const unsigned bytes = (unsigned)ch.layer[l].K * TN * 2;          // one part (hi or lo)
    mbar_expect_tx(&sm.wbar[l & 1], (SPLIT ? 2 : 1) * bytes);
    bulk_g2s(sm.w[l & 1][0], ch.layer[l].w, bytes, &sm.wbar[l & 1]);
    if (SPLIT) bulk_g2s(sm.w[l & 1][1], ch.layer[l].w + (size_t)ch.layer[l].K * TN, bytes, &sm.wbar[l & 1]);
  };
  auto load_tile = [&](int t) {                                      // WIDE: ring tile t into slot t & 1
    const int l = t < ns ? 0 : t - ns + 1;
    const int K = ch.layer[l].K, k0 = t < ns ? t * KMAX : 0;
    const unsigned bytes = (unsigned)(t < ns ? min(KMAX, K - k0) : K) * TN * 2;
    mbar_expect_tx(&sm.wbar[t & 1], (SPLIT ? 2 : 1) * bytes);
    bulk_g2s(sm.w[t & 1][0], ch.layer[l].w + (size_t)k0 * TN, bytes, &sm.wbar[t & 1]);
    if (SPLIT) bulk_g2s(sm.w[t & 1][1], ch.layer[l].w + (size_t)(K + k0) * TN, bytes, &sm.wbar[t & 1]);
  };
  if (tid == 0) {
    mbar_init(&sm.wbar[0], 1); mbar_init(&sm.wbar[1], 1);
    mbar_init(&sm.dbar[0], 1); mbar_init(&sm.dbar[1], 1);
    mbar_init(&sm.bbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned bbytes = (unsigned)nl * TN * 4;
    mbar_expect_tx(&sm.bbar, bbytes);
    bulk_g2s(sm.bias, ch.bias, bbytes, &sm.bbar);
    if (WIDE) {
      mbar_init(&sm.sbar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      load_tile(0);
      load_tile(1);
    } else {
      load_weights(0);
      if (nl > 1) load_weights(1);
    }
  }
  __syncwarp();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(&sm.tmem_base)), "r"(2 * TN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // everything above is independent of the previous kernel; from here on we read its results
  smz_pdl_wait();
  smz_pdl_launch_dependents();

  // ---- first A operand: epilogue thread i stages K-chunk (i >> 6) of tile row (i & 63) (+ chunk 8 + (i >> 6) for
  //      wide observations); requested before the row count of the branch is known ------------------------------
  const int srow = tid & 63, skc = (tid >> 6) & 7;
  int sidx = -1, sact = -1;                   // output index and one-hot position of the staged row
  uint4 h0 = make_uint4(0, 0, 0, 0), l0 = h0, h1 = h0, l1 = h0, h2 = h0, l2 = h0;
  int count = job.n_rows;
  if (job.input_kind == IN_GATHER) {
    if (!is_issuer_warp) {
      const size_t ri = smz_row_index(a, sim, branch, min(tile * TM + srow, a.B - 1));
      const int4 rec = a.rows4[ri];           // {tree, parent slot, action, -}
      h0 = a.xin[ri * ROWQ + skc];            // the descent copied the parent's row next to the record
      if (SPLIT) l0 = a.xin[ri * ROWQ + 8 + skc];
      sidx = rec.x; sact = rec.z;
    }
    count = a.branch_count[sim * 2 + branch];
  } else if (job.input_kind == IN_FEAT) {
    if (!is_issuer_warp) {
      const int row = min(tile * TM + srow, a.B - 1);
      sidx = a.rows4[smz_row_index(a, sim, branch, row)].x;
      const float* src = job.feat + ((size_t)(head * 2 + branch) * a.B + row) * KVIS;
      float v[8];
#pragma unroll
      for (int part = 0; part < 3; ++part) {
        const int kc = skc + 8 * part;
        if (kc * 8 < KVIS) {
          const float4 lo4 = *reinterpret_cast<const float4*>(src + kc * 8), hi4 = *reinterpret_cast<const float4*>(src + kc * 8 + 4);
          v[0] = lo4.x; v[1] = lo4.y; v[2] = lo4.z; v[3] = lo4.w; v[4] = hi4.x; v[5] = hi4.y; v[6] = hi4.z; v[7] = hi4.w;
          if (part == 0) split8(v, h0, l0); else if (part == 1) split8(v, h1, l1); else split8(v, h2, l2);
        }
      }
    }
    count = a.branch_count[sim * 2 + branch];
  } else if (!is_issuer_warp) {
    const int row = tile * TM + srow;
    if (row < count) {
      sidx = row;
      float v[8];
      if (job.input_kind == IN_OBS) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int kc = skc + 8 * half;
          if (kc * 8 < ch.kin) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = kc * 8 + j;
              v[j] = c < job.obs ? job.in[(size_t)row * job.obs + c] : 0.f;
            }
            if (half) split8(v, h1, l1); else split8(v, h0, l0);
          }
        }
      } else {
        const float4 lo4 = *reinterpret_cast<const float4*>(job.in + (size_t)row * SMZ_SP + skc * 8);
        const float4 hi4 = *reinterpret_cast<const float4*>(job.in + (size_t)row * SMZ_SP + skc * 8 + 4);
        v[0] = lo4.x; v[1] = lo4.y; v[2] = lo4.z; v[3] = lo4.w; v[4] = hi4.x; v[5] = hi4.y; v[6] = hi4.z; v[7] = hi4.w;
        split8(v, h0, l0);
        sact = job.idx ? job.idx[row] : -1;
      }
    }
  }
  if (tile * TM >= count) {        // nothing to do for this CTA: drain the prefetches, give TMEM back, leave
    if (tid == 0) {
      mbar_wait(&sm.bbar, 0);
      mbar_wait(&sm.wbar[0], 0);
      if (nl > 1) mbar_wait(&sm.wbar[1], 0);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 0)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(sm.tmem_base), "r"(2 * TN) : "memory");
    return;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = sm.tmem_base;

  if (is_issuer_warp) {
    // =========================== issuer warp: weight ring + 3 x tcgen05.mma per K-step ==========================
    const unsigned long long ad = umma_desc(s32(sm.a[0]), CH, 128);
    if (WIDE) {
      for (int s = 0; s + 1 < ns; ++s) {      // every K slice of the first layer but the last
        mbar_wait(&sm.wbar[s & 1], (s >> 1) & 1);
        const unsigned long long bd_hi = umma_desc(s32(sm.w[s & 1][0]), CHUNK_W, 128);
        const unsigned long long bd_lo = umma_desc(s32(sm.w[s & 1][1]), CHUNK_W, 128);
        nb_sync(2);                         // slice s is in shared memory (the epilogue arrives on both round barriers)
        nb_sync(3);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < KMAX / 16; ++k) {
            const unsigned long long oa = (unsigned long long)(k * ((2 * CH) >> 4));
            const unsigned long long ow = (unsigned long long)(k * ((2 * CHUNK_W) >> 4));
            umma<SPLIT>(tmem, ad + oa, bd_hi + ow, (s > 0 || k > 0) ? 1u : 0u);
            if (SPLIT) umma<SPLIT>(tmem, ad + oa, bd_lo + ow, 1u);
          }
        }
        __syncwarp();
        if (lane == 0) umma_commit(&sm.sbar);
        __syncwarp();
        mbar_wait(&sm.sbar, s & 1);         // slot s & 1 and the A operand are free again
        if (lane == 0) load_tile(s + 2);    // s + 2 <= ns: the last slice or layer 1
        __syncwarp();
      }
    }
    for (int l = 0; l < nl; ++l) {
      const int t = WIDE ? l + ns - 1 : l;  // ring tile of layer l
      const int nk = (WIDE && l == 0) ? (ch.kin - (ns - 1) * KMAX) / 16 : ch.layer[l].K / 16;
      mbar_wait(&sm.wbar[t & 1], (t >> 1) & 1);
      const unsigned long long bd_hi = umma_desc(s32(sm.w[t & 1][0]), CHUNK_W, 128);
      const unsigned long long bd_lo = umma_desc(s32(sm.w[t & 1][1]), CHUNK_W, 128);
      const unsigned d = tmem + (unsigned)((l & 1) * TN);
      for (int c = 0; c < 2; ++c) {
        nb_sync(2 + c);                     // the A columns of round c are in shared memory
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < KA / 16; ++k)
            if (k >= (c ? R0 / 16 : 0) && k < (c ? KA / 16 : R0 / 16) && k < nk) {
              const unsigned long long oa = (unsigned long long)(k * ((2 * CH) >> 4));
              const unsigned long long ow = (unsigned long long)(k * ((2 * CHUNK_W) >> 4));
              umma<SPLIT>(d, ad + oa, bd_hi + ow, (k > 0 || (WIDE && l == 0)) ? 1u : 0u);
              if (SPLIT) umma<SPLIT>(d, ad + oa, bd_lo + ow, 1u);
            }
        }
        __syncwarp();
      }
      if (lane == 0) umma_commit(&sm.dbar[l & 1]);
      __syncwarp();
      if (l + 2 < nl) {                     // ring slot l&1 is reusable once these MMAs have completed
        mbar_wait(&sm.dbar[l & 1], (l >> 1) & 1);
        if (lane == 0) {
          if (WIDE) load_tile(t + 2); else load_weights(l + 2);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue warps ===================================================================
    {
      const bool valid = tile * TM + srow < count;
      const uint4 z = make_uint4(0, 0, 0, 0);
      unsigned char* const ph = sm.a[0] + (SPLIT ? 32 * (srow >> 4) + (srow & 15) : srow) * 16;   // hi row of the staged leaf
      unsigned char* const pl = ph + 16 * 16;                                                      // its lo row (SPLIT)
      sts16(ph + skc * CH, valid ? h0 : z);
      if (SPLIT) sts16(pl + skc * CH, valid ? l0 : z);
      if (job.input_kind == IN_OBS || job.input_kind == IN_FEAT) {
        if ((skc + 8) * 8 < ch.kin) {
          sts16(ph + (skc + 8) * CH, valid ? h1 : z);
          if (SPLIT) sts16(pl + (skc + 8) * CH, valid ? l1 : z);
        }
        if (KA > 128 && (skc + 16) * 8 < ch.kin) {
          sts16(ph + (skc + 16) * CH, valid ? h2 : z);
          if (SPLIT) sts16(pl + (skc + 16) * CH, valid ? l2 : z);
        }
      } else if (skc < ch.onehot_pad / 8) {              // one-hot action / code: a single fp16 1.0 in the hi part
        const int act = valid ? sact : -1;
        unsigned w4[4] = {0, 0, 0, 0};
        if (act >= skc * 8 && act < skc * 8 + 8) {
          const int j = act - skc * 8;
          w4[j >> 1] = (j & 1) ? 0x3C000000u : 0x00003C00u;
        }
        sts16(ph + (8 + skc) * CH, make_uint4(w4[0], w4[1], w4[2], w4[3]));
        if (SPLIT) sts16(pl + (8 + skc) * CH, z);
      }
      if (skc == 0) sm.rowidx[srow] = valid ? sidx : -1;
    }
    fence_async_smem();
    for (int c = 0; c < 2; ++c) nb_arrive(2 + c);
    if (WIDE) {
      // the remaining K slices of the observation: the next slice's loads are in flight while the MMAs of the last run
      const int row = tile * TM + srow;
      const bool valid = row < count;
      const uint4 z = make_uint4(0, 0, 0, 0);
      unsigned char* const ph = sm.a[0] + (SPLIT ? 32 * (srow >> 4) + (srow & 15) : srow) * 16;
      unsigned char* const pl = ph + 16 * 16;
      for (int s = 1; s < ns; ++s) {
        const int k0 = s * KMAX, kw = min(KMAX, ch.kin - k0);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int kc = skc + 8 * half;
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int c = k0 + kc * 8 + j;
            v[j] = (valid && c < job.obs) ? job.in[(size_t)row * job.obs + c] : 0.f;
          }
          if (half) split8(v, h1, l1); else split8(v, h0, l0);
        }
        mbar_wait(&sm.sbar, (s - 1) & 1);
        __syncwarp();
        tc_fence_after();
        if (skc * 8 < kw) {
          sts16(ph + skc * CH, valid ? h0 : z);
          if (SPLIT) sts16(pl + skc * CH, valid ? l0 : z);
        }
        if ((skc + 8) * 8 < kw) {
          sts16(ph + (skc + 8) * CH, valid ? h1 : z);
          if (SPLIT) sts16(pl + (skc + 8) * CH, valid ? l1 : z);
        }
        fence_async_smem();
        for (int c = 0; c < 2; ++c) nb_arrive(2 + c);
      }
    }
    mbar_wait(&sm.bbar, 0);
    epi_sync();                              // rowidx is read by other threads from here on
    const unsigned lane_t = tmem + ((unsigned)(q * 32) << 16);
    const unsigned lane_lo = lane_t + (16u << 16);
    const int S = job.S;
    const int idxA = sm.rowidx[rA], idxB = sm.rowidx[rB];

    for (int l = 0; l < nl; ++l) {
      const int kind = ch.layer[l].kind;
      const unsigned dcol = (unsigned)((l & 1) * TN);
      const float isc = ch.inv_scale[l];
      // hidden layers: this warp's bias pairs are fetched before the accumulator wait (the asm volatile stores below are
      // compiler barriers: a load placed after one of them waits for it)
      constexpr int G0 = R0 / 32, G1 = (TN - R0) / 32;          // 8-column groups per warp in round 0 / 1
      float2 bi[G0 + G1];
      if (kind == LK_HIDDEN) {
#pragma unroll
        for (int g = 0; g < G0 + G1; ++g)
          bi[g] = *reinterpret_cast<const float2*>(sm.bias[l] + (g < G0 ? cb * 8 * G0 + g * 8 : R0 + cb * 8 * G1 + (g - G0) * 8) + cq);
      }
      mbar_wait(&sm.dbar[l & 1], (l >> 1) & 1);
      __syncwarp();
      tc_fence_after();
      if (kind == LK_HIDDEN) {
        // two rounds: columns [0, 96) and [96, 128); this warp owns a quarter of each round for its 16 rows.  All the
        // arithmetic of both rounds first (independent chains), then stores + fence per round.
        unsigned raw[4 * (G0 + G1)];
        tmem_ld16x256_x2(lane_t + dcol + cb * 24, raw);
        tmem_ld16x256_x1(lane_t + dcol + cb * 24 + 16, raw + 8);
        tmem_ld16x256_x1(lane_t + dcol + 96 + cb * 8, raw + 12);
        if (SPLIT) {                      // the lo rows' accumulators: lanes + 16, same fragment positions
          unsigned rlo[4 * (G0 + G1)];
          tmem_ld16x256_x2(lane_lo + dcol + cb * 24, rlo);
          tmem_ld16x256_x1(lane_lo + dcol + cb * 24 + 16, rlo + 8);
          tmem_ld16x256_x1(lane_lo + dcol + 96 + cb * 8, rlo + 12);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 4 * (G0 + G1); ++i) raw[i] = __float_as_uint(__uint_as_float(raw[i]) + __uint_as_float(rlo[i]));
        }
        tmem_wait_ld();
        unsigned ah[G0 + G1], al[G0 + G1], bh[G0 + G1], bl[G0 + G1];
#pragma unroll
        for (int g = 0; g < G0 + G1; ++g) {
          const unsigned* rr = raw + 4 * g;
          const float a0 = act32<EXACT, RELU>(fmaf(__uint_as_float(rr[0]), isc, bi[g].x)), a1 = act32<EXACT, RELU>(fmaf(__uint_as_float(rr[1]), isc, bi[g].y));
          const float b0 = act32<EXACT, RELU>(fmaf(__uint_as_float(rr[2]), isc, bi[g].x)), b1 = act32<EXACT, RELU>(fmaf(__uint_as_float(rr[3]), isc, bi[g].y));
          if (SPLIT) {
            split2(a0, a1, ah[g], al[g]);
            split2(b0, b1, bh[g], bl[g]);
          } else {
            ah[g] = pack_f16(a0, a1); bh[g] = pack_f16(b0, b1);
          }
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
#pragma unroll
          for (int g = 0; g < (c ? G1 : G0); ++g) {
            const int col = (c ? R0 + cb * 8 * G1 : cb * 8 * G0) + g * 8 + cq;
            const int i = (c ? G0 : 0) + g;
            sts4(a_at<CH>(sm.a[0], oA, col), ah[i]);
            sts4(a_at<CH>(sm.a[0], oB, col), bh[i]);
            if (SPLIT) {
              sts4(a_at<CH>(sm.a[0], oA + 16, col), al[i]);
              sts4(a_at<CH>(sm.a[0], oB + 16, col), bl[i]);
            }
          }
          fence_async_smem();
          if (c == 1) tc_fence_before();
          nb_arrive(2 + c);
        }
      } else {
        // head layer: this warp owns the 32-column block cb of its 16 rows (fragment: 4 groups x {rowA, rowB} x 2 columns).
        // Columns [0,64) = state or value logits, [64,128) = reward or policy logits; exponentials with expf here: the
        // categorical expectation feeds inverse_transform_with_support, which amplifies its rounding error ~100x.
        const int c0 = cb * 32;
        unsigned raw[16];
        tmem_ld16x256_x4(lane_t + dcol + c0, raw);
        if (SPLIT) {
          unsigned rlo[16];
          tmem_ld16x256_x4(lane_lo + dcol + c0, rlo);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; ++i) raw[i] = __float_as_uint(__uint_as_float(raw[i]) + __uint_as_float(rlo[i]));
        }
        tmem_wait_ld();
        float xa[8], xb[8];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float2 bi = *reinterpret_cast<const float2*>(sm.bias[l] + c0 + g * 8 + cq);
          xa[2 * g] = fmaf(__uint_as_float(raw[4 * g + 0]), isc, bi.x); xa[2 * g + 1] = fmaf(__uint_as_float(raw[4 * g + 1]), isc, bi.y);
          xb[2 * g] = fmaf(__uint_as_float(raw[4 * g + 2]), isc, bi.x); xb[2 * g + 1] = fmaf(__uint_as_float(raw[4 * g + 3]), isc, bi.y);
        }
        const bool state_seg = (kind == LK_STATE || kind == LK_STATE_REWARD) && cb < 2;
        const bool soft_seg = (kind == LK_STATE_REWARD && cb >= 2) || (kind == LK_PRED && cb < 2);
        SoftPart spa{-1e30f, 0.f, 0.f}, spb{-1e30f, 0.f, 0.f};
        if (state_seg) {
          float loa = INFINITY, hia = -INFINITY, lob = INFINITY, hib = -INFINITY;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            loa = fminf(loa, xa[i]); hia = fmaxf(hia, xa[i]);
            lob = fminf(lob, xb[i]); hib = fmaxf(hib, xb[i]);
          }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            loa = fminf(loa, __shfl_xor_sync(0xffffffffu, loa, off)); hia = fmaxf(hia, __shfl_xor_sync(0xffffffffu, hia, off));
            lob = fminf(lob, __shfl_xor_sync(0xffffffffu, lob, off)); hib = fmaxf(hib, __shfl_xor_sync(0xffffffffu, hib, off));
          }
          if ((lane & 3) == 0) {
            sm.part[cb][rA] = make_float4(loa, hia, 0.f, 0.f);
            sm.part[cb][rB] = make_float4(lob, hib, 0.f, 0.f);
          }
        } else if (soft_seg) {
          // two passes over the row: the row maximum first (partials of both column blocks meet in shared memory), so that
          // every exponent is taken against the same maximum as torch.softmax does
          float ma = -1e30f, mb = -1e30f;
#pragma unroll
          for (int i = 0; i < 8; ++i) { ma = fmaxf(ma, xa[i]); mb = fmaxf(mb, xb[i]); }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            ma = fmaxf(ma, __shfl_xor_sync(0xffffffffu, ma, off));
            mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, off));
          }
          spa.m = ma; spb.m = mb;
          if ((lane & 3) == 0) {
            sm.part[cb][rA] = make_float4(ma, 0.f, 0.f, 0.f);
            sm.part[cb][rB] = make_float4(mb, 0.f, 0.f, 0.f);
          }
        }
        epi_sync();
        unsigned pend_ah[4], pend_al[4], pend_bh[4], pend_bl[4];
        bool have_pend = false;
        if (state_seg) {
          // scale_to_bound_action (mlp:349-357): fp32 / split copy to HBM, split copy = the next network's A operand
          const float4 oa = sm.part[cb ^ 1][rA], ob = sm.part[cb ^ 1][rB], ma4 = sm.part[cb][rA], mb4 = sm.part[cb][rB];
          const float loa = fminf(ma4.x, oa.x), hia = fmaxf(ma4.y, oa.y), lob = fminf(mb4.x, ob.x), hib = fmaxf(mb4.y, ob.y);
          float sa = hia - loa, sb = hib - lob;
          if (sa < 1e-5f) sa += 1e-5f;
          if (sb < 1e-5f) sb += 1e-5f;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int col = c0 + g * 8 + cq;
            const float a0 = __fdiv_rn(xa[2 * g] - loa, sa), a1 = __fdiv_rn(xa[2 * g + 1] - loa, sa);
            const float b0 = __fdiv_rn(xb[2 * g] - lob, sb), b1 = __fdiv_rn(xb[2 * g + 1] - lob, sb);
            if (SPLIT) {
              split2(a0, a1, pend_ah[g], pend_al[g]);
              split2(b0, b1, pend_bh[g], pend_bl[g]);
              sts4(a_at<CH>(sm.a[0], oA + 16, col), pend_al[g]);
              sts4(a_at<CH>(sm.a[0], oB + 16, col), pend_bl[g]);
            } else {
              pend_ah[g] = pack_f16(a0, a1); pend_bh[g] = pack_f16(b0, b1);
            }
            sts4(a_at<CH>(sm.a[0], oA, col), pend_ah[g]);
            sts4(a_at<CH>(sm.a[0], oB, col), pend_bh[g]);
            if (job.hidden_dst) {
              if (idxA >= 0) *reinterpret_cast<float2*>(job.hidden_dst + (size_t)idxA * SMZ_SP + col) = make_float2(a0, a1);
              if (idxB >= 0) *reinterpret_cast<float2*>(job.hidden_dst + (size_t)idxB * SMZ_SP + col) = make_float2(b0, b1);
            }
          }
          have_pend = job.hidden_split_dst != nullptr;
        } else if (soft_seg) {
          const int other = cb ^ 1;
          const float ma = fmaxf(spa.m, sm.part[other][rA].x), mb = fmaxf(spb.m, sm.part[other][rB].x);
          float za = 0.f, ya = 0.f, zb = 0.f, yb = 0.f;
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const float pos = (float)(((c0 + g * 8 + cq + j) & 63) - S / 2);
              const float ea = exp_head<SPLIT>(xa[2 * g + j] - ma), eb = exp_head<SPLIT>(xb[2 * g + j] - mb);   // padded logits sit at -1e30: e == 0
              za += ea; ya = fmaf(pos, ea, ya);
              zb += eb; yb = fmaf(pos, eb, yb);
            }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            za += __shfl_xor_sync(0xffffffffu, za, off); ya += __shfl_xor_sync(0xffffffffu, ya, off);
            zb += __shfl_xor_sync(0xffffffffu, zb, off); yb += __shfl_xor_sync(0xffffffffu, yb, off);
          }
          spa = SoftPart{ma, za, ya}; spb = SoftPart{mb, zb, yb};
        }
        if (kind == LK_STATE_REWARD || kind == LK_PRED) {
          // second exchange (CTA-uniform condition): the two column blocks' sums, taken against the same maximum
          if (soft_seg && (lane & 3) == 0) {
            sm.part2[cb][rA] = make_float4(spa.m, spa.z, spa.y, 0.f);
            sm.part2[cb][rB] = make_float4(spb.m, spb.z, spb.y, 0.f);
          }
          epi_sync();
          if (soft_seg && (cb & 1) == 0 && (lane & 3) == 0) {
            const float4 oa = sm.part2[cb + 1][rA], ob = sm.part2[cb + 1][rB];
            float* dst = (kind == LK_PRED) ? value_dst : job.reward_dst;
            if (dst) {
              if (idxA >= 0) dst[idxA] = support_scalar(spa, SoftPart{oa.x, oa.y, oa.z});
              if (idxB >= 0) dst[idxB] = support_scalar(spb, SoftPart{ob.x, ob.y, ob.z});
            }
          }
        }
        if ((kind == LK_PRED && cb == 2) || (kind == LK_CODE && cb == 0)) {
          // policy softmax (muzero_model.py:837) / Encoder code distribution + argmax (mlp:209-250)
          const int n = ch.n_policy;
          float ma = -1e30f, mb = -1e30f;
          int ia = 0, ib = 0;
#pragma unroll
          for (int g = 0; g < 4; ++g)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const int i = g * 8 + cq + j;
              if (xa[2 * g + j] > ma) { ma = xa[2 * g + j]; ia = i; }
              if (xb[2 * g + j] > mb) { mb = xb[2 * g + j]; ib = i; }
            }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            const float oma = __shfl_xor_sync(0xffffffffu, ma, off), omb = __shfl_xor_sync(0xffffffffu, mb, off);
            const int oia = __shfl_xor_sync(0xffffffffu, ia, off), oib = __shfl_xor_sync(0xffffffffu, ib, off);
            if (oma > ma || (oma == ma && oia < ia)) { ma = oma; ia = oia; }      // ties -> first index (argmax)
            if (omb > mb || (omb == mb && oib < ib)) { mb = omb; ib = oib; }
          }
          float za = 0.f, zb = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            xa[i] = exp_head<SPLIT>(xa[i] - ma); za += xa[i];
            xb[i] = exp_head<SPLIT>(xb[i] - mb); zb += xb[i];
          }
#pragma unroll
          for (int off = 1; off <= 2; off <<= 1) {
            za += __shfl_xor_sync(0xffffffffu, za, off);
            zb += __shfl_xor_sync(0xffffffffu, zb, off);
          }
          if (policy_dst) {
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const int i = g * 8 + cq + j;
                if (i < n) {
                  if (idxA >= 0) policy_dst[(size_t)idxA * job.pstride + i] = __fdiv_rn(xa[2 * g + j], za);
                  if (idxB >= 0) policy_dst[(size_t)idxB * job.pstride + i] = __fdiv_rn(xb[2 * g + j], zb);
                }
              }
          }
          if (kind == LK_CODE && job.code_dst && (lane & 3) == 0) {
            if (idxA >= 0) job.code_dst[idxA] = ia;
            if (idxB >= 0) job.code_dst[idxB] = ib;
          }
        }
        if (l + 1 < nl) {
          fence_async_smem();
          tc_fence_before();
          for (int c = 0; c < 2; ++c) nb_arrive(2 + c);
        }
        if (have_pend) {          // arena row: [hi 64 halves | lo 64 halves]
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int col = c0 + g * 8 + cq;
            if (idxA >= 0) {
              __half* row = job.hidden_split_dst + (size_t)idxA * (ROWQ * 8);
              *reinterpret_cast<unsigned*>(row + col) = pend_ah[g];
              if (SPLIT) *reinterpret_cast<unsigned*>(row + SMZ_SP + col) = pend_al[g];
            }
            if (idxB >= 0) {
              __half* row = job.hidden_split_dst + (size_t)idxB * (ROWQ * 8);
              *reinterpret_cast<unsigned*>(row + col) = pend_bh[g];
              if (SPLIT) *reinterpret_cast<unsigned*>(row + SMZ_SP + col) = pend_bl[g];
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(2 * TN) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// weight image: torch Linear W[out][in] (fp32 blob) -> fp16 hi / lo canonical B operands [K/8][128][8] of W * 2^s
// ---------------------------------------------------------------------------------------------
__global__ void k_absmax(const float* __restrict__ src, int n, unsigned* __restrict__ out) {
  unsigned m = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    m = max(m, __float_as_uint(fabsf(src[i])));      // non-negative floats order like their bit patterns
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}
// s = largest power of two with max|W| * 2^s < 2^14 (fp16 keeps 11 bits above, the lo part 11 more, all normal)
__global__ void k_scale_from_absmax(const unsigned* __restrict__ absmax, float* __restrict__ scale, float* __restrict__ inv_scale) {
  const float m = __uint_as_float(*absmax);
  int e = 0;
  if (m > 0.f && isfinite(m)) {
    frexpf(m, &e);                       // m = f * 2^e, 0.5 <= f < 1
    e = 14 - e;                          // m * 2^(14 - e) in [2^13, 2^14)
    e = max(-100, min(100, e));
  }
  *scale = ldexpf(1.f, e);
  *inv_scale = ldexpf(1.f, -e);
}
__global__ void k_pack_split(__half* __restrict__ dst, int K, const float* __restrict__ src, const float* __restrict__ scale,
                             int n_rows, int in_stride, int seg0, int seg1_dst, int seg1_src, int seg1_n, int dst_n0) {
  // dst k in [0, seg0) <- src column k;  dst k in [seg1_dst, seg1_dst + seg1_n) <- src column seg1_src + (k - seg1_dst)
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per_row = seg0 + seg1_n;
  if (i >= n_rows * per_row) return;
  const int n = i / per_row, j = i % per_row;
  const int k = j < seg0 ? j : seg1_dst + (j - seg0);
  const int c = j < seg0 ? j : seg1_src + (j - seg0);
  const float v = src[(size_t)n * in_stride + c] * *scale;
  const __half hi = __float2half_rn(v);
  const __half lo = __float2half_rn(v - __half2float(hi));
  const size_t o = ((size_t)(k >> 3) * TN + dst_n0 + n) * 8 + (k & 7);
  dst[o] = hi;
  dst[(size_t)K * TN + o] = lo;
}
// state head: columns [S, 64) replicate column 0 so that they never move the row min / max
__global__ void k_replicate_col0(__half* __restrict__ w, float* __restrict__ b, int S, int K) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;      // over (64 - S) * K
  const int npad = 64 - S;
  if (i >= npad * K) return;
  const int n = S + i / K, k = i % K;
  for (int part = 0; part < 2; ++part) {
    __half* p = w + (size_t)part * K * TN;
    p[((size_t)(k >> 3) * TN + n) * 8 + (k & 7)] = p[((size_t)(k >> 3) * TN + 0) * 8 + (k & 7)];
  }
  if (k == 0) b[n] = b[0];
}
__global__ void k_fill_f32(float* __restrict__ dst, float v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = v;
}
__global__ void k_copy_f32(float* __restrict__ dst, const float* __restrict__ src, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}
__global__ void k_split_to_f32(float* __restrict__ dst, const __half* __restrict__ src, int n_rows, int row_halves) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * SMZ_SP) return;
  const int r = i / SMZ_SP, c = i % SMZ_SP;
  const __half* row = src + (size_t)r * row_halves;
  dst[i] = __half2float(row[c]) + (row_halves > SMZ_SP ? __half2float(row[SMZ_SP + c]) : 0.f);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct NetImgT {
  __half *in_w, *mid_w, *head_w;            // each [hi | lo]
  float *in_b, *mid_b, *head_b;             // 128 floats each
  float *scales;                            // device [3][2]: {scale, inv_scale} of in / mid / head
  int kin, head_kind, n_policy, onehot_pad;
};

struct SmzTc32Image {
  SmzNetShape sh;
  NetImgT net[6];          // repr, pred, adyn, apred, dyn, enc
  Chain chain_after, chain_dyn, chain_root, chain_single[6];
  float* bias_pool;        // device: per chain [n_layers][128]
  unsigned char* pool;     // device: all images
  size_t pool_bytes;
  unsigned* absmax;        // device [18]
  float* scales;           // device [18][2]
  int smem_bytes;
  int exact_elu;
  int nprod;               // 3: fp32-grade split operands (SMZ_NET_TC32); 1: plain fp16 operands (SMZ_NET_F16)
};

static int round16(int v) { return (v + 15) / 16 * 16; }

int smz_tc32_create(const SmzNetShape& sh, int nprod, SmzTc32Image** out, char* err, size_t err_len) {
  if (2 * (sh.L + 2) > MAXL) {
    snprintf(err, err_len, "SMZ_NET_TC32: number_of_hidden_layer %d exceeds %d", sh.L, MAXL / 2 - 2);
    return SMZ_E_CAPACITY;
  }
  if (sh.OH > 32) {
    snprintf(err, err_len, "SMZ_NET_TC32: one-hot width %d exceeds 32", sh.OH);
    return SMZ_E_CAPACITY;
  }
  SmzTc32Image* im = new SmzTc32Image();
  memset(im, 0, sizeof(*im));
  im->sh = sh;
  const int ohp = round16(sh.OH);
  const int kin[6] = {round16(sh.obs), 64, 64 + ohp, 64, 64 + ohp, round16(sh.obs)};
  const int kind[6] = {LK_STATE, LK_PRED, LK_STATE, LK_PRED, LK_STATE_REWARD, LK_CODE};
  const int npol[6] = {0, sh.A, 0, sh.C, 0, sh.C};
  // pool: per net in (kin x 128) + mid (128 x 128) + head (128 x 128), hi + lo fp16 each, + 3 x 128 fp32 biases; chain biases
  size_t bytes = 0;
  for (int i = 0; i < 6; ++i) bytes += (size_t)(kin[i] + 2 * KMAX) * TN * 2 * 2 + 3 * TN * 4;
  const size_t chain_bias_floats = (size_t)(3 + 6) * MAXL * TN;
  bytes += chain_bias_floats * 4;
  if (cudaMalloc(&im->pool, bytes) != cudaSuccess || cudaMalloc(&im->absmax, 18 * sizeof(unsigned)) != cudaSuccess ||
      cudaMalloc(&im->scales, 36 * sizeof(float)) != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_TC32: cudaMalloc of the weight image failed");
    cudaFree(im->pool); cudaFree(im->absmax); cudaFree(im->scales);
    delete im;
    return SMZ_E_CUDA;
  }
  im->pool_bytes = bytes;
  unsigned char* p = im->pool;
  for (int i = 0; i < 6; ++i) {
    NetImgT& n = im->net[i];
    n.kin = kin[i]; n.head_kind = kind[i]; n.n_policy = npol[i]; n.onehot_pad = (i == 2 || i == 4) ? ohp : 0;
    n.in_w = (__half*)p; p += (size_t)kin[i] * TN * 2 * 2;
    n.mid_w = (__half*)p; p += (size_t)KMAX * TN * 2 * 2;
    n.head_w = (__half*)p; p += (size_t)KMAX * TN * 2 * 2;
    n.in_b = (float*)p; p += TN * 4;
    n.mid_b = (float*)p; p += TN * 4;
    n.head_b = (float*)p; p += TN * 4;
    n.scales = im->scales + i * 6;
  }
  im->bias_pool = (float*)p;
  im->smem_bytes = (int)sizeof(SmemT<KMAX>) + 1024;
  im->nprod = nprod == 1 ? 1 : 3;
  im->exact_elu = (im->nprod == 3 && getenv("SMZ_TC32_POLY")) ? atoi(getenv("SMZ_TC32_POLY")) : 0;
  for (const void* f : {(const void*)k_tc32_chain_m64<3, false, false, KMAX, false>, (const void*)k_tc32_chain_m64<3, true, false, KMAX, false>,
                        (const void*)k_tc32_chain_m64<1, false, false, KMAX, false>, (const void*)k_tc32_chain_m64<3, false, false, KMAX, true>,
                        (const void*)k_tc32_chain_m64<3, true, false, KMAX, true>, (const void*)k_tc32_chain_m64<1, false, false, KMAX, true>})
    cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, im->smem_bytes);
  *out = im;
  return SMZ_OK;
}

void smz_tc32_destroy(SmzTc32Image* im) {
  if (!im) return;
  cudaFree(im->pool);
  cudaFree(im->absmax);
  cudaFree(im->scales);
  delete im;
}

// scales are device-resident until the end of smz_tc32_pack, which copies them to the host for the Chain structs
static void build_chain(SmzTc32Image* im, Chain* ch, const int* nets, int n_nets, float* bias_dst, const float* host_scales,
                        cudaStream_t s) {
  memset(ch, 0, sizeof(*ch));
  int l = 0;
  for (int t = 0; t < n_nets; ++t) {
    const NetImgT& n = im->net[nets[t]];
    const float* sc = host_scales + nets[t] * 6;
    auto add = [&](const __half* w, const float* b, int K, int kind, float inv_scale) {
      ch->layer[l].w = w; ch->layer[l].K = K; ch->layer[l].kind = kind;
      ch->inv_scale[l] = inv_scale;
      k_copy_f32<<<1, TN, 0, s>>>(bias_dst + (size_t)l * TN, b, TN);
      ++l;
    };
    add(n.in_w, n.in_b, n.kin, LK_HIDDEN, sc[1]);
    for (int i = 0; i < im->sh.L; ++i) add(n.mid_w, n.mid_b, KMAX, LK_HIDDEN, sc[3]);
    add(n.head_w, n.head_b, KMAX, n.head_kind, sc[5]);
    if (n.n_policy) ch->n_policy = n.n_policy;
  }
  ch->n_layers = l;
  ch->bias = bias_dst;
  ch->kin = im->net[nets[0]].kin;
  ch->onehot_pad = im->net[nets[0]].onehot_pad;
}

int smz_tc32_pack(SmzTc32Image* im, const SmzNetShape& sh, const float* blob, cudaStream_t s, char* err, size_t err_len) {
  if (cudaMemsetAsync(im->pool, 0, im->pool_bytes, s) != cudaSuccess || cudaMemsetAsync(im->absmax, 0, 18 * sizeof(unsigned), s) != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_TC32: memset failed");
    return SMZ_E_CUDA;
  }
  const int S = sh.S, H = sh.H, A = sh.A, C = sh.C, OH = sh.OH;
  const int in_dim[6] = {sh.obs, S, S + OH, S, S + OH, sh.obs};
  // head widths in blob order (first head, second head; 0 = none): repr out | pred policy, value | adyn state |
  // apred policy, value | dyn reward, state | enc code
  const int head_a[6] = {S, A, S, C, S, C}, head_b[6] = {0, S, 0, S, S, 0};
  // ---- pass 1: per-image max |w| -> power-of-two scale (the two heads of a net share one image, hence one scale)
  size_t off = 0;
  for (int t = 0; t < 6; ++t) {
    auto mx = [&](int slot, size_t n) { k_absmax<<<64, 256, 0, s>>>(blob + off, (int)n, im->absmax + t * 3 + slot); off += n; };
    mx(0, (size_t)H * in_dim[t]); off += H;
    if (sh.L > 0) { mx(1, (size_t)H * H); off += H; }
    mx(2, (size_t)head_a[t] * H); off += head_a[t];
    if (head_b[t]) { mx(2, (size_t)head_b[t] * H); off += head_b[t]; }
  }
  for (int i = 0; i < 18; ++i) k_scale_from_absmax<<<1, 1, 0, s>>>(im->absmax + i, im->scales + 2 * i, im->scales + 2 * i + 1);
  // ---- pass 2: scaled hi / lo images
  off = 0;
  for (int t = 0; t < 6; ++t) {
    NetImgT& n = im->net[t];
    auto pack = [&](__half* dst, int K, int slot, int n_rows, int in_stride, int seg0, int seg1_dst, int seg1_src, int seg1_n, int dst_n0) {
      const int cnt = n_rows * (seg0 + seg1_n);
      k_pack_split<<<(cnt + 255) / 256, 256, 0, s>>>(dst, K, blob + off, n.scales + 2 * slot, n_rows, in_stride, seg0, seg1_dst,
                                                     seg1_src, seg1_n, dst_n0);
      off += (size_t)n_rows * in_stride;
    };
    auto vec = [&](float* dst, int cnt) { k_copy_f32<<<1, 128, 0, s>>>(dst, blob + off, cnt); off += cnt; };
    auto neg = [&](float* dst, int cnt) { if (cnt > 0) k_fill_f32<<<1, 128, 0, s>>>(dst, -1e30f, cnt); };
    auto rep = [&]() { const int c = (64 - S) * KMAX; if (c > 0) k_replicate_col0<<<(c + 255) / 256, 256, 0, s>>>(n.head_w, n.head_b, S, KMAX); };
    const bool oh = (t == 2 || t == 4);
    pack(n.in_w, n.kin, 0, H, in_dim[t], oh ? S : in_dim[t], 64, S, oh ? OH : 0, 0);
    vec(n.in_b, H);
    if (sh.L > 0) { pack(n.mid_w, KMAX, 1, H, H, H, 0, 0, 0, 0); vec(n.mid_b, H); }
    switch (t) {
      case 0: case 2: pack(n.head_w, KMAX, 2, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); rep(); break;            // state
      case 1: case 3: {                                                                                        // policy, value
        const int P = t == 1 ? A : C;
        neg(n.head_b + S, 64 - S); neg(n.head_b + POL_OFF + P, 64 - P);
        pack(n.head_w, KMAX, 2, P, H, H, 0, 0, 0, POL_OFF); vec(n.head_b + POL_OFF, P);
        pack(n.head_w, KMAX, 2, S, H, H, 0, 0, 0, 0); vec(n.head_b, S);
        break;
      }
      case 4: neg(n.head_b + POL_OFF + S, 64 - S);                                                             // reward, state
              pack(n.head_w, KMAX, 2, S, H, H, 0, 0, 0, POL_OFF); vec(n.head_b + POL_OFF, S);
              pack(n.head_w, KMAX, 2, S, H, H, 0, 0, 0, 0); vec(n.head_b, S); rep(); break;
      case 5: neg(n.head_b + C, 128 - C);
              pack(n.head_w, KMAX, 2, C, H, H, 0, 0, 0, 0); vec(n.head_b, C); break;                           // code
    }
  }
  float host_scales[36];
  if (cudaMemcpyAsync(host_scales, im->scales, sizeof(host_scales), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_TC32: reading the layer scales back failed: %s", cudaGetErrorString(cudaGetLastError()));
    return SMZ_E_CUDA;
  }
  float* bp = im->bias_pool;
  { const int nets[2] = {2, 3}; build_chain(im, &im->chain_after, nets, 2, bp, host_scales, s); bp += MAXL * TN; }
  { const int nets[2] = {4, 1}; build_chain(im, &im->chain_dyn, nets, 2, bp, host_scales, s); bp += MAXL * TN; }
  { const int nets[2] = {0, 1}; build_chain(im, &im->chain_root, nets, 2, bp, host_scales, s); bp += MAXL * TN; }
  for (int i = 0; i < 6; ++i) { const int nets[1] = {i}; build_chain(im, &im->chain_single[i], nets, 1, bp, host_scales, s); bp += MAXL * TN; }
  if (cudaGetLastError() != cudaSuccess) {
    snprintf(err, err_len, "SMZ_NET_TC32: weight packing launch failed");
    return SMZ_E_CUDA;
  }
  return SMZ_OK;
}

void smz_tc32_read_hidden(const SmzArena& a, int slot, int n_trees, float* out, cudaStream_t s) {
  const int n = n_trees * SMZ_SP;
  const int row_halves = a.xin_q * 8;           // 128: [hi | lo], 64: plain fp16
  k_split_to_f32<<<(n + 255) / 256, 256, 0, s>>>(out, reinterpret_cast<const __half*>(a.hidden) + (size_t)slot * a.B * row_halves,
                                                 n_trees, row_halves);
}

static void launch(SmzTc32Image* im, dim3 grid, cudaStream_t s, bool pdl, const SmzArena& a, const Chain& c0, const Chain& c1,
                   Job job, int sim) {
  job.exact_elu = im->exact_elu;
  // observations wider than one K tile: the instantiation that streams the first layer's K in slices
  const bool wide = job.input_kind == IN_OBS && c0.kin > KMAX;
  auto* k = wide ? (im->nprod == 1 ? k_tc32_chain_m64<1, false, false, KMAX, true>
                                   : (im->exact_elu ? k_tc32_chain_m64<3, true, false, KMAX, true> : k_tc32_chain_m64<3, false, false, KMAX, true>))
                 : (im->nprod == 1 ? k_tc32_chain_m64<1, false, false, KMAX, false>
                                   : (im->exact_elu ? k_tc32_chain_m64<3, true, false, KMAX, false> : k_tc32_chain_m64<3, false, false, KMAX, false>));
  smz_launch(k, grid, dim3(NTHR), (size_t)im->smem_bytes, s, pdl, a, c0, c1, job, sim);
}

void smz_tc32_root(SmzTc32Image* im, const SmzArena& a, const SmzNetShape& sh, int n_trees, const float* obs, cudaStream_t s) {
  Job job{};
  job.input_kind = IN_OBS; job.n_rows = n_trees; job.in = obs; job.obs = sh.obs; job.S = sh.S;
  job.hidden_split_dst = reinterpret_cast<__half*>(a.hidden);          // slot 0
  job.policy_dst = a.out_policy; job.value_dst = a.out_value; job.pstride = a.W;
  launch(im, dim3((n_trees + TM - 1) / TM), s, false, a, im->chain_root, im->chain_root, job, 0);
}

void smz_tc32_sim(SmzTc32Image* im, const SmzArena& a, const SmzNetShape& sh, int n_trees, int sim, bool pdl, cudaStream_t s) {
  Job job{};
  job.input_kind = IN_GATHER; job.n_rows = n_trees; job.S = sh.S;
  job.hidden_split_dst = reinterpret_cast<__half*>(a.hidden) + (size_t)(sim + 1) * a.B * (a.xin_q * 8);
  job.policy_dst = a.out_policy; job.value_dst = a.out_value; job.reward_dst = a.out_reward; job.pstride = a.W;
  launch(im, dim3(2 * ((n_trees + TM - 1) / TM)), s, pdl, a, im->chain_after, im->chain_dyn, job, sim);
}

void smz_tc32_eval(SmzTc32Image* im, const SmzNetShape& sh, int which, int n_rows, const float* in, const int* idx,
                   float* hidden_out, float* policy_out, float* value_out, float* reward_out, int* code_out,
                   int policy_stride, cudaStream_t s) {
  Job job{};
  job.input_kind = (which == 0 || which == 5) ? IN_OBS : IN_ROWS;
  job.n_rows = n_rows; job.in = in; job.idx = idx; job.obs = sh.obs; job.S = sh.S;
  job.hidden_dst = hidden_out; job.policy_dst = policy_out; job.value_dst = value_out; job.reward_dst = reward_out;
  job.code_dst = code_out; job.pstride = policy_stride;
  SmzArena dummy{};
  launch(im, dim3((n_rows + TM - 1) / TM), s, false, dummy, im->chain_single[which], im->chain_single[which], job, 0);
}

// ---------------------------------------------------------------------------------------------
// vision family: the MLP heads (147 -> H -> L x [H -> H] -> S or A, ReLU; neural_network_vision_model.py:188-199,
// :262-296) of a simulation step on the same chain kernel, fp32-grade (three products), five (branch, head) chains
// ---------------------------------------------------------------------------------------------
struct SmzTc32VisionHeads {
  int A, S, H, L;
  unsigned char* pool;     // weight images + biases + chain biases
  size_t pool_bytes;
  __half* w[5][3];         // in (K = 160), mid, out images, each [hi | lo]
  float* b[5][3];
  float* bias_pool;        // [5][MAXL][128]
  unsigned* absmax;        // device [15]
  float* scales;           // device [15][2]
  Chain* chains_dev;       // device [5]
  int smem_bytes;
};

int smz_tc32_vision_create(int A, int S, int H, int L, SmzTc32VisionHeads** out, char* err, size_t err_len) {
  if (L + 2 > MAXL || H > KMAX || S > 64 || A > 32) {
    snprintf(err, err_len, "vision heads on tcgen05: need L <= %d, H <= %d, S <= 64, A <= 32", MAXL - 2, KMAX);
    return SMZ_E_CAPACITY;
  }
  SmzTc32VisionHeads* im = new SmzTc32VisionHeads();
  memset(im, 0, sizeof(*im));
  im->A = A; im->S = S; im->H = H; im->L = L;
  const size_t per_head = (size_t)(KVIS + 2 * KMAX) * TN * 2 * 2 + 3 * TN * 4;
  im->pool_bytes = 5 * per_head + (size_t)5 * MAXL * TN * 4;
  if (cudaMalloc(&im->pool, im->pool_bytes) != cudaSuccess || cudaMalloc(&im->absmax, 15 * sizeof(unsigned)) != cudaSuccess ||
      cudaMalloc(&im->scales, 30 * sizeof(float)) != cudaSuccess || cudaMalloc(&im->chains_dev, 5 * sizeof(Chain)) != cudaSuccess) {
    snprintf(err, err_len, "vision heads on tcgen05: cudaMalloc failed");
    cudaFree(im->pool); cudaFree(im->absmax); cudaFree(im->scales); cudaFree(im->chains_dev);
    delete im;
    return SMZ_E_CUDA;
  }
  unsigned char* p = im->pool;
  for (int h = 0; h < 5; ++h) {
    const int K[3] = {KVIS, KMAX, KMAX};
    for (int i = 0; i < 3; ++i) { im->w[h][i] = (__half*)p; p += (size_t)K[i] * TN * 2 * 2; }
    for (int i = 0; i < 3; ++i) { im->b[h][i] = (float*)p; p += TN * 4; }
  }
  im->bias_pool = (float*)p;
  im->smem_bytes = (int)sizeof(SmemT<KVIS>) + 1024;
  if (cudaFuncSetAttribute((const void*)k_tc32_chain_m64<3, false, true, KVIS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           im->smem_bytes) != cudaSuccess) {
    snprintf(err, err_len, "vision heads on tcgen05: %d bytes of shared memory per CTA are not available", im->smem_bytes);
    smz_tc32_vision_destroy(im);
    return SMZ_E_CAPACITY;
  }
  *out = im;
  return SMZ_OK;
}

void smz_tc32_vision_destroy(SmzTc32VisionHeads* im) {
  if (!im) return;
  cudaFree(im->pool); cudaFree(im->absmax); cudaFree(im->scales); cudaFree(im->chains_dev);
  delete im;
}

int smz_tc32_vision_pack(SmzTc32VisionHeads* im, const float* blob, const SmzVisionHeadSrc* src, cudaStream_t s, char* err,
                         size_t err_len) {
  if (cudaMemsetAsync(im->pool, 0, im->pool_bytes, s) != cudaSuccess || cudaMemsetAsync(im->absmax, 0, 15 * sizeof(unsigned), s) != cudaSuccess) {
    snprintf(err, err_len, "vision heads on tcgen05: memset failed");
    return SMZ_E_CUDA;
  }
  const int H = im->H, L = im->L, FLATK = 147;
  for (int h = 0; h < 5; ++h) {
    const SmzVisionHeadSrc& q = src[h];
    k_absmax<<<64, 256, 0, s>>>(blob + q.in_w, H * FLATK, im->absmax + h * 3 + 0);
    if (L > 0) k_absmax<<<64, 256, 0, s>>>(blob + q.mid_w, H * H, im->absmax + h * 3 + 1);
    k_absmax<<<64, 256, 0, s>>>(blob + q.out_w, q.n_out * H, im->absmax + h * 3 + 2);
  }
  for (int i = 0; i < 15; ++i) k_scale_from_absmax<<<1, 1, 0, s>>>(im->absmax + i, im->scales + 2 * i, im->scales + 2 * i + 1);
  for (int h = 0; h < 5; ++h) {
    const SmzVisionHeadSrc& q = src[h];
    const float* sc = im->scales + h * 6;
    k_pack_split<<<(H * FLATK + 255) / 256, 256, 0, s>>>(im->w[h][0], KVIS, blob + q.in_w, sc + 0, H, FLATK, FLATK, 0, 0, 0, 0);
    k_copy_f32<<<1, 128, 0, s>>>(im->b[h][0], blob + q.in_b, H);
    if (L > 0) {
      k_pack_split<<<(H * H + 255) / 256, 256, 0, s>>>(im->w[h][1], KMAX, blob + q.mid_w, sc + 2, H, H, H, 0, 0, 0, 0);
      k_copy_f32<<<1, 128, 0, s>>>(im->b[h][1], blob + q.mid_b, H);
    }
    k_pack_split<<<(q.n_out * H + 255) / 256, 256, 0, s>>>(im->w[h][2], KMAX, blob + q.out_w, sc + 4, q.n_out, H, H, 0, 0, 0, 0);
    k_fill_f32<<<1, 128, 0, s>>>(im->b[h][2], -1e30f, TN);          // padded logits: probability exactly 0
    k_copy_f32<<<1, 128, 0, s>>>(im->b[h][2], blob + q.out_b, q.n_out);
  }
  float host_scales[30];
  if (cudaMemcpyAsync(host_scales, im->scales, sizeof(host_scales), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess) {
    snprintf(err, err_len, "vision heads on tcgen05: reading the layer scales back failed");
    return SMZ_E_CUDA;
  }
  Chain chains[5];
  for (int h = 0; h < 5; ++h) {
    Chain& ch = chains[h];
    memset(&ch, 0, sizeof(ch));
    float* bias_dst = im->bias_pool + (size_t)h * MAXL * TN;
    int l = 0;
    auto add = [&](int i, int K, int kind) {
      ch.layer[l].w = im->w[h][i]; ch.layer[l].K = K; ch.layer[l].kind = kind;
      ch.inv_scale[l] = host_scales[h * 6 + 2 * i + 1];
      k_copy_f32<<<1, TN, 0, s>>>(bias_dst + (size_t)l * TN, im->b[h][i], TN);
      ++l;
    };
    add(0, KVIS, LK_HIDDEN);
    for (int i = 0; i < L; ++i) add(1, KMAX, LK_HIDDEN);
    add(2, KMAX, src[h].is_policy ? LK_CODE : LK_PRED);
    ch.n_layers = l; ch.bias = bias_dst; ch.kin = KVIS; ch.onehot_pad = 0;
    ch.n_policy = src[h].is_policy ? src[h].n_out : 0;
  }
  if (cudaMemcpyAsync(im->chains_dev, chains, sizeof(chains), cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
    snprintf(err, err_len, "vision heads on tcgen05: weight packing failed");
    return SMZ_E_CUDA;
  }
  return SMZ_OK;
}

// heads of simulation `sim` for the compacted rows of both branches; feat as written by the convolution stage
void smz_tc32_vision_heads(SmzTc32VisionHeads* im, const SmzArena& a, int n_trees, int sim, const float* feat, bool pdl,
                           cudaStream_t s) {
  Job job{};
  job.input_kind = IN_FEAT; job.n_rows = n_trees; job.S = im->S;
  job.feat = feat; job.vchains = im->chains_dev;
  job.policy_dst = a.out_policy; job.value_dst = a.out_value; job.reward_dst = a.out_reward; job.pstride = a.W;
  Chain none{};
  smz_launch(k_tc32_chain_m64<3, false, true, KVIS, false>, dim3(5 * ((n_trees + TM - 1) / TM)), dim3(NTHR), (size_t)im->smem_bytes, s, pdl,
             a, none, none, job, sim);
}
