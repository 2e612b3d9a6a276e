// Microbenchmark: the hand-off of a hidden layer's activations to the next layer's tcgen05.mma in the 64-row chain
// (k_bf16_chain_m32 / _m64), with A read from shared memory (SS) or from tensor memory (TS).
//   One CTA: 16 epilogue warps (warp w: TMEM lane quarter w % 4, column slice w / 4 of every round) + 1 issuer warp,
//   M = 64, N = 128, K = 128 bf16 (8 MMAs of K = 16 per layer), the kernel's descriptors and named barriers.
//   SS: st.shared of the packed bf16 pairs + fence.proxy.async + bar.arrive (tcgen05 fence on the last round), two
//       accumulators used alternately — the chain kernel before it read A from TMEM.
//   TS: tcgen05.st.16x128b into the A columns of TMEM + tcgen05.wait::st + tcgen05.fence::before_thread_sync +
//       bar.arrive, one accumulator (128 columns) + the A operand (64 columns).
// R = 1, 2 or 4 rounds per layer: round c hands over K columns [c * 128 / R, (c + 1) * 128 / R) and the issuer issues
// their K-steps as soon as that round's barrier completes.
// Clock stamps of epilogue warp 0: "accumulator seen" (mbarrier wait returned) and "accumulator in registers"
// (tcgen05.wait::ld returned) of every layer.  hand-off = next layer's "seen" - this layer's "in registers".
// Known answer: layers 0 .. NL-2 multiply by the identity (the activations pass through unchanged, as bf16 integers),
// the last layer by a random integer matrix, so the final accumulator must equal A0 * B^T exactly (host GEMM).
// Layout probe: which (lane, column) each register of tcgen05.st.16x128b.x2 lands in, read back with 32x32b.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../stochastic-muzero_b200/csrc -o a_operand_handoff a_operand_handoff.cu
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <vector>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include "smz_tc_ptx.cuh"
using namespace smz_tc;

constexpr int M = 64, N = 128, K = 128, NL = 12, NEPI = 512, NTHR = NEPI + 32;
constexpr int CHUNK_A = M * 16, CHUNK_B = N * 16;
constexpr unsigned IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
constexpr int SMEM = CHUNK_A * (K / 8) + 2 * CHUNK_B * (K / 8) + 1024;

__device__ __forceinline__ void nb_arrive(int id) { __syncwarp(); asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(NTHR) : "memory"); }
__device__ __forceinline__ void nb_sync(int id) { __syncwarp(); asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NTHR) : "memory"); }
__device__ __forceinline__ void umma_ss(unsigned d, unsigned long long ad, unsigned long long bd, unsigned acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d), "l"(ad), "l"(bd), "r"(IDESC), "r"(acc) : "memory");
}

// a0: [M][K] bf16 row-major; bid, brand: [N][K] bf16 row-major; out: [M][N] fp32; stamps: [NL][2]
template <bool TS, int R>
__global__ void __launch_bounds__(NTHR, 1) k_chain(const __nv_bfloat16* a0, const __nv_bfloat16* bid, const __nv_bfloat16* brand,
                                                   float* out, long long* stamps) {
  extern __shared__ unsigned char raw_smem[];
  unsigned char* sa = (unsigned char*)(((uintptr_t)raw_smem + 1023) & ~uintptr_t(1023));
  unsigned char* sb[2] = {sa + CHUNK_A * (K / 8), sa + CHUNK_A * (K / 8) + CHUNK_B * (K / 8)};
  __shared__ unsigned long long bar;
  __shared__ unsigned tmem_base;
  __shared__ long long st_smem[NL][2];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // canonical K-major no-swizzle images: (k / 8) * CHUNK + row * 16 + (k % 8) * 2
  for (int i = tid; i < M * K; i += NTHR) {
    const int m = i / K, kk = i % K;
    *(__nv_bfloat16*)(sa + (kk / 8) * CHUNK_A + m * 16 + (kk % 8) * 2) = a0[i];
  }
  for (int i = tid; i < N * K; i += NTHR) {
    const int n = i / K, kk = i % K;
    *(__nv_bfloat16*)(sb[0] + (kk / 8) * CHUNK_B + n * 16 + (kk % 8) * 2) = bid[i];
    *(__nv_bfloat16*)(sb[1] + (kk / 8) * CHUNK_B + n * 16 + (kk % 8) * 2) = brand[i];
  }
  if (tid == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(&tmem_base)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = tmem_base;
  constexpr int KPR = 8 / R;            // K-steps per round
  constexpr int GPR = 4 / R;            // 8-column accumulator groups per warp and round

  if (warp == NEPI / 32) {
    const unsigned long long ad = umma_desc(s32(sa), CHUNK_A, 128);
    for (int l = 0; l < NL; ++l) {
      const unsigned long long bd = umma_desc(s32(sb[l == NL - 1]), CHUNK_B, 128);
      const unsigned d = TS ? tmem : tmem + (unsigned)((l & 1) * N);
      for (int c = 0; c < R; ++c) {
        if (l > 0) nb_sync(2 + c);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < KPR; ++j) {
            const int k = c * KPR + j;
            const unsigned long long bk = bd + (unsigned long long)(k * ((2 * CHUNK_B) >> 4));
            if (TS && l > 0)
              umma_ts(d, tmem + N + 8 * k, bk, IDESC, k > 0 ? 1u : 0u);
            else
              umma_ss(d, ad + (unsigned long long)(k * ((2 * CHUNK_A) >> 4)), bk, k > 0 ? 1u : 0u);
          }
        }
        __syncwarp();
      }
      if (lane == 0) umma_commit(&bar);
      __syncwarp();
    }
  } else {
    const int q = warp & 3, cb = warp >> 2;
    const int rA = 16 * q + (lane >> 2), rB = rA + 8, cq = 2 * (lane & 3);
    const unsigned lane_t = tmem + ((unsigned)(q * 32) << 16);
    for (int l = 0; l < NL; ++l) {
      const unsigned dcol = TS ? 0u : (unsigned)((l & 1) * N);
      mbar_wait(&bar, l & 1);
      if (tid == 0) st_smem[l][0] = clock64();
      __syncwarp();
      tc_fence_after();
      unsigned r[16];
#pragma unroll
      for (int c = 0; c < R; ++c) {
        const unsigned col = (unsigned)(c * (N / R) + cb * 8 * GPR);
        if constexpr (R == 1) tmem_ld16x256_x4(lane_t + dcol + col, r);
        else if constexpr (R == 2) tmem_ld16x256_x2(lane_t + dcol + col, r + 8 * c);
        else tmem_ld16x256_x1(lane_t + dcol + col, r + 4 * c);
      }
      tmem_wait_ld();
      if (tid == 0) st_smem[l][1] = clock64();
      if (l == NL - 1) {
#pragma unroll
        for (int c = 0; c < R; ++c)
#pragma unroll
          for (int g = 0; g < GPR; ++g) {
            const int col = c * (N / R) + cb * 8 * GPR + g * 8 + cq;
            const unsigned* rr = r + 4 * (c * GPR + g);
            out[rA * N + col] = __uint_as_float(rr[0]); out[rA * N + col + 1] = __uint_as_float(rr[1]);
            out[rB * N + col] = __uint_as_float(rr[2]); out[rB * N + col + 1] = __uint_as_float(rr[3]);
          }
        break;
      }
#pragma unroll
      for (int c = 0; c < R; ++c) {
        unsigned p[2 * GPR];          // {row rA, row rB} per group
#pragma unroll
        for (int g = 0; g < GPR; ++g) {
          const unsigned* rr = r + 4 * (c * GPR + g);
          p[2 * g] = pack_bf16(__uint_as_float(rr[0]), __uint_as_float(rr[1]));
          p[2 * g + 1] = pack_bf16(__uint_as_float(rr[2]), __uint_as_float(rr[3]));
        }
        const int col0 = c * (N / R) + cb * 8 * GPR;
        if constexpr (TS) {
          const unsigned ta = lane_t + N + col0 / 2;
          if constexpr (GPR == 1) tmem_st16x128_x1(ta, p[0], p[1]);
          else if constexpr (GPR == 2) tmem_st16x128_x2(ta, p);
          else tmem_st16x128_x4(ta, p);
          tmem_wait_st();
          tc_fence_before();
        } else {
#pragma unroll
          for (int g = 0; g < GPR; ++g) {
            const int col = col0 + g * 8 + cq;
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(s32(sa + (col >> 3) * CHUNK_A + rA * 16 + (col & 7) * 2)), "r"(p[2 * g]) : "memory");
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(s32(sa + (col >> 3) * CHUNK_A + rB * 16 + (col & 7) * 2)), "r"(p[2 * g + 1]) : "memory");
          }
          fence_async_smem();
          if (c == R - 1) tc_fence_before();
        }
        nb_arrive(2 + c);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 2 * NL) stamps[tid] = st_smem[tid / 2][tid % 2];
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256) : "memory");
}

// layout probe: warp 0 stores register j of thread t (value 0x100 * t + j + 1) with tcgen05.st.16x128b.x2 at column 0,
// then reads lanes 0..31 x columns 0..7 back with 32x32b (thread t <-> lane t)
__global__ void k_probe(unsigned* out) {
  __shared__ unsigned tmem_base;
  const int lane = threadIdx.x;
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(&tmem_base)), "r"(32) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = tmem_base;
  unsigned z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(tmem), "r"(z[0]), "r"(z[1]),
               "r"(z[2]), "r"(z[3]), "r"(z[4]), "r"(z[5]), "r"(z[6]), "r"(z[7]) : "memory");
  tmem_wait_st();
  unsigned v[4];
  for (int j = 0; j < 4; ++j) v[j] = 0x100u * lane + j + 1;
  tmem_st16x128_x2(tmem, v);
  tmem_wait_st();
  unsigned r[8];
  tmem_ld8_nowait(tmem, r);
  tmem_wait_ld();
  for (int c = 0; c < 8; ++c) out[lane * 8 + c] = r[c];
  __syncwarp();
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(32) : "memory");
}

static float bf2f(__nv_bfloat16 b) { return __bfloat162float(b); }

template <bool TS, int R>
static bool run(const char* name, const __nv_bfloat16* d_a, const __nv_bfloat16* d_bid, const __nv_bfloat16* d_br, float* d_out,
                long long* d_st, const std::vector<float>& ref) {
  cudaFuncSetAttribute(k_chain<TS, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
  std::vector<double> hand, per;
  bool exact = true;
  for (int rep = 0; rep < 7; ++rep) {
    cudaMemset(d_out, 0, M * N * 4);
    k_chain<TS, R><<<1, NTHR, SMEM>>>(d_a, d_bid, d_br, d_out, d_st);
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: %s\n", name, cudaGetErrorString(e)); return false; }
    long long st[NL][2];
    std::vector<float> out(M * N);
    cudaMemcpy(st, d_st, sizeof(st), cudaMemcpyDeviceToHost);
    cudaMemcpy(out.data(), d_out, M * N * 4, cudaMemcpyDeviceToHost);
    for (int i = 0; i < M * N; ++i) exact &= out[i] == ref[i];
    if (rep == 0) continue;            // first launch: module load, cold instruction cache
    double h = 0, p = 0;
    for (int l = 1; l < NL - 1; ++l) { h += st[l + 1][0] - st[l][1]; p += st[l + 1][0] - st[l][0]; }
    hand.push_back(h / (NL - 2)); per.push_back(p / (NL - 2));
  }
  std::sort(hand.begin(), hand.end()); std::sort(per.begin(), per.end());
  printf("%-4s %d round%s: accumulator in registers -> next accumulator seen  median %6.0f  (min %6.0f, max %6.0f) cycles | "
         "layer period median %6.0f | known answer %s\n",
         name, R, R > 1 ? "s" : " ", hand[hand.size() / 2], hand.front(), hand.back(), per[per.size() / 2], exact ? "exact" : "MISMATCH");
  return exact;
}

int main() {
  // A0, B: small integers (exact in bf16; every product sum is exact in fp32)
  srand(1234);
  std::vector<__nv_bfloat16> a(M * K), bid(N * K), br(N * K);
  for (auto& x : a) x = __float2bfloat16((float)(rand() % 9 - 4));
  for (auto& x : br) x = __float2bfloat16((float)(rand() % 9 - 4));
  for (int n = 0; n < N; ++n)
    for (int k = 0; k < K; ++k) bid[n * K + k] = __float2bfloat16(n == k ? 1.f : 0.f);
  std::vector<float> ref(M * N);
  for (int m = 0; m < M; ++m)
    for (int n = 0; n < N; ++n) {
      float s = 0.f;
      for (int k = 0; k < K; ++k) s += bf2f(a[m * K + k]) * bf2f(br[n * K + k]);
      ref[m * N + n] = s;
    }
  __nv_bfloat16 *d_a, *d_bid, *d_br;
  float* d_out;
  long long* d_st;
  unsigned* d_probe;
  cudaMalloc(&d_a, M * K * 2); cudaMalloc(&d_bid, N * K * 2); cudaMalloc(&d_br, N * K * 2);
  cudaMalloc(&d_out, M * N * 4); cudaMalloc(&d_st, NL * 2 * 8); cudaMalloc(&d_probe, 32 * 8 * 4);
  cudaMemcpy(d_a, a.data(), M * K * 2, cudaMemcpyHostToDevice);
  cudaMemcpy(d_bid, bid.data(), N * K * 2, cudaMemcpyHostToDevice);
  cudaMemcpy(d_br, br.data(), N * K * 2, cudaMemcpyHostToDevice);

  k_probe<<<1, 32>>>(d_probe);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("probe: %s\n", cudaGetErrorString(e)); return 1; }
  unsigned pr[32 * 8];
  cudaMemcpy(pr, d_probe, sizeof(pr), cudaMemcpyDeviceToHost);
  int bad = 0;
  for (int lane = 0; lane < 32; ++lane)
    for (int c = 0; c < 8; ++c) {
      // expected: repetition i = c / 4 -> thread t with t % 4 == c % 4 writes reg 2i to lane t / 4, reg 2i + 1 to lane t / 4 + 8
      unsigned want = 0;
      if (lane < 16) {
        const int t = 4 * (lane % 8) + c % 4, j = 2 * (c / 4) + (lane >= 8);
        want = 0x100u * t + j + 1;
      }
      if (pr[lane * 8 + c] != want) {
        if (bad++ < 8) printf("probe: lane %2d column %d holds %#x, expected %#x\n", lane, c, pr[lane * 8 + c], want);
      }
    }
  printf("tcgen05.st.16x128b.x2 layout (reg 2i -> lane t/4, reg 2i+1 -> lane t/4+8, column 4i + t%%4; lanes 16-31 untouched): %s\n",
         bad ? "MISMATCH" : "confirmed");
  bool ok = true;
  ok &= run<false, 1>("SS", d_a, d_bid, d_br, d_out, d_st, ref);
  ok &= run<true, 1>("TS", d_a, d_bid, d_br, d_out, d_st, ref);
  ok &= run<false, 2>("SS", d_a, d_bid, d_br, d_out, d_st, ref);
  ok &= run<true, 2>("TS", d_a, d_bid, d_br, d_out, d_st, ref);
  ok &= run<false, 4>("SS", d_a, d_bid, d_br, d_out, d_st, ref);
  ok &= run<true, 4>("TS", d_a, d_bid, d_br, d_out, d_st, ref);
  return ok && !bad ? 0 : 1;
}
