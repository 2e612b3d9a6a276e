// smz_kernels.h — host-side launchers shared between the translation units of libsmz.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "smz_common.cuh"

// ---- tree kernels (smz_tree.cu, compiled with -fmad=false) ---------------------------------------
void smz_launch_root_expand(const SmzArena& a, int lanes, int n_trees, const float* policy, int pstride,
                            const int* root_to_play, int train, const double* dirichlet, const uint32_t* legal,
                            const int* budget, const unsigned char* explore, cudaStream_t s);
void smz_launch_select(const SmzArena& a, int lanes, int n_trees, int sim, int* o_slot, int* o_action, int* o_branch,
                       cudaStream_t s);
void smz_launch_expand_backup(const SmzArena& a, int lanes, int n_trees, int sim, const float* policy, int pstride,
                              const float* value, const float* reward, cudaStream_t s);
// expand+backup of `sim` fused with the descent of `sim + 1` (internal-network loop)
void smz_launch_backup_select(const SmzArena& a, int lanes, int n_trees, int sim, bool pdl, cudaStream_t s);
void smz_launch_read_roots(const SmzArena& a, int n_trees, int* visits, float* values, double* priors, float* rewards,
                           int* error_out, cudaStream_t s);
void smz_launch_begin_search(const SmzArena& a, cudaStream_t s);
void smz_launch_set_seed(unsigned long long* dst, unsigned long long seed, unsigned long long tree_id_offset, cudaStream_t s);
void smz_launch_dirichlet(const SmzArena& a, int n_trees, const uint32_t* legal, int train, const int* budget,
                          const unsigned char* explore, cudaStream_t s);
void smz_launch_select_actions(const SmzArena& a, int n_trees, double temperature, const double* u, int* actions,
                               double* policy, double* stored, cudaStream_t s);
// Gumbel searches: root values, logits and Gumbels after the root expansion; the action / improved-policy read-out
void smz_launch_gumbel_root(const SmzArena& a, int n_trees, const float* root_value, int train, const double* given,
                            const unsigned char* explore, cudaStream_t s);
void smz_launch_read_gumbel(const SmzArena& a, int n_trees, int* actions, double* improved, double* gumbels,
                            cudaStream_t s);

// ---- network (smz_net_f32.cu / smz_net_bf16.cu) --------------------------------------------------
// Model shape and the padded fp32 weight image the CUDA-core path reads (built by smz_net_pack).
struct SmzNetShape {
  int obs, A, C, S, H, L, OH;   // OH = max(A, C): one-hot width of actions and chance codes
  int obs_pad;                  // obs rounded up to 32
};

// One network in the padded fp32 image: every matrix is stored transposed, Wt[k][SMZ_HP] (k-major,
// output channel contiguous, zero padded), so a k-slab is one contiguous, coalesced 512-byte row.
struct SmzNetF32 {
  const float* in_wt;    // [kin_pad][HP]
  const float* in_b;     // [HP]
  const float* emb;      // [OH][HP] columns S.. of the first layer (one-hot folded in), or null
  const float* mid_wt;   // [HP][HP] (tied across the L hidden layers)
  const float* mid_b;    // [HP]
  const float* head_wt;  // [HP][HP] concatenated output heads, see smz_net_f32.cu
  const float* head_b;   // [HP]
  int kin_pad;
};

struct SmzNetImageF32 {
  SmzNetF32 repr, pred, adyn, apred, dyn, enc;
};

// floats needed for the fp32 image
size_t smz_net_f32_image_floats(const SmzNetShape& sh);
// blob_dev: the caller's fp32 blob already on the device; image_dev: engine-owned buffer
void smz_net_f32_pack(const SmzNetShape& sh, const float* blob_dev, float* image_dev, SmzNetImageF32* out,
                      cudaStream_t s);
uint64_t smz_blob_floats(const SmzNetShape& sh);

// root: representation + prediction for trees [0, n_trees) from obs -> hidden slot 0, out_policy/out_value
void smz_net_f32_root(const SmzArena& a, const SmzNetShape& sh, const SmzNetImageF32& img, int n_trees,
                      const float* obs, cudaStream_t s);
// one simulation: compacted afterstate / dynamics rows of simulation `sim`
void smz_net_f32_sim(const SmzArena& a, const SmzNetShape& sh, const SmzNetImageF32& img, int n_trees, int sim,
                     cudaStream_t s);
// stand-alone evaluation on caller rows (smz_net_eval)
void smz_net_f32_eval(const SmzNetShape& sh, const SmzNetImageF32& img, int which, int n_rows, const float* in,
                      const int* idx, float* hidden_out, float* policy_out, float* value_out, float* reward_out,
                      int* code_out, int policy_stride, cudaStream_t s);
