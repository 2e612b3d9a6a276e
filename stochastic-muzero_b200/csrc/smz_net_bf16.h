// smz_net_bf16.h — bf16 tcgen05/TMEM network step (throughput mode); see smz_net_bf16.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "smz_kernels.h"

struct SmzBf16Image;

int smz_bf16_create(const SmzNetShape& sh, const SmzArena& a, SmzBf16Image** out, char* err, size_t err_len);
void smz_bf16_destroy(SmzBf16Image* im);
int smz_bf16_pack(SmzBf16Image* im, const SmzNetShape& sh, const float* blob_dev, cudaStream_t s, char* err,
                  size_t err_len);
void smz_bf16_root(SmzBf16Image* im, const SmzArena& a, const SmzNetShape& sh, int n_trees, const float* obs,
                   cudaStream_t s);
void smz_bf16_sim(SmzBf16Image* im, const SmzArena& a, const SmzNetShape& sh, int n_trees, int sim, bool pdl,
                  cudaStream_t s);
void smz_bf16_eval(SmzBf16Image* im, const SmzNetShape& sh, int which, int n_rows, const float* in, const int* idx,
                   float* hidden_out, float* policy_out, float* value_out, float* reward_out, int* code_out,
                   int policy_stride, cudaStream_t s);
// bf16 mode keeps the arena's hidden-state store in bf16 ([slot][B][64]); this widens one slot to fp32 rows
void smz_bf16_read_hidden(const SmzArena& a, int slot, int n_trees, float* out, cudaStream_t s);
