// Shared device/host helpers for libpertgnn (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pertgnn.h"  // prototypes + PERT_ERR_* (keeps definitions and ABI header in sync)

#define PERT_NUM_SMS 148          // B200: 2 dies x 74 SMs

#define PERT_LAUNCH_CHECK()                          \
  do {                                               \
    cudaError_t e__ = cudaPeekAtLastError();         \
    if (e__ != cudaSuccess) return (int)e__;         \
  } while (0)

static inline int pert_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float4 ld4(const float* p) {
  return *reinterpret_cast<const float4*>(p);
}
__device__ __forceinline__ void st4(float* p, float4 v) {
  *reinterpret_cast<float4*>(p) = v;
}
__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 f4fma(float s, float4 a, float4 acc) {
  return make_float4(fmaf(s, a.x, acc.x), fmaf(s, a.y, acc.y), fmaf(s, a.z, acc.z), fmaf(s, a.w, acc.w));
}
__device__ __forceinline__ float f4dot(float4 a, float4 b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
__device__ __forceinline__ float4 f4max(float4 a, float4 b) {
  return make_float4(fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}
__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4scale(float s, float4 a) {
  return make_float4(s * a.x, s * a.y, s * a.z, s * a.w);
}
// 16-byte vector reduction to global memory (REDG.E.ADD.F32x4, sm_90+).
__device__ __forceinline__ void red4(float* p, float4 v) {
  atomicAdd(reinterpret_cast<float4*>(p), v);
}
// butterfly sum over a sub-warp group of LPR lanes; every lane of the group gets the sum.
template <int LPR>
__device__ __forceinline__ float group_sum(float v, unsigned gmask) {
#pragma unroll
  for (int off = LPR >> 1; off > 0; off >>= 1) v += __shfl_xor_sync(gmask, v, off);
  return v;
}

// ---------------------------------------------------------------- dropout masks (counter-based, no stored state)
// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants).  Pure function of (counter, key): any unit's mask can
// be recomputed from (seed, offset, layer, position) alone -- by the backward pass, by pert_dropout_mask and by the
// numpy restatement the tests compare against -- and does not depend on the launch geometry.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k.x += 0x9E3779B9u;
      k.y += 0xBB67AE85u;
    }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}
// The four words that decide columns 4*(j % (H/4)) + 0..3 of row j / (H/4) of an [N, H] activation:
// key = (seed lo, seed hi), counter = (j lo, j hi, layer, offset).  Unit k is dropped iff word k < t.
__device__ __forceinline__ uint4 dropout_words(unsigned long long seed, unsigned long long offset, int layer,
                                               unsigned long long j) {
  return philox4x32_10(make_uint4((uint32_t)j, (uint32_t)(j >> 32), (uint32_t)layer, (uint32_t)offset),
                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}
struct PertDropout {            // by-value kernel argument of the fused BatchNorm-apply dropout
  const long long* rng;         // device (seed, offset), caller-owned
  unsigned long long t;         // drop iff word < t;  t = floor(p 2^32)  (2^32 at p = 1: everything dropped)
  float scale;                  // 1 / (1 - p);  0 at p = 1
  int layer;
};
// host: threshold and scale of a dropout probability; false if p is NaN or outside [0, 1]
static inline bool pert_dropout_params(float p, unsigned long long* t, float* scale) {
  if (!(p >= 0.f && p <= 1.f)) return false;
  const double pd = (double)p;
  *t = (unsigned long long)floor(pd * 4294967296.0);
  *scale = p == 1.f ? 0.f : (float)(1.0 / (1.0 - pd));
  return true;
}

// engine-internal entry points (not part of the C-ABI)
struct PertTiles {            // graph-aligned tile list of one batch for one row width (csrc/tconv_tile.cu)
  const int* tile_ptr;        // [*ntiles + 1] node boundaries (device)
  const int* ntiles;          // device scalar
  int max_tiles, T, ecap;     // capacity of tile_ptr; nodes / staged edges a tile may hold
};
unsigned int* pert_ticket_slot();   // next slot of the self-resetting ticket ring (csrc/gemm_tc.cu)
long long pert_tile_list_ints(long long N, long long B);
bool pert_tile_fixed_ok(long long N, long long E, long long B, int H, int n_rpc);
int pert_tile_list_view(long long N, long long E, long long B, int H, int n_rpc, int* tiles_mem, PertTiles* out);
int pert_tile_list_bounds(const int64_t* batch, long long N, long long B, int* tiles_mem, cudaStream_t st);
int pert_tile_list_build(int has_batch, long long N, long long E, long long B, const int* rowptr, int H, int n_rpc,
                         int* tiles_mem, PertTiles* out, cudaStream_t st);
int pert_tconv_fwd_stats(const float* q, const float* k, const float* v, const float* s, int ld, const int* rowptr,
                         const int* csr_src, const int* csr_if, const int* csr_rpc, const float* t_if,
                         const float* t_rpc, float* out, int ld_out, float* alpha, int n_rpc, long long N, long long E,
                         long long B_hint, int H, double* bn_acc, int* fused, const PertTiles* tiles, void* stream);
int pert_tconv_bwd_tiles(const float* g, int ld_g, const float* q, const float* k, const float* v, int ld,
                         const int* rowptr, const int* csr_src, const int* csr_if, const int* csr_rpc,
                         const int* colptr, const int* csc_pos, const int* csc_dst, const float* t_if,
                         const float* t_rpc, const float* alpha, float* dq, float* dk, float* dv, int ld_d, float* dsp,
                         float* rpc_ws, float* dt_if, float* dt_rpc, int n_rpc, long long N, long long E,
                         long long B_hint, int H, const PertTiles* tiles, void* stream);
int pert_bn_fwd_ex(const float* x, int ld_x, const float* gamma, const float* beta, float* running_mean,
                   float* running_var, long long* num_batches_tracked, float eps, float momentum, int training,
                   int relu, float* mean, float* rstd, float* y, int ld_y, long long N, int H, void* workspace,
                   long long workspace_bytes, int stats_ready, float dropout_p, const long long* rng_state,
                   int layer, void* stream);
int pert_bn_bwd_ex(const float* dy, int ld_dy, const float* y, int ld_y, const float* x, int ld_x, const float* mean,
                   const float* rstd, const float* gamma, int relu, int training, float dropout_scale, float* dx,
                   int ld_dx, float* dgamma, float* dbeta, float* sums, long long N, int H, void* stream);
