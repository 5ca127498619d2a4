// Whole-model step engine: SAGEDeterministic forward / backward (reference model.py:76-114 and its autograd
// backward, driven by pert_gnn.py:233-247) as ONE C call each.  The Python-orchestrated path issues ~130 launches
// per step through ctypes + autograd (~4.4 ms of host time at cfg2, 2x the GPU time); here the same kernels are
// issued back-to-back from C++ so the GPU, not the interpreter, bounds the step.
//
// Parameters stay in the reference's layout (one flat fp32 buffer + offsets, PertModelDesc); a small pack kernel
// per layer builds the fused operands each step (W4 = [Wq;Wk;Wv;Ws] with conv-0 columns permuted/padded to the
// [cat_embeds | x | pad] input layout, W4^T for the data gradient, the two halves of lin_edge and their transposes)
// and an unpack kernel scatters the packed gradients back (+=) into the flat gradient buffer.
#include "common.cuh"

#include <stdlib.h>
#include <string.h>
#include <mutex>

namespace {

// ------------------------------------------------------------------ grouped small GEMM (heads, edge tables)
struct SmallGemm {
  const float* A;     // A(m,k) = A[m*sam + k*sak]
  const float* B;     // B(k,n) = B[k*sbk + n*sbn];  nullptr => all ones
  const float* bias;  // [N] or null
  const float* mask;  // same shape/ld as C: result *= (mask > 0)   (ReLU backward) or null
  float* C;           // C[m*ldc + n]
  int M, N, K;
  int sam, sak, sbk, sbn, ldc;
  int relu, accumulate, ksplit;
  int atomic;         // accumulate with atomicAdd (several problems of one launch add into the same C)
};
#define SG_MAX 12
struct SmallGemmBatch {
  SmallGemm p[SG_MAX];
  int count;
};
// BK = 64: these problems are latency-bound chains of (load -> sync -> fma) steps; fewer, fatter steps
constexpr int SG_BM = 32, SG_BN = 64, SG_BK = 64;

__global__ void __launch_bounds__(256) k_small_gemm(SmallGemmBatch batch) {
  const SmallGemm& g = batch.p[blockIdx.y];
  const int tiles_m = (g.M + SG_BM - 1) / SG_BM, tiles_n = (g.N + SG_BN - 1) / SG_BN;
  const int ks = g.ksplit > 0 ? g.ksplit : 1;
  int t = blockIdx.x;
  if (t >= tiles_m * tiles_n * ks) return;
  const int kpart = t % ks;
  t /= ks;
  const int m0 = (t / tiles_n) * SG_BM, n0 = (t % tiles_n) * SG_BN;
  const int klen = (g.K + ks - 1) / ks;
  const int kbeg = kpart * klen, kend = min(g.K, kbeg + klen);
  __shared__ float As[SG_BK][SG_BM + 1];
  __shared__ float Bs[SG_BK][SG_BN + 1];
  const int tid = threadIdx.x;
  const int ty = tid / 16, tx = tid % 16;  // 16x16 threads: 2 rows x 4 cols each
  float acc[2][4] = {};
  for (int k0 = kbeg; k0 < kend; k0 += SG_BK) {
    // all global loads of the step are issued before the first shared-memory store (the compiler cannot hoist
    // loads over possibly-aliasing stores: a load->store loop would serialise 24 DRAM/L2 latencies per step)
    float ra[SG_BM * SG_BK / 256], rb[SG_BN * SG_BK / 256];
#pragma unroll
    for (int u = 0; u < SG_BM * SG_BK / 256; ++u) {
      const int x = tid + u * 256;
      int mm, kk;   // the index that is contiguous in memory is the fast thread index
      if (g.sak == 1) { kk = x % SG_BK; mm = x / SG_BK; } else { mm = x % SG_BM; kk = x / SG_BM; }
      const int m = m0 + mm, k = k0 + kk;
      ra[u] = (m < g.M && k < kend) ? __ldg(g.A + (size_t)m * g.sam + (size_t)k * g.sak) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < SG_BN * SG_BK / 256; ++u) {
      const int x = tid + u * 256;
      int nn, kk;
      if (g.sbk == 1) { kk = x % SG_BK; nn = x / SG_BK; } else { nn = x % SG_BN; kk = x / SG_BN; }
      const int n = n0 + nn, k = k0 + kk;
      float v = 0.f;
      if (n < g.N && k < kend) v = g.B ? __ldg(g.B + (size_t)k * g.sbk + (size_t)n * g.sbn) : 1.f;
      rb[u] = v;
    }
#pragma unroll
    for (int u = 0; u < SG_BM * SG_BK / 256; ++u) {
      const int x = tid + u * 256;
      int mm, kk;
      if (g.sak == 1) { kk = x % SG_BK; mm = x / SG_BK; } else { mm = x % SG_BM; kk = x / SG_BM; }
      As[kk][mm] = ra[u];
    }
#pragma unroll
    for (int u = 0; u < SG_BN * SG_BK / 256; ++u) {
      const int x = tid + u * 256;
      int nn, kk;
      if (g.sbk == 1) { kk = x % SG_BK; nn = x / SG_BK; } else { nn = x % SG_BN; kk = x / SG_BN; }
      Bs[kk][nn] = rb[u];
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SG_BK; ++kk) {
      float a0 = As[kk][ty * 2], a1 = As[kk][ty * 2 + 1];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float b = Bs[kk][tx * 4 + j];
        acc[0][j] = fmaf(a0, b, acc[0][j]);
        acc[1][j] = fmaf(a1, b, acc[1][j]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    int m = m0 + ty * 2 + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j];
      if (g.bias && kpart == 0) v += __ldg(g.bias + n);
      float* c = g.C + (size_t)m * g.ldc + n;
      if (ks > 1 || g.atomic) {
        atomicAdd(c, v);  // split-K: C pre-zeroed / accumulating, no relu/mask
      } else {
        if (g.relu) v = fmaxf(v, 0.f);
        if (g.mask && !(g.mask[(size_t)m * g.ldc + n] > 0.f)) v = 0.f;
        *c = g.accumulate ? (*c + v) : v;
      }
    }
  }
}

int launch_small(const SmallGemmBatch& b, cudaStream_t st) {
  int maxt = 1;
  for (int i = 0; i < b.count; ++i) {
    const SmallGemm& g = b.p[i];
    int ks = g.ksplit > 0 ? g.ksplit : 1;
    int t = ((g.M + SG_BM - 1) / SG_BM) * ((g.N + SG_BN - 1) / SG_BN) * ks;
    if (t > maxt) maxt = t;
  }
  k_small_gemm<<<dim3(maxt, b.count), 256, 0, st>>>(b);
  return 0;
}
SmallGemm sg(const float* A, int sam, int sak, const float* B, int sbk, int sbn, const float* bias, float* C,
             int ldc, int M, int N, int K, int relu = 0, int accumulate = 0, int ksplit = 1,
             const float* mask = nullptr) {
  SmallGemm g;
  g.A = A; g.B = B; g.bias = bias; g.mask = mask; g.C = C; g.M = M; g.N = N; g.K = K;
  g.sam = sam; g.sak = sak; g.sbk = sbk; g.sbn = sbn; g.ldc = ldc;
  g.relu = relu; g.accumulate = accumulate; g.ksplit = ksplit;
  g.atomic = 0;
  return g;
}

// ------------------------------------------------------------------ parameter pack / gradient unpack
struct Seg {
  long long src;  // offset (floats) into the flat parameter (or gradient) buffer
  long long dst;  // offset (floats) into the packed workspace
  int rows, cols, src_ld, dst_ld;
  int transpose;  // dst[c*dst_ld + r] = src[r*src_ld + c]
};
#define SEG_MAX 96   // 96 x 40 B of kernel parameters; layers are grouped into as few launches as fit
struct SegList {
  Seg s[SEG_MAX];
  int count;
};
__global__ void k_pack(const float* __restrict__ params, float* __restrict__ packed, SegList L) {
  const Seg& s = L.s[blockIdx.y];
  int n = s.rows * s.cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int r = i / s.cols, c = i - r * s.cols;
    float v = params[s.src + (size_t)r * s.src_ld + c];
    if (s.transpose) packed[s.dst + (size_t)c * s.dst_ld + r] = v;
    else packed[s.dst + (size_t)r * s.dst_ld + c] = v;
  }
}
// grads[src...] += packed_grad[dst...]   (non-transposed segments only)
__global__ void k_unpack(float* __restrict__ grads, const float* __restrict__ packed, SegList L) {
  const Seg& s = L.s[blockIdx.y];
  if (s.transpose) return;
  int n = s.rows * s.cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int r = i / s.cols, c = i - r * s.cols;
    grads[s.src + (size_t)r * s.src_ld + c] += packed[s.dst + (size_t)r * s.dst_ld + c];
  }
}

// ------------------------------------------------------------------ fused global head (reference model.py: global_linear1 -> ReLU -> global_linear2)
// HEAD_G graphs per CTA, one warp per graph.  z = [pool | entry_emb[entry_id]], h1 = relu(W1 z + b1), out = W2 h1 + b2.
// W1 is staged in shared memory once per CTA (all loads in flight together): transposed [2H][H] for the forward
// (lane = output feature, conflict free, no shuffles), row-major [H][2H] for the backward (lane = input column).
constexpr int HEAD_G = 8;
constexpr int HEAD_T = HEAD_G * 32;
__global__ void __launch_bounds__(HEAD_T) k_head_fwd(const float* __restrict__ pool, const float* __restrict__ table,
                                                     int n_rows, const int64_t* __restrict__ ids,
                                                     const float* __restrict__ W1, const float* __restrict__ b1,
                                                     const float* __restrict__ W2, const float* __restrict__ b2,
                                                     float* __restrict__ z, float* __restrict__ h1,
                                                     float* __restrict__ out, int B, int H, int* status,
                                                     long long* rng_state) {
  extern __shared__ float hs[];                       // W1t [2H][H] | z [HEAD_G][2H]
  // dropout: every BatchNorm apply of this forward has finished (stream order) -> advance the offset for the next one
  if (rng_state && blockIdx.x == 0 && threadIdx.x == 0) rng_state[1] += 1;
  float* w1t = hs;
  float* zs_all = hs + (size_t)2 * H * H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K2 = 2 * H, kq = K2 / 4;
  // lanes along n: the global reads are 16-byte pieces of different rows (32 KB, L2 resident), the transposing
  // shared-memory stores are conflict free
  for (int base = 0; base < H * kq; base += 8 * HEAD_T) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int x = base + u * HEAD_T + threadIdx.x;
      v[u] = x < H * kq ? ldg4(W1 + (size_t)(x % H) * K2 + (x / H) * 4) : f4zero();
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int x = base + u * HEAD_T + threadIdx.x;
      if (x < H * kq) {
        const int n = x % H, k = (x / H) * 4;
        w1t[(k + 0) * H + n] = v[u].x; w1t[(k + 1) * H + n] = v[u].y;
        w1t[(k + 2) * H + n] = v[u].z; w1t[(k + 3) * H + n] = v[u].w;
      }
    }
  }
  const int b = blockIdx.x * HEAD_G + w;
  const bool act = b < B;
  float* zs = zs_all + (size_t)w * K2;
  if (act) {
    int64_t r = ids[b];
    if (r < 0 || r >= n_rows) {
      if (status && lane == 0) atomicExch(status, PERT_ERR_RANGE);
      r = 0;
    }
    for (int c = lane; c < K2; c += 32) {
      const float v = c < H ? pool[(size_t)b * H + c] : __ldg(table + (size_t)r * H + (c - H));
      zs[c] = v;
      z[(size_t)b * K2 + c] = v;
    }
  }
  __syncthreads();
  if (!act) return;
  float o = 0.f;
  for (int n = lane; n < H; n += 32) {
    float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
    for (int k = 0; k < K2; k += 2) {
      a0 = fmaf(w1t[k * H + n], zs[k], a0);
      a1 = fmaf(w1t[(k + 1) * H + n], zs[k + 1], a1);
    }
    const float hv = fmaxf(a0 + a1 + __ldg(b1 + n), 0.f);
    h1[(size_t)b * H + n] = hv;
    o = fmaf(hv, __ldg(W2 + n), o);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) o += __shfl_xor_sync(0xffffffffu, o, off);
  if (lane == 0) out[b] = o + __ldg(b2);
}

// the offset advance of k_head_fwd for a batch without graphs (B == 0: no head launch)
__global__ void k_rng_advance(long long* rng_state) { rng_state[1] += 1; }

// Backward of the head for HEAD_G graphs per CTA: dh1 = dg W2 (h1 > 0); dz = dh1 W1 -> dpool | entry-embedding rows
// (atomic scatter); dW2 += dg h1; db2 += dg; dW1 += dh1^T z; db1 += dh1 (block-level sums, then one atomic per value).
__global__ void __launch_bounds__(HEAD_T) k_head_bwd(const float* __restrict__ dg, const float* __restrict__ z,
                                                     const float* __restrict__ h1, const float* __restrict__ W1,
                                                     const float* __restrict__ W2, const int64_t* __restrict__ ids,
                                                     int n_rows, float* __restrict__ dpool, float* __restrict__ g_entry,
                                                     float* __restrict__ gW1, float* __restrict__ gb1,
                                                     float* __restrict__ gW2, float* __restrict__ gb2, int B, int H) {
  extern __shared__ float hs[];                       // W1 [H][2H] | z [HEAD_G][2H] | dh [HEAD_G][H]
  const int K2 = 2 * H;
  float* w1 = hs;
  float* zs_all = hs + (size_t)H * K2;
  float* dh_all = zs_all + (size_t)HEAD_G * K2;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int base = 0; base < H * K2 / 4; base += 8 * HEAD_T) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int x = base + u * HEAD_T + threadIdx.x;
      v[u] = x < H * K2 / 4 ? ldg4(W1 + (size_t)x * 4) : f4zero();
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int x = base + u * HEAD_T + threadIdx.x;
      if (x < H * K2 / 4) st4(w1 + (size_t)x * 4, v[u]);
    }
  }
  const int b = blockIdx.x * HEAD_G + w;
  const bool act = b < B;
  float* zs = zs_all + (size_t)w * K2;
  float* dh = dh_all + (size_t)w * H;
  const float d = act ? dg[b] : 0.f;
  for (int c = lane; c < K2; c += 32) zs[c] = act ? z[(size_t)b * K2 + c] : 0.f;
  for (int n = lane; n < H; n += 32) {
    const float hv = act ? h1[(size_t)b * H + n] : 0.f;
    dh[n] = hv > 0.f ? d * __ldg(W2 + n) : 0.f;
  }
  __syncthreads();
  if (act) {
    int64_t r = ids[b];
    if (r < 0 || r >= n_rows) r = 0;                  // (the forward pass already raised the status flag)
    for (int c = lane; c < K2; c += 32) {
      float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
      for (int n = 0; n < H; n += 2) {
        a0 = fmaf(dh[n], w1[n * K2 + c], a0);
        a1 = fmaf(dh[n + 1], w1[(n + 1) * K2 + c], a1);
      }
      const float acc = a0 + a1;
      if (c < H) {
        if (dpool) dpool[(size_t)b * H + c] = acc;
      } else {
        atomicAdd(g_entry + (size_t)r * H + (c - H), acc);
      }
    }
  }
  // weight gradients of the block's graphs
  for (int x = threadIdx.x; x < H * K2; x += blockDim.x) {
    const int n = x / K2, c = x - n * K2;
    float t = 0.f;
#pragma unroll
    for (int g = 0; g < HEAD_G; ++g) t = fmaf(dh_all[g * H + n], zs_all[g * K2 + c], t);
    if (t != 0.f) atomicAdd(gW1 + x, t);
  }
  for (int n = threadIdx.x; n < H; n += blockDim.x) {
    float t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int g = 0; g < HEAD_G; ++g) {
      t1 += dh_all[g * H + n];
      const int bb = blockIdx.x * HEAD_G + g;
      if (bb < B) t2 = fmaf(dg[bb], h1[(size_t)bb * H + n], t2);
    }
    if (t1 != 0.f) atomicAdd(gb1 + n, t1);
    if (t2 != 0.f) atomicAdd(gW2 + n, t2);
  }
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int g = 0; g < HEAD_G; ++g) {
      const int bb = blockIdx.x * HEAD_G + g;
      if (bb < B) t += dg[bb];
    }
    atomicAdd(gb2, t);
  }
}


inline long long al64(long long n) { return (n + 63) / 64 * 64; }

struct Ws {
  // packed parameters (zero-initialised region: pads must stay 0)
  float *w4[PERT_MAX_CONVS], *b4[PERT_MAX_CONVS], *w4t[PERT_MAX_CONVS];
  float *weA[PERT_MAX_CONVS], *weB[PERT_MAX_CONVS], *weAt[PERT_MAX_CONVS], *weBt[PERT_MAX_CONVS];
  // packed gradients + table gradients (zeroed at the start of every backward, one memset)
  float* gzero_begin;
  float *dw4[PERT_MAX_CONVS], *db4[PERT_MAX_CONVS], *dweA[PERT_MAX_CONVS], *dweB[PERT_MAX_CONVS];
  float *dt_if[PERT_MAX_CONVS], *dt_rpc[PERT_MAX_CONVS];
  float* gzero_end;
  // forward state
  float *t_if[PERT_MAX_CONVS], *t_rpc[PERT_MAX_CONVS];
  float *x[PERT_MAX_CONVS], *planes[PERT_MAX_CONVS], *out[PERT_MAX_CONVS], *alpha[PERT_MAX_CONVS];
  float* bn_stats[PERT_MAX_CONVS];
  float *bn_part, *pool, *z, *h1;
  // backward temporaries
  float *dplanes, *dx, *dsp, *rpc_ws, *sums, *dpool, *dzent, *dh1;
  int* tiles;      // graph-aligned tile list of the batch (pert_tile_list_ints ints), built in forward, reused in backward
  long long total;  // floats
  long long packed_floats;
};

int k_of(const PertModelDesc* d, int l) { return l == 0 ? d->k0 : d->H; }

Ws carve(const PertModelDesc* d, long long N, long long E, long long B, float* base) {
  Ws w;
  memset(&w, 0, sizeof(w));
  long long off = 0;
  auto take = [&](long long n) {
    float* p = base ? base + off : nullptr;
    off += al64(n > 0 ? n : 1);
    return p;
  };
  const int H = d->H, L = d->n_convs;
  for (int l = 0; l < L; ++l) {
    int K = k_of(d, l);
    w.w4[l] = take(4LL * H * K);
    w.b4[l] = take(4LL * H);
    w.w4t[l] = take(4LL * H * K);
    w.weA[l] = take((long long)H * H);
    w.weB[l] = take((long long)H * H);
    w.weAt[l] = take((long long)H * H);
    w.weBt[l] = take((long long)H * H);
  }
  w.packed_floats = off;
  w.gzero_begin = base ? base + off : nullptr;
  for (int l = 0; l < L; ++l) {
    int K = k_of(d, l);
    w.dw4[l] = take(4LL * H * K);
    w.db4[l] = take(4LL * H);
    w.dweA[l] = take((long long)H * H);
    w.dweB[l] = take((long long)H * H);
    w.dt_if[l] = take((long long)d->n_if * H);
    w.dt_rpc[l] = take((long long)d->n_rpc * H);
  }
  w.gzero_end = base ? base + off : nullptr;
  for (int l = 0; l < L; ++l) {
    int K = k_of(d, l);
    w.t_if[l] = take((long long)d->n_if * H);
    w.t_rpc[l] = take((long long)d->n_rpc * H);
    if (l == 0) w.x[l] = take(N * K);
    w.planes[l] = take(4LL * N * H);
    w.out[l] = take(N * H);
    if (l + 1 < L) w.x[l + 1] = take(N * H);
    w.alpha[l] = take(E);
    w.bn_stats[l] = take(2LL * H);
  }
  w.bn_part = take(pert_bn_workspace_bytes(N, H) / 4 + 16);
  w.tiles = (int*)take(pert_tile_list_ints(N, B));
  w.pool = take(B * H);
  w.z = take(B * 2 * H);
  w.h1 = take(B * H);
  w.dplanes = take(4LL * N * H);
  int kmax = d->k0 > H ? d->k0 : H;
  w.dx = take(N * kmax);
  w.dsp = take(E);
  w.rpc_ws = take(N * PERT_TCONV_RPC_WS_FLOATS);
  w.sums = take(2LL * H);
  w.dpool = take(B * H);
  w.dzent = take(B * H);
  w.dh1 = take(B * H);
  w.total = off;
  return w;
}

// segment list of conv layer l: weights -> W4 / W4^T (conv 0: columns permuted to [emb | x | pad]), biases,
// lin_edge halves and their transposes
constexpr int SEGS_PER_LAYER_MAX = 24;
void append_layer_segs(SegList& S, const PertModelDesc* d, const Ws& w, float* base, int l) {
  const int H = d->H, F = d->F, K = k_of(d, l);
  const int Din = (l == 0) ? F + H : H;
  auto add = [&](long long src, float* dst, int rows, int cols, int src_ld, int dst_ld, int tr) {
    Seg& s = S.s[S.count++];
    s.src = src; s.dst = dst - base; s.rows = rows; s.cols = cols; s.src_ld = src_ld; s.dst_ld = dst_ld;
    s.transpose = tr;
  };
  const long long* wq[4] = {&d->off_wq[l], &d->off_wk[l], &d->off_wv[l], &d->off_ws[l]};
  const long long* bq[4] = {&d->off_bq[l], &d->off_bk[l], &d->off_bv[l], &d->off_bs[l]};
  for (int p = 0; p < 4; ++p) {
    float* dstw = w.w4[l] + (size_t)p * H * K;  // rows p*H..
    float* dstt = w.w4t[l] + (size_t)p * H;     // W4^T [K, 4H]: column block p
    if (l == 0) {
      // reference input order [x(F) | emb(H)] -> internal [emb(H) | x(F) | pad]
      add(*wq[p] + F, dstw, H, H, Din, K, 0);          // emb columns -> cols 0..H
      add(*wq[p], dstw + H, H, F, Din, K, 0);          // x columns   -> cols H..H+F
      add(*wq[p] + F, dstt, H, H, Din, 4 * H, 1);
      add(*wq[p], dstt + (size_t)H * 4 * H, H, F, Din, 4 * H, 1);
    } else {
      add(*wq[p], dstw, H, H, Din, K, 0);
      add(*wq[p], dstt, H, H, Din, 4 * H, 1);
    }
    add(*bq[p], w.b4[l] + (size_t)p * H, 1, H, H, H, 0);
  }
  add(d->off_we[l], w.weA[l], H, H, 2 * H, H, 0);
  add(d->off_we[l] + H, w.weB[l], H, H, 2 * H, H, 0);
  add(d->off_we[l], w.weAt[l], H, H, 2 * H, H, 1);
  add(d->off_we[l] + H, w.weBt[l], H, H, 2 * H, H, 1);
}
// same list but pointing at the packed-gradient buffers (for k_unpack)
void append_layer_grad_segs(SegList& S, const PertModelDesc* d, const Ws& w, float* base, int l) {
  const int first = S.count;
  append_layer_segs(S, d, w, base, l);
  // remap dst from parameter pack to gradient pack (same relative layout inside each buffer)
  for (int i = first; i < S.count; ++i) {
    Seg& s = S.s[i];
    if (s.transpose) continue;
    float* p = base + s.dst;
    const int H = d->H, K = k_of(d, l);
    if (p >= w.w4[l] && p < w.w4[l] + 4LL * H * K) s.dst = (w.dw4[l] + (p - w.w4[l])) - base;
    else if (p >= w.b4[l] && p < w.b4[l] + 4LL * H) s.dst = (w.db4[l] + (p - w.b4[l])) - base;
    else if (p == w.weA[l]) s.dst = w.dweA[l] - base;
    else if (p == w.weB[l]) s.dst = w.dweB[l] - base;
  }
}

// Auxiliary stream for the few places where independent small kernels can run beside the main chain (input prologue
// next to the parameter pack + edge tables; edge-table gradients next to the conv-0 GEMMs).  Fork / join with events,
// so the dependencies also hold inside a CUDA-graph capture.  Created on first (eager) use per device;
// PERT_ENGINE_FORK=0 keeps everything on the caller's stream.
struct AuxStream {
  cudaStream_t s = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int state = 0;   // 0 untried, 1 ready, -1 unavailable
};
// host-side issue of engine calls is serialised per process: the fork/join events of the auxiliary stream are shared
std::mutex& engine_mutex() {
  static std::mutex m;
  return m;
}
// Graph-aligned tile lists (csrc/tconv_tile.cu:k_build_tiles) are OFF by default: measured on B200 (round 2,
// profiles/r2_tile_list_ab.md) the fixed T-node tiles win on every BASELINE shape -- uniform cfg2 0.649 vs 0.690 ms/step,
// cfg2 with +-20 % graph sizes 0.721 vs 0.804, power-law cfg3 1.331 vs 1.388 -- because a fixed tiling has the minimal
// number of tiles (one wave of CTAs at cfg2) and the global-gather variant that cut graphs need is only ~10 % slower
// than the all-in-tile variant, while whole-graph tiles cost a packing kernel per batch and more, unevenly filled
// tiles.  PERT_TILE_LIST=1 turns them on.
bool tiles_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("PERT_TILE_LIST");
    on = (e && e[0] == '1') ? 1 : 0;
  }
  return on == 1;
}
bool bn_fuse_enabled() {   // PERT_BN_FUSE=0: statistics by the separate k_bn_partial pass (debug A/B)
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("PERT_BN_FUSE");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on == 1;
}
AuxStream* aux_stream() {
  static AuxStream aux[64];
  static int enabled = -1;
  if (enabled < 0) {
    const char* e = getenv("PERT_ENGINE_FORK");
    enabled = (e && e[0] == '0') ? 0 : 1;
  }
  if (!enabled) return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  AuxStream& a = aux[dev];
  if (a.state == 0) {
    a.state = -1;
    if (cudaStreamCreateWithFlags(&a.s, cudaStreamNonBlocking) == cudaSuccess &&
        cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming) == cudaSuccess &&
        cudaEventCreateWithFlags(&a.join, cudaEventDisableTiming) == cudaSuccess)
      a.state = 1;
    else
      (void)cudaGetLastError();
  }
  return a.state == 1 ? &a : nullptr;
}
bool aux_fork(AuxStream* a, cudaStream_t st) {
  return a && cudaEventRecord(a->fork, st) == cudaSuccess && cudaStreamWaitEvent(a->s, a->fork, 0) == cudaSuccess;
}
int aux_join(AuxStream* a, cudaStream_t st) {
  cudaError_t e = cudaEventRecord(a->join, a->s);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(st, a->join, 0);
  return e == cudaSuccess ? PERT_OK : (int)e;
}

int check_desc(const PertModelDesc* d) {
  if (!d) return PERT_ERR_BADARG;
  if (d->n_convs < 2 || d->n_convs > PERT_MAX_CONVS || d->n_cat < 1 || d->n_cat > PERT_MAX_CAT) return PERT_ERR_BADARG;
  if (d->H <= 0 || d->F <= 0 || d->k0 < d->F + d->H || d->k0 % 4) return PERT_ERR_BADARG;
  if (!pert_tconv_supported_width(d->H)) return PERT_ERR_UNSUPPORTED;
  return PERT_OK;
}

#define PROBE_START(kid, lay)                                                              \
  do {                                                                                     \
    if (probe && probe->kernel == (kid) && probe->layer == (lay) && probe->ev_start)       \
      cudaEventRecord((cudaEvent_t)probe->ev_start, st);                                   \
  } while (0)
#define PROBE_STOP(kid, lay)                                                               \
  do {                                                                                     \
    if (probe && probe->kernel == (kid) && probe->layer == (lay) && probe->ev_stop)        \
      cudaEventRecord((cudaEvent_t)probe->ev_stop, st);                                    \
  } while (0)

#define TRY(expr)            \
  do {                       \
    int rc__ = (expr);       \
    if (rc__ != 0) return rc__; \
  } while (0)

}  // namespace

extern "C" {

long long pert_model_workspace_bytes(const PertModelDesc* d, long long N, long long E, long long B) {
  if (check_desc(d) || N < 0 || E < 0 || B < 0) return PERT_ERR_BADARG;
  Ws w = carve(d, N, E, B, nullptr);
  return w.total * 4;
}
// Test / debug aid: where a saved activation lives inside the workspace (floats from its start): which = 0 -> the input of
// conv `layer` >= 1, i.e. the post-BatchNorm-ReLU activations [N, H]; which = 1 -> the global head's hidden layer
// relu(global_linear1(.)) [B, H].  Returns the offset or a negative PERT_ERR_*.
long long pert_model_workspace_offset(const PertModelDesc* d, long long N, long long E, long long B, int which,
                                      int layer) {
  if (check_desc(d) || N < 0 || E < 0 || B < 0) return PERT_ERR_BADARG;
  float* base = reinterpret_cast<float*>(4096);     // carve() only does pointer arithmetic
  Ws w = carve(d, N, E, B, base);
  if (which == 0 && layer >= 1 && layer < d->n_convs) return w.x[layer] - base;
  if (which == 1) return w.h1 - base;
  return PERT_ERR_BADARG;
}
long long pert_model_packed_bytes(const PertModelDesc* d) {
  if (check_desc(d)) return PERT_ERR_BADARG;
  Ws w = carve(d, 0, 0, 0, nullptr);
  return w.packed_floats * 4;
}

int pert_model_forward(const PertModelDesc* d, const float* params, float* bn_running, long long* bn_nbt,
                       const float* x, const int64_t* cat_X, const int64_t* entry_id, const float* probs,
                       const float* pnn, const int64_t* batch, long long N, long long E, long long B,
                       const int* rowptr, const int* csr_src, const int* csr_if, const int* csr_rpc, void* workspace,
                       long long workspace_bytes, int training, float dropout_p, long long* rng_state,
                       float* global_pred, float* local_pred, int* status, const PertProbe* probe, void* index_ready,
                       void* stream) {
  TRY(check_desc(d));
  if (!(dropout_p >= 0.f && dropout_p <= 1.f)) return PERT_ERR_BADARG;
  const bool drop = training && dropout_p > 0.f;
  if (drop && !rng_state) return PERT_ERR_BADARG;
  std::lock_guard<std::mutex> issue_lock(engine_mutex());
  if (!params || !x || !cat_X || !entry_id || !probs || !pnn || !batch || !rowptr || !workspace || !global_pred)
    return PERT_ERR_BADARG;
  if (E > 0 && (!csr_src || !csr_if || !csr_rpc)) return PERT_ERR_BADARG;
  float* base = (float*)workspace;
  Ws w = carve(d, N, E, B, base);
  if (workspace_bytes < w.total * 4) return PERT_ERR_BADARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int H = d->H, L = d->n_convs;
  // the input prologue (2.) does not depend on the packed parameters: it runs on the auxiliary stream beside 1.
  AuxStream* ax = aux_stream();
  const bool forked = aux_fork(ax, st);
  cudaStream_t s2 = forked ? ax->s : st;
  // 1. pack parameters (one launch per layer) and build the edge tables of all layers (one grouped launch each <=6)
  {
    SegList S;
    S.count = 0;
    for (int l = 0; l < L; ++l) {
      append_layer_segs(S, d, w, base, l);
      if (S.count + SEGS_PER_LAYER_MAX > SEG_MAX || l == L - 1) {
        k_pack<<<dim3(8, S.count), 256, 0, st>>>(params, base, S);
        S.count = 0;
      }
    }
  }
  {
    SmallGemmBatch gb;
    gb.count = 0;
    for (int l = 0; l < L; ++l) {
      // T_if = if_emb . WeA^T ;  T_rpc = rpc_emb . WeB^T      (B(k,n) = WeA[n,k])
      gb.p[gb.count++] = sg(params + d->off_if, H, 1, w.weA[l], 1, H, nullptr, w.t_if[l], H, d->n_if, H, H);
      gb.p[gb.count++] = sg(params + d->off_rpc, H, 1, w.weB[l], 1, H, nullptr, w.t_rpc[l], H, d->n_rpc, H, H);
      if (gb.count + 2 > SG_MAX || l == L - 1) {
        launch_small(gb, st);
        gb.count = 0;
      }
    }
  }
  // 2. prologue: X0 = [sum_i cat_emb_i[cat_X[:,i]] | x | 0]
  for (int i = 0; i < d->n_cat; ++i)
    TRY(pert_embedding_fwd(params + d->off_cat[i], d->cat_rows[i], cat_X + i, d->n_cat, w.x[0], d->k0, N, H, i > 0,
                           status, s2));
  TRY(pert_copy_cols(x, d->F, w.x[0], d->k0, H, N, s2));
  // graph boundaries of the batch for the tile list (needs only the batch vector): beside the prologue as well
  const bool want_tiles = tiles_enabled() && E > 0 && N > 0 && !pert_tile_fixed_ok(N, E, B, H, d->n_rpc);
  if (want_tiles) TRY(pert_tile_list_bounds(batch, N, B, w.tiles, s2));
  if (forked) TRY(aux_join(ax, st));
  // 3. conv stack
  PertTiles tiles{};
  bool have_tiles = false;
  for (int l = 0; l < L; ++l) {
    const int K = k_of(d, l);
    PROBE_START(3, l);
    TRY(pert_gemm_nt(w.x[l], K, 0, 0, w.w4[l], K, w.b4[l], w.planes[l], H, H, N * (long long)H, N, 4 * H, K, 0, 0, st));
    PROBE_STOP(3, l);
    float* pl = w.planes[l];
    if (l == 0 && index_ready) {      // the graph index was built on another stream: first use is here
      cudaError_t we = cudaStreamWaitEvent(st, (cudaEvent_t)index_ready, 0);
      if (we != cudaSuccess) return (int)we;
    }
    if (l == 0 && want_tiles) {   // graph-aligned tile list (whole graphs per tile), once per batch
      int trc = pert_tile_list_build(batch != nullptr && B > 0, N, E, B, rowptr, H, d->n_rpc, w.tiles, &tiles, st);
      have_tiles = trc == PERT_OK;
      if (!have_tiles && trc != PERT_ERR_UNSUPPORTED) return trc;
    }
    // BatchNorm statistics of out[l] are produced by the conv kernel's epilogue (training, staged tile path)
    int stats_fused = 0;
    double* bn_acc = nullptr;
    if (l + 1 < L && training && bn_fuse_enabled()) {
      bn_acc = (double*)w.bn_part;
      cudaError_t me = cudaMemsetAsync(bn_acc, 0, (size_t)2 * H * sizeof(double), st);
      if (me != cudaSuccess) return (int)me;
    }
    PROBE_START(1, l);
    TRY(pert_tconv_fwd_stats(pl, pl + N * H, pl + 2 * N * H, pl + 3 * N * H, H, rowptr, csr_src, csr_if, csr_rpc,
                             w.t_if[l], w.t_rpc[l], w.out[l], H, w.alpha[l], d->n_rpc, N, E, B, H, bn_acc, &stats_fused,
                             have_tiles ? &tiles : nullptr, st));
    PROBE_STOP(1, l);
    if (l + 1 < L) {
      float* rm = bn_running ? bn_running + (size_t)l * 2 * H : nullptr;
      float* rv = rm ? rm + H : nullptr;
      PROBE_START(6, l);
      TRY(pert_bn_fwd_ex(w.out[l], H, params + d->off_bn_g[l], params + d->off_bn_b[l], rm, rv,
                         (training && bn_nbt) ? bn_nbt + l : nullptr, d->bn_eps, d->bn_momentum, training, 1,
                         w.bn_stats[l], w.bn_stats[l] + H, w.x[l + 1], H, N, H, w.bn_part,
                         pert_bn_workspace_bytes(N, H), stats_fused, drop ? dropout_p : 0.f,
                         drop ? rng_state : nullptr, l, st));
      PROBE_STOP(6, l);
    }
  }
  // 4. local head + weighted add-pool, global head
  TRY(pert_pool_fwd(w.out[L - 1], H, probs, pnn, batch, params + d->off_local_w, params + d->off_local_b, local_pred,
                    w.pool, N, B, H, status, st));
  if (B > 0) {
    const size_t hsm = ((size_t)2 * H * H + (size_t)HEAD_G * 2 * H) * sizeof(float);
    if (hsm > 48 * 1024) {
      cudaError_t he = cudaFuncSetAttribute(k_head_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsm);
      if (he != cudaSuccess) return (int)he;
    }
    k_head_fwd<<<pert_cdiv(B, HEAD_G), HEAD_T, hsm, st>>>(
        w.pool, params + d->off_entry, d->n_entry, entry_id, params + d->off_g1_w, params + d->off_g1_b,
        params + d->off_g2_w, params + d->off_g2_b, w.z, w.h1, global_pred, (int)B, H, status,
        drop ? rng_state : nullptr);
  } else if (drop) {
    k_rng_advance<<<1, 1, 0, st>>>(rng_state);
  }
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

// d_global [B] = dL/d global_pred, d_local [N] or NULL.  grads: flat buffer, same offsets as params, accumulated (+=).
int pert_model_backward(const PertModelDesc* d, const float* params, float* grads, const int64_t* cat_X,
                        const int64_t* entry_id, const float* probs, const float* pnn, const int64_t* batch,
                        long long N, long long E, long long B, const int* rowptr, const int* csr_src,
                        const int* csr_if, const int* csr_rpc, const int* colptr, const int* csc_pos,
                        const int* csc_dst, void* workspace, long long workspace_bytes, int training, float dropout_p,
                        const float* d_global, const float* d_local, const PertProbe* probe, void* stream) {
  TRY(check_desc(d));
  unsigned long long drop_t;
  float drop_scale;
  if (!pert_dropout_params(dropout_p, &drop_t, &drop_scale)) return PERT_ERR_BADARG;
  if (!(training && dropout_p > 0.f)) drop_scale = 1.f;
  std::lock_guard<std::mutex> issue_lock(engine_mutex());
  if (!params || !grads || !cat_X || !entry_id || !probs || !pnn || !batch || !rowptr || !colptr || !workspace ||
      !d_global)
    return PERT_ERR_BADARG;
  float* base = (float*)workspace;
  Ws w = carve(d, N, E, B, base);
  if (workspace_bytes < w.total * 4) return PERT_ERR_BADARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int H = d->H, L = d->n_convs;
  cudaError_t e = cudaMemsetAsync(w.gzero_begin, 0, (size_t)(w.gzero_end - w.gzero_begin) * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  // ---- global head backward
  if (B > 0) {
    const size_t hsm = ((size_t)2 * H * H + (size_t)HEAD_G * 3 * H) * sizeof(float);
    if (hsm > 48 * 1024) {
      cudaError_t he = cudaFuncSetAttribute(k_head_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsm);
      if (he != cudaSuccess) return (int)he;
    }
    k_head_bwd<<<pert_cdiv(B, HEAD_G), HEAD_T, hsm, st>>>(
        d_global, w.z, w.h1, params + d->off_g1_w, params + d->off_g2_w, entry_id, d->n_entry, w.dpool,
        grads + d->off_entry, grads + d->off_g1_w, grads + d->off_g1_b, grads + d->off_g2_w, grads + d->off_g2_b,
        (int)B, H);
  }
  // ---- pool / local head backward: g = dL/d out[L-1], written straight into the skip plane of dplanes
  float* dq = w.dplanes;
  float* dk = dq + N * H;
  float* dv = dk + N * H;
  float* dskip = dv + N * H;
  TRY(pert_pool_bwd(B > 0 ? w.dpool : nullptr, d_local, w.out[L - 1], H, probs, pnn, batch, params + d->off_local_w,
                    dskip, H, grads + d->off_local_w, grads + d->off_local_b, N, B, H, st));
  // ---- edge tables: dWeA = dT_if^T . if_emb ; d if_emb += dT_if . WeA   (and the rpc halves), all layers grouped.
  // They depend only on the conv backward passes (dT tables), so they run on the auxiliary stream beside the conv-0
  // GEMMs and the embedding scatters; the unpack at the end waits for them.
  auto table_grads = [&](cudaStream_t ts) {
    SmallGemmBatch gb;
    gb.count = 0;
    for (int l = 0; l < L; ++l) {
      int ks_if = d->n_if >= 512 ? 8 : 1, ks_rpc = 1;
      gb.p[gb.count++] = sg(w.dt_if[l], 1, H, params + d->off_if, H, 1, nullptr, w.dweA[l], H, H, H, d->n_if, 0, 1, ks_if);
      gb.p[gb.count++] = sg(w.dt_rpc[l], 1, H, params + d->off_rpc, H, 1, nullptr, w.dweB[l], H, H, H, d->n_rpc, 0, 1, ks_rpc);
      // every layer adds into the same embedding-gradient rows: atomic accumulation, all layers in one launch
      gb.p[gb.count] = sg(w.dt_if[l], H, 1, w.weA[l], H, 1, nullptr, grads + d->off_if, H, d->n_if, H, H, 0, 1);
      gb.p[gb.count++].atomic = 1;
      gb.p[gb.count] = sg(w.dt_rpc[l], H, 1, w.weB[l], H, 1, nullptr, grads + d->off_rpc, H, d->n_rpc, H, H, 0, 1);
      gb.p[gb.count++].atomic = 1;
      if (gb.count + 4 > SG_MAX || l == 0 + L - 1) {
        launch_small(gb, ts);
        gb.count = 0;
      }
    }
  };
  AuxStream* ax = aux_stream();
  bool forked = false;
  PertTiles tiles{};            // the list forward built for this batch (same geometry: a pure function of the sizes)
  const bool have_tiles = tiles_enabled() && E > 0 && !pert_tile_fixed_ok(N, E, B, H, d->n_rpc) &&
                          pert_tile_list_view(N, E, B, H, d->n_rpc, w.tiles, &tiles) == PERT_OK;
  for (int l = L - 1; l >= 0; --l) {
    const int K = k_of(d, l);
    float* pl = w.planes[l];
    PROBE_START(2, l);
    TRY(pert_tconv_bwd_tiles(dskip, H, pl, pl + N * H, pl + 2 * N * H, H, rowptr, csr_src, csr_if, csr_rpc, colptr,
                             csc_pos, csc_dst, w.t_if[l], w.t_rpc[l], w.alpha[l], dq, dk, dv, H, w.dsp, w.rpc_ws,
                             w.dt_if[l], w.dt_rpc[l], d->n_rpc, N, E, B, H, have_tiles ? &tiles : nullptr, st));
    PROBE_STOP(2, l);
    if (l == 0) {                       // every dT table is complete now
      forked = aux_fork(ax, st);
      if (forked) table_grads(ax->s);
    }
    // weight / bias gradients of the fused node linear (packed), data gradient
    PROBE_START(4, l);
    TRY(pert_gemm_tn(w.dplanes, H, H, N * (long long)H, w.x[l], K, 0, 0, w.dw4[l], K, w.db4[l], N, 4 * H, K, st));
    PROBE_STOP(4, l);
    PROBE_START(5, l);
    // (conv 0: only the embedding columns [0, H) of dX0 are needed -- x and the pad columns carry no parameters)
    TRY(pert_gemm_nt(w.dplanes, H, H, N * (long long)H, w.w4t[l], 4 * H, nullptr, w.dx, K, 0, 0, N, l == 0 ? H : K, 4 * H,
                     0, 0, st));
    PROBE_STOP(5, l);
    if (l > 0) {
      // BN(+ReLU) backward of layer l-1: dx (grad wrt x[l]) -> g of conv l-1, into the skip plane
      // (with dropout, x[l] is the post-dropout output: x[l] > 0 <=> kept and active; dz = dx * scale there)
      TRY(pert_bn_bwd_ex(w.dx, K, w.x[l], H, w.out[l - 1], H, w.bn_stats[l - 1], w.bn_stats[l - 1] + H,
                         params + d->off_bn_g[l - 1], 1, training, drop_scale, dskip, H, grads + d->off_bn_g[l - 1],
                         grads + d->off_bn_b[l - 1], w.sums, N, H, st));
    }
  }
  if (forked) TRY(aux_join(ax, st));
  else table_grads(st);
  // ---- categorical embedding gradients from dX0[:, 0:H] (auxiliary stream) beside the gradient unpack (main stream)
  const bool forked2 = aux_fork(ax, st);
  for (int i = 0; i < d->n_cat; ++i)
    TRY(pert_embedding_bwd(w.dx, d->k0, cat_X + i, d->n_cat, grads + d->off_cat[i], d->cat_rows[i], N, H,
                           forked2 ? ax->s : st));
  {
    SegList S;
    S.count = 0;
    for (int l = 0; l < L; ++l) {
      append_layer_grad_segs(S, d, w, base, l);
      if (S.count + SEGS_PER_LAYER_MAX > SEG_MAX || l == L - 1) {
        k_unpack<<<dim3(8, S.count), 256, 0, st>>>(grads, base, S);
        S.count = 0;
      }
    }
  }
  if (forked2) TRY(aux_join(ax, st));
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

}  // extern "C"
