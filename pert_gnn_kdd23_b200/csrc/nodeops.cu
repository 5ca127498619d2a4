// Node-/graph-level pieces of the hot path around the fused conv (all HBM-bound elementwise / reduction work):
//   embedding gather / scatter-add           reference model.py:87-97,108  (nn.Embedding fwd / dense bwd)
//   feature concat                           model.py:90
//   BatchNorm1d (+ReLU) fwd / bwd            model.py:101-102 (training: batch stats, eps 1e-5, momentum 0.1)
//   local head + prob-weighted add-pool      model.py:105-107 (local_linear, x*probs/num_nodes, global_add_pool)
//   pinball loss, Adam                       pert_gnn.py:191-193,245-247
#include "common.cuh"
#include <type_traits>

namespace {

// ---------------------------------------------------------------- embeddings
// out[n, 0:H] (+)= table[ids[n*id_stride], :]
__global__ void k_embedding_fwd(const float* __restrict__ table, int n_rows, const int64_t* __restrict__ ids,
                                int id_stride, float* __restrict__ out, int ld_out, long long N, int H,
                                int accumulate, int* status) {
  const int vec_per_row = H >> 2;
  long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= N * vec_per_row) return;
  long long n = id / vec_per_row;
  int c = (int)(id % vec_per_row) * 4;
  int64_t r = ids[n * id_stride];
  if (r < 0 || r >= n_rows) {
    if (status) atomicExch(status, PERT_ERR_RANGE);
    r = 0;
  }
  float4 v = ldg4(table + (size_t)r * H + c);
  float* o = out + (size_t)n * ld_out + c;
  if (accumulate) v = f4add(v, ld4(o));
  st4(o, v);
}

// dtable[ids[n*id_stride], :] += dy[n, 0:H]      (REDG.128; nn.Embedding dense backward)
// One thread owns one float4 column of EB_RUN consecutive rows and merges equal ids before the atomic: the stage nodes
// of a microservice are consecutive in a PERT graph (misc.py:238-250: 2c+1 nodes per caller share cat_X), so real
// batches send runs of rows to the same table row.
constexpr int EB_RUN = 8;
__global__ void k_embedding_bwd(const float* __restrict__ dy, int ld_dy, const int64_t* __restrict__ ids,
                                int id_stride, float* __restrict__ dtable, int n_rows, long long N, int H) {
  const int vec_per_row = H >> 2;
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long chunks = (N + EB_RUN - 1) / EB_RUN;
  if (id >= chunks * vec_per_row) return;
  const long long n0 = (id / vec_per_row) * EB_RUN;
  const int c = (int)(id % vec_per_row) * 4;
  int64_t cur = -1;
  float4 acc = f4zero();
#pragma unroll
  for (int k = 0; k < EB_RUN; ++k) {
    const long long n = n0 + k;
    if (n >= N) break;
    const int64_t r = ids[n * id_stride];
    if (r != cur) {
      if (cur >= 0 && cur < n_rows) red4(dtable + (size_t)cur * H + c, acc);
      cur = r;
      acc = f4zero();
    }
    acc = f4add(acc, ldg4(dy + (size_t)n * ld_dy + c));
  }
  if (cur >= 0 && cur < n_rows) red4(dtable + (size_t)cur * H + c, acc);
}

// out[n, col0 : col0+F] = x[n, 0:F]; out[n, col0+F : ld_out) = 0
__global__ void k_copy_cols(const float* __restrict__ x, int F, float* __restrict__ out, int ld_out, int col0,
                            long long N) {
  const int w = ld_out - col0;
  long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= N * w) return;
  long long n = id / w;
  int c = (int)(id % w);
  out[(size_t)n * ld_out + col0 + c] = (c < F) ? x[(size_t)n * F + c] : 0.f;
}

// ---------------------------------------------------------------- batch norm
constexpr int BN_ROWS = 128;      // rows per CTA chunk (forward statistics)
constexpr int BN_BWD_ROWS = 64;   // rows per CTA (backward reductions: atomics, so the chunk count is free)

// per-chunk (mean, M2) with a two-pass centred sum in fp32; the chunks are combined in double precision:
// acc[c] += n_b mean_b,  acc[H + c] += M2_b + n_b mean_b^2  (fp64 atomics; sum and sum of squares of fp32 data are
// exact enough in fp64 that  M2 = S2 - S1^2 / N  has no cancellation problem), so no finalize kernel is needed --
// k_bn_apply derives mean / rstd from acc in its prologue.
__global__ void __launch_bounds__(256) k_bn_partial(const float* __restrict__ x, int ld, long long N, int H,
                                                     double* __restrict__ acc /*[2][H], zeroed*/) {
  extern __shared__ float sm[];  // [rl][H] scratch, then mean[H]
  const int vpr = H >> 2;              // float4 lanes per row
  const int rl_n = blockDim.x / vpr;   // row lanes
  const int cl = threadIdx.x % vpr, rl = threadIdx.x / vpr;
  const long long r0 = (long long)blockIdx.x * BN_ROWS;
  const int rows = (int)min((long long)BN_ROWS, N - r0);
  float* s_red = sm;             // [rl_n][H]
  float* s_mean = sm + rl_n * H; // [H]
  float4 s = f4zero();
  if (rl < rl_n)
    for (int rb = rl; rb < rows; rb += 8 * rl_n) {   // 8 independent row loads in flight per thread
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int r = rb + u * rl_n;
        v[u] = (r < rows) ? ldg4(x + (size_t)(r0 + r) * ld + cl * 4) : f4zero();
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) s = f4add(s, v[u]);
    }
  if (rl < rl_n) st4(s_red + rl * H + cl * 4, s);
  __syncthreads();
  if (threadIdx.x < H) {
    float t = 0.f;
    for (int i = 0; i < rl_n; ++i) t += s_red[i * H + threadIdx.x];
    s_mean[threadIdx.x] = t / (float)rows;
  }
  __syncthreads();
  float4 mu = (rl < rl_n) ? ld4(s_mean + cl * 4) : f4zero();
  float4 q = f4zero();
  if (rl < rl_n)
    for (int rb = rl; rb < rows; rb += 8 * rl_n) {
      float4 vv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int r = rb + u * rl_n;
        vv[u] = (r < rows) ? ldg4(x + (size_t)(r0 + r) * ld + cl * 4) : mu;   // mu => contributes 0
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float4 v = vv[u];
        float dx = v.x - mu.x, dy = v.y - mu.y, dz = v.z - mu.z, dw = v.w - mu.w;
        q.x = fmaf(dx, dx, q.x); q.y = fmaf(dy, dy, q.y); q.z = fmaf(dz, dz, q.z); q.w = fmaf(dw, dw, q.w);
      }
    }
  __syncthreads();
  if (rl < rl_n) st4(s_red + rl * H + cl * 4, q);
  __syncthreads();
  if (threadIdx.x < H) {
    float t = 0.f;
    for (int i = 0; i < rl_n; ++i) t += s_red[i * H + threadIdx.x];
    const double m = (double)s_mean[threadIdx.x], n = (double)rows;
    atomicAdd(acc + threadIdx.x, n * m);
    atomicAdd(acc + H + threadIdx.x, (double)t + n * m * m);
  }
}

// eval mode: mean = running_mean, rstd = 1/sqrt(running_var + eps)
__global__ void k_bn_eval_stats(const float* __restrict__ rm, const float* __restrict__ rv, float eps, int H,
                                float* __restrict__ mean, float* __restrict__ rstd) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= H) return;
  mean[c] = rm[c];
  rstd[c] = 1.0f / sqrtf(rv[c] + eps);
}

// y = (relu)((x - mean) rstd gamma + beta).  acc != null (training): mean / rstd come from the fp64 sums of
// k_bn_partial (every CTA derives them in its prologue; CTA 0 also stores them for the backward pass and updates the
// running statistics); acc == null (eval): mean / rstd arrays are read.
// DROP (training dropout, p > 0): y *= keep * scale in the same pass, keep from dropout_words(seed, offset, layer, j)
// with j = the float4 index n * H/4 + c/4 -- exactly `id` below.  DROP = false is the plain kernel, no Philox in it.
template <bool DROP>
__global__ void __launch_bounds__(256) k_bn_apply(const float* __restrict__ x, int ld_x, float* __restrict__ mean,
                                                   float* __restrict__ rstd, const float* __restrict__ gamma,
                                                   const float* __restrict__ beta, float* __restrict__ y, int ld_y,
                                                   long long N, int H, int relu, const double* __restrict__ acc,
                                                   float eps, float momentum, float* running_mean,
                                                   float* running_var, long long* num_batches_tracked,
                                                   PertDropout dr) {
  extern __shared__ float s_par[];   // mean | rstd | gamma | beta
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float mu, rs;
    if (acc) {
      const double n = (double)N;
      const double m = acc[c] / n;
      double m2 = acc[H + c] - n * m * m;
      if (m2 < 0.0) m2 = 0.0;
      const double var = m2 / n;       // biased, used to normalise
      mu = (float)m;
      rs = (float)(1.0 / sqrt(var + (double)eps));
      if (blockIdx.x == 0) {
        mean[c] = mu;
        rstd[c] = rs;
        if (running_mean) {
          const double unbiased = (N > 1) ? m2 / (n - 1.0) : var;
          running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mu;
          running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
        }
        if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;
      }
    } else {
      mu = mean[c];
      rs = rstd[c];
    }
    s_par[c] = mu;
    s_par[H + c] = rs;
    s_par[2 * H + c] = gamma[c];
    s_par[3 * H + c] = beta[c];
  }
  __syncthreads();
  unsigned long long seed = 0, offset = 0;
  if (DROP) {
    seed = (unsigned long long)dr.rng[0];
    offset = (unsigned long long)dr.rng[1];
  }
  const int vpr = H >> 2;
  const long long total = N * vpr;
  for (long long id0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; id0 < total;
       id0 += 4LL * gridDim.x * blockDim.x) {
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {       // 4 independent row loads in flight
      const long long id = id0 + (long long)u * gridDim.x * blockDim.x;
      v[u] = id < total ? ldg4(x + (size_t)(id / vpr) * ld_x + (int)(id % vpr) * 4) : f4zero();
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long id = id0 + (long long)u * gridDim.x * blockDim.x;
      if (id >= total) break;
      const int c = (int)(id % vpr) * 4;
      const float4 mu = ld4(s_par + c), rs = ld4(s_par + H + c), ga = ld4(s_par + 2 * H + c), be = ld4(s_par + 3 * H + c);
      float4 o;
      o.x = fmaf((v[u].x - mu.x) * rs.x, ga.x, be.x);
      o.y = fmaf((v[u].y - mu.y) * rs.y, ga.y, be.y);
      o.z = fmaf((v[u].z - mu.z) * rs.z, ga.z, be.z);
      o.w = fmaf((v[u].w - mu.w) * rs.w, ga.w, be.w);
      if (relu) o = f4max(o, f4zero());
      if (DROP) {
        const uint4 wd = dropout_words(seed, offset, dr.layer, (unsigned long long)id);
        o.x = wd.x >= dr.t ? o.x * dr.scale : 0.f;
        o.y = wd.y >= dr.t ? o.y * dr.scale : 0.f;
        o.z = wd.z >= dr.t ? o.z * dr.scale : 0.f;
        o.w = wd.w >= dr.t ? o.w * dr.scale : 0.f;
      }
      st4(y + (size_t)(id / vpr) * ld_y + c, o);
    }
  }
}

// sums[0:H] += sum_n dz,  sums[H:2H] += sum_n dz*xhat   with dz = dy * (y > 0 if relu) * scale.
// scale = the dropout scale 1/(1-p) of the forward (1 without dropout: then dz is dy bit for bit): y = relu(.) keep scale,
// so for scale >= 1, y > 0 <=> (kept and relu active) and the saved output is the only mask needed.  SCALED = false: the
// kernel without the multiply (its register budget, and so its occupancy, is that of the plain kernel).
template <bool SCALED>
__global__ void __launch_bounds__(256) k_bn_bwd_reduce(const float* __restrict__ dy, int ld_dy,
                                                        const float* __restrict__ y, int ld_y,
                                                        const float* __restrict__ x, int ld_x,
                                                        const float* __restrict__ mean,
                                                        const float* __restrict__ rstd, long long N, int H, int relu,
                                                        float scale, float* __restrict__ sums) {
  extern __shared__ float sm[];  // [rl_n][2H]
  const int vpr = H >> 2;
  const int rl_n = blockDim.x / vpr;
  const int cl = threadIdx.x % vpr, rl = threadIdx.x / vpr;
  const long long r0 = (long long)blockIdx.x * BN_BWD_ROWS;
  const int rows = (int)min((long long)BN_BWD_ROWS, N - r0);
  float4 s1 = f4zero(), s2 = f4zero();
  if (rl < rl_n) {
    const float4 mu = ldg4(mean + cl * 4), rs = ldg4(rstd + cl * 4);
    for (int rb = rl; rb < rows; rb += 4 * rl_n) {   // 4 rows x 3 operands = 12 independent loads in flight
      float4 gg[4], yy4[4], vv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int r = rb + u * rl_n;
        const bool ok = r < rows;
        gg[u] = ok ? ldg4(dy + (size_t)(r0 + r) * ld_dy + cl * 4) : f4zero();
        yy4[u] = (ok && relu) ? ldg4(y + (size_t)(r0 + r) * ld_y + cl * 4) : make_float4(1.f, 1.f, 1.f, 1.f);
        vv[u] = ok ? ldg4(x + (size_t)(r0 + r) * ld_x + cl * 4) : mu;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float4 g = gg[u];
        const float4 yy = yy4[u], v = vv[u];
        g.x = yy.x > 0.f ? g.x : 0.f; g.y = yy.y > 0.f ? g.y : 0.f;
        g.z = yy.z > 0.f ? g.z : 0.f; g.w = yy.w > 0.f ? g.w : 0.f;
        if (SCALED) g = f4scale(scale, g);
        s1 = f4add(s1, g);
        s2.x = fmaf(g.x, (v.x - mu.x) * rs.x, s2.x); s2.y = fmaf(g.y, (v.y - mu.y) * rs.y, s2.y);
        s2.z = fmaf(g.z, (v.z - mu.z) * rs.z, s2.z); s2.w = fmaf(g.w, (v.w - mu.w) * rs.w, s2.w);
      }
    }
    st4(sm + rl * 2 * H + cl * 4, s1);
    st4(sm + rl * 2 * H + H + cl * 4, s2);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * H; c += blockDim.x) {
    float t = 0.f;
    for (int i = 0; i < rl_n; ++i) t += sm[i * 2 * H + c];
    atomicAdd(sums + c, t);
  }
}

// training: dx = gamma*rstd*(dz - sum_dz/N - xhat*sum_dzxhat/N); eval: dx = gamma*rstd*dz
__global__ void k_bn_bwd_apply(const float* __restrict__ dy, int ld_dy, const float* __restrict__ y, int ld_y,
                               const float* __restrict__ x, int ld_x, const float* __restrict__ mean,
                               const float* __restrict__ rstd, const float* __restrict__ gamma,
                               const float* __restrict__ sums, float* __restrict__ dx, int ld_dx, long long N, int H,
                               int relu, float scale, int training, float* dgamma, float* dbeta) {
  const int vpr = H >> 2;
  long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x == 0)  // parameter grads accumulate (+=) like autograd
    for (int c = threadIdx.x; c < H; c += blockDim.x) {
      if (dbeta) dbeta[c] += sums[c];
      if (dgamma) dgamma[c] += sums[H + c];
    }
  if (id >= N * vpr) return;
  long long n = id / vpr;
  int c = (int)(id % vpr) * 4;
  float4 g = ldg4(dy + (size_t)n * ld_dy + c);
  if (relu) {
    float4 yy = ldg4(y + (size_t)n * ld_y + c);
    g.x = yy.x > 0.f ? g.x : 0.f; g.y = yy.y > 0.f ? g.y : 0.f;
    g.z = yy.z > 0.f ? g.z : 0.f; g.w = yy.w > 0.f ? g.w : 0.f;
    if (scale != 1.f) g = f4scale(scale, g);     // dropout (see k_bn_bwd_reduce)
  }
  const float4 rs = ldg4(rstd + c), ga = ldg4(gamma + c);
  float4 o;
  if (training) {
    const float invn = 1.0f / (float)N;
    const float4 v = ldg4(x + (size_t)n * ld_x + c), mu = ldg4(mean + c);
    const float4 a = ldg4(sums + c), b = ldg4(sums + H + c);
    o.x = ga.x * rs.x * (g.x - a.x * invn - (v.x - mu.x) * rs.x * b.x * invn);
    o.y = ga.y * rs.y * (g.y - a.y * invn - (v.y - mu.y) * rs.y * b.y * invn);
    o.z = ga.z * rs.z * (g.z - a.z * invn - (v.z - mu.z) * rs.z * b.z * invn);
    o.w = ga.w * rs.w * (g.w - a.w * invn - (v.w - mu.w) * rs.w * b.w * invn);
  } else {
    o = make_float4(ga.x * rs.x * g.x, ga.y * rs.y * g.y, ga.z * rs.z * g.z, ga.w * rs.w * g.w);
  }
  st4(dx + (size_t)n * ld_dx + c, o);
}

// keep[n, c] = 1 iff unit (n, c) of BatchNorm `layer` survives dropout (the mask k_bn_apply<true> applies)
__global__ void k_dropout_mask(unsigned long long seed, unsigned long long offset, int layer, long long N, int H,
                               unsigned long long t, uint8_t* __restrict__ keep) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N * (H >> 2)) return;
  const uint4 wd = dropout_words(seed, offset, layer, (unsigned long long)j);
  uchar4 k;
  k.x = wd.x >= t; k.y = wd.y >= t; k.z = wd.z >= t; k.w = wd.w >= t;
  reinterpret_cast<uchar4*>(keep)[j] = k;
}

// ---------------------------------------------------------------- local head + weighted add-pool
constexpr int POOL_ROWS = 8;  // consecutive rows per lane group (run-length pre-aggregation of the pool atomics)

template <int LPR, int VPL>
__global__ void __launch_bounds__(256) k_pool_fwd(const float* __restrict__ x, int ld, const float* __restrict__ probs,
                                                   const float* __restrict__ pnn, const int64_t* __restrict__ batch,
                                                   const float* __restrict__ w_local, const float* __restrict__ b_local,
                                                   float* __restrict__ local, float* __restrict__ pool, long long N,
                                                   int B, int* status) {
  constexpr int H = 4 * LPR * VPL;
  const int lane = threadIdx.x & 31, lig = lane % LPR, grp = lane / LPR;
  const unsigned gmask = (LPR == 32) ? 0xffffffffu : (((1u << LPR) - 1u) << (grp * LPR));
  const long long gid = (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / LPR) + grp;
  const long long r0 = gid * POOL_ROWS;
  if (r0 >= N) return;
  float4 w[VPL], acc[VPL];
#pragma unroll
  for (int u = 0; u < VPL; ++u) {
    w[u] = w_local ? ldg4(w_local + lig * 4 + u * LPR * 4) : f4zero();
    acc[u] = f4zero();
  }
  const float bl = b_local ? __ldg(b_local) : 0.f;
  long long cur = -1;
  const int rows = (int)min((long long)POOL_ROWS, N - r0);
  for (int r = 0; r < rows; ++r) {
    const long long n = r0 + r;
    float4 v[VPL];
    float d = 0.f;
#pragma unroll
    for (int u = 0; u < VPL; ++u) {
      v[u] = ldg4(x + (size_t)n * ld + lig * 4 + u * LPR * 4);
      d += f4dot(v[u], w[u]);
    }
    if (local) {
      d = group_sum<LPR>(d, gmask);
      if (lig == 0) local[n] = d + bl;
    }
    long long g = batch[n];
    if (g < 0 || g >= B) {
      if (status) atomicExch(status, PERT_ERR_RANGE);
      continue;
    }
    if (g != cur) {
      if (cur >= 0) {
#pragma unroll
        for (int u = 0; u < VPL; ++u) red4(pool + (size_t)cur * H + lig * 4 + u * LPR * 4, acc[u]);
      }
#pragma unroll
      for (int u = 0; u < VPL; ++u) acc[u] = f4zero();
      cur = g;
    }
    const float pr = __ldg(probs + n), nn = __ldg(pnn + n);
#pragma unroll
    for (int u = 0; u < VPL; ++u) {
      // reference order: (x * p) / n  (model.py:106) -- keep the two roundings
      acc[u].x += (v[u].x * pr) / nn;
      acc[u].y += (v[u].y * pr) / nn;
      acc[u].z += (v[u].z * pr) / nn;
      acc[u].w += (v[u].w * pr) / nn;
    }
  }
  if (cur >= 0) {
#pragma unroll
    for (int u = 0; u < VPL; ++u) red4(pool + (size_t)cur * H + lig * 4 + u * LPR * 4, acc[u]);
  }
}

// dx[n] = dlocal[n]*w_local + dpool[batch[n]] * probs[n]/pnn[n];  dw_local += sum dlocal[n]*x[n]; db_local += sum dlocal
template <int LPR, int VPL>
__global__ void __launch_bounds__(256) k_pool_bwd(const float* __restrict__ dpool, const float* __restrict__ dlocal,
                                                   const float* __restrict__ x, int ld,
                                                   const float* __restrict__ probs, const float* __restrict__ pnn,
                                                   const int64_t* __restrict__ batch,
                                                   const float* __restrict__ w_local, float* __restrict__ dx,
                                                   int ld_dx, float* __restrict__ dw_local,
                                                   float* __restrict__ db_local, long long N, int B) {
  constexpr int H = 4 * LPR * VPL;
  __shared__ float s_dw[H];
  __shared__ float s_db;
  const bool has_local = dlocal != nullptr;
  if (has_local) {
    for (int c = threadIdx.x; c < H; c += blockDim.x) s_dw[c] = 0.f;
    if (threadIdx.x == 0) s_db = 0.f;
    __syncthreads();
  }
  const int lane = threadIdx.x & 31, lig = lane % LPR, grp = lane / LPR;
  const long long gid = (((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / LPR) + grp;
  const long long r0 = gid * POOL_ROWS;
  float4 w[VPL], dw[VPL];
  float db = 0.f;
#pragma unroll
  for (int u = 0; u < VPL; ++u) {
    w[u] = (has_local && w_local) ? ldg4(w_local + lig * 4 + u * LPR * 4) : f4zero();
    dw[u] = f4zero();
  }
  if (r0 < N) {
    const int rows = (int)min((long long)POOL_ROWS, N - r0);
    for (int r = 0; r < rows; ++r) {
      const long long n = r0 + r;
      const long long g = batch[n];
      const float sc = __ldg(probs + n) / __ldg(pnn + n);
      const float dl = has_local ? __ldg(dlocal + n) : 0.f;
      db += dl;
#pragma unroll
      for (int u = 0; u < VPL; ++u) {
        float4 o = f4zero();
        if (dpool && g >= 0 && g < B) o = f4scale(sc, ldg4(dpool + (size_t)g * H + lig * 4 + u * LPR * 4));
        if (has_local) {
          o = f4fma(dl, w[u], o);
          dw[u] = f4fma(dl, ldg4(x + (size_t)n * ld + lig * 4 + u * LPR * 4), dw[u]);
        }
        st4(dx + (size_t)n * ld_dx + lig * 4 + u * LPR * 4, o);
      }
    }
  }
  if (has_local) {
#pragma unroll
    for (int u = 0; u < VPL; ++u) {
      float* p = s_dw + lig * 4 + u * LPR * 4;
      atomicAdd(p + 0, dw[u].x); atomicAdd(p + 1, dw[u].y); atomicAdd(p + 2, dw[u].z); atomicAdd(p + 3, dw[u].w);
    }
    if (lig == 0) atomicAdd(&s_db, db);
    __syncthreads();
    if (dw_local)
      for (int c = threadIdx.x; c < H; c += blockDim.x) atomicAdd(dw_local + c, s_dw[c]);
    if (db_local && threadIdx.x == 0) atomicAdd(db_local, s_db);
  }
}

template <typename F>
int dispatch_h(int H, F&& f) {
  switch (H) {
    case 4: return f(std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{});
    case 8: return f(std::integral_constant<int, 2>{}, std::integral_constant<int, 1>{});
    case 16: return f(std::integral_constant<int, 4>{}, std::integral_constant<int, 1>{});
    case 32: return f(std::integral_constant<int, 8>{}, std::integral_constant<int, 1>{});
    case 64: return f(std::integral_constant<int, 16>{}, std::integral_constant<int, 1>{});
    case 96: return f(std::integral_constant<int, 8>{}, std::integral_constant<int, 3>{});
    case 128: return f(std::integral_constant<int, 32>{}, std::integral_constant<int, 1>{});
    case 192: return f(std::integral_constant<int, 16>{}, std::integral_constant<int, 3>{});
    case 256: return f(std::integral_constant<int, 32>{}, std::integral_constant<int, 2>{});
    default: return PERT_ERR_UNSUPPORTED;
  }
}

// ---------------------------------------------------------------- small elementwise
__global__ void k_relu_bwd(const float* __restrict__ y, float* __restrict__ dy, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && !(y[i] > 0.f)) dy[i] = 0.f;
}

// pinball loss (pert_gnn.py:191-193): loss = mean(max(tau*e, (tau-1)*e)), e = y - yhat; dyhat = dloss/dyhat
__global__ void k_pinball(const int64_t* __restrict__ y, const float* __restrict__ yhat, float tau, int B,
                          float grad_scale, float* __restrict__ loss, float* __restrict__ dyhat) {
  __shared__ float red[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < B; i += blockDim.x) {
    float e = (float)y[i] - yhat[i];
    float a = tau * e, b = (tau - 1.f) * e;
    s += fmaxf(a, b);
    if (dyhat) {
      // torch.maximum backward: ties split the gradient evenly
      float d = (a > b) ? -tau : ((a < b) ? (1.f - tau) : 0.5f * (1.f - 2.f * tau));
      dyhat[i] = grad_scale * d / (float)B;
    }
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0 && loss) *loss = t / (float)B;
  }
}

// torch.optim.Adam (amsgrad=False, maximize=False) over one flat buffer
__global__ void k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                       float* __restrict__ v, long long n, float lr, float b1, float b2, float eps, float wd,
                       float bc1, float bc2_sqrt, float grad_scale) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float gi = g[i] * grad_scale;
  float pi = p[i];
  if (wd != 0.f) gi = fmaf(wd, pi, gi);
  float mi = m[i] + (1.f - b1) * (gi - m[i]);             // lerp, as torch's foreach path
  float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] = pi - (lr / bc1) * (mi / denom);
}

inline bool al16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }

}  // namespace


// ---- eval metrics (reference pert_gnn.py:284-289, :249): block sums in double, one atomic per block and metric
__global__ void __launch_bounds__(256) k_eval_metrics(const int64_t* __restrict__ y, const float* __restrict__ yhat,
                                                      float tau, int B, double* __restrict__ acc) {
  double mae = 0.0, mape = 0.0, q = 0.0;
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const float yt = (float)y[b];                 // y.float() / int64 -> float32 promotion of the reference
    const float e = yt - yhat[b];
    const float ae = fabsf(yhat[b] - yt);
    mae += (double)ae;
    mape += (double)(ae / yt);
    q += (double)fmaxf(tau * e, (tau - 1.0f) * e);
  }
  __shared__ double red[3][8];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    mae += __shfl_xor_sync(0xffffffffu, mae, off);
    mape += __shfl_xor_sync(0xffffffffu, mape, off);
    q += __shfl_xor_sync(0xffffffffu, q, off);
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { red[0][w] = mae; red[1][w] = mape; red[2][w] = q; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
    atomicAdd(acc + threadIdx.x, t);
  }
}

extern "C" {

int pert_embedding_fwd(const float* table, int n_rows, const int64_t* ids, int id_stride, float* out, int ld_out,
                       long long N, int H, int accumulate, int* status, void* stream) {
  if (N < 0 || H <= 0 || H % 4 || ld_out % 4 || !table || !out || n_rows <= 0 || !al16(table) || !al16(out))
    return PERT_ERR_BADARG;
  if (N == 0) return PERT_OK;
  long long total = N * (H / 4);
  k_embedding_fwd<<<pert_cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(table, n_rows, ids, id_stride, out,
                                                                         ld_out, N, H, accumulate, status);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_embedding_bwd(const float* dy, int ld_dy, const int64_t* ids, int id_stride, float* dtable, int n_rows,
                       long long N, int H, void* stream) {
  if (N < 0 || H <= 0 || H % 4 || ld_dy % 4 || !dy || !dtable || !al16(dy) || !al16(dtable)) return PERT_ERR_BADARG;
  if (N == 0) return PERT_OK;
  long long total = ((N + EB_RUN - 1) / EB_RUN) * (H / 4);
  k_embedding_bwd<<<pert_cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(dy, ld_dy, ids, id_stride, dtable,
                                                                         n_rows, N, H);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_copy_cols(const float* x, int F, float* out, int ld_out, int col0, long long N, void* stream) {
  if (N < 0 || F < 0 || !out || col0 < 0 || col0 + F > ld_out) return PERT_ERR_BADARG;
  if (N == 0 || ld_out == col0) return PERT_OK;
  long long total = N * (ld_out - col0);
  k_copy_cols<<<pert_cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x, F, out, ld_out, col0, N);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

long long pert_bn_workspace_bytes(long long N, int H) {
  (void)N;
  return 2LL * H * 8 + 64;   // fp64 (sum, sum of squares) per column
}

// training != 0: batch statistics (and running-stat update when running_* given); else running statistics.
// Writes mean[H], rstd[H] (saved for backward) and y = (relu)(xhat*gamma + beta).
int pert_bn_fwd(const float* x, int ld_x, const float* gamma, const float* beta, float* running_mean,
                float* running_var, long long* num_batches_tracked, float eps, float momentum, int training,
                int relu, float* mean, float* rstd, float* y, int ld_y, long long N, int H, void* workspace,
                long long workspace_bytes, void* stream) {
  return pert_bn_fwd_ex(x, ld_x, gamma, beta, running_mean, running_var, num_batches_tracked, eps, momentum, training,
                        relu, mean, rstd, y, ld_y, N, H, workspace, workspace_bytes, 0, 0.f, nullptr, 0, stream);
}

int pert_dropout_mask(long long seed, long long offset, int layer, long long N, int H, float p, uint8_t* keep,
                      void* stream) {
  unsigned long long t;
  float scale;
  if (!pert_dropout_params(p, &t, &scale)) return PERT_ERR_BADARG;
  if (N < 0 || H <= 0 || H % 4 || !keep || ((uintptr_t)keep & 3)) return PERT_ERR_BADARG;
  if (N == 0) return PERT_OK;
  k_dropout_mask<<<pert_cdiv(N * (H / 4), 256), 256, 0, (cudaStream_t)stream>>>(
      (unsigned long long)seed, (unsigned long long)offset, layer, N, H, t, keep);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

}  // extern "C"

// stats_ready != 0 (training): the fp64 column sums / sums of squares already sit in `workspace` (written by the producer
// of x, csrc/tconv_tile.cu) -- only the apply pass runs.
// training with dropout_p > 0: y = relu(bn(x)) * keep / (1 - dropout_p), keep from the device (seed, offset) at
// rng_state and the BatchNorm index `layer` (see dropout_words); rng_state is only read.  Otherwise dropout is off.
int pert_bn_fwd_ex(const float* x, int ld_x, const float* gamma, const float* beta, float* running_mean,
                   float* running_var, long long* num_batches_tracked, float eps, float momentum, int training,
                   int relu, float* mean, float* rstd, float* y, int ld_y, long long N, int H, void* workspace,
                   long long workspace_bytes, int stats_ready, float dropout_p, const long long* rng_state, int layer,
                   void* stream) {
  if (N < 0 || H <= 0 || H % 4 || H > 1024 || ld_x % 4 || ld_y % 4 || !x || !gamma || !beta || !mean || !rstd || !y)
    return PERT_ERR_BADARG;
  if (!al16(x) || !al16(gamma) || !al16(beta) || !al16(mean) || !al16(rstd) || !al16(y)) return PERT_ERR_BADARG;
  PertDropout dr{rng_state, 0, 1.f, layer};
  if (!pert_dropout_params(dropout_p, &dr.t, &dr.scale)) return PERT_ERR_BADARG;
  const bool drop = training && dropout_p > 0.f;
  if (drop && !rng_state) return PERT_ERR_BADARG;
  if (N == 0) return PERT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  double* acc = nullptr;
  if (training) {
    if (!workspace || workspace_bytes < pert_bn_workspace_bytes(N, H)) return PERT_ERR_BADARG;
    int chunks = pert_cdiv(N, BN_ROWS);
    int vpr = H / 4;
    int threads = 256;
    if (threads < H) threads = (H + 31) / 32 * 32;
    int rl_n = threads / vpr;
    if (rl_n < 1) return PERT_ERR_UNSUPPORTED;
    size_t smem = ((size_t)rl_n * H + H) * sizeof(float);
    if (smem > 48 * 1024) return PERT_ERR_UNSUPPORTED;
    if ((uintptr_t)workspace & 7) return PERT_ERR_BADARG;
    acc = (double*)workspace;
    if (!stats_ready) {
      cudaError_t e = cudaMemsetAsync(acc, 0, (size_t)2 * H * sizeof(double), st);
      if (e != cudaSuccess) return (int)e;
      k_bn_partial<<<chunks, threads, smem, st>>>(x, ld_x, N, H, acc);
    }
  } else {
    if (!running_mean || !running_var) return PERT_ERR_BADARG;
    k_bn_eval_stats<<<pert_cdiv(H, 128), 128, 0, st>>>(running_mean, running_var, eps, H, mean, rstd);
  }
  long long total = N * (H / 4);
  long long blocks = pert_cdiv(total, 256 * 4);
  if (blocks > 8LL * PERT_NUM_SMS) blocks = 8LL * PERT_NUM_SMS;
  const size_t smem = (size_t)4 * H * sizeof(float);
  float* rm = training ? running_mean : nullptr;
  float* rv = training ? running_var : nullptr;
  long long* nbt = training ? num_batches_tracked : nullptr;
  if (drop)
    k_bn_apply<true><<<(int)blocks, 256, smem, st>>>(x, ld_x, mean, rstd, gamma, beta, y, ld_y, N, H, relu, acc, eps,
                                                     momentum, rm, rv, nbt, dr);
  else
    k_bn_apply<false><<<(int)blocks, 256, smem, st>>>(x, ld_x, mean, rstd, gamma, beta, y, ld_y, N, H, relu, acc,
                                                      eps, momentum, rm, rv, nbt, dr);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

extern "C" {

// sums: [2H] scratch (zeroed here).  dgamma/dbeta accumulate (+=).
int pert_bn_bwd(const float* dy, int ld_dy, const float* y, int ld_y, const float* x, int ld_x, const float* mean,
                const float* rstd, const float* gamma, int relu, int training, float* dx, int ld_dx, float* dgamma,
                float* dbeta, float* sums, long long N, int H, void* stream) {
  return pert_bn_bwd_ex(dy, ld_dy, y, ld_y, x, ld_x, mean, rstd, gamma, relu, training, 1.f, dx, ld_dx, dgamma, dbeta,
                        sums, N, H, stream);
}

}  // extern "C"

// dropout_scale: 1/(1-p) of a training forward that applied dropout to y (relu only), else 1.
int pert_bn_bwd_ex(const float* dy, int ld_dy, const float* y, int ld_y, const float* x, int ld_x, const float* mean,
                   const float* rstd, const float* gamma, int relu, int training, float dropout_scale, float* dx,
                   int ld_dx, float* dgamma, float* dbeta, float* sums, long long N, int H, void* stream) {
  if (N < 0 || H <= 0 || H % 4 || H > 1024 || !dy || !x || !mean || !rstd || !gamma || !dx || !sums)
    return PERT_ERR_BADARG;
  if (dropout_scale != 1.f && !(relu && dropout_scale >= 0.f)) return PERT_ERR_BADARG;
  if (relu && !y) return PERT_ERR_BADARG;
  if (ld_dy % 4 || ld_x % 4 || ld_dx % 4 || (relu && ld_y % 4)) return PERT_ERR_BADARG;
  if (!al16(dy) || !al16(y) || !al16(x) || !al16(mean) || !al16(rstd) || !al16(gamma) || !al16(dx) || !al16(sums))
    return PERT_ERR_BADARG;
  if (N == 0) return PERT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(sums, 0, sizeof(float) * 2 * H, st);
  if (e != cudaSuccess) return (int)e;
  int vpr = H / 4;
  int threads = 256;
  if (threads < vpr) threads = (vpr + 31) / 32 * 32;
  int rl_n = threads / vpr;
  size_t smem = (size_t)rl_n * 2 * H * sizeof(float);
  if (smem > 48 * 1024) return PERT_ERR_UNSUPPORTED;
  if (dropout_scale != 1.f)
    k_bn_bwd_reduce<true><<<pert_cdiv(N, BN_BWD_ROWS), threads, smem, st>>>(dy, ld_dy, y, ld_y, x, ld_x, mean, rstd, N,
                                                                           H, relu, dropout_scale, sums);
  else
    k_bn_bwd_reduce<false><<<pert_cdiv(N, BN_BWD_ROWS), threads, smem, st>>>(dy, ld_dy, y, ld_y, x, ld_x, mean, rstd,
                                                                            N, H, relu, 1.f, sums);
  long long total = N * vpr;
  k_bn_bwd_apply<<<pert_cdiv(total, 256), 256, 0, st>>>(dy, ld_dy, y, ld_y, x, ld_x, mean, rstd, gamma, sums, dx,
                                                       ld_dx, N, H, relu, dropout_scale, training, dgamma, dbeta);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

extern "C" {

// local[n] = <x_n, w_local> + b_local (optional);  pool[batch[n]] += x_n * probs[n] / pnn[n]  (pool zeroed here)
int pert_pool_fwd(const float* x, int ld, const float* probs, const float* pnn, const int64_t* batch,
                  const float* w_local, const float* b_local, float* local, float* pool, long long N, long long B,
                  int H, int* status, void* stream) {
  if (N < 0 || B < 0 || !x || !probs || !pnn || !batch || !pool || ld % 4 || !al16(x) || !al16(w_local) ||
      !al16(pool))
    return PERT_ERR_BADARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (B > 0) {
    cudaError_t e = cudaMemsetAsync(pool, 0, sizeof(float) * B * H, st);
    if (e != cudaSuccess) return (int)e;
  }
  if (N == 0) return PERT_OK;
  int rc = dispatch_h(H, [&](auto lpr, auto vpl) {
    constexpr int LPR = decltype(lpr)::value, VPL = decltype(vpl)::value;
    long long groups = (N + POOL_ROWS - 1) / POOL_ROWS;
    long long threads = groups * LPR;
    k_pool_fwd<LPR, VPL><<<pert_cdiv(threads, 256), 256, 0, st>>>(x, ld, probs, pnn, batch, w_local, b_local, local,
                                                                 pool, N, (int)B, status);
    return PERT_OK;
  });
  if (rc) return rc;
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_pool_bwd(const float* dpool, const float* dlocal, const float* x, int ld, const float* probs,
                  const float* pnn, const int64_t* batch, const float* w_local, float* dx, int ld_dx,
                  float* dw_local, float* db_local, long long N, long long B, int H, void* stream) {
  if (N < 0 || !probs || !pnn || !batch || !dx || ld % 4 || ld_dx % 4 || !al16(dpool) || !al16(x) ||
      !al16(w_local) || !al16(dx))
    return PERT_ERR_BADARG;
  if (dlocal && (!x || !w_local)) return PERT_ERR_BADARG;
  if (N == 0) return PERT_OK;
  int rc = dispatch_h(H, [&](auto lpr, auto vpl) {
    constexpr int LPR = decltype(lpr)::value, VPL = decltype(vpl)::value;
    long long groups = (N + POOL_ROWS - 1) / POOL_ROWS;
    long long threads = groups * LPR;
    k_pool_bwd<LPR, VPL><<<pert_cdiv(threads, 256), 256, 0, (cudaStream_t)stream>>>(
        dpool, dlocal, x, ld, probs, pnn, batch, w_local, dx, ld_dx, dw_local, db_local, N, (int)B);
    return PERT_OK;
  });
  if (rc) return rc;
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_relu_bwd(const float* y, float* dy, long long n, void* stream) {
  if (n < 0 || !y || !dy) return PERT_ERR_BADARG;
  if (n == 0) return PERT_OK;
  k_relu_bwd<<<pert_cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(y, dy, n);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_pinball_loss(const int64_t* y, const float* yhat, float tau, long long B, float grad_scale, float* loss,
                      float* dyhat, void* stream) {
  if (B <= 0 || !y || !yhat) return PERT_ERR_BADARG;
  k_pinball<<<1, 256, 0, (cudaStream_t)stream>>>(y, yhat, tau, (int)B, grad_scale, loss, dyhat);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, long long step, float grad_scale, void* stream) {
  if (n < 0 || step < 1 || !p || !g || !m || !v) return PERT_ERR_BADARG;
  if (n == 0) return PERT_OK;
  float bc1 = 1.f - powf(beta1, (float)step);
  float bc2 = 1.f - powf(beta2, (float)step);
  k_adam<<<pert_cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay,
                                                             bc1, sqrtf(bc2), grad_scale);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

int pert_eval_metrics(const int64_t* y, const float* yhat, float tau, long long B, double* acc, void* stream) {
  if (B < 0 || !y || !yhat || !acc) return PERT_ERR_BADARG;
  if (B == 0) return PERT_OK;
  int grid = pert_cdiv(B, 256);
  if (grid > 64) grid = 64;
  k_eval_metrics<<<grid, 256, 0, (cudaStream_t)stream>>>(y, yhat, tau, (int)B, acc);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

}  // extern "C"
