// Index construction (integer, bit-exact): COO edge_index (int64) -> int32 CSR-by-target +
// CSC-by-source, both STABLE (ascending original edge id inside a segment), and the edge
// attributes permuted into CSR order.  Built once per batch, reused by every layer and by
// backward.  Replaces what PyG's MessagePassing does implicitly on COO (reference call sites
// model.py:100,104; collation pert_gnn.py:107-119,201-209).  Numpy definition of the
// layout: oracle/index_oracle.py:build_index.
//
// HBM-bound integer work: ~40 B/edge of traffic in 9 small launches.  Stability without a
// radix sort: unordered atomic fill, then every segment is sorted by edge id -- a segment is a
// node's in- (or out-) edge list, a handful of entries, so one thread does an insertion sort;
// segments longer than SORT_SMALL go to a CTA-wide rank sort.
#include "common.cuh"

#define SORT_SMALL 32
#define SCAN_THREADS 1024
#define SCAN_ITEMS 4
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

namespace {

__global__ void k_count(const int64_t* __restrict__ ei, int E, int N, int* __restrict__ rowptr,
                        int* __restrict__ colptr, int* status) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= E) return;
  int64_t s = ei[t], d = ei[(size_t)E + t];
  if (s < 0 || s >= N || d < 0 || d >= N) {
    if (status) atomicExch(status, PERT_ERR_RANGE);
    return;
  }
  atomicAdd(&rowptr[d + 1], 1);
  atomicAdd(&colptr[s + 1], 1);
}

// ---- 3-phase inclusive scan over two int arrays (blockIdx.y selects the array) ----
__device__ __forceinline__ int block_scan_inclusive(int v, int* smem_warp /*32*/) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  if (lane == 31) smem_warp[w] = v;
  __syncthreads();
  if (w == 0) {
    int x = smem_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += u;
    }
    smem_warp[lane] = x;
  }
  __syncthreads();
  int base = (w == 0) ? 0 : smem_warp[w - 1];
  __syncthreads();
  return v + base;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_sums(const int* a0, const int* a1, int L,
                                                                  int* bsum, int nb) {
  __shared__ int sw[32];
  const int* a = blockIdx.y ? a1 : a0;
  int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  int s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i)
    if (base + i < L) s += a[base + i];
  int incl = block_scan_inclusive(s, sw);
  if (threadIdx.x == SCAN_THREADS - 1) bsum[blockIdx.y * nb + blockIdx.x] = incl;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_block_sums(int* bsum, int nb) {
  __shared__ int sw[32];
  __shared__ int carry_s;
  int* b = bsum + blockIdx.y * nb;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += SCAN_THREADS) {
    int i = base + threadIdx.x;
    int v = (i < nb) ? b[i] : 0;
    int incl = block_scan_inclusive(v, sw);
    int carry = carry_s;
    __syncthreads();
    if (i < nb) b[i] = carry + incl - v;   // exclusive prefix of tile sums
    if (threadIdx.x == SCAN_THREADS - 1) carry_s = carry + incl;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(int* a0, int* a1, int L, const int* bsum,
                                                              int nb) {
  __shared__ int sw[32];
  int* a = blockIdx.y ? a1 : a0;
  int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
  int v[SCAN_ITEMS];
  int s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    v[i] = (base + i < L) ? a[base + i] : 0;
    s += v[i];
  }
  int incl = block_scan_inclusive(s, sw);
  int run = incl - s + bsum[blockIdx.y * nb + blockIdx.x];
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    run += v[i];
    if (base + i < L) a[base + i] = run;
  }
}

__global__ void k_fill(const int64_t* __restrict__ ei, int E, int N, const int* __restrict__ rowptr,
                       const int* __restrict__ colptr, int* __restrict__ fill, int* __restrict__ slot_csr,
                       int* __restrict__ slot_csc) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= E) return;
  int64_t s = ei[t], d = ei[(size_t)E + t];
  if (s < 0 || s >= N || d < 0 || d >= N) return;
  int p = rowptr[d] + atomicAdd(&fill[d], 1);
  slot_csr[p] = t;
  int c = colptr[s] + atomicAdd(&fill[N + s], 1);
  slot_csc[c] = t;
}

// one thread per (node, side): sort the segment's edge ids ascending (== stable order)
__global__ void k_sort_small(int N, const int* __restrict__ rowptr, const int* __restrict__ colptr,
                             const int* __restrict__ slot_csr, const int* __restrict__ slot_csc,
                             int* __restrict__ perm, int* __restrict__ cperm, int* __restrict__ long_list,
                             int* __restrict__ long_count) {
  int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= 2 * N) return;
  int side = id >= N;
  int n = side ? id - N : id;
  const int* ptr = side ? colptr : rowptr;
  const int* in = side ? slot_csc : slot_csr;
  int* out = side ? cperm : perm;
  int b = ptr[n], len = ptr[n + 1] - b;
  if (len <= 0) return;
  if (len > SORT_SMALL) {
    int k = atomicAdd(long_count, 1);
    long_list[k] = id;
    return;
  }
  // rank sort straight from the (L1-resident) slots: ids are unique, so rank = #smaller.  (An insertion sort in a
  // dynamically indexed local array lives in local memory: 24 us at N = 51k; typical segments have ~3 entries.)
  for (int i = 0; i < len; ++i) {
    const int x = __ldg(in + b + i);
    int rank = 0;
    for (int j = 0; j < len; ++j) rank += (__ldg(in + b + j) < x);
    out[b + rank] = x;
  }
}

// CTA per long segment: rank sort (ids are unique -> rank = #smaller)
__global__ void k_sort_long(int N, const int* __restrict__ rowptr, const int* __restrict__ colptr,
                            const int* __restrict__ slot_csr, const int* __restrict__ slot_csc,
                            int* __restrict__ perm, int* __restrict__ cperm,
                            const int* __restrict__ long_list, const int* __restrict__ long_count) {
  __shared__ int tile[1024];
  int cnt = *long_count;
  for (int k = blockIdx.x; k < cnt; k += gridDim.x) {
    int id = long_list[k];
    int side = id >= N;
    int n = side ? id - N : id;
    const int* ptr = side ? colptr : rowptr;
    const int* in = (side ? slot_csc : slot_csr) + ptr[n];
    int* out = (side ? cperm : perm) + ptr[n];
    int len = ptr[n + 1] - ptr[n];
    for (int i0 = 0; i0 < len; i0 += blockDim.x) {
      int i = i0 + threadIdx.x;
      int x = (i < len) ? in[i] : 0;
      int rank = 0;
      for (int j0 = 0; j0 < len; j0 += 1024) {
        int m = min(1024, len - j0);
        __syncthreads();
        for (int j = threadIdx.x; j < m; j += blockDim.x) tile[j] = in[j0 + j];
        __syncthreads();
        if (i < len)
          for (int j = 0; j < m; ++j) rank += (tile[j] < x);
      }
      if (i < len) out[rank] = x;
    }
    __syncthreads();
  }
}

__global__ void k_finalize_csr(const int64_t* __restrict__ ei, const int64_t* __restrict__ attr, int attr_cols,
                               int E, int n_if, int n_rpc, const int* __restrict__ perm,
                               int* __restrict__ csr_src, int* __restrict__ csr_if, int* __restrict__ csr_rpc,
                               int* __restrict__ inv, int* status, const int* __restrict__ nvalid) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= E) return;
  if (p >= *nvalid) {     // edges dropped by the range check (status = PERT_ERR_RANGE): slots past the last segment
    csr_src[p] = 0;       // hold no edge -- keep them addressable instead of leaving uninitialised ids behind
    if (attr) { csr_if[p] = 0; csr_rpc[p] = 0; }
    return;
  }
  int t = perm[p];
  csr_src[p] = (int)ei[t];
  inv[t] = p;
  if (attr) {
    int64_t a = attr[(size_t)t * attr_cols], b = attr[(size_t)t * attr_cols + 1];
    if (a < 0 || a >= n_if || b < 0 || b >= n_rpc) {
      if (status) atomicExch(status, PERT_ERR_RANGE);
      a = 0;
      b = 0;
    }
    csr_if[p] = (int)a;
    csr_rpc[p] = (int)b;
  }
}

__global__ void k_finalize_csc(const int64_t* __restrict__ ei, int E, const int* __restrict__ cperm,
                               const int* __restrict__ inv, int* __restrict__ csc_pos,
                               int* __restrict__ csc_dst, const int* __restrict__ nvalid) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= E) return;
  if (c >= *nvalid) {
    csc_pos[c] = 0;
    csc_dst[c] = 0;
    return;
  }
  int t = cperm[c];
  csc_pos[c] = inv[t];
  csc_dst[c] = (int)ei[(size_t)E + t];
}

// ---- per-graph multi-source min-depth (level index), one CTA per graph --------------
// Restates reference misc.py:59-63 (relaxing DFS == BFS distance over out-edges); -1 = unreachable.
__global__ void k_min_depth(const int* __restrict__ gptr, const int* __restrict__ colptr,
                            const int* __restrict__ csc_dst, const int* __restrict__ roots, int* __restrict__ depth) {
  int g = blockIdx.x;
  int n0 = gptr[g], n1 = gptr[g + 1];
  __shared__ int changed;
  for (int n = n0 + threadIdx.x; n < n1; n += blockDim.x) depth[n] = 0x7fffffff;
  __syncthreads();
  if (threadIdx.x == 0) {
    int r = roots[g];
    if (r >= n0 && r < n1) depth[r] = 0;
  }
  __syncthreads();
  // level-synchronous relaxation; at most (n1-n0) rounds, normally max-depth+1
  for (int round = 0; round < n1 - n0; ++round) {
    if (threadIdx.x == 0) changed = 0;
    __syncthreads();
    for (int n = n0 + threadIdx.x; n < n1; n += blockDim.x) {
      int d = depth[n];
      if (d == round) {
        for (int c = colptr[n]; c < colptr[n + 1]; ++c) {
          int v = csc_dst[c];
          if (atomicMin(&depth[v], d + 1) > d + 1) changed = 1;
        }
      }
    }
    __syncthreads();
    int ch = changed;
    __syncthreads();
    if (!ch) break;
  }
  for (int n = n0 + threadIdx.x; n < n1; n += blockDim.x)
    if (depth[n] == 0x7fffffff) depth[n] = -1;
}


// ---- stored node_depth tensor (reference misc.py:159-175 + the long cast of :215 / :368), one CTA per graph ----------
// unreachable (-1) -> 0; divide by the graph's max depth (1 if that is 0) in float64 like numpy does; the
// torch.tensor(float ndarray, dtype=torch.long) of the reference truncates toward zero -> values in {0, 1}.
__global__ void k_node_depth(const int* __restrict__ gptr, const int* __restrict__ depth, int64_t* __restrict__ out) {
  const int g = blockIdx.x;
  const int n0 = gptr[g], n1 = gptr[g + 1];
  __shared__ int smax;
  if (threadIdx.x == 0) smax = 0;
  __syncthreads();
  int m = 0;
  for (int n = n0 + threadIdx.x; n < n1; n += blockDim.x) m = max(m, depth[n]);   // -1 never wins against 0
  m = __reduce_max_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0) atomicMax(&smax, m);
  __syncthreads();
  const double norm = smax > 0 ? (double)smax : 1.0;
  for (int n = n0 + threadIdx.x; n < n1; n += blockDim.x) {
    const int d = depth[n];
    out[n] = (int64_t)((double)(d < 0 ? 0 : d) / norm);
  }
}

// ---- level-major node order inside each graph (BASELINE north_star "per-level index layout"; definition:
// oracle/index_oracle.py:level_order): order = stable sort of the graph's nodes by level, unreachable (-1) last.
// One CTA per graph: histogram of levels in shared memory (levels <= LV_MAX, deeper ones clamp into the last bucket
// and are ordered there by a rank pass), exclusive scan, stable placement by counting the earlier nodes of the
// same level (graphs are a few hundred nodes: O(n * n / threads) compares, no atomics -> deterministic).
constexpr int LV_MAX = 1023;
__global__ void __launch_bounds__(256) k_level_order(const int* __restrict__ gptr, const int* __restrict__ depth,
                                                     int* __restrict__ order) {
  const int g = blockIdx.x;
  const int n0 = gptr[g], n1 = gptr[g + 1], n = n1 - n0;
  __shared__ int hist[LV_MAX + 2];
  for (int x = threadIdx.x; x < LV_MAX + 2; x += blockDim.x) hist[x] = 0;
  __syncthreads();
  auto key = [&](int v) {
    const int d = depth[n0 + v];
    return d < 0 ? LV_MAX + 1 : (d > LV_MAX ? LV_MAX : d);
  };
  for (int v = threadIdx.x; v < n; v += blockDim.x) atomicAdd(&hist[key(v)], 1);
  __syncthreads();
  if (threadIdx.x == 0) {                       // exclusive scan of <= 1025 buckets
    int run = 0;
    for (int b = 0; b < LV_MAX + 2; ++b) {
      const int c = hist[b];
      hist[b] = run;
      run += c;
    }
  }
  __syncthreads();
  for (int v = threadIdx.x; v < n; v += blockDim.x) {
    const int kv = key(v);
    const int dv = depth[n0 + v];
    int rank = 0;
    // earlier nodes of the same bucket; inside the clamped bucket order by (true depth, id)
    for (int u = 0; u < n; ++u) {
      if (key(u) != kv) continue;
      const int du = depth[n0 + u];
      rank += (du < dv) || (du == dv && u < v);
    }
    order[n0 + hist[kv] + rank] = n0 + v;
  }
}

__global__ void k_graph_ptr_count(const int64_t* __restrict__ batch, int N, int B, int* __restrict__ ptr, int* status) {
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  int64_t g = batch[n];
  if (g < 0 || g >= B) {
    if (status) atomicExch(status, PERT_ERR_RANGE);
    return;
  }
  atomicAdd(&ptr[g + 1], 1);
}

}  // namespace

extern "C" {

int pert_version(void) { return 2005; }

long long pert_index_workspace_bytes(long long N, long long E) {
  if (N < 0 || E < 0) return PERT_ERR_BADARG;
  long long nb = (N + 1 + SCAN_TILE - 1) / SCAN_TILE;
  long long ints = 2 * N      /* fill counters  */
                   + 2 * E    /* unordered slots */
                   + E        /* cperm */
                   + E        /* inv */
                   + 2 * nb   /* tile sums */
                   + 2 * N    /* long-segment list */
                   + 4;       /* long_count (+pad) */
  return ints * 4 + 256;
}

int pert_build_index(const int64_t* edge_index, const int64_t* edge_attr, int attr_cols, long long N_, long long E_,
                     int n_if, int n_rpc, int* rowptr, int* perm, int* csr_src, int* csr_if, int* csr_rpc,
                     int* colptr, int* csc_pos, int* csc_dst, void* workspace, long long workspace_bytes,
                     int* status, void* stream_) {
  if (N_ < 0 || E_ < 0 || N_ > 0x7ffffff0LL || E_ > 0x7ffffff0LL) return PERT_ERR_BADARG;
  if (!rowptr || !colptr || !workspace) return PERT_ERR_BADARG;
  if (E_ > 0 && (!edge_index || !perm || !csr_src || !csc_pos || !csc_dst)) return PERT_ERR_BADARG;
  if (edge_attr && (attr_cols < 2 || !csr_if || !csr_rpc)) return PERT_ERR_BADARG;
  if (workspace_bytes < pert_index_workspace_bytes(N_, E_)) return PERT_ERR_BADARG;
  cudaStream_t st = (cudaStream_t)stream_;
  int N = (int)N_, E = (int)E_;
  int L = N + 1;
  int nb = pert_cdiv(L, SCAN_TILE);
  int* w = (int*)workspace;
  int* fill = w;                 w += 2 * (size_t)N;
  int* slot_csr = w;             w += E;
  int* slot_csc = w;             w += E;
  int* cperm = w;                w += E;
  int* inv = w;                  w += E;
  int* bsum = w;                 w += 2 * nb;
  int* long_list = w;            w += 2 * (size_t)N;
  int* long_count = w;

  cudaError_t e;
  if ((e = cudaMemsetAsync(rowptr, 0, sizeof(int) * L, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(colptr, 0, sizeof(int) * L, st)) != cudaSuccess) return (int)e;
  if (N > 0 && (e = cudaMemsetAsync(fill, 0, sizeof(int) * 2 * (size_t)N, st)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(long_count, 0, sizeof(int), st)) != cudaSuccess) return (int)e;
  if (E == 0) return PERT_OK;

  const int T = 256;
  k_count<<<pert_cdiv(E, T), T, 0, st>>>(edge_index, E, N, rowptr, colptr, status);
  k_scan_tile_sums<<<dim3(nb, 2), SCAN_THREADS, 0, st>>>(rowptr, colptr, L, bsum, nb);
  k_scan_block_sums<<<dim3(1, 2), SCAN_THREADS, 0, st>>>(bsum, nb);
  k_scan_apply<<<dim3(nb, 2), SCAN_THREADS, 0, st>>>(rowptr, colptr, L, bsum, nb);
  k_fill<<<pert_cdiv(E, T), T, 0, st>>>(edge_index, E, N, rowptr, colptr, fill, slot_csr, slot_csc);
  k_sort_small<<<pert_cdiv(2LL * N, T), T, 0, st>>>(N, rowptr, colptr, slot_csr, slot_csc, perm, cperm, long_list,
                                                   long_count);
  k_sort_long<<<PERT_NUM_SMS, 256, 0, st>>>(N, rowptr, colptr, slot_csr, slot_csc, perm, cperm, long_list,
                                            long_count);
  k_finalize_csr<<<pert_cdiv(E, T), T, 0, st>>>(edge_index, edge_attr, attr_cols, E, n_if, n_rpc, perm, csr_src,
                                                csr_if, csr_rpc, inv, status, rowptr + N);
  k_finalize_csc<<<pert_cdiv(E, T), T, 0, st>>>(edge_index, E, cperm, inv, csc_pos, csc_dst, rowptr + N);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

// ptr[B+1] (int32) from a PyG batch vector: count per graph + inclusive scan.
int pert_graph_ptr(const int64_t* batch, long long N_, long long B_, int* ptr, void* workspace,
                   long long workspace_bytes, int* status, void* stream_) {
  if (N_ < 0 || B_ < 0 || !ptr || !workspace) return PERT_ERR_BADARG;
  int N = (int)N_, B = (int)B_, L = B + 1;
  int nb = pert_cdiv(L, SCAN_TILE);
  if (workspace_bytes < (long long)(2 * nb + 2) * 4) return PERT_ERR_BADARG;
  cudaStream_t st = (cudaStream_t)stream_;
  cudaError_t e;
  if ((e = cudaMemsetAsync(ptr, 0, sizeof(int) * L, st)) != cudaSuccess) return (int)e;
  if (N == 0) return PERT_OK;
  int* bsum = (int*)workspace;
  k_graph_ptr_count<<<pert_cdiv(N, 256), 256, 0, st>>>(batch, N, B, ptr, status);
  k_scan_tile_sums<<<dim3(nb, 1), SCAN_THREADS, 0, st>>>(ptr, ptr, L, bsum, nb);
  k_scan_block_sums<<<dim3(1, 1), SCAN_THREADS, 0, st>>>(bsum, nb);
  k_scan_apply<<<dim3(nb, 1), SCAN_THREADS, 0, st>>>(ptr, ptr, L, bsum, nb);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

// depth[N] (int32): min hop count from roots[g] inside graph g over out-edges; -1 unreachable.
int pert_min_depth(const int* gptr, long long B_, const int* colptr, const int* csc_dst, const int* roots,
                   int* depth, void* stream_) {
  if (B_ < 0 || !gptr || !colptr || !roots || !depth) return PERT_ERR_BADARG;
  if (B_ == 0) return PERT_OK;
  k_min_depth<<<(int)B_, 128, 0, (cudaStream_t)stream_>>>(gptr, colptr, csc_dst, roots, depth);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

// node_depth[N] int64 = the tensor the reference stores on every Data (misc.py:159-175,215,368) from the raw min-depth.
int pert_node_depth(const int* gptr, long long B_, const int* depth, int64_t* node_depth, void* stream_) {
  if (B_ < 0 || !gptr || !depth || !node_depth) return PERT_ERR_BADARG;
  if (B_ == 0) return PERT_OK;
  k_node_depth<<<(int)B_, 128, 0, (cudaStream_t)stream_>>>(gptr, depth, node_depth);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

// order[N] int32: node ids in (graph, level, id) order, unreachable last inside their graph.
int pert_level_order(const int* gptr, long long B_, const int* depth, int* order, void* stream_) {
  if (B_ < 0 || !gptr || !depth || !order) return PERT_ERR_BADARG;
  if (B_ == 0) return PERT_OK;
  k_level_order<<<(int)B_, 256, 0, (cudaStream_t)stream_>>>(gptr, depth, order);
  PERT_LAUNCH_CHECK();
  return PERT_OK;
}

}  // extern "C"
