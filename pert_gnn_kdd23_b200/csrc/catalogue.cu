// Trace catalogue on the GPU: runtime patterns, per-trace targets and entry pattern probabilities from a span table
// (the integer-coded part of preprocess.py:main(), :269-375).
//
// Input: the span table in file order (int64 columns) and `perm`, the row order grouped by traceid (a stable sort of
// the traceid column, so rows keep file order inside a trace), with row_ptr[T+1] over that order.  Traces are numbered
// by ascending traceid ("trace position").
//   summary      one warp per trace, any length: row count, an order-sensitive 64-bit hash of the (um, dm, interface)
//                sequence (:280-289), max |rt| (:290-292), floor(min timestamp / 30000) * 30000 (:39), the entry id
//                (status PERT_ERR_RANGE if the rows disagree)
//   verify       after sorting traces by (key, position): every member of a run is compared row by row with the
//                run's head, so equal keys never stand in for equal sequences
//   rekey        members that differ from their head get key = mix(key, hash with a new seed); repeated until no
//                member differs.  Traces with equal sequences always share key, head and mismatch flag, so they stay
//                together; the combined key is a full 64-bit value, so a masked (test) hash still separates in time
//   ids          first trace of every pattern in position order + an exclusive scan = factorize order (:293)
//   pattern      per pattern: representative = first trace in (entry, traceid) order (atomicMin), occurrences
//   pairs/probs  per (entry, pattern): count, first position inside the entry, count / total in float64 (:371-375)
// Every output is an integer or a correctly rounded division, so the result is deterministic whatever the atomics'
// order.
#include "common.cuh"

namespace {

constexpr int kWarpsPerBlock = 8;

__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {   // splitmix64 finaliser
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// Hash of the (um, dm, interface) sequence of rows [r0, r1) of the grouped order.  Each row's mix is keyed by its
// position inside the trace; the keyed mixes are added (mod 2^64), so the lane split does not matter but a permuted
// sequence hashes differently.  The row count is folded in at the end.
__device__ unsigned long long warp_seq_hash(const int64_t* perm, long long r0, long long r1, const int64_t* um,
                                            const int64_t* dm, const int64_t* itf, unsigned long long seed,
                                            int lane) {
  unsigned long long acc = 0;
  for (long long r = r0 + lane; r < r1; r += 32) {
    const long long i = perm[r];
    unsigned long long h = mix64((unsigned long long)um[i] + seed);
    h = mix64(h ^ (unsigned long long)dm[i]);
    h = mix64(h ^ (unsigned long long)itf[i]);
    acc += mix64(h ^ mix64((unsigned long long)(r - r0) * 0x9E3779B97F4A7C15ull + seed));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return mix64(acc ^ mix64((unsigned long long)(r1 - r0) ^ (seed * 0xD1B54A32D192ED03ull)));
}

__device__ __forceinline__ long long floor_div(long long a, long long b) {
  const long long q = a / b;
  return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}

struct SummaryArgs {
  const int64_t *perm, *row_ptr, *um, *dm, *itf, *rt, *ts, *entry;
  long long T;
  unsigned long long seed, mask;
  int64_t *nrows, *hash, *y, *ts_bucket, *trace_entry;
  int* status;
};

__global__ void __launch_bounds__(32 * kWarpsPerBlock) k_catalogue_summary(SummaryArgs a) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (t >= a.T) return;
  const long long r0 = a.row_ptr[t], r1 = a.row_ptr[t + 1];
  const unsigned long long h = warp_seq_hash(a.perm, r0, r1, a.um, a.dm, a.itf, a.seed, lane) & a.mask;
  const int64_t e0 = a.entry[a.perm[r0]];
  long long amax = 0, tmin = INT64_MAX;
  int bad = 0;
  for (long long r = r0 + lane; r < r1; r += 32) {
    const long long i = a.perm[r];
    const long long v = a.rt[i];
    amax = max(amax, v < 0 ? -v : v);
    tmin = min(tmin, (long long)a.ts[i]);
    bad |= a.entry[i] != e0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    amax = max(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    tmin = min(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
  }
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) {
    a.nrows[t] = r1 - r0;
    a.hash[t] = (int64_t)h;
    a.y[t] = amax;
    a.ts_bucket[t] = floor_div(tmin, 30000) * 30000;
    a.trace_entry[t] = e0;
    if (bad && a.status) atomicExch(a.status, PERT_ERR_RANGE);
  }
}

// Sorted position i of trace order[i]; head[i] = sorted position of its run's head.
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
    k_catalogue_verify(const int64_t* order, const int64_t* head, long long T, const int64_t* perm,
                       const int64_t* row_ptr, const int64_t* um, const int64_t* dm, const int64_t* itf,
                       int32_t* mismatch, unsigned long long* n_mismatch) {
  const int lane = threadIdx.x & 31;
  const long long i = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (i >= T) return;
  const long long t = order[i], h = order[head[i]];
  int diff = 0;
  if (t != h) {
    const long long a0 = row_ptr[t], n = row_ptr[t + 1] - a0, b0 = row_ptr[h];
    diff = n != row_ptr[h + 1] - b0;               // uniform across the warp, like every trip of the loop below
    for (long long k0 = 0; k0 < n && !diff; k0 += 32) {
      const long long k = k0 + lane;
      bool d = false;
      if (k < n) {
        const long long x = perm[a0 + k], y = perm[b0 + k];
        d = um[x] != um[y] || dm[x] != dm[y] || itf[x] != itf[y];
      }
      diff = __any_sync(0xffffffffu, d);
    }
  }
  if (lane == 0) {
    mismatch[t] = diff;
    if (diff) atomicAdd(n_mismatch, 1ull);
  }
}

__global__ void __launch_bounds__(32 * kWarpsPerBlock)
    k_catalogue_rekey(const int64_t* perm, const int64_t* row_ptr, long long T, const int64_t* um, const int64_t* dm,
                      const int64_t* itf, const int32_t* mismatch, unsigned long long seed, unsigned long long mask,
                      int64_t* key) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (t >= T || !mismatch[t]) return;
  const unsigned long long h = warp_seq_hash(perm, row_ptr[t], row_ptr[t + 1], um, dm, itf, seed, lane) & mask;
  if (lane == 0) key[t] = (int64_t)mix64((unsigned long long)key[t] * 0x9E3779B97F4A7C15ull ^ mix64(h + seed));
}

__global__ void k_run_flags(const int64_t* key, long long n, int64_t* flag, int64_t* mark) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t f = i == 0 || key[i] != key[i - 1];
  flag[i] = f;
  if (mark) mark[i] = f ? i : 0;
}

__global__ void k_catalogue_canon(const int64_t* order, const int64_t* head, long long T, int64_t* canon,
                                  int64_t* first) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  const long long t = order[i], h = order[head[i]];
  canon[t] = h;
  first[t] = t == h;
}

__global__ void k_catalogue_rid(const int64_t* canon, const int64_t* first_incl, long long T, int64_t* rid) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < T) rid[t] = first_incl[canon[t]] - 1;
}

__global__ void k_catalogue_pattern(const int64_t* eorder, const int64_t* eidx, long long T, const int64_t* rid,
                                    long long P, unsigned long long* rep_epos, unsigned long long* occ,
                                    int64_t* pair_key) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= T) return;
  const long long r = rid[eorder[j]];
  atomicMin(rep_epos + r, (unsigned long long)j);
  atomicAdd(occ + r, 1ull);
  pair_key[j] = eidx[j] * P + r;
}

__global__ void k_catalogue_pairs(const int64_t* pstart, long long NP, long long T, const int64_t* pidx,
                                  const int64_t* eorder, const int64_t* rid, const int64_t* eidx, int64_t* count,
                                  int64_t* first, int64_t* pent, int64_t* prid) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= NP) return;
  const long long s = pstart[p], e = p + 1 < NP ? pstart[p + 1] : T;
  const long long j = pidx[s];                  // stable sort: the run's first entry-order position
  count[p] = e - s;
  first[p] = j;
  pent[p] = eidx[j];
  prid[p] = rid[eorder[j]];
}

__global__ void k_catalogue_probs(const int64_t* pent, const int64_t* count, long long NP, const int64_t* ent_start,
                                  long long E, long long T, double* prob, int64_t* ent_ptr) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= NP) return;
  const long long e = pent[q];
  const long long total = (e + 1 < E ? ent_start[e + 1] : T) - ent_start[e];
  prob[q] = (double)count[q] / (double)total;   // IEEE division: == Python's int / int for counts < 2^53
  if (q == 0 || pent[q - 1] != e) ent_ptr[e] = q;
  if (q == NP - 1) ent_ptr[E] = NP;
}

inline unsigned warp_grid(long long n) { return (unsigned)((n + kWarpsPerBlock - 1) / kWarpsPerBlock); }
inline unsigned flat_grid(long long n) { return (unsigned)((n + 255) / 256); }

}  // namespace

extern "C" int pert_catalogue_run_flags(const int64_t* key, long long n, int64_t* flag, int64_t* mark, void* stream) {
  if (!key || !flag || n < 0) return PERT_ERR_BADARG;
  if (n == 0) return 0;
  k_run_flags<<<flat_grid(n), 256, 0, (cudaStream_t)stream>>>(key, n, flag, mark);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_summary(const int64_t* perm, const int64_t* row_ptr, long long T, const int64_t* um,
                                      const int64_t* dm, const int64_t* interface, const int64_t* rt,
                                      const int64_t* timestamp, const int64_t* entryid, unsigned long long seed,
                                      unsigned long long hash_mask, int64_t* nrows, int64_t* hash, int64_t* y,
                                      int64_t* ts_bucket, int64_t* trace_entry, int* status, void* stream) {
  if (!perm || !row_ptr || !um || !dm || !interface || !rt || !timestamp || !entryid || !nrows || !hash || !y ||
      !ts_bucket || !trace_entry || T < 0)
    return PERT_ERR_BADARG;
  if (T == 0) return 0;
  SummaryArgs a{perm, row_ptr, um, dm, interface, rt, timestamp, entryid, T, seed, hash_mask,
                nrows, hash, y, ts_bucket, trace_entry, status};
  k_catalogue_summary<<<warp_grid(T), 32 * kWarpsPerBlock, 0, (cudaStream_t)stream>>>(a);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_verify(const int64_t* order, const int64_t* head, long long T, const int64_t* perm,
                                     const int64_t* row_ptr, const int64_t* um, const int64_t* dm,
                                     const int64_t* interface, int32_t* mismatch, unsigned long long* n_mismatch,
                                     void* stream) {
  if (!order || !head || !perm || !row_ptr || !um || !dm || !interface || !mismatch || !n_mismatch || T < 0)
    return PERT_ERR_BADARG;
  cudaError_t e = cudaMemsetAsync(n_mismatch, 0, sizeof(unsigned long long), (cudaStream_t)stream);
  if (e != cudaSuccess) return (int)e;
  if (T == 0) return 0;
  k_catalogue_verify<<<warp_grid(T), 32 * kWarpsPerBlock, 0, (cudaStream_t)stream>>>(order, head, T, perm, row_ptr,
                                                                                      um, dm, interface, mismatch,
                                                                                      n_mismatch);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_rekey(const int64_t* perm, const int64_t* row_ptr, long long T, const int64_t* um,
                                    const int64_t* dm, const int64_t* interface, const int32_t* mismatch,
                                    unsigned long long seed, unsigned long long hash_mask, int64_t* key,
                                    void* stream) {
  if (!perm || !row_ptr || !um || !dm || !interface || !mismatch || !key || T < 0) return PERT_ERR_BADARG;
  if (T == 0) return 0;
  k_catalogue_rekey<<<warp_grid(T), 32 * kWarpsPerBlock, 0, (cudaStream_t)stream>>>(perm, row_ptr, T, um, dm,
                                                                                     interface, mismatch, seed,
                                                                                     hash_mask, key);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_canon(const int64_t* order, const int64_t* head, long long T, int64_t* canon,
                                    int64_t* first, void* stream) {
  if (!order || !head || !canon || !first || T < 0) return PERT_ERR_BADARG;
  if (T == 0) return 0;
  k_catalogue_canon<<<flat_grid(T), 256, 0, (cudaStream_t)stream>>>(order, head, T, canon, first);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_runtime_ids(const int64_t* canon, const int64_t* first_incl, long long T, int64_t* rid,
                                          void* stream) {
  if (!canon || !first_incl || !rid || T < 0) return PERT_ERR_BADARG;
  if (T == 0) return 0;
  k_catalogue_rid<<<flat_grid(T), 256, 0, (cudaStream_t)stream>>>(canon, first_incl, T, rid);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_patterns(const int64_t* eorder, const int64_t* eidx, long long T, const int64_t* rid,
                                       long long P, int64_t* rep_epos, int64_t* occurrences, int64_t* pair_key,
                                       void* stream) {
  if (!eorder || !eidx || !rid || !rep_epos || !occurrences || !pair_key || T < 0 || P < 0) return PERT_ERR_BADARG;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(rep_epos, 0x7f, P * sizeof(int64_t), st);   // 0x7f7f.. > any position
  if (e == cudaSuccess) e = cudaMemsetAsync(occurrences, 0, P * sizeof(int64_t), st);
  if (e != cudaSuccess) return (int)e;
  if (T == 0) return 0;
  k_catalogue_pattern<<<flat_grid(T), 256, 0, st>>>(eorder, eidx, T, rid, P,
                                                     reinterpret_cast<unsigned long long*>(rep_epos),
                                                     reinterpret_cast<unsigned long long*>(occurrences), pair_key);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_pairs(const int64_t* pstart, long long NP, long long T, const int64_t* pidx,
                                    const int64_t* eorder, const int64_t* rid, const int64_t* eidx, int64_t* count,
                                    int64_t* first, int64_t* pair_entry, int64_t* pair_rid, void* stream) {
  if (!pstart || !pidx || !eorder || !rid || !eidx || !count || !first || !pair_entry || !pair_rid || NP < 0 || T < 0)
    return PERT_ERR_BADARG;
  if (NP == 0) return 0;
  k_catalogue_pairs<<<flat_grid(NP), 256, 0, (cudaStream_t)stream>>>(pstart, NP, T, pidx, eorder, rid, eidx, count,
                                                                      first, pair_entry, pair_rid);
  PERT_LAUNCH_CHECK();
  return 0;
}

extern "C" int pert_catalogue_probs(const int64_t* pair_entry, const int64_t* count, long long NP,
                                    const int64_t* ent_start, long long E, long long T, double* prob,
                                    int64_t* ent_ptr, void* stream) {
  if (!pair_entry || !count || !ent_start || !prob || !ent_ptr || NP < 0 || E < 0 || T < 0) return PERT_ERR_BADARG;
  if (NP == 0) return 0;
  k_catalogue_probs<<<flat_grid(NP), 256, 0, (cudaStream_t)stream>>>(pair_entry, count, NP, ent_start, E, T, prob,
                                                                      ent_ptr);
  PERT_LAUNCH_CHECK();
  return 0;
}
