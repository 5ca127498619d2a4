/* libpertgnn -- C-ABI of the B200 (sm_100a) hot path of PERT-GNN.
 *
 * The reference (handasontam/PERT-GNN-KDD23) is pure Python on top of torch_geometric 2.4.0 and has no
 * FFI of its own; the "interface each entry point replaces" is therefore the Python/PyG call the
 * reference makes at the cited file:line.  INTEGRATION.md shows the ctypes binding (the one this
 * repository ships in pert_gnn_kdd23_b200/_lib.py) a maintainer of the reference would add.
 *
 * Conventions (all entry points):
 *   - every data buffer (inputs, outputs, workspaces, scratch) is a CALLER-OWNED DEVICE pointer: the library
 *     allocates no device memory for data (the one exception is pert_peer_alloc, whose purpose is to allocate the
 *     IPC-shareable exchange buffer);  fp32 row-major, `ld*` = row stride in floats; indices int32 inside the library,
 *     int64 where the reference's tensors are int64 (edge_index, edge_attr, batch, ids);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous, nothing synchronises; every call acts on the
 *     CURRENT CUDA device, which must be the device that owns the buffers and the stream (the Python binding enters
 *     torch.cuda.device(tensor.device) around each call);
 *   - return value: 0 = ok; > 0 = cudaError_t of a failed launch/memset; < 0 = library code
 *     (PERT_ERR_*).  Never throws, never exits.  Out-of-range indices found ON THE DEVICE are
 *     reported by writing PERT_ERR_RANGE into the optional device word `status`;
 *   - library-owned state (all of it; none of it is data): (1) a per-device ring of 8192 self-resetting tile-ticket
 *     counters for the dynamically scheduled tensor-core GEMMs -- every launch takes the next slot (host atomic), so
 *     concurrent launches on different streams / threads / captured graphs do not share a counter unless 8192 GEMM
 *     launches separate them while the first is still running; (2) per device, one auxiliary non-blocking stream and
 *     two events the step engine (pert_model_forward/backward) uses to run independent small kernels beside the main
 *     chain (fork/join by events, capture-safe; PERT_ENGINE_FORK=0 disables); the host-side issue of engine calls on
 *     one device is serialised by a mutex, so engines driven from several host threads / streams stay correct (their
 *     side work shares that one auxiliary stream); (3) the cached
 *     cuTensorMapEncodeTiled driver entry point; (4) environment switches read once (debug / measurement A/B only):
 *     PERT_GEMM_TC, PERT_GEMM_TMA, PERT_GEMM_TN_ACC, PERT_TCONV_TILE, PERT_TCONV_VPL, PERT_TCONV_VPL_BWD,
 *     PERT_TILE_LIST, PERT_BN_FUSE, PERT_ENGINE_FORK, PERT_PEER_MODE.
 *     With that, operator-level calls are re-entrant and thread-safe across streams;
 *   - rows of float matrices must be 16-byte aligned (ld % 4 == 0, base pointer 16-byte aligned)
 *     unless stated otherwise.
 */
#ifndef PERTGNN_H_
#define PERTGNN_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PERT_OK 0
#define PERT_ERR_BADARG (-1)
#define PERT_ERR_UNSUPPORTED (-2)
#define PERT_ERR_RANGE (-3)
#define PERT_ERR_PEER_TIMEOUT (-4)

/* ABI version (major*1000 + minor).  2000: pert_tconv_bwd takes rpc_ws; node_depth / eval-metric entry points.
 * 2001: pert_pert_graph_count / pert_pert_graph_build.  2002: pert_allreduce_adam timing[5], reduce-scatter form.
 * 2003: pert_span_graph_count / pert_span_graph_build.  2004: training-mode dropout in the step engine
 * (pert_model_forward gains dropout_p + rng_state, pert_model_backward gains dropout_p), pert_dropout_mask.
 * 2005: pert_catalogue_* (trace catalogue). */
int pert_version(void);

/* ---- index construction (integer, bit-exact) ---------------------------------------------------
 * Replaces the COO handling PyG MessagePassing does implicitly for TransformerConv.propagate
 * (reference model.py:100,104) and the edge_index offsetting/collation of pert_gnn.py:107-119,
 * 201-209: builds, once per batch, a STABLE CSR by target and CSC by source.
 *   edge_index int64 [2,E] (row 0 source, row 1 target);  edge_attr int64 [E,attr_cols] or NULL
 *   (columns 0,1 = interface id, rpctype id -- reference model.py:93-94), ids checked < n_if/n_rpc.
 * out (int32): rowptr[N+1], perm[E] (original edge id at CSR slot), csr_src[E], csr_if[E], csr_rpc[E],
 *              colptr[N+1], csc_pos[E] (CSR slot of the edge at CSC slot), csc_dst[E].
 * Definition of the layout: oracle/index_oracle.py:build_index. */
long long pert_index_workspace_bytes(long long N, long long E);
int pert_build_index(const int64_t* edge_index, const int64_t* edge_attr, int attr_cols, long long N, long long E,
                     int n_if, int n_rpc, int* rowptr, int* perm, int* csr_src, int* csr_if, int* csr_rpc,
                     int* colptr, int* csc_pos, int* csc_dst, void* workspace, long long workspace_bytes,
                     int* status, void* stream);

/* ptr[B+1] int32 from the PyG `batch` vector (Batch.ptr; pert_gnn.py:201-209 collation).
 * workspace >= 64 KiB is always enough for B < 2^22. */
int pert_graph_ptr(const int64_t* batch, long long N, long long B, int* ptr, void* workspace,
                   long long workspace_bytes, int* status, void* stream);

/* Level index: min hop depth from roots[g] over out-edges inside graph g, -1 if unreachable.
 * Replaces misc.py:52-63 (DFS.dfs_min_node_depth) + :107-136.  gptr[B+1], colptr/csc_dst from
 * pert_build_index, roots[B] global node ids, depth[N] int32 out. */
int pert_min_depth(const int* gptr, long long B, const int* colptr, const int* csc_dst, const int* roots,
                   int* depth, void* stream);

/* The tensor the reference stores as Data.node_depth (misc.py:159-175: unreachable -> 0, divide by the graph's max
 * depth or 1; misc.py:215,368: torch.tensor(float, dtype=long) truncation -> {0,1}) from pert_min_depth's output.
 * gptr[B+1], depth[N] int32 (-1 unreachable), node_depth[N] int64 (viewed [N,1] by the caller). */
int pert_node_depth(const int* gptr, long long B, const int* depth, int64_t* node_depth, void* stream);

/* Level-major node order inside each graph (BASELINE north_star "per-level index layout for coalescing"):
 * order[N] int32 = node ids sorted by (graph, level, id), unreachable nodes last inside their graph
 * (definition: oracle/index_oracle.py:level_order).  The reference has no counterpart (its model never reads
 * node_depth, SURVEY.md fact 3); it is a layout key for collation. */
int pert_level_order(const int* gptr, long long B, const int* depth, int* order, void* stream);

/* ---- segmented reduce (the scatter-max / scatter-add metric kernel) -----------------------------
 * out[i,:] = reduce over CSR segment i of msg rows; op 0 = sum, 1 = max; empty segment -> 0.
 * Replaces torch_geometric.utils.scatter(reduce='max'|'sum') as used by utils.softmax and
 * aggr='add' (call sites model.py:100,104) and global_add_pool (model.py:107).
 * perm NULL: msg rows already in CSR order; else row of slot p is perm[p]. */
int pert_segment_reduce_fwd(const float* msg, const int* rowptr, const int* perm, float* out, long long N, int H,
                            int op, void* stream);
int pert_segment_reduce_bwd(const float* dout, const float* msg, const float* out, const int* rowptr,
                            const int* perm, float* dmsg, long long N, int H, int op, void* stream);

/* ---- fused TransformerConv message passing -------------------------------------------------------
 * Replaces torch_geometric.nn.TransformerConv.propagate/message/aggregate (heads=1, edge_dim set,
 * root_weight) -- reference model.py:26-51 (construction), :100,:104 (calls).  q,k,v,s: [N,H] planes with
 * row stride ld (s = lin_skip(x), may be NULL); t_if [n_if,H], t_rpc [n_rpc,H] = embedding tables already
 * multiplied by the two halves of lin_edge.weight (NULL,NULL = no edge features).  out [N,H];
 * alpha [E] (CSR order) is saved for backward.  H in {4,8,16,32,64,96,128,192,256}.
 * E = number of edges, B_hint = number of graphs in the batch (0 if unknown): only used to size the shared-memory
 * node tiles of the staged kernels (csrc/tconv_tile.cu); n_rpc = rows of t_rpc. */
int pert_tconv_supported_width(int H);
int pert_tconv_fwd(const float* q, const float* k, const float* v, const float* s, int ld, const int* rowptr,
                   const int* csr_src, const int* csr_if, const int* csr_rpc, const float* t_if, const float* t_rpc,
                   float* out, int ld_out, float* alpha, int n_rpc, long long N, long long E, long long B_hint, int H,
                   void* stream);
/* g = dL/dout [N,H] (stride ld_g).  Writes dq,dk,dv [N,H] (stride ld_d), dsp [E] scratch; ACCUMULATES
 * (+=, atomics) into dt_if [n_if,H] and dt_rpc [n_rpc,H] (caller zeroes them once per step).
 * rpc_ws: caller scratch of PERT_TCONV_RPC_WS_FLOATS * N floats (per-target sums of alpha / ds by rpc type, written by
 * the target pass and consumed by the source pass of the same call) or NULL; with NULL, or n_rpc > 8, the rpc-table
 * gradient falls back to per-edge shared-memory atomics (same result, slower). */
#define PERT_TCONV_RPC_WS_FLOATS 16
int pert_tconv_bwd(const float* g, int ld_g, const float* q, const float* k, const float* v, int ld,
                   const int* rowptr, const int* csr_src, const int* csr_if, const int* csr_rpc, const int* colptr,
                   const int* csc_pos, const int* csc_dst, const float* t_if, const float* t_rpc, const float* alpha,
                   float* dq, float* dk, float* dv, int ld_d, float* dsp, float* rpc_ws, float* dt_if, float* dt_rpc,
                   int n_rpc, long long N, long long E, long long B_hint, int H, void* stream);

/* ---- dense linears (exact fp32) --------------------------------------------------------------------
 * Replace torch_geometric.nn.Linear / the lin_* of TransformerConv (model.py:26-55,105,110-112).
 * "Blocked" matrices: element (r,c) at base + (c / cb)*cbs + r*ld + (c % cb); cb <= 0 means a plain matrix.
 *   NT: C[M,Nc] (=|+=) A[M,K] . B[Nc,K]^T (+ bias) (relu)
 *   TN: C[Mc,Nc] += A[R,Mc]^T . B[R,Nc]      (atomic accumulation; weight gradients)
 *   colsum: out[c] += sum_r A[r,c]            (bias gradients) */
int pert_gemm_nt(const float* A, int lda, int a_cb, long long a_cbs, const float* B, int ldb, const float* bias,
                 float* C, int ldc, int c_cb, long long c_cbs, long long M, int Nc, int K, int relu, int accumulate,
                 void* stream);
/* a_colsum (optional, [Mc]): also accumulates a_colsum[m] += sum_r A[r,m] (the bias gradient of the same linear,
 * fused into the producer of the tensor-core kernel: A is read once for both). */
int pert_gemm_tn(const float* A, int lda, int a_cb, long long a_cbs, const float* B, int ldb, int b_cb,
                 long long b_cbs, float* C, int ldc, float* a_colsum, long long R, int Mc, int Nc, void* stream);
int pert_colsum(const float* A, int lda, int a_cb, long long a_cbs, float* out, long long R, int Cc, void* stream);

/* ---- embeddings / concat (model.py:87-97,108) -------------------------------------------------------
 * fwd: out[n,0:H] (=|+=) table[ids[n*id_stride]];  bwd: dtable[ids[n*id_stride]] += dy[n,0:H]. */
int pert_embedding_fwd(const float* table, int n_rows, const int64_t* ids, int id_stride, float* out, int ld_out,
                       long long N, int H, int accumulate, int* status, void* stream);
int pert_embedding_bwd(const float* dy, int ld_dy, const int64_t* ids, int id_stride, float* dtable, int n_rows,
                       long long N, int H, void* stream);
/* out[n, col0:col0+F] = x[n,0:F] (x dense [N,F], any F), out[n, col0+F:ld_out] = 0. */
int pert_copy_cols(const float* x, int F, float* out, int ld_out, int col0, long long N, void* stream);

/* ---- BatchNorm1d (+ fused ReLU) (model.py:33,43,101-102) ---------------------------------------------
 * training: batch statistics (biased var), running stats updated with `momentum` (unbiased var),
 * num_batches_tracked += 1; eval: running statistics.  mean/rstd [H] are outputs saved for backward. */
long long pert_bn_workspace_bytes(long long N, int H);
int pert_bn_fwd(const float* x, int ld_x, const float* gamma, const float* beta, float* running_mean,
                float* running_var, long long* num_batches_tracked, float eps, float momentum, int training,
                int relu, float* mean, float* rstd, float* y, int ld_y, long long N, int H, void* workspace,
                long long workspace_bytes, void* stream);
/* dy = grad wrt the (post-ReLU) output y; sums = [2H] scratch; dgamma/dbeta (+=) may be NULL. */
int pert_bn_bwd(const float* dy, int ld_dy, const float* y, int ld_y, const float* x, int ld_x, const float* mean,
                const float* rstd, const float* gamma, int relu, int training, float* dx, int ld_dx, float* dgamma,
                float* dbeta, float* sums, long long N, int H, void* stream);

/* ---- dropout after BatchNorm+ReLU (model.py:103, F.dropout(p, training)) ------------------------------------------
 * The step engine applies dropout inside the BatchNorm-apply kernel with a counter-based generator, so no mask is
 * stored: Philox4x32-10 with key = (seed & 0xffffffff, seed >> 32) and counter = (j & 0xffffffff, j >> 32, layer,
 * offset), where j = n * (H/4) + c/4 is the float4 index of unit (n, c) of the [N, H] output of BatchNorm `layer`;
 * output word c % 4 drops the unit iff it is < floor(p * 2^32) (computed in double; p = 1 drops everything).  Kept
 * units are scaled by 1/(1-p) in fp32.  Test / debug aid: writes that keep mask, keep[n*H + c] = 1 (kept) or 0, for
 * the given (seed, offset, layer).  p NaN or outside [0, 1] -> PERT_ERR_BADARG. */
int pert_dropout_mask(long long seed, long long offset, int layer, long long N, int H, float p, uint8_t* keep,
                      void* stream);

/* ---- local head + probability-weighted add-pool (model.py:105-107) -----------------------------------
 * local[n] = <x_n, w_local> + b_local (skipped when local NULL);
 * pool[batch[n], :] += (x_n * probs[n]) / pnn[n]   (pool [B,H] is zeroed by the call). */
int pert_pool_fwd(const float* x, int ld, const float* probs, const float* pnn, const int64_t* batch,
                  const float* w_local, const float* b_local, float* local, float* pool, long long N, long long B,
                  int H, int* status, void* stream);
int pert_pool_bwd(const float* dpool, const float* dlocal, const float* x, int ld, const float* probs,
                  const float* pnn, const int64_t* batch, const float* w_local, float* dx, int ld_dx,
                  float* dw_local, float* db_local, long long N, long long B, int H, void* stream);

/* dy[i] = 0 where y[i] <= 0 (F.relu backward, model.py:111). */
int pert_relu_bwd(const float* y, float* dy, long long n, void* stream);

/* Pinball loss (pert_gnn.py:191-193): loss[0] = mean(max(tau*e,(tau-1)*e)), e = y - yhat;
 * dyhat[B] = grad_scale * dloss/dyhat (either output may be NULL). */
int pert_pinball_loss(const int64_t* y, const float* yhat, float tau, long long B, float grad_scale, float* loss,
                      float* dyhat, void* stream);

/* Eval / epoch metrics without host syncs (pert_gnn.py:249, :284-289): acc[0] += sum|yhat - y|, acc[1] += sum(|yhat - y| / y),
 * acc[2] += B * pinball_tau(y, yhat)  (= sum of the per-graph pinball terms).  acc: 3 doubles on the device, zeroed by
 * the caller at the start of an epoch and read back once at its end. */
int pert_eval_metrics(const int64_t* y, const float* yhat, float tau, long long B, double* acc, void* stream);

/* torch.optim.Adam step (pert_gnn.py:343,247) over one flat parameter buffer; g is scaled by grad_scale. */
int pert_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, long long step, float grad_scale, void* stream);

/* ---- gradient all-reduce fused with Adam over NVLink peer memory (csrc/peer.cu) ---------------------------
 * Data-parallel form of pert_adam_step, one kernel per step and no NCCL on the step path: every rank publishes its
 * flat gradient in an IPC-shared exchange buffer and signals the peers; rank r then sums slice r of all gradients in
 * rank order (1/world of each peer's buffer over NVLink), applies Adam to that slice (m, v are only maintained for the
 * owned slice, ZeRO-1 style) and stores the new parameters into every peer's buffer; a second flag round collects the
 * other slices (replicas bit-identical by construction).  That form runs for world > 4; up to 4 ranks every rank pulls
 * whole gradients and runs the full Adam with ONE flag round (cheaper while the volume is small; measured both ways at
 * 2 and 8 GPUs).  PERT_PEER_MODE=ag|rs (environment, same on all ranks) forces one form.
 * path.  Setup: pert_peer_alloc on every rank, exchange the 64-byte handles out of band (torch.distributed
 * all_gather), pert_peer_open the peers'.  `xbufs` is a HOST array of `world` device pointers (index = rank).
 * `step` = 1, 2, ... must equal the number of calls so far on every rank (the arrival counter is monotonic).
 * A peer that never arrives makes the kernel write PERT_ERR_PEER_TIMEOUT to `status` after ~3 s instead of hanging. */
long long pert_peer_exchange_bytes(long long n);
int pert_peer_alloc(long long bytes, void** ptr, unsigned char* handle64);
int pert_peer_open(const unsigned char* handle64, void** ptr);
int pert_peer_close(void* ptr);
int pert_peer_free(void* ptr);
int pert_allreduce_adam(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                        float eps, float weight_decay, long long step, float grad_scale, void* const* xbufs, int rank,
                        int world, int* status, long long* timing, void* stream);
/* timing (optional device int64[5]): CTA 0 adds the nanoseconds (%globaltimer) it spent in (0) publishing the gradient
 * + grid arrival, (1) waiting for the peers' flags -- the slowest rank's skew plus the flag round trip --, (2) the
 * rank-ordered reduce + Adam of its slice + parameter push + second arrival, (3) waiting for the peers' slices and
 * copying them, and (4) += 1 per call: the per-phase evidence behind the scaling curve (bench.py `peer`). */

/* ---- whole-model step engine --------------------------------------------------------------------------
 * SAGEDeterministic.forward (model.py:76-114) and its backward as one call each: the same kernels as above,
 * issued back-to-back from C++ (no interpreter between launches).  Parameters live in ONE flat fp32 buffer in
 * the reference's own tensor shapes; PertModelDesc gives the offset (in floats, each 16-byte aligned) of every
 * tensor, named after the reference's state_dict keys.  Gradients go to a second flat buffer with the same
 * offsets and are ACCUMULATED (+=), like autograd.  The workspace holds packed operands, saved activations and
 * temporaries; its first pert_model_packed_bytes() bytes must be zero when first used (padding columns). */
#define PERT_MAX_CONVS 8
#define PERT_MAX_CAT 4
typedef struct PertModelDesc {
  int32_t F;        /* in_channels of the model (raw node features, 9)             model.py:13  */
  int32_t H;        /* hidden_channels                                              model.py:18  */
  int32_t n_convs;  /* max(2, num_layers)                                           model.py:24-52 */
  int32_t n_cat;    /* len(cat_dims)                                                model.py:57-60 */
  int32_t cat_rows[PERT_MAX_CAT];
  int32_t n_entry, n_if, n_rpc; /* rows of entry_embeds / interface_embeds / rpctype_embeds  model.py:63-67 */
  int32_t k0;       /* padded input width of conv 0: round_up(F + H, 8)                          */
  float bn_eps, bn_momentum;
  long long off_cat[PERT_MAX_CAT];                 /* cat_embedding.{i}.weight [rows,H] */
  long long off_entry, off_if, off_rpc;            /* *_embeds.weight                   */
  long long off_wq[PERT_MAX_CONVS], off_bq[PERT_MAX_CONVS]; /* convs.{l}.lin_query.{weight [H,Din],bias} */
  long long off_wk[PERT_MAX_CONVS], off_bk[PERT_MAX_CONVS]; /* lin_key   */
  long long off_wv[PERT_MAX_CONVS], off_bv[PERT_MAX_CONVS]; /* lin_value */
  long long off_ws[PERT_MAX_CONVS], off_bs[PERT_MAX_CONVS]; /* lin_skip  */
  long long off_we[PERT_MAX_CONVS];                         /* lin_edge.weight [H,2H] */
  long long off_bn_g[PERT_MAX_CONVS], off_bn_b[PERT_MAX_CONVS]; /* bns.{l}.weight / bias */
  long long off_local_w, off_local_b;              /* local_linear   [1,H],[1]  */
  long long off_g1_w, off_g1_b;                    /* global_linear1 [H,2H],[H] */
  long long off_g2_w, off_g2_b;                    /* global_linear2 [1,H],[1]  */
} PertModelDesc;

long long pert_model_workspace_bytes(const PertModelDesc* desc, long long N, long long E, long long B);
long long pert_model_packed_bytes(const PertModelDesc* desc);
/* Test / debug aid: offset (in floats) inside the workspace of a saved activation of the last forward:
 * which = 0: input of conv `layer` (>= 1) = post-BatchNorm-ReLU activations [N,H]; which = 1: relu(global_linear1) [B,H].
 * Lets a reference be differentiated on the same linear piece of the network (which ReLUs were active). */
long long pert_model_workspace_offset(const PertModelDesc* desc, long long N, long long E, long long B, int which,
                                      int layer);
/* bn_running: [n_convs-1][2][H] (running_mean | running_var), bn_nbt: [n_convs-1] int64 (either may be NULL in
 * training mode); index arrays from pert_build_index (built with edge_attr); probs/pnn [N] fp32.
 * Outputs: global_pred [B], local_pred [N] (NULL to skip). */
/* Optional measurement probe: the engine records the two caller-created cudaEvent_t around ONE kernel family of ONE
 * layer, on the launching stream (bench.py: in-step duration of the dominant kernel).  kernel: 1 = fused conv forward,
 * 2 = fused conv backward (target + source pass), 3 = node-linear forward GEMM, 4 = weight-gradient GEMM,
 * 5 = data-gradient GEMM, 6 = BatchNorm apply (+ fused dropout) of BatchNorm `layer`.  NULL = no probe. */
typedef struct PertProbe {
  int32_t kernel, layer;
  void* ev_start;
  void* ev_stop;
} PertProbe;
int pert_model_forward(const PertModelDesc* desc, const float* params, float* bn_running, long long* bn_nbt,
                       const float* x, const int64_t* cat_X, const int64_t* entry_id, const float* probs,
                       const float* pnn, const int64_t* batch, long long N, long long E, long long B,
                       const int* rowptr, const int* csr_src, const int* csr_if, const int* csr_rpc, void* workspace,
                       long long workspace_bytes, int training, float dropout_p, long long* rng_state,
                       float* global_pred, float* local_pred, int* status, const PertProbe* probe, void* index_ready,
                       void* stream);
/* index_ready: optional cudaEvent_t recorded (on another stream) after the graph index was built: the forward waits
 * for it only right before the first attention kernel, so the index build overlaps the parameter pack, the input
 * prologue and the first GEMM.  NULL = the index is already complete in `stream` order.
 * dropout_p in [0, 1] (else PERT_ERR_BADARG before any launch): with training and dropout_p > 0 every BatchNorm+ReLU
 * output is passed through dropout (see pert_dropout_mask for the mask).  rng_state: caller-owned device int64[2] =
 * (seed, offset), read by the BatchNorm kernels; the forward then adds 1 to the offset ON THE DEVICE after the last of
 * them, so a replayed CUDA graph draws fresh masks on every replay.  May be NULL when training == 0 or dropout_p == 0.
 * Must follow pert_model_forward on the same workspace, with the same training / dropout_p.  d_global [B], d_local [N]
 * or NULL. */
int pert_model_backward(const PertModelDesc* desc, const float* params, float* grads, const int64_t* cat_X,
                        const int64_t* entry_id, const float* probs, const float* pnn, const int64_t* batch,
                        long long N, long long E, long long B, const int* rowptr, const int* csr_src,
                        const int* csr_if, const int* csr_rpc, const int* colptr, const int* csc_pos,
                        const int* csc_dst, void* workspace, long long workspace_bytes, int training, float dropout_p,
                        const float* d_global, const float* d_local, const PertProbe* probe, void* stream);

/* ---- device-side batch assembly from a resident pattern store (csrc/store.cu) ---------------------------------------
 * Replaces the host-side sample assembly + collation + per-step probability expansion of the reference:
 * get_entry_data / get_x / get_cat_X / get_node_depth / get_edge_index / get_edge_attr / get_pattern_num_nodes
 * (pert_gnn.py:40-173), torch_geometric DataLoader collation (:201-209) and transform_pattern_probs (:122-131,
 * :220-230).  All pointers are caller-owned device arrays, built once from the reference's artefacts
 * (runtime2graph, entry2runtimes, resource_df, tr2data -- pert_gnn.py:297-305) by pert_gnn_kdd23_b200/store.py.
 *   patterns p = 0..n_pat-1 (the runtime ids in the order the store assigned):
 *     pat_nptr/pat_eptr [n_pat+1] node / edge offsets into the concatenated arrays;  pat_ms [sum n] = ms_id (cat_X);
 *     pat_depth [sum n] = node_depth;  pat_last [sum n] = 1 iff the node is the LAST one of its ms inside the pattern
 *     (get_x's ms2nid dict, pert_gnn.py:54-65);  pat_src/pat_dst [sum e] pattern-local edge_index;  pat_attr [sum e, attr_cols]
 *   entries: ent_ptr [n_ent+1] into ent_pat (pattern index) / ent_prob (float32 probability), in the dict order of
 *     entry2runtimes[entry];  ent_nodes / ent_edges [n_ent] totals over the entry's patterns
 *   resources: res_keys [n_res] sorted int64 = timestamp * n_ms + ms, res_vals [n_res, 8] float32,
 *     ms_has_res [n_ms] = 1 iff ms has a row at ANY timestamp (pert_gnn.py:138)
 *   traces: trace_entry [n_traces] int32, trace_ts [n_traces] int64, trace_y [n_traces] int64. */
typedef struct PertStore {
  int32_t n_pat, n_ent, n_res, n_ms, attr_cols;
  long long n_traces;
  const int32_t *pat_nptr, *pat_eptr;
  const int64_t *pat_ms, *pat_depth;
  const uint8_t* pat_last;
  const int32_t *pat_src, *pat_dst;
  const int64_t* pat_attr;
  const int32_t *ent_ptr, *ent_pat;
  const float* ent_prob;
  const int32_t *ent_nodes, *ent_edges;
  const int64_t* res_keys;
  const float* res_vals;
  const uint8_t* ms_has_res;
  const int32_t* trace_entry;
  const int64_t *trace_ts, *trace_y;
} PertStore;
/* Output = the collated Batch of pert_gnn.py:163-173 + PyG collate + the per-node probability of :220-230. */
typedef struct PertBatchOut {
  float* x;                  /* [N, 9]  */
  int64_t* cat_X;            /* [N, 1]  */
  int64_t* node_depth;       /* [N, 1]  */
  float* pattern_num_nodes;  /* [N, 1]  */
  float* rt_probs;           /* [N, 1]  per-node pattern probability (transform_pattern_probs) */
  int64_t* batch;            /* [N]     */
  int64_t* edge_index;       /* [2, E]  */
  int64_t* edge_attr;        /* [E, attr_cols] */
  int64_t* entry_id;         /* [B]     */
  int64_t* y;                /* [B]     */
  int64_t* ptr;              /* [B+1]   */
  float* pattern_probs;      /* [sum_b patterns(entry_b), 1] */
} PertBatchOut;
/* trace_ids [B] int64 (device): which traces form the batch.  N, E = node / edge totals of the batch (the caller sizes
 * the outputs from its host copy of ent_nodes / ent_edges -- no device sync); offsets: int32 scratch of 3 * (B + 1).
 * status: PERT_ERR_RANGE for a trace id out of range or a (timestamp, ms) row missing for a resourced ms (the
 * reference raises KeyError there). */
int pert_store_assemble(const PertStore* store, const int64_t* trace_ids, long long B, long long N, long long E,
                        int* offsets, const PertBatchOut* out, int* status, void* stream);

/* ---- PERT-graph construction (SURVEY 8f row N2) ---------------------------------------------------------------
 * Replaces misc.py:221-319 (GraphConstruct.get_pert_edge_index) for T traces at once.  Input: the cleaned span rows
 * (what misc.py:87-105 drop_wrong_edges leaves) of all traces concatenated, row_ptr[T+1]; per row um, dm, interface,
 * rpctype, t_start (= timestamp), t_end (= endTimestamp), all int64 [R]; root_ms[T] (misc.py:138-142).
 * Output per trace: nodes = 2*rows + distinct microservices, edges = 4*rows (edge slots of trace t start at
 * 4*row_ptr[t]); ms_id[N] = sorted_span_id; edge_index[2,4R] with trace-local node ids (global_ids = 0, the
 * per-pattern tensors the reference stores) or batch-global ids (global_ids = 1); edge_attr[4R,4] =
 * [interface, rpctype, call, same_ms]; root_nid[T] = GLOBAL id of stage 0 of the root microservice (-1 + PERT_ERR_RANGE
 * in status if the root is absent; the reference raises KeyError).  Node numbering is the canonical order documented
 * in csrc/pertgraph.cu (the reference's is pandas / set iteration order); edge order is the reference's.
 * Two passes so the caller can size the outputs: _count writes node_cnt[T]; the caller scans it into node_ptr[T+1].
 * max_rows >= the longest trace (<= PERT_PERT_GRAPH_MAX_ROWS); a longer trace sets PERT_ERR_RANGE. */
#define PERT_PERT_GRAPH_MAX_ROWS 2048
int pert_pert_graph_count(const int64_t* row_ptr, long long T, const int64_t* um, const int64_t* dm, int max_rows,
                          int64_t* node_cnt, int* status, void* stream);
int pert_pert_graph_build(const int64_t* row_ptr, long long T, long long R, const int64_t* um, const int64_t* dm,
                          const int64_t* interface, const int64_t* rpctype, const int64_t* t_start,
                          const int64_t* t_end, const int64_t* root_ms, const int64_t* node_ptr, int max_rows,
                          int global_ids, int64_t* ms_id, int64_t* edge_index, int64_t* edge_attr, int64_t* root_nid,
                          int* status, void* stream);
/* Span graph of T traces (misc.py:190-219 get_span_edge_index; `--graph_type span` is pert_gnn.py's default): nodes =
 * the trace's sorted unique microservice ids (ms_id[N], N from pert_span_graph_count), edge_index[2,R] = positions of
 * um / dm in that list (one edge per row, table order; edge slots of trace t start at row_ptr[t]), edge_attr[R,2] =
 * [interface, rpctype], root_nid[T] as above.  Bit-identical to the reference's tensors. */
int pert_span_graph_count(const int64_t* row_ptr, long long T, const int64_t* um, const int64_t* dm, int max_rows,
                          int64_t* node_cnt, int* status, void* stream);
int pert_span_graph_build(const int64_t* row_ptr, long long T, long long R, const int64_t* um, const int64_t* dm,
                          const int64_t* interface, const int64_t* rpctype, const int64_t* root_ms,
                          const int64_t* node_ptr, int max_rows, int global_ids, int64_t* ms_id, int64_t* edge_index,
                          int64_t* edge_attr, int64_t* root_nid, int* status, void* stream);

/* ---- trace catalogue (csrc/catalogue.cu; Python: pert_gnn_kdd23_b200/catalogue.py) -------------------------------
 * Replaces the integer-coded part of preprocess.py:main() (:269-375): the per-trace pattern strings and their
 * factorize (:280-293), tr2ts_map (:39), tr2delay (:290-292), the per-entry Python loop (:295-367) and the
 * normalisation (:371-375).  All arrays int64 unless stated.  Traces are numbered by ascending traceid; `perm[R]` is
 * the row order grouped by traceid (stable, file order inside a trace), row_ptr[T+1] its trace offsets.
 *
 * run_flags: flag[i] = (i == 0 || key[i] != key[i-1]); mark[i] = flag[i] ? i : 0 (mark may be NULL). */
int pert_catalogue_run_flags(const int64_t* key, long long n, int64_t* flag, int64_t* mark, void* stream);
/* Per trace (one warp each, no row limit): nrows, hash = order-sensitive 64-bit hash of the (um, dm, interface) row
 * sequence (:280-289) & hash_mask, y = max |rt| (:290-292), ts_bucket = floor(min timestamp / 30000) * 30000 (:39),
 * trace_entry = entryid of the first row; PERT_ERR_RANGE in status if the trace's rows carry different entryids. */
int pert_catalogue_summary(const int64_t* perm, const int64_t* row_ptr, long long T, const int64_t* um,
                           const int64_t* dm, const int64_t* interface, const int64_t* rt, const int64_t* timestamp,
                           const int64_t* entryid, unsigned long long seed, unsigned long long hash_mask,
                           int64_t* nrows, int64_t* hash, int64_t* y, int64_t* ts_bucket, int64_t* trace_entry,
                           int* status, void* stream);
/* Exact check of a grouping by key (:293 factorize compares the strings): order[T] = traces sorted by (key, trace),
 * head[i] = sorted position of the first member of i's run.  mismatch[order[i]] = 1 iff that trace's sequence differs
 * from its head's; n_mismatch (device uint64, zeroed by the call) counts them. */
int pert_catalogue_verify(const int64_t* order, const int64_t* head, long long T, const int64_t* perm,
                          const int64_t* row_ptr, const int64_t* um, const int64_t* dm, const int64_t* interface,
                          int32_t* mismatch, unsigned long long* n_mismatch, void* stream);
/* For every trace with mismatch[t]: key[t] = mix(key[t], sequence hash with `seed` & hash_mask). */
int pert_catalogue_rekey(const int64_t* perm, const int64_t* row_ptr, long long T, const int64_t* um,
                         const int64_t* dm, const int64_t* interface, const int32_t* mismatch, unsigned long long seed,
                         unsigned long long hash_mask, int64_t* key, void* stream);
/* canon[order[i]] = order[head[i]] (first trace of the pattern), first[t] = (canon[t] == t). */
int pert_catalogue_canon(const int64_t* order, const int64_t* head, long long T, int64_t* canon, int64_t* first,
                         void* stream);
/* rid[t] = first_incl[canon[t]] - 1 (first_incl = inclusive scan of `first`): runtime ids in factorize order (:293). */
int pert_catalogue_runtime_ids(const int64_t* canon, const int64_t* first_incl, long long T, int64_t* rid,
                               void* stream);
/* eorder[T] = traces in (entry, traceid) order (the order of :295-299), eidx[j] = rank of the entry of eorder[j].
 * Per pattern (P of them): rep_epos = smallest j showing it (its representative, :317-318), occurrences (:342);
 * pair_key[j] = eidx[j] * P + rid[eorder[j]]. */
int pert_catalogue_patterns(const int64_t* eorder, const int64_t* eidx, long long T, const int64_t* rid, long long P,
                            int64_t* rep_epos, int64_t* occurrences, int64_t* pair_key, void* stream);
/* (entry, pattern) pairs (:310-316): pstart[NP] = run starts of the stably sorted pair_key, pidx[T] its sort indices.
 * Per pair: count, first = entry-order position of its first trace, pair_entry (entry rank), pair_rid. */
int pert_catalogue_pairs(const int64_t* pstart, long long NP, long long T, const int64_t* pidx, const int64_t* eorder,
                         const int64_t* rid, const int64_t* eidx, int64_t* count, int64_t* first, int64_t* pair_entry,
                         int64_t* pair_rid, void* stream);
/* Pairs sorted by `first` (entry-major, then first appearance): prob (double) = count / traces of the entry
 * (:371-375, bit-identical to Python's int / int), ent_ptr[E+1] = the entry CSR over the pairs; ent_start[E] = first
 * entry-order position of every entry. */
int pert_catalogue_probs(const int64_t* pair_entry, const int64_t* count, long long NP, const int64_t* ent_start,
                         long long E, long long T, double* prob, int64_t* ent_ptr, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PERTGNN_H_ */
