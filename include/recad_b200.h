/* recad_b200.h -- C ABI of the B200-native RecAD victim hot path.
 *
 * The reference (gusye1234/recad) is pure Python over stock torch ops: it has NO
 * FFI of its own.  Each entry point below therefore cites the reference
 * FUNCTION it replaces (paths relative to the reference checkout); the Python
 * classes in recad_b200/ bind these with ctypes and re-expose the reference's
 * own plugin interface (model.from_config('victim', ..).I(), dataset
 * .generate_batch()/.inject_data(), workflow .execute()).  INTEGRATION.md shows
 * the binding a maintainer would add on the reference side.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types;
 *   - every pointer marked [dev] is a device pointer on the CURRENT CUDA device,
 *     [host] a host pointer; buffers are owned by the caller;
 *   - `stream` is a cudaStream_t passed as void*; all device work is enqueued
 *     on it asynchronously unless the function says "synchronises";
 *   - return value: 0 = ok, < 0 = error (RECAD_ERR_*), message via
 *     recad_last_error() (thread-local); no exception crosses the boundary;
 *   - indices: users/items/samples int64 as in the reference; CSR column
 *     indices int32 (N < 2^31), row pointers int64;
 *   - all floating point is IEEE fp32 (no fast-math), loss accumulators fp64.
 */
#ifndef RECAD_B200_H
#define RECAD_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RECAD_ABI_VERSION 2

enum {
  RECAD_OK = 0,
  RECAD_ERR_ARG = -1,         /* bad argument (null pointer, negative size, id out of range) */
  RECAD_ERR_CUDA = -2,        /* a CUDA runtime call or kernel launch failed */
  RECAD_ERR_UNSUPPORTED = -3, /* shape not compiled (e.g. embedding width) */
  RECAD_ERR_OVERFLOW = -4,    /* size exceeds an index type */
  RECAD_ERR_SCRATCH = -5      /* scratch buffer too small */
};

int recad_abi_version(void);
const char* recad_last_error(void);
/* sm_count / cc of the current device; fails unless it is an sm_100 part. */
int recad_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------ *
 * Graph construction  (recad/dataset/implicit.py:206-213, 243-298, 320-326)
 * ------------------------------------------------------------------------ */

/* Bytes of [dev] scratch recad_csr_build_structure needs for n_edges edges. */
int64_t recad_csr_build_scratch_bytes(int64_t n_edges, int64_t n_users, int64_t n_items);

/* Edge list -> structure of the symmetric bipartite adjacency over
 * N = n_users + n_items rows, entries ordered by (row, col) exactly as
 * `Graph.coalesce()` orders them (implicit.py:296).  Duplicate (u, i) pairs are
 * merged and counted, as scipy's csr_matrix sums them (implicit.py:206-209).
 *   users, items [dev] int64[n_edges]
 *   rowptr  [dev] int64[N + 1]            out
 *   colidx  [dev] int32[2 * n_edges]      out (first nnz valid)
 *   mult    [dev] float[2 * n_edges]      out multiplicity of each entry (1.0 normally)
 *   degree  [dev] int32[N]                out row sums of multiplicities (implicit.py:269)
 *   nnz_out [host] int64*                 out number of distinct directed entries
 * Synchronises the stream (nnz is returned to the host). */
int recad_csr_build_structure(const int64_t* users, const int64_t* items, int64_t n_edges,
                              int64_t n_users, int64_t n_items, int64_t* rowptr, int32_t* colidx,
                              float* mult, int32_t* degree, int64_t* nnz_out, void* scratch,
                              int64_t scratch_bytes, void* stream);

/* vals[e] = (d_inv[row] * mult[e]) * d_inv[col]: two successive fp32 products, the
 * order scipy's D.dot(A).dot(D) evaluates them in (implicit.py:273-276).  d_inv
 * comes from the host: the reference's `np.power(rowsum + 1e-14, -0.5)` in
 * float32 is not reproducible by any device expression (SURVEY.md section 7). */
int recad_csr_normalize(const int64_t* rowptr, const int32_t* colidx, const float* mult,
                        const float* d_inv, int64_t n_rows, float* vals, void* stream);

/* In-place fake-user injection (implicit.py:482-494 + base.py:108-118, which the
 * reference implements as a full dataset rebuild): append F user rows after row
 * n_users-1.  Item rows shift down by F, item column ids in user rows shift by
 * +F, every touched item row gains the new user ids at its END (they are larger
 * than all existing user ids, so (row, col) order is preserved).  No sort.
 *   fake_rowptr [dev] int64[F + 1], fake_items [dev] int32[]: per fake user, its
 *   DISTINCT items ascending (np.where order, implicit.py:109).
 * new_* buffers must hold nnz_old + 2 * fake_rowptr[F] entries. */
int recad_csr_append_users(const int64_t* rowptr, const int32_t* colidx, const float* mult,
                           int64_t n_users, int64_t n_items, int64_t n_fake,
                           const int64_t* fake_rowptr, const int32_t* fake_items, int64_t n_fake_edges,
                           int64_t* new_rowptr, int32_t* new_colidx, float* new_mult,
                           int32_t* new_degree, void* scratch, int64_t scratch_bytes, void* stream);
int64_t recad_csr_append_scratch_bytes(int64_t n_users, int64_t n_items, int64_t n_fake, int64_t n_fake_edges);

/* The weights -> values chain of the normalisation above for caller-supplied per-entry weights w [dev] float[nnz]
 * (in place of mult):  vals_k = d_r w_k d_c,  d_r = (s_r + 1e-14)^(-1/2).
 * recad_csr_row_sums: sums [dev] float[n_rows] = s_r, the weights of row r added in a fixed order in double and rounded
 *   to float once (the host then evaluates d_inv from them, as from the degrees).
 * recad_csr_normalize_backward: for a square, structurally symmetric matrix, the gradient gw [dev] float[nnz] of
 *   sum_k gv_k vals_k:  gw_k = gv_k d_r d_c - 0.5 d_r^3 P_r,  P_r = sum over row r's entries k' of
 *   (gv_k' w_k' + gv_{T k'} w_{T k'}) d_{c(k')}, where tperm [dev] int64[nnz] maps entry (r, c) to the position of (c, r).
 *   Two passes: a per-row reduction into coef [dev] float[n_rows] (work) in a fixed order, then a per-entry epilogue;
 *   deterministic.  d_inv [dev] float[n_rows] is the forward's.
 * Both read rowptr[n_rows] back (synchronising the stream) and return RECAD_ERR_ARG unless it equals nnz. */
int recad_csr_row_sums(const int64_t* rowptr, const float* w, int64_t n_rows, int64_t nnz, float* sums, void* stream);
int recad_csr_normalize_backward(const int64_t* rowptr, const int32_t* colidx, const int64_t* tperm, const float* w,
                                 const float* d_inv, const float* gv, int64_t n_rows, int64_t nnz, float* coef, float* gw,
                                 void* stream);

/* ------------------------------------------------------------------------ *
 * Propagation  (recad/model/victim/lightgcn.py:82-113 `computer`; its autograd
 * backward is the same product because A_hat is symmetric)
 * ------------------------------------------------------------------------ */

/* A CSR matrix plus its work plan.  rowptr / colidx / vals are the canonical arrays (bit-exact against the
 * reference's coalesced graph, implicit.py:295-296); the kernels read two derived arrays:
 *   cv       [dev] int32[nnz, 2]   interleaved (colidx, bits of vals) pairs (recad_spmm_pack_cv)
 *   seg_meta [dev] int32[n_seg, 4] the PLAN: one entry per segment = at most 1024 consecutive entries of one row,
 *            {first entry low 32 bits, high 32 bits, row, (slot + 1) << 11 | count}; a segment is the unit of work
 *            of one warp.  Rows cut into several segments (long rows, or item rows cut at L2-sized column blocks)
 *            own consecutive partial-sum slots; slot = -1 (field 0) for single-segment rows.  Built by
 *            recad_b200.ops.PackedPlan (index arithmetic, once per graph).
 * Rectangular matrices are allowed (colidx indexes rows of X), which is what the shards of the multi-GPU path use.
 * A matrix must not be used by two launches at the same time (row_cnt / partials are per-matrix scratch). */
typedef struct recad_csr {
  int64_t n_rows;
  int64_t n_cols;
  int64_t nnz;
  const int64_t* rowptr;   /* [dev] int64[n_rows + 1] */
  const int32_t* colidx;   /* [dev] int32[nnz] */
  const float* vals;       /* [dev] float[nnz] */
  const void* cv;          /* [dev] int32[nnz, 2] */
  int64_t n_seg;           /* plan: number of segments (>= n_rows) */
  const void* seg_meta;    /* [dev] int32[n_seg, 4] */
  int64_t n_mrow;          /* rows with > 1 segment */
  const void* row_mseg;    /* [dev] int32[n_rows, 2] (first partial slot, number of segments) of multi-segment rows */
  int32_t* row_cnt;        /* [dev] int32[n_rows] arrival counters, zero between launches */
  float* partials;         /* [dev] float[n_slot * D] scratch for multi-segment rows */
} recad_csr;

/* cv[e] = (colidx[e], bits of vals[e]). */
int recad_spmm_pack_cv(const int32_t* colidx, const float* vals, int64_t nnz, void* cv, void* stream);

/* Y = A X (written if Y != NULL) and Z = alpha * (C + A X) (written if Z != NULL;
 * C == NULL means 0; Z may alias C).  X, Y, C, Z: [dev] float[rows, D] row-major,
 * 16-byte aligned.  This one kernel is every layer of the forward propagate
 * fused with the running layer mean (lightgcn.py:99-111: Y = next layer,
 * Z = accumulated mean) and every Horner step of the backward (Z = g + A t). */
int recad_spmm(const recad_csr* A, const float* X, float* Y, const float* C, float* Z,
               float alpha, int32_t D, void* stream);

/* SDDMM, the gradient of an SpMM with respect to the matrix's values: out[k] = alpha * <G[r_k], X[c_k]> for every stored
 * entry k = (r_k, c_k) of A (accumulate != 0: out[k] += ...).  G [dev] float[n_rows, D], X [dev] float[n_cols, D], 16-byte
 * aligned; out [dev] float[nnz] in A's CSR entry order.  Driven by A's plan (reads seg_meta and colidx, not cv or vals);
 * every entry has one writer: atomic-free and bit-stable.  Same bytes as one SpMM (no-reuse model). */
int recad_csr_sddmm(const recad_csr* A, const float* G, const float* X, int32_t D, float alpha, int32_t accumulate,
                    float* out, void* stream);

/* Sharded path (SURVEY.md 8e): Y = A X where row i is not stored locally but written, as soon as it is
 * finished, to dst[i / slice_rows] + (i % slice_rows) * D.  dst[r] [host array of n_dst <= 16 device pointers]
 * is rank r's staging block for THIS sender, mapped into this process over NVLink (torch symmetric memory):
 * the partial item rows of lightgcn.py:99-108 travel to their owner inside the SpMM epilogue instead of
 * through a separate all-reduce.  D in {32, 64, 128}. */
int recad_spmm_scatter(const recad_csr* A, const float* X, float* const* dst, int32_t n_dst,
                       int64_t slice_rows, int32_t D, void* stream);
/* The owner's half of that exchange: out[r][e] = sum over s < n_src of stage[s * src_stride + e], e < n_floats,
 * for every r < n_out (<= 16): partial rows summed in rank order (identical bits on every replica) and stored
 * directly into each peer's table.  multicast != 0: n_out == 1 and out[0] is an NVSwitch multicast address
 * (same offset in every rank's buffer): one multimem.st per element instead of n_out peer stores.
 * The caller brackets it with cross-device barriers. */
int recad_peer_reduce_bcast(const float* stage, int32_t n_src, int64_t src_stride, int64_t n_floats,
                            float* const* out, int32_t n_out, int32_t multicast, void* stream);

/* ------------------------------------------------------------------------ *
 * LightGCN BPR step  (recad/model/victim/lightgcn.py:122-172)
 * ------------------------------------------------------------------------ */

/* Fused gather + dot + softplus + L2-reg + gradient scatter for one batch.
 *   O [dev] float[N, D] propagated mean (users first), E [dev] float[N, D] ego table
 *   samples [dev] int64[*, 3] rows (user, pos, neg) (item ids WITHOUT the n_users offset);
 *   perm [dev] int64[B] row index of each of the B samples of this batch (NULL = rows 0..B-1)
 *   grad_scale = 1 / (L + 1): folded into the scattered gradient so that gO is
 *     already d loss / d (sum of layers)
 *   gO  [dev] float[N, D]  += ; must be zeroed by the caller
 *   cnt [dev] float[N]     += number of times each row occurs in the batch
 *                             (drives the L2-reg gradient lambda/B * cnt * E in Adam)
 *   loss_acc [dev] double[4]: [0] += sum softplus(x), [1] += sum (|E_u|^2+|E_p|^2+|E_n|^2),
 *                             [3] is set non-zero (as an int) if a sample id is out of range */
int recad_bpr_fwd_bwd(const float* O, const float* E, int64_t n_users, int64_t n_items,
                      const int64_t* samples, const int64_t* perm, int64_t B, int64_t B_norm,
                      float grad_scale, float* gO, float* cnt, double* loss_acc, int32_t D,
                      void* stream);
/* B_norm: the batch size the mean loss / gradients are normalised by.  B_norm == B on one GPU; in the
 * user-sharded multi-GPU path each rank passes only its own users' B rows of a global batch of B_norm. */

/* z = a * x + b * y over n floats (n % 4 == 0; z may alias x or y): the layer-mean / Horner accumulation of the
 * sharded path, where the item rows of an SpMM result must be all-reduced BEFORE they are accumulated. */
int recad_axpby(float* z, float a, const float* x, float b, const float* y, int64_t n, void* stream);

/* Dense Adam over n elements (torch.optim.Adam defaults, lightgcn.py:17-19):
 *   G = g + reg_scale * cnt[i / D] * p   (cnt may be NULL)
 *   m = b1 m + (1-b1) G; v = b2 v + (1-b2) G^2;
 *   p -= (lr / (1-b1^t)) * m / (sqrt(v) / sqrt(1-b2^t) + eps)
 * Every element is updated every step (Embedding(sparse=False), lightgcn.py:40-45). */
int recad_adam(float* p, const float* g, const float* cnt, float reg_scale, float* m, float* v,
               int64_t n, int32_t D, float lr, float b1, float b2, float eps, int64_t step,
               void* stream);

/* State of one LightGCN victim on one device; all buffers caller-owned. */
typedef struct recad_lightgcn {
  const recad_csr* graph;  /* N x N normalised adjacency */
  int64_t n_users, n_items;
  int32_t D, n_layers;
  float lambda, lr, beta1, beta2, eps;
  int32_t _pad;
  float* E;                /* [dev] float[N, D] ego embeddings (users then items) */
  float* m;                /* [dev] float[N, D] Adam first moment */
  float* v;                /* [dev] float[N, D] Adam second moment */
  float* O;                /* [dev] float[N, D] propagated mean (output of `computer`) */
  float* X0;               /* [dev] float[N, D] work: layer ping */
  float* X1;               /* [dev] float[N, D] work: layer pong */
  float* g;                /* [dev] float[N, D] work: gradient wrt the layer sum */
  float* cnt;              /* [dev] float[N]    work: batch multiplicities */
  double* loss_acc;        /* [dev] double[4]   {sum softplus, sum sq, epoch loss sum, spare} */
  const recad_csr* graph_t;/* NULL (the usual case: A_hat is symmetric, the backward is the same product), or the TRANSPOSE of
                            * `graph` for the backward pass -- graph dropout (lightgcn.py:62-80) drops (u, i) and (i, u)
                            * independently, so the dropped matrix is not symmetric */
} recad_lightgcn;

/* O = mean_k A^k E (lightgcn.py:82-113).  L fused SpMMs, nothing else. */
int recad_lightgcn_propagate(const recad_lightgcn* st, void* stream);

/* One epoch of `train_step` (lightgcn.py:132-172) over pre-sampled triples
 * samples [dev] int64[n_samples, 3] = (user, pos, neg) rows in SAMPLER order, visited in the
 * order perm [dev] int64[n_samples] (the epoch shuffle of implicit.py:18-35; NULL = identity):
 * batch b is rows perm[b*batch .. (b+1)*batch) (last ragged, implicit.py:38-47).  The shuffle
 * is an index indirection inside the kernels, the sample array is never rewritten.
 * Per batch: propagate, BPR, Horner backward, dense Adam.
 * step0 = Adam steps taken before this epoch.  The mean of the per-batch losses
 * is left in loss_acc[2] / n_batches: read it with ONE device->host copy after
 * the epoch (the reference syncs once per batch, lightgcn.py:169). */
int recad_lightgcn_train_epoch(const recad_lightgcn* st, const int64_t* samples, const int64_t* perm,
                               int64_t n_samples, int64_t batch, int64_t step0, void* stream);

/* 32-bit forms of the two calls above (samples [dev] int32[*, 3], perm [dev] int32[*]): what the large-epoch path
 * uses -- the host sampler emits 32-bit arrays (recad_mt19937_pairwise_soa + recad_samples_expand), halving the
 * host->device traffic of an epoch. */
int recad_bpr_fwd_bwd_i32(const float* O, const float* E, int64_t n_users, int64_t n_items,
                          const int32_t* samples, const int32_t* perm, int64_t B, int64_t B_norm,
                          float grad_scale, float* gO, float* cnt, double* loss_acc, int32_t D, void* stream);
int recad_lightgcn_train_epoch_i32(const recad_lightgcn* st, const int32_t* samples, const int32_t* perm,
                                   int64_t n_samples, int64_t batch, int64_t step0, void* stream);

/* Candidate users of the evaluation (normal.py:133-143), built on the device: users with a non-empty train row (or, when
 * is_key [dev] uint8[n_users] is given, the users that are KEYS of train_dict), none of the targets in their train
 * row, and at least one candidate item left; ascending ids into users_out [dev] int64[n_users], count into *n_out [host]
 * (the call synchronises the stream to return it).  train rows sorted ascending.  targets [dev] int32[n_targets].
 * scratch [dev]: recad_eligible_users_scratch_bytes(n_users) bytes. */
int64_t recad_eligible_users_scratch_bytes(int64_t n_users);
int recad_eligible_users(const int64_t* train_rowptr, const int32_t* train_col, int64_t n_users, int64_t n_items,
                         const int32_t* targets, int32_t n_targets, const uint8_t* is_key, int64_t* users_out,
                         int64_t* n_out, void* scratch, int64_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * User-sharded LightGCN epoch (SURVEY.md 8e; same math as recad_lightgcn_train_epoch,
 * lightgcn.py:82-172), one process per GPU, exchanges over NVLink peer memory only.
 * ------------------------------------------------------------------------ */

/* One epoch's samples on the device, in either form (the other form's pointers NULL):
 *   rows   int64[n_samples, 3] (GLOBAL user, pos, neg) in sampler order + perm64 int64[n_samples] (or NULL = identity)
 *   users / rel / negs  uint32[n_samples] as recad_mt19937_pairwise_soa emits them (GLOBAL user id, index of the
 *          positive inside the user's row, negative) + perm32 int32[n_samples] (or NULL = identity).
 * Every rank holds the WHOLE epoch (0.8 GB at 50 M samples) and keeps the samples whose user it owns. */
typedef struct recad_epoch_samples {
  int64_t n_samples;
  const int64_t* rows;
  const int64_t* perm64;
  const uint32_t* users;
  const uint32_t* rel;
  const uint32_t* negs;
  const int32_t* perm32;
} recad_epoch_samples;

/* State of one rank.  Tables are [n_users_local + n_items, D] (own users first, then a replica of ALL items).
 * Everything peers read or write lives in one symmetric block per rank, mapped into every process
 * (torch.distributed._symmetric_memory): peer_base[r] is rank r's block as mapped HERE, off_* are byte offsets inside it:
 *   off_X0 / off_X1 / off_O / off_g : float[max_r(n_users_local_r) + n_items, D]   layer ping / pong, propagated mean, gradient
 *   off_cnt    : float[max_r(n_users_local_r) + n_items]        batch multiplicities
 *   off_stage  : float[2, world, slice, D]   (double buffered) slot s receives rank s's partial rows of the items THIS rank owns
 *   off_signal : uint32[64], zero-initialised: [0, world) barrier pad, [32] barrier epoch, [33] timeout flag
 * Rank r owns items [r * slice, (r + 1) * slice).  mc_base: NVSwitch multicast mapping of the block (one store lands in
 * every rank's copy) or NULL; used only when every rank has the same n_users_local. */
typedef struct recad_lightgcn_shard {
  int32_t rank, world, D, n_layers;
  int64_t n_users_local, n_items, user_lo, slice;
  float lambda, lr, beta1, beta2, eps;
  int32_t _pad;
  const recad_csr* g_user;     /* [n_users_local x n_items]: own user rows (gather the item replica) */
  const recad_csr* g_item;     /* [n_items x n_users_local]: item rows over own users (partial sums) */
  const int64_t* pos_rowptr;   /* [dev] int64[n_users_local + 1]: own users' sorted distinct positives (may be NULL with `rows`) */
  const int32_t* pos_col;      /* [dev] int32[]: item id + pos_col_offset */
  int64_t pos_col_offset;
  float* E;                    /* [dev] local tables */
  float* m;
  float* v;
  double* loss_acc;            /* [dev] double[4] as in recad_lightgcn; partial sums of THIS rank's samples */
  void* const* peer_base;      /* [host] void*[world] */
  void* mc_base;
  const int64_t* peer_users;   /* [host] int64[world]: n_users_local of every rank */
  int64_t off_X0, off_X1, off_O, off_g, off_cnt, off_stage, off_signal;
} recad_lightgcn_shard;

/* O = mean_k A^k E over the sharded matrix: L x (item-row SpMM pushing partial rows to their owners | user-row SpMM |
 * barrier | owner reduce + store into every replica | barrier).  Collective: every rank must call it. */
int recad_lightgcn_shard_propagate(const recad_lightgcn_shard* st, void* stream);
/* One epoch over the GLOBAL sample list: per batch propagate, BPR on the rank's own users' samples (1/B of the global
 * batch), gradient-block exchange, Horner backward, dense Adam on the own user rows and the item replica.  Nothing
 * synchronises with the host; loss_acc[2] holds the rank's part of the sum of batch losses afterwards (sum over ranks /
 * n_batches = the epoch loss).  trace_ms [host] double[8] or NULL: when given, the call synchronises the stream and
 * returns the time spent per phase {0 item-row SpMM + push, 1 user-row SpMM, 2 barriers, 3 slice reduce + store,
 * 4 zeroing, 5 BPR, 6 gradient exchange, 7 Adam} (CUDA events). */
int recad_lightgcn_shard_train_epoch(const recad_lightgcn_shard* st, const recad_epoch_samples* ep, int64_t batch,
                                     int64_t step0, double* trace_ms, void* stream);
/* state2 [host] uint32[2] = {barriers passed, 1 if a barrier wait ever timed out}; synchronises the stream. */
int recad_lightgcn_shard_barrier_state(const recad_lightgcn_shard* st, uint32_t* state2, void* stream);

/* ------------------------------------------------------------------------ *
 * WMF surrogate of the AIA / Leg-UP attack loop  (recad/model/attacker/aia.py:222-247, 283-289, 393-489)
 * ------------------------------------------------------------------------ */
typedef struct recad_wmf {
  int64_t n_rows, n_items;   /* rows = genuine users + fake users (aia.py:133-141) */
  int32_t dim, batch;        /* hidden_dim_s in {8, 16, 32}, batch_size_s <= 32 (default.py:179, 182) */
  float lr, beta1, beta2, eps, weight_decay, weight_pos, weight_neg;
  int32_t _pad;
  float* P;                  /* [dev] float[n_rows, dim] */
  float* Q;                  /* [dev] float[n_items, dim] */
  float* mP; float* vP; float* mQ; float* vQ;   /* [dev] Adam state, same shapes */
} recad_wmf;

/* n_epochs epochs of WMFTrainer.fit_adv (aia.py:443-487) in ONE persistent cluster kernel: per batch of `batch` rows
 * (row ids orders [dev] int32[n_epochs, n_rows], the np.random.shuffle'd idx_list of each epoch, aia.py:447 / 468)
 * weighted-MSE gradient against data [dev] float[n_rows, n_items] and a dense Adam step with weight decay on P and Q.
 * unrolled == 0: torch.optim.Adam arithmetic (the plain epochs); unrolled != 0: higher.optim.DifferentiableAdam
 * arithmetic (the epochs inside higher.innerloop_ctx), and when snap != NULL every step records what the reverse pass
 * needs (recad_wmf_snapshot_floats(st, n_epochs) floats).  step0 = optimiser steps taken before this call. */
int64_t recad_wmf_snapshot_floats(const recad_wmf* st, int32_t n_epochs);
int recad_wmf_fit(const recad_wmf* st, const float* data, const int32_t* orders, int32_t n_epochs, int64_t step0,
                  int32_t unrolled, float* snap, void* stream);
/* Reverse pass through the unrolled epochs: Pbar / Qbar [dev] = d loss / d (final P, Q) on entry (overwritten);
 * d_data [dev] float[n_rows, n_items] += d loss / d data; scratch [dev] 2 * (n_rows + n_items) * dim + 1024 floats.
 * Same data / orders / step0 / snap as the recad_wmf_fit call that recorded the snapshots. */
int recad_wmf_backward(const recad_wmf* st, const float* data, const int32_t* orders, int32_t n_epochs, int64_t step0,
                       const float* snap, float* Pbar, float* Qbar, float* scratch, float* d_data, void* stream);

/* ------------------------------------------------------------------------ *
 * AUSH generator / discriminator step  (recad/model/attacker/aush.py:78-180, 182-230, 254-283)
 * ------------------------------------------------------------------------ */

/* The discriminator's parameters (Linear(I,150)-Sigmoid-Linear(150,150)-Sigmoid-Linear(150,150)-Sigmoid-Linear(150,1)-Sigmoid,
 * aush.py:269-283) live in one flat [dev] float buffer; offsets [host] int64[9] = float offsets of
 *   main.0.weight^T [I, 152], main.0.bias [152], main.2.weight [150, 152], main.2.bias [152], main.4.weight [150, 152],
 *   main.4.bias [152], main.6.weight [152], main.6.bias [4], and the TOTAL float count
 * (rows padded from 150 to 152 floats; the padding must be zero-initialised and stays zero). */
int recad_aush_d_layout(int64_t n_items, int64_t* offsets);

typedef struct recad_aush {
  int64_t n_items;
  int32_t n_sel;             /* |selected_ids| (default.py:166), <= 64 */
  int32_t filler_num;        /* default.py:161 */
  float lr, beta1, beta2, eps;   /* the discriminator's Adam (aush.py:32-35; lr_d, default.py:163) */
  /* generator Linear(I,128)-Sigmoid-Linear(128,I)-Sigmoid, x 5 (aush.py:254-266).  Read only: the reference detaches the
   * generator's output before every loss (aush.py:128), so its optimizer never sees a gradient. */
  const float* G_W1t;        /* [dev] float[I, 128] = main.0.weight^T */
  const float* G_b1;         /* [dev] float[128] */
  const float* G_W2;         /* [dev] float[I, 128] = main.2.weight */
  const float* G_b2;         /* [dev] float[I] */
  float* D;                  /* [dev] float[recad_aush_d_layout total] */
  float* Dm;                 /* [dev] Adam first moment, same layout  (training only) */
  float* Dv;                 /* [dev] Adam second moment              (training only) */
  const int32_t* selected;   /* [dev] int32[n_sel], ascending */
  float* work;               /* [dev] float[recad_aush_work_floats]   (training only) */
} recad_aush;

/* The sparse form of one epoch of batches (aush.py:100-121).  Row r of the epoch = the r-th user the dataset's batch
 * generator handed out; batch k = rows [k * batch, min(n_rows, (k + 1) * batch)).  F = filler_num, S = n_sel, slots s in
 * the order of recad_aush.selected. */
typedef struct recad_aush_epoch {
  int64_t n_rows;
  int32_t batch;
  int32_t _pad;
  const int32_t* cols;       /* [dev] int32[n_rows, F] the filler columns sample_fillers drew (repeats kept) */
  const float* tval;         /* [dev] float[n_rows, F] input_template at that column = real rating (0 for a repeated column) */
  const float* dval;         /* [dev] float[n_rows, F] real * (fillers_mask + selects_mask) at that column, 0 for a repeated
                                                       or a selected column (those are carried by rsel) */
  const float* rsel;         /* [dev] float[n_rows, S] real * (fillers_mask + selects_mask) at the selected columns */
  const float* tsel;         /* [dev] float[n_rows, S] input_template at the selected columns */
  const float* msel;         /* [dev] float[n_rows, S] fillers_mask + selects_mask at the selected columns */
  const float* zr;           /* [dev] float[n_rows, S] ZR_mask at the selected columns (aush.py:111-117) */
  const int32_t* colptr;     /* [dev] int32[n_batches, I + 1]  column index of every batch (recad_aush_plan_columns) */
  const int32_t* ent;        /* [dev] int32[n_rows * F] */
} recad_aush_epoch;

int64_t recad_aush_work_floats(int64_t n_items, int64_t n_rows, int32_t batch, int32_t n_sel);
/* HOST: per batch, the (row, filler slot) pairs grouped by item column (row-major inside a column):
 * colptr [host] int32[n_batches, I + 1] (offsets relative to the batch's first entry), ent [host] int32[n_rows * F]
 * = row_in_batch * F + slot.  This index gives the first-layer gradient a fixed summation order without atomics (the
 * selected columns, present in every row, are reduced on the device). */
int recad_aush_plan_columns(const int32_t* cols, int64_t n_rows, int32_t batch, int32_t F, int64_t n_items, int32_t* colptr,
                            int32_t* ent);
/* One epoch of Aush.train_step (aush.py:100-170): per batch the generator's forward on the selected columns, the
 * discriminator's forward / backward on the real and the fake rows, its dense Adam step (step0 = steps taken before), and
 * the forward of the updated discriminator on the fake rows.  loss_out [dev] double[4] = the tuple train_step returns:
 * means over the batches of d_loss, g_loss_rec, g_loss_shilling, g_loss_gan (aush.py:171-176). */
int recad_aush_train_epoch(const recad_aush* st, const recad_aush_epoch* ep, int64_t step0, double* loss_out, void* stream);
/* Generator forward of generate_fake (aush.py:213-216): gen_out [dev] float[n_rows, S] = netG(input_template)[:, selected]. */
int recad_aush_generate(const recad_aush* st, const int32_t* cols, const float* tval, int64_t n_rows, float* gen_out, void* stream);
/* HOST: the global-generator draws of ONE batch, bit-exact (aush.py:59-76 sample_fillers = np.random.choice with
 * replacement per row from the row's candidate list; 113-117 np.random.shuffle of the argwhere'd ZR pool).
 * users [host] int64[B]; cand_ptr / cand_items / cand_vals: per-user candidate lists in the order of the reference's
 * list(set(nonzero columns) & filler_pool) and their ratings; zero_sel [host] uint8[B, S] = (real == 0) at the selected
 * columns, slots in ascending column order; cols_out [host] int32[B, F]; tval_out [host] float[B, F] (may be NULL) = the
 * rating at the drawn column, 0 where the row already drew that column; zr_out [host] float[B, S]. */
int recad_mt19937_aush_batch(uint32_t* key, int32_t* pos, int64_t B, const int64_t* users, const int64_t* cand_ptr,
                             const int32_t* cand_items, const float* cand_vals, int32_t F, int32_t S, const uint8_t* zero_sel,
                             double zr_ratio, int32_t* cols_out, float* tval_out, float* zr_out);

/* scores[b] = <O[users[b]], O[n_users + items[b]]> (lightgcn.py:174-183 after a
 * propagate; O must be current). */
int recad_dot_scores(const float* O, int64_t n_users, const int64_t* users, const int64_t* items,
                     int64_t B, int32_t D, float* scores, void* stream);

/* ------------------------------------------------------------------------ *
 * Autograd backward passes of the victims' scores (what `loss.backward()` through
 * lightgcn.py:82-113 / 174-183, mf.py:40-47 and ncf.py:112-131 computes)
 * ------------------------------------------------------------------------ */

/* Backward of pair scores s_b = <Xa[ia[b]], Xb[ib[b]]> (+ ba[ia[b]] + bb[ib[b]]) for the upstream gradient g [dev] float[B]:
 *   dXa [dev] float[n_a, D] = sum over the b with ia[b] = r of g[b] Xb[ib[b]], dXb [dev] float[n_b, D] likewise (dense:
 *   rows no sample names are zero), dba [dev] float[n_a] / dbb [dev] float[n_b] = sum of g[b] per row (NULL: not wanted).
 * Atomic-free and bit-stable from run to run at any B: the samples of a row are grouped by a stable radix sort and added in
 * ascending sample order by the row's only writer.  Xa / Xb and the outputs are 16-byte aligned, D % 4 == 0; dXa and dXb
 * may be two halves of one buffer.  scratch [dev]: recad_pair_scores_backward_scratch_bytes(B) bytes.  Synchronises the
 * stream: an id outside its table gives RECAD_ERR_ARG (no memory outside the tables is addressed; the outputs are then
 * unspecified). */
int64_t recad_pair_scores_backward_scratch_bytes(int64_t B);
int recad_pair_scores_backward(const float* Xa, int64_t n_a, const float* Xb, int64_t n_b, int32_t D, const int64_t* ia,
                               const int64_t* ib, int64_t B, const float* g, float* dXa, float* dXb, float* dba, float* dbb,
                               void* scratch, int64_t scratch_bytes, void* stream);

/* Backward of recad_lightgcn_propagate: gE [dev] float[N, D] = (1 / (L + 1)) sum_l (A^T)^l gO for gO [dev] float[N, D]
 * (A^T = st->graph_t when set, else st->graph), by the Horner loop of the epoch driver.  Reads st->graph / graph_t,
 * n_users, n_items, D, n_layers; uses X0 (L >= 2) and X1 (L >= 3) as work; E, O, g, cnt, m, v and loss_acc are not
 * touched, so a caller may pass a copy of its state with work buffers of its own. */
int recad_lightgcn_backward(const recad_lightgcn* st, const float* gO, float* gE, void* stream);

/* The same backward with respect to the values of st->graph as well:
 *   gvals [dev] float[nnz] (st->graph's entry order) = (1 / (L + 1)) sum_{j < L} <t_j[r_k], X_{L-1-j}[c_k]>,
 *   t_0 = gO, t_{j+1} = gO + A^T t_j (the Horner iterates; A^T = graph_t when set, which it must be unless the values are
 *   symmetric), X [host] array of L device pointers to the forward's layers X_0 = E, X_1 = A E, .., X_{L-1}.
 * One Horner loop: the SDDMM of step j (recad_csr_sddmm over st->graph) runs next to its SpMM.  gE as in
 * recad_lightgcn_backward, or NULL (then the last SpMM is skipped).  L = 0: gvals = 0.  Work buffers as above. */
int recad_lightgcn_backward_values(const recad_lightgcn* st, const float* gO, const float* const* X, float* gE, float* gvals,
                                   void* stream);

/* ------------------------------------------------------------------------ *
 * Hessian-vector products of the training losses (LightGCN's BPR, MF's BCE)
 * ------------------------------------------------------------------------ */

/* The pair backward with a second gather source: outA [dev] float[n_a, D] = sum over the b with ia[b] = r of
 * (alpha[b] Xb[ib[b]] + beta[b] Vb[ib[b]]), outB [dev] float[n_b, D] likewise with Xa / Va, dba / dbb = sum of alpha[b] per
 * row (NULL: not wanted).  beta NULL: Va / Vb are not read and the result is recad_pair_scores_backward's, bit for bit.
 * Same sort, scratch (recad_pair_scores_backward_scratch_bytes(B)), determinism and id check as that entry. */
int recad_pair_scores_hvp(const float* Xa, const float* Va, int64_t n_a, const float* Xb, const float* Vb, int64_t n_b,
                          int32_t D, const int64_t* ia, const int64_t* ib, int64_t B, const float* alpha, const float* beta,
                          float* outA, float* outB, float* dba, float* dbb, void* scratch, int64_t scratch_bytes, void* stream);

/* Per-sample seeds of H_O dO for the BPR loss (1/B_norm) sum_b softplus(x_b), x_b = <O_u, O_n> - <O_u, O_p>, over the n rows
 * samples [dev] int64[n, 3] = (user, pos, neg); O, dO [dev] float[n_users + n_items, D] (users first).  With
 * dx_b = <dO_u, O_n - O_p> + <O_u, dO_n - dO_p>, l' = sigmoid(x), l'' = l'(1 - l') (x > 20: 1 and 0, torch's softplus):
 *   alpha [dev] float[2n]: alpha[b] = l''(x_b) dx_b / B_norm, alpha[n + b] = -alpha[b];
 *   beta  [dev] float[2n]: beta[b] = l'(x_b) / B_norm, beta[n + b] = -beta[b],
 * i.e. the seeds of recad_pair_scores_hvp over the pairs (u, neg) then (u, pos).  dloss [dev] float[n] (NULL: not wanted) =
 * l'(x_b) dx_b + lambda (<V_u, E_u> + <V_p, E_p> + <V_n, E_n>), the unnormalised derivative of sample b's loss along V when
 * dO = P V; E and V are then needed.  bad [dev] int32 work flag.  Deterministic.  Synchronises the stream: an id outside
 * its table gives RECAD_ERR_ARG. */
int recad_bpr_hvp_seeds(const float* O, const float* dO, int64_t n_users, int64_t n_items, const int64_t* samples, int64_t n,
                        int64_t B_norm, int32_t D, const float* E, const float* V, float lambda, float* alpha, float* beta,
                        float* dloss, int32_t* bad, void* stream);

/* Mixed second derivative of the BPR training loss L = (1/n) sum_b l_b (the loss recad_bpr_hvp_seeds differentiates, over
 * the n rows samples [dev] int64[n, 3]) with respect to the values v of st->graph, along S [dev] float[N, D] (users first):
 *   gvals [dev] float[nnz] (st->graph's entry order) = d/dv <S, grad_E L>, at the state's tables st->E.
 * With O = P E, dO = P S (P = (1 / (L + 1)) sum_l A^l), a_b / c_b the seeds of recad_bpr_hvp_seeds (B_norm = n), G_O the
 * H_O dO of recad_pair_scores_hvp and G_dO = the pair backward of c over O, gvals is the edge-value gradient of
 * <G_O, O> + <G_dO, dO> with G held: (1 / (L + 1)) sum_{j < L} <t_j[r_k], Y_{L-1-j}[c_k]> over the 2D columns of the
 * interleaved rows t_j (Horner iterates of [G_O | G_dO]) and Y_l = A^l [E | S].  The regulariser does not depend on v;
 * L = 0: gvals = 0.  One recurrence at width 2D: A2 is st->graph's struct for width 2D (its own partial-sum scratch);
 * st->graph_t must be NULL (symmetric values).  The state's buffers are not written.  work [dev] of
 * recad_lightgcn_loss_mixed_values_work_bytes(N, D, n_layers, n) bytes (L + 2 buffers of N * 2D floats, one more
 * for L >= 3, plus O(n)).  Atomic-free and bit-stable at any n; synchronises the stream once: an id outside its
 * table gives RECAD_ERR_ARG. */
int64_t recad_lightgcn_loss_mixed_values_work_bytes(int64_t n_rows, int32_t D, int32_t n_layers, int64_t n);
int recad_lightgcn_loss_mixed_values(const recad_lightgcn* st, const recad_csr* A2, const float* S, const int64_t* samples,
                                     int64_t n, float* gvals, void* work, int64_t work_bytes, void* stream);

/* Gradient of f(W) = <gO, O> + <S, grad_E L> with respect to one weight W put on both entries (u, U + i), (U + i, u) of
 * an interaction, for the users sel [dev] int64[n_sel] against every item, stored or not:
 *   out [dev] float[n_sel, n_items] (row-major) = d_u d_i (g_v(u, U+i) + g_v(U+i, u)) + coef_u + coef_{U+i} + sample part,
 * at the state's tables and the base point W = mult (0 where not stored).  O = P E as in recad_lightgcn_propagate; L the
 * loss of recad_lightgcn_loss_mixed_values over the n rows samples [dev] int64[n, 3], each row weighted by w_k / mult_k
 * when its positive pair k = (u, U + pos) is stored; g_v the SDDMM formula of that entry with the seed G = its mixed seed
 * + [gO | 0] (valid at unstored pairs as well); coef the per-row term of recad_csr_normalize_backward (pass 1) from g_v at
 * the stored entries; the sample part (1 / (n mult_k)) sum of the row derivatives along S (the dloss of
 * recad_bpr_hvp_seeds with lambda) over the rows with positive pair k, at the stored pairs of sel's rows.
 * gO, S [dev] float[N, D] (users first) or NULL (zero); n = 0: no rows (S and samples may be NULL).  mult [dev] float[nnz],
 * tperm [dev] int64[nnz] (the transpose permutation) and d_inv [dev] float[N] are st->graph's multiplicities, structure
 * transpose and normalisation factors (d_r = (s_r + 1e-14)^(-1/2)); A2 is st->graph's struct at width 2D; st->graph_t
 * must be NULL.  One recurrence at width 2D whose Horner pass also gathers the split GEMM operands, then one 3xTF32
 * tensor-core GEMM [n_sel, 4 L D + 1] x [n_items, 4 L D + 1]^T with the column bias coef_{U+i}; L = 0: the sample part
 * only.  work [dev] of recad_lightgcn_candidate_weight_grads_work_bytes bytes.  D <= 512.  Atomic-free and bit-stable;
 * synchronises the stream once: an id of sel outside [0, n_users) or of samples outside its table gives RECAD_ERR_ARG. */
int64_t recad_lightgcn_candidate_weight_grads_work_bytes(int64_t n_users, int64_t n_items, int32_t D, int32_t n_layers,
                                                         int64_t n, int64_t nnz, int64_t n_sel);
int recad_lightgcn_candidate_weight_grads(const recad_lightgcn* st, const recad_csr* A2, const float* mult,
                                          const int64_t* tperm, const float* d_inv, const float* gO, const float* S,
                                          const int64_t* samples, int64_t n, float lambda, const int64_t* sel, int64_t n_sel,
                                          float* out, void* work, int64_t work_bytes, void* stream);

/* out [dev] float[n_out] = per index r, the sum of x[b] over the b with idx[b] = r, in ascending b, in double (0 where
 * none); idx [dev] int64[n] with entries < 0 skipped.  One stable radix sort and one writer per output: atomic-free and
 * bit-stable.  scratch [dev] of recad_pair_scores_backward_scratch_bytes(n) bytes.  Synchronises the stream: an index
 * >= n_out gives RECAD_ERR_ARG. */
int recad_index_sums(const int64_t* idx, const float* x, int64_t n, int64_t n_out, float* out, void* scratch,
                     int64_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------ *
 * MF pointwise BCE step  (recad/model/victim/mf.py:40-69)
 * ------------------------------------------------------------------------ */
typedef struct recad_mf {
  int64_t n_users, n_items;
  int32_t D;
  float mean, lr, beta1, beta2, eps;
  float *Ue, *Ub, *Ie, *Ib;         /* [dev] params: [U,D] [U] [I,D] [I] */
  float *mUe, *mUb, *mIe, *mIb;     /* Adam m */
  float *vUe, *vUb, *vIe, *vIb;     /* Adam v */
  float *gUe, *gUb, *gIe, *gIb;     /* work: dense gradients */
  double* loss_acc;                 /* [dev] double[4] {batch sum, spare, epoch sum, spare} */
} recad_mf;

/* pred[b] = <Ue[u], Ie[i]> + Ub[u] + Ib[i] + mean (mf.py:40-47, dropout 0). */
int recad_mf_forward(const recad_mf* st, const int64_t* users, const int64_t* items, int64_t B,
                     float* pred, void* stream);
/* One epoch of MF.train_step (mf.py:49-69): BCEWithLogits (mean) + dense Adam on
 * the four tables, per batch.  samples [dev] int64[n, 3] = (user, item, label) rows, perm as in
 * recad_lightgcn_train_epoch.  Loss as in the LightGCN epoch. */
int recad_mf_train_epoch(const recad_mf* st, const int64_t* samples, const int64_t* perm,
                         int64_t n_samples, int64_t batch, int64_t step0, void* stream);
/* The gradient half of ONE step (mf.py:58-64, forward + backward, no optimiser): g* = d(BCE sum / B_norm)
 * over the B rows samples[perm[0..B)] (perm NULL: rows 0..B-1), g* zeroed here; loss_acc[0] += BCE sum
 * (the caller zeroes loss_acc).  For data-parallel training the rows of a batch are split over ranks,
 * B_norm is the GLOBAL batch size, the caller all-reduces g* and applies recad_adam (SURVEY.md 8e).  B = 0 is
 * allowed (zero gradient). */
int recad_mf_grad(const recad_mf* st, const int64_t* samples, const int64_t* perm, int64_t B, int64_t B_norm,
                  void* stream);
/* Per-row seeds of the Hessian-vector product of (1/B_norm) sum_b BCEWithLogits(y_b, label_b) over the n rows samples [dev]
 * int64[n, 3] = (user, item, label), y = <Ue_u, Ie_i> + Ub_u + Ib_i + st->mean (mean held constant), along the direction
 * (dUe [U, D], dUb [U], dIe [I, D], dIb [I]) [dev]: with dy_b = <dUe_u, Ie_i> + <Ue_u, dIe_i> + dUb_u + dIb_i,
 * l' = sigmoid(y) - label, l'' = sigmoid(y)(1 - sigmoid(y)):  alpha [dev] float[n] = l'' dy / B_norm,
 * beta [dev] float[n] = l' / B_norm (the seeds of recad_pair_scores_hvp over the pairs (user, item); its bias outputs are
 * the bias rows of the product), dloss [dev] float[n] (NULL: not wanted) = l' dy.  Reads the parameter tables only.
 * bad [dev] int32 work flag.  Deterministic.  Synchronises the stream: an id outside its table gives RECAD_ERR_ARG. */
int recad_mf_hvp_seeds(const recad_mf* st, const float* dUe, const float* dUb, const float* dIe, const float* dIb,
                       const int64_t* samples, int64_t n, int64_t B_norm, float* alpha, float* beta, float* dloss, int32_t* bad,
                       void* stream);

/* ------------------------------------------------------------------------ *
 * NCF / NeuMF-end pointwise BCE step  (recad/model/victim/ncf.py:32-53, 112-153)
 * ------------------------------------------------------------------------ */

/* All parameters live in one flat [dev] float buffer.  offsets [host]
 * int64[4 + 2 * n_layers + 3] = float offsets of
 *   embed_user_GMF [U, f], embed_item_GMF [I, f], embed_user_MLP [U, w], embed_item_MLP [I, w],
 *   then per MLP layer l: weight [in_l / 2, in_l] (torch Linear layout), bias [in_l / 2],
 *   predict weight [2 f], predict bias [1], and the TOTAL float count
 * with w = f * 2^(n_layers - 1), in_l = f * 2^(n_layers - l) (ncf.py:32-53).  Each piece starts
 * on a multiple of 4 floats; the padding must be zero-initialised. */
int recad_ncf_layout(int32_t factor, int32_t n_layers, int64_t n_users, int64_t n_items, int64_t* offsets);
int64_t recad_ncf_work_floats(int32_t factor, int32_t n_layers, int64_t max_batch);

typedef struct recad_ncf {
  int64_t n_users, n_items;
  int32_t factor, n_layers;
  float lr, beta1, beta2, eps;
  int32_t tower_fp32; /* 0: tower GEMMs on tcgen05 (3xTF32, fp32-accurate); 1: exact fp32 CUDA-core GEMMs (bit-stable
                         ReLU masks; what the strict parity tests use) */
  int32_t variant;    /* ncf.py:49-53, 112-131: 0 = NeuMF (predict on cat(GMF, MLP), 2f inputs; 'NeuMF-end' / 'NeuMF-pre'),
                         1 = 'GMF' (predict on the GMF product, f inputs), 2 = 'MLP' (predict on the tower output, f inputs).
                         The layout is the same for all three; the unused predict weights stay zero. */
  float* params;      /* [dev] float[n_params] */
  float* m;           /* [dev] Adam first moment  (training only) */
  float* v;           /* [dev] Adam second moment (training only) */
  float* grads;       /* [dev] float[n_params] work (training only) */
  int64_t n_params;   /* = offsets[last] of recad_ncf_layout */
  float* work;        /* [dev] float[work_floats] activations */
  int64_t work_floats;
  int64_t max_batch;  /* largest batch the work buffer was sized for */
  double* loss_acc;   /* [dev] double[4] {batch sum, spare, epoch sum, bad-id flag} */
} recad_ncf;

/* pred[b] = NeuMF(users[b], items[b]) (ncf.py:112-131, dropout 0), B <= max_batch. */
int recad_ncf_forward(const recad_ncf* st, const int64_t* users, const int64_t* items, int64_t B,
                      float* pred, void* stream);
/* Full ranking (normal.py:57-93 scores every (user, item) pair): the first tower layer is linear in cat(um[u], im[i]), so it
 * is evaluated once per user and once per item instead of once per pair (75 % of the tower's multiply-adds).
 *   recad_ncf_rank_work_floats  size of the path's own workspace for blocks of up to max_pairs pairs
 *   recad_ncf_rank_floats       size of PUI for n_eval_users users (negative: bad argument)
 *   recad_ncf_rank_prepare      PUI [dev] = [PU (n_eval_users x w) | PI (n_items x w)], PU = um[users] W_0[:, :w]^T,
 *                               PI = im W_0[:, w:]^T + b_0; also stages every layer's split weights in `work`.
 *                               RECAD_ERR_UNSUPPORTED when the model has to use recad_ncf_forward (exact fp32 tower, a
 *                               single layer)
 *   recad_ncf_rank_block        scores [dev] float[nu, n_items] of the evaluation users u0 .. u0 + nu (slots of `users`)
 *                               against every item; nu * n_items <= max_pairs; same work / PUI as the prepare call */
int64_t recad_ncf_rank_work_floats(int32_t factor, int32_t n_layers, int64_t max_pairs);
int64_t recad_ncf_rank_floats(const recad_ncf* st, int64_t n_eval_users);
int recad_ncf_rank_prepare(const recad_ncf* st, const int64_t* users, int64_t n_eval_users, float* PUI, float* work,
                           int64_t work_floats, int64_t max_pairs, void* stream);
int recad_ncf_rank_block(const recad_ncf* st, const float* PUI, const int64_t* users, int64_t n_eval_users, int64_t u0, int64_t nu,
                         float* scores, float* work, int64_t work_floats, int64_t max_pairs, void* stream);
/* One epoch of NCF.train_step (ncf.py:133-153); loss bookkeeping as in the MF epoch. */
int recad_ncf_train_epoch(const recad_ncf* st, const int64_t* samples, const int64_t* perm,
                          int64_t n_samples, int64_t batch, int64_t step0, void* stream);
/* Batches replayed from the captured graph so far in this process (diagnostic: tests check that the graph path ran). */
int64_t recad_ncf_graph_launches(void);
/* The gradient half of ONE step (ncf.py:139-148): as recad_mf_grad, into st->grads (layout of recad_ncf_layout). */
int recad_ncf_grad(const recad_ncf* st, const int64_t* samples, const int64_t* perm, int64_t B, int64_t B_norm,
                   void* stream);
/* Backward of recad_ncf_forward for an upstream gradient dpred [dev] float[B] (autograd): grads [dev] float[n_params]
 * (layout of recad_ncf_layout, written whole) = sum_b dpred[b] d pred[b] / d params over the pairs (users[b], items[b]),
 * B <= max_batch.  The forward is recomputed in the model's tower precision; st->grads, st->m, st->v and st->loss_acc
 * are not touched.  The embedding rows are added in ascending sample order (bit-stable) for B <= 8192.  Synchronises the
 * stream: an id out of range gives RECAD_ERR_ARG (no memory outside the tables is addressed). */
int recad_ncf_backward(const recad_ncf* st, const int64_t* users, const int64_t* items, int64_t B, const float* dpred,
                       float* grads, void* stream);
/* Hessian-vector product of the training loss (ncf.py:112-153): L = (1/n) sum_b BCEWithLogits(pred_b, label_b) over the n rows
 * samples [dev] int64[n, 3] = (user, item, label) taken as one batch (what train_step minimises for it; no regulariser, no
 * dropout), at the current parameters, in the model's tower precision.  vec [dev] float[n_params] is the direction in the
 * layout of recad_ncf_layout; out [dev] float[n_params] (NULL: not wanted) = H vec, written whole (padding zero; the branch a
 * variant does not read gets exactly zero); dloss [dev] float[n] (NULL: not wanted) = each row's unnormalised directional
 * derivative l'_b dpred_b = <grad l_b, vec>.  With out NULL only the R-forward and the seeds run.  Rows are processed in
 * chunks of max_batch, in order, the seeds normalised by the full n; no atomics, so the result is bit-stable at any n.
 * work [dev] float[work_floats], work_floats >= recad_ncf_hvp_work_floats(factor, n_layers, st->max_batch); st->work is
 * used as well.  st->params, m, v, grads and loss_acc are not touched.  Synchronises the stream: an id outside its table
 * gives RECAD_ERR_ARG (no memory outside the tables is addressed). */
int64_t recad_ncf_hvp_work_floats(int32_t factor, int32_t n_layers, int64_t max_batch);
int recad_ncf_hvp(const recad_ncf* st, const int64_t* samples, int64_t n, const float* vec, float* out, float* dloss,
                  float* work, int64_t work_floats, void* stream);

/* The tensor-core GEMM of the NCF tower, exposed for testing: C[M, N] = A[M, K] . B[N, K]^T (+ bias[N]) (ReLU) on
 * tcgen05 (kind::tf32, fp32 accumulators in TMEM, TMA operands) with the 3xTF32 operand split, i.e. fp32-accurate.
 * A, B, C row-major [dev]; scratch [dev] float[2 * (M + N) * ((K + 3) / 4 * 4)]. */
int recad_gemm_tn_tf32x3(const float* A, const float* B, int32_t M, int32_t N, int32_t K, const float* bias,
                         int32_t relu, float* C, float* scratch, void* stream);

/* ------------------------------------------------------------------------ *
 * Full-ranking evaluation  (recad/workflow/normal.py:57-93, 111-160;
 * lightgcn.py:115-120 getUsersRating)
 * ------------------------------------------------------------------------ */

/* item_T[d * ld + i] = item_emb[i * D + d]  (ld >= n_items, multiple of 4). */
int recad_transpose_items(const float* item_emb, int64_t n_items, int32_t D, float* item_T,
                          int64_t ld, void* stream);

/* For each of n_eval users: score EVERY item (s = <user_emb[u], item_emb[i]>, fp32
 * FMA in ascending d), drop the user's train items, and produce
 *   topk_idx/topk_val [dev] int32/float[n_eval, K]  best K by (score desc, id asc); -1/-inf padded
 *   target_rank  [dev] int32[n_eval, T]  #{non-train i: s_i > s_t or (s_i == s_t and i < t)},
 *                                        -1 when the target is one of the user's train items
 *   target_score [dev] float[n_eval, T]
 * without materialising the score matrix.  HR@k = mean[rank < k] and pred_shift
 * (normal.py:155-159) follow on the host from these.  Tie rule documented in
 * DESIGN.md (the reference's pandas quicksort leaves ties undefined, normal.py:86-88).
 *   user_emb [dev] float[*, D]; user_ids [dev] int64[n_eval] rows of user_emb
 *   train_rowptr [dev] int64[n_users_total + 1], train_col [dev] int32[] ascending per user
 *   targets [dev] int32[T] (T <= 8), K <= 128 */
int recad_fullrank_eval(const float* user_emb, const float* item_T, int64_t ld, int64_t n_items,
                        int32_t D, const int64_t* user_ids, int64_t n_eval,
                        const int64_t* train_rowptr, const int32_t* train_col,
                        const int32_t* targets, int32_t T, int32_t K, int32_t* topk_idx,
                        float* topk_val, int32_t* target_rank, float* target_score, void* stream);

/* The same evaluation on the tensor cores: tcgen05.mma kind::tf32 with fp32 accumulators in TMEM, operand
 * tiles fed by TMA, every operand split x = tf32(x) + tf32(x - tf32(x)) and three MMAs per tile ("3xTF32":
 * |score error| ~ 2^-21 |u||i|, so ranks can differ from recad_fullrank_eval only between near-tied items).
 * item_emb is the ROW-major [n_items, D] table (no transpose needed), D <= 64, K <= 32.
 * item_bias [dev] float[n_items] or NULL is added to every score (MF's b_i; b_u and the mean do not
 * change a user's ranking and are added to target_score by the caller).
 * scratch [dev] float[recad_fullrank_tc_scratch_floats(n_eval, n_items)], 256-byte aligned. */
int64_t recad_fullrank_tc_scratch_floats(int64_t n_eval, int64_t n_items);
int recad_fullrank_eval_tc(const float* user_emb, const float* item_emb, int64_t n_items, int32_t D,
                           const int64_t* user_ids, int64_t n_eval, const int64_t* train_rowptr,
                           const int32_t* train_col, const int32_t* targets, int32_t T, int32_t K,
                           const float* item_bias, int32_t* topk_idx, float* topk_val,
                           int32_t* target_rank, float* target_score, float* scratch,
                           int64_t scratch_floats, void* stream);

/* Same outputs as recad_fullrank_eval from a MATERIALISED score block, for victims whose
 * score is not an inner product (NCF): scores [dev] float[n_rows, n_items], row r belongs
 * to user user_ids[r].  One warp per row. */
int recad_rank_from_scores(const float* scores, int64_t n_rows, int64_t n_items,
                           const int64_t* user_ids, const int64_t* train_rowptr,
                           const int32_t* train_col, const int32_t* targets, int32_t T, int32_t K,
                           int32_t* topk_idx, float* topk_val, int32_t* target_rank,
                           float* target_score, void* stream);

/* Recall@K / NDCG@K sums over users from top-K lists and a ground-truth CSR
 * (implicit.py:461-476 test batches; definition in oracle/evaluate.py, parity
 * unpinned in the reference).  out [dev] double[3] += {sum recall, sum ndcg, n users with gt}. */
int recad_recall_ndcg(const int32_t* topk_idx, int64_t n_eval, int32_t K, const int64_t* user_ids,
                      const int64_t* gt_rowptr, const int32_t* gt_col, double* out, void* stream);

/* ------------------------------------------------------------------------ *
 * Samplers: bit-exact replay of the legacy np.random MT19937 stream on the host
 * (recad/dataset/implicit.py:18-35, 50-74, 77-91; recad/__init__.py:11-14)
 * ------------------------------------------------------------------------ */

/* key[624] / *pos: numpy's legacy state (np.random.get_state()[1:3]); advanced in
 * place so the caller can write it back with np.random.set_state.
 * out [host] int64[train_size * 3] (user, pos, neg) rows; *n_out = rows produced
 * (users without positives are dropped, implicit.py:63-64). */
int recad_mt19937_pairwise(uint32_t* key, int32_t* pos, int64_t n_users, int64_t n_items,
                           int64_t train_size, const int64_t* allpos_rowptr,
                           const int32_t* allpos_col, int64_t* out, int64_t* n_out);
int recad_host_advise_huge(void* ptr, int64_t bytes);   /* madvise(MADV_HUGEPAGE) on an untouched host buffer; best effort */
/* Per-user filter blocks of recad_mt19937_pairwise_soa for users [u_lo, n_users); the other users' blocks are left
 * untouched (dataset injection: the parent's blocks are copied, only the appended fake users' are built).
 * filter [host] uint64[n_users * 16]: word 0 = the user's row start | row length << 40, words 1..7 = 448 filter bits,
 * words 8..15 = 512 more bits consulted only when the first probe hits; no false negatives, a "maybe" falls back to
 * the exact search.  ext [host] uint32[nnz of allpos] = second-level filter of the users with more than 96 positives. */
int recad_pairwise_filter_build_range(const int64_t* allpos_rowptr, const int32_t* allpos_col, int64_t u_lo, int64_t n_users,
                                      uint64_t* filter, uint32_t* ext, int32_t n_threads);

/* Per user k (dict order): its |pos| positives (label 1, stored order) then
 * ratio * |pos| negatives drawn with replacement from the ascending complement.
 * pos_sorted: the same lists sorted ascending (for the complement).
 * out [host] int64[(1 + ratio) * n_pos_total * 3]. */
int recad_mt19937_pointwise(uint32_t* key, int32_t* pos, int64_t n_dict_users, const int64_t* user_ids,
                            const int64_t* pos_rowptr, const int64_t* pos_items,
                            const int64_t* pos_sorted, int64_t n_items, int32_t ratio, int64_t* out);
/* np.random.shuffle(np.arange(n)) (implicit.py:24-25): perm [host] int64[n]. */
int recad_mt19937_permutation(uint32_t* key, int32_t* pos, int64_t n, int64_t* perm);
/* The same shuffle in two halves (identical result and stream consumption): _draw is the only part that
 * consumes the stream (j_out [host] uint32[n], j_out[i] = random_interval(i) for i = n-1 .. 1), _apply turns
 * the draws into the permutation without touching the generator -- so the caller can start drawing the next
 * epoch while another thread applies the swaps of this one. */
int recad_mt19937_permutation_draw(uint32_t* key, int32_t* pos, int64_t n, uint32_t* j_out);
/* Epoch sampler for 10^7..10^8 samples: same samples and stream consumption as recad_mt19937_pairwise
 * (+ recad_mt19937_permutation_draw when j_out != NULL), in 32-bit structure-of-arrays form (n_users, n_items and
 * train_size at most 2^31 - 1):
 *   users / rel / negs [host] uint32[train_size]: user id, INDEX of the positive inside the user's row of allPos,
 *   negative item; the positive ITEM is looked up on the device by recad_samples_expand.
 * A producer thread generates the MT19937 stream into a ring, helper threads gather row lengths and verify the
 * optimistically drawn negatives; the calling thread runs the sequential parse (csrc/sampler.cpp).
 * filter / ext: built by recad_pairwise_filter_build_range. */
int recad_mt19937_pairwise_soa(uint32_t* key, int32_t* pos, int64_t n_users, int64_t n_items, int64_t train_size,
                               const int64_t* allpos_rowptr, const int32_t* allpos_col, const uint64_t* filter,
                               const uint32_t* ext, int32_t n_threads, uint32_t* users, uint32_t* rel, uint32_t* negs,
                               int64_t* n_out, uint32_t* j_out);
int recad_permutation_apply32(int64_t n, const uint32_t* j, int32_t* perm);
/* rows[k] = (users[k], allpos_col[allpos_rowptr[users[k]] + rel[k]], negs[k]) as int32[n, 3] on the device
 * (the positive-item gather of implicit.py:66-67, done where the CSR lives).
 * users / rel / negs [dev] uint32[n], allpos_rowptr [dev] int64[n_users + 1], allpos_col [dev] int32[]. */
int recad_samples_expand(const int64_t* allpos_rowptr, const int32_t* allpos_col, const uint32_t* users,
                         const uint32_t* rel, const uint32_t* negs, int64_t n, int32_t* rows, void* stream);
int recad_permutation_apply(int64_t n, const uint32_t* j, int64_t* perm);

#ifdef __cplusplus
}
#endif
#endif /* RECAD_B200_H */
