/*
 * daisy_b200.h -- C ABI of libdaisy_b200.so: the B200 (sm_100a) implementation of Daisy's
 * BPR-MF / funk-SVD training hot path and its top-K evaluation.
 *
 * The reference (NotFoundGG/recommend-lib) has no FFI of its own: the hot path sits behind Python
 * object protocols (SURVEY.md section 8b).  Each entry point below names the reference code it
 * replaces (file:line relative to the reference root); INTEGRATION.md shows the ctypes binding a
 * maintainer adds on the reference side.
 *
 * Conventions
 *  - every function returns 0 on success or a negative DAISY_E* code; daisy_last_error() returns a
 *    thread-local message for the last failing call on this thread;
 *  - device buffers (tables, index arrays, outputs) are OWNED BY THE CALLER (e.g. torch.Tensor.data_ptr());
 *    the handle owns only its workspace;
 *  - every call is asynchronous on the CUDA stream passed in (a cudaStream_t cast to void*; NULL = the
 *    legacy default stream);  a handle is bound to one device and is not thread-safe;
 *  - row ids are validated on the device: an out-of-range id never faults, it raises a sticky flag that
 *    daisy_check() reports as DAISY_EINDEX (mirrors nn.Embedding's IndexError / predict's ValueError);
 *  - tables are row-major contiguous fp32 [rows, dim], dim % 4 == 0, dim <= 512, base 16-byte aligned.
 */
#ifndef DAISY_B200_H
#define DAISY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAISY_OK 0
#define DAISY_EINVAL (-1)       /* bad argument */
#define DAISY_ECUDA (-2)        /* CUDA runtime error (message has the cudaError string) */
#define DAISY_EINDEX (-3)       /* a user / item id was out of range (sticky until daisy_check) */
#define DAISY_EUNSUPPORTED (-4) /* shape not supported by this build */
#define DAISY_ENOMEM (-5)

#define DAISY_ABI_VERSION 1

#if defined(__GNUC__)
#define DAISY_API __attribute__((visibility("default")))
#else
#define DAISY_API
#endif

typedef struct daisy_ctx *daisy_handle_t;
typedef void *daisy_stream_t; /* cudaStream_t */

/* create flags */
#define DAISY_FLAG_DEFAULT 0u
#define DAISY_FLAG_EAGER_DECAY 1u /* apply the dense L2 shrink to every row every step (reference-literal,
                                     BPRMFRecommender.py:154,176) instead of the exact lazy scale */

DAISY_API int daisy_abi_version(void);
DAISY_API const char *daisy_last_error(void);

/* Workspace for one model: tables of user_num x dim and item_num x dim, batches of at most max_batch.
 * Replaces: BPR.__init__ allocation side (BPRMFRecommender.py:29-40) + optim.SGD construction (:154). */
DAISY_API int daisy_create(daisy_handle_t *out, int device, int64_t user_num, int64_t item_num, int dim,
                 int64_t max_batch, unsigned flags);
DAISY_API int daisy_destroy(daisy_handle_t h);

/* Synchronise `stream` and report (then clear) the sticky device-side index error.  On DAISY_EINDEX the
 * message names the first offending position.  Mirrors IndexError of nn.Embedding (BPRMFRecommender.py:43-45). */
DAISY_API int daisy_check(daisy_handle_t h, daisy_stream_t stream);

/* ---- lazy L2 decay ------------------------------------------------------------------------------
 * optim.SGD(weight_decay) shrinks EVERY row by (1 - lr*wd) each step (BPRMFRecommender.py:154,176).
 * The library stores W_hat = W / c and keeps the scalar c per handle; scores use c^2.  The true tables
 * are W = c * W_hat; daisy_materialize() multiplies both tables by c and resets c = 1 (one pass over the
 * tables) -- call it before anything outside the library reads the weights (eval by foreign code,
 * torch.save, predict).  daisy_get_scale() returns c. */
DAISY_API int daisy_get_scale(daisy_handle_t h, double *c);
DAISY_API int daisy_set_scale(daisy_handle_t h, double c);
DAISY_API int daisy_materialize(daisy_handle_t h, float *P, float *Q, daisy_stream_t stream);

/* BPR.forward (BPRMFRecommender.py:42-50): pred_i[t] = <P[u_t],Q[i_t]>, pred_j[t] = <P[u_t],Q[j_t]>.
 * triples: device int32 [B,3] packed (u,i,j).  Honours the handle's lazy scale. */
DAISY_API int daisy_bpr_forward(daisy_handle_t h, const float *P, const float *Q, const int32_t *triples, int64_t B,
                      float *pred_i, float *pred_j, daisy_stream_t stream);

/* One training step = model.zero_grad(); forward; loss = -(pi-pj).sigmoid().log().sum(); loss.backward();
 * optimizer.step()  (BPRMFRecommender.py:172-176) fused: gradients at the pre-step tables, repeated rows
 * accumulate deterministically (sort-by-row segmented reduction, no float atomics), SGD + L2.
 * loss_accum (device double, may be NULL): the batch-sum loss is ADDED to it.
 * triples: device int32 [B,3], B <= max_batch. */
DAISY_API int daisy_bpr_step(daisy_handle_t h, float *P, float *Q, const int32_t *triples, int64_t B, float lr, float wd,
                   double *loss_accum, daisy_stream_t stream);

/* The integer bookkeeping of a step (sorting the batch by row) depends on the triples only, so the library runs
 * it on a private stream where, for step n+1, it overlaps the table kernels of step n.  By default
 * daisy_bpr_step assumes `triples` may still be being produced by earlier work on `stream` and orders its
 * bookkeeping after that work (which also orders it after step n: no overlap).  Declare with on = 1 that device
 * triples passed to daisy_bpr_step are complete at call time (e.g. batches uploaded and synchronised up front)
 * to get the overlap.  daisy_bpr_step_host always overlaps (host memory is complete at call time).
 * The flag stays set until it is changed.  It is read by daisy_bpr_step, daisy_gmf_step and the row-sharded steps
 * (daisy_bpr_shard_step, daisy_shard_step, daisy_shard_compute, daisy_shard_prepare) only.  daisy_bpr_epoch and
 * daisy_gmf_epoch with device input order their bookkeeping once per call behind the work already on `stream`, and
 * daisy_bpr_adam_step and daisy_bprfm_adagrad_step at every call, whatever the flag says. */
DAISY_API int daisy_set_inputs_ready(daisy_handle_t h, int on);

/* Same step fed from HOST memory (the reference's `user.cuda(); item_i.cuda(); item_j.cuda()`,
 * BPRMFRecommender.py:163-166): triples_host is int32 [B,3] in host memory (pinned for a truly async
 * copy); the library copies it into its own device buffer on `stream` and runs the step. */
DAISY_API int daisy_bpr_step_host(daisy_handle_t h, float *P, float *Q, const int32_t *triples_host, int64_t B, float lr,
                        float wd, double *loss_accum, daisy_stream_t stream);

/* One epoch of steps = the body of `for user, item_i, item_j in train_loader:` (BPRMFRecommender.py:162-178) run
 * by the library: triples is int32 [n,3] (every triple of the epoch, already shuffled), consumed in consecutive
 * batches of `batch` (<= max_batch; the last one may be short), each one exactly daisy_bpr_step /
 * daisy_bpr_step_host.  One call per epoch instead of one per step: with small batches (the reference's default is
 * 4 096) the step takes ~20 us on the device and the per-call cost of the host language would dominate.
 * on_host = 1: triples is host memory (pinned), each batch is copied in as the head of its bookkeeping chain.
 * on_host = 0: device memory, produced by earlier work on `stream` at the latest (e.g. daisy_sample_triples). */
DAISY_API int daisy_bpr_epoch(daisy_handle_t h, float *P, float *Q, const int32_t *triples, int64_t n, int64_t batch,
                    int on_host, float lr, float wd, double *loss_accum, daisy_stream_t stream);

/* ---- row-sharded tables (no Daisy counterpart; SURVEY.md section 8e) --------------------------------
 * One process per GPU owns a block of user rows and a block of item rows.  Triples are routed to the owner of
 * their user, so P is local; the item rows a batch needs are fetched from their owners into `cache`
 * [cache_rows, dim] (exchange done by the host code over NCCL) and the triples' item ids are indices into it.
 * daisy_bpr_shard_step runs the same fused pipeline as daisy_bpr_step: users get SGD + lazy L2 in place, and
 * instead of updating the cache it writes the complete descent sum of every cache row to grad_out [cache_rows, dim]
 * (every cache row must be referenced by at least one triple).  The handle is created with the LOCAL table sizes;
 * cache_rows <= 2 * max_batch. */
DAISY_API int daisy_bpr_shard_step(daisy_handle_t h, float *P_local, const float *cache, int64_t cache_rows,
                                   const int32_t *triples, int64_t B, float lr, float wd, float *grad_out,
                                   double *loss_accum, daisy_stream_t stream);
/* Owner side: rows [n] (local item row ids, concatenated in sender-rank order, each sender's list duplicate-free)
 * and grads [n, dim] (their descent sums).  Applies Q_local[row] += lr/(1-lr*wd) * sum over senders, contributions
 * of a row summed in sender-rank order (stable sort): deterministic. */
DAISY_API int daisy_owner_apply(daisy_handle_t h, float *Q_local, const int32_t *rows, const float *grads, int64_t n,
                                float lr, float wd, daisy_stream_t stream);

/* ---- row-sharded tables over PEER MEMORY (NVLink / NVSwitch), one process per GPU -------------------------
 * The fused compute + exchange path for catalogues larger than one GPU (BASELINE.json configs[4]): no collective
 * library on the data path.  Rows are block-sharded: rank r owns items [r*i_per, (r+1)*i_per), i_per =
 * ceil(item_num_global / world), and a block of users; a triple is (LOCAL user row, GLOBAL positive item, GLOBAL
 * negative item) and is fed to the rank that owns its user.  The handle is created with the LOCAL row counts.
 *
 *   daisy_shard_init    sets up this rank's ARENA (its item rows + receive regions + barrier flags, one contiguous
 *                       buffer of daisy_shard_arena_size bytes with the same layout on every rank).  arena != NULL:
 *                       caller-owned memory that the caller has mapped into the peer processes -- the product path
 *                       passes a torch symmetric-memory buffer (cuMem VMM mapping; measured 625 GB/s per direction
 *                       for random 512-byte row reads from the peer).  arena == NULL: the library cudaMallocs it and
 *                       exports it through legacy CUDA IPC (daisy_shard_ipc_handle; that mapping was measured at
 *                       300 GB/s for the same reads, profiles/r01_peer_mapping_bw.md).
 *                       daisy_shard_arena returns the arena and the item-shard pointer q_local [item rows, dim]
 *                       (fill it before the first step; it is the rank's block of BPR.embed_item.weight)
 *   daisy_shard_attach  gives the library the peers' arenas as mapped into THIS process: either the ranks' 64-byte
 *                       CUDA IPC handles (exchanged by any transport, e.g. torch.distributed.all_gather) or their
 *                       addresses (arena_ptrs [world]).  in_process = 1: all ranks live in this process on one
 *                       device (single-GPU emulation in the tests) -- the caller orders the phases, no barriers.
 *   daisy_shard_step    one training step of this rank: pre-step item rows are READ from their owners by peer loads,
 *                       the fused step kernels STORE every finished item-row sum straight into its owner's memory,
 *                       a flag barrier across the GPUs, the owner-side deterministic merge + update, a second barrier.
 *                       Every rank must call it the same number of times (B may be 0).  Asynchronous, no host sync.
 *   daisy_shard_compute / _barrier / _apply   the phases of daisy_shard_step, for callers that drive several ranks
 *                       from one process in lockstep (all computes, then all applies; no barrier kernels).
 *   daisy_shard_prepare / _classify   the same lockstep protocol with the EXCLUSIVE-ROW BYPASS of daisy_shard_step
 *                       (DAISY_SHARD_BYPASS): all prepares (bookkeeping + id lists into the owners), all classifies
 *                       (every owner tells every sender which of its rows no other rank references this step), all
 *                       computes (same B; a sender stores the UPDATED row of an exclusive row straight into its
 *                       owner's shard instead of a sum the owner would have to add), all applies (shared rows only).
 *                       Results are bit-identical with and without the bypass.
 *   daisy_shard_materialize   daisy_materialize on (P_local, q_local) + barrier (peers read q_local).
 * Semantics = daisy_bpr_step on the global batch (gradients at the pre-step tables, repeated rows accumulate);
 * contributions to a row are added in sender-rank order, so results are bit-reproducible. */
DAISY_API int daisy_shard_arena_size(int dim, int64_t max_batch, int world, int64_t item_num_global, int64_t *bytes);
DAISY_API int daisy_shard_init(daisy_handle_t h, int rank, int world, int64_t item_num_global, void *arena);
DAISY_API int daisy_shard_arena(daisy_handle_t h, void **arena, float **q_local, int64_t *arena_bytes);
DAISY_API int daisy_shard_ipc_handle(daisy_handle_t h, void *out64);
DAISY_API int daisy_shard_attach(daisy_handle_t h, const void *ipc_handles /* [world][64] or NULL */,
                                 void *const *arena_ptrs /* [world] or NULL */, int in_process);
DAISY_API int daisy_shard_step(daisy_handle_t h, float *P_local, const int32_t *triples, int64_t B, float lr, float wd,
                               double *loss_accum, daisy_stream_t stream);
DAISY_API int daisy_shard_step_host(daisy_handle_t h, float *P_local, const int32_t *triples_host, int64_t B, float lr,
                                    float wd, double *loss_accum, daisy_stream_t stream);
DAISY_API int daisy_shard_compute(daisy_handle_t h, float *P_local, const int32_t *triples, int64_t B, float lr, float wd,
                                  double *loss_accum, daisy_stream_t stream);
DAISY_API int daisy_shard_prepare(daisy_handle_t h, float *P_local, const int32_t *triples, int64_t B, daisy_stream_t stream);
DAISY_API int daisy_shard_classify(daisy_handle_t h, daisy_stream_t stream);
DAISY_API int daisy_shard_barrier(daisy_handle_t h, daisy_stream_t stream);
DAISY_API int daisy_shard_apply(daisy_handle_t h, float lr, float wd, daisy_stream_t stream);
DAISY_API int daisy_shard_materialize(daisy_handle_t h, float *P_local, daisy_stream_t stream);
/* The schedule of the fused step kernel (no device call): *chunk = the chunk of sorted triples that warp `warp` of a
 * launch over `nchunks` chunks takes when the chunks are dealt round-robin over `interleave` ranges of the
 * owner-grouped order (the sharded step uses interleave = world size; 0 / 1 = sorted order), -1 if the warp has none.
 * Every chunk is taken by exactly one warp of the ceil(nchunks / interleave) * interleave launched. */
DAISY_API int daisy_shard_schedule(int warp, int nchunks, int interleave, int *chunk);
/* Reporting: owner_off_out [world+1] = first cache row of every owner in the most recent step of this rank, so
 * owner_off_out[o+1] - owner_off_out[o] distinct item rows were fetched from / pushed to rank o.  Synchronises. */
/* The item shard of `rank` as mapped into this process (diagnostics). */
DAISY_API int daisy_shard_peer_q(daisy_handle_t h, int rank, float **q);
/* Row gather dst[c] = src[idx[c]] (rows of `dim` floats; src may be a peer address mapped into this process):
 * the building block of the fetch, exposed for bandwidth diagnostics (tools/peer_map_bw.py). */
DAISY_API int daisy_gather_rows(daisy_handle_t h, const float *src, const int32_t *idx, int64_t n, float *dst,
                                daisy_stream_t stream);
/* With daisy_set_timing(h, 2): average device ms of the phases of daisy_shard_step since the last call, in order
 * bookkeeping, fetch, compute+push, barrier, apply, barrier (the step is then serialised on the caller's stream and
 * synchronised once per step -- a diagnostic, not a bench mode). */
DAISY_API int daisy_shard_phase_ms(daisy_handle_t h, double *avg_ms6, int64_t *steps);
DAISY_API int daisy_shard_last_counts(daisy_handle_t h, uint32_t *owner_off_out, daisy_stream_t stream);

/* Lazy sparse Adam variant of the step (no Daisy counterpart -- BPR-MF uses SGD only; semantics =
 * torch.optim.SparseAdam: only rows present in the batch change, weights and moments alike).
 * mP,vP [user_num,dim], mQ,vQ [item_num,dim] fp32 moments owned by the caller; step_no is 1-based.  The betas are
 * doubles: torch forms 1 - beta in double before it meets the fp32 tensors (1.f - 0.999f is off by 1.3e-5). */
DAISY_API int daisy_bpr_adam_step(daisy_handle_t h, float *P, float *Q, float *mP, float *vP, float *mQ, float *vQ,
                        const int32_t *triples, int64_t B, float lr, double beta1, double beta2, float eps,
                        int64_t step_no, double *loss_accum, daisy_stream_t stream);

/* ---- BPR-FM with two one-hot features per example (SURVEY.md section 8f, row N3) ------------------
 * BPRFM (BPRFMRecommender.py:29-80) with batch_norm = False and drop_prob = [0, 0], features [user, user_num + item],
 * values [1, 1]:  pred = <e_u, e_i> + b_u + b_i + bias_,  loss = -(pred_i - pred_j).sigmoid().log().sum()  (:214-219),
 * optimiser torch.optim.Adagrad(lr, initial_accumulator_value) (:191-193), which moves only elements with a gradient.
 * The handle is created with dim = num_factors + 4.  E [user_num + item_num, dim]: AUGMENTED rows
 * [e_0 .. e_{F-1}, x, 0, 0, 0] with x = 1 for user rows (constant) and x = b_i for item rows; acc: Adagrad state_sum,
 * same layout, initialised to initial_accumulator_value.  triples: device int32 [B,3] (user, item_i, item_j) with
 * item ids relative to the item block.  The user bias and bias_ cancel in pred_i - pred_j and never move. */
DAISY_API int daisy_bprfm_adagrad_step(daisy_handle_t h, float *E, float *acc, const int32_t *triples, int64_t B, float lr,
                             float eps, double *loss_accum, daisy_stream_t stream);

/* ---- NCF, GMF variant (SURVEY.md section 8f, row N3) -----------------------------------------------
 * NCF.forward with model == 'GMF' (NCFRecommender.py:105-125): pred[t] = w . (P[u_t] * Q[i_t]) + b.
 * samples: device int32 [B,3] packed (user, item, label); the label column is ignored here.
 * P = embed_user_GMF.weight [user_num, dim], Q = embed_item_GMF.weight [item_num, dim], w = predict_layer.weight
 * [dim] (16-byte aligned), b = predict_layer.bias [1]. */
DAISY_API int daisy_gmf_forward(daisy_handle_t h, const float *P, const float *Q, const float *w, const float *b,
                      const int32_t *samples, int64_t B, float *pred, daisy_stream_t stream);

/* One training step of the script's loop (NCFRecommender.py:283-287 with :255, :260):
 *   model.zero_grad(); prediction = model(user, item); loss = nn.BCEWithLogitsLoss()(prediction, label);
 *   loss.backward(); optim.Adam(lr).step()
 * fused: gradients at the pre-step parameters, repeated rows accumulate deterministically (sort-by-row segmented
 * reduction, no float atomics), then torch-default Adam over EVERY element of both tables and of the predict layer
 * (dense Adam: a row without a gradient still moves while its first moment decays).
 * mP,vP [user_num,dim], mQ,vQ [item_num,dim]: Adam moments of the tables; mwb [2*(dim+1)]: moments of (w.., b):
 * first moments, then second moments.  step_no is 1-based.  loss_accum (device double, may be NULL): the batch's
 * MEAN loss is added to it.  B <= 8192 (the reference's batch is 256); labels are 0 / 1 in column 2 of samples. */
DAISY_API int daisy_gmf_step(daisy_handle_t h, float *P, float *Q, float *w, float *b, float *mP, float *vP, float *mQ,
                   float *vQ, float *mwb, const int32_t *samples, int64_t B, float lr, float beta1, float beta2,
                   float eps, int64_t step_no, double *loss_accum, daisy_stream_t stream);

/* The loop `for user, item, label in train_loader:` of one epoch (NCFRecommender.py:268-288) inside the library:
 * samples int32 [n,3] (already shuffled), consumed in consecutive batches of `batch`, step numbers
 * first_step_no, first_step_no + 1, ...; on_host = 1: (pinned) host memory, copied in batch by batch.
 * loss_accum receives the SUM of the batches' mean losses. */
DAISY_API int daisy_gmf_epoch(daisy_handle_t h, float *P, float *Q, float *w, float *b, float *mP, float *vP, float *mQ,
                    float *vQ, float *mwb, const int32_t *samples, int64_t n, int64_t batch, int on_host, float lr,
                    float beta1, float beta2, float eps, int64_t first_step_no, double *loss_accum,
                    daisy_stream_t stream);

/* metric_eval / _bpr_topk (util/metrics.py:46-66,88-94), all groups in one launch:
 * for n < N: score[c] = <P[users[n]], Q[cand[n,c]]>, c < C; the K best in (score desc, position asc) order.
 * out_pos [N,K] int32 = candidate positions (the `indices` of torch.topk), out_item [N,K] = cand ids
 * (`torch.take`), out_score [N,K].  C <= 8192, K <= 128, K <= C. */
DAISY_API int daisy_topk_candidates(daisy_handle_t h, const float *P, const float *Q, const int32_t *users,
                          const int32_t *cand, int64_t N, int C, int K, int32_t *out_pos, int32_t *out_item,
                          float *out_score, daisy_stream_t stream);

/* Full-catalogue score + top-K (replaces the per-candidate scalar loop BPRMFRecommender.py:196-207):
 * for n < N the K best items of score[i] = <P[users[n]], Q[i]>, i < item_num, order (score desc, item asc).
 * Optional exclusion lists in CSR form (excl_ptr [N+1] int64, excl_idx int32: the user's training positives).
 * K <= 128. */
DAISY_API int daisy_topk_full(daisy_handle_t h, const float *P, const float *Q, const int32_t *users, int64_t N, int K,
                    const int64_t *excl_ptr, const int32_t *excl_idx, int32_t *out_item, float *out_score,
                    daisy_stream_t stream);
/* Which strategy served the last daisy_topk_full call on h: *path = DAISY_TOPK_PATH_EXACT (materialised scores +
 * radix select), _SIMT (fp32 CUDA-core candidate filter) or _TC (BF16 tensor-core candidate filter); *filtered = users
 * whose top K came from the candidate list, *redone = users the exact path redid because their list overflowed or
 * held fewer than K admissible items (both 0 on the exact path).  Host state only: no device call. */
#define DAISY_TOPK_PATH_EXACT 0
#define DAISY_TOPK_PATH_SIMT 1
#define DAISY_TOPK_PATH_TC 2
DAISY_API int daisy_topk_full_path(daisy_handle_t h, int *path, int64_t *filtered, int64_t *redone);

/* ---- device-side negative sampler (SURVEY.md section 8f, row N1) ------------------------------------
 * Replaces BPRData.ng_sample (util/data_loader.py:680-690) + the DataLoader(shuffle=True) permutation
 * (BPRMFRecommender.py:141-142) for one epoch: for every training positive pairs[p] = (u, i), num_ng triples
 * (u, i, j) with j uniform over [0, item_num) re-drawn while (u, j) is a training positive; triples_out is
 * int32 [n_pairs * num_ng, 3] on the device, in the reference's features_fill order (positive-major) or, with
 * shuffle != 0, permuted by one epoch-keyed permutation.  pos_keys: the sorted, duplicate-free int64 keys
 * u * item_num + i of the training positives on the device (the role of train_mat).  Deterministic: every draw is
 * Philox4x32-10(key = seed, counter = (slot, epoch, attempt)) -- the rule is restated in oracle/sampler_oracle.py
 * and the two agree bit for bit.  A user whose items are (almost) all positive raises the sticky error flag
 * (daisy_check -> DAISY_EINDEX) after 4096 rejected draws. */
DAISY_API int daisy_sample_triples(daisy_handle_t h, const int32_t *pairs, int64_t n_pairs, int num_ng,
                                   const int64_t *pos_keys, int64_t n_keys, uint64_t seed, uint32_t epoch, int shuffle,
                                   int32_t *triples_out, daisy_stream_t stream);

/* Row-sharded training (SURVEY.md section 8e; no counterpart in the single-device reference): the share of rank
 * [u0, u1) of a GLOBAL epoch.  triples int32 [n,3] (device; global ids, the same on every rank, already shuffled) ->
 * out: the triples whose user lies in [u0, u1), order kept, user column made local; batch_off [ceil(n/batch)+1]
 * (device, int64): where the rank's share of each global batch of `batch` triples starts in out.  Step k of every
 * rank then runs on out[batch_off[k] .. batch_off[k+1]) and the sharded step equals daisy_bpr_step on global batch k. */
DAISY_API int daisy_route_triples(daisy_handle_t h, const int32_t *triples, int64_t n, int64_t batch, int64_t u0,
                                  int64_t u1, int32_t *out, int64_t *batch_off, daisy_stream_t stream);

/* ---- funk-SVD / RSVD (util/matrix_factorization.pyx) ---------------------------------------------
 * variant: 0 = SVD (:132-151), 1 = RSVD version 1, 2 = RSVD version 2 (:41-61).
 * One call runs `n_epochs` passes over the n ratings IN THE GIVEN ORDER with the reference's strictly
 * sequential semantics (update t+1 sees update t): the kernel is a dataflow over per-row version
 * counters, so independent ratings run in parallel and dependent ones in sequence order.
 * Tables are float64 like the reference's (pu [U,dim], qi [I,dim], bu [U], bi [I]); users/items int32,
 * ratings float64, all on the device.  sse_out (device double[n_epochs], may be NULL) receives the sum
 * of squared errors of each epoch. */
typedef struct {
    int variant;
    int biased; /* SVD only */
    double lr_bu, lr_bi, lr_pu, lr_qi;
    double reg_bu, reg_bi, reg_pu, reg_qi;
    double reg2;        /* RSVD2 */
    double global_mean; /* SVD: mu if biased else 0;  RSVD2: mu in the bias coupling */
} daisy_mf_params;

DAISY_API int daisy_mf_fit(daisy_handle_t h, double *pu, double *qi, double *bu, double *bi, const int32_t *users,
                 const int32_t *items, const double *ratings, int64_t n, int n_epochs,
                 const daisy_mf_params *prm, double *sse_out, daisy_stream_t stream);

/* SVD.predict / RSVD.predict (util/matrix_factorization.pyx:157-167, 68-78), batched:
 * est[n] = (with_bias ? mu + bu[u] + bi[i] : 0) + <pu[u], qi[i]>.  Out-of-range codes raise DAISY_EINDEX
 * at daisy_check (ValueError('Invalid user code' / 'Invalid item code') in the reference). */
DAISY_API int daisy_mf_predict(daisy_handle_t h, const double *pu, const double *qi, const double *bu, const double *bi,
                     const int32_t *users, const int32_t *items, int64_t n, int with_bias, double mu,
                     double *est, daisy_stream_t stream);

/* ---- SVD++ (SURVEY section 8f, row N4): SVDpp.fit / SVDpp.predict, util/matrix_factorization.pyx:193-288 -----------
 * GPU-verified in round 2 (tests/test_svdpp_gpu.py); csrc/svdpp.cu has the measured state and the plan.
 * daisy_svdpp_fit runs `n_epochs` passes over the n ratings IN THE GIVEN ORDER with the reference's strictly sequential
 * semantics (loop body :238-263): every rating of user u updates bu[u], bi[i], pu[u], qi[i] and the implicit-feedback
 * row yj[j] of EVERY item j in the user's history.  Tables are float64 like the reference's (pu [U,dim], qi [I,dim],
 * yj [I,dim], bu [U], bi [I]; U, I, dim are the handle's); users/items int32, ratings float64, all on the device.
 * The histories (`ur`, :231-234) come in CSR form: ur_ptr int64 [U+1], ur_idx int32 [ur_ptr[U]] = per user the items
 * of its ratings in frame order.  ur_mult (int32, parallel to ur_idx, may be NULL when no history holds an item twice):
 * the number of occurrences of ur_idx[k] in its user's list if k is the first occurrence, else 0 -- a repeated
 * (user, item) rating makes the reference apply that row's update twice per rating, and so does the kernel.
 * sse_out (device double[n_epochs], may be NULL) receives the sum of squared errors of each epoch.  Out-of-range ids
 * raise DAISY_EINDEX at daisy_check and leave the tables untouched. */
typedef struct {
    double lr_bu, lr_bi, lr_pu, lr_qi, lr_yj;
    double reg_bu, reg_bi, reg_pu, reg_qi, reg_yj;
    double global_mean;
} daisy_svdpp_params;

DAISY_API int daisy_svdpp_fit(daisy_handle_t h, double *pu, double *qi, double *yj, double *bu, double *bi,
                    const int32_t *users, const int32_t *items, const double *ratings, int64_t n, int n_epochs,
                    const int64_t *ur_ptr, const int32_t *ur_idx, const int32_t *ur_mult,
                    const daisy_svdpp_params *prm, double *sse_out, daisy_stream_t stream);

/* The user side of SVDpp.predict (:281-286): z_out[u] = pu[u] + sum_{j in Iu} yj[j] / sqrt|Iu| for every user
 * (a user without history keeps pu[u]); est = global_mean + bu[u] + bi[i] + <qi[i], z[u]> is then
 * daisy_mf_predict(z, qi, bu, bi, ..., with_bias = 1, mu = global_mean). */
DAISY_API int daisy_svdpp_user_factors(daisy_handle_t h, const double *pu, const double *yj, const int64_t *ur_ptr,
                             const int32_t *ur_idx, double *z_out, daisy_stream_t stream);

/* ---- BPR-FM at the reference script's defaults: batch norm + dropout (SURVEY section 8f, row N3) ---------------------
 * GPU-verified in round 2 (tests/test_bprfm_bn_gpu.py); batch_norm off + dropout 0 is daisy_bprfm_adagrad_step.
 * Replaces, for features = [user, user_num + item] with values 1 (util/data_loader.py:159-172, 595-614):
 *   BPRFM._out with nn.BatchNorm1d(num_factors) + nn.Dropout(drop_prob[0])   BPRFMRecommender.py:45-80
 *   the training step + optim.Adagrad over every parameter                    BPRFMRecommender.py:191-193, 214-219
 * All pointers are device pointers owned by the caller (the module's parameter / buffer tensors and the optimizer's
 * state_sum tensors), fp32, contiguous. */
typedef struct {
    float *E;            /* [num_features, F]  embeddings.weight */
    float *bias;         /* [num_features]     biases.weight */
    float *accE, *accb;  /* Adagrad state_sum of the two tables (step only) */
    float *gamma, *beta; /* [F]  FM_layers[0].weight / .bias */
    float *acc_gamma, *acc_beta;        /* their Adagrad state_sum (step only) */
    float *running_mean, *running_var;  /* [F]  FM_layers[0] buffers */
    float lr, eps;       /* Adagrad: lr, eps (torch default 1e-10) */
    float bn_eps, momentum; /* BatchNorm1d: 1e-5, 0.1 */
    int64_t user_num, num_features;     /* features [0, user_num) are users, the rest items */
    int F;               /* num_factors, 1..255 */
} daisy_fmbn_params;

/* Bytes of device scratch daisy_fmbn_step needs for batches of up to B triples (no device call). */
DAISY_API int daisy_fmbn_scratch_bytes(int64_t B, int F, int64_t *bytes);
/* One training step on B >= 2 triples (user, item_i, item_j; item ids relative to user_num).  mask_i / mask_j [B, F]:
 * the dropout masks of the positive / negative _out call, kept elements already scaled by 1 / (1 - p); NULL = no
 * dropout.  loss_accum += -sum log sigmoid(pred_i - pred_j).  Batch statistics, running statistics (updated once per
 * _out call, positive first) and every reduction are computed in a fixed order: bit-reproducible.  Asynchronous. */
DAISY_API int daisy_fmbn_step(daisy_handle_t h, const daisy_fmbn_params *p, const int32_t *triples, int64_t B,
                    const float *mask_i, const float *mask_j, void *scratch, int64_t scratch_bytes,
                    double *loss_accum, daisy_stream_t stream);
/* Evaluation-mode forward (running statistics, no dropout): pred = sum_f BN(e_u * e_item)_f + b_item; the caller adds
 * the user bias and bias_ (equal for every item of a user). */
DAISY_API int daisy_fmbn_forward(daisy_handle_t h, const daisy_fmbn_params *p, const int32_t *triples, int64_t B,
                       float *pred_i, float *pred_j, daisy_stream_t stream);
/* Ranking tables of the evaluation-mode model (BPRFMRecommender.py:57-80 after model.eval()): with
 * a_f = gamma_f / sqrt(running_var_f + bn_eps), P_out [user_num, W] = [a (.) e_u, 1, 0...], Q_out [item_num, W] =
 * [e_i, b_i, 0...] and *c0_out = sum_f (beta_f - a_f running_mean_f), so that the forward score is
 * <P[u], Q[i]> + b_u + bias_ + c0.  W % 4 == 0, W >= F + 1 (the 16-byte rows of the ranking kernels); rank with
 * daisy_topk_candidates / daisy_topk_full on a handle of dim W, then add b_u + bias_ + c0 per user.  Only the forward
 * fields of p are read.  Deterministic: the same bits on every call. */
DAISY_API int daisy_fmbn_rank_tables(daisy_handle_t h, const daisy_fmbn_params *p, int W, float *P_out, float *Q_out,
                                     float *c0_out, daisy_stream_t stream);

/* ---- Item2Vec / skip-gram with negative sampling (SURVEY section 8f, row N4) ---------------------------------------
 * GPU-verified in round 2 (tests/test_sgns_gpu.py).
 * Replaces Item2Vec.forward_i / forward_o + SGNS.forward (Item2VecRecommender.py:60-97) with the negatives given, and
 * loss.backward() + optim.Adam(sgns.parameters()).step() (:266, 274-277; torch's Adam is dense: every row of both
 * tables is stepped).  Device pointers owned by the caller, fp32, contiguous. */
typedef struct {
    float *iv, *ov;                  /* [vocab, D]  embedding.ivectors.weight / embedding.ovectors.weight */
    float *m_iv, *v_iv, *m_ov, *v_ov; /* Adam exp_avg / exp_avg_sq of the two tables */
    float lr, beta1, beta2, eps;     /* torch defaults: 1e-3, 0.9, 0.999, 1e-8 */
    int64_t vocab;
    int D;                           /* embedding size, 1..512 */
    int padding_idx;                 /* row that receives no gradient (nn.Embedding(padding_idx=0)); -1 = none */
} daisy_sgns_params;

/* Bytes of device scratch daisy_sgns_step needs (no device call). */
DAISY_API int daisy_sgns_scratch_bytes(int64_t B, int C, int n_negs, int64_t vocab, int D, int64_t *bytes);
/* One training step: iword [B], owords [B, C], nwords [B, C * n_negs] (the layout of :86-87), step_no 1-based (Adam's
 * bias correction).  loss_accum += the batch loss of :97 (mean form).  Fixed-order reductions: bit-reproducible. */
DAISY_API int daisy_sgns_step(daisy_handle_t h, const daisy_sgns_params *p, const int32_t *iword, const int32_t *owords,
                    const int32_t *nwords, int64_t B, int C, int n_negs, int64_t step_no, void *scratch,
                    int64_t scratch_bytes, double *loss_accum, daisy_stream_t stream);

/* ---- NCF with an MLP tower: model 'MLP' and the script's default 'NeuMF-end' (SURVEY section 8f, row N3) ----------
 * GPU-verified in round 2 (tests/test_neumf_gpu.py); the GMF variant is daisy_gmf_step.
 * Replaces NCF.forward (NCFRecommender.py:105-125) with dropout 0 and the training step :283-287 with
 * nn.BCEWithLogitsLoss() (:255) and optim.Adam(model.parameters(), lr) (:260).  Device pointers owned by the caller (the
 * module's parameter tensors and the optimizer's exp_avg / exp_avg_sq), fp32, contiguous; torch's Linear layout
 * W_l [out_l, in_l] with in_0 = 2 * factor * 2^(num_layers - 1), out_l = in_l / 2. */
#define DAISY_NEUMF_MAX_LAYERS 6
typedef struct {
    int neumf;               /* 0: model 'MLP' (the GMF tables are not touched), 1: 'NeuMF-end' */
    int num_layers, factor;  /* factor * 2^num_layers <= 1024 */
    int64_t user_num, item_num;
    float *Pg, *Qg;          /* embed_user_GMF / embed_item_GMF  [n, factor]                     (neumf only) */
    float *Pm, *Qm;          /* embed_user_MLP / embed_item_MLP  [n, factor * 2^(num_layers-1)] */
    float *W[DAISY_NEUMF_MAX_LAYERS], *b[DAISY_NEUMF_MAX_LAYERS];   /* MLP_layers Linear weights / biases */
    float *wp, *bp;          /* predict_layer weight [factor or 2 * factor: GMF part first], bias [1] */
    float *m_Pg, *v_Pg, *m_Qg, *v_Qg, *m_Pm, *v_Pm, *m_Qm, *v_Qm;   /* Adam moments (step only) */
    float *m_W[DAISY_NEUMF_MAX_LAYERS], *v_W[DAISY_NEUMF_MAX_LAYERS], *m_b[DAISY_NEUMF_MAX_LAYERS], *v_b[DAISY_NEUMF_MAX_LAYERS];
    float *m_wp, *v_wp, *m_bp, *v_bp;
    float lr, beta1, beta2, eps;
} daisy_neumf_params;

/* Bytes of device scratch daisy_neumf_step needs for batches of up to B samples (no device call). */
DAISY_API int daisy_neumf_scratch_bytes(const daisy_neumf_params *p, int64_t B, int64_t *bytes);
/* logits[B] of (user, item, label) int32 samples (the label column is ignored). */
DAISY_API int daisy_neumf_forward(daisy_handle_t h, const daisy_neumf_params *p, const int32_t *samples, int64_t B,
                        float *logits, daisy_stream_t stream);
/* One training step on B (user, item, label) samples; step_no is 1-based (Adam's bias correction);
 * loss_accum += the batch's mean BCE.  Fixed-order reductions: bit-reproducible. */
DAISY_API int daisy_neumf_step(daisy_handle_t h, const daisy_neumf_params *p, const int32_t *samples, int64_t B,
                     int64_t step_no, void *scratch, int64_t scratch_bytes, double *loss_accum, daisy_stream_t stream);

/* Ranking with the tower: score(u, i) = the logit NCF.forward returns (NCFRecommender.py:105-125), up to the fp32
 * reassociation of layer 0, which is split into a per-user and a per-item half.  Only the forward fields of p are read
 * (the Adam moment pointers may be NULL).  Scores are fp32 sums in a fixed order: a user's results are the same bits
 * whether it is ranked alone or with others, and in both entry points.
 * metric_eval(model, test_loader, top_k, algo='ncf') -> _ncf_topk (util/metrics.py:68-86,88-94), all groups at once:
 * for n < N the K best of score(users[n], cand[n,c]), c < C, in (score desc, position asc) order; out_pos [N,K] =
 * candidate positions, out_item [N,K] = cand ids, out_score [N,K].  C <= 8192, K <= 128, K <= C
 * (the layout of daisy_topk_candidates). */
DAISY_API int daisy_neumf_topk_candidates(daisy_handle_t h, const daisy_neumf_params *p, const int32_t *users,
                                          const int32_t *cand, int64_t N, int C, int K, int32_t *out_pos,
                                          int32_t *out_item, float *out_score, daisy_stream_t stream);
/* Full catalogue: for n < N the K best items of score(users[n], i), i < item_num, order (score desc, item asc), with
 * optional CSR exclusion lists (the user's training positives) as in daisy_topk_full.  K <= 128. */
DAISY_API int daisy_neumf_topk_full(daisy_handle_t h, const daisy_neumf_params *p, const int32_t *users, int64_t N, int K,
                                    const int64_t *excl_ptr, const int32_t *excl_idx, int32_t *out_item,
                                    float *out_score, daisy_stream_t stream);

/* ---- introspection for tests / bench ------------------------------------------------------------- */
/* Number of kernels launched by this handle since creation (the bench's gpu_launches claim). */
DAISY_API int daisy_launch_count(daisy_handle_t h, int64_t *n);
/* Device time (ms) of the dominant kernel of the last daisy_bpr_step, measured with CUDA events on the
 * launching stream when timing was enabled with daisy_set_timing(h, 1).  Synchronises. */
DAISY_API int daisy_set_timing(daisy_handle_t h, int on);
DAISY_API int daisy_last_step_timing(daisy_handle_t h, float *ms_main_kernel, float *ms_total);
/* Timing mode 1 (asynchronous, main fused kernel only): average device time of that kernel over the steps
 * issued since daisy_set_timing(h, 1), and how many launches were measured.  Synchronises on the events. */
DAISY_API int daisy_main_kernel_ms(daisy_handle_t h, double *avg_ms, int64_t *count);
/* daisy_topk_full with timing on (daisy_set_timing(h, 1)): device time of the tensor-core filter kernel (k_filter_tc)
 * and of the whole call's filtered path, averaged over the calls since the last query; *count = filter launches
 * measured (0: the tensor-core filter did not run).  Synchronises on the events; resets the averages. */
DAISY_API int daisy_topk_tc_ms(daisy_handle_t h, double *filter_ms, double *rescore_ms, int64_t *count);
/* Timing mode 2 (synchronises once per step): average device time of each phase of the step, in launch order:
 * prep, sort_i, refs, sort_u, sort_q, slots, main, seg_u, seg_q, heavy, loss (11 values). */
#define DAISY_NUM_PHASES 11
DAISY_API int daisy_phase_ms(daisy_handle_t h, double *avg_ms, int n, int64_t *steps);
/* Timeline of the first 48 steps after daisy_trace(h, 1, NULL, 0, NULL): per step 4 offsets in ms from the first
 * event -- bookkeeping begin, bookkeeping end (bookkeeping stream), table kernels begin, end (caller's stream).
 * A call with ms != NULL dumps what was recorded (synchronises) before applying `on`. */
DAISY_API int daisy_trace(daisy_handle_t h, int on, double *ms, int cap, int *n_steps);
/* Pin rows [0, n_rows) of the item table in L2 through a stream access-policy window
 * (hot items first when the catalogue is popularity-ordered).  n_rows = 0 clears the window. */
DAISY_API int daisy_set_l2_window(daisy_handle_t h, const float *Q, int64_t n_rows, float hit_ratio,
                        daisy_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DAISY_B200_H */
