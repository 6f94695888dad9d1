/*
 * c2v_b200.h -- C ABI of the B200-native path-attention engine (libc2v_b200.so).
 *
 * This is the drop-in boundary for code2vec's ONE hot path.  The reference (tech-srl/code2vec)
 * has no FFI of its own: its seam is the Python ABC Code2VecModelBase (model_base.py:37-182)
 * whose TensorFlow backend runs the whole path inside sess.run() calls.  Each entry point below
 * names the reference statement(s) it replaces (file:line relative to the reference root), so a
 * maintainer can bind it from a third backend (`--framework b200`, see INTEGRATION.md).
 *
 * Conventions
 *   - plain C, no CUDA / torch types: device pointers are `void*`/`float*`/`int32_t*` holding
 *     device addresses, a stream is the `cudaStream_t` value passed as `void*` (NULL = default).
 *   - every function returns 0 (C2V_OK) or a negative c2v_status; the message of the last
 *     failure is kept per engine (c2v_last_error).  Nothing throws across the boundary.
 *   - the caller owns all big buffers (parameters, gradients, Adam slots, workspace) -- in the
 *     Python backend they are torch tensors used purely as storage.  The engine allocates
 *     nothing on the device after c2v_create.
 *   - all calls are asynchronous w.r.t. the host on `stream`, except the *_host entry points,
 *     which synchronise the stream before returning because they hand results back to the host.
 *   - one host thread per engine at a time; engines are independent.
 *   - layouts: row-major, float32 parameters, int32 indices, float32 0/1 mask -- the dtypes the
 *     reference reader emits (path_context_reader.py:32-44,214; vocabularies.py:112).
 */
#ifndef C2V_B200_H_
#define C2V_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C2V_ABI_VERSION 1

typedef struct c2v_engine c2v_engine;

typedef enum c2v_status {
  C2V_OK = 0,
  C2V_ERR_INVALID = -1,      /* bad argument (NULL, size out of range, unsupported dims)   */
  C2V_ERR_CUDA = -2,         /* a CUDA runtime call or kernel launch failed                */
  C2V_ERR_STATE = -3,        /* call order violated (e.g. train step before binding grads) */
  C2V_ERR_UNSUPPORTED = -4   /* valid request this build cannot serve                      */
} c2v_status;

/* Shapes of the model (config.py:60-68; vocab sizes include the special words,
 * vocabularies.py:51-55).  code_dim is CODE_VECTOR_SIZE (= 3*embed_dim by default). */
typedef struct c2v_dims {
  int32_t token_vocab;   /* T: rows of WORDS_VOCAB          (tensorflow_model.py:206-209) */
  int32_t path_vocab;    /* P: rows of PATHS_VOCAB          (tensorflow_model.py:217-220) */
  int32_t target_vocab;  /* Y: rows of TARGET_WORDS_VOCAB   (tensorflow_model.py:210-213) */
  int32_t embed_dim;     /* d: TOKEN/PATH_EMBEDDINGS_SIZE, multiple of 4                  */
  int32_t code_dim;      /* D: CODE_VECTOR_SIZE, multiple of 4, <= 1024                   */
  int32_t max_contexts;  /* C: MAX_CONTEXTS                                               */
  int32_t max_batch;     /* largest batch any call will pass                              */
  int32_t top_k;         /* TOP_K_WORDS_CONSIDERED_DURING_PREDICTION (<= 64)              */
} c2v_dims;

/* The five variables of the model, in the order the reference creates them
 * (tensorflow_model.py:32-36,205-220,249-250).  Used for parameters, gradients and Adam slots.
 *   tok  [T, d]   WORDS_VOCAB            path [P, d]   PATHS_VOCAB
 *   tgt  [Y, D]   TARGET_WORDS_VOCAB     W    [3d, D]  TRANSFORM          a [D] ATTENTION */
typedef struct c2v_tensors {
  float* tok;
  float* path;
  float* tgt;
  float* W;
  float* a;
} c2v_tensors;

/* Arithmetic of the three big matrix products (projection, logits, their gradients).
 *   C2V_MATH_FP32  : fp32 FFMA on the SIMT pipe -- the reference's own arithmetic class
 *                    (cuBLAS/Eigen SGEMM); used for bit-level top-k parity.
 *   C2V_MATH_TF32  : tcgen05.mma kind::tf32 (fp32 storage, 10-bit mantissa operands, fp32
 *                    accumulate in TMEM) -- what TensorFlow itself runs on Ampere+ GPUs.
 *   C2V_MATH_3XTF32: the same tensor-core kernels at fp32-equivalent accuracy: every operand is
 *                    split into tf32 high and low parts (x = hi + lo up to 2^-22 |x|) and a product
 *                    is issued as a_lo.b_hi + a_hi.b_lo + a_hi.b_hi into the same fp32 TMEM
 *                    accumulator (the dropped a_lo.b_lo term is O(2^-22) relative); tanh / exp in the
 *                    epilogues use the correctly rounded library forms.  The reference's arithmetic
 *                    class (fp32 tf.matmul, tensorflow_model.py:226,252,297) on tensor cores. */
typedef enum c2v_math_mode { C2V_MATH_FP32 = 0, C2V_MATH_TF32 = 1, C2V_MATH_3XTF32 = 2 } c2v_math_mode;

int c2v_abi_version(void);

/* Message of the last failed call on `e`; with e == NULL, of the last failed c2v_create /
 * c2v_workspace_bytes on this thread.  Never NULL. */
const char* c2v_last_error(const c2v_engine* e);

/* Bytes of device scratch the engine needs for `dims` (activations kept for the backward pass,
 * the [B, Y] logits slab, split-K partials, host-API staging).  0 on invalid dims. */
size_t c2v_workspace_bytes(const c2v_dims* dims);

/* Create an engine for CUDA device `device`.  Replaces Code2VecModel.__init__'s
 * tf.compat.v1.Session() (tensorflow_model.py:19-38). */
int c2v_create(const c2v_dims* dims, int device, c2v_engine** out);

/* Replaces close_session() (tensorflow_model.py:439-440).  NULL is a no-op. */
void c2v_destroy(c2v_engine* e);

int c2v_bind_workspace(c2v_engine* e, void* dev_ptr, size_t bytes);   /* >= c2v_workspace_bytes, 256-B aligned */
int c2v_bind_params(c2v_engine* e, const c2v_tensors* theta);         /* tf.get_variable x5, :205-220,249-250   */
int c2v_bind_grads(c2v_engine* e, const c2v_tensors* grads);          /* autodiff outputs of minimize(), :232   */
int c2v_bind_adam_state(c2v_engine* e, const c2v_tensors* m, const c2v_tensors* v);  /* Adam slots, :232       */

/* Options: "math_mode" (c2v_math_mode), "deterministic" (reserved: only 0 is accepted -- the
 * embedding scatter-add uses float atomics; every other reduction is fixed-order), "cta_pair"
 * (tcgen05 GEMMs as CTA pairs, tcgen05.mma.cta_group::2: 0 never, 1 always, 2 auto = per GEMM,
 * wherever it measured faster; default 2), "dy_late" (where the target-table gradient GEMM dY = P^T.v -- with the
 * target table's Adam step in its epilogue when armed -- runs: 0 = right after dv on the caller's
 * stream, "target_grads_ready" fires earliest; 1 = default: inside the context backward pass, next
 * to the embedding scatter-add; 2 = on an engine-owned stream right after dv, joined before the
 * step returns.  All three measure within 1 % of each other on one GPU: the persistent GEMM CTAs
 * fill the register file, so kernels on other streams mostly wait for them), "profile" (0/1: per-phase
 * CUDA-event timing, read with c2v_phase_stats), "lazy_adam" (0/1, single-GPU replicated tables:
 * the dense TF1 Adam update of an embedding row is deferred -- its gradient stays in the bound
 * gradient table -- and replayed bit-exactly (one step with that gradient, then the zero-gradient
 * steps) when a later batch references the row; same results as the dense update, one pass over
 * the batch's rows per step instead of 9 GB of traffic.  While it is on, the token / path gradient
 * tables are engine state (deferred steps), every c2v_train_step must be followed by
 * c2v_adam_step with consecutive t, and c2v_sync_tables brings every row up to date),
 * "adam_step_count" (the number of Adam steps already applied: optimizer reset / restore),
 * "grad_scale_inverse" (n: embedding scatter-adds are scaled by 1/n), "fuse_target_adam" (0/1,
 * default 0: c2v_train_batch_host arms c2v_arm_target_adam itself), "target_adam_fused_step"
 * (read: the step count whose target-table update the dY epilogue has already applied, 0 = none;
 * writing 0 acknowledges it for callers that drive c2v_adam_step_range themselves),
 * "early_catchup_count" (read-only: how many train steps used a c2v_hint_next_batch hint),
 * "adam_rows_occupancy" (4 or 5 resident blocks per SM for the lazy-Adam row pass; default 4),
 * "adam_sweep_period" (R, default 32, 0 = off: with lazy_adam every c2v_adam_step also brings rows
 * [rows*(t mod R)/R, rows*(t mod R + 1)/R) of each lazily updated table up to date, so that no row is
 * ever more than R steps behind -- this bounds the replay a rarely referenced row costs when a batch
 * finally reads it, and the cost of c2v_sync_tables, whatever the index distribution; results are
 * unchanged, the deferred steps are only applied earlier), "adam_rest_shortcut" (0/1, default 1: a row's
 * zero-gradient replay stops dividing / taking square roots once an update no longer changes any element of
 * the row -- updates shrink monotonically from there, so the parameters provably stay put and only the
 * slots keep decaying; bit-identical to the full replay for 0 < beta1 <= 0.95 and 0.99 <= beta2 < 1, and
 * not applied outside that range), "exp_slab" (0/1, default 1; tensor-core math modes, single-GPU full-softmax
 * train step): the logits GEMM's epilogue writes U = exp(logit - true-class logit) instead of the logits, one element
 * per row is patched and the softmax's 1 / sum is applied as a per-example factor by the two target-side gradient
 * GEMMs, so no pass re-reads the [B, Y] slab to normalise it; a step in which some row's largest U leaves the fp32
 * window [1e-26, 1e30] is redone on the device as the two-pass schedule (logits stored, then rewritten) -- read-only
 * "exp_slab_fallbacks" counts those steps (the read synchronises the device), "sort_peer_access" (row-sharded
 * tables over peer memory: 0 never, 1 = default: when a table exceeds 2 GB, 2 always -- the step's row indices are
 * counting-sorted by (owner, 2 MB page) before the peer gather / scatter-add).
 * Experimental schedules, all correct, all measured slower on B200 and therefore 0 by default (DESIGN.md sections
 * 4.6 - 4.8): "fuse_gather" (the gather feeds the context GEMM's shared-memory stages directly), "fuse_softmax_grad"
 * (dv / dY turn logits into dL/dlogits as their A tiles land; tf32 mode), "recompute_logits" (the logits GEMM runs
 * twice instead of storing logits), "adam_epilogue_prefetch" (the dY GEMM's Adam epilogue prefetches the (theta, m, v)
 * lines of its next tile into L2: dY 0.77 ms instead of 0.69). */
int c2v_set_option(c2v_engine* e, const char* key, int64_t value);
int c2v_get_option(const c2v_engine* e, const char* key, int64_t* value);

/* _calculate_weighted_contexts(..., is_evaluating=True)  (tensorflow_model.py:236-265):
 * three gathers, concat, tanh(x.W), attention score, log-mask, softmax over the bag, weighted
 * sum.  src/path/tgt/mask: device [B, C].  code_vec: device [B, D].  attn: device [B, C] or
 * NULL.  A bag with no valid context yields NaN (as tf.nn.softmax of all -inf does). */
int c2v_forward(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt,
                const float* mask, int32_t B, float* code_vec, float* attn, void* stream);

/* scores = code_vec . TARGET_WORDS_VOCAB^T ; tf.nn.top_k(scores, k) sorted descending, ties to
 * the lower index (tensorflow_model.py:297-306).  normalize: 0 = raw scores (evaluate); 1 =
 * softmax over the k values (TF backend's predict, :305-306); 2 = probabilities of the softmax
 * over the whole target vocabulary (Keras backend: Dense(softmax) then top_k,
 * keras_model.py:69-70, keras_topk_word_predictions_layer.py:30-35).
 * idx: device int32 [B, k]; val: device float [B, k]. */
int c2v_topk(c2v_engine* e, const float* code_vec, int32_t B, int32_t* idx, float* val,
             int32_t normalize, void* stream);

/* ---- Nearest-neighbour search: gensim's KeyedVectors.most_similar on a device-resident matrix -----------
 * What the reference README runs on the --save_t2v / --save_w2v text files (README.md:236-251), and the search
 * of a code-vector corpus (--export_code_vectors, c2v_predict_batch_host) for the methods closest to a snippet.
 * bank: device fp32 [rows, dim], row-major, 16-byte aligned, dim % 4 == 0, dim <= 1024, 1 <= rows < 2^31 -- a bound
 * table (theta.tgt / tok / path; with "lazy_adam" on, call c2v_sync_tables first, otherwise deferred rows are read
 * stale) or any caller matrix such as code vectors.  Row norms are computed in the same pass as the dot products
 * (nothing is cached), in fp32 FFMA.  Neither call uses the workspace or changes engine state, so a search
 * between two train steps leaves the next step bit-identical.  Both are asynchronous on `stream`.
 *
 *   c2v_nearest_scratch_bytes : device scratch c2v_nearest needs for (rows, n, k) (per-CTA candidate lists); 0 when
 *                               the arguments are out of range.
 *   c2v_compose_queries       : gensim's query vector, unitvec(mean_t(w_t * x_t)), for n queries of up to
 *                               max_terms (<= 16) terms each.  term_rows / term_weights: device [n, max_terms];
 *                               term_rows[q, t] >= 0: x_t = bank row / its norm (a zero row adds nothing);
 *                               -2: x_t = term_vectors[q, t, :] as given (device [n, max_terms, dim], may be NULL
 *                               when no -2 occurs); -1 (or a row outside the bank): no term.  weights: +1 for a
 *                               positive term, -1 for a negative one.  queries: device [n, dim] output; a query
 *                               with no term or a zero mean is all zeros.
 *   c2v_nearest               : cosine top-k of n query vectors (device [n, dim], any n: chunked internally)
 *                               against the bank: idx / val device [n, k], score descending, ties to the lower
 *                               row.  1 <= k <= 64.  exclude: device [n, n_exclude] row ids never returned for
 *                               that query (-1 = padding), n_exclude <= 16, NULL when 0.  Zero rows and rows whose
 *                               score is NaN are never returned; a zero query returns nothing; slots beyond the
 *                               available results hold idx = -1, val = -inf.  Results do not depend on n or on how
 *                               the queries are batched.  scratch: 16-byte aligned device memory of at least
 *                               c2v_nearest_scratch_bytes(rows, n, k) bytes. */
size_t c2v_nearest_scratch_bytes(int64_t rows, int32_t n, int32_t k);
int c2v_compose_queries(c2v_engine* e, const float* bank, int64_t rows, int32_t dim, const int32_t* term_rows,
                        const float* term_weights, const float* term_vectors, int32_t n, int32_t max_terms,
                        float* queries, void* stream);
int c2v_nearest(c2v_engine* e, const float* bank, int64_t rows, int32_t dim, const float* queries, int32_t n,
                int32_t k, const int32_t* exclude, int32_t n_exclude, int32_t* idx, float* val, void* scratch,
                size_t scratch_bytes, void* stream);

/* Mean sparse-softmax cross entropy of code_vec against `target` without gradients
 * (tensorflow_model.py:226-230).  loss_out: device float[1]. */
int c2v_loss(c2v_engine* e, const float* code_vec, const int32_t* target, int32_t B,
             float* loss_out, void* stream);

/* Forward + backward of the training graph (tensorflow_model.py:197-234 without the Adam
 * update): dropout with keep probability `keep_prob` (config.py:69; 1.0 disables it), full
 * softmax loss, gradients of all five variables written to the bound gradient tensors
 * (overwriting them; embedding rows that received no contribution are exactly 0).
 *   dropout_mask : NULL -> counter-based Philox4x32-10 mask from (seed, step), regenerated in
 *                  the backward pass; or device float [B*C, 3d] of 0/1 supplied by the caller.
 *   loss_out     : device float[1], mean loss over the B examples (dynamic batch, :227).
 * target: device int32 [B]. */
int c2v_train_step(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt,
                   const float* mask, const int32_t* target, int32_t B, float keep_prob,
                   uint64_t seed, uint64_t step, const float* dropout_mask, float* loss_out,
                   void* stream);

/* Same with a sampled softmax over {target_b} U sampled[0..S) instead of the full softmax.
 * NOT IN THE REFERENCE (BASELINE config 3; semantics defined in DESIGN.md after
 * tf.nn.sampled_softmax_loss): logq_* are the log expected counts subtracted from the logits,
 * a sampled class equal to a row's target is masked out for that row. */
int c2v_sampled_train_step(c2v_engine* e, const int32_t* src, const int32_t* path,
                           const int32_t* tgt, const float* mask, const int32_t* target,
                           int32_t B, const int32_t* sampled, int32_t S, const float* logq_true,
                           const float* logq_sampled, float keep_prob, uint64_t seed,
                           uint64_t step, const float* dropout_mask, float* loss_out,
                           void* stream);

/* tf.compat.v1.train.AdamOptimizer() update of all five variables from the bound gradients
 * (tensorflow_model.py:232): lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v decay on EVERY row (TF1's
 * sparse apply is not lazy); theta -= lr_t*m/(sqrt(v)+eps).  t is the 1-based step count. */
int c2v_adam_step(c2v_engine* e, float lr, float beta1, float beta2, float eps, int64_t t,
                  void* stream);

/* Folds the TARGET_WORDS_VOCAB part of that update into the backward pass (tcgen05 path, full
 * softmax): once armed, the next target-gradient product dY = P^T.v applies Adam step t to
 * (theta, m, v) of the target table in its epilogue -- bit-identical to c2v_adam_step, but dY is
 * never written (the bound target gradient buffer keeps stale values) and the 401 MB table is not
 * re-read.  The following c2v_adam_step(t) with the same hyper-parameters skips the target table
 * (different ones are an error).  If the step that follows cannot fuse (fp32 path, sampled
 * softmax) the arming is dropped and c2v_adam_step updates the table as usual.  Same semantics as
 * tensorflow_model.py:232; no reference statement of its own. */
int c2v_arm_target_adam(c2v_engine* e, float lr, float beta1, float beta2, float eps, int64_t t);

/* Next-batch hint for "lazy_adam" (one-shot, optional; tf.data's prefetch, path_context_reader.py:150,
 * is what makes the next batch known in the reference too): the index arrays [B, C] of the batch
 * the NEXT train step will run on.  If the current step is armed (c2v_arm_target_adam supplies the
 * step's hyper-parameters) the deferred updates of that batch's embedding rows are applied during
 * the current step's backward pass, on the engine's side stream next to the dY / dW GEMMs,
 * instead of at the head of the next step.  Results are identical with or without the hint; a
 * wrong hint only costs the overlap.  Device pointers must stay valid until the next train step
 * has been issued; the _host variant copies from host memory into the engine's staging area. */
int c2v_hint_next_batch(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt,
                        int32_t B);
int c2v_hint_next_batch_host(c2v_engine* e, const int32_t* h_src, const int32_t* h_path,
                             const int32_t* h_tgt, int32_t B, void* stream);

/* ---- Phase-split train step for the fully sharded schedule (BASELINE config 5) -----------------------
 * The target table is row-sharded too: this engine is created with target_vocab = the number of
 * LOCAL rows and max_batch = the GLOBAL batch Bt.  Between the phases the caller moves only small
 * tensors: all-gather of code vectors [Bt, D], all-gather of per-row (max, sum exp) [Bt] and an
 * all-reduce of the true logits [Bt], reduce-scatter of dv [Bt, D] -- never a [*, Y] slab and
 * never a table gradient.
 *   c2v_context_forward : training forward of the local examples (dropout as c2v_train_step) ->
 *                         code_vec [B, D]; activations stay in the workspace for the backward pass.
 *   c2v_target_forward  : S = code_all . Ytab_local^T for all Bt examples; row_max / row_sum [Bt] =
 *                         max and sum exp(. - max) over the local classes; this engine's rows are
 *                         global rows [row_offset, row_offset + target_vocab): true_logit [Bt] =
 *                         S[b, target[b] - row_offset] if that row lives here, else 0
 *                         (target = global class ids of all Bt examples).
 *   c2v_lse_combine     : the ranks' partials maxes / sums [world, Bt] (after all-gather) and the
 *                         all-reduced true logits -> lse [Bt], mean loss (inv_batch = 1/Bt).
 *   c2v_target_backward : S <- (exp(S - lse) - onehot(target - row_offset)) * inv_batch; dv_partial [Bt, D] =
 *                         P . Ytab_local; the bound target gradient (local rows) = P^T . code_all.
 *   c2v_context_backward: rest of the backward pass of the local examples given dv [B, D]
 *                         (after the reduce-scatter): attention, TRANSFORM / ATTENTION gradients,
 *                         scatter-add into the (sharded) embedding gradient tables. */
int c2v_context_forward(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt,
                        const float* mask, int32_t B, float keep_prob, uint64_t seed, uint64_t step,
                        const float* dropout_mask, float* code_vec, void* stream);
int c2v_target_forward(c2v_engine* e, const float* code_all, int32_t Bt, const int32_t* target,
                       int32_t row_offset, float* row_max, float* row_sum, float* true_logit,
                       void* stream);
int c2v_lse_combine(c2v_engine* e, const float* maxes, const float* sums, int32_t world, int32_t Bt,
                    const float* true_logit, float inv_batch, float* lse_out, float* loss_out,
                    void* stream);
int c2v_target_backward(c2v_engine* e, const float* code_all, int32_t Bt, const float* lse,
                        const int32_t* target, int32_t row_offset, float inv_batch, float* dv_partial,
                        void* stream);
int c2v_context_backward(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt,
                         const float* mask, int32_t B, float keep_prob, uint64_t seed, uint64_t step,
                         const float* dropout_mask, const float* dv, void* stream);

/* With "lazy_adam" on: replay all deferred updates so that the bound token / path tables (and their
 * Adam slots) hold exactly what the dense optimizer would hold after the steps applied so far.  Call
 * before reading the parameter tensors from outside the engine (export, checkpoint).  No-op otherwise. */
int c2v_sync_tables(c2v_engine* e, void* stream);

/* The same update on one contiguous slice of caller-provided device arrays (count % 4 == 0,
 * 16-byte aligned): the sharded-optimizer path of a data-parallel run, where each rank owns
 * 1/world of the flat parameter buffer (reduce-scatter grads -> this -> all-gather params). */
int c2v_adam_step_range(c2v_engine* e, float* theta, float* grad, float* m, float* v,
                        size_t count, float lr, float beta1, float beta2, float eps, int64_t t,
                        int32_t zero_grad, void* stream);

/* Row-sharded embedding tables over the GPUs of one NVSwitch domain (data-parallel runs).  Global
 * row r of WORDS_VOCAB / PATHS_VOCAB lives on rank (r % world) at local row (r / world); tok[i] /
 * path[i] are device pointers to rank i's shard -- the caller's own allocation for i == rank,
 * CUDA-IPC mappings of the peers' allocations otherwise.  The forward gather then reads peer
 * memory directly and the backward scatter-add issues red.global.add to the owning rank, scaled
 * by grad_scale (1/world for a mean over the global batch): no table gradient is ever
 * all-reduced and each rank updates only its own rows with c2v_adam_step_range.  The caller
 * provides the cross-rank ordering (all scatters done before Adam; all Adams done before the next
 * gather).  world must be 1, 2, 4 or 8.  grads may be NULL (inference). */
typedef struct c2v_table_shards {
  int32_t world;
  int32_t rank;
  float* tok[8];
  float* path[8];
} c2v_table_shards;
int c2v_bind_table_shards(c2v_engine* e, const c2v_table_shards* params, const c2v_table_shards* grads,
                          float grad_scale);

/* Push-based embedding-gradient exchange for row-sharded tables.  Every rank owns an INBOX in peer-visible memory
 * (c2v_ipc_alloc, c2v_scatter_inbox_bytes(dims, world) bytes) with one region per sending rank.  With inboxes bound,
 * the backward pass no longer issues 16-byte red.global.add over NVLink: it sorts its 3 B C gradient rows by owning
 * rank and writes each owner's rows -- (local row id, d floats) -- DENSELY into its region of that owner's inbox with
 * plain coalesced stores; after the caller's cross-rank barrier (the same one that ordered the remote red.adds before)
 * each owner folds its inbox into its own gradient shards with local atomics (c2v_apply_scatter_inbox).
 * inbox[r] = rank r's inbox as mapped into this process (r == rank: the local allocation). */
size_t c2v_scatter_inbox_bytes(const c2v_dims* dims, int32_t world);
int c2v_bind_scatter_inbox(c2v_engine* e, void* const* inbox, int32_t world, int32_t rank);
int c2v_apply_scatter_inbox(c2v_engine* e, void* stream);

/* cudaMalloc'ed, zero-filled, IPC-shareable device memory for the shards (not tied to an engine;
 * errors are reported through c2v_last_error(NULL)).  handle64 is a 64-byte cudaIpcMemHandle_t. */
int c2v_ipc_alloc(int device, size_t bytes, void** dev_ptr, unsigned char* handle64);
int c2v_ipc_open(int device, const unsigned char* handle64, void** dev_ptr);
int c2v_ipc_close(int device, void* dev_ptr);
int c2v_ipc_free(int device, void* dev_ptr);

/* Register a cudaEvent_t (passed as void*; NULL unregisters) that c2v_train_step records on its
 * stream at a named point, so the caller can start communication early on another stream:
 *   "target_grads_ready" : the TARGET_WORDS_VOCAB gradient is complete (right after dY), while
 *                          the context backward pass is still to run. */
int c2v_set_event(c2v_engine* e, const char* name, void* cuda_event);

/* --- host-buffer entry points: what the backend's train()/evaluate()/predict() call -------- */

/* One `sess.run([optimizer, train_loss])` (tensorflow_model.py:80): copies the batch from host
 * memory (pinned memory makes the copies asynchronous), runs c2v_train_step + c2v_adam_step
 * with the TF defaults given, copies the loss back and synchronises.  h_* are HOST pointers. */
int c2v_train_batch_host(c2v_engine* e, const int32_t* h_src, const int32_t* h_path,
                         const int32_t* h_tgt, const float* h_mask, const int32_t* h_target,
                         int32_t B, float keep_prob, uint64_t seed, int64_t t, float lr,
                         float beta1, float beta2, float eps, float* h_loss, void* stream);

/* The same step WITHOUT waiting for it: the asynchronous half of the batcher that replaces tf.data's prefetch
 * (path_context_reader.py:150).  The five h_* arrays must be page-locked host memory that stays untouched until
 * `upload_done_event` (a cudaEvent_t, may be NULL) has completed: the copies run on an engine-owned copy stream, behind the
 * step that last used the same one of two device staging sets, so the upload of batch t+1 overlaps the kernels of batch t.
 * The step itself (arm target Adam if "fuse_target_adam", train step, Adam step t) is queued on `stream` behind the upload;
 * the loss is copied to h_loss (page-locked, 4 bytes) on `stream` and is valid once `stream` has been synchronised. */
int c2v_train_batch_async(c2v_engine* e, const int32_t* h_src, const int32_t* h_path, const int32_t* h_tgt,
                          const float* h_mask, const int32_t* h_target, int32_t B, float keep_prob,
                          uint64_t seed, int64_t t, float lr, float beta1, float beta2, float eps,
                          float* h_loss, void* upload_done_event, void* stream);

/* One `sess.run([top_words, top_values, ..., code_vectors])` of the test graph
 * (tensorflow_model.py:157-161,331-335).  Outputs are HOST pointers; h_code_vec [B, D] and
 * h_attn [B, C] may be NULL. */
int c2v_predict_batch_host(c2v_engine* e, const int32_t* h_src, const int32_t* h_path,
                           const int32_t* h_tgt, const float* h_mask, int32_t B,
                           int32_t normalize, int32_t* h_topk_idx, float* h_topk_val,
                           float* h_code_vec, float* h_attn, void* stream);

/* Test hook for the tcgen05 GEMM building block: C = A . B with tf32 operands.  a_mn / b_mn
 * select the operand layout (0: K contiguous, element (x,k) at p[x*ld+k]; 1: M resp. N
 * contiguous, element (x,k) at p[k*ld+x]); bn is the N tile (192 or 256); with splits > 1,
 * slice s of the K range is written to C + s*M*ldc.  Returns the number of slices (> 0) or an
 * error (< 0).  All pointers are device pointers. */
int c2v_selftest_gemm(c2v_engine* e, int32_t a_mn, int32_t b_mn, int32_t bn, int32_t M, int32_t N,
                      int32_t K, int32_t splits, const float* A, size_t lda, const float* B,
                      size_t ldb, float* C, size_t ldc, void* stream);

/* The same product as 3xTF32 (C2V_MATH_3XTF32): A / A_lo and B / B_lo hold the tf32 high parts and
 * residuals of the fp32 operands (same layout and pitch); c2v_selftest_split produces them
 * (hi = rna_tf32(x), lo = rna_tf32(x - hi); count % 4 == 0, 16-byte aligned device pointers). */
int c2v_selftest_gemm3(c2v_engine* e, int32_t a_mn, int32_t b_mn, int32_t bn, int32_t M, int32_t N,
                       int32_t K, int32_t splits, const float* A, const float* A_lo, size_t lda,
                       const float* B, const float* B_lo, size_t ldb, float* C, size_t ldc,
                       void* stream);
int c2v_selftest_split(c2v_engine* e, const float* x, float* hi, float* lo, size_t count, void* stream);

/* Introspection for tests and bench: number of kernels the engine has launched so far. */
int64_t c2v_launch_count(const c2v_engine* e);

/* Per-phase device timing (option "profile" = 1): CUDA events bracket every phase of a pass on
 * the launching stream.  c2v_phase_stats synchronises, folds the pending events into the
 * running totals and returns them (reset != 0 clears the totals afterwards). */
int c2v_phase_count(void);
const char* c2v_phase_name(int phase);
int c2v_phase_stats(c2v_engine* e, int phase, double* total_ms, int64_t* count, int reset);

#ifdef __cplusplus
}
#endif
#endif /* C2V_B200_H_ */
