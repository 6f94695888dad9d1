// C ABI of the path-attention engine (see include/c2v_b200.h) and the orchestration of one
// forward / train / predict pass.  Host code only launches kernels: all arithmetic of the path
// (tensorflow_model.py:197-309) runs in the kernels of sgemm.cuh / kernels.cuh / umma_gemm.cuh.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <utility>
#include <vector>

#include "../../include/c2v_b200.h"
#include "common.cuh"
#include "kernels.cuh"
#include "sgemm.cuh"
#include "umma_gemm.cuh"
#include "umma_gemm2.cuh"
#include "ctx_fused.cuh"
#include "similarity.cuh"

using namespace c2v;

namespace {

thread_local std::string g_create_error = "";

constexpr size_t kAlign = 256;
inline size_t align_up(size_t x, size_t a = kAlign) { return (x + a - 1) / a * a; }

constexpr int kSplitDv = 18;   // split-K slices for dv = P . Y      (K = |Y|)
constexpr int kSplitDw = 48;   // split-K slices for dW = X'^T . dU  (K = B*C)

// Carve-up of the caller-provided workspace (offsets in bytes).
struct Workspace {
  size_t H, Xg, dXg, alpha, v, dv, S, loss_b, lse, loss, part, da_part, lse_part, dl;
  size_t Xg_lo, H_lo, S_lo, tgt_hi, tgt_lo, W_hi, W_lo, v_hi, v_lo;     // 3xTF32 operand splits
  size_t true_logit, rscale, v_scaled, slab_flag;                  // exp_slab schedule: row factors, scaled code vectors, {range flag, fallback count}
  size_t st_src, st_pth, st_tgt, st_mask, st_target, st_topk_idx, st_topk_val, st_code, st_attn;
  size_t nx_src, nx_pth, nx_tgt;                                  // indices of the hinted NEXT batch (host entry point)
  size_t sb_src, sb_pth, sb_tgt, sb_mask, sb_target;              // second staging set (c2v_train_batch_async double buffer)
  size_t stamp_tok, stamp_path, last_tok, last_path, lr_tab;     // lazy Adam bookkeeping
  size_t stamp_tgt, last_tgt;                                    // ... of the target table (sampled softmax)
  size_t perm, bkt_count, bkt_cursor, bkt_starts;                            // locality-sorted peer gather / scatter (sharded tables)
  size_t total;
  size_t ldS;
};

bool dims_ok(const c2v_dims* d, std::string* why) {
  auto bad = [&](const char* m) { if (why) *why = m; return false; };
  if (!d) return bad("dims is NULL");
  if (d->token_vocab < 1 || d->path_vocab < 1 || d->target_vocab < 1) return bad("vocab sizes must be >= 1");
  if (d->embed_dim < 4 || d->embed_dim % 4) return bad("embed_dim must be a positive multiple of 4");
  if (d->code_dim < 4 || d->code_dim % 4 || d->code_dim > 1024) return bad("code_dim must be a multiple of 4 in [4, 1024]");
  if (d->max_contexts < 1) return bad("max_contexts must be >= 1");
  if (d->max_batch < 1) return bad("max_batch must be >= 1");
  if (d->top_k < 1 || d->top_k > 64) return bad("top_k must be in [1, 64]");
  if ((double)d->max_batch * d->max_contexts > 2.0e9) return bad("max_batch * max_contexts overflows int32");
  return true;
}

Workspace carve(const c2v_dims& d) {
  Workspace w{};
  const size_t N = (size_t)d.max_batch * d.max_contexts, D = d.code_dim, B = d.max_batch, X = 3 * (size_t)d.embed_dim;
  w.ldS = align_up((size_t)d.target_vocab, 64);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  w.H = take(N * D * 4);
  w.Xg = take(N * X * 4);      // gathered context matrix X' (tf32 path), kept for dW
  w.dXg = take(N * X * 4);     // dX' (tf32 path): its scatter-add overlaps the dW GEMM, which still reads X'
  w.alpha = take(N * 4);
  w.v = take(B * D * 4);
  w.dv = take(B * D * 4);
  w.S = take(B * w.ldS * 4);
  w.loss_b = take(B * 4);
  w.lse = take(B * 4);
  w.true_logit = take(B * 4);
  w.rscale = take(B * 4);
  w.v_scaled = take(B * D * 4);
  w.slab_flag = take(64);
  w.loss = take(64);
  size_t part = (size_t)kSplitDv * B * D;
  if ((size_t)kSplitDw * X * D > part) part = (size_t)kSplitDw * X * D;
  w.part = take(part * 4);
  w.da_part = take(B * D * 4);
  w.lse_part = take(B * 2 * (((size_t)d.target_vocab + 255) / 256) * 8);   // (max, sum exp) per (row, 128-col half tile)
  w.dl = take(B * (size_t)(kMaxSampled + 1) * 4);     // sampled softmax: dL/dlogits [B, 1+S]
  w.st_src = take(N * 4);
  w.st_pth = take(N * 4);
  w.st_tgt = take(N * 4);
  w.st_mask = take(N * 4);
  w.nx_src = take(N * 4);
  w.nx_pth = take(N * 4);
  w.nx_tgt = take(N * 4);
  w.st_target = take(B * 4);
  w.sb_src = take(N * 4);
  w.sb_pth = take(N * 4);
  w.sb_tgt = take(N * 4);
  w.sb_mask = take(N * 4);
  w.sb_target = take(B * 4);
  w.st_topk_idx = take(B * (size_t)d.top_k * 4);
  w.st_topk_val = take(B * (size_t)d.top_k * 4);
  w.st_code = take(B * D * 4);
  w.st_attn = take(N * 4);
  w.stamp_tok = take((size_t)d.token_vocab * 4);
  w.stamp_path = take((size_t)d.path_vocab * 4);
  w.last_tok = take((size_t)d.token_vocab * 4);
  w.last_path = take((size_t)d.path_vocab * 4);
  w.lr_tab = take((size_t)kLrRing * 4);
  w.perm = take(3 * N * 4);
  w.bkt_count = take((size_t)kMaxBuckets * 4);
  w.bkt_cursor = take((size_t)kMaxBuckets * 4);
  w.bkt_starts = take((size_t)(kMaxBuckets + 1) * 4);
  w.stamp_tgt = take((size_t)d.target_vocab * 4);
  w.last_tgt = take((size_t)d.target_vocab * 4);
  // 3xTF32 (C2V_MATH_3XTF32): low parts of the GEMM operands that are produced inside a step, and the
  // (hi, lo) split of the operands that must keep their fp32 originals
  w.Xg_lo = take(N * X * 4);
  w.H_lo = take(N * D * 4);
  w.S_lo = take(B * w.ldS * 4);
  w.tgt_hi = take((size_t)d.target_vocab * D * 4);
  w.tgt_lo = take((size_t)d.target_vocab * D * 4);
  w.W_hi = take(X * D * 4);
  w.W_lo = take(X * D * 4);
  w.v_hi = take(B * D * 4);
  w.v_lo = take(B * D * 4);
  w.total = off;
  return w;
}

}  // namespace

// Phases of a pass, for per-kernel timing (option "profile"): CUDA events bracket each phase on
// the launching stream; c2v_phase_stats() resolves them.
enum Phase { PH_CTX_FWD = 0, PH_ATTN_FWD, PH_LOGITS, PH_XENT, PH_DV, PH_DY, PH_ATTN_BWD, PH_DW, PH_DX_SCATTER,
             PH_ADAM, PH_TOPK, PH_SAMPLED, PH_GATHER, PH_DX_GEMM, PH_ADAM_CATCHUP, PH_SPLIT, PH_ADAM_SWEEP, PH_PEER_SORT, PH_INBOX_APPLY,
             PH_COUNT };
const char* const kPhaseNames[PH_COUNT] = {"ctx_fwd", "attn_fwd", "logits", "xent", "dv", "dY", "attn_bwd", "dW",
                                           "dx_scatter", "adam", "topk", "sampled_softmax", "gather", "dx_gemm",
                                           "adam_catchup", "split", "adam_sweep", "peer_sort", "inbox_apply"};
struct PhaseLog {
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> free_list;
  double total_ms = 0.0;
  int64_t count = 0;
};

struct c2v_engine {
  PhaseLog phase[PH_COUNT];
  int profile = 0;
  c2v_dims dims;
  int device;
  Workspace ws;
  char* wbase;
  size_t wbytes;
  c2v_tensors theta, grad, am, av;
  ShardedTable th_tok{}, th_path{}, gr_tok{}, gr_path{};   // how kernels reach the two embedding tables
  int table_world = 1;       // > 1: tables are row-sharded over peers (c2v_bind_table_shards)
  float grad_scale = 1.f;
  // lazy-but-exact dense Adam for the embedding tables (option "lazy_adam")
  int lazy = 0;
  int adam_rows_occ = 4;
  int sweep_period = 32;                // lazy Adam: every step brings a 1/R slice of each table up to date, so no row
                                        // is ever more than R steps behind (bounds the replay of rarely used rows and
                                        // the cost of c2v_sync_tables); 0 = off
  int64_t full_flush_t = 0;             // step count as of which every row was last known to be current
  int rest_shortcut = 1;                // option "adam_rest_shortcut": replay_row may stop dividing once theta rests
  bool tgt_lazy = false;                // the target table's rows are updated lazily too (sampled softmax steps)
  bool tgt_split_valid = false;         // 3xTF32: ws.tgt_hi / tgt_lo hold the split of the current target table
  bool lazy_grads_pending = false;  // a train step's embedding gradients are in the tables and c2v_adam_step has not followed
  int64_t adam_t_done = 0;   // Adam steps applied so far
  int32_t mark_epoch = 0;
  float hp_lr = 0.f, hp_b1 = 0.f, hp_b2 = 0.f, hp_eps = 0.f;
  bool hp_set = false;
  bool has_theta, has_grad, has_adam;
  bool emb_grads_clean;      // token/path gradient tables are known to be all-zero
  int math_mode;
  const int32_t* sorted_src = nullptr;   // ws.perm / ws.bkt_starts hold the bucket order of THIS batch (set by the forward pass)
  int sorted_rows = 0;
  InboxSet inbox{};          // push-based gradient exchange (c2v_bind_scatter_inbox); world == 0: not bound
  int sort_peer = 1;         // option "sort_peer_access": sharded tables are gathered / scattered in (owner, 2 MB page) order
  bool bkt_zeroed = false;   // the bucket counters have been cleared once (bucket_scan_kernel leaves them cleared)
  int recompute = 0;         // option "recompute_logits" (tensor-core modes, single-GPU step): the logits GEMM runs twice -- once for the
                             // log-sum-exp only, once writing dL/dlogits from its epilogue -- instead of writing logits and rewriting them.
                             // Measured: logits 0.42 + xent 0.36 -> 0.69 + 0.02 ms in tf32 (the LSE-only pass is epilogue-bound too), but
                             // 6.3 -> 7.1 ms in 3xTF32 (a third 3x GEMM and a second table split): off by default
  int exp_slab = 1;          // option "exp_slab" (tensor-core modes, single-GPU full-softmax step; default on): the logits epilogue writes
                             // U = exp(s - true logit) and the softmax's normalisation is deferred into per-row factors applied by the
                             // dv / dY GEMMs, so no pass re-reads the slab to turn logits into dL/dlogits (DESIGN.md section 4.9).  Rows
                             // outside the fp32 window make that step fall back, on the device, to the two-pass schedule.
  bool slab_flag_zeroed = false;
  bool slab_exp_live = false;         // c2v_target_forward left U (not logits) in the slab: c2v_target_backward finishes that schedule
  int gather_occ[2] = {0, 0};         // resident CTAs per SM of gather_ctx_kernel<false / true>, queried once
  int adam_epi_prefetch = 0; // option "adam_epilogue_prefetch" (measured slower, off): the dY epilogue's Adam update prefetches its (theta, m, v)
                             // lines into L2 one tile ahead
  const float* row_scale = nullptr;   // while the step's dv GEMM runs: the per-example factor its split-K reduction applies
  int fuse_sg = 0;           // option "fuse_softmax_grad": dv / dY compute dL/dlogits from the logits slab on the fly (tf32 mode).
                             // Correct, and it removes the 2.1 GB softmax-gradient pass (0.36 -> 0.02 ms), but with 32-bit operands the two
                             // GEMMs are already shared-memory-bandwidth bound and the in-place rewrite of the A stage costs more than
                             // it saves on B200 (dv 0.34 -> 0.63 ms, dY 0.69 -> 1.02 ms): off by default
  bool sg_live = false;      // ws.S holds LOGITS and sg describes how dv / dY turn them into dL/dlogits
  umma::SoftmaxGradArgs sg{};
  int fuse_gather = 0;       // option "fuse_gather": gather -> projection -> tanh as one kernel on the tf32 path (ctx_fused.cuh);
                             // bit-identical to the two-kernel path, but measured slower on B200 so far (0.31 vs 0.27 ms forward) -> off
  int cta_pair = 2;          // tcgen05 GEMMs as CTA pairs (cta_group::2, UMMA 256 x BN): 0 never, 1 always, 2 auto
  int num_sms;
  cudaEvent_t ev_tgt_ready = nullptr;   // recorded after dY (caller-owned)
  int dy_late = 1;                      // where dY = P^T.v runs: 0 after dv, 1 inside context_backward, 2 on side2 after dv
  const float* pending_dy_v = nullptr;  // code vectors of the deferred dY product
  int pending_dy_B = 0;
  cudaStream_t side = nullptr;          // engine-owned: the embedding scatter-add runs here, next to the dY / dW GEMMs
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t copy = nullptr;          // engine-owned: host -> device copies of c2v_train_batch_async
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_used[2] = {nullptr, nullptr};
  bool used_valid[2] = {false, false};
  uint64_t async_n = 0;
  cudaStream_t side2 = nullptr;         // engine-owned: the dY (+ target Adam) GEMM with dy_late == 2
  cudaEvent_t ev_fork2 = nullptr, ev_join2 = nullptr;
  bool dy_in_flight = false;            // a dY launched on side2 has not been joined yet
  // target-table Adam folded into the dY epilogue (c2v_arm_target_adam)
  bool tgt_armed = false;               // the next tcgen05 dY product applies the update instead of storing dY
  float tgt_lr = 0.f, tgt_b1 = 0.f, tgt_b2 = 0.f, tgt_eps = 0.f;
  int64_t tgt_t = 0;
  int64_t armed_t = 0;                  // step whose hyper-parameters c2v_arm_target_adam declared (0 = none)
  // next-batch hint (c2v_hint_next_batch): the deferred embedding-row updates of the NEXT batch's rows are
  // applied on the side stream during this step's backward, next to the dY / dW GEMMs
  const int32_t* hint_src = nullptr;
  const int32_t* hint_pth = nullptr;
  const int32_t* hint_tgt = nullptr;
  int hint_B = 0;
  int64_t early_t = 0;                  // step count the early catch-up already assumed applied (0 = none)
  int64_t early_count = 0;              // how many steps used the hint (option "early_catchup_count", read-only)
  int fuse_tgt = 0;                     // option "fuse_target_adam": c2v_train_batch_host arms itself
  int64_t tgt_fused_t = 0;              // step count whose target update has already been applied (0 = none)
  int deterministic;
  int64_t launches;
  std::string err;
};

namespace {

int fail(c2v_engine* e, int code, const std::string& msg) {
  if (e) e->err = msg; else g_create_error = msg;
  return code;
}

struct PhaseTimer {
  c2v_engine* e; int ph; cudaStream_t st; cudaEvent_t stop = nullptr;
  PhaseTimer(c2v_engine* e_, int ph_, cudaStream_t st_) : e(e_), ph(ph_), st(st_) {
    if (!e->profile) return;
    PhaseLog& L = e->phase[ph];
    std::pair<cudaEvent_t, cudaEvent_t> ev;
    if (!L.free_list.empty()) { ev = L.free_list.back(); L.free_list.pop_back(); }
    else { cudaEventCreate(&ev.first); cudaEventCreate(&ev.second); }
    cudaEventRecord(ev.first, st);
    stop = ev.second;
    L.pending.push_back(ev);
  }
  ~PhaseTimer() { if (stop) cudaEventRecord(stop, st); }
};

#define C2V_CUDA(e, expr)                                                                         \
  do {                                                                                            \
    cudaError_t _c = (expr);                                                                      \
    if (_c != cudaSuccess)                                                                        \
      return fail((e), C2V_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_c));         \
  } while (0)

// every kernel launch goes through this so the launch counter is truthful
#define C2V_LAUNCH(e, ...)                                                                        \
  do {                                                                                            \
    __VA_ARGS__;                                                                                  \
    cudaError_t _c = cudaGetLastError();                                                          \
    if (_c != cudaSuccess)                                                                        \
      return fail((e), C2V_ERR_CUDA, std::string("kernel launch failed: ") + cudaGetErrorString(_c)); \
    (e)->launches++;                                                                              \
  } while (0)

// adam_rows_kernel as one wave of num_sms * occupancy blocks (option "adam_rows_occupancy": 4 or 5)
#define C2V_ADAM_ROWS(e, MODE, stream, ...)                                                                    \
  do {                                                                                                         \
    if ((e)->adam_rows_occ == 5)                                                                               \
      C2V_LAUNCH(e, (adam_rows_kernel<MODE, 5><<<(e)->num_sms * 5, 256, 0, stream>>>(__VA_ARGS__)));           \
    else                                                                                                       \
      C2V_LAUNCH(e, (adam_rows_kernel<MODE, 4><<<(e)->num_sms * 4, 256, 0, stream>>>(__VA_ARGS__)));           \
  } while (0)

// the "theta rests" exit of the row replay (kernels.cuh, replay_row) is proven for these hyper-parameter ranges only
inline int rest_ok(const c2v_engine* e) {
  return (e->rest_shortcut && e->hp_b1 > 0.f && e->hp_b1 <= 0.95f && e->hp_b2 >= 0.99f && e->hp_b2 < 1.f && e->hp_eps > 0.f) ? 1 : 0;
}
inline bool is_tc(const c2v_engine* e) { return e->math_mode != C2V_MATH_FP32; }          // tcgen05 GEMMs
inline bool is_3x(const c2v_engine* e) { return e->math_mode == C2V_MATH_3XTF32; }        // ... as 3xTF32

// tcgen05 GEMM launchers: single-CTA (UMMA 128 x BN) or CTA-pair (UMMA 256 x BN).  Option "cta_pair":
// 0 = never, 1 = always, 2 = auto (default): pairs wherever they measured faster on B200 -- every GEMM
// except the two whose work items are few and long (dW: 3x2 tiles x split-K; dY: 1024-deep K), where the
// halved item count costs more than the halved B traffic saves (profiles/r01_bench_*).
#define C2V_PAIR(site_default) (e->cta_pair == 1 || (e->cta_pair == 2 && (site_default)))
#define C2V_UMMA_192(...) (C2V_PAIR(true) ? umma::launch2<192, 6>(__VA_ARGS__) : umma::launch<192, 4>(__VA_ARGS__))
#define C2V_UMMA_192_SINGLE(...) (C2V_PAIR(false) ? umma::launch2<192, 6>(__VA_ARGS__) : umma::launch<192, 4>(__VA_ARGS__))
#define C2V_UMMA_256(...) (C2V_PAIR(true) ? umma::launch2<256, 6>(__VA_ARGS__) : umma::launch<256, 4>(__VA_ARGS__))
// the same with the operand majors fixed at compile time (the fused-epilogue GEMMs each have one layout, so only
// that instantiation is built): AMN / BMN = operand is M- resp. N-contiguous in memory
#define C2V_UMMA_FIXED(BN, AMN, BMN, pair_default, EPI, ...)                                   \
  (C2V_PAIR(pair_default) ? umma::launch2_cfg<BN, 6, AMN, BMN, EPI>(__VA_ARGS__) : umma::launch_cfg<BN, 4, AMN, BMN, EPI>(__VA_ARGS__))

template <class T> T* wsp(c2v_engine* e, size_t off) { return reinterpret_cast<T*>(e->wbase + off); }

inline bool has_all(const c2v_tensors* t) { return t && t->tok && t->path && t->tgt && t->W && t->a; }

Dropout make_dropout(const c2v_dims& d, float keep, uint64_t seed, uint64_t step, const float* ext) {
  Dropout dp{};
  dp.ctx_dim = 3 * d.embed_dim;
  dp.enabled = (keep < 1.0f) ? 1 : 0;
  dp.ext = ext;
  dp.scale = 1.0f / keep;
  double thr = (double)keep * 4294967296.0;
  dp.thr = thr >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)thr;
  dp.key = make_uint2((uint32_t)(seed & 0xFFFFFFFFull), (uint32_t)(seed >> 32));
  dp.step = make_uint2((uint32_t)(step & 0xFFFFFFFFull), (uint32_t)(step >> 32));
  return dp;
}

int check_batch(c2v_engine* e, int32_t B) {
  if (!e) return C2V_ERR_INVALID;
  if (B < 1 || B > e->dims.max_batch) return fail(e, C2V_ERR_INVALID, "batch size out of range [1, max_batch]");
  if (!e->wbase) return fail(e, C2V_ERR_STATE, "workspace not bound (c2v_bind_workspace)");
  if (!e->has_theta) return fail(e, C2V_ERR_STATE, "parameters not bound (c2v_bind_params)");
  return C2V_OK;
}

// ---- attention kernels: dispatch on ceil(D / 128) ------------------------------------------------
int launch_attn_fwd(c2v_engine* e, cudaStream_t st, const float* H, const float* mask, int B, float* alpha, float* v) {
  const int C = e->dims.max_contexts, D = e->dims.code_dim;
  const size_t smem = ((size_t)((C + 3) & ~3) + 32 + kAttnWarps + (size_t)kAttnWarps * D) * sizeof(float);
  const float* a = e->theta.a;
  PhaseTimer pt(e, PH_ATTN_FWD, st);
#define C2V_AF(NV)                                                                                        \
  do {                                                                                                    \
    if (smem > 48 * 1024)                                                                                 \
      C2V_CUDA(e, cudaFuncSetAttribute(attn_fwd_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    C2V_LAUNCH(e, (attn_fwd_kernel<NV><<<B, kAttnThreads, smem, st>>>(H, a, mask, C, D, alpha, v)));      \
  } while (0)
  switch ((D + 127) / 128) {
    case 1: C2V_AF(1); break;
    case 2: C2V_AF(2); break;
    case 3: C2V_AF(3); break;
    case 4: C2V_AF(4); break;
    case 5: case 6: C2V_AF(6); break;
    default: C2V_AF(8); break;
  }
#undef C2V_AF
  return C2V_OK;
}

// v: the code vectors the forward pass produced for these examples (ws.v)
int launch_attn_bwd(c2v_engine* e, cudaStream_t st, float* H, const float* alpha, const float* dv, const float* v, int B,
                    float* da_part, float* H_lo) {
  const int C = e->dims.max_contexts, D = e->dims.code_dim;
  const size_t smem = (size_t)kAttnWarps * D * sizeof(float);
  const float* a = e->theta.a;
  PhaseTimer pt(e, PH_ATTN_BWD, st);
#define C2V_AB(NV)                                                                                        \
  do {                                                                                                    \
    if (H_lo) {                                                                                           \
      if (smem > 48 * 1024)                                                                               \
        C2V_CUDA(e, cudaFuncSetAttribute(attn_bwd_kernel<NV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      C2V_LAUNCH(e, (attn_bwd_kernel<NV, true><<<B, kAttnThreads, smem, st>>>(H, alpha, dv, v, a, C, D, da_part, H_lo))); \
    } else {                                                                                              \
      if (smem > 48 * 1024)                                                                               \
        C2V_CUDA(e, cudaFuncSetAttribute(attn_bwd_kernel<NV, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      C2V_LAUNCH(e, (attn_bwd_kernel<NV, false><<<B, kAttnThreads, smem, st>>>(H, alpha, dv, v, a, C, D, da_part, nullptr))); \
    }                                                                                                     \
  } while (0)
  switch ((D + 127) / 128) {
    case 1: C2V_AB(1); break;
    case 2: C2V_AB(2); break;
    case 3: C2V_AB(3); break;
    case 4: C2V_AB(4); break;
    case 5: case 6: C2V_AB(6); break;
    default: C2V_AB(8); break;
  }
#undef C2V_AB
  return C2V_OK;
}

// row_scale (optional): the n results are rows of length row_len; row i is multiplied by row_scale[i]
int launch_colsum(c2v_engine* e, cudaStream_t st, const float* in, size_t stride, int R, int n, float* out,
                  const float* row_scale = nullptr, int row_len = 0) {
  if (R <= 64 && n % 4 == 0 && stride % 4 == 0 && (!row_scale || row_len % 4 == 0)) {          // split-K slices: few rows, many columns
    size_t blocks = ((size_t)n / 4 + 255) / 256;
    if (blocks > (size_t)e->num_sms * 16) blocks = (size_t)e->num_sms * 16;
    C2V_LAUNCH(e, (slice_sum_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, stride, R, (size_t)n / 4, out, row_scale, row_scale ? row_len / 4 : 1)));
    return C2V_OK;
  }
  C2V_LAUNCH(e, (colsum_kernel<<<(n + 31) / 32, dim3(32, 32), 0, st>>>(in, stride, R, n, out)));
  if (row_scale) C2V_LAUNCH(e, (scale_rows_kernel<<<(unsigned)(((size_t)n + 255) / 256), 256, 0, st>>>(out, row_scale, out, row_len, (size_t)n)));
  return C2V_OK;
}

ContextSource make_source(c2v_engine* e, const int32_t* src, const int32_t* pth, const int32_t* tgt, int B) {
  ContextSource cs{};
  cs.src = src; cs.pth = pth; cs.tgt = tgt;
  cs.tok = e->th_tok; cs.path = e->th_path;
  cs.d = e->dims.embed_dim;
  cs.rows = B * e->dims.max_contexts;
  return cs;
}

// Lazy Adam: stamp the rows this batch references and replay their pending zero-gradient steps so the
// gather below reads exactly what a dense Adam would have left there.
int prepare_rows(c2v_engine* e, cudaStream_t st, const ContextSource& cs) {
  if (!e->lazy) return C2V_OK;
  PhaseTimer pt(e, PH_ADAM_CATCHUP, st);
  const c2v_dims& d = e->dims;
  int32_t* stamp_tok = wsp<int32_t>(e, e->ws.stamp_tok);
  int32_t* stamp_path = wsp<int32_t>(e, e->ws.stamp_path);
  e->mark_epoch++;
  C2V_LAUNCH(e, (mark_rows_kernel<<<(cs.rows + 255) / 256, 256, 0, st>>>(cs.src, cs.pth, cs.tgt, cs.rows, stamp_tok, stamp_path,
                                                                        e->mark_epoch)));
  if (e->adam_t_done > 0) {
    const float* lr_tab = wsp<float>(e, e->ws.lr_tab);
    C2V_ADAM_ROWS(e, ADAM_ROWS_CATCHUP, st,
                  e->theta.tok, e->grad.tok, e->am.tok, e->av.tok, d.token_vocab, d.embed_dim, stamp_tok, e->mark_epoch,
                      wsp<int32_t>(e, e->ws.last_tok), (int32_t)e->adam_t_done, lr_tab, e->hp_b1, e->hp_b2, e->hp_eps, rest_ok(e));
    C2V_ADAM_ROWS(e, ADAM_ROWS_CATCHUP, st,
                  e->theta.path, e->grad.path, e->am.path, e->av.path, d.path_vocab, d.embed_dim, stamp_path, e->mark_epoch,
                      wsp<int32_t>(e, e->ws.last_path), (int32_t)e->adam_t_done, lr_tab, e->hp_b1, e->hp_b2, e->hp_eps, rest_ok(e));
  }
  return C2V_OK;
}

// every row of one table that is behind step t: replay (one warp per row)
int launch_sweep(c2v_engine* e, cudaStream_t st, float* p, float* g, float* m, float* v, int rows, int dim, int32_t* last, int64_t t) {
  if (rows <= 0) return C2V_OK;
  int blocks = (rows + 7) / 8;
  if (blocks > e->num_sms * 4) blocks = e->num_sms * 4;
  C2V_LAUNCH(e, (adam_sweep_kernel<4><<<blocks, 256, 0, st>>>(p, g, m, v, rows, dim, last, (int32_t)t, wsp<float>(e, e->ws.lr_tab), e->hp_b1,
                                                             e->hp_b2, e->hp_eps, rest_ok(e))));
  return C2V_OK;
}

// Lazy Adam: bring every row of both embedding tables up to date (export, checkpoint, mode switches).
int flush_rows(c2v_engine* e, cudaStream_t st) {
  if (!e->lazy || e->adam_t_done == 0) return C2V_OK;
  const c2v_dims& d = e->dims;
  const float* lr_tab = wsp<float>(e, e->ws.lr_tab);
  { int rcw = launch_sweep(e, st, e->theta.tok, e->grad.tok, e->am.tok, e->av.tok, d.token_vocab, d.embed_dim, wsp<int32_t>(e, e->ws.last_tok), e->adam_t_done);
    if (rcw) return rcw; }
  { int rcw = launch_sweep(e, st, e->theta.path, e->grad.path, e->am.path, e->av.path, d.path_vocab, d.embed_dim, wsp<int32_t>(e, e->ws.last_path), e->adam_t_done);
    if (rcw) return rcw; }
  if (e->tgt_lazy)
    { int rcw = launch_sweep(e, st, e->theta.tgt, e->grad.tgt, e->am.tgt, e->av.tgt, d.target_vocab, d.code_dim, wsp<int32_t>(e, e->ws.last_tgt), e->adam_t_done);
    if (rcw) return rcw; }
  e->full_flush_t = e->adam_t_done;
  return C2V_OK;
}

// The target table leaves the lazily updated set (a full-softmax step, a full-vocabulary read): bring its rows
// up to date first.  Its gradient rows are zero afterwards (cleared as they are applied).
int end_target_lazy(c2v_engine* e, cudaStream_t st) {
  if (!e->tgt_lazy) return C2V_OK;
  if (e->adam_t_done > 0) {
    const c2v_dims& d = e->dims;
    { int rcw = launch_sweep(e, st, e->theta.tgt, e->grad.tgt, e->am.tgt, e->av.tgt, d.target_vocab, d.code_dim, wsp<int32_t>(e, e->ws.last_tgt), e->adam_t_done);
    if (rcw) return rcw; }
  }
  e->tgt_lazy = false;
  return C2V_OK;
}

// Lazy Adam sweep: rows [rows*ph/R, rows*(ph+1)/R) of every lazily updated table are brought up to date each
// step (ph = t mod R), so a row is never more than R steps behind whatever the data looks like: the replay
// of a rarely referenced row costs at most R iterations, and c2v_sync_tables at most R per row.
int sweep_rows(c2v_engine* e, cudaStream_t st, int64_t t) {
  const int R = e->sweep_period;
  if (!e->lazy || R <= 0) return C2V_OK;
  if (R == 1) return flush_rows(e, st);
  PhaseTimer pt(e, PH_ADAM_SWEEP, st);
  const c2v_dims& d = e->dims;
  const float* lr_tab = wsp<float>(e, e->ws.lr_tab);
  const int64_t ph = t % R;
  auto slice = [&](float* p, float* g, float* m, float* v, int rows, int dim, int32_t* last) -> int {
    const int64_t lo = (int64_t)rows * ph / R, hi = (int64_t)rows * (ph + 1) / R;
    if (hi <= lo) return C2V_OK;
    const size_t o = (size_t)lo * dim;
    return launch_sweep(e, st, p + o, g + o, m + o, v + o, (int)(hi - lo), dim, last + lo, t);
  };
  int rc;
  if ((rc = slice(e->theta.tok, e->grad.tok, e->am.tok, e->av.tok, d.token_vocab, d.embed_dim, wsp<int32_t>(e, e->ws.last_tok)))) return rc;
  if ((rc = slice(e->theta.path, e->grad.path, e->am.path, e->av.path, d.path_vocab, d.embed_dim, wsp<int32_t>(e, e->ws.last_path)))) return rc;
  if (e->tgt_lazy &&
      (rc = slice(e->theta.tgt, e->grad.tgt, e->am.tgt, e->av.tgt, d.target_vocab, d.code_dim, wsp<int32_t>(e, e->ws.last_tgt)))) return rc;
  if (ph == R - 1) e->full_flush_t = t - R + 1;      // every row has been visited at or after step t - R + 1
  return C2V_OK;
}

// Lazy Adam + next-batch hint: once this step's scatter-add is queued on the side stream, the rows the NEXT
// batch references can already be brought up to date through THIS step (its hyper-parameters are known
// from c2v_arm_target_adam): their deferred updates then run next to the dY / dW GEMMs instead of at the
// head of the next step.  Same kernels, same arithmetic, only earlier; anything not covered here is
// handled by the next step's prepare_rows as usual.
int early_catchup(c2v_engine* e, cudaStream_t side) {
  const int32_t *hs = e->hint_src, *hp = e->hint_pth, *ht = e->hint_tgt;
  const int hB = e->hint_B;
  e->hint_src = e->hint_pth = e->hint_tgt = nullptr;          // one-shot
  e->hint_B = 0;
  if (!hs || !e->lazy || e->table_world > 1) return C2V_OK;
  const int64_t t = e->armed_t;
  if (t != e->adam_t_done + 1) return C2V_OK;
  // pending steps were recorded under e->hp_*: only valid to run ahead if this step keeps them
  if (!e->hp_set || e->tgt_lr != e->hp_lr || e->tgt_b1 != e->hp_b1 || e->tgt_b2 != e->hp_b2 || e->tgt_eps != e->hp_eps)
    return C2V_OK;
  const c2v_dims& d = e->dims;
  const double lr_t = (double)e->tgt_lr * sqrt(1.0 - pow((double)e->tgt_b2, (double)t)) / (1.0 - pow((double)e->tgt_b1, (double)t));
  float* lr_tab = wsp<float>(e, e->ws.lr_tab);
  int32_t* stamp_tok = wsp<int32_t>(e, e->ws.stamp_tok);
  int32_t* stamp_path = wsp<int32_t>(e, e->ws.stamp_path);
  PhaseTimer pt(e, PH_ADAM_CATCHUP, side);
  C2V_LAUNCH(e, (set_float_kernel<<<1, 1, 0, side>>>(lr_tab + (t & kLrRingMask), (float)lr_t)));
  e->mark_epoch++;
  const int rows = hB * d.max_contexts;
  C2V_LAUNCH(e, (mark_rows_kernel<<<(rows + 255) / 256, 256, 0, side>>>(hs, hp, ht, rows, stamp_tok, stamp_path, e->mark_epoch)));
  C2V_ADAM_ROWS(e, ADAM_ROWS_CATCHUP, side,
                  e->theta.tok, e->grad.tok, e->am.tok, e->av.tok, d.token_vocab, d.embed_dim, stamp_tok, e->mark_epoch,
                    wsp<int32_t>(e, e->ws.last_tok), (int32_t)t, lr_tab, e->hp_b1, e->hp_b2, e->hp_eps, rest_ok(e));
  C2V_ADAM_ROWS(e, ADAM_ROWS_CATCHUP, side,
                  e->theta.path, e->grad.path, e->am.path, e->av.path, d.path_vocab, d.embed_dim, stamp_path, e->mark_epoch,
                    wsp<int32_t>(e, e->ws.last_path), (int32_t)t, lr_tab, e->hp_b1, e->hp_b2, e->hp_eps, rest_ok(e));
  e->early_t = t;
  e->early_count++;
  return C2V_OK;
}

// 3xTF32: (hi, lo) tf32 split of a whole fp32 buffer into two workspace regions.
int split_small(c2v_engine* e, cudaStream_t st, const float* x, size_t n, size_t off_hi, size_t off_lo) {
  PhaseTimer pt(e, PH_SPLIT, st);
  const size_t n4 = n / 4;                 // every split buffer here is a multiple of 4 floats (dims_ok)
  size_t blocks = (n4 + 255) / 256;
  if (blocks > (size_t)e->num_sms * 16) blocks = (size_t)e->num_sms * 16;
  if (blocks < 1) blocks = 1;
  C2V_LAUNCH(e, (split_tf32_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, wsp<float>(e, off_hi), wsp<float>(e, off_lo), n4)));
  return C2V_OK;
}

// Sharded tables: bucket the batch's 3 B C context entries by (owner rank, 2 MB page of the owner's shard) into ws.perm.
// Returns false when the plan does not apply (tables not sharded, option off, too many buckets).
bool plan_buckets(c2v_engine* e, BucketPlan* bp, bool force = false) {
  if (e->table_world <= 1) return false;
  const c2v_dims& d = e->dims;
  // sort_peer_access: 0 never, 1 (default) when the tables are large enough for random peer accesses to thrash the TLB
  // (measured: a loss at 1.1 GB of tables, 1.8-3.4x faster at 5 GB), 2 always; the inbox exchange always needs the order
  const double table_bytes = ((double)d.token_vocab + d.path_vocab) * d.embed_dim * 4.0;
  if (!force && (e->sort_peer == 0 || (e->sort_peer == 1 && table_bytes < 2.0e9))) return false;
  const int W = e->table_world;
  int rows_per_page = (int)((2u << 20) / ((size_t)d.embed_dim * 4));
  int ps = 0;
  while ((2 << ps) <= rows_per_page) ++ps;
  bp->shift = e->th_tok.shift; bp->mask = e->th_tok.mask; bp->page_shift = ps;
  const int rows_tok = (d.token_vocab + W - 1) / W, rows_path = (d.path_vocab + W - 1) / W;
  bp->pages_tok = (rows_tok >> ps) + 1;
  bp->pages_path = (rows_path >> ps) + 1;
  bp->n_buckets = W * (bp->pages_tok + bp->pages_path);
  return bp->n_buckets <= kMaxBuckets;
}
int sort_entries(c2v_engine* e, cudaStream_t st, const ContextSource& cs, const BucketPlan& bp) {
  PhaseTimer pt(e, PH_PEER_SORT, st);
  int32_t* counts = wsp<int32_t>(e, e->ws.bkt_count);
  int32_t* cursor = wsp<int32_t>(e, e->ws.bkt_cursor);
  if (!e->bkt_zeroed) {
    C2V_CUDA(e, cudaMemsetAsync(counts, 0, (size_t)kMaxBuckets * 4, st));
    e->bkt_zeroed = true;
  }
  const int total = 3 * cs.rows;
  int blocks = (total + 255) / 256;
  if (blocks > e->num_sms * 8) blocks = e->num_sms * 8;
  C2V_LAUNCH(e, (bucket_count_kernel<<<blocks, 256, (size_t)bp.n_buckets * 4, st>>>(cs, bp, counts)));
  C2V_LAUNCH(e, (bucket_scan_kernel<<<1, 1024, 0, st>>>(counts, cursor, wsp<int32_t>(e, e->ws.bkt_starts), bp.n_buckets)));
  C2V_LAUNCH(e, (bucket_fill_kernel<<<blocks, 256, 0, st>>>(cs, bp, cursor, wsp<int32_t>(e, e->ws.perm))));
  return C2V_OK;
}

// Grid of the gather: one wave of resident CTAs (8 warps each; a warp strides over the rows), never more CTAs than rows / 8.
unsigned gather_blocks(c2v_engine* e, int rows, bool split) {
  int& occ = e->gather_occ[split ? 1 : 0];
  if (occ == 0) {
    int n = 0;
    cudaError_t rc = split ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, gather_ctx_kernel<true>, 256, 0)
                           : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, gather_ctx_kernel<false>, 256, 0);
    occ = (rc == cudaSuccess && n > 0) ? n : 4;
  }
  const long want = (rows + 7) / 8, wave = (long)e->num_sms * occ;
  return (unsigned)(want < wave ? want : wave);
}

// H = tanh(X' . W)   (tensorflow_model.py:238-252)
int run_ctx_fwd(c2v_engine* e, cudaStream_t st, const ContextSource& cs, const Dropout& dp, float* H, bool keep_x) {
  const int D = e->dims.code_dim, K = 3 * e->dims.embed_dim;
  { int rc0 = prepare_rows(e, st, cs); if (rc0) return rc0; }
  if (is_tc(e) && !is_3x(e) && e->fuse_gather && e->dims.embed_dim % 32 == 0 && cs.rows % 4 == 0 &&
      (((uintptr_t)cs.src | (uintptr_t)cs.pth | (uintptr_t)cs.tgt) % 16) == 0) {
    // gather -> dropout -> projection -> tanh in one kernel (ctx_fused.cuh); X' is written out only when a backward
    // pass will need it (dW = X'^T . dU)
    PhaseTimer pt(e, PH_CTX_FWD, st);
    umma::EpiTanhStore ep{H, (size_t)D};
    C2V_LAUNCH(e, C2V_CUDA(e, (umma::launch_ctx_fused<192, 4>(st, cs.rows, D, e->theta.W, (size_t)D, cs, dp,
                                                              keep_x ? wsp<float>(e, e->ws.Xg) : nullptr, ep, e->num_sms))));
    return C2V_OK;
  }
  if (is_tc(e)) {
    float* Xg = wsp<float>(e, e->ws.Xg);
    const bool x3 = is_3x(e);
    {
      PhaseTimer pt(e, PH_GATHER, st);
      BucketPlan bp;
      e->sorted_src = nullptr;
      if (e->inbox.world > 1 && plan_buckets(e, &bp, true) && !plan_buckets(e, &bp)) {
        // the backward pass will push gradient rows owner by owner: bucket the batch now, while the SMs are free (in
        // the backward pass the same three small kernels would queue behind the persistent dW GEMM)
        int rcs = sort_entries(e, st, cs, bp);
        if (rcs) return rcs;
        e->sorted_src = cs.src; e->sorted_rows = cs.rows;
      }
      if (plan_buckets(e, &bp)) {           // peer shards: walk the entries page by page
        int rcs = sort_entries(e, st, cs, bp);
        if (rcs) return rcs;
        e->sorted_src = cs.src; e->sorted_rows = cs.rows;
        const int32_t* perm = wsp<int32_t>(e, e->ws.perm);
        if (x3) C2V_LAUNCH(e, (gather_sorted_kernel<true><<<(3 * cs.rows + 7) / 8, 256, 0, st>>>(cs, dp, perm, Xg, wsp<float>(e, e->ws.Xg_lo))));
        else C2V_LAUNCH(e, (gather_sorted_kernel<false><<<(3 * cs.rows + 7) / 8, 256, 0, st>>>(cs, dp, perm, Xg, nullptr)));
      } else if (x3) C2V_LAUNCH(e, (gather_ctx_kernel<true><<<gather_blocks(e, cs.rows, true), 256, 0, st>>>(cs, dp, Xg, wsp<float>(e, e->ws.Xg_lo))));
      else C2V_LAUNCH(e, (gather_ctx_kernel<false><<<gather_blocks(e, cs.rows, false), 256, 0, st>>>(cs, dp, Xg, nullptr)));
    }
    if (x3) { int rcs = split_small(e, st, e->theta.W, (size_t)K * D, e->ws.W_hi, e->ws.W_lo); if (rcs) return rcs; }
    PhaseTimer pt(e, PH_CTX_FWD, st);
    umma::Operand opA{Xg, (size_t)K, false, x3 ? wsp<float>(e, e->ws.Xg_lo) : nullptr};
    umma::Operand opB{x3 ? wsp<float>(e, e->ws.W_hi) : e->theta.W, (size_t)D, true, x3 ? wsp<float>(e, e->ws.W_lo) : nullptr};
    if (x3) {
      umma::EpiTanhStorePrecise ep{H, (size_t)D};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(192, false, true, true, umma::EpiTanhStorePrecise, st, cs.rows, D, K, 1, opA, opB, ep, e->num_sms))));
    } else {
      umma::EpiTanhStore ep{H, (size_t)D};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(192, false, true, true, umma::EpiTanhStore, st, cs.rows, D, K, 1, opA, opB, ep, e->num_sms))));
    }
    return C2V_OK;
  }
  PhaseTimer pt(e, PH_CTX_FWD, st);
  simt::GatherRowsK al{cs, dp};
  simt::ColsX bl{e->theta.W, (size_t)D};
  simt::TanhStore ep{H, (size_t)D};
  C2V_LAUNCH(e, C2V_CUDA(e, simt::launch(st, cs.rows, D, K, 1, al, bl, ep)));
  return C2V_OK;
}

// S[B, Y] = v . Ytab^T   (tensorflow_model.py:226,297)
// with_lse (tf32 path only): also emit per-(row, 256-column tile) log-sum-exp partials into ws.lse_part.
// grad != nullptr: the pass writes dL/dlogits (EpiSoftmaxGrad); lse_only: nothing but the log-sum-exp partials.
struct LogitsGrad { const float* lse; const int32_t* target; int row0; float inv_batch; };
// exp_offset != nullptr: the pass writes U = exp(logit - exp_offset[row]) and (max U, sum U) partials (EpiExpSum).
// gate != nullptr (with_lse): the launch is the exp_slab schedule's fallback, a no-op while *gate == 0; it reuses the operand
// splits the step's first pass made.
int run_logits(c2v_engine* e, cudaStream_t st, const float* v, int B, float* S, bool with_lse = false, bool lse_only = false,
               const LogitsGrad* grad = nullptr, const float* exp_offset = nullptr, const int* gate = nullptr) {
  const int D = e->dims.code_dim, Y = e->dims.target_vocab;
  { int rcl = end_target_lazy(e, st); if (rcl) return rcl; }      // a pass over the whole table needs every row current
  if (is_tc(e) && (reinterpret_cast<uintptr_t>(v) % 16 == 0)) {
    const bool x3 = is_3x(e);
    umma::Operand opA{v, (size_t)D, false};
    umma::Operand opB{e->theta.tgt, (size_t)D, false};
    if (x3) {      // fp32-faithful: both operands as tf32 (hi, lo) pairs; the table is re-split on every pass over it
      int rcs;
      if (!gate) {
        if ((rcs = split_small(e, st, v, (size_t)B * D, e->ws.v_hi, e->ws.v_lo))) return rcs;
        if ((rcs = split_small(e, st, e->theta.tgt, (size_t)Y * D, e->ws.tgt_hi, e->ws.tgt_lo))) return rcs;
      }
      e->tgt_split_valid = true;
      opA.base = wsp<float>(e, e->ws.v_hi); opA.lo = wsp<float>(e, e->ws.v_lo);
      opB.base = wsp<float>(e, e->ws.tgt_hi); opB.lo = wsp<float>(e, e->ws.tgt_lo);
    }
    PhaseTimer pt(e, PH_LOGITS, st);
    const int slots = 2 * ((Y + 255) / 256);
    if (exp_offset && x3) {
      umma::EpiExpSumT<true, true> ep{S, wsp<float>(e, e->ws.S_lo), e->ws.ldS, exp_offset, wsp<float2>(e, e->ws.lse_part), slots};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (exp_offset) {
      umma::EpiExpSumT<false, false> ep{S, nullptr, e->ws.ldS, exp_offset, wsp<float2>(e, e->ws.lse_part), slots};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (gate && x3) {
      umma::EpiStoreLseGatedT<true> ep{{S, e->ws.ldS, wsp<float2>(e, e->ws.lse_part), slots}, gate};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (gate) {
      umma::EpiStoreLseGatedT<false> ep{{S, e->ws.ldS, wsp<float2>(e, e->ws.lse_part), slots}, gate};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (grad && x3) {
      umma::EpiSoftmaxGradT<true, true> ep{S, wsp<float>(e, e->ws.S_lo), e->ws.ldS, grad->lse, grad->target, grad->row0, grad->inv_batch, B};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (grad) {
      umma::EpiSoftmaxGradT<false, false> ep{S, nullptr, e->ws.ldS, grad->lse, grad->target, grad->row0, grad->inv_batch, B};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (lse_only && x3) {
      umma::EpiLseOnlyT<true> ep{{S, e->ws.ldS, wsp<float2>(e, e->ws.lse_part), slots}};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (lse_only) {
      umma::EpiLseOnlyT<false> ep{{S, e->ws.ldS, wsp<float2>(e, e->ws.lse_part), slots}};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, decltype(ep), st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (with_lse && x3) {
      umma::EpiStoreLsePrecise ep{S, e->ws.ldS, wsp<float2>(e, e->ws.lse_part), 2 * ((Y + 255) / 256)};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, umma::EpiStoreLsePrecise, st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else if (with_lse) {
      umma::EpiStoreLse ep{S, e->ws.ldS, wsp<float2>(e, e->ws.lse_part), 2 * ((Y + 255) / 256)};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(256, false, false, true, umma::EpiStoreLse, st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    } else {
      umma::EpiStore ep{S, e->ws.ldS, 0};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_256(st, B, Y, D, 1, opA, opB, ep, e->num_sms))));
    }
    return C2V_OK;
  }
  PhaseTimer pt(e, PH_LOGITS, st);
  simt::RowsK al{v, (size_t)D};
  simt::RowsK bl{e->theta.tgt, (size_t)D};
  simt::StoreC ep{S, e->ws.ldS, 0};
  C2V_LAUNCH(e, C2V_CUDA(e, simt::launch(st, B, Y, D, 1, al, bl, ep)));
  return C2V_OK;
}

int forward_impl(c2v_engine* e, cudaStream_t st, const int32_t* src, const int32_t* pth, const int32_t* tgt,
                 const float* mask, int B, const Dropout& dp, float* code_vec, float* attn, bool keep_x = false) {
  ContextSource cs = make_source(e, src, pth, tgt, B);
  float* H = wsp<float>(e, e->ws.H);
  int rc = run_ctx_fwd(e, st, cs, dp, H, keep_x);
  if (rc) return rc;
  if ((rc = launch_attn_fwd(e, st, H, mask, B, attn, code_vec))) return rc;
  if (keep_x && code_vec != wsp<float>(e, e->ws.v))      // a backward pass follows (phase-split API): it needs the code vectors
    C2V_CUDA(e, cudaMemcpyAsync(wsp<float>(e, e->ws.v), code_vec, (size_t)B * e->dims.code_dim * 4, cudaMemcpyDeviceToDevice, st));
  return C2V_OK;
}

int topk_impl(c2v_engine* e, cudaStream_t st, const float* code_vec, int B, int32_t* idx, float* val, int normalize) {
  if (normalize < 0 || normalize > 2) return fail(e, C2V_ERR_INVALID, "normalize must be 0 (logits), 1 (softmax over k) or 2 (full softmax)");
  float* S = wsp<float>(e, e->ws.S);
  int rc = run_logits(e, st, code_vec, B, S);
  if (rc) return rc;
  const int Y = e->dims.target_vocab;
  const int k = e->dims.top_k < Y ? e->dims.top_k : Y;
  PhaseTimer pt(e, PH_TOPK, st);
  if (k <= 16)
    C2V_LAUNCH(e, (topk_kernel<16><<<B, kTopkThreads, 0, st>>>(S, e->ws.ldS, Y, k, normalize, idx, val)));
  else
    C2V_LAUNCH(e, (topk_iter_kernel<<<B, kTopkThreads, 0, st>>>(S, e->ws.ldS, Y, k, normalize, idx, val)));
  if (normalize == 2) C2V_LAUNCH(e, (topk_full_softmax_kernel<<<B, 256, 0, st>>>(S, e->ws.ldS, Y, k, val)));
  return C2V_OK;
}

// Backward of everything below the code vector, given dv: gradients of a, W and the two
// embedding tables (SURVEY A.2).
int run_dy(c2v_engine* e, cudaStream_t st, const float* v, int B);

int context_backward(c2v_engine* e, cudaStream_t st, const ContextSource& cs, const float* mask, int B,
                     const Dropout& dp, const float* dv) {
  const int D = e->dims.code_dim, d = e->dims.embed_dim, K3 = 3 * d, N = cs.rows;
  float* H = wsp<float>(e, e->ws.H);
  float* alpha = wsp<float>(e, e->ws.alpha);
  float* da_part = wsp<float>(e, e->ws.da_part);
  float* part = wsp<float>(e, e->ws.part);
  int rc;
  if (e->pending_dy_v && !is_tc(e)) {   // fp32 path: nothing to overlap with, run it first
    const float* pv = e->pending_dy_v;
    e->pending_dy_v = nullptr;
    if ((rc = run_dy(e, st, pv, e->pending_dy_B))) return rc;
  }
  const bool x3 = is_tc(e) && is_3x(e);
  float* H_lo = x3 ? wsp<float>(e, e->ws.H_lo) : nullptr;
  rc = launch_attn_bwd(e, st, H, alpha, dv, wsp<float>(e, e->ws.v), B, da_part, H_lo);    // H now holds dU (3xTF32: its high parts, H_lo the rest)
  if (rc) return rc;
  rc = launch_colsum(e, st, da_part, (size_t)D, B, D, e->grad.a);
  if (rc) return rc;
  if (is_tc(e)) {
    float* Xg = wsp<float>(e, e->ws.Xg);
    float* dXg = wsp<float>(e, e->ws.dXg);
    {  // dX' = dU . W^T
      PhaseTimer pt(e, PH_DX_GEMM, st);
      // 3xTF32: W's split was made by this step's forward pass (run_ctx_fwd) and W has not changed since
      umma::Operand opA{H, (size_t)D, false, H_lo};
      umma::Operand opB{x3 ? wsp<float>(e, e->ws.W_hi) : e->theta.W, (size_t)D, false, x3 ? wsp<float>(e, e->ws.W_lo) : nullptr};
      umma::EpiStore ep{dXg, (size_t)K3, 0};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_192(st, N, K3, D, 1, opA, opB, ep, e->num_sms))));
    }
    if (e->lazy) {
      if (e->lazy_grads_pending)
        return fail(e, C2V_ERR_STATE, "lazy_adam: every train step must be followed by c2v_adam_step before the next one");
      e->lazy_grads_pending = true;
    } else if (!e->emb_grads_clean && e->table_world == 1) {
      C2V_CUDA(e, cudaMemsetAsync(e->grad.tok, 0, (size_t)e->dims.token_vocab * d * 4, st));
      C2V_CUDA(e, cudaMemsetAsync(e->grad.path, 0, (size_t)e->dims.path_vocab * d * 4, st));
    }
    // fork: the scatter-add of dX' rows (memory / NVLink bound, no shared memory) runs on the engine's
    // side stream while the dW GEMM (tensor bound) runs on the caller's stream; join before returning.
    C2V_CUDA(e, cudaEventRecord(e->ev_fork, st));
    C2V_CUDA(e, cudaStreamWaitEvent(e->side, e->ev_fork, 0));
    {
      PhaseTimer pt(e, PH_DX_SCATTER, e->side);
      BucketPlan bp;
      if (e->inbox.world > 1 && plan_buckets(e, &bp, true)) {
        // push: every owner's rows go densely into this rank's region of the owner's inbox (plain coalesced stores over
        // NVLink); the owners fold them in with local atomics after the caller's barrier (c2v_apply_scatter_inbox)
        if (e->sorted_src != cs.src || e->sorted_rows != cs.rows) {     // not bucketed by this step's forward pass
          if ((rc = sort_entries(e, e->side, cs, bp))) return rc;
        }
        e->sorted_src = nullptr;
        const int32_t* starts = wsp<int32_t>(e, e->ws.bkt_starts);
        C2V_LAUNCH(e, (inbox_counts_kernel<<<1, 32, 0, e->side>>>(e->inbox, bp, starts)));
        C2V_LAUNCH(e, (scatter_inbox_kernel<<<(3 * N + 7) / 8, 256, 0, e->side>>>(cs, dp, mask, wsp<int32_t>(e, e->ws.perm), starts, bp, dXg,
                                                                              e->inbox, e->grad_scale)));
      } else if (plan_buckets(e, &bp)) {    // peer shards: the red.adds walk the owners' pages in order
        if ((rc = sort_entries(e, e->side, cs, bp))) return rc;
        C2V_LAUNCH(e, (scatter_sorted_kernel<<<(3 * N + 7) / 8, 256, 0, e->side>>>(cs, dp, mask, wsp<int32_t>(e, e->ws.perm), dXg, e->gr_tok,
                                                                               e->gr_path, e->grad_scale)));
      } else {
        C2V_LAUNCH(e, (scatter_dx_kernel<<<(N + 7) / 8, 256, 0, e->side>>>(cs, dp, mask, dXg, e->gr_tok, e->gr_path, e->grad_scale)));
      }
    }
    if ((rc = early_catchup(e, e->side))) return rc;
    C2V_CUDA(e, cudaEventRecord(e->ev_join, e->side));
    if (e->pending_dy_v) {   // deferred dYtab = P^T . v, concurrent with the scatter-add
      const float* pv = e->pending_dy_v;
      e->pending_dy_v = nullptr;
      if ((rc = run_dy(e, st, pv, e->pending_dy_B))) return rc;
    }
    {  // dW = X'^T . dU on the gathered X' kept from the forward pass
      PhaseTimer pt(e, PH_DW, st);
      umma::Operand opA{Xg, (size_t)K3, true, x3 ? wsp<float>(e, e->ws.Xg_lo) : nullptr};
      umma::Operand opB{H, (size_t)D, true, H_lo};
      const int ks = umma::effective_splits(N, kSplitDw);
      umma::EpiStore ep{part, (size_t)D, (size_t)K3 * D};
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_192_SINGLE(st, K3, D, N, kSplitDw, opA, opB, ep, e->num_sms))));
      rc = launch_colsum(e, st, part, (size_t)K3 * D, ks, K3 * D, e->grad.W);
      if (rc) return rc;
    }
    C2V_CUDA(e, cudaStreamWaitEvent(st, e->ev_join, 0));
    if (e->dy_in_flight) {
      C2V_CUDA(e, cudaStreamWaitEvent(st, e->ev_join2, 0));
      e->dy_in_flight = false;
    }
    e->emb_grads_clean = false;
    return C2V_OK;
  }
  {  // dW = X'^T . dU   (split-K over the B*C contexts, fixed-order reduction)
    PhaseTimer pt(e, PH_DW, st);
    simt::GatherColsX al{cs, dp};
    simt::ColsX bl{H, (size_t)D};
    const int ks = simt::effective_ksplit(N, kSplitDw);
    simt::StoreC ep{part, (size_t)D, (size_t)K3 * D};
    C2V_LAUNCH(e, C2V_CUDA(e, simt::launch(st, K3, D, N, kSplitDw, al, bl, ep)));
    rc = launch_colsum(e, st, part, (size_t)K3 * D, ks, K3 * D, e->grad.W);
    if (rc) return rc;
  }
  {  // dX' = dU . W^T -> dropout backward -> scatter-add into the embedding gradient tables
    if (e->lazy) {
      if (e->lazy_grads_pending)
        return fail(e, C2V_ERR_STATE, "lazy_adam: every train step must be followed by c2v_adam_step before the next one");
      e->lazy_grads_pending = true;
    } else if (!e->emb_grads_clean && e->table_world == 1) {
      C2V_CUDA(e, cudaMemsetAsync(e->grad.tok, 0, (size_t)e->dims.token_vocab * d * 4, st));
      C2V_CUDA(e, cudaMemsetAsync(e->grad.path, 0, (size_t)e->dims.path_vocab * d * 4, st));
    }
    PhaseTimer pt(e, PH_DX_SCATTER, st);
    simt::RowsK al{H, (size_t)D};
    simt::RowsK bl{e->theta.W, (size_t)D};
    simt::ScatterDx ep{cs, e->gr_tok, e->gr_path, mask, dp, e->grad_scale};
    C2V_LAUNCH(e, C2V_CUDA(e, simt::launch(st, N, K3, D, 1, al, bl, ep)));
    e->emb_grads_clean = false;
  }
  return C2V_OK;
}

// Given P = dL/dlogits in the S slab:  dv = P . Ytab  (split-K over |Y|, fixed-order reduction).
int run_dv(c2v_engine* e, cudaStream_t st, int B, float* dv) {
  const int D = e->dims.code_dim, Y = e->dims.target_vocab;
  float* S = wsp<float>(e, e->ws.S);
  float* part = wsp<float>(e, e->ws.part);
  PhaseTimer pt(e, PH_DV, st);
  if (is_tc(e)) {
    umma::Operand opA{S, e->ws.ldS, false};
    umma::Operand opB{e->theta.tgt, (size_t)D, true};
    if (is_3x(e)) {      // P was written as its split by softmax_grad_kernel; the table's split dates from the logits pass
      if (!e->tgt_split_valid) {
        int rcs = split_small(e, st, e->theta.tgt, (size_t)Y * D, e->ws.tgt_hi, e->ws.tgt_lo);
        if (rcs) return rcs;
        e->tgt_split_valid = true;
      }
      opA.lo = wsp<float>(e, e->ws.S_lo);
      opB.base = wsp<float>(e, e->ws.tgt_hi); opB.lo = wsp<float>(e, e->ws.tgt_lo);
    }
    // enough split-K slices to fill the SMs about twice; few when the batch already gives many tiles
    const int tiles = ((B + 127) / 128) * ((D + 191) / 192);
    int want = (2 * e->num_sms + tiles - 1) / tiles;
    if (want > kSplitDv) want = kSplitDv;
    const int ks = umma::effective_splits(Y, want);
    umma::EpiStore ep{part, (size_t)D, (size_t)B * D};
    if (e->sg_live) {       // A = the logits slab, rewritten to dL/dlogits tile by tile in shared memory
      umma::AXSoftmaxGradK<4> ax{e->sg};
      C2V_LAUNCH(e, C2V_CUDA(e, (umma::launch_cfg<192, 4, false, true, umma::EpiStore, umma::AXSoftmaxGradK<4>>(st, B, D, Y, want, opA, opB, ep,
                                                                                                            e->num_sms, ax))));
    } else {
      C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_192(st, B, D, Y, want, opA, opB, ep, e->num_sms))));
    }
    return launch_colsum(e, st, part, (size_t)B * D, ks, B * D, dv, e->row_scale, D);
  }
  simt::RowsK al{S, e->ws.ldS};
  simt::ColsX bl{e->theta.tgt, (size_t)D};
  const int ks = simt::effective_ksplit(Y, kSplitDv);
  simt::StoreC ep{part, (size_t)D, (size_t)B * D};
  C2V_LAUNCH(e, C2V_CUDA(e, simt::launch(st, B, D, Y, kSplitDv, al, bl, ep)));
  return launch_colsum(e, st, part, (size_t)B * D, ks, B * D, dv);
}

// dYtab = P^T . v  into the bound target-table gradient; then the caller's "target_grads_ready" event.
int run_dy(c2v_engine* e, cudaStream_t st, const float* v, int B) {
  const int D = e->dims.code_dim, Y = e->dims.target_vocab;
  float* S = wsp<float>(e, e->ws.S);
  {
    PhaseTimer pt(e, PH_DY, st);
    if (is_3x(e) && (reinterpret_cast<uintptr_t>(v) % 16 != 0))
      return fail(e, C2V_ERR_INVALID, "3xTF32: the code vectors must be 16-byte aligned");
    if (is_tc(e) && (reinterpret_cast<uintptr_t>(v) % 16 == 0)) {
      umma::Operand opA{S, e->ws.ldS, true};
      umma::Operand opB{v, (size_t)D, true};
      if (is_3x(e)) {
        int rcs = split_small(e, st, v, (size_t)B * D, e->ws.v_hi, e->ws.v_lo);
        if (rcs) return rcs;
        opA.lo = wsp<float>(e, e->ws.S_lo);
        opB.base = wsp<float>(e, e->ws.v_hi); opB.lo = wsp<float>(e, e->ws.v_lo);
      }
      if (e->tgt_armed && e->has_adam) {
        // dYtab never reaches memory: the epilogue applies TF1 Adam to the target table in place
        const double lr_t = (double)e->tgt_lr * sqrt(1.0 - pow((double)e->tgt_b2, (double)e->tgt_t)) /
                            (1.0 - pow((double)e->tgt_b1, (double)e->tgt_t));
        umma::EpiAdam ep{e->theta.tgt, e->am.tgt, e->av.tgt, (size_t)D, (float)lr_t, e->tgt_b1, e->tgt_b2, e->tgt_eps,
                         1.f - e->tgt_b1, 1.f - e->tgt_b2, e->adam_epi_prefetch};
        if (e->sg_live) {
          umma::AXSoftmaxGradMN<2> ax{e->sg};
          C2V_LAUNCH(e, C2V_CUDA(e, (umma::launch_cfg<192, 4, true, true, umma::EpiAdam, umma::AXSoftmaxGradMN<2>>(st, Y, D, B, 1, opA, opB, ep,
                                                                                                               e->num_sms, ax))));
        } else {
          C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_FIXED(192, true, true, false, umma::EpiAdam, st, Y, D, B, 1, opA, opB, ep, e->num_sms))));
        }
        e->tgt_armed = false;
        e->tgt_fused_t = e->tgt_t;
        e->tgt_split_valid = false;
      } else {
        umma::EpiStore ep{e->grad.tgt, (size_t)D, 0};
        if (e->sg_live) {
          umma::AXSoftmaxGradMN<2> ax{e->sg};
          C2V_LAUNCH(e, C2V_CUDA(e, (umma::launch_cfg<192, 4, true, true, umma::EpiStore, umma::AXSoftmaxGradMN<2>>(st, Y, D, B, 1, opA, opB, ep,
                                                                                                                e->num_sms, ax))));
        } else {
          C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_192_SINGLE(st, Y, D, B, 1, opA, opB, ep, e->num_sms))));
        }
      }
    } else {
      simt::ColsX al{S, e->ws.ldS};
      simt::ColsX bl{v, (size_t)D};
      simt::StoreC ep{e->grad.tgt, (size_t)D, 0};
      C2V_LAUNCH(e, C2V_CUDA(e, simt::launch(st, Y, D, B, 1, al, bl, ep)));
    }
  }
  if (e->ev_tgt_ready) C2V_CUDA(e, cudaEventRecord(e->ev_tgt_ready, st));
  return C2V_OK;
}

// The two target-table gradient products.  With option "dy_late" (default) only dv runs here and dY is
// deferred into context_backward, where it overlaps the NVLink / L2-atomic bound scatter-add of the
// embedding gradients (dY needs P and v only, not the context backward).
int target_grad_gemms(c2v_engine* e, cudaStream_t st, const float* v, int B, float* dv) {
  int rc = run_dv(e, st, B, dv);
  if (rc) return rc;
  if (e->dy_late == 2 && is_tc(e)) {
    // dY (and the target table's Adam step in its epilogue) is HBM-bound and independent of the context
    // backward pass: it runs on its own stream from here until context_backward joins it
    C2V_CUDA(e, cudaEventRecord(e->ev_fork2, st));
    C2V_CUDA(e, cudaStreamWaitEvent(e->side2, e->ev_fork2, 0));
    if ((rc = run_dy(e, e->side2, v, B))) return rc;
    C2V_CUDA(e, cudaEventRecord(e->ev_join2, e->side2));
    e->dy_in_flight = true;
    return C2V_OK;
  }
  if (e->dy_late) {
    e->pending_dy_v = v;
    e->pending_dy_B = B;
    return C2V_OK;
  }
  return run_dy(e, st, v, B);
}

int train_step_impl(c2v_engine* e, cudaStream_t st, const int32_t* src, const int32_t* pth, const int32_t* tgt,
                    const float* mask, const int32_t* target, int B, float keep, uint64_t seed, uint64_t step,
                    const float* ext_mask, float* loss_out) {
  if (!e->has_grad) return fail(e, C2V_ERR_STATE, "gradients not bound (c2v_bind_grads)");
  if (!(keep > 0.f) || keep > 1.f) return fail(e, C2V_ERR_INVALID, "keep_prob must be in (0, 1]");
  const int Y = e->dims.target_vocab;
  const Dropout dp = make_dropout(e->dims, keep, seed, step, ext_mask);
  ContextSource cs = make_source(e, src, pth, tgt, B);
  float* H = wsp<float>(e, e->ws.H);
  float* alpha = wsp<float>(e, e->ws.alpha);
  float* v = wsp<float>(e, e->ws.v);
  float* dv = wsp<float>(e, e->ws.dv);
  float* S = wsp<float>(e, e->ws.S);
  float* loss_b = wsp<float>(e, e->ws.loss_b);
  float* lse = wsp<float>(e, e->ws.lse);
  int rc;
  if ((rc = run_ctx_fwd(e, st, cs, dp, H, true))) return rc;
  if ((rc = launch_attn_fwd(e, st, H, mask, B, alpha, v))) return rc;
  const bool fused_lse = (is_tc(e));
  const float invB = 1.0f / (float)B;
  if (fused_lse && e->recompute && !e->fuse_sg) {
    // the slab is written ONCE, as dL/dlogits: pass 1 of the logits GEMM leaves only log-sum-exp partials, the true-class
    // logit comes from a B-row dot product, pass 2 repeats the product and its epilogue writes (softmax - onehot) / B
    if ((rc = run_logits(e, st, v, B, S, false, true))) return rc;
    float* tl = wsp<float>(e, e->ws.true_logit);
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (true_logit_kernel<<<(B + 7) / 8, 256, 0, st>>>(v, e->theta.tgt, target, 0, Y, e->dims.code_dim, B, tl)));
      C2V_LAUNCH(e, (xent_combine_kernel<<<B, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), 2 * ((Y + 255) / 256), S, e->ws.ldS, target,
                                                            loss_b, lse, tl)));
      C2V_LAUNCH(e, (loss_reduce_kernel<<<1, 256, 0, st>>>(loss_b, B, invB, loss_out)));
    }
    e->sg_live = false;
    const LogitsGrad lg{lse, target, 0, invB};
    if ((rc = run_logits(e, st, v, B, S, false, false, &lg))) return rc;
    if ((rc = target_grad_gemms(e, st, v, B, dv))) return rc;
    return context_backward(e, st, cs, mask, B, dp, dv);
  }
  if (fused_lse && e->exp_slab && !e->fuse_sg) {
    // deferred normalisation: U = exp(s - true logit) from the logits epilogue, one patched element and one factor per row;
    // the gated kernels after the combine are the two-pass schedule, run by the device only when a row left the fp32 window
    const int D = e->dims.code_dim;
    const int n_tiles = 2 * ((Y + 255) / 256);
    float* tl = wsp<float>(e, e->ws.true_logit);
    float* rscale = wsp<float>(e, e->ws.rscale);
    float* vs = wsp<float>(e, e->ws.v_scaled);
    int* flag = wsp<int>(e, e->ws.slab_flag);
    float* S_lo = is_3x(e) ? wsp<float>(e, e->ws.S_lo) : nullptr;
    if (!e->slab_flag_zeroed) {
      C2V_CUDA(e, cudaMemsetAsync(flag, 0, 64, st));
      e->slab_flag_zeroed = true;
    }
    if ((rc = end_target_lazy(e, st))) return rc;      // the true-class rows are read below: every target row must be current
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (true_logit_kernel<<<(B + 7) / 8, 256, 0, st>>>(v, e->theta.tgt, target, 0, Y, D, B, tl, flag)));
    }
    if ((rc = run_logits(e, st, v, B, S, false, false, nullptr, tl))) return rc;
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (expsum_combine_kernel<<<B, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), n_tiles, S, S_lo, e->ws.ldS, Y, target, tl, tl, invB,
                                                              loss_b, lse, rscale, flag)));
    }
    if ((rc = run_logits(e, st, v, B, S, true, false, nullptr, nullptr, flag))) return rc;
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (xent_combine_kernel<<<B, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), n_tiles, S, e->ws.ldS, target, loss_b, lse, nullptr, flag,
                                                            rscale, reinterpret_cast<unsigned*>(flag) + 1)));
      const int chunks = 2;        // the fallback only has to be correct; a small grid keeps the closed gate cheap
      if (S_lo) C2V_LAUNCH(e, (softmax_grad_kernel<true><<<dim3(chunks, B), 256, 0, st>>>(S, e->ws.ldS, Y, lse, target, invB, 0, S_lo, flag)));
      else C2V_LAUNCH(e, (softmax_grad_kernel<false><<<dim3(chunks, B), 256, 0, st>>>(S, e->ws.ldS, Y, lse, target, invB, 0, nullptr, flag)));
      C2V_LAUNCH(e, (scale_rows_kernel<<<(unsigned)(((size_t)B * D + 255) / 256), 256, 0, st>>>(v, rscale, vs, D, (size_t)B * D)));
      C2V_LAUNCH(e, (loss_reduce_kernel<<<1, 256, 0, st>>>(loss_b, B, invB, loss_out)));
    }
    e->sg_live = false;
    e->row_scale = rscale;
    rc = target_grad_gemms(e, st, vs, B, dv);
    e->row_scale = nullptr;
    if (rc) return rc;
    return context_backward(e, st, cs, mask, B, dp, dv);
  }
  if ((rc = run_logits(e, st, v, B, S, fused_lse))) return rc;
  {
    PhaseTimer pt(e, PH_XENT, st);
    if (fused_lse) {
      const int n_tiles = 2 * ((Y + 255) / 256);       // partial slots per row
      C2V_LAUNCH(e, (xent_combine_kernel<<<B, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), n_tiles, S, e->ws.ldS, target,
                                                            loss_b, lse)));
      const int chunks = (int)((e->ws.ldS / 4 + 256 * 8 - 1) / (256 * 8));
      e->sg_live = false;
      if (is_3x(e))
        C2V_LAUNCH(e, (softmax_grad_kernel<true><<<dim3(chunks, B), 256, 0, st>>>(S, e->ws.ldS, Y, lse, target, invB, 0, wsp<float>(e, e->ws.S_lo))));
      else if (e->fuse_sg) {
        // no pass over the slab: the dv and dY GEMMs turn logits into (softmax - onehot) / B as their A tiles land
        e->sg = umma::SoftmaxGradArgs{lse, target, 0, invB};
        e->sg_live = true;
      } else
        C2V_LAUNCH(e, (softmax_grad_kernel<false><<<dim3(chunks, B), 256, 0, st>>>(S, e->ws.ldS, Y, lse, target, invB, 0, nullptr)));
    } else {
      C2V_LAUNCH(e, (xent_kernel<<<B, kXentThreads, 0, st>>>(S, e->ws.ldS, target, Y, invB, loss_b, lse, 1)));
    }
    C2V_LAUNCH(e, (loss_reduce_kernel<<<1, 256, 0, st>>>(loss_b, B, invB, loss_out)));
  }
  if ((rc = target_grad_gemms(e, st, v, B, dv))) return rc;
  return context_backward(e, st, cs, mask, B, dp, dv);
}

int sampled_train_step_impl(c2v_engine* e, cudaStream_t st, const int32_t* src, const int32_t* pth, const int32_t* tgt,
                             const float* mask, const int32_t* target, int B, const int32_t* sampled, int S,
                             const float* logq_true, const float* logq_samp, float keep, uint64_t seed, uint64_t step,
                             const float* ext_mask, float* loss_out) {
  if (!e->has_grad) return fail(e, C2V_ERR_STATE, "gradients not bound (c2v_bind_grads)");
  if (!(keep > 0.f) || keep > 1.f) return fail(e, C2V_ERR_INVALID, "keep_prob must be in (0, 1]");
  if (S < 1 || S > kMaxSampled) return fail(e, C2V_ERR_INVALID, "number of sampled classes must be in [1, 1024]");
  const int D = e->dims.code_dim;
  const Dropout dp = make_dropout(e->dims, keep, seed, step, ext_mask);
  ContextSource cs = make_source(e, src, pth, tgt, B);
  float* H = wsp<float>(e, e->ws.H);
  float* alpha = wsp<float>(e, e->ws.alpha);
  float* v = wsp<float>(e, e->ws.v);
  float* dv = wsp<float>(e, e->ws.dv);
  float* loss_b = wsp<float>(e, e->ws.loss_b);
  float* dl = wsp<float>(e, e->ws.dl);
  int rc;
  if ((rc = run_ctx_fwd(e, st, cs, dp, H, true))) return rc;
  if ((rc = launch_attn_fwd(e, st, H, mask, B, alpha, v))) return rc;
  const float invB = 1.0f / (float)B;
  if (e->lazy && e->has_adam && e->table_world == 1) {
    // TF1 applies sampled-softmax gradients as IndexedSlices: every row of the table still decays m, v and moves
    // (SURVEY A.3), exactly as for the embedding tables -- so the same deferred, bit-exact row replay applies, and
    // a step touches only the B + S rows it reads instead of streaming 24 B x 100 M parameters.
    PhaseTimer pt(e, PH_ADAM_CATCHUP, st);
    const c2v_dims& d = e->dims;
    int32_t* stamp = wsp<int32_t>(e, e->ws.stamp_tgt);
    int32_t* last = wsp<int32_t>(e, e->ws.last_tgt);
    if (!e->tgt_lazy) {          // the table joins the lazily updated set: every row is current as of adam_t_done
      C2V_CUDA(e, cudaMemsetAsync(e->grad.tgt, 0, (size_t)d.target_vocab * D * 4, st));
      C2V_LAUNCH(e, (fill_i32_kernel<<<256, 256, 0, st>>>(last, (size_t)d.target_vocab, (int32_t)e->adam_t_done)));
      C2V_CUDA(e, cudaMemsetAsync(stamp, 0, (size_t)d.target_vocab * 4, st));
      e->tgt_lazy = true;
    }
    e->mark_epoch++;
    C2V_LAUNCH(e, (mark_list_kernel<<<(B + 255) / 256, 256, 0, st>>>(target, B, stamp, e->mark_epoch)));
    C2V_LAUNCH(e, (mark_list_kernel<<<(S + 255) / 256, 256, 0, st>>>(sampled, S, stamp, e->mark_epoch)));
    if (e->adam_t_done > 0)
      C2V_ADAM_ROWS(e, ADAM_ROWS_CATCHUP, st,
                    e->theta.tgt, e->grad.tgt, e->am.tgt, e->av.tgt, d.target_vocab, d.code_dim, stamp, e->mark_epoch, last,
                    (int32_t)e->adam_t_done, wsp<float>(e, e->ws.lr_tab), e->hp_b1, e->hp_b2, e->hp_eps, rest_ok(e));
  }
  {
    PhaseTimer pt(e, PH_SAMPLED, st);
    const size_t smem = ((size_t)D + S + 1) * sizeof(float);
    C2V_LAUNCH(e, (sampled_softmax_fwd_kernel<<<B, kSampledThreads, smem, st>>>(v, e->theta.tgt, target, sampled, S, logq_true,
                                                                                 logq_samp, D, invB, loss_b, dl, dv)));
    C2V_LAUNCH(e, (loss_reduce_kernel<<<1, 256, 0, st>>>(loss_b, B, invB, loss_out)));
    // the target-table gradient is sparse here (B + S rows).  Lazy Adam: the rows were brought up to date (and
    // their gradient rows cleared) before the forward kernel read them; the update of this step is deferred
    // like an embedding row's.  Dense Adam: the bound buffer is dense, so it is cleared first.
    if (!e->tgt_lazy) C2V_CUDA(e, cudaMemsetAsync(e->grad.tgt, 0, (size_t)e->dims.target_vocab * D * 4, st));
    C2V_LAUNCH(e, (sampled_softmax_bwd_kernel<<<B + S * ((B + kSampledChunk - 1) / kSampledChunk), kSampledThreads, 0, st>>>(
        v, dl, target, sampled, B, S, D, e->grad.tgt)));
  }
  if (e->ev_tgt_ready) C2V_CUDA(e, cudaEventRecord(e->ev_tgt_ready, st));
  return context_backward(e, st, cs, mask, B, dp, dv);
}

int adam_impl(c2v_engine* e, cudaStream_t st, float lr, float b1, float b2, float eps, int64_t t) {
  if (!e->has_grad || !e->has_adam) return fail(e, C2V_ERR_STATE, "gradients / Adam state not bound");
  if (e->table_world > 1)
    return fail(e, C2V_ERR_STATE, "embedding tables are sharded: update each slice with c2v_adam_step_range");
  if (t < 1) return fail(e, C2V_ERR_INVALID, "Adam step count t must be >= 1");
  e->tgt_armed = false;                 // an unconsumed arming (fp32 path, sampled softmax) falls back to the dense update
  e->armed_t = 0;
  e->hint_src = e->hint_pth = e->hint_tgt = nullptr;      // a hint the step could not use is dropped
  bool skip_tgt = false;
  if (e->tgt_fused_t || e->early_t) {
    const int64_t done_t = e->tgt_fused_t ? e->tgt_fused_t : e->early_t;
    if (done_t != t || lr != e->tgt_lr || b1 != e->tgt_b1 || b2 != e->tgt_b2 || eps != e->tgt_eps)
      return fail(e, C2V_ERR_STATE, "part of this Adam step was already applied inside the train step (c2v_arm_target_adam) with a different step count / hyper-parameters");
    skip_tgt = e->tgt_fused_t != 0;
    e->tgt_fused_t = 0;
    e->early_t = 0;
  }
  const double lr_t_d = (double)lr * sqrt(1.0 - pow((double)b2, (double)t)) / (1.0 - pow((double)b1, (double)t));
  const float lr_t = (float)lr_t_d;
  const c2v_dims& d = e->dims;
  const size_t n[5] = {(size_t)d.token_vocab * d.embed_dim, (size_t)d.path_vocab * d.embed_dim,
                       (size_t)d.target_vocab * d.code_dim, (size_t)3 * d.embed_dim * d.code_dim, (size_t)d.code_dim};
  float* P[5] = {e->theta.tok, e->theta.path, e->theta.tgt, e->theta.W, e->theta.a};
  float* G[5] = {e->grad.tok, e->grad.path, e->grad.tgt, e->grad.W, e->grad.a};
  float* M[5] = {e->am.tok, e->am.path, e->am.tgt, e->am.W, e->am.a};
  float* V[5] = {e->av.tok, e->av.path, e->av.tgt, e->av.W, e->av.a};
  int first_dense = 0;
  if (e->lazy) {
    if (t != e->adam_t_done + 1) return fail(e, C2V_ERR_STATE, "lazy Adam needs consecutive step counts (t == previous t + 1)");
    if (e->hp_set && (lr != e->hp_lr || b1 != e->hp_b1 || b2 != e->hp_b2 || eps != e->hp_eps)) {
      int rcf = flush_rows(e, st);                  // pending steps must use the old hyper-parameters
      if (rcf) return rcf;
    }
    // the learning rates of pending steps live in a ring: no row may fall a whole ring behind (only possible
    // with the sweep switched off)
    if (t - e->full_flush_t >= kLrRing - 2) {
      int rcf = flush_rows(e, st);
      if (rcf) return rcf;
    }
    e->hp_lr = lr; e->hp_b1 = b1; e->hp_b2 = b2; e->hp_eps = eps; e->hp_set = true;
    float* lr_tab = wsp<float>(e, e->ws.lr_tab);
    // the embedding rows' step t is deferred: their gradient rows keep this step's scatter-add until the
    // rows are next referenced (prepare_rows), swept (sweep_rows) or flushed; only the learning rate of the
    // step is recorded
    C2V_LAUNCH(e, (set_float_kernel<<<1, 1, 0, st>>>(lr_tab + (t & kLrRingMask), lr_t)));
    e->lazy_grads_pending = false;
    first_dense = 2;
  }
  e->adam_t_done = t;
  e->tgt_split_valid = false;
  if (e->lazy) { int rcs = sweep_rows(e, st, t); if (rcs) return rcs; }
  for (int i = first_dense; i < 5; ++i) {
    if (i == 2 && (skip_tgt || e->tgt_lazy)) continue;     // lazy target rows: deferred like the embedding rows
    const size_t n4 = n[i] / 4;
    size_t blocks = (n4 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    const int zero = (i < 2) ? 1 : 0;   // embedding gradient tables are cleared for the next scatter-add
    PhaseTimer pt(e, PH_ADAM, st);
    C2V_LAUNCH(e, (adam_kernel<<<(unsigned)blocks, 256, 0, st>>>(P[i], G[i], M[i], V[i], n4, lr_t, b1, b2, eps, zero)));
  }
  e->emb_grads_clean = !e->lazy;     // lazy: the gradient tables hold deferred steps, cleared row by row as they are applied
  return C2V_OK;
}

// ---- nearest-neighbour search (similarity.cuh) ----------------------------------------------------
// Touches neither the workspace nor any engine state: a search between two train steps leaves the next step unchanged.
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int check_bank(c2v_engine* e, const float* bank, int64_t rows, int32_t dim) {
  if (!bank) return fail(e, C2V_ERR_INVALID, "bank is NULL");
  if (rows < 1 || rows > INT32_MAX) return fail(e, C2V_ERR_INVALID, "rows must be in [1, 2^31)");
  if (dim < 4 || dim > 1024 || dim % 4) return fail(e, C2V_ERR_INVALID, "dim must be a multiple of 4 in [4, 1024]");
  if (!aligned16(bank)) return fail(e, C2V_ERR_INVALID, "bank must be 16-byte aligned");
  return C2V_OK;
}

template <int QB>
int launch_nearest(c2v_engine* e, cudaStream_t st, const float* bank, int rows, int dim, const float* queries, int n, int k,
                   const int32_t* exclude, int n_exclude, const sim::Layout& L, int slices, ValIdx* cand) {
  C2V_CUDA(e, cudaFuncSetAttribute(sim::nearest_kernel<QB>, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
  const dim3 grid((unsigned)((n + L.qc - 1) / L.qc), (unsigned)slices);
  C2V_LAUNCH(e, (sim::nearest_kernel<QB><<<grid, sim::kThreads, L.total, st>>>(bank, rows, dim, queries, n, k, exclude,
                                                                                n_exclude, L, cand)));
  return C2V_OK;
}

int nearest_impl(c2v_engine* e, cudaStream_t st, const float* bank, int rows, int dim, const float* queries, int n, int k,
                 const int32_t* exclude, int n_exclude, int32_t* idx, float* val, void* scratch) {
  const sim::Layout L = sim::make_layout(dim, k);
  const int slices = sim::slices_for(rows);
  ValIdx* cand = reinterpret_cast<ValIdx*>(scratch);
  // register block of 1, 2, 4 or 8 queries: a single query does not pay for seven zero ones
  int rc;
  if (n == 1) rc = launch_nearest<1>(e, st, bank, rows, dim, queries, n, k, exclude, n_exclude, L, slices, cand);
  else if (n == 2) rc = launch_nearest<2>(e, st, bank, rows, dim, queries, n, k, exclude, n_exclude, L, slices, cand);
  else if (n <= 4) rc = launch_nearest<4>(e, st, bank, rows, dim, queries, n, k, exclude, n_exclude, L, slices, cand);
  else rc = launch_nearest<8>(e, st, bank, rows, dim, queries, n, k, exclude, n_exclude, L, slices, cand);
  if (rc) return rc;
  C2V_LAUNCH(e, (sim::merge_kernel<<<n, kTopkThreads, 0, st>>>(cand, slices, k, idx, val)));
  return C2V_OK;
}

}  // namespace

// ================================== C ABI =======================================================
extern "C" {

int c2v_abi_version(void) { return C2V_ABI_VERSION; }

const char* c2v_last_error(const c2v_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

size_t c2v_workspace_bytes(const c2v_dims* dims) {
  std::string why;
  if (!dims_ok(dims, &why)) { g_create_error = why; return 0; }
  return carve(*dims).total;
}

int c2v_create(const c2v_dims* dims, int device, c2v_engine** out) {
  if (!out) return fail(nullptr, C2V_ERR_INVALID, "out is NULL");
  *out = nullptr;
  std::string why;
  if (!dims_ok(dims, &why)) return fail(nullptr, C2V_ERR_INVALID, why);
  int ndev = 0;
  cudaError_t c = cudaGetDeviceCount(&ndev);
  if (c != cudaSuccess || ndev < 1)
    return fail(nullptr, C2V_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(c));
  if (device < 0 || device >= ndev) return fail(nullptr, C2V_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  c = cudaGetDeviceProperties(&prop, device);
  if (c != cudaSuccess) return fail(nullptr, C2V_ERR_CUDA, cudaGetErrorString(c));
  if (prop.major != 10)
    return fail(nullptr, C2V_ERR_UNSUPPORTED, "this library is built for sm_100a (B200) only");
  c2v_engine* e = new c2v_engine();
  e->dims = *dims;
  e->device = device;
  e->ws = carve(*dims);
  e->wbase = nullptr;
  e->wbytes = 0;
  e->has_theta = e->has_grad = e->has_adam = false;
  e->emb_grads_clean = false;
  e->math_mode = C2V_MATH_FP32;
  e->num_sms = prop.multiProcessorCount;
  cudaSetDevice(device);
  if (cudaStreamCreateWithFlags(&e->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->side2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_fork2, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_join2, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->copy, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_h2d[0], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_h2d[1], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_used[0], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_used[1], cudaEventDisableTiming) != cudaSuccess) {
    delete e;
    return fail(nullptr, C2V_ERR_CUDA, "could not create the engine's side stream / events");
  }
  e->deterministic = 0;
  e->launches = 0;
  *out = e;
  return C2V_OK;
}

void c2v_destroy(c2v_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->side) cudaStreamDestroy(e->side);
  if (e->ev_fork2) cudaEventDestroy(e->ev_fork2);
  if (e->ev_join2) cudaEventDestroy(e->ev_join2);
  if (e->side2) cudaStreamDestroy(e->side2);
  for (int i = 0; i < 2; ++i) {
    if (e->ev_h2d[i]) cudaEventDestroy(e->ev_h2d[i]);
    if (e->ev_used[i]) cudaEventDestroy(e->ev_used[i]);
  }
  if (e->copy) cudaStreamDestroy(e->copy);
  for (auto& L : e->phase) {
    for (auto& ev : L.pending) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    for (auto& ev : L.free_list) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
  }
  delete e;
}

int c2v_bind_workspace(c2v_engine* e, void* dev_ptr, size_t bytes) {
  if (!e) return C2V_ERR_INVALID;
  if (!dev_ptr) return fail(e, C2V_ERR_INVALID, "workspace pointer is NULL");
  if (((uintptr_t)dev_ptr) % kAlign) return fail(e, C2V_ERR_INVALID, "workspace must be 256-byte aligned");
  if (bytes < e->ws.total) return fail(e, C2V_ERR_INVALID, "workspace smaller than c2v_workspace_bytes()");
  e->wbase = (char*)dev_ptr;
  e->wbytes = bytes;
  e->bkt_zeroed = false;
  e->slab_flag_zeroed = false;
  return C2V_OK;
}

int c2v_bind_params(c2v_engine* e, const c2v_tensors* t) {
  if (!e) return C2V_ERR_INVALID;
  if (!has_all(t)) return fail(e, C2V_ERR_INVALID, "all five parameter pointers must be non-NULL");
  e->theta = *t; e->has_theta = true;
  e->th_tok = ShardedTable{}; e->th_path = ShardedTable{};
  e->th_tok.base[0] = t->tok; e->th_path.base[0] = t->path;
  e->table_world = 1; e->grad_scale = 1.f;
  return C2V_OK;
}

int c2v_bind_grads(c2v_engine* e, const c2v_tensors* t) {
  if (!e) return C2V_ERR_INVALID;
  if (!has_all(t)) return fail(e, C2V_ERR_INVALID, "all five gradient pointers must be non-NULL");
  e->grad = *t; e->has_grad = true; e->emb_grads_clean = false;
  e->gr_tok = ShardedTable{}; e->gr_path = ShardedTable{};
  e->gr_tok.base[0] = t->tok; e->gr_path.base[0] = t->path;
  return C2V_OK;
}

int c2v_bind_adam_state(c2v_engine* e, const c2v_tensors* m, const c2v_tensors* v) {
  if (!e) return C2V_ERR_INVALID;
  if (!has_all(m) || !has_all(v)) return fail(e, C2V_ERR_INVALID, "all ten Adam slot pointers must be non-NULL");
  e->am = *m; e->av = *v; e->has_adam = true;
  return C2V_OK;
}

int c2v_set_option(c2v_engine* e, const char* key, int64_t value) {
  if (!e || !key) return C2V_ERR_INVALID;
  if (!strcmp(key, "math_mode")) {
    if (value != C2V_MATH_FP32 && value != C2V_MATH_TF32 && value != C2V_MATH_3XTF32)
      return fail(e, C2V_ERR_INVALID, "unknown math_mode");
    if (value != C2V_MATH_FP32 && !umma::get_encode_fn())
      return fail(e, C2V_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled not available from the driver");
    e->math_mode = (int)value;
    return C2V_OK;
  }
  if (!strcmp(key, "deterministic")) {
    if (value) return fail(e, C2V_ERR_UNSUPPORTED, "deterministic (sorted) embedding scatter-add is not built; float atomics only");
    e->deterministic = 0;
    return C2V_OK;
  }
  if (!strcmp(key, "profile")) { e->profile = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "dy_late")) {
    if (value < 0 || value > 2) return fail(e, C2V_ERR_INVALID, "dy_late must be 0, 1 or 2");
    e->dy_late = (int)value;
    return C2V_OK;
  }
  if (!strcmp(key, "fuse_target_adam")) { e->fuse_tgt = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "fuse_gather")) { e->fuse_gather = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "fuse_softmax_grad")) { e->fuse_sg = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "exp_slab")) { e->exp_slab = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "adam_epilogue_prefetch")) { e->adam_epi_prefetch = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "recompute_logits")) { e->recompute = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "sort_peer_access")) {
    if (value < 0 || value > 2) return fail(e, C2V_ERR_INVALID, "sort_peer_access must be 0 (never), 1 (auto) or 2 (always)");
    e->sort_peer = (int)value;
    return C2V_OK;
  }
  if (!strcmp(key, "adam_rest_shortcut")) { e->rest_shortcut = value ? 1 : 0; return C2V_OK; }
  if (!strcmp(key, "adam_sweep_period")) {
    if (value < 0 || value > kLrRing / 2) return fail(e, C2V_ERR_INVALID, "adam_sweep_period must be in [0, 32768]");
    e->sweep_period = (int)value;
    return C2V_OK;
  }
  if (!strcmp(key, "adam_rows_occupancy")) {
    if (value != 4 && value != 5) return fail(e, C2V_ERR_INVALID, "adam_rows_occupancy must be 4 or 5");
    e->adam_rows_occ = (int)value;
    return C2V_OK;
  }
  if (!strcmp(key, "cta_pair")) {
    if (value < 0 || value > 2) return fail(e, C2V_ERR_INVALID, "cta_pair must be 0 (never), 1 (always) or 2 (auto)");
    e->cta_pair = (int)value;
    return C2V_OK;
  }
  if (!strcmp(key, "grad_scale_inverse")) {               // scatter-add scale = 1 / value (1 = unscaled)
    if (value < 1) return fail(e, C2V_ERR_INVALID, "grad_scale_inverse must be >= 1");
    e->grad_scale = 1.0f / (float)value;
    return C2V_OK;
  }
  if (!strcmp(key, "lazy_adam")) {
    if (!e->wbase || !e->has_theta || !e->has_grad || !e->has_adam)
      return fail(e, C2V_ERR_STATE, "bind workspace, parameters, gradients and Adam state before lazy_adam");
    if (value && e->table_world > 1) return fail(e, C2V_ERR_STATE, "lazy_adam is for replicated (single-GPU) tables");
    C2V_CUDA(e, cudaSetDevice(e->device));
    if (!value && e->lazy) {                              // bring every row up to date, then go dense
      int rc = flush_rows(e, 0);
      if (rc) return rc;
      C2V_CUDA(e, cudaStreamSynchronize(0));
      e->emb_grads_clean = !e->lazy_grads_pending;        // every applied gradient row was cleared on the way
      e->lazy_grads_pending = false;
      e->tgt_lazy = false;
    }
    if (value && !e->lazy) {                              // all rows are current as of adam_t_done
      const c2v_dims& d = e->dims;
      if (!e->emb_grads_clean) {                          // deferred steps read the gradient rows: they must start from zero
        C2V_CUDA(e, cudaMemset(e->grad.tok, 0, (size_t)d.token_vocab * d.embed_dim * 4));
        C2V_CUDA(e, cudaMemset(e->grad.path, 0, (size_t)d.path_vocab * d.embed_dim * 4));
      }
      e->lazy_grads_pending = false;
      C2V_LAUNCH(e, (fill_i32_kernel<<<256, 256>>>(wsp<int32_t>(e, e->ws.last_tok), (size_t)d.token_vocab, (int32_t)e->adam_t_done)));
      C2V_LAUNCH(e, (fill_i32_kernel<<<256, 256>>>(wsp<int32_t>(e, e->ws.last_path), (size_t)d.path_vocab, (int32_t)e->adam_t_done)));
      C2V_CUDA(e, cudaMemset(wsp<int32_t>(e, e->ws.stamp_tok), 0, (size_t)d.token_vocab * 4));
      C2V_CUDA(e, cudaMemset(wsp<int32_t>(e, e->ws.stamp_path), 0, (size_t)d.path_vocab * 4));
      e->mark_epoch = 0;
      e->full_flush_t = e->adam_t_done;
      e->tgt_lazy = false;
      C2V_CUDA(e, cudaDeviceSynchronize());
    }
    e->lazy = value ? 1 : 0;
    return C2V_OK;
  }
  if (!strcmp(key, "target_adam_fused_step")) {           // callers that run c2v_adam_step_range themselves acknowledge with 0
    if (value) return fail(e, C2V_ERR_INVALID, "target_adam_fused_step can only be cleared (0)");
    e->tgt_fused_t = 0;
    return C2V_OK;
  }
  if (!strcmp(key, "adam_step_count")) {                  // optimizer reset / checkpoint restore
    C2V_CUDA(e, cudaSetDevice(e->device));
    if (e->lazy) {
      int rc = flush_rows(e, 0);
      if (rc) return rc;
      const c2v_dims& d = e->dims;
      C2V_LAUNCH(e, (fill_i32_kernel<<<256, 256>>>(wsp<int32_t>(e, e->ws.last_tok), (size_t)d.token_vocab, (int32_t)value)));
      C2V_LAUNCH(e, (fill_i32_kernel<<<256, 256>>>(wsp<int32_t>(e, e->ws.last_path), (size_t)d.path_vocab, (int32_t)value)));
      C2V_CUDA(e, cudaDeviceSynchronize());
      e->tgt_lazy = false;                                // flush_rows brought the target rows up to date as well
      e->full_flush_t = value;
    }
    e->adam_t_done = value;
    e->hp_set = false;
    return C2V_OK;
  }
  return fail(e, C2V_ERR_INVALID, std::string("unknown option: ") + key);
}

int c2v_get_option(const c2v_engine* e, const char* key, int64_t* value) {
  if (!e || !key || !value) return C2V_ERR_INVALID;
  if (!strcmp(key, "math_mode")) { *value = e->math_mode; return C2V_OK; }
  if (!strcmp(key, "deterministic")) { *value = e->deterministic; return C2V_OK; }
  if (!strcmp(key, "profile")) { *value = e->profile; return C2V_OK; }
  if (!strcmp(key, "lazy_adam")) { *value = e->lazy; return C2V_OK; }
  if (!strcmp(key, "adam_sweep_period")) { *value = e->sweep_period; return C2V_OK; }
  if (!strcmp(key, "adam_rest_shortcut")) { *value = e->rest_shortcut; return C2V_OK; }
  if (!strcmp(key, "adam_rows_occupancy")) { *value = e->adam_rows_occ; return C2V_OK; }
  if (!strcmp(key, "cta_pair")) { *value = e->cta_pair; return C2V_OK; }
  if (!strcmp(key, "dy_late")) { *value = e->dy_late; return C2V_OK; }
  if (!strcmp(key, "fuse_target_adam")) { *value = e->fuse_tgt; return C2V_OK; }
  if (!strcmp(key, "fuse_gather")) { *value = e->fuse_gather; return C2V_OK; }
  if (!strcmp(key, "fuse_softmax_grad")) { *value = e->fuse_sg; return C2V_OK; }
  if (!strcmp(key, "exp_slab")) { *value = e->exp_slab; return C2V_OK; }
  if (!strcmp(key, "adam_epilogue_prefetch")) { *value = e->adam_epi_prefetch; return C2V_OK; }
  if (!strcmp(key, "exp_slab_fallbacks")) {       // steps so far that left the fp32 window and ran the two-pass schedule (synchronises)
    *value = 0;
    if (e->wbase && e->slab_flag_zeroed) {
      unsigned n = 0;
      if (cudaDeviceSynchronize() != cudaSuccess ||
          cudaMemcpy(&n, e->wbase + e->ws.slab_flag + 4, 4, cudaMemcpyDeviceToHost) != cudaSuccess)
        return C2V_ERR_CUDA;
      *value = n;
    }
    return C2V_OK;
  }
  if (!strcmp(key, "recompute_logits")) { *value = e->recompute; return C2V_OK; }
  if (!strcmp(key, "sort_peer_access")) { *value = e->sort_peer; return C2V_OK; }
  if (!strcmp(key, "adam_step_count")) { *value = e->adam_t_done; return C2V_OK; }
  if (!strcmp(key, "target_adam_fused_step")) { *value = e->tgt_fused_t; return C2V_OK; }
  if (!strcmp(key, "early_catchup_count")) { *value = e->early_count; return C2V_OK; }
  return C2V_ERR_INVALID;
}

int c2v_forward(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt, const float* mask,
                int32_t B, float* code_vec, float* attn, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!src || !path || !tgt || !mask || !code_vec) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  const Dropout dp = make_dropout(e->dims, 1.0f, 0, 0, nullptr);
  return forward_impl(e, (cudaStream_t)stream, src, path, tgt, mask, B, dp, code_vec, attn);
}

int c2v_topk(c2v_engine* e, const float* code_vec, int32_t B, int32_t* idx, float* val, int32_t normalize,
             void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!code_vec || !idx || !val) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  return topk_impl(e, (cudaStream_t)stream, code_vec, B, idx, val, normalize);
}

size_t c2v_nearest_scratch_bytes(int64_t rows, int32_t n, int32_t k) {
  if (rows < 1 || rows > INT32_MAX || n < 1 || k < 1 || k > sim::kMaxK) return 0;
  return (size_t)n * (size_t)sim::slices_for(rows) * (size_t)k * sizeof(ValIdx);
}

int c2v_compose_queries(c2v_engine* e, const float* bank, int64_t rows, int32_t dim, const int32_t* term_rows,
                        const float* term_weights, const float* term_vectors, int32_t n, int32_t max_terms,
                        float* queries, void* stream) {
  if (!e) return C2V_ERR_INVALID;
  int rc = check_bank(e, bank, rows, dim);
  if (rc) return rc;
  if (!term_rows || !term_weights || !queries) return fail(e, C2V_ERR_INVALID, "NULL argument");
  if (n < 1) return fail(e, C2V_ERR_INVALID, "n must be >= 1");
  if (max_terms < 1 || max_terms > sim::kMaxTerms) return fail(e, C2V_ERR_INVALID, "max_terms must be in [1, 16]");
  if (!aligned16(queries) || (term_vectors && !aligned16(term_vectors)))
    return fail(e, C2V_ERR_INVALID, "queries / term_vectors must be 16-byte aligned");
  C2V_CUDA(e, cudaSetDevice(e->device));
  C2V_LAUNCH(e, (sim::compose_kernel<<<n, sim::kThreads, 0, (cudaStream_t)stream>>>(bank, rows, dim, term_rows, term_weights,
                                                                                     term_vectors, max_terms, queries)));
  return C2V_OK;
}

int c2v_nearest(c2v_engine* e, const float* bank, int64_t rows, int32_t dim, const float* queries, int32_t n, int32_t k,
                const int32_t* exclude, int32_t n_exclude, int32_t* idx, float* val, void* scratch, size_t scratch_bytes,
                void* stream) {
  if (!e) return C2V_ERR_INVALID;
  int rc = check_bank(e, bank, rows, dim);
  if (rc) return rc;
  if (!queries || !idx || !val || !scratch) return fail(e, C2V_ERR_INVALID, "NULL argument");
  if (n < 1) return fail(e, C2V_ERR_INVALID, "n must be >= 1");
  if (k < 1 || k > sim::kMaxK) return fail(e, C2V_ERR_INVALID, "k must be in [1, 64]");
  if (n_exclude < 0 || n_exclude > sim::kMaxExclude) return fail(e, C2V_ERR_INVALID, "n_exclude must be in [0, 16]");
  if (n_exclude > 0 && !exclude) return fail(e, C2V_ERR_INVALID, "exclude is NULL with n_exclude > 0");
  if (!aligned16(queries)) return fail(e, C2V_ERR_INVALID, "queries must be 16-byte aligned");
  if (!aligned16(scratch)) return fail(e, C2V_ERR_INVALID, "scratch must be 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(idx) % 4 || reinterpret_cast<uintptr_t>(val) % 4)
    return fail(e, C2V_ERR_INVALID, "idx / val must be 4-byte aligned");
  if (scratch_bytes < c2v_nearest_scratch_bytes(rows, n, k))
    return fail(e, C2V_ERR_INVALID, "scratch smaller than c2v_nearest_scratch_bytes()");
  C2V_CUDA(e, cudaSetDevice(e->device));
  return nearest_impl(e, (cudaStream_t)stream, bank, (int)rows, dim, queries, n, k, exclude, n_exclude, idx, val, scratch);
}

int c2v_loss(c2v_engine* e, const float* code_vec, const int32_t* target, int32_t B, float* loss_out, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!code_vec || !target || !loss_out) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  float* S = wsp<float>(e, e->ws.S);
  const float invB = 1.0f / (float)B;
  const int Y = e->dims.target_vocab;
  const bool fused = is_tc(e) && (reinterpret_cast<uintptr_t>(code_vec) % 16 == 0);
  if ((rc = run_logits(e, st, code_vec, B, S, fused))) return rc;
  {
    PhaseTimer pt(e, PH_XENT, st);
    if (fused)      // the logits epilogue already folded each tile into (max, sum exp) partials
      C2V_LAUNCH(e, (xent_combine_kernel<<<B, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), 2 * ((Y + 255) / 256), S, e->ws.ldS, target,
                                                            wsp<float>(e, e->ws.loss_b), wsp<float>(e, e->ws.lse))));
    else
      C2V_LAUNCH(e, (xent_kernel<<<B, kXentThreads, 0, st>>>(S, e->ws.ldS, target, Y, invB, wsp<float>(e, e->ws.loss_b),
                                                              wsp<float>(e, e->ws.lse), 0)));
    C2V_LAUNCH(e, (loss_reduce_kernel<<<1, 256, 0, st>>>(wsp<float>(e, e->ws.loss_b), B, invB, loss_out)));
  }
  return C2V_OK;
}

int c2v_train_step(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt, const float* mask,
                   const int32_t* target, int32_t B, float keep_prob, uint64_t seed, uint64_t step,
                   const float* dropout_mask, float* loss_out, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!src || !path || !tgt || !mask || !target || !loss_out) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  return train_step_impl(e, (cudaStream_t)stream, src, path, tgt, mask, target, B, keep_prob, seed, step,
                         dropout_mask, loss_out);
}

int c2v_sampled_train_step(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt, const float* mask,
                           const int32_t* target, int32_t B, const int32_t* sampled, int32_t S, const float* logq_true,
                           const float* logq_sampled, float keep_prob, uint64_t seed, uint64_t step,
                           const float* dropout_mask, float* loss_out, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!src || !path || !tgt || !mask || !target || !sampled || !logq_true || !logq_sampled || !loss_out)
    return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  return sampled_train_step_impl(e, (cudaStream_t)stream, src, path, tgt, mask, target, B, sampled, S, logq_true,
                                 logq_sampled, keep_prob, seed, step, dropout_mask, loss_out);
}

int c2v_arm_target_adam(c2v_engine* e, float lr, float beta1, float beta2, float eps, int64_t t) {
  if (!e) return C2V_ERR_INVALID;
  if (!e->has_theta || !e->has_adam) return fail(e, C2V_ERR_STATE, "parameters / Adam state not bound");
  if (t < 1) return fail(e, C2V_ERR_INVALID, "Adam step count t must be >= 1");
  if (e->tgt_fused_t)
    return fail(e, C2V_ERR_STATE, "a fused target update is still unacknowledged: call c2v_adam_step (or clear target_adam_fused_step)");
  if (e->early_t) return fail(e, C2V_ERR_STATE, "the previous armed step is still unacknowledged: call c2v_adam_step");
  e->tgt_lr = lr; e->tgt_b1 = beta1; e->tgt_b2 = beta2; e->tgt_eps = eps; e->tgt_t = t;
  e->tgt_armed = true;
  e->armed_t = t;
  return C2V_OK;
}

int c2v_hint_next_batch(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt, int32_t B) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!src || !path || !tgt) return fail(e, C2V_ERR_INVALID, "NULL argument");
  e->hint_src = src; e->hint_pth = path; e->hint_tgt = tgt; e->hint_B = B;
  return C2V_OK;
}

int c2v_hint_next_batch_host(c2v_engine* e, const int32_t* h_src, const int32_t* h_path, const int32_t* h_tgt, int32_t B,
                             void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!h_src || !h_path || !h_tgt) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nb = (size_t)B * e->dims.max_contexts * 4;
  int32_t* src = wsp<int32_t>(e, e->ws.nx_src);
  int32_t* pth = wsp<int32_t>(e, e->ws.nx_pth);
  int32_t* tgt = wsp<int32_t>(e, e->ws.nx_tgt);
  C2V_CUDA(e, cudaMemcpyAsync(src, h_src, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(pth, h_path, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(tgt, h_tgt, nb, cudaMemcpyHostToDevice, st));
  return c2v_hint_next_batch(e, src, pth, tgt, B);
}

int c2v_adam_step(c2v_engine* e, float lr, float beta1, float beta2, float eps, int64_t t, void* stream) {
  if (!e) return C2V_ERR_INVALID;
  if (!e->has_theta) return fail(e, C2V_ERR_STATE, "parameters not bound");
  C2V_CUDA(e, cudaSetDevice(e->device));
  return adam_impl(e, (cudaStream_t)stream, lr, beta1, beta2, eps, t);
}

int c2v_bind_table_shards(c2v_engine* e, const c2v_table_shards* params, const c2v_table_shards* grads, float grad_scale) {
  if (!e) return C2V_ERR_INVALID;
  if (!params) return fail(e, C2V_ERR_INVALID, "params shards are NULL");
  if (!e->has_theta) return fail(e, C2V_ERR_STATE, "bind the replicated tensors first (c2v_bind_params)");
  const int w = params->world;
  if (!(w == 1 || w == 2 || w == 4 || w == 8)) return fail(e, C2V_ERR_INVALID, "world must be 1, 2, 4 or 8");
  if (grads && grads->world != w) return fail(e, C2V_ERR_INVALID, "params / grads world mismatch");
  int shift = 0;
  while ((1 << shift) < w) ++shift;
  auto fill = [&](ShardedTable& t, float* const* ptrs) -> bool {
    t = ShardedTable{};
    t.shift = shift; t.mask = w - 1;
    for (int i = 0; i < w; ++i) { if (!ptrs[i]) return false; t.base[i] = ptrs[i]; }
    return true;
  };
  if (!fill(e->th_tok, params->tok) || !fill(e->th_path, params->path)) return fail(e, C2V_ERR_INVALID, "NULL shard pointer");
  if (grads) {
    if (!fill(e->gr_tok, grads->tok) || !fill(e->gr_path, grads->path)) return fail(e, C2V_ERR_INVALID, "NULL shard pointer");
  }
  e->table_world = w;
  e->grad_scale = grad_scale;
  return C2V_OK;
}

size_t c2v_scatter_inbox_bytes(const c2v_dims* dims, int32_t world) {
  std::string why;
  if (!dims_ok(dims, &why) || world < 1 || world > kMaxShards) { g_create_error = why.empty() ? "bad world" : why; return 0; }
  const size_t cap = (size_t)3 * dims->max_batch * dims->max_contexts;
  return inbox_val_offset(world, cap) + (size_t)world * cap * dims->embed_dim * 4;
}

int c2v_bind_scatter_inbox(c2v_engine* e, void* const* inbox, int32_t world, int32_t rank) {
  if (!e) return C2V_ERR_INVALID;
  if (!inbox) { e->inbox = InboxSet{}; return C2V_OK; }           // unbind: back to remote red.add
  if (world != e->table_world || world < 2) return fail(e, C2V_ERR_STATE, "bind the table shards first (same world)");
  if (rank < 0 || rank >= world) return fail(e, C2V_ERR_INVALID, "rank out of range");
  InboxSet s{};
  for (int i = 0; i < world; ++i) {
    if (!inbox[i]) return fail(e, C2V_ERR_INVALID, "NULL inbox pointer");
    s.base[i] = (char*)inbox[i];
  }
  s.cap = (size_t)3 * e->dims.max_batch * e->dims.max_contexts;
  s.world = world; s.rank = rank;
  e->inbox = s;
  return C2V_OK;
}

int c2v_apply_scatter_inbox(c2v_engine* e, void* stream) {
  if (!e) return C2V_ERR_INVALID;
  if (e->inbox.world < 2) return fail(e, C2V_ERR_STATE, "no scatter inbox bound (c2v_bind_scatter_inbox)");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  PhaseTimer pt(e, PH_INBOX_APPLY, st);
  C2V_LAUNCH(e, (inbox_apply_kernel<<<e->num_sms * 8, 256, 0, st>>>(e->inbox, e->dims.embed_dim, e->gr_tok.base[e->inbox.rank],
                                                                    e->gr_path.base[e->inbox.rank])));
  return C2V_OK;
}

int c2v_ipc_alloc(int device, size_t bytes, void** dev_ptr, unsigned char* handle64) {
  if (!dev_ptr || !handle64 || bytes == 0) return fail(nullptr, C2V_ERR_INVALID, "bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  C2V_CUDA((c2v_engine*)nullptr, cudaSetDevice(device));
  C2V_CUDA((c2v_engine*)nullptr, cudaMalloc(dev_ptr, bytes));
  C2V_CUDA((c2v_engine*)nullptr, cudaMemset(*dev_ptr, 0, bytes));
  cudaIpcMemHandle_t h;
  C2V_CUDA((c2v_engine*)nullptr, cudaIpcGetMemHandle(&h, *dev_ptr));
  memcpy(handle64, &h, 64);
  return C2V_OK;
}

int c2v_ipc_open(int device, const unsigned char* handle64, void** dev_ptr) {
  if (!dev_ptr || !handle64) return fail(nullptr, C2V_ERR_INVALID, "bad argument");
  C2V_CUDA((c2v_engine*)nullptr, cudaSetDevice(device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  C2V_CUDA((c2v_engine*)nullptr, cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return C2V_OK;
}

int c2v_ipc_close(int device, void* dev_ptr) {
  C2V_CUDA((c2v_engine*)nullptr, cudaSetDevice(device));
  C2V_CUDA((c2v_engine*)nullptr, cudaIpcCloseMemHandle(dev_ptr));
  return C2V_OK;
}

int c2v_ipc_free(int device, void* dev_ptr) {
  C2V_CUDA((c2v_engine*)nullptr, cudaSetDevice(device));
  C2V_CUDA((c2v_engine*)nullptr, cudaFree(dev_ptr));
  return C2V_OK;
}

// ---- phase-split training step: the fully sharded schedule (target table row-sharded too) ------------
int c2v_context_forward(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt, const float* mask,
                        int32_t B, float keep_prob, uint64_t seed, uint64_t step, const float* dropout_mask,
                        float* code_vec, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!src || !path || !tgt || !mask || !code_vec) return fail(e, C2V_ERR_INVALID, "NULL argument");
  if (!(keep_prob > 0.f) || keep_prob > 1.f) return fail(e, C2V_ERR_INVALID, "keep_prob must be in (0, 1]");
  C2V_CUDA(e, cudaSetDevice(e->device));
  const Dropout dp = make_dropout(e->dims, keep_prob, seed, step, dropout_mask);
  return forward_impl(e, (cudaStream_t)stream, src, path, tgt, mask, B, dp, code_vec, wsp<float>(e, e->ws.alpha), true);
}

int c2v_target_forward(c2v_engine* e, const float* code_all, int32_t Bt, const int32_t* target, int32_t row_offset,
                       float* row_max, float* row_sum, float* true_logit, void* stream) {
  int rc = check_batch(e, Bt);
  if (rc) return rc;
  if (!code_all || !target || !row_max || !row_sum || !true_logit) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  float* S = wsp<float>(e, e->ws.S);
  const int Y = e->dims.target_vocab;
  const bool fused = (is_tc(e)) && (reinterpret_cast<uintptr_t>(code_all) % 16 == 0);
  const int n_tiles = 2 * ((Y + 255) / 256);
  e->slab_exp_live = false;
  if (fused && e->exp_slab && !e->fuse_sg && e->has_grad) {
    // deferred normalisation over a row-sharded table: (c_b, sum U) stand in for (row max, sum exp) in the cross-rank combine
    float* tl = wsp<float>(e, e->ws.true_logit);
    int* flag = wsp<int>(e, e->ws.slab_flag);
    if (!e->slab_flag_zeroed) {
      C2V_CUDA(e, cudaMemsetAsync(flag, 0, 64, st));
      e->slab_flag_zeroed = true;
    }
    if ((rc = end_target_lazy(e, st))) return rc;
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (true_logit_kernel<<<(Bt + 7) / 8, 256, 0, st>>>(code_all, e->theta.tgt, target, row_offset, Y, e->dims.code_dim, Bt, tl, flag)));
      C2V_CUDA(e, cudaMemcpyAsync(true_logit, tl, (size_t)Bt * 4, cudaMemcpyDeviceToDevice, st));
    }
    if ((rc = run_logits(e, st, code_all, Bt, S, false, false, nullptr, tl))) return rc;
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (expsum_rows_kernel<<<Bt, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), n_tiles, tl, row_max, row_sum, flag)));
    }
    // a row left the fp32 window: the statistics that go to the other ranks are redone the classic way (gated, usually a no-op)
    if ((rc = run_logits(e, st, code_all, Bt, S, true, false, nullptr, nullptr, flag))) return rc;
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (row_maxsum_kernel<<<Bt, 256, 0, st>>>(wsp<float2>(e, e->ws.lse_part), n_tiles, S, e->ws.ldS, Y, target, row_offset, row_max,
                                                           row_sum, true_logit, 1, flag)));
    }
    e->slab_exp_live = true;
    return C2V_OK;
  }
  if ((rc = run_logits(e, st, code_all, Bt, S, fused))) return rc;
  PhaseTimer pt(e, PH_XENT, st);
  C2V_LAUNCH(e, (row_maxsum_kernel<<<Bt, 256, 0, st>>>(fused ? wsp<float2>(e, e->ws.lse_part) : nullptr, n_tiles, S, e->ws.ldS, Y, target,
                                                       row_offset, row_max, row_sum, true_logit)));
  return C2V_OK;
}

int c2v_lse_combine(c2v_engine* e, const float* maxes, const float* sums, int32_t world, int32_t Bt, const float* true_logit,
                    float inv_batch, float* lse_out, float* loss_out, void* stream) {
  if (!e || !maxes || !sums || !true_logit || !lse_out || !loss_out) return C2V_ERR_INVALID;
  if (Bt < 1 || Bt > e->dims.max_batch || world < 1) return fail(e, C2V_ERR_INVALID, "bad size");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  float* loss_b = wsp<float>(e, e->ws.loss_b);
  C2V_LAUNCH(e, (lse_combine_kernel<<<(Bt + 255) / 256, 256, 0, st>>>(maxes, sums, world, Bt, true_logit, lse_out, loss_b)));
  C2V_LAUNCH(e, (loss_reduce_kernel<<<1, 256, 0, st>>>(loss_b, Bt, inv_batch, loss_out)));
  return C2V_OK;
}

int c2v_target_backward(c2v_engine* e, const float* code_all, int32_t Bt, const float* lse, const int32_t* target,
                        int32_t row_offset, float inv_batch, float* dv_partial, void* stream) {
  int rc = check_batch(e, Bt);
  if (rc) return rc;
  if (!code_all || !lse || !target || !dv_partial) return fail(e, C2V_ERR_INVALID, "NULL argument");
  if (!e->has_grad) return fail(e, C2V_ERR_STATE, "gradients not bound (c2v_bind_grads)");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  float* S = wsp<float>(e, e->ws.S);
  if (e->slab_exp_live) {
    // the slab holds U = exp(s - c_b): patch the true-class elements, hand the rows' factors to the two GEMMs
    e->slab_exp_live = false;
    e->sg_live = false;
    const int Y = e->dims.target_vocab, D = e->dims.code_dim;
    float* tl = wsp<float>(e, e->ws.true_logit);
    float* rscale = wsp<float>(e, e->ws.rscale);
    float* vs = wsp<float>(e, e->ws.v_scaled);
    int* flag = wsp<int>(e, e->ws.slab_flag);
    float* S_lo = is_3x(e) ? wsp<float>(e, e->ws.S_lo) : nullptr;
    {
      PhaseTimer pt(e, PH_XENT, st);
      C2V_LAUNCH(e, (expsum_finish_kernel<<<(Bt + 255) / 256, 256, 0, st>>>(S, S_lo, e->ws.ldS, Y, target, row_offset, tl, lse, inv_batch, Bt, rscale, flag)));
    }
    // fallback (gated): logits again, then the classic rewrite with the global log-sum-exp; the rows' factors become 1
    if ((rc = run_logits(e, st, code_all, Bt, S, true, false, nullptr, nullptr, flag))) return rc;
    {
      PhaseTimer pt(e, PH_XENT, st);
      if (S_lo) C2V_LAUNCH(e, (softmax_grad_kernel<true><<<dim3(2, Bt), 256, 0, st>>>(S, e->ws.ldS, Y, lse, target, inv_batch, row_offset, S_lo, flag, rscale,
                                                                                    reinterpret_cast<unsigned*>(flag) + 1)));
      else C2V_LAUNCH(e, (softmax_grad_kernel<false><<<dim3(2, Bt), 256, 0, st>>>(S, e->ws.ldS, Y, lse, target, inv_batch, row_offset, nullptr, flag, rscale,
                                                                                 reinterpret_cast<unsigned*>(flag) + 1)));
      C2V_LAUNCH(e, (scale_rows_kernel<<<(unsigned)(((size_t)Bt * D + 255) / 256), 256, 0, st>>>(code_all, rscale, vs, D, (size_t)Bt * D)));
    }
    e->row_scale = rscale;
    rc = target_grad_gemms(e, st, vs, Bt, dv_partial);
    e->row_scale = nullptr;
    return rc;
  }
  {
    PhaseTimer pt(e, PH_XENT, st);
    const int chunks = (int)((e->ws.ldS / 4 + 256 * 8 - 1) / (256 * 8));
    e->sg_live = false;
    if (is_3x(e))
      C2V_LAUNCH(e, (softmax_grad_kernel<true><<<dim3(chunks, Bt), 256, 0, st>>>(S, e->ws.ldS, e->dims.target_vocab, lse, target, inv_batch,
                                                                               row_offset, wsp<float>(e, e->ws.S_lo))));
    else if (is_tc(e) && e->fuse_sg) {
      e->sg = umma::SoftmaxGradArgs{lse, target, row_offset, inv_batch};
      e->sg_live = true;
    } else
      C2V_LAUNCH(e, (softmax_grad_kernel<false><<<dim3(chunks, Bt), 256, 0, st>>>(S, e->ws.ldS, e->dims.target_vocab, lse, target, inv_batch,
                                                                                row_offset, nullptr)));
  }
  return target_grad_gemms(e, st, code_all, Bt, dv_partial);
}

int c2v_context_backward(c2v_engine* e, const int32_t* src, const int32_t* path, const int32_t* tgt, const float* mask,
                         int32_t B, float keep_prob, uint64_t seed, uint64_t step, const float* dropout_mask,
                         const float* dv, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!src || !path || !tgt || !mask || !dv) return fail(e, C2V_ERR_INVALID, "NULL argument");
  if (!e->has_grad) return fail(e, C2V_ERR_STATE, "gradients not bound (c2v_bind_grads)");
  C2V_CUDA(e, cudaSetDevice(e->device));
  const Dropout dp = make_dropout(e->dims, keep_prob, seed, step, dropout_mask);
  ContextSource cs = make_source(e, src, path, tgt, B);
  return context_backward(e, (cudaStream_t)stream, cs, mask, B, dp, dv);
}

int c2v_sync_tables(c2v_engine* e, void* stream) {
  if (!e) return C2V_ERR_INVALID;
  C2V_CUDA(e, cudaSetDevice(e->device));
  return flush_rows(e, (cudaStream_t)stream);
}

int c2v_set_event(c2v_engine* e, const char* name, void* cuda_event) {
  if (!e || !name) return C2V_ERR_INVALID;
  if (!strcmp(name, "target_grads_ready")) { e->ev_tgt_ready = (cudaEvent_t)cuda_event; return C2V_OK; }
  return fail(e, C2V_ERR_INVALID, std::string("unknown event: ") + name);
}

int c2v_adam_step_range(c2v_engine* e, float* theta, float* grad, float* m, float* v, size_t count, float lr,
                        float beta1, float beta2, float eps, int64_t t, int32_t zero_grad, void* stream) {
  if (!e) return C2V_ERR_INVALID;
  if (!theta || !grad || !m || !v) return fail(e, C2V_ERR_INVALID, "NULL argument");
  if (count % 4 || ((uintptr_t)theta | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) % 16)
    return fail(e, C2V_ERR_INVALID, "slice must be a multiple of 4 floats and 16-byte aligned");
  if (t < 1) return fail(e, C2V_ERR_INVALID, "Adam step count t must be >= 1");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const float lr_t = (float)((double)lr * sqrt(1.0 - pow((double)beta2, (double)t)) / (1.0 - pow((double)beta1, (double)t)));
  const size_t n4 = count / 4;
  if (n4 == 0) return C2V_OK;
  size_t blocks = (n4 + 255) / 256;
  if (blocks > (size_t)e->num_sms * 16) blocks = (size_t)e->num_sms * 16;
  PhaseTimer pt(e, PH_ADAM, st);
  C2V_LAUNCH(e, (adam_kernel<<<(unsigned)blocks, 256, 0, st>>>(theta, grad, m, v, n4, lr_t, beta1, beta2, eps,
                                                               zero_grad ? 1 : 0)));
  return C2V_OK;
}

int c2v_train_batch_host(c2v_engine* e, const int32_t* h_src, const int32_t* h_path, const int32_t* h_tgt,
                         const float* h_mask, const int32_t* h_target, int32_t B, float keep_prob, uint64_t seed,
                         int64_t t, float lr, float beta1, float beta2, float eps, float* h_loss, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!h_src || !h_path || !h_tgt || !h_mask || !h_target || !h_loss) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nb = (size_t)B * e->dims.max_contexts * 4;
  int32_t* src = wsp<int32_t>(e, e->ws.st_src);
  int32_t* pth = wsp<int32_t>(e, e->ws.st_pth);
  int32_t* tgt = wsp<int32_t>(e, e->ws.st_tgt);
  float* mask = wsp<float>(e, e->ws.st_mask);
  int32_t* target = wsp<int32_t>(e, e->ws.st_target);
  float* loss = wsp<float>(e, e->ws.loss);
  C2V_CUDA(e, cudaMemcpyAsync(src, h_src, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(pth, h_path, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(tgt, h_tgt, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(mask, h_mask, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(target, h_target, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  if (e->fuse_tgt && (rc = c2v_arm_target_adam(e, lr, beta1, beta2, eps, t))) return rc;
  // the Adam step count doubles as the dropout stream position
  if ((rc = train_step_impl(e, st, src, pth, tgt, mask, target, B, keep_prob, seed, (uint64_t)t, nullptr, loss))) return rc;
  if ((rc = adam_impl(e, st, lr, beta1, beta2, eps, t))) return rc;
  C2V_CUDA(e, cudaMemcpyAsync(h_loss, loss, 4, cudaMemcpyDeviceToHost, st));
  C2V_CUDA(e, cudaStreamSynchronize(st));
  return C2V_OK;
}

int c2v_train_batch_async(c2v_engine* e, const int32_t* h_src, const int32_t* h_path, const int32_t* h_tgt, const float* h_mask,
                          const int32_t* h_target, int32_t B, float keep_prob, uint64_t seed, int64_t t, float lr, float beta1,
                          float beta2, float eps, float* h_loss, void* upload_done_event, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!h_src || !h_path || !h_tgt || !h_mask || !h_target || !h_loss) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int i = (int)(e->async_n++ & 1);
  const size_t nb = (size_t)B * e->dims.max_contexts * 4;
  int32_t* src = wsp<int32_t>(e, i ? e->ws.sb_src : e->ws.st_src);
  int32_t* pth = wsp<int32_t>(e, i ? e->ws.sb_pth : e->ws.st_pth);
  int32_t* tgt = wsp<int32_t>(e, i ? e->ws.sb_tgt : e->ws.st_tgt);
  float* mask = wsp<float>(e, i ? e->ws.sb_mask : e->ws.st_mask);
  int32_t* target = wsp<int32_t>(e, i ? e->ws.sb_target : e->ws.st_target);
  float* loss = wsp<float>(e, e->ws.loss) + 1 + i;          // one device slot per buffer: the previous step's read-back may be in flight
  // upload on the copy stream, behind the step that last read this staging set; the step waits for the upload only
  if (e->used_valid[i]) C2V_CUDA(e, cudaStreamWaitEvent(e->copy, e->ev_used[i], 0));
  C2V_CUDA(e, cudaMemcpyAsync(src, h_src, nb, cudaMemcpyHostToDevice, e->copy));
  C2V_CUDA(e, cudaMemcpyAsync(pth, h_path, nb, cudaMemcpyHostToDevice, e->copy));
  C2V_CUDA(e, cudaMemcpyAsync(tgt, h_tgt, nb, cudaMemcpyHostToDevice, e->copy));
  C2V_CUDA(e, cudaMemcpyAsync(mask, h_mask, nb, cudaMemcpyHostToDevice, e->copy));
  C2V_CUDA(e, cudaMemcpyAsync(target, h_target, (size_t)B * 4, cudaMemcpyHostToDevice, e->copy));
  C2V_CUDA(e, cudaEventRecord(e->ev_h2d[i], e->copy));
  if (upload_done_event) C2V_CUDA(e, cudaEventRecord((cudaEvent_t)upload_done_event, e->copy));
  C2V_CUDA(e, cudaStreamWaitEvent(st, e->ev_h2d[i], 0));
  if (e->fuse_tgt && (rc = c2v_arm_target_adam(e, lr, beta1, beta2, eps, t))) return rc;
  if ((rc = train_step_impl(e, st, src, pth, tgt, mask, target, B, keep_prob, seed, (uint64_t)t, nullptr, loss))) return rc;
  if ((rc = adam_impl(e, st, lr, beta1, beta2, eps, t))) return rc;
  C2V_CUDA(e, cudaMemcpyAsync(h_loss, loss, 4, cudaMemcpyDeviceToHost, st));
  C2V_CUDA(e, cudaEventRecord(e->ev_used[i], st));
  e->used_valid[i] = true;
  return C2V_OK;
}

int c2v_predict_batch_host(c2v_engine* e, const int32_t* h_src, const int32_t* h_path, const int32_t* h_tgt,
                           const float* h_mask, int32_t B, int32_t normalize, int32_t* h_topk_idx, float* h_topk_val,
                           float* h_code_vec, float* h_attn, void* stream) {
  int rc = check_batch(e, B);
  if (rc) return rc;
  if (!h_src || !h_path || !h_tgt || !h_mask || !h_topk_idx || !h_topk_val) return fail(e, C2V_ERR_INVALID, "NULL argument");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nb = (size_t)B * e->dims.max_contexts * 4;
  int32_t* src = wsp<int32_t>(e, e->ws.st_src);
  int32_t* pth = wsp<int32_t>(e, e->ws.st_pth);
  int32_t* tgt = wsp<int32_t>(e, e->ws.st_tgt);
  float* mask = wsp<float>(e, e->ws.st_mask);
  float* code = wsp<float>(e, e->ws.st_code);
  float* attn = wsp<float>(e, e->ws.st_attn);
  int32_t* tki = wsp<int32_t>(e, e->ws.st_topk_idx);
  float* tkv = wsp<float>(e, e->ws.st_topk_val);
  C2V_CUDA(e, cudaMemcpyAsync(src, h_src, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(pth, h_path, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(tgt, h_tgt, nb, cudaMemcpyHostToDevice, st));
  C2V_CUDA(e, cudaMemcpyAsync(mask, h_mask, nb, cudaMemcpyHostToDevice, st));
  const Dropout dp = make_dropout(e->dims, 1.0f, 0, 0, nullptr);
  if ((rc = forward_impl(e, st, src, pth, tgt, mask, B, dp, code, attn))) return rc;
  if ((rc = topk_impl(e, st, code, B, tki, tkv, normalize))) return rc;
  const int Y = e->dims.target_vocab;
  const int k = e->dims.top_k < Y ? e->dims.top_k : Y;
  C2V_CUDA(e, cudaMemcpyAsync(h_topk_idx, tki, (size_t)B * k * 4, cudaMemcpyDeviceToHost, st));
  C2V_CUDA(e, cudaMemcpyAsync(h_topk_val, tkv, (size_t)B * k * 4, cudaMemcpyDeviceToHost, st));
  if (h_code_vec) C2V_CUDA(e, cudaMemcpyAsync(h_code_vec, code, (size_t)B * e->dims.code_dim * 4, cudaMemcpyDeviceToHost, st));
  if (h_attn) C2V_CUDA(e, cudaMemcpyAsync(h_attn, attn, nb, cudaMemcpyDeviceToHost, st));
  C2V_CUDA(e, cudaStreamSynchronize(st));
  return C2V_OK;
}

int c2v_selftest_gemm(c2v_engine* e, int32_t a_mn, int32_t b_mn, int32_t bn, int32_t M, int32_t N, int32_t K,
                      int32_t splits, const float* A, size_t lda, const float* Bm, size_t ldb, float* C, size_t ldc,
                      void* stream) {
  return c2v_selftest_gemm3(e, a_mn, b_mn, bn, M, N, K, splits, A, nullptr, lda, Bm, nullptr, ldb, C, ldc, stream);
}

int c2v_selftest_gemm3(c2v_engine* e, int32_t a_mn, int32_t b_mn, int32_t bn, int32_t M, int32_t N, int32_t K,
                       int32_t splits, const float* A, const float* A_lo, size_t lda, const float* Bm, const float* B_lo,
                       size_t ldb, float* C, size_t ldc, void* stream) {
  if (!e || !A || !Bm || !C) return C2V_ERR_INVALID;
  if ((A_lo != nullptr) != (B_lo != nullptr)) return fail(e, C2V_ERR_INVALID, "3xTF32 needs the low parts of both operands");
  C2V_CUDA(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  umma::Operand opA{A, lda, a_mn != 0, A_lo};
  umma::Operand opB{Bm, ldb, b_mn != 0, B_lo};
  if (!umma::operand_ok(opA) || !umma::operand_ok(opB)) return fail(e, C2V_ERR_INVALID, "operand not TMA-compatible");
  umma::EpiStore ep{C, ldc, (size_t)M * ldc};
  if (bn == 256) C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_256(st, M, N, K, splits, opA, opB, ep, e->num_sms))));
  else if (bn == 192) C2V_LAUNCH(e, C2V_CUDA(e, (C2V_UMMA_192(st, M, N, K, splits, opA, opB, ep, e->num_sms))));
  else return fail(e, C2V_ERR_INVALID, "bn must be 192 or 256");
  return umma::effective_splits(K, splits);
}

int c2v_selftest_split(c2v_engine* e, const float* x, float* hi, float* lo, size_t count, void* stream) {
  if (!e || !x || !hi || !lo) return C2V_ERR_INVALID;
  if (count % 4 || ((uintptr_t)x | (uintptr_t)hi | (uintptr_t)lo) % 16) return fail(e, C2V_ERR_INVALID, "count % 4 and 16-byte alignment");
  C2V_CUDA(e, cudaSetDevice(e->device));
  size_t blocks = (count / 4 + 255) / 256;
  if (blocks > (size_t)e->num_sms * 16) blocks = (size_t)e->num_sms * 16;
  if (blocks < 1) blocks = 1;
  C2V_LAUNCH(e, (split_tf32_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, hi, lo, count / 4)));
  return C2V_OK;
}

int64_t c2v_launch_count(const c2v_engine* e) { return e ? e->launches : 0; }

int c2v_phase_count(void) { return PH_COUNT; }

const char* c2v_phase_name(int phase) { return (phase >= 0 && phase < PH_COUNT) ? kPhaseNames[phase] : ""; }

int c2v_phase_stats(c2v_engine* e, int phase, double* total_ms, int64_t* count, int reset) {
  if (!e || phase < 0 || phase >= PH_COUNT) return C2V_ERR_INVALID;
  C2V_CUDA(e, cudaSetDevice(e->device));
  PhaseLog& L = e->phase[phase];
  if (!L.pending.empty()) C2V_CUDA(e, cudaDeviceSynchronize());
  for (auto& ev : L.pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) { L.total_ms += ms; L.count++; }
    L.free_list.push_back(ev);
  }
  L.pending.clear();
  if (total_ms) *total_ms = L.total_ms;
  if (count) *count = L.count;
  if (reset) { L.total_ms = 0.0; L.count = 0; }
  return C2V_OK;
}

}  // extern "C"
