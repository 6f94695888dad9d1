#!/usr/bin/env python
"""bench.py -- path-contexts/sec of one code2vec train step (batch 1024 x 200, java14m shape).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA engine through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port of the reference
                                                             # graph on the box's host cores (TensorFlow
                                                             # itself is not installable here, see DESIGN.md)
    python bench.py --math 3xtf32        # the same step at fp32-equivalent accuracy on the tensor cores
    python bench.py --mode fwd_loss      # BASELINE configs[2]: forward + full-softmax loss only
    python bench.py --mode sampled       # BASELINE configs[3]: train step with sampled softmax (25 negatives)
    python bench.py --workload large     # BASELINE configs[4]'s model: 3M/2M vocab, d=256 (run it with --gpus 8)
    python bench.py --dump-outputs DIR   # also write what the last timed step computed to DIR/*.npy (see dump_outputs)

A "step" is one pass of the hot path over one batch of synthetic path-context bags: three
embedding gathers, tanh(x.W), masked softmax attention, full-softmax logits + loss, the whole
backward pass including the sparse embedding-gradient scatter-add, and the TF1-faithful dense Adam
update (tensorflow_model.py:80 `sess.run([optimizer, train_loss])`).  One JSON line on stdout.

Timing: W >= 3 warm-up steps, then exactly K steps bracketed by barrier + synchronize, CUDA events
on the launching stream, max over ranks.  No L2 flush is needed: each step streams > 9 GB of
parameter / optimizer state through a 126 MB L2 and cycles through distinct input batches.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json configs[1]: java14m shape (config.py:60-68; vocab + 1 special word)
WORKLOADS = {
    "java14m": dict(token_vocab=1301137, path_vocab=911418, target_vocab=261246, embed_dim=128, code_dim=384,
                    max_contexts=200, batch=1024),
    # BASELINE.json configs[4]: large-vocab stress (3M tokens / 2M paths + the special word, d = 256, D = 768);
    # the target vocabulary is java14m's (the config does not name one)
    "large": dict(token_vocab=3000001, path_vocab=2000001, target_vocab=261246, embed_dim=256, code_dim=768,
                  max_contexts=200, batch=1024),
    "tiny": dict(token_vocab=1001, path_vocab=501, target_vocab=1001, embed_dim=32, code_dim=96,
                 max_contexts=20, batch=64),
}
KEEP_PROB = 0.75      # config.py:69 DROPOUT_KEEP_RATE
NUM_SAMPLED = 25      # BASELINE.json configs[2]: "sampled_softmax (neg=25)"
NVLINK_PEER_GBS = 770.0   # measured peer copy per direction per GPU (/opt/skills/guides/B200_PROFILING.md)
N_BATCHES = 16        # distinct input batches the timed loop cycles through
REFERENCE_BUDGET_S = 240.0   # --impl reference: most CPU seconds the timed + warm-up steps may take
DUMP_TABLE_BYTES = 16 << 20  # --dump-outputs: most bytes written per embedding table (a seeded sample of its rows)


def workload_string(name, w, mode):
    step = {"train": "train step: full softmax, dropout keep 0.75, TF1 dense Adam",
            "fwd_loss": "forward + full-softmax loss (no backward)",
            "sampled": "train step: sampled softmax (25 log-uniform negatives), dropout keep 0.75, TF1 dense Adam"}[mode]
    return "%s-shape %s; T=%d P=%d Y=%d d=%d D=%d C=%d" % (name, step, w["token_vocab"], w["path_vocab"], w["target_vocab"],
                                                      w["embed_dim"], w["code_dim"], w["max_contexts"])


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return dict(hbm=float(j["hbm_gbs"]), tensor=float(j["bf16_tflops"]),
                        tensor_sustained=float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), source="measured")
        except Exception:
            pass
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback")


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0, period_ms=100):
        self.idx, self.period = gpu_index, period_ms
        self.proc, self.lines, self.thread = None, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for ln in self.proc.stdout:
                self.lines.append((time.time(), ln.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ts, ln in self.lines:
            if t0 is not None and not (t0 <= ts <= t1 + 0.2):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_batches(w, n_batches, seed, bags="full", zipf=False):
    """bags: "full" = every bag has all MAX_CONTEXTS valid contexts (the HBM worst case the roofline is judged on,
    SURVEY 8d); "normal" = n_b ~ clip(N(120, 60), 1, 200); "ragged" = n_b ~ U{1..C}.  zipf: Zipfian indices."""
    from code2vec_b200.synthetic import synthetic_batch
    return [synthetic_batch(w["token_vocab"], w["path_vocab"], w["target_vocab"], w["max_contexts"], w["batch"],
                            seed=seed + 7919 * i, full_bags=(bags == "full"), normal_bags=(bags == "normal"), zipf=zipf)
            for i in range(n_batches)]


def algorithmic_work(w, B, touched_rows=None, world=1, fused_target_adam=False, terms=1, remote_frac=0.0, sweep_period=0):
    """Per-step algorithmic FLOPs / bytes of each phase (SURVEY section 8d).

    adam: the dense TF1 update streams theta, m, v in and out = 24 B per parameter.  With the
    lazy-but-exact scheme (single GPU) only the rows the batch references are streamed, once: 32 B
    per element (theta, m, v and the deferred gradient, in and out) in the catch-up pass; the dense
    part is the target table (unless fused into dY), TRANSFORM and ATTENTION.  Under table sharding each rank updates 1/world of every table.
    fused_target_adam: the target table's update runs in the dY epilogue, so its 24 B/param move
    from "adam" to "dY", which then is HBM-bound (P^T read once + the update) rather than tensor-bound."""
    d, D, C, Y = w["embed_dim"], w["code_dim"], w["max_contexts"], w["target_vocab"]
    N = B * C
    emb = (w["token_vocab"] + w["path_vocab"]) * d
    rest = Y * D + 3 * d * D + D
    # tensor work is counted as the fp32 products of the reference (2*M*N*K); 3xTF32 issues three tf32 MMAs for each
    proj = 2.0 * N * 3 * d * D
    logit = 2.0 * B * D * Y
    if fused_target_adam:
        rest -= Y * D
    if touched_rows is not None:
        # lazy Adam: one pass over the batch's rows (theta, m, v, g in and out); the dense kernels keep the rest
        adam, catchup = 24.0 * rest, 32.0 * touched_rows * d
    else:
        adam, catchup = 24.0 * (emb + rest) / world, 0.0
    dy = ("hbm", 24.0 * Y * D + 4.0 * terms_bytes(terms) * B * Y) if fused_target_adam else ("tensor", logit)
    gather_bytes = N * (3 * d * 4 + 16)                # SURVEY 8d: table rows + indices + mask per context (read side only)
    if remote_frac > 0:
        # row-sharded tables: (world-1)/world of the rows cross NVLink -- that link, not HBM, bounds the two kernels
        gather = ("nvlink", remote_frac * 4.0 * N * 3 * d)
        scatter = ("nvlink", remote_frac * 4.0 * N * 3 * d)
    else:
        gather = ("hbm", gather_bytes)
        scatter = ("hbm", 4.0 * N * 3 * d + 2 * 4.0 * N * 3 * d)     # dX' in, read-modify-write of the table rows
    sweep = ("hbm", 32.0 * emb / sweep_period) if sweep_period else ("hbm", 0.0)
    return {
        "gather": gather, "dx_scatter": scatter, "adam_sweep": sweep,
        "split": ("hbm", 12.0 * Y * D),                 # 3xTF32: the target table read once, (hi, lo) written
        "ctx_fwd": ("tensor", proj), "dW": ("tensor", proj), "dx_gemm": ("tensor", proj),
        "logits": ("tensor", logit), "dv": ("tensor", logit), "dY": dy,
        "adam": ("hbm", adam), "adam_catchup": ("hbm", catchup),
        "attn_fwd": ("hbm", 4.0 * N * D), "attn_bwd": ("hbm", 3 * 4.0 * N * D),
        "xent": ("hbm", 2 * 4.0 * B * Y),
    }


def terms_bytes(terms):
    """3xTF32 keeps the slab operand as two arrays (hi, lo)."""
    return 2 if terms == 3 else 1


def ncu_traffic():
    """DRAM bytes per launch measured by `ncu --set full` (profiles/r02_traffic.json, else round 1's), keyed by phase."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))
        except Exception:
            continue
    return {}


def sampled_inputs(w, batch, seed):
    """Per-batch inputs of the sampled-softmax step (SURVEY 8a A12): one shared set of NUM_SAMPLED log-uniform
    classes and the log expected counts of the true / sampled classes (tf.nn.sampled_softmax_loss defaults)."""
    Y = w["target_vocab"]
    rng = np.random.default_rng(seed)
    u = rng.random(NUM_SAMPLED)
    sampled = np.minimum((np.exp(u * np.log(Y + 1.0)) - 1.0).astype(np.int64), Y - 1).astype(np.int32)

    def logq(ids):
        ids = ids.astype(np.float64)
        p = (np.log(ids + 2.0) - np.log(ids + 1.0)) / np.log(Y + 1.0)
        return np.log(NUM_SAMPLED * p).astype(np.float32)
    return sampled, logq(batch[4]), logq(sampled)


def dump_outputs(out_dir, eng, mode, loss, code=None):
    """Writes what a caller of the timed step holds after its last step, as float32 DIR/<name>.npy: `loss` ([1]); for
    the train modes the parameters that step left behind (W and a whole; of tok, path and tgt the rows drawn by
    np.random.default_rng(0) without replacement, sorted, at most DUMP_TABLE_BYTES per table); for fwd_loss the code
    vectors `code` [B, D].  The inputs and the initialisation are seeded, so two builds run with the same arguments can
    be compared array for array."""
    import torch
    out = {"loss": loss}
    if mode == "fwd_loss":
        out["code"] = code
    else:
        eng.sync_tables()                # lazy Adam: bring every deferred row up to date before it is read
        for k in ("tok", "path", "tgt", "W", "a"):
            p = eng.params[k]
            if k in ("W", "a"):
                out[k] = p
                continue
            n, row_bytes = p.shape[0], p.shape[1] * 4
            rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_TABLE_BYTES // row_bytes), replace=False))
            out[k] = p.index_select(0, torch.from_numpy(rows).to(p.device))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ================================ our arm ========================================================
def run_ours(args):
    import torch
    import torch.distributed as dist
    from code2vec_b200.engine import MATH_MODES, EngineDims, PathAttentionEngine
    from code2vec_b200.trainer import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", local_rank)
    mode = args.mode
    if world > 1 and mode != "train":
        raise SystemExit("--mode %s is a single-GPU workload (BASELINE configs[1]/[2])" % mode)
    if world > 1 and args.dump_outputs:
        raise SystemExit("--dump-outputs is single-GPU (the multi-GPU schedules keep the tables in row shards)")

    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w["batch"] = args.batch
    B, C = w["batch"], w["max_contexts"]
    gdims = EngineDims(w["token_vocab"], w["path_vocab"], w["target_vocab"], w["embed_dim"], w["code_dim"], C, B, 10)
    if world not in (2, 4, 8) and args.dp_schedule in ("fully_sharded", "table_sharded"):
        args.dp_schedule = "sharded"              # peer-memory table sharding needs a power-of-two world <= 8
    if world > 1 and args.dp_schedule == "fully_sharded":
        from code2vec_b200.trainer import make_fully_sharded_engine
        eng = make_fully_sharded_engine(gdims, B, device=local_rank)
    else:
        eng = PathAttentionEngine(gdims, device=local_rank, training=(mode != "fwd_loss"))
    eng.init_params(seed=4321)                       # replicated: same seed on every rank
    eng.set_option("math_mode", MATH_MODES[args.math])
    eng.set_option("cta_pair", args.cta_pair)
    if args.no_sort_peer:
        eng.set_option("sort_peer_access", 0)
    if args.fuse_gather:
        eng.set_option("fuse_gather", 1)
    if args.fuse_softmax_grad:
        eng.set_option("fuse_softmax_grad", 1)
    if args.recompute_logits >= 0:
        eng.set_option("recompute_logits", args.recompute_logits)
    if args.no_exp_slab:
        eng.set_option("exp_slab", 0)
    if args.adam_prefetch:
        eng.set_option("adam_epilogue_prefetch", 1)
    trainer = None
    if mode != "fwd_loss":
        trainer = Trainer(eng, keep_prob=KEEP_PROB, seed=99, schedule=args.dp_schedule, fuse_target_adam=not args.no_fuse_adam,
                          lazy_adam=not args.no_lazy_adam, push_grads=args.push_grads)
        if args.dy_late >= 0:
            eng.set_option("dy_late", args.dy_late)
        if args.adam_rows_occ:
            eng.set_option("adam_rows_occupancy", args.adam_rows_occ)
        if args.sweep_period >= 0:
            eng.set_option("adam_sweep_period", args.sweep_period)
    schedule = trainer.schedule if trainer else "single"
    # a training loop knows its next batch (the reader prefetches); --hint passes it on so lazy Adam can run ahead
    n_batches = N_BATCHES
    nxt = (lambda seq, i: seq[(i + 1) % n_batches]) if (args.hint and mode == "train") else (lambda seq, i: None)
    host = make_batches(w, n_batches, seed=1234 + 100003 * rank, bags=args.bags, zipf=args.zipf)
    if mode == "sampled":
        host = [tuple(b) + sampled_inputs(w, b, seed=77 + i) for i, b in enumerate(host)]
    pinned = [[torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in b] for b in host]
    devb = [[t.to(dev) for t in b] for b in pinned]
    stage = [torch.empty_like(t, device=dev) for t in pinned[0]]      # e2e: this step's inputs are copied here
    last_code = [None]                                                  # fwd_loss: the code vectors of the latest step

    def step_dev(i):
        b = devb[i % n_batches]
        if mode == "train":
            return trainer.step_device(*b, next_batch=nxt(devb, i))
        if mode == "sampled":
            return trainer.step_device_sampled(*b)
        code, _ = eng.forward(b[0], b[1], b[2], b[3], want_attention=False)
        last_code[0] = code
        return eng.loss(code, b[4])

    loss_pin = torch.zeros(1, dtype=torch.float32).pin_memory()
    loss_hist = torch.zeros(max(args.steps, 16) + 8, dtype=torch.float32).pin_memory()

    def step_e2e(i):
        """The user-facing call with HOST buffers: pinned host -> device copies of this step's inputs, the step, and
        the loss read back -- all inside the timed region."""
        b = pinned[i % n_batches]
        if mode == "train" and world == 1 and not args.sync_e2e:
            # what Code2VecModel.train() calls per batch: c2v_train_batch_async -- this step's host -> device copies (engine copy
            # stream), the step, and the loss copied back into pinned host memory; the host does not wait per step (the timed
            # region ends with a synchronize, after which all K losses are on the host)
            eng.train_batch_async(*b[:5], rows=B, loss_out=loss_hist[i % loss_hist.numel():i % loss_hist.numel() + 1], keep=KEEP_PROB,
                                  seed=trainer.seed, **trainer.adam)
            return None
        if mode == "train":
            return trainer.step_host(*b, next_batch=nxt(pinned, i))     # c2v_train_batch_host (copies inside the C call, waits for the loss)
        for dst, src_t in zip(stage, b):
            dst.copy_(src_t, non_blocking=True)
        if mode == "sampled":
            l = trainer.step_device_sampled(*stage)
        else:
            code, _ = eng.forward(stage[0], stage[1], stage[2], stage[3], want_attention=False)
            l = eng.loss(code, stage[4])
        loss_pin.copy_(l, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return float(loss_pin[0])

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, K, W):
        for i in range(W):
            fn(i)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for i in range(K):
            out = fn(W + i)
        e1.record()
        sync_all()
        return e0.elapsed_time(e1), out

    # ---- device-resident timing (value) ---------------------------------------------------
    W, K = max(args.warmup, 3), args.steps
    for i in range(W):
        step_dev(i)
    sync_all()
    eng.set_option("profile", 1)
    eng.phase_stats(reset=True)
    clocks = ClockSampler(local_rank, period_ms=20)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    sync_all()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record()
    for i in range(K):
        loss_dev = step_dev(W + i)
    ev1.record()
    sync_all()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - launches0
    phases = eng.phase_stats(reset=True)
    eng.set_option("profile", 0)
    clk = clocks.stop(t_wall0, t_wall1) if rank == 0 else None
    last_loss = float(loss_dev.cpu()[0])
    if args.dump_outputs:
        # before the e2e and 3xTF32 passes below train the model further
        dump_outputs(args.dump_outputs, eng, mode, loss_dev, last_code[0])

    # ---- end to end through the host-buffer API (e2e) ---------------------------------------
    ms_e2e, _ = timed(step_e2e, K, 2)

    # ---- the same step at fp32-equivalent accuracy (3xTF32), when the headline ran plain tf32 --------------
    fp32_eq = None
    if args.math == "tf32" and world == 1 and not args.no_fp32_equivalent:
        eng.set_option("math_mode", MATH_MODES["3xtf32"])
        k3 = max(3, min(K, 10))
        ms3, l3 = timed(step_dev, k3, 3)
        ms3e, _ = timed(step_e2e, k3, 1)
        fp32_eq = {"math_mode": "3xtf32", "dtype": "fp32-equivalent: tf32 (hi, lo) operand splits, 3 tcgen05 MMAs per product, fp32 accumulate",
                   "value": round(B * C * k3 / (ms3 * 1e-3), 1), "e2e_value": round(B * C * k3 / (ms3e * 1e-3), 1),
                   "unit": "path-contexts/s", "ms_per_step": round(ms3 / k3, 4), "steps": k3,
                   "last_loss": round(float(l3.cpu()[0]), 5)}
        eng.set_option("math_mode", MATH_MODES[args.math])

    if world > 1:
        t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    contexts = float(world) * B * C * K
    value = contexts / (ms * 1e-3)
    e2e_value = contexts / (ms_e2e * 1e-3)
    peaks = _peaks()
    touched = None
    lazy_on = bool(trainer) and schedule == "single" and bool(eng.get_option("lazy_adam"))
    if lazy_on:
        touched = float(np.mean([len(np.unique(np.concatenate([b[0].ravel(), b[2].ravel()]))) + len(np.unique(b[1]))
                                 for b in host]))
    tc = args.math != "fp32"
    fused = bool(getattr(trainer, "fuse_tgt", False)) and tc and mode == "train"
    sharded_tables = schedule in ("table_sharded", "fully_sharded")
    work = algorithmic_work(w, B * (world if schedule == "fully_sharded" else 1), touched_rows=touched,
                            world=world if sharded_tables else 1, fused_target_adam=fused,
                            terms=3 if args.math == "3xtf32" else 1,
                            remote_frac=(world - 1.0) / world if sharded_tables else 0.0,
                            sweep_period=int(eng.get_option("adam_sweep_period")) if lazy_on else 0)
    if schedule == "fully_sharded":
        # each rank runs the context side on its own B bags and the target side on its 1/world of the classes for all world*B
        w_local = dict(w, target_vocab=(w["target_vocab"] + world - 1) // world)
        tgt_side = algorithmic_work(w_local, B * world, world=world, fused_target_adam=fused,
                                    terms=3 if args.math == "3xtf32" else 1)
        ctx_side = algorithmic_work(w, B, world=world, remote_frac=(world - 1.0) / world)
        work = dict(ctx_side, **{k: tgt_side[k] for k in ("logits", "dv", "dY", "xent", "split")})
        work["adam"] = ("hbm", 24.0 * ((w["token_vocab"] + w["path_vocab"]) * w["embed_dim"]) / world)
    slab_on = (mode == "train" and tc and bool(eng.get_option("exp_slab")) and not args.fuse_softmax_grad and
               (schedule == "fully_sharded" or args.recompute_logits <= 0))
    if slab_on:
        # deferred normalisation: no pass over the slab -- the phase is the true-class rows, the per-tile partials and the patches
        rows = B * (world if schedule == "fully_sharded" else 1)
        y_loc = (w["target_vocab"] + world - 1) // world if schedule == "fully_sharded" else w["target_vocab"]
        work["xent"] = ("hbm", 4.0 * rows * (w["code_dim"] * 3 + 2 * 2 * ((y_loc + 255) // 256) + 8))
    traffic = ncu_traffic()
    phase_out = {}
    dominant, dom_ms = None, -1.0
    for name, (tot_ms, n) in phases.items():
        avg = tot_ms / K                      # per step (a phase may be several launches)
        entry = {"ms": round(avg, 4), "share": round(tot_ms / ms, 4)}
        if name in work and work[name][1] > 0:
            kind, amount = work[name]
            if kind == "tensor":
                entry["tflops"] = round(amount / (avg * 1e-3) / 1e12, 2)
            else:
                entry["gbs"] = round(amount / (avg * 1e-3) / 1e9, 1)
                if kind == "nvlink":
                    entry["link"] = "nvlink"
            if avg > dom_ms:
                dominant, dom_ms = name, avg
        phase_out[name] = entry

    def roofline_of(name, avg_ms):
        kind, amount = work[name]
        if kind == "tensor":
            ach = amount / (avg_ms * 1e-3) / 1e12
            peak = peaks["tensor_sustained"]
            return {"kernel": name, "bound": "tensor", "achieved": round(ach, 2), "peak": peak, "unit": "TFLOP/s",
                    "frac": round(ach / peak, 4), "traffic": traffic.get(name),
                    "peak_source": peaks["source"] + " bf16 dense (sustained); tcgen05 kind::tf32 peaks at half of it"
                                   + ("; FLOPs counted as the reference's fp32 products (each costs 3 tf32 MMAs)" if args.math == "3xtf32" else "")}
        ach = amount / (avg_ms * 1e-3) / 1e9
        if kind == "nvlink":
            return {"kernel": name, "bound": "nvlink", "achieved": round(ach, 1), "peak": NVLINK_PEER_GBS, "unit": "GB/s",
                    "frac": round(ach / NVLINK_PEER_GBS, 4), "traffic": None,
                    "peak_source": "measured peer copy per direction per GPU (B200_PROFILING.md); bytes = the rows that cross NVLink"}
        peak = peaks["hbm"]
        return {"kernel": name, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach / peak, 4), "traffic": traffic.get(name), "peak_source": peaks["source"] + " copy bandwidth"}

    roofline = roofline_of(dominant, dom_ms) if dominant else None
    # north_star's own yardstick, whatever the dominant kernel is: the embedding gather against the HBM roofline on
    # SURVEY 8d's bytes (table rows + indices + mask; the X' it writes is not counted as useful work)
    gather_roofline = None
    if "gather" in phase_out and "gather" in work:
        gather_roofline = roofline_of("gather", phase_out["gather"]["ms"])
    elif "ctx_fwd" in phase_out and "gather" in work:
        # fused gather -> projection kernel: the gather has no launch of its own.  Its bytes over the WHOLE fused kernel's
        # time (which also runs the projection GEMM and writes H) is a lower bound of the gather's bandwidth; "kernel_total"
        # counts everything the fused kernel moves (rows in; H out; X' out when training) against the same time.
        gather_roofline = roofline_of("gather", phase_out["ctx_fwd"]["ms"])
        if gather_roofline["bound"] == "hbm":
            N, D, d3 = B * C, w["code_dim"], 3 * w["embed_dim"]
            total = work["gather"][1] + 4.0 * N * D + (4.0 * N * d3 if mode != "fwd_loss" else 0.0)
            ach = total / (phase_out["ctx_fwd"]["ms"] * 1e-3) / 1e9
            gather_roofline.update({"kernel": "ctx_fused (gather + projection + tanh)", "lower_bound": True,
                                    "kernel_total": {"bytes": total, "achieved": round(ach, 1), "frac": round(ach / peaks["hbm"], 4)}})

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(w, host[0][:5], steps=1, threads=args.cpu_threads or None, mode=mode)

    h2d = sum(int(a.nbytes) for a in host[0])
    if world == 1 and args.hint and fused:
        h2d += sum(int(a.nbytes) for a in host[0][:3])      # the next batch's index arrays are copied once more as the hint
    dtype = {"tf32": "tf32 operands / fp32 accumulate+storage", "fp32": "f32",
             "3xtf32": "fp32-equivalent (3xTF32: tf32 hi/lo operand splits, fp32 accumulate+storage)"}[args.math]
    metric = {"train": "path-contexts/sec (train step, batch 1024x200)",
              "fwd_loss": "path-contexts/sec (forward + loss, batch 1024x200)",
              "sampled": "path-contexts/sec (sampled-softmax train step, batch 1024x200)"}[mode]
    out = {
        "metric": metric, "value": round(value, 1), "unit": "path-contexts/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(ms / K, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": dtype,
        "data": "synthetic",
        "config": {"workload": workload_string(args.workload, w, mode),
                   "batch_per_gpu": B, "global_batch": B * world, "contexts_per_example": C,
                   "parallelism": "dp%d (%s)" % (world, schedule) if world > 1 else "single",
                   "l2": "no flush: >9 GB of parameter/optimizer traffic per step and %d rotating input batches exceed the 126 MB L2" % n_batches,
                   "math_mode": args.math, "fused_target_adam": fused, "lazy_adam": lazy_on,
                   "adam_sweep_period": int(eng.get_option("adam_sweep_period")) if lazy_on else None,
                   "exp_slab": slab_on,
                   "exp_slab_fallbacks": int(eng.get_option("exp_slab_fallbacks")),
                   "next_batch_hint": bool(world == 1 and args.hint and fused), "last_loss": round(last_loss, 5),
                   "inputs": "%s bags, %s indices; all %d slots per example are counted in the metric" % (
                       args.bags, "zipf(1.2)" if args.zipf else "uniform", C),
                   "valid_context_fraction": round(float(np.mean([b[3].mean() for b in host])), 4)},
        "e2e": {"value": round(e2e_value, 1), "unit": "path-contexts/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / K, 4),
                "api": ("c2v_train_batch_async (pinned host buffers; copies on the engine's copy stream; loss to pinned memory every step)"
                        if (mode == "train" and world == 1 and not args.sync_e2e) else
                        "c2v_train_batch_host" if mode == "train" else "torch H2D + device entry points + loss read-back")},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": roofline,
        "gather_roofline": gather_roofline,
        "fp32_equivalent": fp32_eq,
        "phases": phase_out,
        "cpu_baseline": cpu,
    }
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


# ================================ CPU arm ========================================================
def default_cpu_threads():
    """Upper bound of the CPU arm's intra-op threads: every host core unless C2V_CPU_THREADS says otherwise."""
    return int(os.environ.get("C2V_CPU_THREADS", "0")) or os.cpu_count() or 1


def pick_cpu_threads(tr, batch, limit):
    """More threads are not always faster (two sockets x SMT: 128 threads ran the step at 9.0 s, 32 at 3.2 s on the
    GPU boxes' Xeons), so the CPU arm gets the best of {all, 1/2, 1/4, 1/8} of the host threads, probed with one
    step on a 64-example slice each (the dense Adam over all 383 M parameters is part of every probe)."""
    import torch
    src, pth, tgt, mask, target = (a[:64] for a in batch)
    cands = sorted({max(1, limit // d) for d in (1, 2, 4, 8)}, reverse=True)
    if limit <= 16 or len(cands) == 1:          # small hosts: every core helps, nothing to probe
        torch.set_num_threads(limit)
        return limit, {}
    timing = {}
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.time()
        tr.train_step(src, pth, tgt, mask, target, keep=1.0)
        timing[c] = round(time.time() - t0, 3)
    best = min(timing, key=timing.get)
    torch.set_num_threads(best)
    return best, timing


def cpu_step_fn(tr, w, batch, mode, extra=None):
    """One timed CPU step of `mode` on `batch` -> seconds."""
    src, pth, tgt, mask, target = batch[:5]
    rng = np.random.default_rng(0)

    def one():
        dm = None
        if mode != "fwd_loss":
            dm = (rng.random((src.shape[0] * src.shape[1], 3 * w["embed_dim"]), dtype=np.float32) < KEEP_PROB).astype(np.float32)
        t0 = time.time()
        if mode == "train":
            tr.train_step(src, pth, tgt, mask, target, keep=KEEP_PROB, dropout_mask=dm)
        elif mode == "sampled":
            tr.sampled_train_step(src, pth, tgt, mask, target, *extra, keep=KEEP_PROB, dropout_mask=dm)
        else:
            tr.forward_loss(src, pth, tgt, mask, target)
        return time.time() - t0
    return one


CPU_WHAT = {"train": "train step(s)", "fwd_loss": "forward + loss pass(es)", "sampled": "sampled-softmax train step(s)"}


def cpu_baseline(w, batch, steps=1, threads=None, mode="train"):
    """The oracle port of the reference graph (torch-CPU, all host threads): forward + backward +
    TF1 dense Adam on the same workload; `steps` full batches (bounded sample)."""
    import torch
    from oracle.path_attention_oracle import Dims, init_params
    from oracle.torch_crosscheck import TorchCpuTrainer
    cores = threads or default_cpu_threads()
    dims = Dims(w["token_vocab"], w["path_vocab"], w["target_vocab"], w["embed_dim"], w["code_dim"], w["max_contexts"])
    params = init_params(dims, seed=4321)
    tr = TorchCpuTrainer(params, threads=cores)
    probed = {}
    if not threads:
        _, probed = pick_cpu_threads(tr, batch[:5], cores)
    one = cpu_step_fn(tr, w, batch, mode, extra=sampled_inputs(w, batch, seed=77) if mode == "sampled" else None)
    sec = float(np.mean([one() for _ in range(steps)]))
    B, C = batch[0].shape
    return {"value": round(B * C / sec, 1), "unit": "path-contexts/s", "cores": int(torch.get_num_threads()), "kind": "port",
            "sample": "%d full %s of the same workload (B=%d x C=%d), torch-CPU restatement of "
                      "tensorflow_model.py:197-265%s; %.2f s/step%s" % (
                          steps, CPU_WHAT[mode], B, C, "" if mode == "fwd_loss" else " incl. dense Adam", sec,
                          "; threads = fastest of a 64-example probe %s (s)" % probed if probed else "")}


def run_reference(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    mode = args.mode
    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w["batch"] = args.batch
    K, W = args.steps, args.warmup
    # Exactly K timed steps after W warm-ups, as asked -- unless that would not end within minutes on this host
    # (REFERENCE_BUDGET_S of CPU work, judged from the first step): then fewer, and the line says how many.
    batch = make_batches(w, 1, seed=1234, bags=args.bags, zipf=args.zipf)[0]
    import torch
    from oracle.path_attention_oracle import Dims, init_params
    from oracle.torch_crosscheck import TorchCpuTrainer
    cores = args.cpu_threads or default_cpu_threads()
    dims = Dims(w["token_vocab"], w["path_vocab"], w["target_vocab"], w["embed_dim"], w["code_dim"], w["max_contexts"])
    tr = TorchCpuTrainer(init_params(dims, seed=4321), threads=cores)
    probed = {}
    if not args.cpu_threads:
        _, probed = pick_cpu_threads(tr, batch, cores)
    one = cpu_step_fn(tr, w, batch, mode, extra=sampled_inputs(w, batch, seed=77) if mode == "sampled" else None)
    first = one()                       # doubles as the first warm-up step
    k_eff, w_eff = K, max(W, 1)
    if first * (K + W) > REFERENCE_BUDGET_S:
        k_eff = max(1, min(K, int(REFERENCE_BUDGET_S / first) - 1))
        w_eff = 1
    for _ in range(w_eff - 1):
        one()
    times = [one() for _ in range(k_eff)]
    sec = float(np.mean(times))
    B, C = batch[0].shape
    value = B * C / sec
    sample = ("%d timed full-batch %s (asked: --steps %d) after %d warm-up, torch-CPU "
              "restatement of the reference graph (TensorFlow not installable here), %d threads%s" % (
                  k_eff, CPU_WHAT[mode], K, w_eff, torch.get_num_threads(),
                  " (fastest of a 64-example probe %s s)" % probed if probed else ""))
    metric = {"train": "path-contexts/sec (train step, batch 1024x200)",
              "fwd_loss": "path-contexts/sec (forward + loss, batch 1024x200)",
              "sampled": "path-contexts/sec (sampled-softmax train step, batch 1024x200)"}[mode]
    out = {"impl": "reference", "metric": metric, "value": round(value, 1),
           "unit": "path-contexts/s", "n_gpus": world, "steps": k_eff, "warmup": w_eff, "steps_requested": K,
           "warmup_requested": W, "ms_per_step": round(sec * 1e3, 2),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload_string(args.workload, w, mode),
                      "batch_per_gpu": B, "global_batch": B, "contexts_per_example": C, "parallelism": "cpu"},
           "cpu_baseline": {"value": round(value, 1), "unit": "path-contexts/s", "cores": int(torch.get_num_threads()),
                            "kind": "port", "sample": sample},
           "e2e": {"value": round(value, 1), "unit": "path-contexts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="java14m", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--math", default=os.environ.get("C2V_MATH", "tf32"), choices=["fp32", "tf32", "3xtf32"],
                    help="arithmetic of the GEMMs: fp32 = FFMA on the SIMT pipe, tf32 = tcgen05 kind::tf32 (default), "
                         "3xtf32 = tcgen05 at fp32-equivalent accuracy (hi/lo operand splits)")
    ap.add_argument("--mode", default="train", choices=["train", "fwd_loss", "sampled"],
                    help="train = BASELINE configs[1] (default); fwd_loss = configs[2] forward + full-softmax loss; "
                         "sampled = configs[3] train step with sampled softmax")
    ap.add_argument("--sync-e2e", action="store_true",
                    help="e2e through c2v_train_batch_host (waits for every step's loss) instead of c2v_train_batch_async")
    ap.add_argument("--no-fp32-equivalent", action="store_true", help="skip the extra 3xTF32 measurement of the default run")
    ap.add_argument("--push-grads", action="store_true",
                    help="row-sharded tables: inbox-based gradient push (c2v_bind_scatter_inbox) instead of remote red.global.add; "
                         "measured slower at 8 GPUs (4.62 vs 4.29 ms), off by default")
    ap.add_argument("--no-sort-peer", action="store_true", help="row-sharded tables: plain (unsorted) peer gather / scatter-add")
    ap.add_argument("--fuse-gather", action="store_true", help="engine option fuse_gather (ctx_fused.cuh)")
    ap.add_argument("--recompute-logits", type=int, default=-1, choices=[-1, 0, 1], help="engine option recompute_logits (-1 = default)")
    ap.add_argument("--adam-prefetch", action="store_true", help="engine option adam_epilogue_prefetch = 1 (measured slower)")
    ap.add_argument("--no-exp-slab", action="store_true", help="engine option exp_slab = 0: the two-pass softmax schedule (logits stored, then rewritten)")
    ap.add_argument("--fuse-softmax-grad", action="store_true", help="engine option fuse_softmax_grad (A-operand transform warps)")
    ap.add_argument("--no-lazy-adam", action="store_true", help="dense Adam over the embedding tables every step")
    ap.add_argument("--sweep-period", type=int, default=-1, help="engine option adam_sweep_period (-1 = default 32, 0 = off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU arm (0 = all host cores)")
    ap.add_argument("--dy-late", type=int, default=-1, choices=[-1, 0, 1, 2],
                    help="engine option dy_late (-1 = the schedule's default)")
    ap.add_argument("--adam-rows-occ", type=int, default=0, choices=[0, 4, 5], help="engine option adam_rows_occupancy (0 = default)")
    ap.add_argument("--hint", action="store_true",
                    help="hint the next batch to the engine (c2v_hint_next_batch); measured no gain on one GPU, off by default")
    ap.add_argument("--no-fuse-adam", action="store_true",
                    help="keep the target table's Adam update as a separate pass instead of the dY epilogue")
    ap.add_argument("--bags", default="full", choices=["full", "normal", "ragged"],
                    help="valid contexts per bag: full (default; worst case for HBM), normal ~N(120,60), ragged ~U{1..C}")
    ap.add_argument("--zipf", action="store_true", help="Zipfian instead of uniform indices (hot rows, L2 reuse)")
    ap.add_argument("--cta-pair", type=int, default=int(os.environ.get("C2V_CTA_PAIR", "2")),
                    help="tcgen05 GEMMs as CTA pairs (cta_group::2): 0 never, 1 always, 2 auto (default)")
    ap.add_argument("--dp-schedule", default=os.environ.get("C2V_DP_SCHEDULE", "fully_sharded"),
                    choices=["fully_sharded", "table_sharded", "sharded", "allreduce"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32, < 64 MB; "
                         "single GPU, our arm)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the CUDA engine computed (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
