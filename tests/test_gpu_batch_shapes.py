"""Parity at the batch sizes, attention widths and schedule options the other GPU tests never reach.

Batch sizes.  Training runs at B = 1024 and every epoch and evaluation ends with a short batch on an engine sized
for the largest one.  So these tests run batches past one 128-row tile of the logits GEMM (rows of m-tile > 0 and of
the peer CTA of a CTA pair land in their own partial slots, true logits and row factors), K tails and K = 1 in
dY = P^T.v, several dv split-K counts, several sampled-softmax chunks, the logits GEMM's n-fastest raster (few
classes, many rows), and they shrink B on one engine so that the workspace still holds the previous, larger
step's rows (S slab, log-sum-exp partials, v, row factors, true logits, split-K partials).

Widths.  The attention kernels are instantiated for NV = ceil(D / 128) in {1, 2, 3, 4, 6, 8}; D here covers
NV = 2, 4, 6 and 8 with and without a partial last 128-column slice, and d = 160 gives the lazy-Adam row replay a
partial second slice.  Top-k runs at k = 1, 16 (the last width of the register kernel), 17 (the first of the
iterative one), 64 (the largest) and k clamped to a 40-class vocabulary.

Options.  dy_late 0 / 2 (dY and the fused target Adam right after dv, on the caller's stream resp. a second engine
stream) and adam_epilogue_prefetch are checked bit for bit against the default schedule.

Tolerances are the per-mode constants of test_gpu_parity.py / test_gpu_tf32.py: fp32 FFMA (math 0) and 3xTF32
(math 2) -- loss 1e-4, gradients 5e-5, code vectors 2e-5, attention 2e-6; tf32 (math 1) -- gradients 1e-2, code
vectors 3e-3, attention 2e-3."""
import dataclasses

import numpy as np
import pytest

from oracle import path_attention_oracle as O
from tests.test_gpu_parity import check_topk_rows
from tests.util import dev_batch, make_engine, rel_err

pytestmark = pytest.mark.gpu

# logits GEMM: M = B up to 3 m-tiles of 128 rows, 24 n-tiles; dY: K = B
WIDE = O.Dims(token_vocab=5003, path_vocab=3001, target_vocab=3001, embed_dim=64, code_dim=256, max_contexts=50)
# 1 n-tile of classes under 3 m-tiles of examples: the logits GEMM walks n fastest
SMALL_Y = dataclasses.replace(WIDE, target_vocab=200)
# java14m's model widths (d = 128, D = 384, C = 200) at a vocabulary the oracle finishes in seconds
JAVA_WIDTHS = O.Dims(token_vocab=5003, path_vocab=3001, target_vocab=3001, embed_dim=128, code_dim=384, max_contexts=200)
# tables wide enough that every step's token and path rows can be distinct (see _distinct_rows_batch)
DISTINCT = O.Dims(token_vocab=50021, path_vocab=30011, target_vocab=3001, embed_dim=64, code_dim=256, max_contexts=50)

LOSS_TOL = 1e-4
SHRINKING = (384, 1, 130, 31, 257, 384)          # larger batches first: the short ones run over stale rows
TRAJECTORY = (384, 97, 384, 1, 200)


def tol(math):
    """(code vectors, attention, gradients) for the arithmetic mode."""
    return (3e-3, 2e-3, 1e-2) if math == 1 else (2e-5, 2e-6, 5e-5)


def _key(dims):
    return tuple(dataclasses.astuple(dims))


_params = {}
_cases = {}


def params_of(dims):
    if _key(dims) not in _params:
        _params[_key(dims)] = O.init_params(dims, seed=4321)
    return _params[_key(dims)]


def _batch(dims, B, seed):
    src, pth, tgt, mask, target = O.synthetic_batch(dims, B, seed=seed)
    src[0, 0] = tgt[0, 0] = src[min(1, B - 1), 0] = 3            # duplicates across src / tgt and across examples
    return src, pth, tgt, mask, target


def _one_and_full_bag_batch(dims, B, seed):
    """Example 0 has exactly one valid context, example 1 a full bag."""
    src, pth, tgt, mask, target = O.synthetic_batch(dims, B, seed=seed)
    full = O.synthetic_batch(dims, B, seed=seed + 1, full_bags=True)
    for a, f in zip((src, pth, tgt, mask), full[:4]):
        a[1] = f[1]
        a[0, 1:] = 0
    assert mask[0].sum() == 1 and mask[1].sum() == dims.max_contexts
    return src, pth, tgt, mask, target


def _distinct_rows_batch(dims, B, seed):
    """A batch in which every token row occurs at most once among src and tgt and every path row at most once, so no
    row of the embedding scatter-add sums more than one term: the float atomics leave nothing to chance and two
    schedules must agree bit for bit on every tensor."""
    rng = np.random.default_rng(seed)
    C = dims.max_contexts
    tok = rng.permutation(np.arange(1, dims.token_vocab, dtype=np.int32))[:2 * B * C].reshape(2, B, C)
    pth = rng.permutation(np.arange(1, dims.path_vocab, dtype=np.int32))[:B * C].reshape(B, C)
    valid = np.arange(C)[None, :] < rng.integers(1, C + 1, size=B)[:, None]
    src, tgt, pth = (np.where(valid, x, 0).astype(np.int32) for x in (tok[0], tok[1], pth))
    target = rng.integers(1, dims.target_vocab, size=B, dtype=np.int32)
    return src, pth, tgt, valid.astype(np.float32), target


def oracle_case(dims, B, seed, k=10, make=_batch):
    """(batch, (loss, grads, top-k indices, top-k values, code vectors, attention, scores)) on params_of(dims); no
    Adam step runs in the tests that use it, so every engine and arithmetic mode shares one computation."""
    key = (_key(dims), B, seed, k, make.__name__)
    if key not in _cases:
        params = params_of(dims)
        batch = make(dims, B, seed)
        loss_ref, g_ref, _ = O.train_loss_and_grads(params, *batch)
        idx_ref, val_ref, v_ref, alpha_ref, scores = O.evaluate_topk(params, *batch[:4], k=k)
        _cases[key] = (batch, (loss_ref, g_ref, idx_ref, val_ref, v_ref, alpha_ref, scores))
    return _cases[key]


def sampled_case(dims, B, seed, S=50):
    """Sampled-softmax step: (sampled, logq_true, logq_sampled, loss, grads of all five tensors) for oracle_case's
    batch.  The context gradients chain the oracle's dv through the full-softmax backward pass."""
    key = ("sampled", _key(dims), B, seed, S)
    if key not in _cases:
        params = params_of(dims)
        (src, pth, tgt, mask, target), _ = oracle_case(dims, B, seed)
        rng = np.random.default_rng(seed)
        sampled = O.log_uniform_sample(rng, S, dims.target_vocab)
        sampled[0] = target[B - 1]                        # an accidental hit
        sampled[1] = sampled[2]                           # a duplicate sampled class
        lq_t = O.log_uniform_logq(target, S, dims.target_vocab)
        lq_s = O.log_uniform_logq(sampled, S, dims.target_vocab)
        v, alpha, cache = O.forward(params, src, pth, tgt, mask)
        loss, dv, g_tgt, _ = O.sampled_softmax_loss_and_grads(params, v, target, sampled, lq_t, lq_s)
        h = cache.h.reshape(B, dims.max_contexts, -1)
        dalpha = np.einsum("bcd,bd->bc", h, dv)
        dz = alpha * (dalpha - (alpha * dalpha).sum(axis=1, keepdims=True))
        dh = alpha[:, :, None] * dv[:, None, :] + dz[:, :, None] * params["a"][None, None, :]
        du = (dh * (1.0 - h * h)).reshape(B * dims.max_contexts, -1).astype(np.float32)
        dx = du @ params["W"].T
        g_tok, g_path, dd = np.zeros_like(params["tok"]), np.zeros_like(params["path"]), dims.embed_dim
        np.add.at(g_tok, src.reshape(-1), dx[:, :dd])
        np.add.at(g_path, pth.reshape(-1), dx[:, dd:2 * dd])
        np.add.at(g_tok, tgt.reshape(-1), dx[:, 2 * dd:])
        grads = {"tok": g_tok, "path": g_path, "tgt": g_tgt, "W": cache.x.T @ du, "a": np.einsum("bc,bcd->d", dz, h)}
        _cases[key] = (sampled, lq_t, lq_s, loss, grads)
    return _cases[key]


# ---- checks shared by the tests ------------------------------------------------------------------------------------

def check_forward(eng, d, ref, math):
    v_ref, alpha_ref = ref[4], ref[5]
    code, attn = eng.forward(*d[:4])
    tc, ta, _ = tol(math)
    assert rel_err(code.cpu().numpy(), v_ref) < tc
    assert np.abs(attn.cpu().numpy() - alpha_ref).max() < ta
    return code


def check_topk(eng, code, ref, k, math, min_frac=0.95):
    """Raw scores (normalize 0), softmax over the k values (1) and full-vocabulary probabilities (2).  min_frac: share
    of the rows whose top-(k+1) gaps must all exceed fp32 rounding (check_topk_rows)."""
    idx_ref, val_ref, scores = ref[2], ref[3], ref[6]
    k = min(k, scores.shape[1])
    idx, val = (x.cpu().numpy() for x in eng.topk(code))
    assert idx.shape == (code.shape[0], k)
    vtol = 3e-3 * max(1.0, np.abs(val_ref).max()) if math == 1 else 1e-5
    if math == 1:        # tf32: top-1 wherever the fp32 margin exceeds the tf32 error bound
        srt = -np.sort(-scores, axis=1)
        clear = (srt[:, 0] - srt[:, 1]) > 2e-3
        assert np.array_equal(idx[clear, 0], idx_ref[clear, 0])
    else:
        check_topk_rows(idx, idx_ref, scores, k, min_frac=min_frac)
    assert np.abs(val - val_ref).max() < vtol
    idx1, val1 = (x.cpu().numpy() for x in eng.topk(code, normalize=1))
    assert np.array_equal(idx1, idx)
    np.testing.assert_allclose(val1, O.softmax_over_k(val), atol=1e-6)
    if math != 1:
        np.testing.assert_allclose(val1, O.softmax_over_k(val_ref), atol=1e-6)
    idx2, val2 = (x.cpu().numpy() for x in eng.topk(code, normalize=2))
    assert np.array_equal(idx2, idx)
    # log p = s - lse: an error e in the logits moves log p by at most 2 e
    p_ref = O.full_softmax_scores(scores, np.take_along_axis(scores, idx, axis=1))
    assert np.abs(np.log(val2) - np.log(p_ref)).max() < 2 * vtol
    return idx


def check_train_step(eng, d, batch, ref, math, dims):
    src, _, tgt, mask, _ = batch
    loss = float(eng.train_step(*d, keep=1.0).cpu()[0])
    assert abs(loss - ref[0]) < LOSS_TOL, (loss, ref[0])
    g = eng.export_grads()
    for name in O.PARAM_NAMES:
        assert rel_err(g[name], ref[1][name]) < tol(math)[2], (name, rel_err(g[name], ref[1][name]))
    touched = np.zeros(dims.token_vocab, bool)                    # rows of an earlier, larger batch are cleared
    touched[src[mask > 0]] = True
    touched[tgt[mask > 0]] = True
    assert np.all(g["tok"][~touched] == 0.0)
    assert eng.get_option("exp_slab_fallbacks") == 0


def check_sampled_step(eng, d, dims, B, seed, math):
    import torch
    sampled, lq_t, lq_s, loss_ref, g_ref = sampled_case(dims, B, seed)
    loss = float(eng.sampled_train_step(*d, eng.to_device(sampled, torch.int32), eng.to_device(lq_t, torch.float32),
                                        eng.to_device(lq_s, torch.float32)).cpu()[0])
    assert abs(loss - loss_ref) < LOSS_TOL, (loss, loss_ref)
    g = eng.export_grads()
    for name in O.PARAM_NAMES:
        assert rel_err(g[name], g_ref[name]) < tol(math)[2], (name, rel_err(g[name], g_ref[name]))


def run_batch(eng, dims, B, seed, math, k=10, make=_batch, topk=True):
    batch, ref = oracle_case(dims, B, seed, k=k, make=make)
    d = dev_batch(eng, *batch)
    code = check_forward(eng, d, ref, math)
    if topk:
        check_topk(eng, code, ref, k, math)
    check_train_step(eng, d, batch, ref, math, dims)
    return d


# ---- 1. multi-tile and short batches -------------------------------------------------------------------------------

SCHEDULES = [(0, 2, 1)] + [(m, p, s) for m in (1, 2) for p in (0, 1) for s in (1, 0)]


@pytest.mark.parametrize("math,cta_pair,exp_slab", SCHEDULES)
def test_multi_tile_and_short_batches_on_one_engine(math, cta_pair, exp_slab):
    """B = 384, 1, 130, 31, 257, 384 on ONE engine sized for 384: forward, top-10 (normalize 0 / 1 / 2), train step
    against the oracle at each, and a sampled-softmax step at B = 130 (three 64-example chunks) and B = 1."""
    dims = WIDE
    eng, _ = make_engine(dims, max_batch=max(SHRINKING), params=params_of(dims))
    eng.set_option("math_mode", math)
    eng.set_option("cta_pair", cta_pair)
    eng.set_option("exp_slab", exp_slab)
    for i, B in enumerate(SHRINKING):
        d = run_batch(eng, dims, B, 100 + i, math)
        if B in (130, 1):
            check_sampled_step(eng, d, dims, B, 100 + i, math)
    eng.close()


@pytest.mark.parametrize("math", [1, 2])
def test_few_classes_many_rows_raster(math):
    """Y = 200 under B = 384: the logits GEMM has fewer n-tiles than m-tiles and walks n fastest; then a short batch."""
    eng, _ = make_engine(SMALL_Y, max_batch=384, params=params_of(SMALL_Y))
    eng.set_option("math_mode", math)
    for B, seed in ((384, 200), (130, 201)):
        run_batch(eng, SMALL_Y, B, seed, math)
    eng.close()


@pytest.mark.parametrize("math", [0, 1, 2])
def test_production_batch_java_widths(math):
    """B = 1024 (bench.py's and the java14m config's batch) at d = 128, D = 384, C = 200."""
    eng, _ = make_engine(JAVA_WIDTHS, max_batch=1024, params=params_of(JAVA_WIDTHS))
    eng.set_option("math_mode", math)
    run_batch(eng, JAVA_WIDTHS, 1024, 300, math)
    eng.close()


@pytest.mark.parametrize("math", [0, 1, 2])
def test_lazy_fused_trajectory_over_changing_batch_sizes(math):
    """Trainer("single") -- lazy Adam with the sweep, target Adam in the dY epilogue, next-batch hints whose B differs
    from the current step's -- over B = 384, 97, 384, 1, 200 against a dense engine running train_step + adam_step.
    Embedding rows are distinct within each step, so only the schedules differ and the target table must come out
    bit-identical.  In fp32 FFMA the dense trajectory also follows the oracle's Adam."""
    import torch
    from code2vec_b200.trainer import Trainer
    dims, keep, seed = DISTINCT, 0.75, 3
    params0 = params_of(dims)
    fast, _ = make_engine(dims, max_batch=max(TRAJECTORY), params=params0)
    dense, _ = make_engine(dims, max_batch=max(TRAJECTORY), params=params0)
    for eng in (fast, dense):
        eng.set_option("math_mode", math)
    tr = Trainer(fast, keep_prob=keep, seed=seed)
    assert tr.schedule == "single" and tr.fuse_tgt and fast.get_option("lazy_adam") == 1
    batches = [_distinct_rows_batch(dims, B, 500 + s) for s, B in enumerate(TRAJECTORY)]
    on_device = [dev_batch(fast, *b) for b in batches]           # hints must stay alive until the next step is issued
    ref = {k: v.copy() for k, v in params0.items()}
    m = {k: np.zeros_like(p) for k, p in ref.items()}
    v = {k: np.zeros_like(p) for k, p in ref.items()}
    for s, batch in enumerate(batches):
        nxt = on_device[s + 1][:3] if s + 1 < len(batches) else None
        la = float(tr.step_device(*on_device[s], next_batch=nxt).cpu()[0])
        lb = float(dense.train_step(*dev_batch(dense, *batch), keep=keep, seed=seed, step=s + 1).cpu()[0])
        dense.adam_step()
        assert abs(la - lb) < 1e-5, (s, la, lb)
        if math == 0:
            dm = O.dropout_keep_mask(seed=seed, step=s + 1, n_rows=batch[0].size, ctx_dim=dims.ctx_dim, keep=keep)
            loss_ref, g_ref, _ = O.train_loss_and_grads(ref, *batch, keep=keep, dropout_mask=dm)
            O.adam_step(ref, g_ref, m, v, s + 1)
            assert abs(lb - loss_ref) < LOSS_TOL, (s, lb, loss_ref)
    # the first step has no hyper-parameters on record to run ahead with, the last one has no next batch; the fp32
    # path has no backward side stream to run them on
    assert fast.get_option("early_catchup_count") == (0 if math == 0 else len(TRAJECTORY) - 2)
    a, b = fast.export_params(), dense.export_params()
    if math != 0:
        assert np.array_equal(a["tgt"], b["tgt"])                # epilogue Adam == adam_kernel, bit for bit
    for k in O.PARAM_NAMES:
        assert np.abs(a[k] - b[k]).max() < 2e-6, k
        if math == 0:
            assert np.abs(b[k] - ref[k]).max() < 5e-5, k
    torch.cuda.synchronize()
    fast.close(); dense.close()


# ---- 2. every attention width --------------------------------------------------------------------------------------

@pytest.mark.parametrize("math", [0, 1, 2])
@pytest.mark.parametrize("embed_dim", [40, 160])
@pytest.mark.parametrize("code_dim", [256, 512, 640, 1020, 1024])
def test_every_attention_width(code_dim, embed_dim, math):
    """NV = ceil(D / 128) = 2, 4, 6 (last slice idle), 8 (last slice partial) and 8 (full); B = 130 then 37 on one
    engine, each batch with a one-context bag and a full bag."""
    dims = O.Dims(token_vocab=1009, path_vocab=503, target_vocab=1201, embed_dim=embed_dim, code_dim=code_dim, max_contexts=13)
    eng, _ = make_engine(dims, max_batch=130, params=params_of(dims))
    eng.set_option("math_mode", math)
    for B, seed in ((130, 40), (37, 41)):
        run_batch(eng, dims, B, seed, math, make=_one_and_full_bag_batch, topk=False)
    eng.close()


# ---- 3. top-k limits -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("math", [0, 1, 2])
@pytest.mark.parametrize("Y,k", [(3001, 1), (3001, 16), (3001, 17), (3001, 64), (40, 64)])
def test_topk_limits(Y, k, math):
    """k = 1 and 16 (register kernel), 17 and 64 (iterative kernel), and k = 64 over 40 classes: clamped to 40, the
    whole row sorted."""
    dims = O.Dims(token_vocab=1009, path_vocab=503, target_vocab=Y, embed_dim=64, code_dim=256, max_contexts=20)
    B = 130
    batch, ref = oracle_case(dims, B, 60, k=k)
    eng, _ = make_engine(dims, max_batch=B, top_k=k, params=params_of(dims))
    eng.set_option("math_mode", math)
    d = dev_batch(eng, *batch)
    code = check_forward(eng, d, ref, math)
    # the 65 largest of 3001 logits lie close together: about 1 row in 10 has a gap below fp32 rounding among them
    idx = check_topk(eng, code, ref, k, math, min_frac=0.85 if k == 64 and Y > k else 0.95)
    if k >= Y:
        assert np.array_equal(np.sort(idx, axis=1), np.tile(np.arange(Y), (B, 1)))
    eng.close()


# ---- 4. lazy-Adam row widths and occupancy -------------------------------------------------------------------------

@pytest.mark.parametrize("period", [0, 32])
@pytest.mark.parametrize("occupancy", [4, 5])
@pytest.mark.parametrize("embed_dim", [160, 20])
def test_long_idle_rows_replay_exactly_at_odd_widths(embed_dim, occupancy, period):
    """As test_gpu_lazy_adam.test_long_idle_rows_replay_exactly, with a row of one full and one partial 128-column
    slice (d = 160) and one much narrower than a slice (d = 20), and the row pass at 4 and 5 blocks per SM."""
    import torch
    B, steps = 8, 300
    dims = O.Dims(token_vocab=1501, path_vocab=701, target_vocab=101, embed_dim=embed_dim, code_dim=64, max_contexts=6)
    first = O.synthetic_batch(dims, B, seed=900)
    later = O.synthetic_batch(dims, B, seed=901)
    later = tuple(np.where(a > 0, 1 + (a % 40), a).astype(a.dtype) if i < 3 else a for i, a in enumerate(later))   # rows 1..40 only
    lazy, params0 = make_engine(dims, max_batch=B)
    dense, _ = make_engine(dims, max_batch=B, params=params0)
    lazy.set_option("lazy_adam", 1)
    lazy.set_option("adam_sweep_period", period)
    lazy.set_option("adam_rows_occupancy", occupancy)
    assert lazy.get_option("adam_rows_occupancy") == occupancy
    for s in range(steps):
        batch = first if s == 0 else later
        for eng in (lazy, dense):
            eng.train_step(*dev_batch(eng, *batch), keep=1.0)
            eng.adam_step()
    a, b = lazy.export_params(), dense.export_params()
    for name, cols in (("tok", (0, 2)), ("path", (1,))):
        counts = np.zeros(a[name].shape[0], dtype=np.int64)
        for c in cols:
            np.add.at(counts, first[c][first[3] > 0], 1)
        idle = counts == 1
        idle[:41] = False                                   # rows the later batches keep using
        assert idle.sum() > 20
        assert np.array_equal(a[name][idle].view(np.uint32), b[name][idle].view(np.uint32)), name
        assert np.abs(a[name][idle] - params0[name][idle]).max() > 1e-4          # they did move, then rested
        never = counts == 0
        never[:41] = False
        assert np.array_equal(a[name][never], params0[name][never])
        sel = torch.from_numpy(idle | never).to(lazy.dev)
        assert torch.equal(lazy.adam_m[name][sel], dense.adam_m[name][sel])
        assert torch.equal(lazy.adam_v[name][sel], dense.adam_v[name][sel])


# ---- 5. schedule options -------------------------------------------------------------------------------------------

def _run_schedule(dims, batches, params0, math, options):
    """Three steps -- two with the target Adam armed into dY, then one unarmed -- on a fresh engine.  Returns the
    losses, the unarmed step's target gradient and the engine; with dy_late = 0, checks that "target_grads_ready"
    fires inside every step."""
    import torch
    eng, _ = make_engine(dims, max_batch=max(len(b[4]) for b in batches), params=params0)
    eng.set_option("math_mode", math)
    for key, value in options.items():
        eng.set_option(key, value)
        assert eng.get_option(key) == value
    ready = None
    if options.get("dy_late") == 0:
        ready = torch.cuda.Event(enable_timing=True)
        eng.set_event("target_grads_ready", ready)
    losses, g_tgt = [], None
    for s, batch in enumerate(batches):
        t = s + 1
        armed = s < 2
        if armed:
            eng.arm_target_adam(t)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        loss = eng.train_step(*dev_batch(eng, *batch), keep=0.75, seed=7, step=t)
        end.record()
        torch.cuda.synchronize()
        losses.append(float(loss.cpu()[0]))
        assert eng.get_option("target_adam_fused_step") == (t if armed else 0)
        if ready is not None:         # recorded after this step started and no later than its end
            assert ready.query() and start.elapsed_time(ready) > 0 and ready.elapsed_time(end) >= 0
        if not armed:
            g_tgt = eng.grads["tgt"].clone()
        eng.adam_step(t=t)
    torch.cuda.synchronize()
    return losses, g_tgt, eng


@pytest.mark.parametrize("math", [1, 2])
@pytest.mark.parametrize("options", [{"dy_late": 0}, {"dy_late": 2}, {"adam_epilogue_prefetch": 1}],
                         ids=["dy_late0", "dy_late2", "adam_epilogue_prefetch"])
def test_schedule_option_is_bit_identical_to_the_default(options, math):
    """dy_late 0 / 2 against the default 1 and adam_epilogue_prefetch 1 against 0, at B = 384, Y = 3001: the same
    kernels in another order or on another stream, so the same bits -- loss, target table and its Adam slots, the
    unarmed step's target gradient, and (every embedding row being referenced once per step) all other tensors."""
    import torch
    dims = DISTINCT
    params0 = params_of(dims)
    batches = [_distinct_rows_batch(dims, 384, 800 + s) for s in range(3)]
    base = _run_schedule(dims, batches, params0, math, {"dy_late": 1, "adam_epilogue_prefetch": 0})
    other = _run_schedule(dims, batches, params0, math, options)
    assert base[0] == other[0]
    assert torch.equal(base[1], other[1])
    e0, e1 = base[2], other[2]
    assert not torch.equal(e0.params["tgt"].cpu(), torch.from_numpy(params0["tgt"]))        # it did move
    for name in O.PARAM_NAMES:
        assert torch.equal(e0.params[name], e1.params[name]), name
    assert torch.equal(e0.adam_m["tgt"], e1.adam_m["tgt"]) and torch.equal(e0.adam_v["tgt"], e1.adam_v["tgt"])
    e0.close(); e1.close()
