"""Nearest-neighbour search on the engine (c2v_compose_queries, c2v_nearest) and gensim's most_similar on the model
and the command line, against float64 numpy.

Tolerances.  The engine computes cosines in fp32 FFMA; the reference computes them in float64.  Scores must agree
within SCORE_TOL at every position.  An index must match the reference's wherever the reference's score gaps to the
neighbouring positions both exceed GAP: closer than that, fp32 rounding may legitimately swap two rows."""
import ctypes
import io
import os

import numpy as np
import pytest

from tests.test_gpu_model import _config, _make_dataset

pytestmark = pytest.mark.gpu

SCORE_TOL = 1e-5
GAP = 1e-5


@pytest.fixture(scope="module")
def eng():
    from code2vec_b200.engine import EngineDims, PathAttentionEngine
    e = PathAttentionEngine(EngineDims(16, 16, 16, 4, 4, 4, 4, 4), device=0, training=False)
    yield e
    e.close()


def ref_search(bank, queries, k, exclude=None):
    """float64 cosine top-k: score descending, ties to the lower row; zero / NaN rows, excluded rows and zero queries
    give nothing.  Returns (idx [n, k+1], val [n, k+1]) padded with -1 / -inf, one position past k for the gap rule."""
    Q = np.asarray(queries, dtype=np.float64)
    rows = bank.shape[0]
    bn = np.empty(rows)
    dots = np.empty((Q.shape[0], rows))
    for r0 in range(0, rows, 65536):                                  # float64 in slices: bounded host memory
        B = np.asarray(bank[r0:r0 + 65536], dtype=np.float64)
        bn[r0:r0 + 65536] = np.linalg.norm(B, axis=1)
        dots[:, r0:r0 + 65536] = Q @ np.nan_to_num(B, nan=0.0).T
    with np.errstate(all="ignore"):
        qn = np.linalg.norm(Q, axis=1)
        S = dots / (qn[:, None] * bn[None, :])
    bad_row = ~(bn > 0) | np.isnan(bn)
    n = Q.shape[0]
    idx = np.full((n, k + 1), -1, dtype=np.int64)
    val = np.full((n, k + 1), -np.inf)
    for q in range(n):
        s = S[q].copy()
        s[bad_row | np.isnan(s)] = -np.inf
        if not qn[q] > 0:
            continue
        if exclude is not None:
            ex = [r for r in exclude[q] if r >= 0]
            s[ex] = -np.inf
        m = min(k + 1, int(np.isfinite(s).sum()))
        part = np.argpartition(-s, min(len(s) - 1, 4 * k + 64))[:4 * k + 65] if len(s) > 4 * k + 65 else np.arange(len(s))
        order = part[np.lexsort((part, -s[part]))][:m]
        idx[q, :m] = order
        val[q, :m] = s[order]
    return idx, val


def check_against_ref(idx, val, ref_idx, ref_val, k):
    idx, val = np.asarray(idx), np.asarray(val, dtype=np.float64)
    n = idx.shape[0]
    for q in range(n):
        valid = ref_idx[q, :k] >= 0
        assert np.array_equal(idx[q] >= 0, valid), (q, idx[q], ref_idx[q, :k])
        assert np.all(np.isneginf(val[q, ~valid]))
        assert np.abs(val[q, valid] - ref_val[q, :k][valid]).max(initial=0.0) <= SCORE_TOL, q
        rv = ref_val[q]
        for p in np.nonzero(valid)[0]:
            before = p == 0 or rv[p - 1] - rv[p] > GAP
            after = not np.isfinite(rv[p + 1]) or rv[p] - rv[p + 1] > GAP
            if before and after:
                assert idx[q, p] == ref_idx[q, p], (q, p, idx[q], ref_idx[q])


def _bank(rows, dim, seed):
    return np.random.default_rng(seed).standard_normal((rows, dim)).astype(np.float32)


def _queries(bank, n, seed):
    """Half perturbed bank rows (close neighbours exist), half random directions."""
    rng = np.random.default_rng(seed)
    q = rng.standard_normal((n, bank.shape[1])).astype(np.float32)
    pick = rng.integers(0, bank.shape[0], size=n)
    near = bank[pick] + 0.3 * q
    return np.where((np.arange(n) % 2 == 0)[:, None], near, q).astype(np.float32)


# (rows, dim, n, k): every value of each axis at least once; n = 17, 9, 65 are one past the per-chunk query capacity
# at dim 384, 1024 and <= 256; 1000 and 4099 rows are not multiples of any row tile (64, 32, 16)
SHAPES = [
    (1, 128, 7, 10), (5, 128, 7, 10), (1000, 128, 7, 10), (4099, 128, 7, 10), (261246, 384, 8, 10),
    (1000, 4, 7, 10), (1000, 20, 7, 10), (1000, 384, 7, 10), (4099, 1024, 7, 10),
    (4099, 128, 1, 10), (4099, 128, 64, 10), (4099, 128, 65, 10), (4099, 384, 17, 10), (1000, 1024, 9, 10),
    (4099, 20, 65, 10), (261246, 128, 1, 10),
    (4099, 384, 7, 1), (4099, 384, 7, 64), (4099, 128, 64, 64), (5, 384, 7, 64), (37, 1024, 3, 64), (1, 4, 2, 1),
]


@pytest.mark.parametrize("rows,dim,n,k", SHAPES)
def test_matches_float64_cosine(eng, rows, dim, n, k):
    import torch
    bank = _bank(rows, dim, seed=rows + dim)
    queries = _queries(bank, n, seed=n + k)
    idx, val = eng.nearest(torch.from_numpy(bank).to(eng.dev), torch.from_numpy(queries).to(eng.dev), k)
    ref_idx, ref_val = ref_search(bank, queries, k)
    check_against_ref(idx.cpu().numpy(), val.cpu().numpy(), ref_idx, ref_val, k)


def test_duplicates_in_different_slices_come_lower_row_first(eng):
    import torch
    bank = _bank(3000, 128, seed=1)
    for r in (2900, 1500, 40):
        bank[r] = bank[7]
    q = bank[7:8] + 0.01 * _bank(1, 128, seed=2)
    idx, val = eng.nearest(torch.from_numpy(bank).to(eng.dev), torch.from_numpy(q).to(eng.dev), 6)
    idx, val = idx.cpu().numpy()[0], val.cpu().numpy()[0]
    assert list(idx[:4]) == [7, 40, 1500, 2900]
    assert val[0] == val[1] == val[2] == val[3] and val[4] < val[3]


def test_results_do_not_depend_on_batching(eng):
    import torch
    bank = torch.from_numpy(_bank(50021, 128, seed=3)).to(eng.dev)
    queries = torch.from_numpy(_queries(bank.cpu().numpy(), 200, seed=4)).to(eng.dev)
    ia, va = eng.nearest(bank, queries, 20)
    ib, vb = eng.nearest(bank, queries, 20)
    assert torch.equal(ia, ib) and torch.equal(va, vb)
    for q in (0, 1, 63, 64, 65, 199):
        i1, v1 = eng.nearest(bank, queries[q:q + 1].clone(), 20)
        assert torch.equal(i1[0], ia[q]) and torch.equal(v1[0], va[q]), q
    i7, v7 = eng.nearest(bank, queries[60:67].clone(), 20)            # 7 queries: another register block width
    assert torch.equal(i7, ia[60:67]) and torch.equal(v7, va[60:67])


def test_excluded_zero_and_nan_rows_are_never_returned(eng):
    import torch
    bank = _bank(2000, 64, seed=5)
    queries = _queries(bank, 9, seed=6)
    zero_rows, nan_rows = [3, 700, 1999], [4, 1200]
    bank[zero_rows] = 0.0
    bank[nan_rows, 5] = np.nan
    queries[2] = 0.0                                                  # a zero query
    d_bank, d_q = torch.from_numpy(bank).to(eng.dev), torch.from_numpy(queries).to(eng.dev)
    idx0, _ = eng.nearest(d_bank, d_q, 10)
    idx0 = idx0.cpu().numpy()
    exclude = np.full((9, 16), -1, dtype=np.int32)
    exclude[:, :3] = idx0[:, :3]                                      # the three best of the plain search
    exclude[:, 3] = 17
    idx, val = eng.nearest(d_bank, d_q, 10, exclude=exclude)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    assert np.all(idx[2] == -1) and np.all(np.isneginf(val[2]))
    for q in range(9):
        returned = set(idx[q][idx[q] >= 0].tolist())
        assert not returned & set(zero_rows + nan_rows)
        assert not returned & set(exclude[q][exclude[q] >= 0].tolist())
        if q != 2:
            assert list(idx[q, :6]) == [r for r in idx0[q, 3:10] if r != 17][:6]       # the rest moves up
    ref_idx, ref_val = ref_search(bank, queries, 10, exclude=exclude)
    check_against_ref(idx, val, ref_idx, ref_val, 10)


def test_padding_when_fewer_than_k_results(eng):
    import torch
    bank = _bank(5, 8, seed=7)
    bank[1] = 0.0
    q = torch.from_numpy(bank[2:4].copy()).to(eng.dev)
    idx, val = eng.nearest(torch.from_numpy(bank).to(eng.dev), q, 10, exclude=np.array([[2, -1], [0, 4]], dtype=np.int32))
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    assert sorted(idx[0, :3].tolist()) == [0, 3, 4] and np.all(idx[0, 3:] == -1) and np.all(np.isneginf(val[0, 3:]))
    assert sorted(idx[1, :2].tolist()) == [2, 3] and np.all(idx[1, 2:] == -1) and np.all(np.isneginf(val[1, 2:]))
    assert idx[1, 0] == 3 and abs(val[1, 0] - 1.0) < 1e-6            # the query is row 3 itself


def test_compose_is_gensims_query_vector(eng):
    import torch
    bank = _bank(300, 40, seed=8)
    vec = np.random.default_rng(9).standard_normal(40).astype(np.float32)
    terms = [[(3, 1.0)], [(3, 1.0), (10, 1.0), (200, -1.0)], [(vec, 1.0), (7, -1.0)], [(vec, 1.0)]]
    out = eng.compose_queries(torch.from_numpy(bank).to(eng.dev), terms).cpu().numpy()
    unit = bank.astype(np.float64) / np.linalg.norm(bank.astype(np.float64), axis=1, keepdims=True)
    for q, t in enumerate(terms):
        mean = np.mean([w * (unit[x] if isinstance(x, int) else x.astype(np.float64)) for x, w in t], axis=0)
        assert np.abs(out[q] - mean / np.linalg.norm(mean)).max() < 1e-6, q


def test_invalid_arguments_are_rejected(eng):
    import torch
    lib, h = eng.lib, eng.h
    bank = torch.zeros((100, 16), dtype=torch.float32, device=eng.dev)
    bank[:, 0] = 1.0
    q = torch.ones((2, 16), dtype=torch.float32, device=eng.dev)
    idx = torch.empty((2, 64), dtype=torch.int32, device=eng.dev)
    val = torch.empty((2, 64), dtype=torch.float32, device=eng.dev)
    nbytes = lib.c2v_nearest_scratch_bytes(100, 2, 10)
    assert nbytes > 0 and lib.c2v_nearest_scratch_bytes(100, 2, 65) == 0 and lib.c2v_nearest_scratch_bytes(0, 2, 10) == 0
    scratch = torch.empty(lib.c2v_nearest_scratch_bytes(100, 2, 64) + 16, dtype=torch.uint8, device=eng.dev)
    ex = torch.full((2, 17), -1, dtype=torch.int32, device=eng.dev)
    good = dict(bank=bank.data_ptr(), rows=100, dim=16, q=q.data_ptr(), n=2, k=10, ex=None, nex=0,
                scratch=scratch.data_ptr(), sb=nbytes)

    def call(**kw):
        a = dict(good, **kw)
        return lib.c2v_nearest(h, a["bank"], a["rows"], a["dim"], a["q"], a["n"], a["k"], a["ex"], a["nex"],
                               idx.data_ptr(), val.data_ptr(), a["scratch"], a["sb"], None)

    assert call() == 0
    torch.cuda.synchronize()
    bad = {"NULL bank": dict(bank=None), "NULL queries": dict(q=None), "NULL scratch": dict(scratch=None),
           "k = 0": dict(k=0), "k = 65": dict(k=65), "dim % 4": dict(dim=18), "dim > 1024": dict(dim=1028),
           "rows = 0": dict(rows=0), "n = 0": dict(n=0), "misaligned bank": dict(bank=bank.data_ptr() + 4),
           "misaligned queries": dict(q=q.data_ptr() + 8), "misaligned scratch": dict(scratch=scratch.data_ptr() + 4),
           "small scratch": dict(sb=nbytes - 1), "n_exclude = 17": dict(ex=ex.data_ptr(), nex=17),
           "NULL exclude": dict(nex=3)}
    for what, kw in bad.items():
        assert call(**kw) == -1, what
        assert len(lib.c2v_last_error(h)) > 0, what
    rows = torch.zeros((2, 1), dtype=torch.int32, device=eng.dev)
    w = torch.ones((2, 1), dtype=torch.float32, device=eng.dev)
    assert lib.c2v_compose_queries(h, bank.data_ptr(), 100, 16, rows.data_ptr(), w.data_ptr(), None, 2, 1, q.data_ptr(), None) == 0
    assert lib.c2v_compose_queries(h, bank.data_ptr(), 100, 16, rows.data_ptr(), w.data_ptr(), None, 2, 17, q.data_ptr(), None) == -1
    assert lib.c2v_compose_queries(h, None, 100, 16, rows.data_ptr(), w.data_ptr(), None, 2, 1, q.data_ptr(), None) == -1
    assert lib.c2v_compose_queries(h, bank.data_ptr(), 100, 16, None, w.data_ptr(), None, 2, 1, q.data_ptr(), None) == -1
    assert len(lib.c2v_last_error(h)) > 0
    torch.cuda.synchronize()


# ---- the model: gensim's most_similar through the --save_t2v / --save_w2v files ------------------------------------

def read_word2vec(path):
    with open(path) as f:
        n, dim = map(int, f.readline().split())
        words, rows = [], []
        for line in f:
            parts = line.rstrip("\n").split(" ")
            words.append(parts[0])
            rows.append(np.array(parts[1:], dtype=np.float32))
    assert len(words) == n and rows[0].shape == (dim,)
    return words, np.stack(rows)


def gensim_most_similar(words, vectors, positive=(), negative=(), topn=10, restrict_vocab=None):
    """numpy restatement of gensim 4's KeyedVectors.most_similar (fill_norms, mean of weighted unit vectors, unitvec,
    dot / norms, drop the query's words, topn) in float64.  Returns [(word, score)] for topn + 1 positions."""
    index = {w: i for i, w in enumerate(words)}
    v = vectors.astype(np.float64)
    norms = np.linalg.norm(v, axis=1)
    terms = [(x, 1.0) for x in positive] + [(x, -1.0) for x in negative]
    mean = np.mean([w * (v[index[x]] / norms[index[x]] if isinstance(x, str) else np.asarray(x, np.float64))
                    for x, w in terms], axis=0)
    mean /= np.linalg.norm(mean)
    limit = len(words) if restrict_vocab is None else restrict_vocab
    dists = (v[:limit] @ mean) / norms[:limit]
    keys = {index[x] for x, _ in terms if isinstance(x, str)}
    order = [i for i in np.lexsort((np.arange(limit), -dists)) if i not in keys]
    return [(words[i], float(dists[i])) for i in order[:topn + 1]]


def check_gensim(got, ref, topn):
    assert len(got) == min(topn, len(ref))
    rv = [s for _, s in ref] + [-np.inf]
    for p, (word, score) in enumerate(got):
        assert abs(score - ref[p][1]) <= SCORE_TOL, (p, got, ref)
        if (p == 0 or rv[p - 1] - rv[p] > GAP) and rv[p] - rv[p + 1] > GAP:
            assert word == ref[p][0], (p, got, ref)


@pytest.fixture(scope="module")
def trained(tmp_path_factory):
    """The small model of test_gpu_model.py after a few batches, with its two word2vec files."""
    from code2vec_b200.b200_model import Code2VecModel
    from code2vec_b200.vocabularies import VocabType
    tmp = tmp_path_factory.mktemp("sim")
    prefix, _ = _make_dataset(tmp)
    model = Code2VecModel(_config(prefix, tmp, TRAIN_DATA_PATH_PREFIX=prefix, NUM_TRAIN_EPOCHS=3, DROPOUT_KEEP_RATE=1.0))
    model.train()
    files = {}
    for vt, name in ((VocabType.Target, "t2v"), (VocabType.Token, "w2v")):
        path = str(tmp / (name + ".txt"))
        model.save_word2vec_format(path, vt)
        files[vt] = read_word2vec(path)
    yield model, files
    model.close_session()


def test_most_similar_matches_gensim_on_the_exported_files(trained):
    from code2vec_b200.vocabularies import VocabType
    model, files = trained
    words, vecs = files[VocabType.Target]
    rng = np.random.default_rng(11)
    vec = rng.standard_normal(vecs.shape[1]).astype(np.float32)
    cases = [dict(positive=["get|name"]), dict(positive=["run", "to|string"]),
             dict(positive=["get|name", "set|name"], negative=["main"]), dict(positive=[vec]),
             dict(positive=[vec, "close"], negative=["is|empty"]), dict(positive="add|item", restrict_vocab=6)]
    for case in cases:
        for topn in (3, 10):
            got = model.most_similar(topn=topn, vocab_type=VocabType.Target, **case)
            pos = case.get("positive")
            pos = [pos] if isinstance(pos, (str, np.ndarray)) else pos
            ref = gensim_most_similar(words, vecs, pos, case.get("negative", ()), topn, case.get("restrict_vocab"))
            check_gensim(got, ref, topn)
    twords, tvecs = files[VocabType.Token]
    for pos, neg in ((["tok1"], []), (["tok3", "tok35"], ["tok9"])):
        got = model.most_similar(positive=pos, negative=neg, topn=10, vocab_type=VocabType.Token)
        check_gensim(got, gensim_most_similar(twords, tvecs, pos, neg, 10), 10)
    code = model.engine.params["tgt"][5].cpu().numpy()
    got = model.similar_by_vector(code, topn=4)
    check_gensim(got, gensim_most_similar(words, vecs, [code], (), 4), 4)
    assert got[0][0] == words[5]                                      # a row's own vector is not excluded
    many = model.most_similar_many([(["run"], []), (["main"], ["close"])], topn=5)
    assert many[0] == model.most_similar(positive=["run"], topn=5)
    with pytest.raises(KeyError):
        model.most_similar(positive=["no|such|name"])
    with pytest.raises(ValueError):
        model.most_similar(positive=[], negative=None)


def test_most_similar_reads_lazily_updated_rows_current(tmp_path):
    """Lazy Adam leaves deferred token rows stale in the table until they are replayed: most_similar, called first
    after training, must see the rows export_params() returns afterwards."""
    import torch
    from code2vec_b200.b200_model import Code2VecModel
    from code2vec_b200.vocabularies import VocabType
    prefix, _ = _make_dataset(tmp_path)
    model = Code2VecModel(_config(prefix, tmp_path, TRAIN_DATA_PATH_PREFIX=prefix, NUM_TRAIN_EPOCHS=4, DROPOUT_KEEP_RATE=1.0))
    try:
        model.train()
        assert model.engine.get_option("lazy_adam") == 1
        raw = model.engine.params["tok"].clone()
        got = [model.most_similar(positive=[w], topn=8, vocab_type=VocabType.Token) for w in ("tok0", "tok17", "tok33")]
        params = model.engine.export_params()
        assert not torch.equal(raw.cpu(), torch.from_numpy(params["tok"]))        # some rows were deferred
        words = [model.vocabs.token_vocab.index_to_word[i] for i in range(params["tok"].shape[0])]
        for w, g in zip(("tok0", "tok17", "tok33"), got):
            check_gensim(g, gensim_most_similar(words, params["tok"], [w], (), 8), 8)
    finally:
        model.close_session()


def test_search_between_train_steps_changes_nothing():
    from code2vec_b200.engine import EngineDims, PathAttentionEngine
    from oracle import path_attention_oracle as O
    from tests.test_gpu_batch_shapes import _distinct_rows_batch
    from tests.util import dev_batch
    import torch
    dims = O.Dims(token_vocab=5003, path_vocab=3001, target_vocab=3001, embed_dim=64, code_dim=256, max_contexts=20)
    params0 = O.init_params(dims, seed=4321)
    batches = [_distinct_rows_batch(dims, 64, 900 + s) for s in range(3)]
    runs = []
    for search in (False, True):
        e = PathAttentionEngine(EngineDims(dims.token_vocab, dims.path_vocab, dims.target_vocab, dims.embed_dim,
                                           dims.code_dim, dims.max_contexts, 64), device=0, training=True)
        e.load_params(params0)
        e.set_option("lazy_adam", 1)
        losses = []
        for s, batch in enumerate(batches):
            losses.append(float(e.train_step(*dev_batch(e, *batch), keep=0.75, seed=3, step=s + 1).cpu()[0]))
            e.adam_step()
            e.sync_tables()                                           # in both runs: the search is the only difference
            if search:
                for name in ("tgt", "tok", "path"):
                    bank = e.params[name]
                    q = e.compose_queries(bank, [[(1, 1.0), (2, -1.0)], [(5, 1.0)]])
                    e.nearest(bank, q, 64, exclude=np.array([[1, 2], [5, -1]], dtype=np.int32))
        torch.cuda.synchronize()
        runs.append((losses, e.export_params(), e))
    (la, pa, ea), (lb, pb, eb) = runs
    assert la == lb
    for name in pa:
        assert np.array_equal(pa[name].view(np.uint32), pb[name].view(np.uint32)), name
    for slot in ("adam_m", "adam_v"):
        for name in pa:
            assert torch.equal(getattr(ea, slot)[name], getattr(eb, slot)[name]), (slot, name)
    ea.close()
    eb.close()


def test_command_line_most_similar(tmp_path, monkeypatch, capsys):
    import tests.test_gpu_model as gm
    from code2vec_b200.__main__ import main
    monkeypatch.setattr(gm, "C", 200)                 # the default MAX_CONTEXTS
    monkeypatch.chdir(tmp_path)
    prefix, _ = _make_dataset(tmp_path)
    save = str(tmp_path / "cli" / "saved")
    assert main(["--data", prefix, "--save", save, "--framework", "b200"]) == 0
    queries = tmp_path / "queries.txt"
    queries.write_text("get|name\n\nrun to|string\tmain\nno|such|name run\n")
    capsys.readouterr()
    assert main(["--load", save, "--most_similar", "target", "--similar_input", str(queries), "--topn", "3"]) == 0
    out = capsys.readouterr().out.splitlines()
    q = [i for i, line in enumerate(out) if line.startswith("Query:\t")]
    assert [out[i] for i in q] == ["Query:\tget|name", "Query:\trun to|string\tmain", "Query:\tno|such|name run"]
    hits = out[q[0] + 1:q[1]]
    assert len(hits) == 3 and all(h.startswith("\t(") and ") " in h for h in hits)
    assert all(h.split(") ", 1)[1] != "get|name" for h in hits)
    hits2 = [h.split(") ", 1)[1] for h in out[q[1] + 1:q[2]] if h.startswith("\t(")]
    assert len(hits2) == 3 and not {"run", "to|string", "main"} & set(hits2)
    from code2vec_b200.b200_model import Code2VecModel
    from code2vec_b200.config import Config
    cfg = Config(set_defaults=True)
    cfg.load_from_args(["--load", save])
    cfg.VERBOSE_MODE = 0
    m = Code2VecModel(cfg)
    try:
        want = m.most_similar(positive=["run", "to|string"], negative=["main"], topn=3)
    finally:
        m.close_session()
    assert hits2 == [w for w, _ in want]
    assert out[q[2] + 1].startswith("Error:\t") and "no|such|name" in out[q[2] + 1]
    assert not any(line.startswith("\t(") for line in out[q[2] + 1:])
    # standard input, token vocabulary, default topn
    import sys
    monkeypatch.setattr(sys, "stdin", io.StringIO("tok1 tok2\n"))
    assert main(["--load", save, "--most_similar", "token"]) == 0
    out = capsys.readouterr().out.splitlines()
    q = [i for i, line in enumerate(out) if line.startswith("Query:\t")]
    assert [out[i] for i in q] == ["Query:\ttok1 tok2"]
    assert len([h for h in out[q[0] + 1:] if h.startswith("\t(")]) == 10
