"""`Code2VecModel` for `--framework b200`: the third backend behind Code2VecModelBase.

Where the reference's TensorFlow backend (tensorflow_model.py:18-447) builds a graph and calls
`sess.run`, this class feeds host batches from the reader to the C-ABI engine:
    train()    : c2v_train_batch_host per batch      == sess.run([optimizer, train_loss])   (:80)
    evaluate() : c2v_predict_batch_host per batch    == sess.run([top_words, top_values, ...]) (:157-161)
    predict()  : c2v_predict_batch_host, batch of 1, normalised scores + attention           (:331-335)
Host-side bookkeeping (logging cadence, save/evaluate cadence, log.txt, .vectors, metrics) follows
the reference method by method; the citations are on each method.
"""
from __future__ import annotations

import json
import os
import struct
import time
from collections import Counter
from functools import partial
from typing import Dict, Iterable, List, Optional, Tuple

import numpy as np

from .common import common
from .config import Config
from .engine import PARAM_NAMES, EngineDims, PathAttentionEngine
from .model_base import Code2VecModelBase, ModelEvaluationResults, ModelPredictionResults
from .path_context_reader import EstimatorAction, ModelInputTensorsFormer, PathContextReader, ReaderInputTensors
from .trainer import Trainer
from .vocabularies import VocabType

def _prefetch(iterable, depth: int = 8):
    """Runs `iterable` (the reader) in a background thread, `depth` batches ahead: the native
    tensoriser and the C-ABI train call both release the GIL, so parsing the next batches overlaps
    the GPU step -- the role tf.data's prefetch(40) plays in the reference (path_context_reader.py:150)."""
    import queue
    import threading
    q: "queue.Queue" = queue.Queue(maxsize=depth)
    done = object()
    stop = threading.Event()

    def put(item) -> bool:
        while not stop.is_set():
            try:
                q.put(item, timeout=0.1)
                return True
            except queue.Full:
                continue
        return False

    def run():
        try:
            for item in iterable:
                if not put(item):
                    return                    # the consumer went away (endless readers end here)
            put(done)
        except BaseException as exc:          # surface reader errors in the consumer
            put(exc)

    threading.Thread(target=run, daemon=True).start()
    try:
        while True:
            item = q.get()
            if item is done:
                return
            if isinstance(item, BaseException):
                raise item
            yield item
    finally:
        stop.set()


def _with_next(iterable):
    """(item, following item or None) pairs: the one-batch lookahead behind the engine's next-batch hint."""
    it = iter(iterable)
    try:
        cur = next(it)
    except StopIteration:
        return
    for nxt in it:
        yield cur, nxt
        cur = nxt
    yield cur, None


def similarity_query_terms(vocab, positive=None, negative=None):
    """A most_similar query -> ([(row or vector, +1 / -1)], [rows of the query's words]).  As gensim: a single word
    or vector may stand for a one-item list, vectors are not excluded from the results, a word outside the
    vocabulary raises KeyError (it is not mapped to the OOV word) and a query without items raises ValueError."""
    def as_list(items):
        if items is None:
            return []
        if isinstance(items, (str, np.ndarray)):
            return [items]
        return list(items)
    terms, exclude = [], []
    for items, weight in ((as_list(positive), 1.0), (as_list(negative), -1.0)):
        for item in items:
            if isinstance(item, str):
                if item not in vocab.word_to_index:
                    raise KeyError("word '%s' not in vocabulary" % item)
                row = int(vocab.word_to_index[item])
                terms.append((row, weight))
                if row not in exclude:
                    exclude.append(row)
            else:
                terms.append((np.asarray(item, dtype=np.float32).reshape(-1), weight))
    if not terms:
        raise ValueError("cannot compute similarity with no input")
    if len(terms) > PathAttentionEngine.MAX_QUERY_TERMS:
        raise ValueError("at most %d words / vectors per query" % PathAttentionEngine.MAX_QUERY_TERMS)
    return terms, exclude


_CKPT_MAGIC = b"C2VB200\0"
_CKPT_SUFFIX = ".c2v_b200"


class Code2VecModel(Code2VecModelBase):
    _ADAM: Optional[dict] = None      # None = tf.compat.v1.train.AdamOptimizer() defaults (tensorflow_model.py:232)

    def __init__(self, config: Config):
        self.engine: Optional[PathAttentionEngine] = None
        self.trainer: Optional[Trainer] = None
        self.eval_reader = None
        self.predict_reader = None
        # the reference's TF variable names, kept for checkpoint metadata (tensorflow_model.py:32-36)
        self.vocab_type_to_tf_variable_name_mapping: Dict[VocabType, str] = {
            VocabType.Token: "WORDS_VOCAB", VocabType.Target: "TARGET_WORDS_VOCAB", VocabType.Path: "PATHS_VOCAB"}
        self._param_of_vocab = {VocabType.Token: "tok", VocabType.Target: "tgt", VocabType.Path: "path"}
        super().__init__(config)

    # ---- engine life cycle -------------------------------------------------------------------
    def _engine_dims(self) -> EngineDims:
        c = self.config
        if c.TOKEN_EMBEDDINGS_SIZE != c.PATH_EMBEDDINGS_SIZE:
            raise ValueError("the b200 backend needs TOKEN_EMBEDDINGS_SIZE == PATH_EMBEDDINGS_SIZE")
        if c.TARGET_EMBEDDINGS_SIZE != c.CODE_VECTOR_SIZE:
            raise ValueError("TARGET_EMBEDDINGS_SIZE must equal CODE_VECTOR_SIZE (logits = code_vectors . targets^T)")
        return EngineDims(token_vocab=self.vocabs.token_vocab.size, path_vocab=self.vocabs.path_vocab.size,
                          target_vocab=self.vocabs.target_vocab.size, embed_dim=c.TOKEN_EMBEDDINGS_SIZE,
                          code_dim=c.CODE_VECTOR_SIZE, max_contexts=c.MAX_CONTEXTS,
                          max_batch=max(c.TRAIN_BATCH_SIZE, c.TEST_BATCH_SIZE, 1),
                          top_k=c.TOP_K_WORDS_CONSIDERED_DURING_PREDICTION)

    def _make_engine(self):
        import torch
        if int(os.environ.get("WORLD_SIZE", "1")) > 1:
            # The multi-GPU schedules live in code2vec_b200.trainer (and bench.py drives them); wiring them into
            # train() also needs per-rank data sharding and sharded checkpoints, which this backend does not do yet.
            raise NotImplementedError("Code2VecModel.train()/evaluate() run one process on one GPU; "
                                      "use code2vec_b200.trainer.Trainer for multi-GPU steps")
        device = int(os.environ.get("LOCAL_RANK", "0")) if torch.cuda.device_count() > 1 else 0
        self.engine = PathAttentionEngine(self._engine_dims(), device=device, training=self.config.is_training)
        # arithmetic of the big matrix products: tensor cores (tf32 operands, fp32 accumulate) for training
        # steps, the reference's own fp32 FMA class for evaluate()/predict() so that top-k is decided on
        # fp32 logits.  C2V_MATH=fp32|tf32 forces one mode for both.
        forced = os.environ.get("C2V_MATH", "").lower()
        modes = {"fp32": 0, "tf32": 1, "3xtf32": 2}
        self._math_train = modes.get(forced, 1)
        # evaluate()/predict(): the tensor cores at fp32-equivalent accuracy (3xTF32), so top-k is decided on fp32-class
        # logits at tensor-core speed; both choices are logged, nothing switches silently
        self._math_eval = modes.get(forced, 2)
        self.log("b200 backend arithmetic: train = %s, evaluate/predict = %s (C2V_MATH=fp32|tf32|3xtf32 forces one for both)" % (
            {0: "fp32 FFMA", 1: "tf32 tensor cores", 2: "3xTF32 tensor cores (fp32-equivalent)"}[self._math_train],
            {0: "fp32 FFMA", 1: "tf32 tensor cores", 2: "3xTF32 tensor cores (fp32-equivalent)"}[self._math_eval]))
        # C2V_HINT_NEXT=1: pass each next batch to the engine (c2v_hint_next_batch); no measured gain on one GPU
        self._hint_next = os.environ.get("C2V_HINT_NEXT", "0") == "1"
        if self.config.is_training:
            self.trainer = Trainer(self.engine, keep_prob=self.config.DROPOUT_KEEP_RATE, seed=int(time.time()) & 0x7FFFFFFF,
                                   adam=self._ADAM)

    def _create_inner_model(self):
        self._make_engine()
        self.engine.init_params()
        n_params = sum(int(np.prod(s)) for s in self.engine.dims.shapes().values())
        self.log("Number of trainable params: {}".format(n_params))
        for name, shape in self.engine.dims.shapes().items():
            self.log("variable name: {} -- shape: {} -- #params: {}".format(name, shape, int(np.prod(shape))))

    def _load_inner_model(self):
        self._make_engine()
        path = self.config.MODEL_LOAD_PATH + _CKPT_SUFFIX
        self.log("Loading model weights from: " + path)
        self._read_checkpoint(path)
        self.log("Done loading model weights")

    def close_session(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None

    # ---- checkpoint: header (json) + raw little-endian float32 tensors -------------------------
    def _save_inner_model(self, path: str, release: bool = False):
        e = self.engine
        e.sync_tables()                                  # lazy Adam: replay deferred row updates before reading the tensors
        tensors = [("theta/" + k, e.params[k]) for k in PARAM_NAMES]
        with_optimizer = (not release) and e.adam_m is not None
        if with_optimizer:
            tensors += [("adam_m/" + k, e.adam_m[k]) for k in PARAM_NAMES]
            tensors += [("adam_v/" + k, e.adam_v[k]) for k in PARAM_NAMES]
        meta = {"format": 1, "dims": vars(e.dims), "adam_t": int(e.adam_t) if with_optimizer else 0,
                "epochs_trained": int(getattr(self, "nr_epochs_trained", 0)),
                "tf_names": {"tok": "model/WORDS_VOCAB", "path": "model/PATHS_VOCAB", "tgt": "model/TARGET_WORDS_VOCAB",
                             "W": "model/TRANSFORM", "a": "model/ATTENTION"},
                "tensors": []}
        offset = 0
        for name, t in tensors:
            n = int(t.numel()) * 4
            meta["tensors"].append({"name": name, "shape": list(t.shape), "offset": offset, "nbytes": n})
            offset += n
        header = json.dumps(meta).encode()
        tmp = path + _CKPT_SUFFIX + ".tmp"
        with open(tmp, "wb") as f:
            f.write(_CKPT_MAGIC)
            f.write(struct.pack("<Q", len(header)))
            f.write(header)
            for _, t in tensors:
                f.write(t.detach().cpu().numpy().astype("<f4", copy=False).tobytes())
        os.replace(tmp, path + _CKPT_SUFFIX)

    def _read_checkpoint(self, file_path: str):
        import torch
        if not os.path.isfile(file_path):
            raise ValueError("There is no model at path `{}`.".format(file_path))
        e = self.engine
        with open(file_path, "rb") as f:
            if f.read(8) != _CKPT_MAGIC:
                raise ValueError("`{}` is not a c2v_b200 checkpoint".format(file_path))
            (hlen,) = struct.unpack("<Q", f.read(8))
            meta = json.loads(f.read(hlen).decode())
            base = f.tell()
            want = vars(e.dims)
            for key in ("token_vocab", "path_vocab", "target_vocab", "embed_dim", "code_dim"):
                if meta["dims"][key] != want[key]:
                    raise ValueError("checkpoint %s=%s does not match the model (%s)" % (key, meta["dims"][key], want[key]))
            dest = {"theta": e.params, "adam_m": e.adam_m, "adam_v": e.adam_v}
            for ent in meta["tensors"]:
                group, name = ent["name"].split("/")
                if dest.get(group) is None:
                    continue
                f.seek(base + ent["offset"])
                arr = np.frombuffer(f.read(ent["nbytes"]), dtype="<f4").reshape(ent["shape"])
                dest[group][name].copy_(torch.from_numpy(arr.copy()))
            e.adam_t = int(meta.get("adam_t", 0))
            if e.training:
                # resuming: the engine's own step counter (lazy Adam needs consecutive steps and marks every row
                # as current as of this step) has to agree with the restored optimizer state
                e.set_option("adam_step_count", e.adam_t)
            if hasattr(self, "nr_epochs_trained"):           # the Keras-schedule backend resumes at this epoch
                self.nr_epochs_trained = int(meta.get("epochs_trained", 0))

    # ---- train (tensorflow_model.py:40-112) ------------------------------------------------------
    def train(self):
        self.log("Starting training")
        start_time = time.time()
        cfg = self.config
        batch_num, sum_loss = 0, 0.0
        multi_batch_start_time = time.time()
        num_batches_to_save_and_eval = max(int(cfg.train_steps_per_epoch * cfg.SAVE_EVERY_EPOCHS), 1)
        train_reader = PathContextReader(vocabs=self.vocabs, model_input_tensors_former=_TrainInputFormer(),
                                         config=cfg, estimator_action=EstimatorAction.Train)
        self.log("Started reader...")
        former = _TrainInputFormer()
        # pinned-host batch ring + copy stream (batch_ring.py): the reader thread draws every batch straight into a
        # page-locked slot, its upload overlaps the previous step, and the loop never waits for the GPU except to read
        # the losses at each progress line.  C2V_BATCH_RING=0 (or a reader without the native tensoriser) keeps the
        # synchronous c2v_train_batch_host path.
        ring = None
        if os.environ.get("C2V_BATCH_RING", "1") != "0" and not self._hint_next and train_reader._native_ready():
            import torch
            from .batch_ring import PinnedBatchRing
            ring = PinnedBatchRing(torch, self.engine.dev, cfg.TRAIN_BATCH_SIZE, cfg.MAX_CONTEXTS)
            train_reader.batch_ring = ring
            loss_hist = torch.zeros(max(int(cfg.NUM_BATCHES_TO_LOG_PROGRESS), 1), dtype=torch.float32).pin_memory()
            n_hist = 0
        self.h2d_bytes = 0
        for batch, following in _with_next(_prefetch(train_reader.get_dataset(), depth=4 if ring else 8)):
            t = former.from_model_input_form(batch)
            nxt = None
            if self._hint_next and following is not None:
                n = former.from_model_input_form(following)
                nxt = (n.path_source_token_indices, n.path_indices, n.path_target_token_indices)
            batch_num += 1
            self.engine.set_option("math_mode", self._math_train)
            if ring is not None:
                rows = int(t.target_index.shape[0])
                self.trainer.step_ring(ring, rows, loss_hist[n_hist:n_hist + 1])      # upload + step queued; nothing waited for
                n_hist += 1
                self.h2d_bytes += rows * (4 * cfg.MAX_CONTEXTS + 1) * 4
                flush = (batch_num % cfg.NUM_BATCHES_TO_LOG_PROGRESS == 0) or (batch_num % num_batches_to_save_and_eval == 0) \
                    or n_hist == loss_hist.numel()
                batch_loss = 0.0
                if flush:                          # the losses of the steps since the last progress line reach the host here
                    torch.cuda.current_stream(self.engine.dev).synchronize()
                    batch_loss = float(loss_hist[:n_hist].sum())
                    n_hist = 0
            else:
                batch_loss = self.trainer.step_host(t.path_source_token_indices, t.path_indices, t.path_target_token_indices,
                                                    t.context_valid_mask, t.target_index, next_batch=nxt)
            sum_loss += batch_loss
            if batch_num % cfg.NUM_BATCHES_TO_LOG_PROGRESS == 0:
                self._trace_training(sum_loss, batch_num, multi_batch_start_time)
                sum_loss = 0.0
                multi_batch_start_time = time.time()
            if batch_num % num_batches_to_save_and_eval == 0:
                epoch_num = int((batch_num / num_batches_to_save_and_eval) * cfg.SAVE_EVERY_EPOCHS)
                if cfg.MODEL_SAVE_PATH:
                    model_save_path = cfg.MODEL_SAVE_PATH + "_iter" + str(epoch_num)
                    self.save(model_save_path)
                    self.log("Saved after %d epochs in: %s" % (epoch_num, model_save_path))
                if cfg.is_testing:
                    results = self.evaluate()
                    text = str(results).replace("topk", "top{}".format(cfg.TOP_K_WORDS_CONSIDERED_DURING_PREDICTION))
                    self.log("After {nr_epochs} epochs -- {evaluation_results}".format(nr_epochs=epoch_num, evaluation_results=text))
        if ring is not None:
            import torch
            torch.cuda.current_stream(self.engine.dev).synchronize()
            if n_hist:
                sum_loss += float(loss_hist[:n_hist].sum())
            ring.close()
            train_reader.batch_ring = None
        self.log("Done training")
        if cfg.MODEL_SAVE_PATH:
            self.save(cfg.MODEL_SAVE_PATH)
            self.log("Model saved in file: %s" % cfg.MODEL_SAVE_PATH)
        elapsed = int(time.time() - start_time)
        self.log("Training time: %sH:%sM:%sS\n" % ((elapsed // 60 // 60), (elapsed // 60) % 60, elapsed % 60))

    # ---- evaluate (tensorflow_model.py:114-195) ------------------------------------------------------
    def evaluate(self) -> Optional[ModelEvaluationResults]:
        eval_start_time = time.time()
        cfg = self.config
        if self.eval_reader is None:
            self.eval_reader = PathContextReader(vocabs=self.vocabs, model_input_tensors_former=_EvaluateInputFormer(),
                                                 config=cfg, estimator_action=EstimatorAction.Evaluate)
        if cfg.MODEL_LOAD_PATH and not cfg.TRAIN_DATA_PATH_PREFIX and cfg.RELEASE:
            release_name = cfg.MODEL_LOAD_PATH + ".release"
            self.log("Releasing model, output model: %s" % release_name)
            self._save_inner_model(release_name, release=True)
            return None                            # as the reference does after --release (:132-136)
        self.engine.set_option("math_mode", self._math_eval)
        special = self.vocabs.target_vocab.special_words
        subtokens_metric = SubtokensEvaluationMetric(partial(common.filter_impossible_names, special))
        topk_metric = TopKAccuracyEvaluationMetric(cfg.TOP_K_WORDS_CONSIDERED_DURING_PREDICTION,
                                                   partial(common.get_first_match_word_from_top_predictions, special))
        total_predictions, total_batches = 0, 0
        code_vectors_file = open(cfg.TEST_DATA_PATH + ".vectors", "w") if cfg.EXPORT_CODE_VECTORS else None
        with open("log.txt", "w") as log_output_file:
            start_time = time.time()
            self.log("Starting evaluation")
            for batch in _prefetch(self.eval_reader.get_dataset()):
                t = _EvaluateInputFormer().from_model_input_form(batch)
                idx, _vals, code_vectors, _attn = self.engine.predict_batch_host(
                    t.path_source_token_indices, t.path_indices, t.path_target_token_indices, t.context_valid_mask,
                    normalize=False, want_code=cfg.EXPORT_CODE_VECTORS, want_attention=False)
                top_words = self.vocabs.target_vocab.lookup_word(idx)          # (batch, top_k) strings   (:302)
                original_names = list(t.target_string)
                self._log_predictions_during_evaluation(zip(original_names, top_words), log_output_file)
                topk_metric.update_batch(zip(original_names, top_words))
                subtokens_metric.update_batch(zip(original_names, top_words))
                total_predictions += len(original_names)
                total_batches += 1
                if code_vectors_file is not None:
                    self._write_code_vectors(code_vectors_file, code_vectors)
                if total_batches % cfg.NUM_BATCHES_TO_LOG_PROGRESS == 0:
                    self._trace_evaluation(total_predictions, time.time() - start_time)
            self.log("Done evaluating, epoch reached")
            log_output_file.write(str(topk_metric.topk_correct_predictions) + "\n")
        if code_vectors_file is not None:
            code_vectors_file.close()
        elapsed = int(time.time() - eval_start_time)
        self.log("Evaluation time: %sH:%sM:%sS" % ((elapsed // 60 // 60), (elapsed // 60) % 60, elapsed % 60))
        return ModelEvaluationResults(topk_acc=topk_metric.topk_correct_predictions,
                                      subtoken_precision=subtokens_metric.precision,
                                      subtoken_recall=subtokens_metric.recall, subtoken_f1=subtokens_metric.f1)

    # ---- predict (tensorflow_model.py:311-368) ----------------------------------------------------------
    def predict(self, predict_data_lines: Iterable[str]) -> List[ModelPredictionResults]:
        if self.predict_reader is None:
            self.predict_reader = PathContextReader(vocabs=self.vocabs, model_input_tensors_former=_EvaluateInputFormer(),
                                                    config=self.config, estimator_action=EstimatorAction.Predict)
        results: List[ModelPredictionResults] = []
        self.engine.set_option("math_mode", self._math_eval)
        for line in predict_data_lines:
            t = _EvaluateInputFormer().from_model_input_form(self.predict_reader.process_input_row(line))
            idx, scores, code_vectors, attn = self.engine.predict_batch_host(
                t.path_source_token_indices, t.path_indices, t.path_target_token_indices, t.context_valid_mask,
                normalize=True, want_code=True, want_attention=True)
            assert idx.shape[0] == 1
            top_words = self.vocabs.target_vocab.lookup_word(idx[0])
            attention_per_context = self._get_attention_weight_per_context(
                t.path_source_token_strings[0], t.path_strings[0], t.path_target_token_strings[0], attn[0])
            results.append(ModelPredictionResults(
                original_name=common.binary_to_string(t.target_string[0]), topk_predicted_words=top_words,
                topk_predicted_words_scores=scores[0], attention_per_context=attention_per_context,
                code_vector=(code_vectors[0] if self.config.EXPORT_CODE_VECTORS else None)))
        return results

    # ---- nearest neighbours: gensim's KeyedVectors.most_similar on the resident tables ----------------------
    # The reference README (README.md:236-251) loads the --save_t2v / --save_w2v text files into gensim for these
    # queries; here the cosine scan and top-k run on the engine (c2v_compose_queries, c2v_nearest).
    def most_similar(self, positive=None, negative=None, topn: int = 10, vocab_type: VocabType = VocabType.Target,
                     restrict_vocab: Optional[int] = None) -> List[Tuple[str, float]]:
        """gensim's most_similar: the `topn` rows closest by cosine to unitvec(mean of the unit vectors of the positive
        words and the negated unit vectors of the negative ones).  Items may be words or numpy vectors (used as given,
        not excluded); the query's words are never returned.  restrict_vocab=N scans the first N rows only (the N most
        frequent words).  Unknown words raise KeyError, an empty query ValueError."""
        return self.most_similar_many([(positive, negative)], topn=topn, vocab_type=vocab_type,
                                      restrict_vocab=restrict_vocab)[0]

    def similar_by_vector(self, vector, topn: int = 10, vocab_type: VocabType = VocabType.Target,
                          restrict_vocab: Optional[int] = None) -> List[Tuple[str, float]]:
        """The names (or tokens) closest to a vector, e.g. a code vector from predict()."""
        return self.most_similar(positive=[np.asarray(vector, dtype=np.float32)], topn=topn, vocab_type=vocab_type,
                                 restrict_vocab=restrict_vocab)

    def most_similar_many(self, queries, topn: int = 10, vocab_type: VocabType = VocabType.Target,
                          restrict_vocab: Optional[int] = None) -> List[List[Tuple[str, float]]]:
        """most_similar for many (positive, negative) queries: one query-composition launch and one search launch
        serve them all."""
        vocab = self.vocabs.get(vocab_type)
        parsed = [similarity_query_terms(vocab, pos, neg) for pos, neg in queries]
        if not parsed:
            return []
        if not 1 <= int(topn) <= PathAttentionEngine.NEAREST_MAX_K:
            raise ValueError("topn must be in [1, %d]" % PathAttentionEngine.NEAREST_MAX_K)
        e = self.engine
        name = self._param_of_vocab[vocab_type]
        if getattr(e, "table_world", 1) > 1 and name != "tgt":
            raise NotImplementedError("most_similar over row-sharded token / path tables is not supported")
        e.sync_tables()                          # lazy Adam: deferred rows must be current before they are scanned
        table = e.params[name]
        queries_dev = e.compose_queries(table, [terms for terms, _ in parsed])   # query words may lie past restrict_vocab
        bank = table if restrict_vocab is None else table[:max(1, min(int(restrict_vocab), table.shape[0]))]
        n_ex = max([len(ex) for _, ex in parsed] + [1])
        exclude = np.full((len(parsed), n_ex), -1, dtype=np.int32)
        for q, (_, ex) in enumerate(parsed):
            exclude[q, :len(ex)] = ex
        idx, val = e.nearest(bank, queries_dev, int(topn), exclude=exclude)
        idx, val = idx.cpu().numpy(), val.cpu().numpy()
        return [[(vocab.index_to_word[int(i)], float(v)) for i, v in zip(ri, rv) if i >= 0] for ri, rv in zip(idx, val)]

    def _get_vocab_embedding_as_np_array(self, vocab_type: VocabType) -> np.ndarray:
        assert vocab_type in VocabType
        self.engine.sync_tables()
        return self.engine.params[self._param_of_vocab[vocab_type]].detach().cpu().numpy()

    # ---- logging helpers (tensorflow_model.py:411-437) ------------------------------------------------------
    def _log_predictions_during_evaluation(self, results, output_file):
        special = self.vocabs.target_vocab.special_words
        for original_name, top_predicted_words in results:
            found = common.get_first_match_word_from_top_predictions(special, original_name, top_predicted_words)
            if found is None:
                output_file.write("No results for predicting: " + original_name)
                continue
            rank, word = found
            if rank == 0:
                output_file.write("Original: " + original_name + ", predicted 1st: " + word + "\n")
            else:
                output_file.write("\t\t predicted correctly at rank: " + str(rank + 1) + "\n")

    def _trace_training(self, sum_loss, batch_num, multi_batch_start_time):
        cfg = self.config
        elapsed = time.time() - multi_batch_start_time
        # the reference divides the summed mean losses by NUM_BATCHES * BATCH_SIZE (:426); kept as is
        avg_loss = sum_loss / (cfg.NUM_BATCHES_TO_LOG_PROGRESS * cfg.TRAIN_BATCH_SIZE)
        throughput = cfg.TRAIN_BATCH_SIZE * cfg.NUM_BATCHES_TO_LOG_PROGRESS / (elapsed if elapsed > 0 else 1)
        self.log("Average loss at batch %d: %f, \tthroughput: %d samples/sec" % (batch_num, avg_loss, throughput))

    def _trace_evaluation(self, total_predictions, elapsed):
        self.log("Evaluated %d examples..." % total_predictions)
        self.log("Prediction throughput: %d samples/sec" % int(total_predictions / (elapsed if elapsed > 0 else 1)))


# ---- host-side metrics (tensorflow_model.py:450-516) ---------------------------------------------------
class SubtokensEvaluationMetric:
    def __init__(self, filter_impossible_names_fn):
        self.nr_true_positives = 0
        self.nr_false_positives = 0
        self.nr_false_negatives = 0
        self.nr_predictions = 0
        self.filter_impossible_names_fn = filter_impossible_names_fn

    def update_batch(self, results):
        for original_name, top_words in results:
            prediction = self.filter_impossible_names_fn(top_words)[0]      # IndexError if none is legal, as upstream
            truth = Counter(common.get_subtokens(original_name))
            guess = Counter(common.get_subtokens(prediction))
            self.nr_true_positives += sum(n for tok, n in guess.items() if tok in truth)
            self.nr_false_positives += sum(n for tok, n in guess.items() if tok not in truth)
            self.nr_false_negatives += sum(n for tok, n in truth.items() if tok not in guess)
            self.nr_predictions += 1

    @property
    def true_positive(self):
        return self.nr_true_positives / self.nr_predictions

    @property
    def false_positive(self):
        return self.nr_false_positives / self.nr_predictions

    @property
    def false_negative(self):
        return self.nr_false_negatives / self.nr_predictions

    @property
    def precision(self):
        return self.nr_true_positives / (self.nr_true_positives + self.nr_false_positives)

    @property
    def recall(self):
        return self.nr_true_positives / (self.nr_true_positives + self.nr_false_negatives)

    @property
    def f1(self):
        p, r = self.precision, self.recall
        return 0 if p + r == 0 else 2 * p * r / (p + r)


class TopKAccuracyEvaluationMetric:
    def __init__(self, top_k: int, get_first_match_word_from_top_predictions_fn):
        self.top_k = top_k
        self.nr_correct_predictions = np.zeros(self.top_k)
        self.nr_predictions = 0
        self.get_first_match_word_from_top_predictions_fn = get_first_match_word_from_top_predictions_fn

    def update_batch(self, results):
        for original_name, top_predicted_words in results:
            self.nr_predictions += 1
            found = self.get_first_match_word_from_top_predictions_fn(original_name, top_predicted_words)
            if found is not None:
                self.nr_correct_predictions[found[0]:self.top_k] += 1

    @property
    def topk_correct_predictions(self):
        return self.nr_correct_predictions / self.nr_predictions


# ---- tuple orders the model consumes (tensorflow_model.py:519-551) ---------------------------------------
class _TrainInputFormer(ModelInputTensorsFormer):
    def to_model_input_form(self, t: ReaderInputTensors):
        return (t.target_index, t.path_source_token_indices, t.path_indices, t.path_target_token_indices,
                t.context_valid_mask)

    def from_model_input_form(self, row) -> ReaderInputTensors:
        return ReaderInputTensors(target_index=row[0], path_source_token_indices=row[1], path_indices=row[2],
                                  path_target_token_indices=row[3], context_valid_mask=row[4])


class _EvaluateInputFormer(ModelInputTensorsFormer):
    def to_model_input_form(self, t: ReaderInputTensors):
        return (t.target_string, t.path_source_token_indices, t.path_indices, t.path_target_token_indices,
                t.context_valid_mask, t.path_source_token_strings, t.path_strings, t.path_target_token_strings)

    def from_model_input_form(self, row) -> ReaderInputTensors:
        return ReaderInputTensors(target_string=row[0], path_source_token_indices=row[1], path_indices=row[2],
                                  path_target_token_indices=row[3], context_valid_mask=row[4],
                                  path_source_token_strings=row[5], path_strings=row[6],
                                  path_target_token_strings=row[7])
