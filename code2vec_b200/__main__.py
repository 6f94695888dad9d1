"""`python -m code2vec_b200 ...`: the reference's command line (code2vec.py:16-38) on the B200 backends.

Same flags (`Config.arguments_parser`, reference config.py:11-44) and the same order of actions:
train, export word2vec files, evaluate (or release), predict.  `--predict` differs in one respect: the
reference's REPL shells out to the Java path extractor (interactive_predict.py:18-21, extractor.py),
which is out of scope here; this entry point reads ALREADY-EXTRACTED lines (`name ctx ctx ...`, the
extractor's output format, SURVEY A.5) from `--predict_input FILE` or standard input, post-processes
them as extractor.py:22-38 does (first MAX_CONTEXTS contexts, path strings replaced by their Java
`String.hashCode`, padding to MAX_CONTEXTS fields) and prints each prediction in the reference's layout
(interactive_predict.py:50-63), attention paths un-hashed when the input carried path strings.

`--most_similar target|token [--similar_input FILE] [--topn N]` answers gensim `most_similar` queries (the workflow
the reference README runs on the --save_t2v / --save_w2v files, README.md:236-251) on the GPU: one query per line
of FILE or standard input, positive words separated by spaces, then optionally a TAB and the negative words.  The
extra flags are taken out of the argument list before `Config` parses it, so config.py stays the reference's.
"""
from __future__ import annotations

import sys
from typing import Iterable, Optional

from . import load_model_dynamically
from .common import common
from .config import Config
from .vocabularies import VocabType

SHOW_TOP_CONTEXTS = 10       # interactive_predict.py:6


def java_string_hashcode(s: str) -> int:
    """Java's String.hashCode (s[0]*31^(n-1) + ... + s[n-1] in wrapping 32-bit arithmetic) as a signed int:
    datasets store paths under this hash (extractor.py:40-49, ProgramRelation.java:18)."""
    h = 0
    for ch in s:
        h = (h * 31 + ord(ch)) % (1 << 32)
    return h - (1 << 32) if h >= (1 << 31) else h


def _looks_hashed(path: str) -> bool:
    body = path[1:] if path[:1] == "-" else path
    return body.isdigit()


def prepare_extracted_lines(lines: Iterable[str], max_contexts: int):
    """Extractor output -> model input lines + {hashed path: path string} (extractor.py:20-38)."""
    out, unhash = [], {}
    for line in lines:
        fields = line.rstrip().split(" ")
        if not fields or not fields[0]:
            continue
        contexts = [c for c in fields[1:] if c]
        kept = []
        for ctx in contexts[:max_contexts]:
            token1, path, token2 = ctx.split(",")
            hashed = path if _looks_hashed(path) else str(java_string_hashcode(path))
            unhash[hashed] = path
            kept.append("%s,%s,%s" % (token1, hashed, token2))
        out.append(" ".join([fields[0]] + kept) + " " * (max_contexts - len(kept)))
    return out, unhash


def print_predictions(config: Config, model, lines: Iterable[str], out=None):
    out = sys.stdout if out is None else out
    lines, unhash = prepare_extracted_lines(lines, config.MAX_CONTEXTS)
    if not lines:
        return
    raw_results = model.predict(lines)
    parsed = common.parse_prediction_results(raw_results, unhash, model.vocabs.target_vocab.special_words,
                                             topk=SHOW_TOP_CONTEXTS)
    for raw, method in zip(raw_results, parsed):
        out.write("Original name:\t" + method.original_name + "\n")
        for pair in method.predictions:
            out.write("\t(%f) predicted: %s\n" % (pair["probability"], pair["name"]))
        out.write("Attention:\n")
        for att in method.attention_paths:
            out.write("%f\tcontext: %s,%s,%s\n" % (att["score"], att["token1"], att["path"], att["token2"]))
        if config.EXPORT_CODE_VECTORS:
            out.write("Code vector:\n")
            out.write(" ".join(map(str, raw.code_vector)) + "\n")


SIMILARITY_VOCABS = {"target": VocabType.Target, "token": VocabType.Token}


def parse_similarity_line(line: str):
    """One nearest-neighbour query line -> (positive words, negative words), or None for a blank line.  Positive
    words are separated by spaces; an optional TAB is followed by the negative words.  (A `-` prefix cannot mark a
    negative word: nothing in the extractor's token normalisation rules out a token that starts with `-`.)"""
    line = line.rstrip("\r\n")
    pos, _, neg = line.partition("\t")
    positive, negative = pos.split(), neg.split()
    if not positive and not negative:
        return None
    return positive, negative


def print_similar(model, lines: Iterable[str], vocab_type: VocabType, topn: int, out=None):
    """gensim's most_similar for every query line (reference README.md:236-251), printed in print_predictions'
    layout: `Query:` then one `\\t(score) word` line per hit.  A line with an unknown word prints one error line."""
    from .b200_model import similarity_query_terms
    out = sys.stdout if out is None else out
    vocab = model.vocabs.get(vocab_type)
    entries = []                                       # (line, query or None, error message or None)
    for line in lines:
        q = parse_similarity_line(line)
        if q is None:
            continue
        try:
            similarity_query_terms(vocab, *q)
            entries.append((line.rstrip("\r\n"), q, None))
        except (KeyError, ValueError) as exc:
            entries.append((line.rstrip("\r\n"), None, exc.args[0] if exc.args else str(exc)))
    valid = [q for _, q, _ in entries if q is not None]
    results = iter(model.most_similar_many(valid, topn=topn, vocab_type=vocab_type) if valid else [])
    for line, q, err in entries:
        out.write("Query:\t" + line + "\n")
        if err is not None:
            out.write("Error:\t%s\n" % err)
            continue
        for word, score in next(results):
            out.write("\t(%f) %s\n" % (score, word))


def _pop_flag(argv, flag: str):
    """Removes `flag VALUE` from argv and returns VALUE (None when absent)."""
    if flag not in argv:
        return None
    i = argv.index(flag)
    if i + 1 >= len(argv):
        raise SystemExit("%s needs a value" % flag)
    value = argv[i + 1]
    del argv[i:i + 2]
    return value


def strip_extra_flags(argv):
    """Takes the flags the reference does not have out of argv before Config parses the rest:
    {"predict_input": FILE, "most_similar": "target" | "token", "similar_input": FILE, "topn": int}."""
    argv = list(argv)
    extra = {"predict_input": _pop_flag(argv, "--predict_input"), "most_similar": _pop_flag(argv, "--most_similar"),
             "similar_input": _pop_flag(argv, "--similar_input"), "topn": _pop_flag(argv, "--topn")}
    if extra["most_similar"] is not None and extra["most_similar"] not in SIMILARITY_VOCABS:
        raise SystemExit("--most_similar must be one of: %s" % ", ".join(sorted(SIMILARITY_VOCABS)))
    extra["topn"] = 10 if extra["topn"] is None else int(extra["topn"])
    return argv, extra


def main(argv: Optional[Iterable[str]] = None) -> int:
    argv, extra = strip_extra_flags(sys.argv[1:] if argv is None else argv)
    predict_input = extra["predict_input"]
    config = Config(set_defaults=True)
    config.load_from_args(argv)
    config.verify()
    model = load_model_dynamically(config)
    config.log("Done creating code2vec model")
    try:
        if config.is_training:
            model.train()
        if config.SAVE_W2V is not None:
            model.save_word2vec_format(config.SAVE_W2V, VocabType.Token)
            config.log("Origin word vectors saved in word2vec text format in: %s" % config.SAVE_W2V)
        if config.SAVE_T2V is not None:
            model.save_word2vec_format(config.SAVE_T2V, VocabType.Target)
            config.log("Target word vectors saved in word2vec text format in: %s" % config.SAVE_T2V)
        if (config.is_testing and not config.is_training) or config.RELEASE:
            eval_results = model.evaluate()
            if eval_results is not None:
                config.log(str(eval_results).replace("topk", "top{}".format(config.TOP_K_WORDS_CONSIDERED_DURING_PREDICTION)))
        if config.PREDICT:
            model.predict([])                          # the reference's warm-up call (interactive_predict.py:16)
            if predict_input:
                with open(predict_input, "r") as f:
                    print_predictions(config, model, f)
            else:
                print_predictions(config, model, sys.stdin)
        if extra["most_similar"] is not None:
            vocab_type = SIMILARITY_VOCABS[extra["most_similar"]]
            if extra["similar_input"]:
                with open(extra["similar_input"], "r") as f:
                    print_similar(model, f, vocab_type, extra["topn"])
            else:
                print_similar(model, sys.stdin, vocab_type, extra["topn"])
    finally:
        model.close_session()
    return 0


if __name__ == "__main__":
    sys.exit(main())
