"""Host side of the nearest-neighbour queries (no device): query-line parsing, the command line's extra flags, and
the vocabulary lookup of most_similar."""
import io

import numpy as np
import pytest

from code2vec_b200.__main__ import parse_similarity_line, print_similar, strip_extra_flags
from code2vec_b200.b200_model import similarity_query_terms
from code2vec_b200.config import Config
from code2vec_b200.vocabularies import Vocab, VocabType


def test_query_lines():
    assert parse_similarity_line("equals to|lower\n") == (["equals", "to|lower"], [])
    assert parse_similarity_line("download send\treceive\n") == (["download", "send"], ["receive"])
    assert parse_similarity_line("a  b \t c\td\n") == (["a", "b"], ["c", "d"])       # a second TAB separates too
    assert parse_similarity_line("\tnegative|only") == ([], ["negative|only"])
    assert parse_similarity_line("-starts|with|dash") == (["-starts|with|dash"], [])    # no `-` prefix rule
    assert parse_similarity_line("\n") is None
    assert parse_similarity_line("   \t  \r\n") is None


def test_extra_flags_are_stripped_before_config():
    argv = ["--load", "m/saved", "--most_similar", "token", "--similar_input", "q.txt", "--topn", "5",
            "--predict_input", "p.txt"]
    rest, extra = strip_extra_flags(argv)
    assert rest == ["--load", "m/saved"]
    assert extra == {"predict_input": "p.txt", "most_similar": "token", "similar_input": "q.txt", "topn": 5}
    assert argv[2] == "--most_similar"                                                  # the caller's list is untouched
    cfg = Config(set_defaults=True)
    cfg.load_from_args(rest)                                                            # the reference's parser accepts the rest
    assert cfg.MODEL_LOAD_PATH == "m/saved"
    rest, extra = strip_extra_flags(["--load", "x", "--most_similar", "target"])
    assert extra["topn"] == 10 and extra["similar_input"] is None
    with pytest.raises(SystemExit):
        strip_extra_flags(["--load", "x", "--most_similar", "path"])
    with pytest.raises(SystemExit):
        strip_extra_flags(["--load", "x", "--topn"])


def _vocab():
    return Vocab(VocabType.Target, ["get|name", "set|name", "run"])


def test_unknown_word_raises_key_error():
    v = _vocab()
    terms, exclude = similarity_query_terms(v, ["get|name", "run"], ["set|name"])
    assert [(r, w) for r, w in terms] == [(0, 1.0), (2, 1.0), (1, -1.0)] and exclude == [0, 2, 1]
    with pytest.raises(KeyError):
        similarity_query_terms(v, ["get|name", "no|such|name"])
    with pytest.raises(KeyError):
        similarity_query_terms(v, None, ["<OOV>"])                                      # never mapped to the OOV word
    with pytest.raises(ValueError):
        similarity_query_terms(v, [], None)
    with pytest.raises(ValueError):
        similarity_query_terms(v, ["run"] * 17)


def test_single_items_and_vectors():
    v = _vocab()
    terms, exclude = similarity_query_terms(v, "run")
    assert terms == [(2, 1.0)] and exclude == [2]
    vec = np.arange(4, dtype=np.float64)
    terms, exclude = similarity_query_terms(v, vec, ["run"])
    assert terms[0][0].dtype == np.float32 and terms[0][1] == 1.0 and terms[1] == (2, -1.0)
    assert exclude == [2]                                                               # vectors are not excluded


def test_print_similar_layout_without_a_device():
    class FakeModel:
        class vocabs:
            @staticmethod
            def get(vt):
                return _vocab()

        def __init__(self):
            self.calls = []

        def most_similar_many(self, queries, topn, vocab_type):
            self.calls.append(list(queries))
            return [[("run", 0.5), ("set|name", -0.25)][:topn] for _ in queries]

    m, out = FakeModel(), io.StringIO()
    print_similar(m, ["get|name\n", "\n", "bogus word\n", "get|name\tset|name\n"], VocabType.Target, 2, out)
    assert m.calls == [[(["get|name"], []), (["get|name"], ["set|name"])]]             # one batched call
    assert out.getvalue() == ("Query:\tget|name\n\t(0.500000) run\n\t(-0.250000) set|name\n"
                              "Query:\tbogus word\nError:\tword 'bogus' not in vocabulary\n"
                              "Query:\tget|name\tset|name\n\t(0.500000) run\n\t(-0.250000) set|name\n")
