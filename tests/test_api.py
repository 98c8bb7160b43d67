"""Drop-in surface (SURVEY.md 8b / Appendix C): the `densephrases` facade, Options flags, tokenizer, QA loader, metrics;
on the GPU: DensePhrases.search() and the evaluate() loop end to end over a synthetic corpus."""
import json
import os

import numpy as np
import pytest

from tests.helpers import jsonable

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def reference_golden(section):
    """What the unmodified reference code returned on the inputs defined in this module (tests/golden/reference_api.json,
    written by tests/golden/make_reference_api_golden.py)."""
    return json.load(open(os.path.join(GOLD, "reference_api.json")))[section]


# ---- inputs shared by the tests below and by tests/golden/make_reference_api_golden.py -----------------------------------------
EVAL_QA = [("which river crosses the city", ["the Seine", "Seine"]), ("who signed the treaty", ["Louis XIV"]), ("what year", ["1648", "in 1648"]),
           ("where", ["Paris"]), ("what is the a an the", ["yes"])]
EVAL_CANNED = {"which river crosses the city": ["Seine", "Loire"], "who signed the treaty": ["Louis XV", "Louis XIV", "x"], "what year": [],
               "where": ["paris.", "Lyon"], "what is the a an the": ["no", "Yes!"]}
SEARCH_UNITS = ["phrase", "sentence", "paragraph", "document"]
SEARCH_QUESTIONS = ["first question", "second question", "third"]
QA_PAIRS_DATA = {"data": [{"id": "a1", "question": "Which river?", "answers": ["Seine"]},
                          {"id": "a2", "origin": "nq.dev.x", "question": "who signed it", "answers": ["Louis", "Anne"], "titles": ["T1", "T2"]},
                          {"id": "a3", "question": "skipped", "answers": []},
                          {"id": "a4", "question": "x" * 400 + " [START_ENT] Paris [END_ENT] " + "y" * 400 + "?", "answers": ["Paris"]},
                          {"id": "a5", "question": "ALL CAPS?", "answers": ["x"]}]}
QA_PAIRS_CONFIGS = [(False, None), (True, None), (False, 1), (False, 3)]          # (do_lower_case, q_idx)
BACKWARD_COMPAT_SD = {"bert_q_start.embeddings.w": 1, "bert_q_end.x": 2, "bert_start.y": 3, "cross_encoder.z": 4, "bert_qd.q": 5, "qa_outputs.w": 6,
                      "query_start_encoder.k": 7, "linear.weight": 8}
OPTION_GROUPS = ("add_model_options", "add_index_options", "add_retrieval_options", "add_data_options")
OPTION_ARGV = ["--cuda", "--top_k", "40", "--nprobe", "64", "--index_name", "start/1048576_flat_OPQ96", "--eval_batch_size", "32", "--agg_strat", "opt2"]


def eval_setup(tmp_path):
    """Question file, parsed options and CPU stand-ins (encoder, phrase index with canned answers) for the evaluate loop."""
    import torch
    from densephrases import Options
    from densephrases_b200.tokenization import WordPieceTokenizer
    json.dump({"data": [{"id": str(i), "question": q, "answers": a} for i, (q, a) in enumerate(EVAL_QA)]}, open(os.path.join(tmp_path, "test.json"), "w"))
    o = Options()
    o.add_model_options(); o.add_index_options(); o.add_retrieval_options(); o.add_data_options()
    args = o.parse(["--test_path", os.path.join(tmp_path, "test.json"), "--load_dir", str(tmp_path), "--top_k", "3", "--eval_batch_size", "2", "--save_pred"])

    class FakeEncoder:
        def __call__(self, input_ids_=None, attention_mask_=None, token_type_ids_=None, return_query=False):
            assert return_query and input_ids_.shape == attention_mask_.shape == token_type_ids_.shape and input_ids_.shape[1] == args.max_query_length
            b = input_ids_.shape[0]
            return torch.ones((b, 1, 768)), torch.zeros((b, 1, 768))

        def eval(self):
            return self

    class FakeMips:
        num_docs_list = [1.0]

        def search(self, query, q_texts=None, nprobe=256, top_k=10, max_answer_length=10, aggregate=False, agg_strat='opt1', return_sent=False):
            assert query.shape == (len(q_texts), 1536) and top_k == 3
            return [[{"answer": a, "context": "ctx " + a, "title": ["T"], "score": 10.0 - j, "start_pos": 4, "end_pos": 4 + len(a)}
                     for j, a in enumerate(EVAL_CANNED[q])] for q in q_texts]

    return args, FakeMips(), FakeEncoder(), WordPieceTokenizer.from_pretrained_or_synthetic(None)


def search_setup(oracle):
    """(query2vec, MIPS over the CPU oracle index, parsed options) that DensePhrases.search runs on."""
    import torch
    from densephrases import Options
    from densephrases_b200 import runtime as R
    from densephrases_b200.mips import MIPS
    from densephrases_b200.tokenization import WordPieceTokenizer
    from tests.test_mips import OracleIndexAdapter, build
    doc_groups, idx_f, _, ref, query = build(oracle)
    mips = MIPS.from_components(OracleIndexAdapter(ref), idx_f, doc_groups, cuda=False)
    qvec = torch.from_numpy(query.astype(np.float32))

    class FakeEncoder:
        def __call__(self, input_ids_=None, attention_mask_=None, token_type_ids_=None, return_query=False):
            b = input_ids_.shape[0]
            return qvec[:b, None, :768], qvec[:b, None, 768:]

    o = Options()
    o.add_model_options(); o.add_index_options(); o.add_retrieval_options(); o.add_data_options()
    args = o.parse([])
    q2v = R.get_query2vec(query_encoder=FakeEncoder(), tokenizer=WordPieceTokenizer.from_pretrained_or_synthetic(None), args=args, batch_size=64)
    return q2v, mips, args


def search_outputs(model, unit):
    """DensePhrases.search results compared across implementations: batch answers, metadata without the vectors, one single query."""
    a = model.search(SEARCH_QUESTIONS, retrieval_unit=unit, top_k=3, truecase=False, return_meta=True)
    strip = [[{k: v for k, v in r.items() if k not in ("start_vec", "end_vec")} for r in ret] for ret in a[1]]
    single = model.search(SEARCH_QUESTIONS[0], retrieval_unit=unit, top_k=2, truecase=False)
    return jsonable({"answers": a[0], "meta": strip, "single": single})


class QaPairsArgs:
    do_lower_case, draft, truecase, truecase_path = False, False, False, ""


def truecase_differential_inputs(tables):
    """Random sentences (x 3 out-of-vocabulary policies) and score queries over the vocabulary of tests/golden/truecase.dist."""
    import random
    rng = random.Random(12345)
    vocab = list(tables["word_casing_lookup"]) + ["zzz", "o'brien", "42", "?", ",", "'s", "x-ray", "Ünïcode", "a.b"]
    cases = []
    for _ in range(400):
        s = " ".join(rng.choice(vocab) for _ in range(rng.randint(0, 12)))
        s = rng.choice([s, s.upper(), s.title(), "  " + s + " "])
        cases += [(s, oov) for oov in ("title", "lower", "as-is")]
    multi = [w for w, c in tables["word_casing_lookup"].items() if len(c) > 1]
    scores = []
    for _ in range(300):
        tok = rng.choice(tables["word_casing_lookup"][rng.choice(multi)])
        scores.append((rng.choice([None] + vocab), tok, rng.choice([None] + vocab)))
    return cases, scores


def test_reference_eval_script_imports_against_facade():
    """Every `densephrases...` / `faiss` import of the reference's eval_phrase_retrieval.py (recorded in the golden file) resolves
    against this repo's facade; the `faiss` stub imports but refuses to be used."""
    import importlib
    for imp in reference_golden("eval_script_imports"):
        mod = importlib.import_module(imp["module"])
        for name in imp["names"]:
            assert hasattr(mod, name), (imp["module"], name)
    import faiss
    with pytest.raises(RuntimeError):
        faiss.read_index


def test_options_defaults_match_reference():
    from densephrases import Options
    o = Options()
    o.add_model_options(); o.add_index_options(); o.add_retrieval_options(); o.add_data_options()
    a = o.parse([])
    assert (a.top_k, a.nprobe, a.eval_batch_size, a.max_query_length, a.max_answer_length) == (10, 256, 64, 64, 10)   # options.py:150-160,38,41
    assert (a.phrase_dir, a.index_path, a.idx2id_path, a.agg_strat, a.cuda) == ("phrase", "index.faiss", "idx2id.hdf5", "opt1", False)
    b = o.parse(["--cuda", "--top_k", "40", "--aggregate", "--index_name", "start/1048576_flat_OPQ96", "--unknown_flag", "1"])
    assert b.cuda and b.top_k == 40 and b.aggregate and b.index_name.endswith("OPQ96")


def test_tokenizer_question_features():
    from densephrases_b200.tokenization import WordPieceTokenizer
    t = WordPieceTokenizer.from_pretrained_or_synthetic(None, extra_words=["river", "##s"])
    ids, mask, tt, toks = t.encode_question("Which rivers?", 12)
    assert toks[0] == "[CLS]" and toks[-1] == "[SEP]" and "river" in toks and "##s" in toks and "?" in toks
    assert len(ids) == len(mask) == len(tt) == 12 and ids[0] == 101 and sum(mask) == len(toks) and set(tt) == {0}
    long_ids, long_mask, _, long_toks = t.encode_question("a " * 100, 8)
    assert len(long_ids) == 8 and sum(long_mask) == 8 and long_toks[-1] == "[SEP]"          # truncated to max_query_length
    assert t.wordpiece("中") == ["[UNK]"]


def test_load_qa_pairs_and_metrics(tmp_path):
    from densephrases_b200.runtime import exact_match_score, f1_score, load_qa_pairs, normalize_answer

    class A:
        do_lower_case = False; draft = False; truecase = False
    p = tmp_path / "qa.json"
    json.dump({"data": [{"id": "1", "question": "Who wrote it?", "answers": ["The Author"]}, {"id": "2", "question": "none", "answers": []},
                        {"id": "3", "origin": "nq.x", "question": "When", "answers": ["1999"], "titles": ["T"]}]}, open(p, "w"))
    ids, qs, ans, titles = load_qa_pairs(str(p), A())
    assert ids == ["1", "nq-3"] and qs == ["Who wrote it", "When"] and titles == [[""], ["T"]]
    assert normalize_answer("The  Author!") == "author" and exact_match_score("the author", "Author")
    assert f1_score("big red dog", "red dog")[0] == pytest.approx(0.8)


def test_load_encoder_raises_without_checkpoint_or_vocab(tmp_path):
    """A wrong load_dir / missing vocab.txt must not silently fall back to random weights (the reference raises, single_utils.py:62-93)."""
    import argparse
    from densephrases_b200.runtime import load_encoder
    args = argparse.Namespace(load_dir=str(tmp_path / "nope"), pretrained_name_or_path="SpanBERT/spanbert-base-cased", tokenizer_name="",
                              cache_dir="", do_lower_case=False)
    with pytest.raises(FileNotFoundError, match="vocab.txt"):
        load_encoder("cuda", args)
    (tmp_path / "tok").mkdir()
    (tmp_path / "tok" / "vocab.txt").write_text("\n".join(["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]", "a", "b"]) + "\n")
    args.tokenizer_name = str(tmp_path / "tok")
    with pytest.raises(FileNotFoundError, match="pytorch_model.bin"):
        load_encoder("cuda", args)
    args.load_dir = "princeton-nlp/densephrases-multi-query-multi"      # hub ids cannot be resolved offline: raise, do not invent weights
    with pytest.raises(FileNotFoundError):
        load_encoder("cuda", args)


@pytest.mark.gpu
def test_densephrases_search_and_evaluate_end_to_end(oracle, tmp_path):
    from densephrases import DensePhrases
    from densephrases_b200 import IvfPqIndex
    from densephrases_b200.mips import MIPS
    from densephrases_b200.runtime import evaluate
    from densephrases_b200.synthetic import make_corpus, make_phrase_index_arrays
    from tests.helpers import opq_matrix
    doc_groups, idx_f, ntotal = make_corpus(30, 5)
    list_len, codes, ids = make_phrase_index_arrays(ntotal, 32, 5)
    index = IvfPqIndex.from_arrays(opq_matrix(5), oracle.gen_centroids(5, 0, 32), oracle.gen_pq(5), list_len, codes, ids)
    mips = MIPS.from_components(index, idx_f, doc_groups, cuda=True)
    model = DensePhrases(load_dir="", dump_dir="unused", mips=mips, allow_random_init=True)
    qs = ["which river crosses the city", "Who signed the treaty", "museum of the island"]   # load_qa_pairs strips a trailing "?"
    single = model.search(qs[0], retrieval_unit="phrase", top_k=5)
    batch, meta = model.search(qs, retrieval_unit="phrase", top_k=5, return_meta=True)
    assert isinstance(single, list) and single == batch[0] and len(batch) == 3
    for rets in meta:
        assert 0 < len(rets) <= 5 and all(r["context"][r["start_pos"]:r["end_pos"]] == r["answer"] for r in rets)
        assert [r["score"] for r in rets] == sorted((r["score"] for r in rets), reverse=True)
    assert all(isinstance(t, str) for t in model.search(qs, retrieval_unit="document", top_k=3)[0])
    sents = model.search(qs, retrieval_unit="sentence", top_k=3)
    assert all(len(s) <= 3 for s in sents)
    # query2vec contract (open_utils.py:94-100): python lists [1][768] + tokens
    out = model.query2vec(qs[:2])
    assert len(out) == 2 and len(out[0][0]) == 1 and len(out[0][0][0]) == 768 and out[0][2][0] == "[CLS]"
    # evaluate loop
    p = tmp_path / "test.json"
    json.dump({"data": [{"id": str(i), "question": q, "answers": [meta[i][0]["answer"]]} for i, q in enumerate(qs)]}, open(p, "w"))
    args = model.args
    args.test_path, args.top_k, args.aggregate = str(p), 5, True
    res = evaluate(args, mips=mips, query_encoder=model.model, tokenizer=model.tokenizer)
    assert res["exact_match_top1"] == 1.0 and res["exact_match_top5"] == 1.0
    res2 = model.evaluate(str(p), top_k=5, aggregate=True)             # DensePhrases.evaluate (model.py:118-128): same loop through the model object
    assert res2["exact_match_top1"] == 1.0 and res2["predictions"] == res["predictions"]


@pytest.mark.parametrize("lower", [False, True])
def test_tokenizer_matches_transformers_bert_tokenizer(tmp_path, lower):
    """Row 8a-a3 pinned against the library the reference calls: same WordPiece sequence as transformers.BertTokenizer (the slow,
    pure-Python tokenizer; squad_utils.py:119-135 feeds it whitespace-split question tokens) on a shared vocabulary, for random
    strings with punctuation, accents, CJK, control / zero-width characters and over-long words; and the same padded features."""
    transformers = pytest.importorskip("transformers")
    import random
    from densephrases_b200.tokenization import WordPieceTokenizer
    words = ["river", "##s", "the", "Who", "who", "sign", "##ed", "treaty", "city", "##ing", "é", "##é", "naïve", "naive", "cafe", "中", "over", "##flow"]
    seed_tok = WordPieceTokenizer.from_pretrained_or_synthetic(None, extra_words=words)
    inv = sorted(seed_tok.vocab.items(), key=lambda kv: kv[1])
    lines = [f"[unused{i}]" for i in range(inv[-1][1] + 1)]
    for tok, i in inv:
        lines[i] = tok
    (tmp_path / "vocab.txt").write_text("\n".join(lines) + "\n", encoding="utf-8")
    hf = transformers.BertTokenizer(str(tmp_path / "vocab.txt"), do_lower_case=lower)
    mine = WordPieceTokenizer.from_pretrained_or_synthetic(str(tmp_path), do_lower_case=lower)
    rng = random.Random(7)
    alphabet = list("abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789") + list(" .,;:!?'\"()[]{}-_/\\@#$%^&*+=<>|~`") + \
        ["é", "ï", "中", "文", "\t", "\n", " ", "​", "\x00", "\x07", "ß", "—", "’", "“", "€", " river ", " rivers ", " signed ", " overflowing "]
    cases = ["Which rivers?", "Who signed the treaty of naïve café?", "a" * 150 + " b", "中文river", "hello world​zero", "x\x00y\x07z", ""]
    cases += ["".join(rng.choice(alphabet) for _ in range(rng.randint(0, 40))) for _ in range(1500)]
    for s in cases:
        assert mine.tokenize(s) == hf.tokenize(s), repr(s)
    for s in cases[:200]:
        enc = hf(s, max_length=16, padding="max_length", truncation=True)
        ids, mask, tt, toks = mine.encode_question(s, 16)
        assert ids == enc["input_ids"] and mask == enc["attention_mask"] and tt == enc["token_type_ids"], repr(s)


def test_metrics_match_reference_golden():
    """normalize_answer / f1 / EM / DrQA matchers against outputs of the unmodified reference functions
    (tests/golden/metrics.json, written by tests/golden/make_metrics_golden.py from eval_utils.py:9-86)."""
    from densephrases_b200 import runtime as R
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "metrics.json")))
    for c in g["pairs"]:
        p, t = c["prediction"], c["truth"]
        assert R.normalize_answer(p) == c["norm_p"] and R.exact_match_score(p, t) == c["em"] and R.drqa_exact_match_score(p, t) == c["drqa_em"]
        assert [float(v) for v in R.f1_score(p, t)] == c["f1"] and R.drqa_normalize(p) == c["drqa_norm"]
    for c in g["regex"]:
        assert R.drqa_regex_match_score(c["prediction"], c["pattern"]) == c["match"], c
    for c in g["max_over"]:
        assert bool(R.drqa_metric_max_over_ground_truths(R.drqa_exact_match_score, c["prediction"], c["truths"])) == c["em"]


def test_unmodified_reference_evaluate_runs_on_the_facade(tmp_path):
    """The reference's own `eval_phrase_retrieval.evaluate` (:49-91) + `evaluate_results` (:94-204), UNMODIFIED, executed over this
    repo's drop-in surface: `Options`, `load_qa_pairs`, `get_query2vec` (+ tokenizer) and the metric functions come from the
    `densephrases` facade; only the phrase index and the encoder are CPU stand-ins with the documented call signatures (eval_setup).
    What it returned and the prediction file it wrote are recorded in the golden file; densephrases_b200.runtime.evaluate gives the
    same numbers (the reference reports percentages), predictions and scores on the same inputs."""
    from densephrases_b200 import runtime as R
    g = reference_golden("evaluate")
    args, mips, enc, tok = eval_setup(tmp_path)
    mine = R.evaluate(args, mips=mips, query_encoder=enc, tokenizer=tok)
    assert (g["em1"], g["f11"], g["emk"], g["f1k"]) == pytest.approx((100 * mine["exact_match_top1"], 100 * mine["f1_score_top1"],
                                                                      100 * mine["exact_match_top3"], 100 * mine["f1_score_top3"]))
    assert g["em1"] == pytest.approx(40.0) and g["emk"] == pytest.approx(80.0)
    pred = g["pred"]                                                                     # written by the reference (:187-196)
    assert pred["1"]["prediction"] == EVAL_CANNED["who signed the treaty"] and pred["2"]["prediction"] == [""]
    assert mine["predictions"] == [pred[str(i)]["prediction"] for i in range(len(EVAL_QA))]
    assert mine["scores"] == [pred[str(i)]["score"] for i in range(len(EVAL_QA))]


@pytest.mark.parametrize("unit", SEARCH_UNITS)
def test_densephrases_search_wrapper_equals_unmodified_reference_class(oracle, unit):
    """model.py:55-109 (`DensePhrases.search`: query2vec -> stacked vectors -> MIPS.search with the unit's aggregation -> field
    selection) run UNMODIFIED over this repo's MIPS / query2vec (search_setup) returned what the golden file records; densephrases_b200's
    DensePhrases.search returns exactly that."""
    from densephrases import DensePhrases
    want = reference_golden("search")[unit]
    ours = DensePhrases.__new__(DensePhrases)
    ours.query2vec, ours.mips, ours.args = search_setup(oracle)
    ours.truecase = None
    got = search_outputs(ours, unit)
    assert len(got["answers"]) == 3 and all(len(x) <= 3 for x in got["answers"])
    assert got["answers"] == want["answers"] and got["single"] == want["single"]
    no_score = lambda meta: [[{k: v for k, v in r.items() if k != "score"} for r in rets] for rets in meta]
    assert no_score(got["meta"]) == no_score(want["meta"])
    # the scores pass through the host BLAS (OPQ matrix, query vectors), whose fp32 summation order depends on the CPU it runs on
    assert [r["score"] for rets in got["meta"] for r in rets] == pytest.approx([r["score"] for rets in want["meta"] for r in rets], rel=1e-5)


def test_open_utils_and_single_utils_helpers_equal_unmodified_reference(tmp_path):
    """`load_qa_pairs` (open_utils.py:103-163) and `backward_compat` (single_utils.py:36-56): the reference's code (its imports of
    squad_utils / embed_utils -- not on this path -- stubbed) on awkward inputs returned what the golden file records; the facade's
    versions return the same."""
    from densephrases.utils import open_utils as mine_open, single_utils as mine_single
    g = reference_golden("qa_pairs")
    p = tmp_path / "qa.json"
    json.dump(QA_PAIRS_DATA, open(p, "w"))
    for (lower, q_idx), want in zip(QA_PAIRS_CONFIGS, g["load_qa_pairs"], strict=True):
        QaPairsArgs.do_lower_case = lower
        got = mine_open.load_qa_pairs(str(p), QaPairsArgs, q_idx=q_idx)
        assert jsonable([list(x) for x in got]) == want
    assert jsonable(mine_single.backward_compat(dict(BACKWARD_COMPAT_SD))) == g["backward_compat"]


def test_option_flags_and_defaults_equal_reference_parser():
    """Every flag of the four option groups eval_phrase_retrieval.py / model.py add (options.py: model, index, retrieval, data)
    exists here with the same default; nothing is renamed.  The reference parser's values are recorded in the golden file."""
    from densephrases import Options
    g = reference_golden("options")
    ours = Options()
    for group in OPTION_GROUPS:
        getattr(ours, group)()
    want, got = g["defaults"], jsonable(vars(ours.parse([])))
    assert not [k for k in want if k not in got]
    assert {k: got[k] for k in want} == want
    got2 = jsonable(vars(ours.parse(OPTION_ARGV)))
    assert {k: got2[k] for k in g["argv"]} == g["argv"]


def test_synthetic_dump_spec_objects(tmp_path):
    """densephrases_b200/synthetic_dump.py: the spec files land where load_phrase_index looks (open_utils.py:28-31), idx2id lookups are
    arithmetic, documents are a pure function of (seed, doc) -- every rank of a sharded job sees the same corpus."""
    import os
    from densephrases_b200 import synthetic_dump as SD
    ntotal = SD.write_synthetic_dump(str(tmp_path), "start/64_flat_OPQ96", 128 * 50 + 3, 64, tokens_per_doc=128, seed=7)
    assert ntotal == 128 * 50
    for rel in ("start/64_flat_OPQ96/index.dph.json", "start/64_flat_OPQ96/idx2id.dph.json", "meta_dph.json", "phrase"):
        assert os.path.exists(tmp_path / rel)
    idx = SD.synthetic_idx2id(ntotal, 128)
    rows = np.array([0, 127, 128, 6399])
    assert idx["0"]["doc"][rows].tolist() == [0, 0, 1, 49] and idx["0"]["word"][rows].tolist() == [0, 127, 0, 127]
    a, b = SD.LazyDocs(128, 7), SD.LazyDocs(128, 7)
    ra, rb = a["13"], b[13]
    assert ra["context"] == rb["context"] and np.array_equal(ra["word2char_end"], rb["word2char_end"]) and ra["title"] == "Doc 13"
    assert len(ra["f2o_start"]) == 128 and ra["word2char_end"][-1] == len(ra["context"])
    w = 17
    assert ra["context"][ra["word2char_start"][w]:ra["word2char_end"][w]] in SD._WORDS
    assert SD.LazyDocs(128, 8)["13"]["context"] != ra["context"]
    assert SD.uniform_list_lengths(10, 4).tolist() == [3, 3, 2, 2]
    qa = SD.write_synthetic_questions(str(tmp_path / "q.json"), 5)
    import json as _json
    assert len(_json.load(open(qa))["data"]) == 5


# ---- truecaser (squad_utils.py:1452-1585, model.py:52,66-67) ------------------------------------------------------
def test_truecaser_matches_reference_golden():
    """tests/golden/truecase.json was produced by the UNMODIFIED reference TrueCaser class on tests/golden/truecase.dist."""
    import json
    from densephrases_b200.truecase import TrueCaser, truecase_questions
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    tc = TrueCaser(os.path.join(here, "truecase.dist"))
    gold = json.load(open(os.path.join(here, "truecase.json")))
    for c in gold["cases"]:
        assert tc.get_true_case(c["sentence"], c["oov"]) == c["truecased"], c
    for s in gold["scores"]:
        assert tc.get_score(s["prev"], s["token"], s["next"]) == s["score"], s          # same float, not approximately
    assert truecase_questions(tc, ["who is the president of france ?", "Already Cased"])[1] == "Already Cased"


def test_truecaser_rejects_other_pickles(tmp_path):
    import pickle
    from densephrases_b200.truecase import TrueCaser
    p = tmp_path / "x.dist"
    pickle.dump({"uni_dist": {}}, open(p, "wb"))
    with pytest.raises(KeyError):
        TrueCaser(str(p))
    with pytest.raises(FileNotFoundError):
        TrueCaser(str(tmp_path / "missing.dist"))


def test_load_qa_pairs_truecases_lower_case_questions(tmp_path, monkeypatch, capsys):
    """open_utils.py:147-156: with args.truecase the all-lower-case questions are re-cased from $DATA_DIR/<truecase_path>; a missing
    statistics file is printed and ignored."""
    import densephrases_b200.runtime as rt
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    gold = {c["sentence"]: c["truecased"] for c in json.load(open(os.path.join(here, "truecase.json")))["cases"] if c["oov"] == "title"}

    class A:
        do_lower_case = False; draft = False; truecase = True; truecase_path = "truecase.dist"
    p = tmp_path / "qa.json"
    json.dump({"data": [{"id": "1", "question": "who is the president of france ?", "answers": ["x"]},
                        {"id": "2", "question": "Who is the President?", "answers": ["y"]}]}, open(p, "w"))
    monkeypatch.setenv("DATA_DIR", here)
    monkeypatch.setattr(rt, "_truecaser", None)
    _, qs, _, _ = rt.load_qa_pairs(str(p), A())
    assert qs == [gold["who is the president of france ?"[:-1]] if "who is the president of france " in gold else rt._truecaser.get_true_case("who is the president of france "),
                  "Who is the President"]
    assert qs[0] != "who is the president of france "           # it was re-cased
    monkeypatch.setenv("DATA_DIR", str(tmp_path))                # no statistics file there
    monkeypatch.setattr(rt, "_truecaser", None)
    _, qs2, _, _ = rt.load_qa_pairs(str(p), A())
    assert qs2[0] == "who is the president of france " and "truecase.dist" in capsys.readouterr().out


def test_truecaser_differential_against_the_reference_class():
    """The UNMODIFIED `TrueCaser` source (cut out of squad_utils.py with `ast`, like tests/golden/make_truecase_golden.py) was run on
    random sentences and score queries (truecase_differential_inputs); ours gives every output string and every score it recorded."""
    import pickle
    from densephrases_b200.truecase import TrueCaser
    here = os.path.join(GOLD, "truecase.dist")
    g = reference_golden("truecase_differential")
    cases, scores = truecase_differential_inputs(pickle.load(open(here, "rb")))
    ours = TrueCaser(here)
    assert len(cases) == len(g["cases"]) and len(scores) == len(g["scores"])
    for (s, oov), want in zip(cases, g["cases"]):
        assert ours.get_true_case(s, oov) == want, (s, oov)
    for (prev, tok, nxt), want in zip(scores, g["scores"]):
        assert ours.get_score(prev, tok, nxt) == want, (prev, tok, nxt)
