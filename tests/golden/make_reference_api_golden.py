"""Golden outputs of the UNMODIFIED reference code for tests/test_api.py, computed on the inputs that module defines: the
`densephrases` / `faiss` imports of eval_phrase_retrieval.py, its `evaluate` (:49-204), model.py's `DensePhrases.search` (:55-109),
open_utils.load_qa_pairs (:103-163) and single_utils.backward_compat (:36-56), the four option groups of options.py, and the
`TrueCaser` class of squad_utils.py (:1452-1585).  Where the reference imports `densephrases`, it gets this repo's facade, as it
would if the facade were installed in its place; imports that are not on these paths are stubbed.

    python tests/golden/make_reference_api_golden.py <reference checkout>   ->   tests/golden/reference_api.json"""
import ast
import importlib.util
import json
import math
import os
import pickle
import string
import sys
import tempfile
import types
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import test_api as T  # noqa: E402
from tests.helpers import jsonable  # noqa: E402


def load(name, path, stubs=None):
    """Executes the file at `path` as module `name`, with `stubs` ({module: attribute names}) importable while it loads."""
    stubs = stubs or {}
    for mod_name, attrs in stubs.items():
        m = types.ModuleType(mod_name)
        for a in attrs:
            setattr(m, a, type(a, (), {}))
        sys.modules[mod_name] = m
    try:
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for mod_name in stubs:
            del sys.modules[mod_name]
    return mod


def cut(path, name):
    src = open(path).read()
    node = next(n for n in ast.parse(src).body if getattr(n, "name", None) == name)
    return ast.get_source_segment(src, node)


def eval_script_imports(ref):
    path = os.path.join(ref, "eval_phrase_retrieval.py")
    mod = load("ref_eval_phrase_retrieval_imports", path)          # every import line resolves against the facade
    assert callable(mod.evaluate) and callable(mod.embed_all_query)
    ours = ("densephrases", "faiss")
    out = []
    for n in ast.parse(open(path).read()).body:
        if isinstance(n, ast.ImportFrom) and n.module.split(".")[0] in ours:
            out.append({"module": n.module, "names": [a.name for a in n.names]})
        elif isinstance(n, ast.Import):
            out += [{"module": a.name, "names": []} for a in n.names if a.name.split(".")[0] in ours]
    return out


def evaluate(ref):
    mod = load("ref_eval_phrase_retrieval", os.path.join(ref, "eval_phrase_retrieval.py"))
    with tempfile.TemporaryDirectory() as tmp:
        args, mips, enc, tok = T.eval_setup(tmp)
        em1, f11, emk, f1k = mod.evaluate(args, mips=mips, query_encoder=enc, tokenizer=tok)
        pred = json.load(open(os.path.join(tmp, "pred", f"test_{len(T.EVAL_QA)}_top{args.top_k}.pred")))
    return {"em1": em1, "f11": f11, "emk": emk, "f1k": f1k, "pred": pred}


def search(ref, oracle):
    mod = load("ref_densephrases_model", os.path.join(ref, "densephrases", "model.py"), {"densephrases.utils.squad_utils": ("TrueCaser",)})
    out = {}
    for unit in T.SEARCH_UNITS:
        theirs = mod.DensePhrases.__new__(mod.DensePhrases)
        theirs.query2vec, theirs.mips, theirs.args = T.search_setup(oracle)
        theirs.truecase = None
        out[unit] = T.search_outputs(theirs, unit)
    return out


def qa_pairs(ref):
    stubs = {"densephrases.utils.squad_utils": ("get_question_dataloader", "TrueCaser"), "densephrases.utils.embed_utils": ("get_question_results",)}
    single = load("ref_single_utils", os.path.join(ref, "densephrases", "utils", "single_utils.py"), stubs)
    open_utils = load("ref_open_utils", os.path.join(ref, "densephrases", "utils", "open_utils.py"), stubs)
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        p = os.path.join(tmp, "qa.json")
        json.dump(T.QA_PAIRS_DATA, open(p, "w"))
        for lower, q_idx in T.QA_PAIRS_CONFIGS:
            T.QaPairsArgs.do_lower_case = lower
            rows.append([list(x) for x in open_utils.load_qa_pairs(p, T.QaPairsArgs, q_idx=q_idx)])
    return {"load_qa_pairs": rows, "backward_compat": single.backward_compat(dict(T.BACKWARD_COMPAT_SD))}


def options(ref):
    theirs = load("ref_options", os.path.join(ref, "densephrases", "options.py")).Options()
    for group in T.OPTION_GROUPS:
        getattr(theirs, group)()
    return {"defaults": vars(theirs.parser.parse_args([])), "argv": vars(theirs.parser.parse_args(T.OPTION_ARGV))}


def truecase_differential(ref):
    ns = {"os": os, "pickle": pickle, "math": math, "string": string}
    exec(cut(os.path.join(ref, "densephrases", "utils", "data_utils.py"), "whitespace_tokenize"), ns)
    exec(cut(os.path.join(ref, "densephrases", "utils", "squad_utils.py"), "TrueCaser"), ns)
    tables = pickle.load(open(os.path.join(T.GOLD, "truecase.dist"), "rb"))
    with tempfile.TemporaryDirectory() as tmp:
        p = os.path.join(tmp, "truecase.dist")                       # the reference indexes its count tables with []
        pickle.dump({k: (defaultdict(int, v) if k != "word_casing_lookup" else v) for k, v in tables.items()}, open(p, "wb"))
        tc = ns["TrueCaser"](p)
    cases, scores = T.truecase_differential_inputs(tables)
    return {"cases": [tc.get_true_case(s, oov) for s, oov in cases], "scores": [tc.get_score(*q) for q in scores]}


def main():
    ref = os.path.abspath(sys.argv[1])
    from oracle import ivfpq_ref as oracle
    oracle.build()
    out = {"eval_script_imports": eval_script_imports(ref), "evaluate": evaluate(ref), "search": search(ref, oracle), "qa_pairs": qa_pairs(ref),
           "options": options(ref), "truecase_differential": truecase_differential(ref)}
    path = os.path.join(T.GOLD, "reference_api.json")
    json.dump(jsonable(out), open(path, "w"), ensure_ascii=True)
    print(path, os.path.getsize(path))


if __name__ == "__main__":
    main()
