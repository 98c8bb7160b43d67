"""Glue between strings and the two CUDA kernels families: the reference's L2/L3 layers (SURVEY.md 1) re-stated for this
package.  Same function names, arguments and return shapes as
  densephrases/utils/open_utils.py  load_phrase_index :26-43, get_query2vec :83-101, load_qa_pairs :104-160
  densephrases/utils/single_utils.py load_encoder :59-118
  densephrases/utils/eval_utils.py  metrics :9-86
  densephrases/model.py             DensePhrases :14-128
  eval_phrase_retrieval.py          embed_all_query :33-46, evaluate :49-91 (the search loop; scoring reduced to EM/F1@1,k)
so the reference's drivers keep working; what changed is where the arithmetic runs."""
import json
import logging
import os
import random
import re
import string
import unicodedata
from collections import Counter

import numpy as np
import torch

from .encoder import BertGeometry, Encoder, random_filter_state_dict, random_state_dict
from .mips import MIPS
from .options import Options
from .tokenization import WordPieceTokenizer
from .truecase import TrueCaser, truecase_questions

logger = logging.getLogger(__name__)
_truecaser = None          # open_utils.py:23: one truecaser per process, loaded on first use


# ---- eval_utils ------------------------------------------------------------------------------------------
def normalize_answer(s):
    s = ''.join(ch for ch in s.lower() if ch not in set(string.punctuation))
    return ' '.join(re.sub(r'\b(a|an|the)\b', ' ', s).split())


def f1_score(prediction, ground_truth):
    p, g = normalize_answer(prediction), normalize_answer(ground_truth)
    if (p in ('yes', 'no', 'noanswer') or g in ('yes', 'no', 'noanswer')) and p != g:
        return (0, 0, 0)
    pt, gt = p.split(), g.split()
    same = sum((Counter(pt) & Counter(gt)).values())
    if same == 0:
        return (0, 0, 0)
    precision, recall = same / len(pt), same / len(gt)
    return 2 * precision * recall / (precision + recall), precision, recall


def exact_match_score(prediction, ground_truth):
    return normalize_answer(prediction) == normalize_answer(ground_truth)


def drqa_normalize(text):
    return unicodedata.normalize('NFD', text)


def drqa_exact_match_score(prediction, ground_truth):
    return normalize_answer(prediction) == normalize_answer(ground_truth)


def drqa_regex_match_score(prediction, pattern):
    try:
        compiled = re.compile(pattern, flags=re.IGNORECASE + re.UNICODE + re.MULTILINE)
    except BaseException:
        return False
    return compiled.match(prediction) is not None


def drqa_metric_max_over_ground_truths(metric_fn, prediction, ground_truths):
    return max(metric_fn(prediction, gt) for gt in ground_truths)


# ---- single_utils.backward_compat / load_encoder ----------------------------------------------------------------
def backward_compat(model_dict):
    """Old checkpoint names -> current ones, teacher / reader heads dropped (single_utils.py:36-56)."""
    dropped = ('cross_encoder', 'bert_qd', 'qa_outputs')
    renamed = (('bert_start', 'phrase_encoder'), ('bert_q_start', 'query_start_encoder'), ('bert_q_end', 'query_end_encoder'))
    out = {}
    for key, val in model_dict.items():
        if key.startswith(dropped):
            continue
        hits = [(old, new) for old, new in renamed if key.startswith(old)]
        if not hits:
            out[key] = val
        for old, new in hits:
            out[key.replace(old, new)] = val
    return out


def _find_vocab(args, load_dir):
    """vocab.txt the way the reference resolves its tokenizer (single_utils.py:72-77): `tokenizer_name`, else
    `pretrained_name_or_path`, looked up as a directory / file and under `cache_dir`; `load_dir` last (a fine-tuned checkpoint
    directory usually carries its own copy)."""
    cands = []
    for name in (getattr(args, 'tokenizer_name', None), getattr(args, 'pretrained_name_or_path', None)):
        if not name:
            continue
        cands += [name, os.path.join(name, 'vocab.txt')]
        cache = getattr(args, 'cache_dir', None)
        if cache:
            cands += [os.path.join(cache, name, 'vocab.txt'), os.path.join(cache, name.replace('/', '--'), 'vocab.txt'),
                      os.path.join(cache, os.path.basename(name), 'vocab.txt')]
    if load_dir:
        cands.append(os.path.join(load_dir, 'vocab.txt'))
    for c in cands:
        if os.path.isfile(c) and c.endswith('.txt'):
            return c
    return None


def load_encoder(device, args, phrase_only=False):
    """-> (model, tokenizer, config) from `args.load_dir/pytorch_model.bin` + a WordPiece `vocab.txt` (single_utils.py:59-118).
    A missing checkpoint or vocabulary raises FileNotFoundError like the reference does; seeded random weights and the
    synthetic character-level vocabulary are used only when the caller opts in with `args.allow_random_init = True` or the
    environment variable DPH_ALLOW_RANDOM_INIT=1 (tests and benchmarks: no checkpoint is reachable offline).
    phrase_only=True (generate_phrase_vecs.py): the phrase tower and the filter head only, like the reference's
    `del model.query_start_encoder` / `del model.query_end_encoder` (single_utils.py:106-114)."""
    load_dir = getattr(args, 'load_dir', '') or ''
    allow_random = bool(getattr(args, 'allow_random_init', False)) or os.environ.get('DPH_ALLOW_RANDOM_INIT', '') == '1'
    config = BertGeometry()
    cfg_json = os.path.join(load_dir, 'config.json')
    if os.path.exists(cfg_json):
        config = BertGeometry(**json.load(open(cfg_json)))
    vocab_file = _find_vocab(args, load_dir)
    if vocab_file is not None:
        tokenizer = WordPieceTokenizer.from_vocab_file(vocab_file, do_lower_case=getattr(args, 'do_lower_case', False))
    elif allow_random:
        tokenizer = WordPieceTokenizer.from_pretrained_or_synthetic(None, do_lower_case=getattr(args, 'do_lower_case', False),
                                                                   vocab_size=config.vocab_size)
        logger.warning('no vocab.txt found: synthetic character-level WordPiece vocabulary (allow_random_init)')
    else:
        raise FileNotFoundError(f'no vocab.txt for the tokenizer (tokenizer_name / pretrained_name_or_path / cache_dir / load_dir={load_dir!r}); '
                                'pass allow_random_init=True for a synthetic vocabulary')
    if len(tokenizer.vocab) > config.vocab_size or max(tokenizer.vocab.values()) >= config.vocab_size:
        raise ValueError(f'vocabulary has ids up to {max(tokenizer.vocab.values())} but the encoder embeds {config.vocab_size} rows')
    ckpt = os.path.join(load_dir, 'pytorch_model.bin')
    if os.path.exists(ckpt):
        sd = backward_compat(torch.load(ckpt, map_location='cpu'))
        logger.info(f'DensePhrases encoder loaded from {load_dir}')
    elif allow_random:
        seed = getattr(args, 'seed', 42)
        if phrase_only:
            sd = random_state_dict(config, seed, prefixes=('phrase_encoder',))
            sd.update(random_filter_state_dict(config, seed))
        else:
            sd = random_state_dict(config, seed)
        logger.warning('no checkpoint found: encoder initialised with seeded random weights (allow_random_init)')
    else:
        raise FileNotFoundError(f'{ckpt} not found (hub ids are not resolvable offline); pass allow_random_init=True for seeded random weights')
    dev_index = torch.cuda.current_device() if str(device).startswith('cuda') else 0
    model = Encoder(config, tokenizer=tokenizer, state_dict=sd, device=dev_index, towers='phrase' if phrase_only else 'query')
    return model, tokenizer, config


# ---- open_utils ------------------------------------------------------------------------------------------------
def load_phrase_index(args, ignore_logging=False):
    phrase_dump_dir = os.path.join(args.dump_dir, args.phrase_dir)
    index_dir = os.path.join(args.dump_dir, args.index_name)
    return MIPS(phrase_dump_dir=phrase_dump_dir, index_path=os.path.join(index_dir, args.index_path),
                idx2id_path=os.path.join(index_dir, args.idx2id_path), cuda=args.cuda,
                logging_level=logging.WARNING if ignore_logging else (logging.DEBUG if args.verbose_logging else logging.INFO))


def get_query2vec(query_encoder, tokenizer, args, batch_size=64):
    """-> query2vec(list[str]) -> list of (start_vec [1][768] list, end_vec [1][768] list, tokens) like open_utils.py:85-100.
    The returned function also carries `query2vec.tensors(list[str]) -> (start [n,768], end [n,768] torch tensors on the encoder's
    device, tokens)`: the same vectors without the per-question Python lists of the reference's contract (768 floats -> list -> back
    to an array costs more than the encoder forward); DensePhrases.search and embed_all_query use it (SURVEY.md 8f #3)."""
    def encode(queries):
        for i in range(0, len(queries), batch_size):
            feats = [tokenizer.encode_question(q, args.max_query_length) for q in queries[i:i + batch_size]]
            ids, mask, tt = (torch.tensor([f[j] for f in feats], dtype=torch.int64) for j in range(3))
            with torch.no_grad():
                start, end = query_encoder(input_ids_=ids, attention_mask_=mask, token_type_ids_=tt, return_query=True)
            yield start, end, feats

    def query2vec(queries):
        outs = []
        for start, end, feats in encode(queries):
            start, end = start.cpu().numpy(), end.cpu().numpy()       # one device->host copy per batch (reference: one per row)
            outs += [(start[j].tolist(), end[j].tolist(), feats[j][3]) for j in range(len(feats))]
        return outs

    def tensors(queries):
        starts, ends, toks = [], [], []
        for start, end, feats in encode(queries):
            starts.append(start[:, 0]); ends.append(end[:, 0]); toks += [f[3] for f in feats]
        if not starts:
            z = torch.zeros((0, 768), dtype=torch.float32)
            return z, z, toks
        return torch.cat(starts, 0), torch.cat(ends, 0), toks
    query2vec.tensors = tensors
    return query2vec


def load_qa_pairs(data_path, args, q_idx=None, draft_num_examples=100, shuffle=False):
    q_ids, questions, answers, titles = [], [], [], []
    for data_idx, item in enumerate(json.load(open(data_path))['data']):
        if q_idx is not None and data_idx != q_idx:
            continue
        if len(item['answers']) == 0:
            continue
        q_id = item['id'] if 'origin' not in item else item['origin'].split('.')[0] + '-' + item['id']
        question = item['question']
        if '[START_ENT]' in question:
            question = question[max(question.index('[START_ENT]') - 300, 0):question.index('[END_ENT]') + 300]
        q_ids.append(q_id)
        questions.append(question[:-1] if question.endswith('?') else question)
        answers.append(item['answers'])
        titles.append(item.get('titles', ['']))
    if getattr(args, 'do_lower_case', False):
        questions = [q.lower() for q in questions]
    if shuffle:
        pack = list(zip(q_ids, questions, answers, titles))
        random.shuffle(pack)
        q_ids, questions, answers, titles = map(list, zip(*pack))
    if getattr(args, 'draft', False):
        q_ids, questions, answers, titles = (x[:draft_num_examples] for x in (q_ids, questions, answers, titles))
    if getattr(args, 'truecase', False):            # open_utils.py:147-156: a missing statistics file is reported, not fatal
        try:
            global _truecaser
            if _truecaser is None:
                logger.info('loading truecaser')
                _truecaser = TrueCaser(os.path.join(os.environ['DATA_DIR'], args.truecase_path))
            logger.info('Truecasing queries')
            questions = truecase_questions(_truecaser, questions)
        except Exception as e:
            print(e)
    logger.info(f'Loading {len(questions)} questions from {data_path}')
    return q_ids, questions, answers, titles


# ---- eval_phrase_retrieval ---------------------------------------------------------------------------------------
def embed_all_query(questions, args, query_encoder, tokenizer, batch_size=64):
    query2vec = get_query2vec(query_encoder=query_encoder, tokenizer=tokenizer, args=args, batch_size=batch_size)
    # open_utils.py:103-117 concatenates the per-question lists; the same array (float64 like an array built from Python floats, same
    # values) comes from one device->host copy per batch
    start, end, _ = query2vec.tensors(questions)
    return np.concatenate([start.cpu().numpy(), end.cpu().numpy()], 1).astype(np.float64)


def evaluate(args, mips=None, query_encoder=None, tokenizer=None, q_idx=None):
    """The search loop of eval_phrase_retrieval.evaluate (:49-91) + EM/F1 at 1 and top_k."""
    qids, questions, answers, _ = load_qa_pairs(args.test_path, args, q_idx)
    if query_encoder is None:
        query_encoder, tokenizer, _ = load_encoder('cuda' if args.cuda else 'cpu', args)
    query_vec = embed_all_query(questions, args, query_encoder, tokenizer)
    if mips is None:
        mips = load_phrase_index(args)
    step = args.eval_batch_size
    predictions, scores = [], []
    for i in range(0, len(questions), step):
        result = mips.search(query_vec[i:i + step], q_texts=questions[i:i + step], nprobe=args.nprobe, top_k=args.top_k,
                             max_answer_length=args.max_answer_length, aggregate=args.aggregate, agg_strat=args.agg_strat,
                             return_sent=args.return_sent)
        predictions += [[r['answer'] for r in out][:args.top_k] if len(out) > 0 else [''] for out in result]
        scores += [[r['score'] for r in out][:args.top_k] if len(out) > 0 else [-1e10] for out in result]
    em1 = np.mean([max(exact_match_score(p[0], a) for a in ans) for p, ans in zip(predictions, answers)])
    f11 = np.mean([max(f1_score(p[0], a)[0] for a in ans) for p, ans in zip(predictions, answers)])
    emk = np.mean([max(exact_match_score(pp, a) for pp in p for a in ans) for p, ans in zip(predictions, answers)])
    f1k = np.mean([max(f1_score(pp, a)[0] for pp in p for a in ans) for p, ans in zip(predictions, answers)])
    logger.info(f'exact_match_top1 {100*em1:.2f} f1_score_top1 {100*f11:.2f} | exact_match_top{args.top_k} {100*emk:.2f} f1 {100*f1k:.2f}')
    return {'exact_match_top1': em1, 'f1_score_top1': f11, f'exact_match_top{args.top_k}': emk, f'f1_score_top{args.top_k}': f1k,
            'predictions': predictions, 'scores': scores}


# ---- model.DensePhrases ----------------------------------------------------------------------------------------------
class DensePhrases(object):
    _AGG = {'phrase': 'opt1', 'sentence': 'opt2', 'paragraph': 'opt2', 'document': 'opt3'}

    def __init__(self, load_dir, dump_dir, index_name='start/1048576_flat_OPQ96', device='cuda', verbose=False, mips=None, **kwargs):
        # kwargs land in args; allow_random_init=True opts into seeded random weights / synthetic vocabulary (tests, benchmarks)
        options = Options()
        options.add_model_options(); options.add_index_options(); options.add_retrieval_options(); options.add_data_options()
        self.args = options.parse([])            # the reference parses the live sys.argv here (model.py:30-35); we do not
        self.args.load_dir, self.args.dump_dir, self.args.index_name = load_dir, dump_dir, index_name
        self.args.cache_dir = os.environ.get('CACHE_DIR', '')
        self.args.cuda = device == 'cuda'
        self.args.__dict__.update(kwargs)
        self.set_encoder(load_dir, device)
        self.mips = mips if mips is not None else load_phrase_index(self.args, ignore_logging=not verbose)
        # model.py:52 loads $DATA_DIR/<truecase_path> unconditionally; here a missing statistics file only disables truecasing
        # (search(truecase=True) then leaves the queries as typed) -- pass truecase_path=... / set DATA_DIR to enable it
        tc_path = os.path.join(os.environ.get('DATA_DIR', ''), self.args.truecase_path)
        self.truecase = TrueCaser(tc_path) if os.path.exists(tc_path) else None
        if self.truecase is None:
            logger.warning(f'truecaser statistics {tc_path} not found: lower-case queries are searched as typed')

    def set_encoder(self, load_dir, device='cuda'):
        self.args.load_dir = load_dir
        self.model, self.tokenizer, self.config = load_encoder(device, self.args)
        self.query2vec = get_query2vec(query_encoder=self.model, tokenizer=self.tokenizer, args=self.args, batch_size=64)

    def evaluate(self, test_path, **kwargs):
        """model.py:118-128: run the evaluation loop of eval_phrase_retrieval.py on `test_path` with this model's index and encoder.
        The reference imports `evaluate` from the script on its path; when that module is importable it is used unmodified, else
        this package's restatement of the same loop (runtime.evaluate)."""
        import copy
        new_args = copy.deepcopy(self.args)
        new_args.test_path = test_path
        new_args.truecase = True
        new_args.__dict__.update(kwargs)
        try:
            from eval_phrase_retrieval import evaluate as evaluate_fn
        except ImportError:
            evaluate_fn = evaluate
        return evaluate_fn(new_args, self.mips, self.model, self.tokenizer)

    def search(self, query='', retrieval_unit='phrase', top_k=10, truecase=True, return_meta=False):
        single = isinstance(query, str)
        batch_query = [query] if single else query
        assert isinstance(batch_query, list)
        if retrieval_unit not in self._AGG:
            raise NotImplementedError(f'"{retrieval_unit}" not supported. Choose one of {self._AGG.keys()}.')
        if truecase and self.truecase is not None:
            # model.py:66-70 binds the truecased list to `query` and then encodes `batch_query`: in the reference the truecased text
            # never reaches the encoder or the result dicts.  Reproduced as is (same results on the same inputs); the evaluation
            # path (load_qa_pairs, open_utils.py:147-154) does use the truecased questions.
            query = truecase_questions(self.truecase, batch_query)
        if hasattr(self.query2vec, 'tensors'):        # encoder output stays a tensor on its device until the index has searched it
            start, end, _ = self.query2vec.tensors(batch_query)
            query_vec = torch.cat([start, end], 1)
        else:                                         # a caller-supplied query2vec with the reference's list contract (model.py:69-73)
            outs = self.query2vec(batch_query)
            query_vec = np.concatenate([np.concatenate([o[0] for o in outs], 0), np.concatenate([o[1] for o in outs], 0)], 1)
        search_top_k = top_k * 2 if retrieval_unit in ('sentence', 'paragraph', 'document') else top_k
        rets = self.mips.search(query_vec, q_texts=batch_query, nprobe=256, top_k=search_top_k, max_answer_length=10, return_idxs=False,
                                aggregate=True, agg_strat=self._AGG[retrieval_unit], return_sent=retrieval_unit == 'sentence')
        rets = [ret[:top_k] for ret in rets]
        field = {'phrase': lambda r: r['answer'], 'sentence': lambda r: r['context'], 'paragraph': lambda r: r['context'],
                 'document': lambda r: r['title'][0]}[retrieval_unit]
        retrieved = [[field(r) for r in ret][:top_k] for ret in rets]
        if single:
            rets, retrieved = rets[0], retrieved[0]
        return (retrieved, rets) if return_meta else retrieved
