"""Encoder: the inference forwards of the DensePhrases encoder on the B200 tensor cores.

Mirror of /root/reference/densephrases/encoder.py (class Encoder):
  query side: `embed_query` (:101-118) and `forward(input_ids_=..., attention_mask_=..., token_type_ids_=..., return_query=True)`
    (:146-152) -> (query_start, query_end), each [B,1,768], computed by two independent BERT-base towers whose weights come from
    the `query_start_encoder.*` / `query_end_encoder.*` entries of the reference state dict;
  phrase side (towers='phrase' or 'all'): `embed_phrase` (:92-99) and `forward(input_ids=..., attention_mask=..., token_type_ids=...,
    return_phrase=True)` (:130-144) -> (start, end, filter_start_logits, filter_end_logits) from the `phrase_encoder.*` tower and
    `filter_linear`, plus `embed_phrase_int8`, the int8 `start` codes that write_phrases stores.
Legacy names `bert_q_start.*` / `bert_q_end.*` / `bert_start.*` are accepted like single_utils.backward_compat (:36-56).  The
training losses and the dump writer are out of scope (SURVEY.md 8a).  Compute: libdph_b200 (tcgen05 GEMMs and attention)."""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

LEGACY = {'bert_q_start': 'query_start_encoder', 'bert_q_end': 'query_end_encoder', 'bert_start': 'phrase_encoder'}
TOWERS = ('query_start_encoder', 'query_end_encoder')
PHRASE_TOWER = 'phrase_encoder'                  # tower 2 of libdph_b200
TOWER_SETS = {'query': (0, 1), 'phrase': (2,), 'all': (0, 1, 2)}


class BertGeometry(object):
    """The subset of HF BertConfig this path needs (SpanBERT-base-cased defaults, options.py:23)."""

    def __init__(self, vocab_size=28996, max_position_embeddings=512, type_vocab_size=2, hidden_size=768, num_hidden_layers=12,
                 num_attention_heads=12, intermediate_size=3072, **_):
        assert (hidden_size, num_hidden_layers, num_attention_heads, intermediate_size) == (768, 12, 12, 3072), \
            'only the BERT-base geometry of the released DensePhrases models is built'
        self.vocab_size, self.max_position_embeddings, self.type_vocab_size = vocab_size, max_position_embeddings, type_vocab_size
        self.hidden_size, self.num_hidden_layers = hidden_size, num_hidden_layers
        self.num_attention_heads, self.intermediate_size = num_attention_heads, intermediate_size


def tower_blob(sd, prefix, config):
    """Pack one tower's tensors into the flat fp32 blob libdph_b200 expects (layout documented in csrc/encoder.cu)."""
    def t(name):
        return sd[f'{prefix}.{name}'].detach().to(torch.float32).cpu().contiguous().view(-1)
    parts = [t('embeddings.word_embeddings.weight'), t('embeddings.position_embeddings.weight'), t('embeddings.token_type_embeddings.weight'),
             t('embeddings.LayerNorm.weight'), t('embeddings.LayerNorm.bias')]
    for l in range(config.num_hidden_layers):
        p = f'encoder.layer.{l}'
        parts += [t(f'{p}.attention.self.query.weight'), t(f'{p}.attention.self.key.weight'), t(f'{p}.attention.self.value.weight'),
                  t(f'{p}.attention.self.query.bias'), t(f'{p}.attention.self.key.bias'), t(f'{p}.attention.self.value.bias'),
                  t(f'{p}.attention.output.dense.weight'), t(f'{p}.attention.output.dense.bias'),
                  t(f'{p}.attention.output.LayerNorm.weight'), t(f'{p}.attention.output.LayerNorm.bias'),
                  t(f'{p}.intermediate.dense.weight'), t(f'{p}.intermediate.dense.bias'),
                  t(f'{p}.output.dense.weight'), t(f'{p}.output.dense.bias'), t(f'{p}.output.LayerNorm.weight'), t(f'{p}.output.LayerNorm.bias')]
    return torch.cat(parts).numpy()


class Encoder(object):
    """towers: 'query' (default; only the two query towers are loaded, even when the checkpoint holds the phrase tower), 'phrase'
    (phrase tower + filter head, like the reference after `del model.query_start_encoder`, single_utils.py:106-114) or 'all'."""

    def __init__(self, config, tokenizer=None, state_dict=None, device=0, precise='bf16x3', towers='query'):
        if towers not in TOWER_SETS:
            raise ValueError(f'towers must be one of {sorted(TOWER_SETS)}, not {towers!r}')
        self.towers = towers
        self.config = config if isinstance(config, BertGeometry) else BertGeometry(**{k: getattr(config, k) for k in
                                                                                     ('vocab_size', 'max_position_embeddings', 'type_vocab_size', 'hidden_size',
                                                                                      'num_hidden_layers', 'num_attention_heads', 'intermediate_size')})
        self.tokenizer = tokenizer
        self.device_index = device
        self.device = torch.device('cuda', device)
        self._h = C.c_void_p()
        L.check(L.lib().dph_encoder_create(C.byref(self._h), device, self.config.vocab_size, self.config.max_position_embeddings,
                                           self.config.type_vocab_size))
        self.training = False
        self.set_precision(precise)
        if state_dict is not None:
            self.load_state_dict(state_dict)

    def __del__(self):
        h, self._h = getattr(self, '_h', None), None
        if h and L is not None and L._lib is not None:
            L._lib.dph_encoder_free(h)

    MODES = {'tf32': 0, '3xtf32': 1, 'bf16x3': 2}      # name -> dph_encoder_set_precision argument

    def set_precision(self, precise):
        """'bf16x3' (default of this class): meets the north star's 1e-3 tolerance on the query vectors at nearly the speed of 'tf32';
        'tf32' / False: 1xTF32 GEMMs (== torch 1.9's default for fp32 matmuls on Ampere+), fastest, ~2e-2;
        '3xtf32' / True: 3xTF32 split, fp32-accurate; 'bf16x3': bf16 (hi, lo) planes, three bf16 MMAs per product -- both meet
        the 1e-3 tolerance of the north star, bf16x3 at the speed of 'tf32'."""
        mode = precise if isinstance(precise, str) else ('3xtf32' if precise else 'tf32')
        if mode not in self.MODES:
            raise ValueError(f'unknown precision mode {mode!r}; choose one of {sorted(self.MODES)}')
        self.mode = mode
        self.precise = mode != 'tf32'
        L.check(L.lib().dph_encoder_set_precision(self._h, self.MODES[mode]))

    def precision_modes(self):
        return list(self.MODES)

    @staticmethod
    def mma_multiplier(mode):
        """Tensor-core work issued per algorithmic flop, in TF32-MMA equivalents (a bf16 MMA costs half a TF32 one)."""
        return {'tf32': 1.0, '3xtf32': 3.0, 'bf16x3': 1.5}[mode]

    def default_mode(self):
        """The fastest mode that meets the north star's 1e-3 tolerance on the [CLS] vectors (tests/test_encoder.py)."""
        return 'bf16x3' if 'bf16x3' in self.MODES else '3xtf32'

    def set_attention(self, tensor_core=True):
        """True (default): tensor-core attention for S <= 64 in the 1xTF32 mode; False: fp32 SIMT attention always."""
        L.check(L.lib().dph_encoder_set_attention(self._h, int(bool(tensor_core))))

    # -- torch.nn.Module-style surface the callers touch (embed_utils.py:393, single_utils.py:116) --
    def eval(self):
        self.training = False
        return self

    def to(self, device):
        return self

    @property
    def has_query(self):
        return self.towers in ('query', 'all')

    @property
    def has_phrase(self):
        return self.towers in ('phrase', 'all')

    def load_state_dict(self, sd, strict=False):
        sd = {next((k.replace(old, new, 1) for old, new in LEGACY.items() if k.startswith(old)), k): v for k, v in sd.items()}
        need = L.lib().dph_encoder_tower_floats(self._h)
        for tower in TOWER_SETS[self.towers]:
            prefix = (TOWERS + (PHRASE_TOWER,))[tower]
            blob = np.ascontiguousarray(tower_blob(sd, prefix, self.config), dtype=np.float32)
            assert blob.size == need, f'{prefix}: {blob.size} floats, expected {need}'
            L.check(L.lib().dph_encoder_load_tower(self._h, tower, blob.ctypes.data_as(C.c_void_p), L.MEM_HOST))
        if self.has_phrase:
            W = np.ascontiguousarray(sd['filter_linear.weight'].detach().to(torch.float32).cpu().numpy())
            b = np.ascontiguousarray(sd['filter_linear.bias'].detach().to(torch.float32).cpu().numpy())
            assert W.shape == (2, self.config.hidden_size) and b.shape == (2,), 'filter_linear must be Linear(768, 2)'
            L.check(L.lib().dph_encoder_load_filter(self._h, W.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), L.MEM_HOST))
        return self

    def _check_ids(self, input_ids, token_type_ids):
        if not input_ids.is_cuda:      # ids normally come from the CPU tokenizer: range check before the copy (torch.nn.Embedding raises IndexError)
            if int(input_ids.min()) < 0 or int(input_ids.max()) >= self.config.vocab_size:
                raise IndexError(f'input_ids outside [0, {self.config.vocab_size})')
            if int(token_type_ids.min()) < 0 or int(token_type_ids.max()) >= self.config.type_vocab_size:
                raise IndexError(f'token_type_ids outside [0, {self.config.type_vocab_size})')

    def embed_query(self, input_ids_, attention_mask_, token_type_ids_):
        """int64 [B,S] tensors (cuda or cpu) -> (query_start, query_end) float32 [B,1,768] on the GPU."""
        if not self.has_query:
            raise NotImplementedError("this Encoder was built with towers='phrase': the query towers are not loaded")
        B, S = input_ids_.shape
        self._check_ids(input_ids_, token_type_ids_)
        ids, mask, tt = (x.to(self.device, dtype=torch.int64).contiguous() for x in (input_ids_, attention_mask_, token_type_ids_))
        start = torch.empty((B, 1, self.config.hidden_size), dtype=torch.float32, device=self.device)
        end = torch.empty_like(start)
        L.check(L.lib().dph_encoder_set_stream(self._h, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        L.check(L.lib().dph_encoder_embed_query(self._h, ids.data_ptr(), mask.data_ptr(), tt.data_ptr(), B, S, start.data_ptr(), end.data_ptr(),
                                                L.MEM_DEVICE))
        return start, end

    def _phrase(self, input_ids, attention_mask, token_type_ids, want_float, want_int8, dense_offset=-2.0, dense_scale=20.0):
        if not self.has_phrase:
            raise NotImplementedError("the phrase tower is not loaded: build the Encoder with towers='phrase' or 'all'")
        assert len(input_ids.size()) == 2
        B, S = input_ids.shape
        self._check_ids(input_ids, token_type_ids)
        ids, mask, tt = (x.to(self.device, dtype=torch.int64).contiguous() for x in (input_ids, attention_mask, token_type_ids))
        out = torch.empty((B, S, self.config.hidden_size), dtype=torch.float32, device=self.device) if want_float else None
        q = torch.empty((B, S, self.config.hidden_size), dtype=torch.int8, device=self.device) if want_int8 else None
        fs = torch.empty((B, S), dtype=torch.float32, device=self.device)
        fe = torch.empty_like(fs)
        L.check(L.lib().dph_encoder_set_stream(self._h, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        L.check(L.lib().dph_encoder_embed_phrase(self._h, ids.data_ptr(), mask.data_ptr(), tt.data_ptr(), B, S,
                                                 out.data_ptr() if want_float else None, fs.data_ptr(), fe.data_ptr(),
                                                 q.data_ptr() if want_int8 else None, float(dense_offset), float(dense_scale), L.MEM_DEVICE))
        return out, q, fs, fe

    def embed_phrase(self, input_ids, attention_mask, token_type_ids):
        """int64 [B,S] tensors (cuda or cpu), S <= 512 -> (start, end) float32 [B,S,768] on the GPU, the phrase tower's last hidden
        state; like the reference (encoder.py:92-99) start and end are the same tensor."""
        out, _, _, _ = self._phrase(input_ids, attention_mask, token_type_ids, True, False)
        return out, out

    def embed_phrase_int8(self, input_ids, attention_mask, token_type_ids, dense_offset=-2, dense_scale=20):
        """-> (start_int8 [B,S,768] int8, filter_start [B,S], filter_end [B,S]) on the GPU: the codes write_phrases stores,
        float_to_int8(start, dense_offset, dense_scale) (embed_utils.py:141-145; defaults options.py:144-145), and the filter logits,
        computed in the same pass without the fp32 vectors."""
        _, q, fs, fe = self._phrase(input_ids, attention_mask, token_type_ids, False, True, dense_offset, dense_scale)
        return q, fs, fe

    def forward(self, input_ids=None, attention_mask=None, token_type_ids=None, input_ids_=None, attention_mask_=None, token_type_ids_=None,
                return_phrase=False, return_query=False, **unused):
        if return_phrase and not return_query and input_ids is not None and input_ids_ is None and self.has_phrase:
            out, _, fs, fe = self._phrase(input_ids, attention_mask, token_type_ids, True, False)
            return out, out, fs, fe                     # (start, end, filter_start_logits, filter_end_logits), encoder.py:143-144
        if input_ids is not None or not return_query:
            raise NotImplementedError('only the inference paths (return_query=True, encoder.py:146-152; return_phrase=True with the '
                                      'phrase tower loaded, :130-144) are on the B200 hot path')
        assert len(input_ids_.size()) == 2
        return self.embed_query(input_ids_, attention_mask_, token_type_ids_)

    __call__ = forward


def random_state_dict(config, seed, prefixes=TOWERS, std=0.02):
    """Seeded random weights in the reference's state-dict naming (no checkpoint is reachable offline).  LayerNorm gains
    are 1 + noise and biases are noise so every parameter matters in parity tests."""
    g = torch.Generator().manual_seed(seed)
    H, FF = config.hidden_size, config.intermediate_size

    def rn(*shape, s=std):
        return torch.randn(*shape, generator=g) * s

    sd = {}
    for prefix in prefixes:
        sd[f'{prefix}.embeddings.word_embeddings.weight'] = rn(config.vocab_size, H)
        sd[f'{prefix}.embeddings.position_embeddings.weight'] = rn(config.max_position_embeddings, H)
        sd[f'{prefix}.embeddings.token_type_embeddings.weight'] = rn(config.type_vocab_size, H)
        sd[f'{prefix}.embeddings.LayerNorm.weight'] = 1.0 + rn(H, s=0.1)
        sd[f'{prefix}.embeddings.LayerNorm.bias'] = rn(H, s=0.1)
        for l in range(config.num_hidden_layers):
            p = f'{prefix}.encoder.layer.{l}'
            for name, shape in (('attention.self.query', (H, H)), ('attention.self.key', (H, H)), ('attention.self.value', (H, H)),
                                ('attention.output.dense', (H, H)), ('intermediate.dense', (FF, H)), ('output.dense', (H, FF))):
                sd[f'{p}.{name}.weight'] = rn(*shape, s=0.04)
                sd[f'{p}.{name}.bias'] = rn(shape[0], s=0.05)
            for name in ('attention.output.LayerNorm', 'output.LayerNorm'):
                sd[f'{p}.{name}.weight'] = 1.0 + rn(H, s=0.1)
                sd[f'{p}.{name}.bias'] = rn(H, s=0.1)
    return sd


def random_filter_state_dict(config, seed, std=0.02):
    """Seeded random `filter_linear` (Linear(768, 2)) weights, from their own generator so random_state_dict's stream is untouched;
    std 0.02 is the reference's init range (Encoder.init_weights), the bias is noise so it matters in parity tests."""
    g = torch.Generator().manual_seed(seed)
    return {'filter_linear.weight': torch.randn(2, config.hidden_size, generator=g) * std,
            'filter_linear.bias': torch.randn(2, generator=g) * 0.1}


def synthetic_context_batch(B, S, vocab_size, seed):
    """Context-side inputs as the dump builds them: [CLS] title [SEP] context [SEP], ragged real lengths (in a batch of several rows
    the first fills S, every other row is padded), zero padding; token type 0 for [CLS] title [SEP] and 1 for the context part, so
    the type embedding is exercised."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.zeros((B, S), dtype=torch.int64)
    mask = torch.zeros((B, S), dtype=torch.int64)
    tt = torch.zeros((B, S), dtype=torch.int64)
    for b in range(B):
        n = S if (b == 0 and B > 1) or S == 1 else int(torch.randint(max(1, S // 3), S, (1,), generator=g))     # real tokens of this row
        ids[b, 0] = 101
        if n >= 2:
            ids[b, n - 1] = 102
        title = min(int(torch.randint(1, 9, (1,), generator=g)), max(0, n - 3))
        ids[b, 1:1 + title] = torch.randint(1000, vocab_size, (title,), generator=g)
        if n >= 3:
            ids[b, 1 + title] = 102
        body = max(0, n - 3 - title)
        ids[b, 2 + title:2 + title + body] = torch.randint(1000, vocab_size, (body,), generator=g)
        tt[b, 2 + title:n] = 1
        mask[b, :n] = 1
    return ids, mask, tt


def synthetic_query_batch(B, S, vocab_size, seed):
    """SURVEY 8d: uniform token ids, 6-20 real tokens + [CLS]/[SEP] (ids 101/102), zero padding to S, all token types 0."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.zeros((B, S), dtype=torch.int64)
    mask = torch.zeros((B, S), dtype=torch.int64)
    for b in range(B):
        n = int(torch.randint(6, 21, (1,), generator=g))
        n = min(n, S - 2)
        ids[b, 0] = 101
        ids[b, 1:1 + n] = torch.randint(1000, vocab_size, (n,), generator=g)
        ids[b, 1 + n] = 102
        mask[b, :n + 2] = 1
    return ids, mask, torch.zeros_like(ids)
