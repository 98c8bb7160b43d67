"""Generates tests/golden/encoder_phrase.npz by running the UNMODIFIED reference class
/root/reference/densephrases/encoder.py:Encoder (fp32, CPU, eager) with return_phrase=True on seeded random weights
(densephrases_b200.encoder.random_state_dict with prefixes=('phrase_encoder',) + random_filter_state_dict) and
synthetic_context_batch inputs.  Stored: inputs, seeds, all filter logits, and the start vectors at a seeded subset of positions
(always position 0, the last real token and a padded position) to keep the file small; the weights are regenerated from the seeds.
Run in the build container (needs /root/reference):  python tests/golden/make_phrase_golden.py"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from densephrases_b200.encoder import BertGeometry, random_filter_state_dict, random_state_dict, synthetic_context_batch  # noqa: E402
from tests import phrase_oracle  # noqa: E402
from tests.golden.make_encoder_golden import load_reference_encoder  # noqa: E402

CASES = {'b3_s40': (3, 40, 8), 'b2_s200': (2, 200, 16), 'b1_s512': (1, 512, 32)}      # name -> (B, S, stored positions per row)


def positions(mask, per_row, seed):
    """[B, per_row] sorted positions per row: 0, the last real token, the first padded position, the rest seeded."""
    g = np.random.default_rng(seed)
    out = []
    for row in mask:
        n, S = int(row.sum()), len(row)
        fixed = {0, n - 1} | ({n} if n < S else set())
        rest = g.choice(np.setdiff1d(np.arange(S), sorted(fixed)), per_row - len(fixed), replace=False)
        out.append(np.sort(np.concatenate([sorted(fixed), rest])))
    return np.stack(out).astype(np.int64)


if __name__ == '__main__':
    from transformers import BertConfig, BertModel
    torch.manual_seed(0)
    seed, filter_seed, vocab = 20261017, 20261018, 28996
    geo = BertGeometry(vocab_size=vocab)
    cfg = BertConfig(vocab_size=vocab, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                     max_position_embeddings=512, type_vocab_size=2, layer_norm_eps=1e-12, hidden_act='gelu',
                     hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
    RefEncoder = load_reference_encoder()
    model = RefEncoder(cfg, tokenizer=None, transformer_cls=BertModel).eval()
    sd = random_state_dict(geo, seed, prefixes=('phrase_encoder',))
    sd.update(random_filter_state_dict(geo, filter_seed))
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all(not m.startswith(('phrase_encoder.encoder', 'phrase_encoder.embeddings.word', 'filter_linear')) for m in missing), missing
    out = {}
    for name, (B, S, per_row) in CASES.items():
        ids, mask, tt = synthetic_context_batch(B, S, vocab, seed + S)
        with torch.no_grad():
            start, end, fs, fe = model(input_ids=ids, attention_mask=mask, token_type_ids=tt, return_phrase=True)
        assert start is end or torch.equal(start, end)
        rs, _, rfs, rfe = phrase_oracle.embed_phrase(sd, ids, mask, tt)
        d = max((start - rs).abs().max().item(), (fs - rfs).abs().max().item(), (fe - rfe).abs().max().item())
        print(name, 'reference class vs torch restatement: max abs diff', d, '| out scale', start.abs().mean().item(),
              '| filter scale', fs.abs().mean().item())
        assert d < 2e-4, d
        pos = positions(mask.numpy(), per_row, seed + S)
        out[f'{name}_ids'], out[f'{name}_mask'], out[f'{name}_tt'] = ids.numpy(), mask.numpy(), tt.numpy()
        out[f'{name}_pos'] = pos
        out[f'{name}_start'] = np.take_along_axis(start.numpy(), pos[:, :, None], axis=1)
        out[f'{name}_fs'], out[f'{name}_fe'] = fs.numpy(), fe.numpy()
    out['seed'], out['filter_seed'], out['vocab'] = np.array(seed), np.array(filter_seed), np.array(vocab)
    path = os.path.join(ROOT, 'tests', 'golden', 'encoder_phrase.npz')
    np.savez_compressed(path, **out)
    print('wrote tests/golden/encoder_phrase.npz,', os.path.getsize(path), 'bytes')
