"""Plain PyTorch fp32 restatement of the phrase side of Encoder.forward(input_ids=..., return_phrase=True)
(/root/reference/densephrases/encoder.py:92-99, 130-144), built on the query oracle's tower_forward (oracle/encoder_ref.py),
and of the int8 dump codes of write_phrases.  Pinned against the reference class by tests/golden/encoder_phrase.npz
(tests/golden/make_phrase_golden.py), so it can stand in for the reference on the GPU machine."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle.encoder_ref import tower_forward


def embed_phrase(sd, ids, mask, tt):
    """-> (start [B,S,768], end (the same tensor), filter_start_logits [B,S], filter_end_logits [B,S]), fp32 on ids.device."""
    with torch.no_grad():
        start = tower_forward(sd, 'phrase_encoder', ids, mask, tt)
        logits = F.linear(start, sd['filter_linear.weight'].to(ids.device, torch.float32), sd['filter_linear.bias'].to(ids.device, torch.float32))
    return start, start, logits[..., 0], logits[..., 1]


def float_to_int8(x, offset, scale):
    """The int8 codes write_phrases stores (embed_utils.py:141-145): (x - offset) * scale on fp32 data, each step rounded to fp32,
    clipped to [-128, 127], rounded half to even, as int8.  x: numpy array or tensor -> numpy int8 array."""
    x = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    t = (x.astype(np.float32, copy=False) - np.float32(offset)) * np.float32(scale)
    return np.rint(np.clip(t, np.float32(-128), np.float32(127))).astype(np.int8)
