"""Phrase encoder (Encoder.forward(input_ids=..., return_phrase=True), embed_phrase_int8) and the long-sequence tensor-core attention.
Oracle chain: UNMODIFIED reference Encoder (run in the build container by tests/golden/make_phrase_golden.py) -> committed fixture
tests/golden/encoder_phrase.npz -> (CPU test) the torch fp32 restatement tests/phrase_oracle.py reproduces it -> (GPU tests) the
CUDA phrase forward is compared with both.

Tolerances: 'bf16x3' and '3xtf32' are fp32-accurate (max |diff| < 1e-3 on start vectors and filter logits); 'tf32' (one TF32 MMA
per product) < 5e-2 with per-token cosine > 0.9995, the bounds of the query encoder tests."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from tests import phrase_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "encoder_phrase.npz")
QUERY_GOLD = os.path.join(ROOT, "tests", "golden", "encoder_query.npz")
CASES = ["b3_s40", "b2_s200", "b1_s512"]
TOL = {"tf32": 5e-2, "3xtf32": 1e-3, "bf16x3": 1e-3}


def load_case(name):
    g = np.load(GOLD)
    t = lambda k: torch.from_numpy(g[f"{name}_{k}"])
    return int(g["seed"]), int(g["filter_seed"]), int(g["vocab"]), t("ids"), t("mask"), t("tt"), t("pos"), t("start"), t("fs"), t("fe")


def phrase_sd(geo, seed, filter_seed):
    from densephrases_b200.encoder import random_filter_state_dict, random_state_dict
    sd = random_state_dict(geo, seed, prefixes=("phrase_encoder",))
    sd.update(random_filter_state_dict(geo, filter_seed))
    return sd


def cos(a, b):
    return torch.nn.functional.cosine_similarity(a.reshape(-1, a.shape[-1]), b.reshape(-1, b.shape[-1]), dim=1)


# ---- CPU ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CASES)
def test_torch_restatement_reproduces_reference_phrase_fixture(name):
    from densephrases_b200.encoder import BertGeometry
    seed, fseed, vocab, ids, mask, tt, pos, start, fs, fe = load_case(name)
    s, e, rfs, rfe = phrase_oracle.embed_phrase(phrase_sd(BertGeometry(vocab_size=vocab), seed, fseed), ids, mask, tt)
    assert s is e and s.shape == ids.shape + (768,)
    got = torch.take_along_dim(s, pos[:, :, None], dim=1)
    assert (got - start).abs().max() < 2e-4
    assert (rfs - fs).abs().max() < 2e-4 and (rfe - fe).abs().max() < 2e-4
    assert (fs - fe).abs().max() > 0.05                      # the two filter rows really are different


def test_fixture_positions_cover_first_last_and_padding():
    g = np.load(GOLD)
    assert os.path.getsize(GOLD) < 1 << 20
    for name in CASES:
        mask, pos = g[f"{name}_mask"], g[f"{name}_pos"]
        assert (mask[:, 1:] <= mask[:, :-1]).all() and (g[f"{name}_tt"] == 1).any()
        for row, p in zip(mask, pos):
            n = int(row.sum())
            assert 0 in p and n - 1 in p
        assert any(int(row.sum()) in p for row, p in zip(mask, pos)), "no padded position stored"


def test_phrase_tower_blob_and_legacy_names():
    from densephrases_b200.encoder import LEGACY, BertGeometry, random_state_dict, tower_blob
    geo = BertGeometry(vocab_size=1000)
    sd = random_state_dict(geo, 1, prefixes=("phrase_encoder",))
    per_layer = 3 * 768 * 768 + 3 * 768 + 768 * 768 + 768 + 2 * 768 + 3072 * 768 + 3072 + 768 * 3072 + 768 + 2 * 768
    assert tower_blob(sd, "phrase_encoder", geo).size == 1000 * 768 + 512 * 768 + 2 * 768 + 2 * 768 + 12 * per_layer
    legacy = {k.replace("phrase_encoder", "bert_start"): v for k, v in sd.items()}
    mapped = {next((k.replace(o, n, 1) for o, n in LEGACY.items() if k.startswith(o)), k): v for k, v in legacy.items()}
    assert np.array_equal(tower_blob(mapped, "phrase_encoder", geo), tower_blob(sd, "phrase_encoder", geo))


def test_random_state_dict_default_stream_unchanged():
    """The query fixtures regenerate their weights from the seed: the default output must not move."""
    from densephrases_b200.encoder import BertGeometry, random_filter_state_dict, random_state_dict, synthetic_context_batch
    from oracle import encoder_ref
    g = np.load(QUERY_GOLD)
    geo = BertGeometry(vocab_size=int(g["vocab"]))
    sd = random_state_dict(geo, int(g["seed"]))
    assert sorted({k.split(".")[0] for k in sd}) == ["query_end_encoder", "query_start_encoder"]
    ids, mask, tt = (torch.from_numpy(g[f"b3_s24_{k}"]) for k in ("ids", "mask", "tt"))
    s, _ = encoder_ref.embed_query(sd, ids, mask, tt)
    assert (s - torch.from_numpy(g["b3_s24_start"])).abs().max() < 2e-4
    f1, f2 = random_filter_state_dict(geo, 5), random_filter_state_dict(geo, 5)
    assert f1["filter_linear.weight"].shape == (2, 768) and torch.equal(f1["filter_linear.weight"], f2["filter_linear.weight"])
    ids, mask, tt = synthetic_context_batch(4, 50, 2000, 3)
    assert (ids[:, 0] == 101).all() and mask[0].all() and not mask[1:, -1].any() and (tt == 1).any() and (tt[mask == 0] == 0).all()


def test_oracle_float_to_int8_rounds_half_to_even_and_clips():
    x = np.array([-2.0, -1.975, -1.925, -1.875, 0.0, 100.0, -100.0, 4.35, 4.4], dtype=np.float32)
    got = phrase_oracle.float_to_int8(x, -2, 20)
    ref = np.round(((x - -2) * 20).clip(-128, 127)).astype(np.int8)           # embed_utils.py:141-145 on fp32 data
    assert np.array_equal(got, ref)
    assert list(phrase_oracle.float_to_int8(np.array([0.5, 1.5, 2.5, -0.5, -1.5], np.float32), 0, 1)) == [0, 2, 2, 0, -2]
    assert phrase_oracle.float_to_int8(np.array([1e6, -1e6], np.float32), 0, 1).tolist() == [127, -128]
    assert phrase_oracle.float_to_int8(torch.tensor([0.05]), -2, 20).dtype == np.int8


def test_long_attention_kernels_compile_without_spills_on_the_tensor_cores():
    log = os.path.join(ROOT, "build", "obj", "attention_long.ptxas.log")
    assert os.path.exists(log), "run `make` / __graft_entry__.build() first"
    txt = open(log).read()
    assert txt.count("attention_long_kernel") >= 2
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", txt)
    assert spills and all(a == "0" and b == "0" for a, b in spills), spills
    lib = os.path.join(ROOT, "densephrases_b200", "lib", "libdph_b200.so")
    cuobjdump = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True, check=True).stdout
    for kernel in ("_Z21attention_long_kernelILb0EEv12AttnLongArgs", "_Z21attention_long_kernelILb1EEv12AttnLongArgs"):
        body = sass.split(f"Function : {kernel}")[1].split("Function : ")[0]
        assert re.search(r"\bUTC\w*MMA", body), kernel
        assert not re.search(r"(?<!UTC)\bHMMA", body), kernel


# ---- GPU ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tf32", "3xtf32", "bf16x3"])
@pytest.mark.parametrize("name", CASES)
def test_cuda_phrase_encoder_matches_reference_fixture(name, mode):
    from densephrases_b200.encoder import BertGeometry, Encoder
    seed, fseed, vocab, ids, mask, tt, pos, start, fs, fe = load_case(name)
    geo = BertGeometry(vocab_size=vocab)
    enc = Encoder(geo, state_dict=phrase_sd(geo, seed, fseed), precise=mode, towers="phrase")
    s, e, gfs, gfe = enc(input_ids=ids, attention_mask=mask, token_type_ids=tt, return_phrase=True)
    assert s is e and s.shape == ids.shape + (768,) and gfs.shape == ids.shape
    got = torch.take_along_dim(s.cpu(), pos[:, :, None], dim=1)
    d = max((got - start).abs().max().item(), (gfs.cpu() - fs).abs().max().item(), (gfe.cpu() - fe).abs().max().item())
    print(f"phrase {name} {mode}: max|diff| {d:.2e}")
    assert torch.isfinite(s).all() and d < TOL[mode]
    if mode == "tf32":
        assert cos(got, start).min() > 0.9995


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tf32", "3xtf32", "bf16x3"])
def test_cuda_phrase_encoder_against_torch_on_gpu(mode):
    """All B*S*768 outputs against the torch fp32 restatement on the GPU (TF32 off): B = 12 at S = 384, 512, and odd lengths."""
    from densephrases_b200.encoder import BertGeometry, Encoder, synthetic_context_batch
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    geo = BertGeometry(vocab_size=28996)
    sd = phrase_sd(geo, 7, 8)
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    enc = Encoder(geo, state_dict=sd, precise=mode, towers="phrase")
    for B, S in [(12, 384), (12, 512), (3, 1), (3, 65), (2, 129), (2, 300)]:
        ids, mask, tt = (t.cuda() for t in synthetic_context_batch(B, S, geo.vocab_size, S))
        s, _, gfs, gfe = enc(input_ids=ids, attention_mask=mask, token_type_ids=tt, return_phrase=True)
        rs, _, rfs, rfe = phrase_oracle.embed_phrase(sd_gpu, ids, mask, tt)
        d = max((s - rs).abs().max().item(), (gfs - rfs).abs().max().item(), (gfe - rfe).abs().max().item())
        print(f"phrase B={B} S={S} {mode}: max|diff| {d:.2e}, min cos {cos(s, rs).min().item():.6f}")
        assert torch.isfinite(s).all() and d < TOL[mode], (B, S, d)
        assert cos(s, rs).min() > 0.9995


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_core,tol", [(1, 1e-2), (2, 1e-4)])      # tcgen05 TF32 | tcgen05 bf16 (hi, lo) planes
@pytest.mark.parametrize("B,S", [(3, 65), (2, 128), (3, 200), (2, 384), (2, 512)])
def test_long_attention_against_torch(B, S, tensor_core, tol):
    """attention_long.cu through the C ABI against torch fp32, ragged masks (a padded tail per row, one fully padded key in the middle)."""
    from densephrases_b200 import _lib as L
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(S)
    qkv = torch.randn((B * S, 2304), generator=g, device="cuda")
    mask = torch.ones((B, S), dtype=torch.int64, device="cuda")
    for b in range(B):
        mask[b, S - 1 - b * (S // 5):] = 0
    mask[0, S // 2] = 0
    ctx = torch.full((B * S, 768), float("nan"), device="cuda")
    L.check(L.lib().dph_attention_bert(qkv.data_ptr(), mask.data_ptr(), B, S, ctx.data_ptr(), tensor_core, None))
    torch.cuda.synchronize()
    q, k, v = (qkv[:, i * 768:(i + 1) * 768].reshape(B, S, 12, 64).permute(0, 2, 1, 3) for i in range(3))
    sc = q @ k.transpose(-1, -2) / 8.0 + ((1.0 - mask.float()) * -10000.0)[:, None, None, :]
    ref = (torch.softmax(sc, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * S, 768)
    d = (ctx - ref).abs().max().item()
    print(f"long attention B={B} S={S} tensor_core={tensor_core}: max|diff| {d:.2e}")
    assert d < tol
    if S == 384:   # the SIMT kernel on the same input (its S <= 384 limit stays)
        ctx0 = torch.zeros_like(ctx)
        L.check(L.lib().dph_attention_bert(qkv.data_ptr(), mask.data_ptr(), B, S, ctx0.data_ptr(), 0, None))
        torch.cuda.synchronize()
        assert (ctx0 - ref).abs().max().item() < 2e-5
    with pytest.raises(RuntimeError):
        L.check(L.lib().dph_attention_bert(qkv.data_ptr(), mask.data_ptr(), 1, 513, ctx.data_ptr(), tensor_core, None))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["tf32", "bf16x3"])
def test_int8_codes(mode):
    """out_q == float_to_int8(out) of the same call, exactly; against the reference fixture every differing code is off by one, and in the
    fp32-accurate mode the reference value lies within 1e-3 * scale of a rounding boundary (tf32 vectors differ by up to ~2e-2, i.e.
    0.4 code steps, so there a code may differ anywhere)."""
    from densephrases_b200 import _lib as L
    from densephrases_b200.encoder import BertGeometry, Encoder
    seed, fseed, vocab, ids, mask, tt, pos, start, fs, fe = load_case("b2_s200")
    geo = BertGeometry(vocab_size=vocab)
    enc = Encoder(geo, state_dict=phrase_sd(geo, seed, fseed), precise=mode, towers="phrase")
    B, S = ids.shape
    di, dm, dt = (x.cuda() for x in (ids, mask, tt))
    out = torch.empty((B, S, 768), device="cuda")
    q = torch.empty((B, S, 768), dtype=torch.int8, device="cuda")
    f0, f1 = torch.empty((B, S), device="cuda"), torch.empty((B, S), device="cuda")
    L.check(L.lib().dph_encoder_embed_phrase(enc._h, di.data_ptr(), dm.data_ptr(), dt.data_ptr(), B, S, out.data_ptr(), f0.data_ptr(),
                                             f1.data_ptr(), q.data_ptr(), -2.0, 20.0, L.MEM_DEVICE))
    torch.cuda.synchronize()
    assert np.array_equal(q.cpu().numpy(), phrase_oracle.float_to_int8(out, -2, 20))
    q2, g0, g1 = enc.embed_phrase_int8(ids, mask, tt)                 # without the fp32 output: same codes and logits
    assert torch.equal(q2, q) and torch.equal(g0, f0) and torch.equal(g1, f1)
    ref_q = phrase_oracle.float_to_int8(start, -2, 20)
    got_q = np.take_along_axis(q.cpu().numpy(), pos.numpy()[:, :, None], axis=1)
    diff = got_q.astype(np.int32) - ref_q.astype(np.int32)
    assert np.abs(diff).max() <= 1
    t = (start.numpy() - np.float32(-2)) * np.float32(20)
    near = np.abs(t - np.floor(t) - 0.5) <= 1e-3 * 20
    if mode != "tf32":
        assert near[diff != 0].all(), f"{int((diff != 0).sum())} codes differ, not all near a rounding boundary"
    # host buffers: the same results through the staging path
    hq = np.empty((B, S, 768), np.int8); hf0 = np.empty((B, S), np.float32); hf1 = np.empty((B, S), np.float32); ho = np.empty((B, S, 768), np.float32)
    ids_np, mask_np, tt_np = (np.ascontiguousarray(x.numpy()) for x in (ids, mask, tt))
    L.check(L.lib().dph_encoder_embed_phrase(enc._h, ids_np.ctypes.data, mask_np.ctypes.data, tt_np.ctypes.data, B, S, ho.ctypes.data,
                                             hf0.ctypes.data, hf1.ctypes.data, hq.ctypes.data, -2.0, 20.0, L.MEM_HOST))
    assert np.array_equal(hq, q.cpu().numpy()) and np.array_equal(ho, out.cpu().numpy()) and np.array_equal(hf0, f0.cpu().numpy())


@pytest.mark.gpu
def test_query_path_isolated_from_phrase_tower():
    from densephrases_b200.encoder import BertGeometry, Encoder, random_filter_state_dict, random_state_dict, synthetic_context_batch
    g = np.load(QUERY_GOLD)
    geo = BertGeometry(vocab_size=int(g["vocab"]))
    sd = random_state_dict(geo, int(g["seed"]), prefixes=("query_start_encoder", "query_end_encoder", "phrase_encoder"))
    sd.update(random_filter_state_dict(geo, 1))
    query_only = Encoder(geo, state_dict=sd)
    both = Encoder(geo, state_dict=sd, towers="all")
    cids, cmask, ctt = (t.cuda() for t in synthetic_context_batch(16, 512, geo.vocab_size, 2))
    for name in ["b4_s64", "b3_s24", "b2_s100"]:
        ids, mask, tt = (torch.from_numpy(g[f"{name}_{k}"]).cuda() for k in ("ids", "mask", "tt"))
        for mode in ["tf32", "3xtf32", "bf16x3"]:
            query_only.set_precision(mode); both.set_precision(mode)
            ref = query_only.embed_query(ids, mask, tt)
            a = both.embed_query(ids, mask, tt)
            both.embed_phrase(cids, cmask, ctt)                       # regrows the workspace (slot 0) to 8192 tokens
            b = both.embed_query(ids, mask, tt)
            for x, y in ((a, ref), (b, ref)):
                assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1]), (name, mode)
    with pytest.raises(NotImplementedError):
        query_only(input_ids=cids, attention_mask=cmask, token_type_ids=ctt, return_phrase=True)
    with pytest.raises(NotImplementedError):                          # training paths stay out of scope
        both(input_ids=cids, attention_mask=cmask, token_type_ids=ctt, input_ids_=ids, attention_mask_=mask, token_type_ids_=tt,
             return_phrase=True, return_query=True)


@pytest.mark.gpu
def test_load_encoder_phrase_only(tmp_path):
    from types import SimpleNamespace
    from densephrases.utils.single_utils import load_encoder
    from densephrases_b200.encoder import BertGeometry, random_filter_state_dict, random_state_dict, synthetic_context_batch
    geo = BertGeometry(vocab_size=2000)
    sd = random_state_dict(geo, 4, prefixes=("phrase_encoder", "query_start_encoder", "query_end_encoder"))
    sd.update(random_filter_state_dict(geo, 4))
    legacy = {k.replace("phrase_encoder", "bert_start"): v for k, v in sd.items()}
    torch.save(legacy, tmp_path / "pytorch_model.bin")
    (tmp_path / "config.json").write_text('{"vocab_size": 2000}')
    vocab = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + [chr(ord("a") + i) for i in range(26)]
    (tmp_path / "vocab.txt").write_text("\n".join(vocab) + "\n")
    model, tok, cfg = load_encoder("cuda", SimpleNamespace(load_dir=str(tmp_path)), phrase_only=True)
    assert model.towers == "phrase"
    ids, mask, tt = synthetic_context_batch(2, 30, 2000, 1)
    s, e, fs, fe = model(input_ids=ids, attention_mask=mask, token_type_ids=tt, return_phrase=True)
    rs, _, rfs, _ = phrase_oracle.embed_phrase({k: v.cuda() for k, v in sd.items()}, ids.cuda(), mask.cuda(), tt.cuda())
    assert (s - rs).abs().max() < 1e-3 and (fs - rfs).abs().max() < 1e-3
    with pytest.raises(NotImplementedError):
        model(input_ids_=ids, attention_mask_=mask, token_type_ids_=tt, return_query=True)


@pytest.mark.gpu
def test_phrase_out_of_range_ids_raise():
    from densephrases_b200.encoder import BertGeometry, Encoder, random_filter_state_dict, random_state_dict
    geo = BertGeometry(vocab_size=500)
    sd = random_state_dict(geo, 1, prefixes=("phrase_encoder",))
    sd.update(random_filter_state_dict(geo, 1))
    enc = Encoder(geo, state_dict=sd, towers="phrase")
    ids = torch.full((2, 100), 3, dtype=torch.int64)
    mask, tt = torch.ones_like(ids), torch.zeros_like(ids)
    enc.embed_phrase(ids, mask, tt)
    bad = ids.clone(); bad[1, 70] = 500
    with pytest.raises(IndexError):
        enc.embed_phrase(bad, mask, tt)                       # host tensor: range-checked before the copy
    with pytest.raises(IndexError):
        enc.embed_phrase_int8(ids, mask, tt + 2)
    enc.embed_phrase(bad.cuda(), mask.cuda(), tt.cuda())      # device tensor: the kernel clamps the row and latches a flag ...
    with pytest.raises(RuntimeError, match="embedding tables"):
        enc.embed_phrase(ids.cuda(), mask.cuda(), tt.cuda())  # ... which the next call reports
    enc.embed_phrase(ids.cuda(), mask.cuda(), tt.cuda())
