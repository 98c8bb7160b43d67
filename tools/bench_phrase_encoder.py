"""Phrase encoder timing: Encoder.forward(input_ids=..., return_phrase=True) (phrase tower + filter head) in every precision mode,
the long-sequence attention kernel alone, and a torch arm on the same GPU (fp32 and fp16 autocast; the latter is the closest
stand-in for the reference's `--fp16` apex O1 dump).

    python tools/bench_phrase_encoder.py --out DIR

Times come from CUDA events around back-to-back calls, after a warm-up, over windows of at least --window seconds; the median
window and the spread (min, max) over --repeats windows are reported.  Algorithmic FLOP from shapes: per token
12 * 2 * (768*2304 + 768*768 + 2*768*3072) + 4*768, plus per sequence 12 * 4 * S^2 * 768.  Tensor work counts the MMAs a mode
issues (Encoder.mma_multiplier, in TF32-MMA equivalents) against NVIDIA's data-sheet dense rate for one B200 (1,125 TFLOP/s TF32 =
half of 2,250 TFLOP/s BF16); a card at a lower power limit, or one that throttles under a sustained matrix load, gets less.
Writes DIR/phrase_encoder_bench.json; fails when no GPU is present."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

SHAPES = [(12, 384), (64, 384), (12, 512), (32, 512)]
MODES = ["tf32", "3xtf32", "bf16x3"]
TF32_PEAK_TFLOPS = 1125.0


def flop(B, S):
    per_token = 12 * 2 * (768 * 2304 + 768 * 768 + 2 * 768 * 3072) + 4 * 768
    return B * S * per_token + B * 12 * 4 * S * S * 768


def timed(fn, window, repeats):
    """-> (median ms per call, min, max) over `repeats` windows of >= `window` seconds each."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    n = max(1, int(window / max(time.perf_counter() - t0, 1e-6)) + 1)
    out = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        while True:
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            if ms >= window * 1e3:
                break
            n = int(n * window * 1e3 / max(ms, 1e-3) * 1.1) + 1
        out.append(ms / n)
    return statistics.median(out), min(out), max(out)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no GPU found: this benchmark only measures on the GPU")
    from densephrases_b200 import _lib as L
    from densephrases_b200.encoder import BertGeometry, Encoder, random_filter_state_dict, random_state_dict, synthetic_context_batch
    from oracle.encoder_ref import tower_forward
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    geo = BertGeometry()
    sd = random_state_dict(geo, 1, prefixes=("phrase_encoder",))
    sd.update(random_filter_state_dict(geo, 1))
    enc = Encoder(geo, state_dict=sd, towers="phrase")
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    res = {"card": card(), "torch": torch.__version__, "window_s": args.window, "repeats": args.repeats,
           "tf32_peak_tflops_datasheet": TF32_PEAK_TFLOPS, "encoder": [], "torch_arm": [], "attention": []}
    print("card:", res["card"])

    def row(kind, B, S, ms, lo, hi, extra):
        r = {"kind": kind, "B": B, "S": S, "ms": round(ms, 4), "ms_min": round(lo, 4), "ms_max": round(hi, 4),
             "tokens_per_s": round(B * S / ms * 1e3), "contexts_per_s": round(B / ms * 1e3, 1),
             "algorithmic_tflops": round(flop(B, S) / ms / 1e9, 1)}
        r.update(extra)
        print(json.dumps(r))
        return r

    for B, S in SHAPES:
        ids, mask, tt = (t.cuda() for t in synthetic_context_batch(B, S, geo.vocab_size, S))
        for mode in MODES:
            enc.set_precision(mode)
            ms, lo, hi = timed(lambda: enc(input_ids=ids, attention_mask=mask, token_type_ids=tt, return_phrase=True), args.window, args.repeats)
            mult = Encoder.mma_multiplier(mode)
            res["encoder"].append(row(mode, B, S, ms, lo, hi, {
                "mma_kind": "tf32" if mode != "bf16x3" else "f16 (bf16 planes)", "mma_multiplier": mult,
                "tensor_share_of_datasheet_peak": round(flop(B, S) * mult / ms / 1e9 / TF32_PEAK_TFLOPS, 4)}))

        def torch_fwd():
            with torch.no_grad():
                x = tower_forward(sd_gpu, "phrase_encoder", ids, mask, tt)
                torch.nn.functional.linear(x, sd_gpu["filter_linear.weight"], sd_gpu["filter_linear.bias"])

        def torch_fp16():
            with torch.autocast("cuda", dtype=torch.float16):
                torch_fwd()
        for kind, fn in (("torch_fp32", torch_fwd), ("torch_fp16_autocast", torch_fp16)):
            ms, lo, hi = timed(fn, args.window, args.repeats)
            res["torch_arm"].append(row(kind, B, S, ms, lo, hi, {}))

    # the attention kernel alone (C ABI; each call ends with a stream synchronisation)
    for B, S, tcs in [(12, 384, (0, 1, 2)), (12, 512, (1, 2)), (64, 384, (0, 1, 2)), (32, 512, (1, 2))]:
        g = torch.Generator(device="cuda").manual_seed(S)
        qkv = torch.randn((B * S, 2304), generator=g, device="cuda")
        mask = torch.ones((B, S), dtype=torch.int64, device="cuda")
        ctx = torch.empty((B * S, 768), device="cuda")
        for tc in tcs:
            ms, lo, hi = timed(lambda: L.check(L.lib().dph_attention_bert(qkv.data_ptr(), mask.data_ptr(), B, S, ctx.data_ptr(), tc, None)),
                               args.window, args.repeats)
            r = {"kernel": {0: "simt_fp32", 1: "long_tc_tf32", 2: "long_tc_bf16x3"}[tc], "B": B, "S": S, "ms": round(ms, 4),
                 "ms_min": round(lo, 4), "ms_max": round(hi, 4), "algorithmic_tflops": round(B * 12 * 4 * S * S * 64 / ms / 1e9, 1)}
            print(json.dumps(r))
            res["attention"].append(r)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "phrase_encoder_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", os.path.join(args.out, "phrase_encoder_bench.json"))


if __name__ == "__main__":
    main()
