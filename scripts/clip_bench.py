"""Times `encode_image` (train_svd.py:857-876: anti-aliased resize + normalisation + the ViT-H/14 image encoder) on 320 x 512
frames at the SVD configuration with bf16 parameters (train_svd.py:672), next to the bounds computed from shapes and the
baselines the reference runs.

    python scripts/clip_bench.py [--out profiles/clip_bench.json] [--calls 200] [--batches 1,2,8]

Per batch size: ours eager and captured in a CUDA graph; the oracle (the same arithmetic in PyTorch ops) under torch bf16
autocast; transformers' CLIPVisionModelWithProjection in bf16 (with the oracle's preprocessing) when transformers is importable.
CUDA events over `--calls` calls after warm-up. The bf16 weights (1.26 GB) exceed the 126 MB L2, so every call streams them from
HBM. The weights are random (seeded): timing does not depend on their values. Card name and power limit are read in the
same run and written with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.svd_clip_oracle import CLIP_CONFIG, CLIPVisionModelWithProjection as Oracle, init_weights, preprocess  # noqa: E402
from svd_xtend_b200.clip import CLIPVisionModelWithProjection as Ours, encode_image  # noqa: E402

DEV = "cuda:0"


def work_per_image(cfg):
    """(linear FLOP, attention FLOP, patch-embedding FLOP, bf16 weight bytes) of one image, from the shapes"""
    C, I, L, P, S = cfg["hidden_size"], cfg["intermediate_size"], cfg["num_hidden_layers"], cfg["projection_dim"], 257
    lin = L * 2.0 * S * (3 * C * C + C * C + 2 * C * I) + 2.0 * C * P
    attn = L * 4.0 * S * S * C
    patch = 2.0 * 256 * 588 * C
    with torch.device("meta"):
        params = sum(v.numel() for v in Oracle(**cfg).state_dict().values())
    return lin, attn, patch, 2.0 * params


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")) * 1e12, d.get("hbm_gbs") * 1e9, "MEASURED_PEAKS.json"
    return 2250e12, 7.7e12, "data sheet (HGX B200, one GPU, dense bf16; not reached)"


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unavailable ({type(e).__name__})"


def time_calls(fn, calls, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def time_graph(fn, calls):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return time_calls(g.replay, calls)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "clip_bench.json"))
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--batches", default="1,2,8")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("clip_bench.py needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    dt = torch.bfloat16
    with torch.device(DEV):
        oracle = init_weights(Oracle(**CLIP_CONFIG), 0).eval().requires_grad_(False)
        ours = Ours(**CLIP_CONFIG).eval().requires_grad_(False)
    ours.load_state_dict(oracle.state_dict())
    ours.to(dt)
    hf = None
    try:
        import transformers
        with torch.device(DEV):
            hf = transformers.CLIPVisionModelWithProjection(transformers.CLIPVisionConfig(**CLIP_CONFIG)).eval().requires_grad_(False)
        hf.load_state_dict(oracle.state_dict())
        hf.to(dt)
        hf_version = transformers.__version__
    except Exception as e:  # noqa: BLE001
        hf_version = f"not run ({type(e).__name__}: {e})"
    lin, attn, patch, wbytes = work_per_image(CLIP_CONFIG)
    peak_f, peak_b, peak_src = peaks()
    res = {"card": card(), "torch": torch.__version__, "transformers": hf_version, "frames": "320x512", "param_dtype": "bf16",
           "calls": args.calls, "peaks": {"bf16_flops": peak_f, "hbm_bytes_per_s": peak_b, "source": peak_src},
           "work_per_image": {"linear_gflop": lin / 1e9, "attention_gflop": attn / 1e9, "patch_gflop": patch / 1e9, "weight_gb_bf16": wbytes / 1e9},
           "row_tile_padding_b1": {"rows": 257, "rows_in_128_row_tiles": 384, "factor": 384 / 257}, "batches": {}}
    with torch.no_grad():
        for B in [int(b) for b in args.batches.split(",")]:
            x = torch.rand(B, 3, 320, 512, generator=torch.Generator(device=DEV).manual_seed(B), device=DEV) * 2 - 1
            flop = B * (lin + attn + patch)
            bound_f, bound_b = flop / peak_f * 1e3, wbytes / peak_b * 1e3
            r = {"gflop": flop / 1e9, "bound_ms_flop": bound_f, "bound_ms_weights": bound_b, "bound_ms": max(bound_f, bound_b)}
            r["ours_eager_ms"] = time_calls(lambda: encode_image(x, ours), args.calls)
            r["ours_graph_ms"] = time_graph(lambda: encode_image(x, ours), args.calls)

            def oracle_autocast():
                with torch.autocast("cuda", dtype=dt):
                    return oracle(preprocess(x)).image_embeds
            r["oracle_bf16_autocast_ms"] = time_calls(oracle_autocast, args.calls)
            if hf is not None:
                r["transformers_bf16_ms"] = time_calls(lambda: hf(preprocess(x).to(dt)).image_embeds, args.calls)
            ref = oracle(preprocess(x)).image_embeds
            got = encode_image(x, ours).float()
            r["rel_l2_vs_fp32_oracle"] = ((got - ref).norm() / ref.norm()).item()
            r["ours_graph_share_of_bound"] = r["bound_ms"] / r["ours_graph_ms"]
            res["batches"][str(B)] = r
            print(B, json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("card:", res["card"], "->", args.out)


if __name__ == "__main__":
    main()
