"""Generates tests/golden/clip_tiny.pt: the CLIP image path of the reference, recorded from the code that defines it.

    python tests/golden/make_clip_golden.py <reference checkout>

Runs on the CPU and needs `transformers`; tests/test_clip.py needs neither it nor the checkout. It records
  * the reference's own anti-aliased resize: the five helpers `_resize_with_antialiasing`, `_compute_padding`, `_filter2d`,
    `_gaussian` and `_gaussian_blur2d` are taken from <checkout>/train_svd.py with `ast` (the file cannot be imported: its
    top level imports diffusers and accelerate) and executed here, in float64, on seeded frames of 320 x 512 and 576 x 1024
    (B = 2) and one up-scaling case (128 x 128): the blur kernel sizes and sigmas they choose, and the norm plus RESIZE_SAMPLES
    seeded samples of each 224 x 224 result;
  * transformers' CLIPImageProcessor normalisation with the script's flags (train_svd.py:864-871) on (resized + 1) / 2;
  * transformers' CLIPVisionModelWithProjection at TINY_CLIP_CONFIG in float64 with the oracle's seeded weights: per-tensor
    state-dict sums, image_embeds, and the norm plus samples of last_hidden_state;
  * the key list, shapes and parameter count of transformers' class at the SVD configuration (meta device).
"""
import ast
import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.svd_clip_oracle import CLIP_CONFIG, TINY_CLIP_CONFIG, CLIPVisionModelWithProjection as Oracle, init_weights  # noqa: E402

SEED = 20261017
RESIZE_CASES = (("320x512", 2, 320, 512), ("576x1024", 2, 576, 1024), ("128x128", 1, 128, 128))
RESIZE_SAMPLES = 4096
HIDDEN_SAMPLES = 4096
HELPERS = ("_resize_with_antialiasing", "_compute_padding", "_filter2d", "_gaussian", "_gaussian_blur2d")


def frames(case_index, B, H, W):
    """seeded frames in [-1, 1) (float64); tests/test_clip.py draws the same"""
    g = torch.Generator().manual_seed(SEED + 100 * case_index)
    return torch.rand(B, 3, H, W, generator=g, dtype=torch.float64) * 2.0 - 1.0


def pixel_values(B):
    g = torch.Generator().manual_seed(SEED + 7)
    return torch.randn(B, 3, 224, 224, generator=g, dtype=torch.float64)


def sample_index(numel, salt):
    return torch.randperm(numel, generator=torch.Generator().manual_seed(SEED + salt))[:RESIZE_SAMPLES].sort().values


def reference_helpers(reference_root):
    path = os.path.join(reference_root, "train_svd.py")
    src = open(path).read()
    tree = ast.parse(src)
    found = {n.name: n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in HELPERS}
    missing = set(HELPERS) - set(found)
    if missing:
        raise RuntimeError(f"{path} lacks {sorted(missing)}")
    mod = ast.Module(body=[found[n] for n in HELPERS], type_ignores=[])
    ns = {"torch": torch}
    exec(compile(mod, path, "exec"), ns)
    return ns, hashlib.sha256("\n".join(ast.get_source_segment(src, found[n]) for n in HELPERS).encode()).hexdigest()


def main(reference_root):
    from transformers import CLIPImageProcessor, CLIPVisionConfig, CLIPVisionModelWithProjection as HF

    ns, helpers_sha = reference_helpers(reference_root)
    blur_calls = []
    blur = ns["_gaussian_blur2d"]

    def recording_blur(x, kernel_size, sigma):
        blur_calls.append((tuple(int(k) for k in kernel_size), tuple(float(s) for s in sigma)))
        return blur(x, kernel_size, sigma)
    ns["_gaussian_blur2d"] = recording_blur

    processor = CLIPImageProcessor()
    resize = {}
    for ci, (name, B, H, W) in enumerate(RESIZE_CASES):
        blur_calls.clear()
        y = ns["_resize_with_antialiasing"](frames(ci, B, H, W), (224, 224))
        assert y.dtype == torch.float64 and tuple(y.shape) == (B, 3, 224, 224) and len(blur_calls) == 1
        idx = sample_index(y.numel(), ci)
        entry = {"B": B, "H": H, "W": W, "kernel_size": blur_calls[0][0], "sigma": blur_calls[0][1], "norm": float(y.norm()),
                 "idx": idx.to(torch.int32), "val": y.reshape(-1)[idx].clone()}
        # CLIPImageProcessor with the flags of train_svd.py:864-871, on the unnormalised resize
        pv = processor(images=(y + 1.0) / 2.0, do_normalize=True, do_center_crop=False, do_resize=False, do_rescale=False,
                       return_tensors="pt").pixel_values
        entry["norm_processor"] = float(pv.double().norm())
        entry["val_processor"] = pv.reshape(-1)[idx].double().clone()
        entry["processor_dtype"] = str(pv.dtype)
        resize[name] = entry

    hf = HF(CLIPVisionConfig(**TINY_CLIP_CONFIG)).double().eval()
    oracle = init_weights(Oracle(**TINY_CLIP_CONFIG).double(), SEED + 1)
    hf.load_state_dict(oracle.state_dict(), strict=True)
    x = pixel_values(2)
    with torch.no_grad():
        out = hf(x)
    lhs = out.last_hidden_state
    lidx = torch.randperm(lhs.numel(), generator=torch.Generator().manual_seed(SEED + 11))[:HIDDEN_SAMPLES].sort().values
    with torch.device("meta"):
        big = HF(CLIPVisionConfig(**CLIP_CONFIG))
    big_keys = [(k, tuple(v.shape)) for k, v in big.state_dict().items()]

    fixture = {
        "seed": SEED,
        "reference_helpers_sha256": helpers_sha,
        "resize": resize,
        "tiny_state_sums": {k: (float(v.sum()), float(v.abs().sum())) for k, v in hf.state_dict().items()},
        "tiny_image_embeds": out.image_embeds.clone(),
        "tiny_hidden_norm": float(lhs.norm()),
        "tiny_hidden_idx": lidx.to(torch.int32),
        "tiny_hidden_val": lhs.reshape(-1)[lidx].clone(),
        "svd_keys_sha256": hashlib.sha256(repr(big_keys).encode()).hexdigest(),
        "svd_keys": big_keys,
        "svd_total_params": sum(v.numel() for v in big.state_dict().values()),
    }
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "clip_tiny.pt")
    torch.save(fixture, path)
    print("wrote", path, {n: (e["kernel_size"], e["sigma"]) for n, e in resize.items()}, "svd params", fixture["svd_total_params"],
          "embeds std", float(out.image_embeds.std()))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(f"usage: python {sys.argv[0]} <reference checkout>")
    main(sys.argv[1])
