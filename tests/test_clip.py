"""CLIP image encoder (train_svd.py:646, :857-876) — CPU checks: the product class and the oracle against the fixture recorded
from the reference's own resize helpers, transformers' CLIPImageProcessor and transformers' CLIPVisionModelWithProjection
(tests/golden/make_clip_golden.py), the host-side blur taps, construction refusals and the CUDA-only guard."""
import hashlib
import os

import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "clip_tiny.pt")


@pytest.fixture(scope="module")
def fx():
    return torch.load(GOLDEN, weights_only=False)


def _frames(seed, case_index, B, H, W):
    g = torch.Generator().manual_seed(seed + 100 * case_index)
    return torch.rand(B, 3, H, W, generator=g, dtype=torch.float64) * 2.0 - 1.0


def _keys(m):
    return [(k, tuple(v.shape)) for k, v in m.state_dict().items()]


def test_census_product_and_oracle(fx):
    from oracle.svd_clip_oracle import CLIP_CONFIG, CLIPVisionModelWithProjection as Oracle
    from svd_xtend_b200.clip import CLIPVisionModelWithProjection as Ours
    with torch.device("meta"):
        ours, oracle = Ours(**CLIP_CONFIG), Oracle(**CLIP_CONFIG)
    for m in (ours, oracle):
        keys = _keys(m)
        assert hashlib.sha256(repr(keys).encode()).hexdigest() == fx["svd_keys_sha256"]
        assert keys == [(k, tuple(s)) for k, s in fx["svd_keys"]]
        assert len(keys) == 520
        assert sum(v.numel() for v in m.state_dict().values()) == fx["svd_total_params"] == 632_076_800
    assert keys[0][0] == "vision_model.embeddings.class_embedding" and keys[-1][0] == "visual_projection.weight"


@pytest.mark.parametrize("case", [0, 1, 2])
def test_oracle_resize_matches_reference_helpers(fx, case):
    from oracle.svd_clip_oracle import antialias_params, resize_antialiased
    from svd_xtend_b200 import raw
    name = ("320x512", "576x1024", "128x128")[case]
    e = fx["resize"][name]
    y = resize_antialiased(_frames(fx["seed"], case, e["B"], e["H"], e["W"]))
    assert abs(float(y.norm()) - e["norm"]) <= 1e-12 * e["norm"]
    assert (y.reshape(-1)[e["idx"].long()] - e["val"]).abs().max().item() <= 1e-12
    # the kernel sizes and sigmas the reference picked: the oracle's rule and the host tap computation of svdx_clip_pixels
    assert antialias_params(e["H"], e["W"]) == (e["kernel_size"], pytest.approx(e["sigma"], abs=1e-15))
    ky, kx, wy, wx, sig = raw.clip_blur_taps(e["H"], e["W"])
    assert (ky, kx) == e["kernel_size"] and sig == pytest.approx(e["sigma"], abs=1e-15)
    for k, w, s in ((ky, wy, sig[0]), (kx, wx, sig[1])):
        ref = torch.exp(-(torch.arange(k, dtype=torch.float64) - k // 2) ** 2 / (2 * s * s))
        assert torch.allclose(torch.tensor(w, dtype=torch.float64), ref / ref.sum(), rtol=0, atol=1e-15)


@pytest.mark.parametrize("case", [0, 1, 2])
def test_oracle_normalisation_matches_processor(fx, case):
    from oracle.svd_clip_oracle import normalize, resize_antialiased
    name = ("320x512", "576x1024", "128x128")[case]
    e = fx["resize"][name]
    x = normalize((resize_antialiased(_frames(fx["seed"], case, e["B"], e["H"], e["W"])) + 1.0) / 2.0)
    # the image processor computes in float32
    assert (x.reshape(-1)[e["idx"].long()] - e["val_processor"]).abs().max().item() <= 1e-6
    assert abs(float(x.norm()) - e["norm_processor"]) <= 1e-6 * e["norm_processor"]


def _tiny_oracle(fx):
    from oracle.svd_clip_oracle import TINY_CLIP_CONFIG, CLIPVisionModelWithProjection as Oracle, init_weights
    m = init_weights(Oracle(**TINY_CLIP_CONFIG).double(), fx["seed"] + 1).eval()
    sums = {k: (float(v.sum()), float(v.abs().sum())) for k, v in m.state_dict().items()}
    assert sums.keys() == fx["tiny_state_sums"].keys()
    for k, (s, a) in sums.items():
        assert s == pytest.approx(fx["tiny_state_sums"][k][0], abs=1e-9) and a == pytest.approx(fx["tiny_state_sums"][k][1], rel=1e-12), k
    return m


def _pixel_values(seed, B):
    return torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(seed + 7), dtype=torch.float64)


def test_oracle_matches_transformers_fixture(fx):
    m = _tiny_oracle(fx)
    with torch.no_grad():
        out = m(_pixel_values(fx["seed"], 2))
    assert (out.image_embeds - fx["tiny_image_embeds"]).abs().max().item() <= 1e-10
    lhs = out.last_hidden_state
    assert (lhs.reshape(-1)[fx["tiny_hidden_idx"].long()] - fx["tiny_hidden_val"]).abs().max().item() <= 1e-10
    assert abs(float(lhs.norm()) - fx["tiny_hidden_norm"]) <= 1e-10 * fx["tiny_hidden_norm"]


def test_oracle_matches_live_transformers(fx):
    transformers = pytest.importorskip("transformers")
    from oracle.svd_clip_oracle import CLIP_CONFIG, TINY_CLIP_CONFIG
    m = _tiny_oracle(fx)
    hf = transformers.CLIPVisionModelWithProjection(transformers.CLIPVisionConfig(**TINY_CLIP_CONFIG)).double().eval()
    hf.load_state_dict(m.state_dict(), strict=True)
    x = torch.randn(3, 3, 224, 224, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    with torch.no_grad():
        a, b = hf(x), m(x)
    assert (a.image_embeds - b.image_embeds).abs().max().item() <= 1e-10
    assert (a.last_hidden_state - b.last_hidden_state).abs().max().item() <= 1e-10
    with torch.device("meta"):
        big = transformers.CLIPVisionModelWithProjection(transformers.CLIPVisionConfig(**CLIP_CONFIG))
    assert _keys(big) == [(k, tuple(s)) for k, s in fx["svd_keys"]]


@pytest.mark.parametrize("bad", [dict(hidden_act="quick_gelu"), dict(num_attention_heads=20), dict(hidden_size=1024),
                                 dict(image_size=336), dict(patch_size=16), dict(intermediate_size=5000)])
def test_construction_refuses_unsupported_configs(bad):
    from oracle.svd_clip_oracle import TINY_CLIP_CONFIG
    from svd_xtend_b200.clip import CLIPVisionModelWithProjection as Ours
    cfg = dict(TINY_CLIP_CONFIG)
    cfg.update(bad)
    with torch.device("meta"), pytest.raises(ValueError):
        Ours(**cfg)


def test_config_object_and_cpu_refusal():
    from oracle.svd_clip_oracle import TINY_CLIP_CONFIG
    from svd_xtend_b200.clip import CLIPVisionModelWithProjection as Ours, encode_image
    from types import SimpleNamespace
    m = Ours(SimpleNamespace(**TINY_CLIP_CONFIG)).requires_grad_(False)
    assert m.config.hidden_size == 160 and m.config.projection_dim == 64
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="CUDA"):
            m(torch.zeros(1, 3, 224, 224))
        with pytest.raises(RuntimeError, match="CUDA"):
            encode_image(torch.zeros(1, 3, 320, 512), m)
        with pytest.raises(NotImplementedError):
            m(torch.zeros(1, 3, 224, 224), output_hidden_states=True)
