"""ORACLE — test infrastructure only. Plain-PyTorch restatement of the CLIP image encoder as `train_svd.py` uses it:

    image_encoder = CLIPVisionModelWithProjection.from_pretrained(..., subfolder="image_encoder")    (train_svd.py:646)
    encode_image(pixel_values)                                                                       (train_svd.py:857-876)
        = image_encoder(normalize((resize_with_antialiasing(pixel_values, (224, 224)) + 1) / 2)).image_embeds

The encoder is transformers' CLIPVisionModelWithProjection (pre-LN ViT: patch conv + class token + learned positions,
pre_layrnorm, L x [LN1 -> multi-head self-attention -> residual, LN2 -> fc1 -> GELU -> fc2 -> residual], post_layernorm on
the class token, bias-free visual_projection). Unlike the UNet and VAE restatements this block arithmetic IS pinned against
its upstream implementation: tests/golden/make_clip_golden.py runs transformers' own class at TINY_CLIP_CONFIG in float64
and tests/test_clip.py holds this file to it (and to live transformers wherever it is importable).

The preprocessing is restated from what the reference's resize helpers compute (a Gaussian anti-aliasing blur, reflect
padded, then bicubic align_corners resampling) and from the CLIPImageProcessor normalisation; the fixture records the
reference's own functions on seeded frames. Parameter names follow the transformers state dict.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

import torch
import torch.nn as nn
import torch.nn.functional as F

CLIP_CONFIG = dict(hidden_size=1280, intermediate_size=5120, num_attention_heads=16, num_hidden_layers=32, patch_size=14,
                   image_size=224, projection_dim=1024, hidden_act="gelu", layer_norm_eps=1e-5, num_channels=3)
TINY_CLIP_CONFIG = dict(hidden_size=160, intermediate_size=640, num_attention_heads=2, num_hidden_layers=2, patch_size=14,
                        image_size=224, projection_dim=64, hidden_act="gelu", layer_norm_eps=1e-5, num_channels=3)
CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)      # CLIPImageProcessor defaults (OpenAI CLIP statistics)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)
CLIP_SIZE = 224


# ----------------------------------------------------------------------------- preprocessing
def antialias_params(h: int, w: int, size=(CLIP_SIZE, CLIP_SIZE)):
    """((k_h, k_w), (sigma_h, sigma_w)) of the blur that precedes resampling an h x w image: sigma = (scale - 1) / 2 with a
    floor of 0.001, window = the integer part of 4 sigma but at least 3, bumped to the next odd number"""
    sig = tuple(max((n / s - 1.0) / 2.0, 0.001) for n, s in zip((h, w), size))
    ks = tuple(k if k % 2 else k + 1 for k in (int(max(4.0 * s, 3.0)) for s in sig))
    return ks, sig


def gaussian_taps(k: int, sigma: float, dtype=torch.float64) -> torch.Tensor:
    """normalised samples of a Gaussian on the k integer offsets centred on the window (k odd)"""
    x = torch.arange(k, dtype=torch.float64) - (k // 2)
    g = torch.exp(-(x * x) / (2.0 * sigma * sigma))
    return (g / g.sum()).to(dtype)


def _blur_axis(x: torch.Tensor, taps: torch.Tensor, dim: int) -> torch.Tensor:
    """correlate every channel with `taps` along H (dim=2) or W (dim=3), reflect padding of (k - 1) / 2 on each side"""
    k = taps.numel()
    p = (k - 1) // 2
    c = x.shape[1]
    if dim == 3:
        xp = F.pad(x, (p, k - 1 - p, 0, 0), mode="reflect")
        w = taps.view(1, 1, 1, k)
    else:
        xp = F.pad(x, (0, 0, p, k - 1 - p), mode="reflect")
        w = taps.view(1, 1, k, 1)
    return F.conv2d(xp, w.to(device=x.device, dtype=x.dtype).expand(c, 1, *w.shape[2:]).contiguous(), groups=c)


def resize_antialiased(x: torch.Tensor, size=(CLIP_SIZE, CLIP_SIZE)) -> torch.Tensor:
    """[B, C, H, W] -> [B, C, size]: Gaussian anti-aliasing blur (W first, then H) and bicubic align_corners resampling"""
    (kh, kw), (sh, sw) = antialias_params(x.shape[-2], x.shape[-1], size)
    y = _blur_axis(x, gaussian_taps(kw, sw, x.dtype), dim=3)
    y = _blur_axis(y, gaussian_taps(kh, sh, x.dtype), dim=2)
    return F.interpolate(y, size=size, mode="bicubic", align_corners=True)


def normalize(x: torch.Tensor, mean=CLIP_MEAN, std=CLIP_STD) -> torch.Tensor:
    m = torch.tensor(mean, dtype=x.dtype, device=x.device).view(1, -1, 1, 1)
    s = torch.tensor(std, dtype=x.dtype, device=x.device).view(1, -1, 1, 1)
    return (x - m) / s


def preprocess(frames: torch.Tensor, mean=CLIP_MEAN, std=CLIP_STD) -> torch.Tensor:
    """encode_image's pixel path: frames in [-1, 1] -> normalised 224 x 224 CLIP input"""
    return normalize((resize_antialiased(frames) + 1.0) / 2.0, mean, std)


def patchify(x: torch.Tensor, patch: int = 14) -> torch.Tensor:
    """[B, C, 224, 224] -> [B * 256, C * patch * patch]: row b * 256 + py * 16 + px = patch (py, px) in (c, ky, kx) order"""
    B, Cc, H, W = x.shape
    n = H // patch
    return x.reshape(B, Cc, n, patch, n, patch).permute(0, 2, 4, 1, 3, 5).reshape(B * n * n, Cc * patch * patch)


# ----------------------------------------------------------------------------- the encoder
class _Embeddings(nn.Module):
    def __init__(self, c, patch, image, channels):
        super().__init__()
        self.class_embedding = nn.Parameter(torch.zeros(c))
        self.patch_embedding = nn.Conv2d(channels, c, patch, stride=patch, bias=False)
        self.position_embedding = nn.Embedding((image // patch) ** 2 + 1, c)

    def forward(self, x):
        p = self.patch_embedding(x.to(self.patch_embedding.weight.dtype)).flatten(2).transpose(1, 2)    # [B, 256, C]
        cls = self.class_embedding.view(1, 1, -1).expand(x.shape[0], 1, -1)
        return torch.cat([cls, p], dim=1) + self.position_embedding.weight.unsqueeze(0)


class _Attention(nn.Module):
    def __init__(self, c, heads):
        super().__init__()
        self.heads = heads
        self.k_proj = nn.Linear(c, c)
        self.v_proj = nn.Linear(c, c)
        self.q_proj = nn.Linear(c, c)
        self.out_proj = nn.Linear(c, c)

    def forward(self, x):
        B, S, C = x.shape
        d = C // self.heads
        split = lambda t: t.view(B, S, self.heads, d).transpose(1, 2)
        q, k, v = split(self.q_proj(x)), split(self.k_proj(x)), split(self.v_proj(x))
        a = torch.softmax((q @ k.transpose(-1, -2)) * d ** -0.5, dim=-1)
        return self.out_proj((a @ v).transpose(1, 2).reshape(B, S, C))


class _MLP(nn.Module):
    def __init__(self, c, inner):
        super().__init__()
        self.fc1 = nn.Linear(c, inner)
        self.fc2 = nn.Linear(inner, c)

    def forward(self, x):
        return self.fc2(F.gelu(self.fc1(x)))


class _Layer(nn.Module):
    def __init__(self, c, heads, inner, eps):
        super().__init__()
        self.self_attn = _Attention(c, heads)
        self.layer_norm1 = nn.LayerNorm(c, eps=eps)
        self.mlp = _MLP(c, inner)
        self.layer_norm2 = nn.LayerNorm(c, eps=eps)

    def forward(self, x):
        x = x + self.self_attn(self.layer_norm1(x))
        return x + self.mlp(self.layer_norm2(x))


class _Encoder(nn.Module):
    def __init__(self, n, *a):
        super().__init__()
        self.layers = nn.ModuleList([_Layer(*a) for _ in range(n)])


class _VisionModel(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        c = cfg["hidden_size"]
        self.embeddings = _Embeddings(c, cfg["patch_size"], cfg["image_size"], cfg["num_channels"])
        self.pre_layrnorm = nn.LayerNorm(c, eps=cfg["layer_norm_eps"])
        self.encoder = _Encoder(cfg["num_hidden_layers"], c, cfg["num_attention_heads"], cfg["intermediate_size"], cfg["layer_norm_eps"])
        self.post_layernorm = nn.LayerNorm(c, eps=cfg["layer_norm_eps"])


class CLIPVisionModelWithProjection(nn.Module):
    """reference semantics of transformers' CLIPVisionModelWithProjection.forward(pixel_values) (gelu models only)"""

    def __init__(self, **cfg):
        super().__init__()
        full = dict(CLIP_CONFIG)
        full.update(cfg)
        if full["hidden_act"] != "gelu":
            raise ValueError("the oracle restates hidden_act='gelu' only")
        self.config = SimpleNamespace(**full)
        self.vision_model = _VisionModel(full)
        self.visual_projection = nn.Linear(full["hidden_size"], full["projection_dim"], bias=False)

    def forward(self, pixel_values):
        vm = self.vision_model
        h = vm.pre_layrnorm(vm.embeddings(pixel_values))
        for layer in vm.encoder.layers:
            h = layer(h)
        pooled = vm.post_layernorm(h[:, 0, :])
        return SimpleNamespace(image_embeds=self.visual_projection(pooled), last_hidden_state=h)


def encode_image(frames: torch.Tensor, model: CLIPVisionModelWithProjection, mean=CLIP_MEAN, std=CLIP_STD) -> torch.Tensor:
    """train_svd.py:857-876: [B, 3, H, W] frames in [-1, 1] -> image_embeds [B, projection_dim]"""
    x = preprocess(frames.to(next(model.parameters()).dtype), mean, std)
    return model(x).image_embeds


@torch.no_grad()
def init_weights(model: nn.Module, seed: int) -> nn.Module:
    """seeded weights for tests, drawn in state-dict order from one generator on the model's device: matrices / conv kernels
    ~ N(0, 1 / fan_in), embeddings ~ N(0, 0.5^2), LayerNorm scales 1 + N(0, 0.1^2), biases and LayerNorm shifts N(0, 0.1^2)
    (every affine path matters). The same call gives the same tensors on any module with these names and shapes."""
    params = dict(model.named_parameters())
    dev = next(model.parameters()).device
    g = torch.Generator(device=dev).manual_seed(seed)
    for name in model.state_dict().keys():
        p = params[name]
        r = torch.randn(p.shape, generator=g, device=dev, dtype=torch.float64 if p.dtype == torch.float64 else torch.float32)
        if "norm" in name and name.endswith("weight"):
            v = 1.0 + 0.1 * r
        elif name.endswith("bias"):
            v = 0.1 * r
        elif "embedding" in name and "patch" not in name:
            v = 0.5 * r
        else:
            v = r / math.sqrt(p[0].numel())
        p.copy_(v)
    return model
