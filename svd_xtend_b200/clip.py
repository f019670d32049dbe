"""`CLIPVisionModelWithProjection` and `encode_image` on B200 — the frozen CLIP image encoder of every training step
(ViT-H/14 at the SVD configuration: 32 layers, 1280 wide, 16 heads of 80, 257 tokens; 632 M parameters) and the embedding the
UNet is conditioned on:

    image_encoder = CLIPVisionModelWithProjection.from_pretrained(..., subfolder="image_encoder")   (train_svd.py:646, :672)
    encoder_hidden_states = encode_image(pixel_values[:, 0])                                       (train_svd.py:857-876, :975)

Path (one token matrix [B * 257, C] bf16, forward only — the reference freezes the encoder, train_svd.py:660):
  1. `svdx_clip_pixels`: anti-aliased bicubic resize to 224 x 224 + CLIPImageProcessor normalisation (encode_image) or the
     already normalised input (forward), cut into the [B * 256, 592] patch matrix;
  2. patch embedding as a GEMM (K = 592) per image with the position embeddings pos[1:] as its residual, written to rows
     1 .. 256 of the image's 257-row block; the class rows (class_embedding + pos[0]) in one launch;
  3. pre_layrnorm, then per layer: LN1 -> fused q|k|v linear -> `svdx_attention_vit_fwd` (head_dim 80, q/k/v read in place)
     -> out_proj + residual -> LN2 -> fc1 with the GELU epilogue -> fc2 + residual (split-K where 257-row GEMMs leave SMs idle);
  4. post_layernorm on the class-token rows only (row stride 257 * C), visual_projection as a GEMV (B <= 8) or GEMM.
No host synchronisation and no host-dependent control flow after the first call for a shape: a call can be captured in a
CUDA graph. Parameter names follow the transformers state dict. No PyTorch / CPU fallback.
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace
from typing import Optional

import torch
import torch.nn as nn

from . import raw
from .engine import Engine, F32, Var, bf16

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)     # CLIPImageProcessor defaults
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)
_CONFIG_FIELDS = ("hidden_size", "intermediate_size", "projection_dim", "num_hidden_layers", "num_attention_heads", "num_channels",
                  "image_size", "patch_size", "hidden_act", "layer_norm_eps")
_DEFAULTS = dict(hidden_size=1280, intermediate_size=5120, projection_dim=1024, num_hidden_layers=32, num_attention_heads=16,
                 num_channels=3, image_size=224, patch_size=14, hidden_act="gelu", layer_norm_eps=1e-5)


class _Embeddings(nn.Module):
    def __init__(self, c, patch, image, channels):
        super().__init__()
        self.class_embedding = nn.Parameter(torch.zeros(c))
        self.patch_embedding = nn.Conv2d(channels, c, patch, stride=patch, bias=False)
        self.position_embedding = nn.Embedding((image // patch) ** 2 + 1, c)


class _Attention(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.k_proj = nn.Linear(c, c)
        self.v_proj = nn.Linear(c, c)
        self.q_proj = nn.Linear(c, c)
        self.out_proj = nn.Linear(c, c)


class _MLP(nn.Module):
    def __init__(self, c, inner):
        super().__init__()
        self.fc1 = nn.Linear(c, inner)
        self.fc2 = nn.Linear(inner, c)


class _Layer(nn.Module):
    def __init__(self, c, inner, eps):
        super().__init__()
        self.self_attn = _Attention(c)
        self.layer_norm1 = nn.LayerNorm(c, eps=eps)
        self.mlp = _MLP(c, inner)
        self.layer_norm2 = nn.LayerNorm(c, eps=eps)


class _Encoder(nn.Module):
    def __init__(self, n, c, inner, eps):
        super().__init__()
        self.layers = nn.ModuleList([_Layer(c, inner, eps) for _ in range(n)])


class _VisionModel(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        c, eps = cfg.hidden_size, cfg.layer_norm_eps
        self.embeddings = _Embeddings(c, cfg.patch_size, cfg.image_size, cfg.num_channels)
        self.pre_layrnorm = nn.LayerNorm(c, eps=eps)
        self.encoder = _Encoder(cfg.num_hidden_layers, c, cfg.intermediate_size, eps)
        self.post_layernorm = nn.LayerNorm(c, eps=eps)


class CLIPVisionModelWithProjection(nn.Module):
    """drop-in for transformers' CLIPVisionModelWithProjection as train_svd.py uses it (ViT with patch 14 at 224 x 224, GELU,
    head_dim 80): same state-dict keys and shapes, forward(pixel_values) -> .image_embeds / .last_hidden_state"""

    config_name = "config.json"

    def __init__(self, config=None, **kw):
        super().__init__()
        fields = dict(_DEFAULTS)
        if config is not None:
            src = config if isinstance(config, dict) else config.to_dict() if hasattr(config, "to_dict") else vars(config)
            fields.update({k: src[k] for k in _CONFIG_FIELDS if k in src})
        fields.update({k: v for k, v in kw.items() if k in _CONFIG_FIELDS})
        cfg = SimpleNamespace(**fields)
        c, heads = cfg.hidden_size, cfg.num_attention_heads
        if cfg.hidden_act != "gelu":
            raise ValueError(f"svd_xtend_b200 CLIP: hidden_act {cfg.hidden_act!r} is not supported (only 'gelu', the erf form)")
        if heads <= 0 or c % heads or c // heads != 80:
            raise ValueError(f"svd_xtend_b200 CLIP: head_dim must be 80 (hidden_size {c}, {heads} heads)")
        if c % 32 or cfg.intermediate_size % 32:
            raise ValueError("svd_xtend_b200 CLIP: hidden_size and intermediate_size must be multiples of 32")
        if cfg.patch_size != 14 or cfg.image_size % cfg.patch_size or (cfg.image_size // cfg.patch_size) ** 2 != 256:
            raise ValueError("svd_xtend_b200 CLIP: only patch_size 14 at image_size 224 (16 x 16 patches) is supported")
        if cfg.num_channels != 3:
            raise ValueError("svd_xtend_b200 CLIP: num_channels must be 3")
        self.config = cfg
        self.vision_model = _VisionModel(cfg)
        self.visual_projection = nn.Linear(c, cfg.projection_dim, bias=False)
        self.image_mean, self.image_std = CLIP_MEAN, CLIP_STD
        self._engine = Engine()

    @property
    def dtype(self):
        return next(self.parameters()).dtype

    @property
    def device(self):
        return next(self.parameters()).device

    @classmethod
    def from_pretrained(cls, path: str, subfolder: Optional[str] = "image_encoder", torch_dtype=None, variant: Optional[str] = None,
                        preprocessor_config: bool = False, **kw):
        """a local checkpoint directory: <path>/<subfolder>/config.json and model[.variant].safetensors or pytorch_model.bin.
        preprocessor_config=True also reads image_mean / image_std from <path>/feature_extractor/preprocessor_config.json
        (the defaults encode_image uses for this model)."""
        d = path if subfolder is None else os.path.join(path, subfolder)
        with open(os.path.join(d, cls.config_name)) as f:
            cfg = json.load(f)
        model = cls(cfg.get("vision_config", cfg))
        stems = ["model"] if variant is None else [f"model.{variant}", "model"]
        names = [s + ".safetensors" for s in stems] + ["pytorch_model" + ("" if variant is None else f".{variant}") + ".bin", "pytorch_model.bin"]
        for name in names:
            p = os.path.join(d, name)
            if not os.path.exists(p):
                continue
            if name.endswith(".safetensors"):
                from safetensors.torch import load_file
                sd = load_file(p)
            else:
                sd = torch.load(p, map_location="cpu")
            break
        else:
            raise FileNotFoundError(f"no model weights (model.safetensors / pytorch_model.bin) under {d}")
        sd = {k: v for k, v in sd.items() if not k.endswith("position_ids")}     # a non-persistent buffer in older checkpoints
        model.load_state_dict({k: v.float() for k, v in sd.items()}, strict=True)
        if torch_dtype is not None:
            model.to(torch_dtype)
        if preprocessor_config:
            with open(os.path.join(path, "feature_extractor", "preprocessor_config.json")) as f:
                pc = json.load(f)
            model.image_mean = tuple(float(v) for v in pc.get("image_mean", CLIP_MEAN))
            model.image_std = tuple(float(v) for v in pc.get("image_std", CLIP_STD))
        return model

    # ------------------------------------------------------------------ checks shared by forward and encode_image
    def _check_call(self, x: torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError("svd_xtend_b200: the CLIP image encoder only runs on a CUDA (sm_100a) device; there is no CPU fallback")
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            raise RuntimeError("svd_xtend_b200: CLIPVisionModelWithProjection is forward-only (the reference freezes the image encoder, "
                               "train_svd.py:660); call image_encoder.requires_grad_(False) / use torch.no_grad()")
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"svd_xtend_b200 CLIP: expected [B, 3, H, W] images, got {tuple(x.shape)}")
        for n, p in self.named_parameters():
            raw.dtype_code(p, f"parameter {n}")

    def forward(self, pixel_values: torch.Tensor, output_attentions: Optional[bool] = None, output_hidden_states: Optional[bool] = None,
                interpolate_pos_encoding: bool = False, return_dict: bool = True):
        """pixel_values [B, 3, 224, 224], already CLIP-normalised -> .image_embeds [B, projection_dim], .last_hidden_state
        [B, 257, hidden] in the parameter dtype"""
        if output_attentions or output_hidden_states:
            raise NotImplementedError("svd_xtend_b200 CLIP: output_attentions / output_hidden_states are not produced")
        if interpolate_pos_encoding:
            raise NotImplementedError("svd_xtend_b200 CLIP: interpolate_pos_encoding is not supported")
        self._check_call(pixel_values)
        if tuple(pixel_values.shape[-2:]) != (224, 224):
            raise ValueError("svd_xtend_b200 CLIP: forward takes 224 x 224 pixel_values (encode_image resizes)")
        B = pixel_values.shape[0]
        patches = torch.empty(B * 256, raw.CLIP_PATCH_KP, device=pixel_values.device, dtype=bf16)
        raw.clip_pixels(pixel_values.contiguous(), patches, resize=False)
        emb, hidden = self._run(patches, B)
        if not return_dict:
            return emb, hidden
        return SimpleNamespace(image_embeds=emb, last_hidden_state=hidden)

    def _run(self, patches: torch.Tensor, B: int):
        E = self._engine
        E.begin(recording=False)
        vm = self.vision_model
        emb = vm.embeddings
        C, S, dev = self.config.hidden_size, 257, patches.device
        heads = self.config.num_attention_heads
        pos = emb.position_embedding.weight
        pos_bf = E.wc.get(("clip_pos", id(pos)), [pos], (S, C), lambda buf: raw.prep_weight(pos.detach(), buf, 0, S, C))
        cls_row = E.wc.get(("clip_cls", id(emb.class_embedding), id(pos)), [emb.class_embedding, pos], (C,),
                           lambda buf: buf.copy_(emb.class_embedding.detach().float() + pos.detach()[0].float()), dtype=F32)
        wp = emb.patch_embedding.weight

        def build_patch(buf):
            tmp = torch.empty(C, raw.CLIP_PATCH_K, device=buf.device, dtype=bf16)
            raw.prep_weight(wp.detach().reshape(C, raw.CLIP_PATCH_K), tmp, 0, C, raw.CLIP_PATCH_K)
            buf.zero_()
            buf[:, :raw.CLIP_PATCH_K].copy_(tmp)
        w_patch = E.wc.get(("clip_patch", id(wp)), [wp], (C, raw.CLIP_PATCH_KP), build_patch)

        x0 = torch.empty(B * S, C, device=dev, dtype=bf16)
        x3 = x0.view(B, S, C)
        for b in range(B):
            raw.tapgemm_auto(patches[b * 256:(b + 1) * 256], w_patch, x3[b, 1:], M=256, N=C, K=raw.CLIP_PATCH_KP, res1=pos_bf[1:])
        raw.fill_rows(x3[:, 0], cls_row)
        _, h = E.layernorm(Var(x0), vm.pre_layrnorm)
        for layer in vm.encoder.layers:
            at = layer.self_attn
            _, y = E.layernorm(h, layer.layer_norm1)
            ws = [at.q_proj.weight, at.k_proj.weight, at.v_proj.weight]
            bs = [at.q_proj.bias, at.k_proj.bias, at.v_proj.bias]
            bcat = E.wc.get(("clip_qkv_bias",) + tuple(id(b) for b in bs), bs, (3 * C,),
                            lambda buf, bs=bs: buf.copy_(torch.cat([b.detach().float() for b in bs])), dtype=F32)
            qkv = E.linear(y, None, bcat, fused=ws).data
            o = torch.empty(B * S, C, device=dev, dtype=bf16)
            raw.attention_vit(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], o, heads=heads, S=S, nseq=B, scale=(C // heads) ** -0.5)
            h = E.linear(Var(o), at.out_proj.weight, at.out_proj.bias, res1=h)
            _, y = E.layernorm(h, layer.layer_norm2)
            f = E.linear(y, layer.mlp.fc1.weight, layer.mlp.fc1.bias, act=raw.ACT_GELU)
            h = E.linear(f, layer.mlp.fc2.weight, layer.mlp.fc2.bias, res1=h)
        pooled = torch.empty(B, C, device=dev, dtype=bf16)
        pln = vm.post_layernorm
        raw.layernorm_fwd(h.data.view(B, S * C)[:, :C], E.vec_f32(pln.weight), E.vec_f32(pln.bias), pln.eps, pooled)
        dt = self.dtype
        P = self.config.projection_dim
        if dt == bf16:
            out = E.linear(Var(pooled), self.visual_projection.weight).data
            hidden = h.data.view(B, S, C)
        else:
            out = E.linear(Var(pooled), self.visual_projection.weight, out_f32=True).data
            hidden = raw.cast_bf16_f32(h.data, torch.empty(B * S, C, device=dev, dtype=F32)).view(B, S, C)
            if dt != F32:
                out, hidden = out.to(dt), hidden.to(dt)
        return out.view(B, P), hidden


def encode_image(pixel_values: torch.Tensor, image_encoder: CLIPVisionModelWithProjection, mean=None, std=None) -> torch.Tensor:
    """train_svd.py:857-876 as one function: [B, 3, H, W] frames in [-1, 1] (H, W >= 14) -> image_embeds [B, projection_dim].
    mean / std default to the model's image_mean / image_std (the CLIPImageProcessor defaults unless from_pretrained read a
    preprocessor config)."""
    image_encoder._check_call(pixel_values)
    mean = image_encoder.image_mean if mean is None else mean
    std = image_encoder.image_std if std is None else std
    B = pixel_values.shape[0]
    patches = torch.empty(B * 256, raw.CLIP_PATCH_KP, device=pixel_values.device, dtype=bf16)
    raw.clip_pixels(pixel_values.contiguous(), patches, resize=True, mean=mean, std=std)
    return image_encoder._run(patches, B)[0]
