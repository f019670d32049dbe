"""ORACLE / test infrastructure — run the reference's OWN top-level file on top of the oracle's blocks.

/root/reference/src/unet_spatio_temporal_condition.py is real reference code (construction :71-246, forward :357-490,
attention-processor plugin API :248-321, gradient-checkpointing hook :323-325, forward chunking :328-355), but it
cannot be imported here because its lines 7-13 import the absent `diffusers`. This module builds a minimal stand-in
`diffusers` package in `sys.modules` — ONLY the names that file imports — whose block classes are the oracle's
restatements, imports the reference file from where it lies, and returns its `UNetSpatioTemporalConditionModel`.

What that pins: the oracle's top-level wiring (oracle.UNetSpatioTemporalConditionModel) against the reference's own
statement of it, on identical blocks: constructor channel bookkeeping, state-dict names, the forward's embedding /
repeat / skip-connection order, the plugin API. What it does NOT pin: the arithmetic inside the blocks, which both
sides take from the oracle (that part stays "parity unpinned" against diffusers — see oracle/svd_unet_oracle.py).

Used by tests/golden/make_ref_wiring_golden.py, which writes the committed fixture that tests/test_reference_wiring.py
checks the oracle against. Nothing here is imported by the product path.
"""
from __future__ import annotations

import contextlib
import functools
import importlib.util
import inspect
import os
import sys
import types

import torch.nn as nn

from . import svd_unet_oracle as O

REFERENCE_FILE = os.path.join("src", "unet_spatio_temporal_condition.py")


def _register_to_config(init):
    """[D] configuration_utils.register_to_config: record the constructor arguments on self.config (attribute access)."""
    sig = inspect.signature(init)

    @functools.wraps(init)
    def wrapped(self, *args, **kwargs):
        bound = sig.bind(self, *args, **kwargs)
        bound.apply_defaults()
        cfg = {k: v for k, v in bound.arguments.items() if k != "self"}
        init(self, *args, **kwargs)
        self.config = types.SimpleNamespace(**cfg)
    return wrapped


class _ModelMixin(nn.Module):
    """[D] modeling_utils.ModelMixin, reduced to what the reference file and train_svd.py:732 use."""

    def enable_gradient_checkpointing(self):
        self.apply(lambda m: self._set_gradient_checkpointing(m, value=True))


class _Empty:
    pass


class _BaseOutput:
    """[D] utils.BaseOutput: a dataclass base with tuple-style access."""

    def __getitem__(self, i):
        return tuple(getattr(self, f) for f in self.__dataclass_fields__)[i]


def _get_down_block(down_block_type, num_layers, in_channels, out_channels, temb_channels, add_downsample, num_attention_heads=None,
                    cross_attention_dim=None, transformer_layers_per_block=1, **ignored):
    # the reference passes resnet_eps / resnet_act_fn too (:170-182); diffusers' get_down_block does not forward them to
    # the spatio-temporal blocks [D], and neither does the oracle's
    return O.get_down_block(down_block_type, num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                            temb_channels=temb_channels, add_downsample=add_downsample, num_attention_heads=num_attention_heads,
                            cross_attention_dim=cross_attention_dim, transformer_layers_per_block=transformer_layers_per_block)


def _get_up_block(up_block_type, num_layers, in_channels, out_channels, prev_output_channel, temb_channels, add_upsample,
                  num_attention_heads=None, cross_attention_dim=None, transformer_layers_per_block=1, **ignored):
    return O.get_up_block(up_block_type, num_layers=num_layers, in_channels=in_channels, out_channels=out_channels,
                          prev_output_channel=prev_output_channel, temb_channels=temb_channels, add_upsample=add_upsample,
                          num_attention_heads=num_attention_heads, cross_attention_dim=cross_attention_dim,
                          transformer_layers_per_block=transformer_layers_per_block)


def _stub_modules():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    class _Logging:
        @staticmethod
        def get_logger(name):
            import logging
            return logging.getLogger(name)

    mods = {
        "diffusers": mod("diffusers", __path__=[]),
        "diffusers.configuration_utils": mod("diffusers.configuration_utils", ConfigMixin=_Empty, register_to_config=_register_to_config),
        "diffusers.loaders": mod("diffusers.loaders", UNet2DConditionLoadersMixin=type("UNet2DConditionLoadersMixin", (), {}),
                                 PeftAdapterMixin=type("PeftAdapterMixin", (), {})),
        "diffusers.utils": mod("diffusers.utils", BaseOutput=_BaseOutput, logging=_Logging),
        "diffusers.models": mod("diffusers.models", __path__=[]),
        "diffusers.models.attention_processor": mod("diffusers.models.attention_processor",
                                                    CROSS_ATTENTION_PROCESSORS=(O.AttnProcessor, O.AttnProcessor2_0),
                                                    AttentionProcessor=object, AttnProcessor=O.AttnProcessor),
        "diffusers.models.embeddings": mod("diffusers.models.embeddings", TimestepEmbedding=O.TimestepEmbedding, Timesteps=O.Timesteps),
        "diffusers.models.modeling_utils": mod("diffusers.models.modeling_utils", ModelMixin=_ModelMixin),
        "diffusers.models.unets": mod("diffusers.models.unets", __path__=[]),
        "diffusers.models.unets.unet_3d_blocks": mod("diffusers.models.unets.unet_3d_blocks",
                                                     UNetMidBlockSpatioTemporal=O.UNetMidBlockSpatioTemporal,
                                                     get_down_block=_get_down_block, get_up_block=_get_up_block),
    }
    return mods


@contextlib.contextmanager
def _stubbed_diffusers():
    mods = _stub_modules()
    saved = {k: sys.modules.get(k) for k in mods}
    sys.modules.update(mods)
    try:
        yield
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def load_reference_unet_class(reference_root: str):
    """import <reference_root>/src/unet_spatio_temporal_condition.py (unmodified, from where it lies) over the stand-in
    diffusers namespace and return its UNetSpatioTemporalConditionModel class"""
    path = os.path.join(reference_root, REFERENCE_FILE)
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    with _stubbed_diffusers():
        spec = importlib.util.spec_from_file_location("_svdx_reference_unet", path)
        module = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(module)
    return module.UNetSpatioTemporalConditionModel
