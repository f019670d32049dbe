"""Launcher shim: run the reference's training scripts UNCHANGED on the B200 path.

    python -m svd_xtend_b200.shim train_svd.py --pretrained_model_name_or_path=... [script args]
    accelerate launch -m svd_xtend_b200.shim train_svd.py ...

Before the script body runs, the replacement class is installed under the two names the reference
imports the UNet from: `diffusers.UNetSpatioTemporalConditionModel` (train_svd.py:49) and
`src.unet_spatio_temporal_condition.UNetSpatioTemporalConditionModel` (train_svd_lora.py:60). When `transformers` is
importable, the CLIP image encoder is also installed as `transformers.CLIPVisionModelWithProjection` (train_svd.py:43,
train_svd_lora.py:43); the scripts' CLIPImageProcessor stays transformers' own.
diffusers / accelerate are NOT part of this image (no network), so this shim is exercised only where a
user's environment provides them; it fails loudly when they are missing.
"""
from __future__ import annotations

import importlib
import runpy
import sys
import types


def install() -> None:
    from .unet import UNetSpatioTemporalConditionModel
    try:
        diffusers = importlib.import_module("diffusers")
    except ModuleNotFoundError as e:
        raise RuntimeError("svd_xtend_b200.shim: the reference scripts need `diffusers`, which is not installed here") from e
    diffusers.UNetSpatioTemporalConditionModel = UNetSpatioTemporalConditionModel
    for modname in ("diffusers.models", "diffusers.models.unets", "diffusers.models.unets.unet_spatio_temporal_condition"):
        try:
            m = importlib.import_module(modname)
            setattr(m, "UNetSpatioTemporalConditionModel", UNetSpatioTemporalConditionModel)
        except Exception:
            pass
    # train_svd_lora.py imports `from src.unet_spatio_temporal_condition import UNetSpatioTemporalConditionModel`
    pkg = sys.modules.get("src") or types.ModuleType("src")
    pkg.__path__ = getattr(pkg, "__path__", [])
    sub = types.ModuleType("src.unet_spatio_temporal_condition")
    sub.UNetSpatioTemporalConditionModel = UNetSpatioTemporalConditionModel
    sys.modules["src"] = pkg
    sys.modules["src.unet_spatio_temporal_condition"] = sub
    pkg.unet_spatio_temporal_condition = sub
    install_clip()


def install_clip() -> bool:
    """install svd_xtend_b200.clip.CLIPVisionModelWithProjection as transformers.CLIPVisionModelWithProjection; False when
    transformers is not importable (the scripts then fail on their own import, as before)"""
    from .clip import CLIPVisionModelWithProjection
    try:
        transformers = importlib.import_module("transformers")
    except ModuleNotFoundError:
        return False
    transformers.CLIPVisionModelWithProjection = CLIPVisionModelWithProjection
    return True


def main(argv=None) -> None:
    argv = list(sys.argv[1:] if argv is None else argv)
    if not argv:
        raise SystemExit("usage: python -m svd_xtend_b200.shim <train_svd.py|train_svd_lora.py> [args...]")
    install()
    script = argv[0]
    sys.argv = argv
    runpy.run_path(script, run_name="__main__")


if __name__ == "__main__":
    main()
