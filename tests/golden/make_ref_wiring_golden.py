"""Generates tests/golden/ref_wiring_tiny.pt by running the REFERENCE'S OWN top-level file.

    python tests/golden/make_ref_wiring_golden.py <reference checkout>

<reference checkout>/src/unet_spatio_temporal_condition.py is imported unmodified from where it lies (oracle/ref_wiring.py
provides a stand-in for the absent `diffusers` package whose block classes are the oracle's), instantiated with the
small test topology and run in fp64 on a batch of TWO clips. The fixture freezes what the reference's file itself
decides: state-dict names and shapes, channel bookkeeping of the down / mid / up blocks, the order of embedding
repeats and skip connections in forward(), the attention-processor key set — so the oracle's top-level restatement
(and through it the CUDA path) is pinned to reference code, not to a recollection of it. The block arithmetic is the
oracle's on both sides and stays unpinned against diffusers (see the header of oracle/svd_unet_oracle.py).

It also records one training-mode step of the reference file (loss = mean square of the output, the as-scripted
trainable set): per-tensor sums of its initial state dict, the loss, and for every trainable parameter the gradient
norm and the gradient at GRAD_SAMPLES seeded positions, plus what its plugin API and gradient-checkpointing hook do.
"""
import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_wiring import REFERENCE_FILE, load_reference_unet_class  # noqa: E402
from oracle.svd_unet_oracle import SVD_CONFIG, TINY_CONFIG, synthetic_batch  # noqa: E402

SEED = 20260923
GRAD_SAMPLES = 64


def build(cls):
    torch.manual_seed(SEED)
    m = cls(**TINY_CONFIG).double()
    with torch.no_grad():      # de-symmetrise what default init leaves at constants, so that every affine / blend path matters
        g = torch.Generator().manual_seed(SEED + 1)
        for n, p in m.named_parameters():
            if "norm" in n or n.endswith("bias") or n.endswith("mix_factor"):
                p.add_(0.1 * torch.randn(p.shape, generator=g, dtype=p.dtype))
    return m.eval()


def batch():
    return synthetic_batch(2, 4, 16, 16, seed=4321, cross_dim=TINY_CONFIG["cross_attention_dim"], dtype=torch.float64)


def train_step(m, b):
    """one training-mode step on the as-scripted trainable set; returns (output, loss)"""
    m.train()
    m.requires_grad_(False)
    for n, p in m.named_parameters():
        if "temporal_transformer_block" in n:
            p.requires_grad_(True)
    out = m(b["sample"], b["timestep"].double(), b["encoder_hidden_states"], b["added_time_ids"]).sample
    loss = out.square().mean()
    loss.backward()
    return out.detach(), loss.detach()


def grad_sample_index(numel):
    """the GRAD_SAMPLES positions (sorted, all of them for a small tensor) at which a gradient is recorded"""
    if numel <= GRAD_SAMPLES:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(SEED + numel))[:GRAD_SAMPLES].sort().values


def state_sums(m):
    return {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in m.state_dict().items()}


def main(reference_root):
    Ref = load_reference_unet_class(reference_root)
    ref = build(Ref)
    b = batch()
    with torch.no_grad():
        out = ref(b["sample"], b["timestep"].double(), b["encoder_hidden_states"], b["added_time_ids"]).sample
        out_t = ref(b["sample"], b["timestep"].double(), b["encoder_hidden_states"], b["added_time_ids"], return_dict=False)[0]
    assert torch.equal(out, out_t)
    with torch.device("meta"):
        big = Ref(**SVD_CONFIG)
    big_keys = [(k, tuple(v.shape)) for k, v in big.state_dict().items()]

    train = build(Ref)
    sums = state_sums(train)
    train_out, train_loss = train_step(train, b)
    assert ((train_out - out).norm() / out.norm()).item() < 1e-12
    grads, zero_grads = {}, []
    for n, p in train.named_parameters():
        if not p.requires_grad:
            continue
        g = p.grad.reshape(-1)
        if g.abs().max() == 0:
            zero_grads.append(n)
            continue
        idx = grad_sample_index(g.numel())
        grads[n] = {"norm": float(g.norm()), "idx": idx, "val": g[idx].clone()}
    train.enable_gradient_checkpointing()
    ckpt_modules = sum(bool(getattr(m, "gradient_checkpointing", False)) for m in train.modules())
    try:
        train.set_attn_processor({})
        mismatch_error = None
    except Exception as e:  # noqa: BLE001
        mismatch_error = type(e).__name__

    fixture = {
        "seed": SEED,
        "reference_file_sha256": hashlib.sha256(open(os.path.join(reference_root, REFERENCE_FILE), "rb").read()).hexdigest(),
        "tiny_keys": [(k, tuple(v.shape)) for k, v in ref.state_dict().items()],
        "tiny_param_checksum": float(sum(p.double().abs().sum() for p in ref.parameters())),
        "tiny_out": out.clone(),
        "tiny_attn_processor_keys": sorted(ref.attn_processors.keys()),
        "svd_keys_sha256": hashlib.sha256(repr(big_keys).encode()).hexdigest(),
        "svd_num_keys": len(big_keys),
        "svd_total_params": sum(v.numel() for v in big.state_dict().values()),
        "svd_temporal_params": sum(p.numel() for n, p in big.named_parameters() if "temporal_transformer_block" in n),
        "svd_num_upsamplers": big.num_upsamplers,
        "svd_attn_processors": len(big.attn_processors),
        "train_state_sums": sums,
        "train_loss": float(train_loss),
        "train_grads": grads,
        "train_zero_grads": zero_grads,
        "grad_ckpt_modules": ckpt_modules,
        "set_attn_processor_mismatch_error": mismatch_error,
    }
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_wiring_tiny.pt")
    torch.save(fixture, path)
    print("wrote", path, "out std", float(out.std()), "svd params", fixture["svd_total_params"], fixture["svd_temporal_params"],
          "processors", fixture["svd_attn_processors"], "train loss", fixture["train_loss"], "sampled grads", len(grads),
          "zero grads", len(zero_grads))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(f"usage: python {sys.argv[0]} <reference checkout>")
    main(sys.argv[1])
