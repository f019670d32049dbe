"""The oracle's (and the product class's) top-level wiring against the REFERENCE'S OWN file.

tests/golden/ref_wiring_tiny.pt was produced by importing the reference's src/unet_spatio_temporal_condition.py unmodified
(tests/golden/make_ref_wiring_golden.py, through oracle/ref_wiring.py) and running it in fp64 on two clips. These CPU tests
need only the committed fixture.
What is pinned: construction (:71-246), forward wiring (:357-490), plugin-API key set (:248-274), parameter census of the SVD
configuration, the gradients of one training-mode step. The arithmetic inside the blocks is the oracle's on both sides
(unpinned against diffusers)."""
import hashlib
import importlib.util
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_wiring_tiny.pt")


def _gen():
    spec = importlib.util.spec_from_file_location("make_ref_wiring_golden", os.path.join(ROOT, "tests", "golden", "make_ref_wiring_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def gold():
    return torch.load(GOLDEN, weights_only=False)


def test_oracle_forward_equals_reference_file_golden(gold):
    from oracle.svd_unet_oracle import UNetSpatioTemporalConditionModel as Oracle
    gen = _gen()
    m = gen.build(Oracle)
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == gold["tiny_keys"]
    chk = float(sum(p.detach().double().abs().sum() for p in m.parameters()))
    assert abs(chk - gold["tiny_param_checksum"]) < 1e-9 * gold["tiny_param_checksum"], "seeded init differs from the generator's"
    b = gen.batch()
    with torch.no_grad():
        out = m(b["sample"], b["timestep"].double(), b["encoder_hidden_states"], b["added_time_ids"]).sample
    assert out.shape == gold["tiny_out"].shape == (2, 4, 4, 16, 16)
    err = ((out - gold["tiny_out"]).norm() / gold["tiny_out"].norm()).item()
    assert err < 1e-12, err      # identical blocks, identical wiring: fp64 round-off only
    assert sorted(m_name + ".processor" for m_name, mod in m.named_modules() if hasattr(mod, "get_processor")) == gold["tiny_attn_processor_keys"]


def test_svd_configuration_census_equals_reference_file(gold):
    """names, shapes and counts the reference's constructor produces for the SVD configuration: oracle AND product class"""
    from oracle.svd_unet_oracle import SVD_CONFIG, UNetSpatioTemporalConditionModel as Oracle
    from svd_xtend_b200.unet import UNetSpatioTemporalConditionModel as Ours
    assert gold["svd_total_params"] == 1_524_623_082 and gold["svd_temporal_params"] == 397_620_480
    for cls in (Oracle, Ours):
        with torch.device("meta"):
            m = cls(**SVD_CONFIG)
        keys = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
        assert len(keys) == gold["svd_num_keys"]
        assert hashlib.sha256(repr(keys).encode()).hexdigest() == gold["svd_keys_sha256"], cls
        assert m.num_upsamplers == gold["svd_num_upsamplers"]
    assert len(m.attn_processors) == gold["svd_attn_processors"] == 64


def test_product_class_plugin_keys_equal_reference_file(gold):
    from oracle.svd_unet_oracle import TINY_CONFIG
    from svd_xtend_b200.unet import UNetSpatioTemporalConditionModel as Ours
    m = Ours(**TINY_CONFIG)
    assert sorted(m.attn_processors.keys()) == gold["tiny_attn_processor_keys"]
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == gold["tiny_keys"]


def test_live_reference_file_vs_oracle(gold):
    """one training-mode step of the oracle against the same step of the reference file, as the fixture recorded it:
    initial state dict, output, loss and every trainable gradient (fp64 on both sides: round-off only), plus the
    reference's gradient-checkpointing hook and its plugin-API error on a mismatched processor dict"""
    from oracle.svd_unet_oracle import TINY_CONFIG, UNetSpatioTemporalConditionModel as Oracle
    from svd_xtend_b200.unet import UNetSpatioTemporalConditionModel as Ours
    gen = _gen()
    ora = gen.build(Oracle)
    sums = gen.state_sums(ora)
    assert list(sums) == list(gold["train_state_sums"])
    for k, (s, a) in gold["train_state_sums"].items():
        assert abs(sums[k][0] - s) <= 1e-12 * a and abs(sums[k][1] - a) <= 1e-12 * a, k
    out, loss = gen.train_step(ora, gen.batch())
    assert ((out - gold["tiny_out"]).norm() / gold["tiny_out"].norm()).item() < 1e-12
    assert abs(float(loss) - gold["train_loss"]) < 1e-12 * gold["train_loss"]
    trainable = {n: p for n, p in ora.named_parameters() if p.requires_grad}
    assert sorted(trainable) == sorted(list(gold["train_grads"]) + gold["train_zero_grads"])
    for n in gold["train_zero_grads"]:
        assert float(trainable[n].grad.abs().max()) == 0.0, n
    for n, rec in gold["train_grads"].items():
        g = trainable[n].grad.reshape(-1)
        assert torch.equal(gen.grad_sample_index(g.numel()), rec["idx"]), n
        assert abs(float(g.norm()) - rec["norm"]) <= 1e-10 * rec["norm"], n
        assert (g[rec["idx"]] - rec["val"]).abs().max().item() <= 1e-10 * rec["norm"], n
    assert sum(1 for m in ora.modules() if hasattr(m, "gradient_checkpointing")) == gold["grad_ckpt_modules"]
    ours = Ours(**TINY_CONFIG)
    ours.enable_gradient_checkpointing()
    assert sum(bool(getattr(m, "gradient_checkpointing", False)) for m in ours.modules()) == gold["grad_ckpt_modules"]
    with pytest.raises(Exception) as err:
        ours.set_attn_processor({})
    assert type(err.value).__name__ == gold["set_attn_processor_mismatch_error"]
