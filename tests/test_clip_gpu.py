"""CLIP image encoder on the B200 path (svd_xtend_b200/clip.py) and its three kernels against fp32 / fp64 references:
the GELU epilogue of svdx_tapgemm (1-CTA, CTA-pair and split-K forms), svdx_attention_vit_fwd (head_dim 80), svdx_clip_pixels,
and the whole encoder against the oracle (oracle/svd_clip_oracle.py, pinned to transformers by tests/test_clip.py), built and
run on the device with TF32 off. Tolerance of the whole encoder, as for the UNet and VAE: rel-L2 of image_embeds and
last_hidden_state <= max(2 x err(oracle under torch bf16 autocast), 2e-2)."""
import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


@pytest.fixture(autouse=True)
def _no_tf32():
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


# ----------------------------------------------------------------------------- GELU epilogue
def _gemm_operands(M, N, K, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    a = torch.randn(M, K, generator=g, device=DEV).to(torch.bfloat16)
    w = (torch.randn(N, K, generator=g, device=DEV) / K ** 0.5).to(torch.bfloat16)
    b = 0.5 * torch.randn(N, generator=g, device=DEV)
    r = torch.randn(M, N, generator=g, device=DEV).to(torch.bfloat16)
    return a, w, b, r


@pytest.mark.parametrize("M", [257, 514, 2056])
@pytest.mark.parametrize("N", [1280, 5120])
@pytest.mark.parametrize("bias,res", [(False, False), (True, False), (True, True)])
def test_gelu_epilogue_whole(M, N, bias, res):
    """one launch: 1-CTA tiles at M = 257, CTA-pair tiles at M >= 512"""
    from svd_xtend_b200 import raw
    K = 1280
    a, w, b, r = _gemm_operands(M, N, K, M + N)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    raw.tapgemm(a, w, out, M=M, N=N, K=K, bias=b if bias else None, res1=r if res else None, act=raw.ACT_GELU, block_n=256)
    ref = F.gelu(a.float() @ w.float().t() + (b if bias else 0.0)) + (r.float() if res else 0.0)
    assert raw.pair_eligible(M, N, 256, False) == (M >= 512)
    assert _rel(out, ref) < 1e-2


@pytest.mark.parametrize("K", [1280, 5120])
@pytest.mark.parametrize("bias,res", [(False, False), (True, False), (True, True)])
def test_gelu_epilogue_split_k(K, bias, res):
    """M = 257 (one image): the split-K path with the activation in svdx_splitk_epilogue_act"""
    from svd_xtend_b200 import raw
    M, N = 257, 1280
    assert raw.split_plan(True, M, N, K) is not None
    a, w, b, r = _gemm_operands(M, N, K, K)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    raw.tapgemm_auto(a, w, out, M=M, N=N, K=K, bias=b if bias else None, res1=r if res else None, act=raw.ACT_GELU)
    ref = F.gelu(a.float() @ w.float().t() + (b if bias else 0.0)) + (r.float() if res else 0.0)
    assert _rel(out, ref) < 1e-2


def test_gelu_epilogue_refused_with_geglu_and_gn_sum():
    from svd_xtend_b200 import raw
    from svd_xtend_b200._lib import SvdxError
    M, N, K = 256, 256, 256
    a, w, _, _ = _gemm_operands(M, N, K, 1)
    with pytest.raises(SvdxError):
        raw.tapgemm(a, w, torch.empty(M, N // 2, device=DEV, dtype=torch.bfloat16), M=M, N=N, K=K, geglu=True, act=raw.ACT_GELU)
    gs = torch.zeros(1, 2, N, device=DEV)
    with pytest.raises(SvdxError):
        raw.tapgemm(a, w, torch.empty(M, N, device=DEV, dtype=torch.bfloat16), M=M, N=N, K=K, gn_sum=gs, gn_rows=M, act=raw.ACT_GELU)
    with pytest.raises(SvdxError):
        raw.tapgemm(a, w, torch.empty(M, N, device=DEV, dtype=torch.float32), M=M, N=N, K=K, act=raw.ACT_GELU)


# ----------------------------------------------------------------------------- attention_vit
@pytest.mark.parametrize("S", [1, 17, 64, 65, 257, 512])
@pytest.mark.parametrize("B", [1, 2, 8])
def test_attention_vit(S, B):
    from svd_xtend_b200 import raw
    H, D = 16, 80
    C = H * D
    g = torch.Generator(device=DEV).manual_seed(S * 31 + B)
    qkv = (2.0 * torch.randn(B * S, 3 * C, generator=g, device=DEV)).to(torch.bfloat16)
    o = torch.full((B * S, C + 16), 7.0, device=DEV, dtype=torch.bfloat16)
    raw.attention_vit(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], o, heads=H, S=S, nseq=B, scale=D ** -0.5)
    q, k, v = (t.float().view(B, S, H, D).transpose(1, 2) for t in qkv.split(C, dim=1))
    ref = torch.softmax((q @ k.transpose(-1, -2)) * D ** -0.5, dim=-1) @ v
    ref = ref.transpose(1, 2).reshape(B * S, C)
    assert _rel(o[:, :C], ref) < 1e-2
    assert bool((o[:, C:] == 7.0).all()), "columns outside the heads were written"


def test_attention_vit_refuses_long_sequences():
    from svd_xtend_b200 import raw
    from svd_xtend_b200._lib import SvdxError
    C = 1280
    qkv = torch.zeros(513, 3 * C, device=DEV, dtype=torch.bfloat16)
    with pytest.raises(SvdxError):
        raw.attention_vit(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], torch.empty(513, C, device=DEV, dtype=torch.bfloat16),
                          heads=16, S=513, nseq=1)


# ----------------------------------------------------------------------------- clip_pixels
def _bf16_ulp_ok(ours, ref64):
    """|ours - bf16(ref)| <= one bf16 ulp at the larger magnitude"""
    refb = ref64.to(torch.bfloat16).double()
    o = ours.double()
    mag = torch.maximum(o.abs(), refb.abs()).clamp_min(1e-30)
    ulp = torch.exp2(torch.floor(torch.log2(mag)) - 7)
    return bool(((o - refb).abs() <= ulp * 1.0000001).all())


@pytest.mark.parametrize("H,W,B", [(320, 512, 2), (576, 1024, 2), (128, 128, 1), (224, 224, 2)])
def test_clip_pixels_resize(H, W, B):
    from oracle.svd_clip_oracle import CLIP_MEAN, CLIP_STD, patchify, preprocess
    from svd_xtend_b200 import raw
    g = torch.Generator(device=DEV).manual_seed(H + W)
    x = torch.rand(B, 3, H, W, generator=g, device=DEV) * 2 - 1
    out = torch.full((B * 256, 592), float("nan"), device=DEV, dtype=torch.bfloat16)
    raw.clip_pixels(x, out, resize=True, mean=CLIP_MEAN, std=CLIP_STD)
    ref = patchify(preprocess(x.double()))
    assert bool((out[:, 588:] == 0).all())
    assert _bf16_ulp_ok(out[:, :588], ref)


def test_clip_pixels_patchify_only():
    from oracle.svd_clip_oracle import patchify
    from svd_xtend_b200 import raw
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator(device=DEV).manual_seed(3), device=DEV)
    out = torch.full((512, 592), float("nan"), device=DEV, dtype=torch.bfloat16)
    raw.clip_pixels(x, out, resize=False)
    assert torch.equal(out[:, :588], patchify(x).to(torch.bfloat16))
    assert bool((out[:, 588:] == 0).all())


# ----------------------------------------------------------------------------- the whole encoder
_MODELS = {}


def _models(name):
    """(oracle fp32, ours fp32) on the device with seeded weights, norms and biases de-symmetrised (built once per config)"""
    if name not in _MODELS:
        from oracle.svd_clip_oracle import CLIP_CONFIG, TINY_CLIP_CONFIG, CLIPVisionModelWithProjection as Oracle, init_weights
        from svd_xtend_b200.clip import CLIPVisionModelWithProjection as Ours
        cfg = CLIP_CONFIG if name == "svd" else TINY_CLIP_CONFIG
        with torch.device(DEV):
            oracle = init_weights(Oracle(**cfg), 1234).eval().requires_grad_(False)
            ours = Ours(**cfg).eval().requires_grad_(False)
        ours.load_state_dict(oracle.state_dict())
        _MODELS.clear()
        _MODELS[name] = (oracle, ours)
    return _MODELS[name]


def _oracle_outputs(oracle, x, path):
    from oracle.svd_clip_oracle import preprocess
    with torch.no_grad():
        px = preprocess(x) if path == "encode" else x
        ref = oracle(px)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ac = oracle(px)
    tol_e = max(2 * _rel(ac.image_embeds.float(), ref.image_embeds), 2e-2)
    tol_h = max(2 * _rel(ac.last_hidden_state.float(), ref.last_hidden_state), 2e-2)
    return ref, tol_e, tol_h


def _inputs(B, path, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    if path == "encode":
        return torch.rand(B, 3, 320, 512, generator=g, device=DEV) * 2 - 1
    return torch.randn(B, 3, 224, 224, generator=g, device=DEV)


@pytest.mark.parametrize("name,B", [("tiny", 1), ("tiny", 3), ("svd", 1), ("svd", 2)])
@pytest.mark.parametrize("path", ["forward", "encode"])
def test_encoder_matches_oracle(name, B, path):
    from svd_xtend_b200.clip import encode_image
    oracle, ours = _models(name)
    x = _inputs(B, path, 10 * B + (path == "encode"))
    ref, tol_e, tol_h = _oracle_outputs(oracle, x, path)
    with torch.no_grad():
        if path == "encode":
            emb = encode_image(x, ours)
            hid = None
        else:
            out = ours(x)
            emb, hid = out.image_embeds, out.last_hidden_state
    torch.cuda.synchronize()
    assert emb.dtype == torch.float32 and emb.shape == ref.image_embeds.shape
    e = _rel(emb, ref.image_embeds)
    assert e <= tol_e, (e, tol_e)
    if hid is not None:
        assert hid.shape == ref.last_hidden_state.shape
        h = _rel(hid, ref.last_hidden_state)
        assert h <= tol_h, (h, tol_h)


@pytest.mark.parametrize("name", ["tiny", "svd"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_encoder_half_precision_parameters(name, dtype):
    """image_encoder.to(dtype=weight_dtype) (train_svd.py:672): outputs in that dtype, checked against the fp32 oracle holding
    the same rounded parameters"""
    import copy
    oracle, ours = _models(name)
    ours_h = copy.deepcopy(ours).to(dtype)
    oracle_r = copy.deepcopy(oracle)
    with torch.no_grad():
        for p_o, p_h in zip(oracle_r.parameters(), ours_h.parameters()):
            p_o.copy_(p_h.float())
    x = _inputs(1, "forward", 77)
    ref, tol_e, tol_h = _oracle_outputs(oracle_r, x, "forward")
    with torch.no_grad():
        out = ours_h(x.to(dtype))
    assert out.image_embeds.dtype == dtype and out.last_hidden_state.dtype == dtype
    assert _rel(out.image_embeds, ref.image_embeds) <= tol_e
    assert _rel(out.last_hidden_state, ref.last_hidden_state) <= tol_h
    del ours_h, oracle_r


def test_encode_image_graph_capture():
    """encode_image at B = 1 captured in a CUDA graph and replayed on new frames. The replay must compute the NEW frames: it
    meets the encoder tolerance against the oracle on them, and it is far closer to an eager call on them than an eager call on
    the capture-time frames is. Against the eager call itself bitwise equality is impossible (split-K fp32 atomics change the
    summation order from call to call); two eager calls on the same frames already differ by ~1e-2 rel-L2 at the SVD
    configuration with random weights (bf16 rounding flips amplified over 32 layers; 1.03e-2 measured between replay and eager
    on a B200), so that comparison is held to the 2e-2 floor of the encoder tolerance."""
    from svd_xtend_b200.clip import encode_image
    oracle, ours = _models("svd")
    static = _inputs(1, "encode", 5)
    with torch.no_grad():
        before = encode_image(static.clone(), ours)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                encode_image(static, ours)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = encode_image(static, ours)
        fresh = _inputs(1, "encode", 6)
        static.copy_(fresh)
        graph.replay()
        torch.cuda.synchronize()
        replayed = out.clone()
        eager = encode_image(fresh, ours)
        eager2 = encode_image(fresh, ours)
        graph.replay()
        torch.cuda.synchronize()
    ref, tol_e, _ = _oracle_outputs(oracle, fresh, "encode")
    d_replay, d_eager, d_frames = _rel(replayed, eager), _rel(eager2, eager), _rel(before, eager)
    print(f"replay vs eager {d_replay:.3g}, eager vs eager {d_eager:.3g}, capture-time frames vs new {d_frames:.3g}")
    assert _rel(replayed, ref.image_embeds) <= tol_e
    assert d_replay <= 2e-2 and d_replay < 0.25 * d_frames
    assert _rel(out, replayed) <= 2e-2        # a second replay


def test_forward_only_refusal():
    oracle, ours = _models("tiny")
    ours.requires_grad_(True)
    try:
        with torch.enable_grad(), pytest.raises(RuntimeError, match="forward-only"):
            ours(_inputs(1, "forward", 1))
    finally:
        ours.requires_grad_(False)
