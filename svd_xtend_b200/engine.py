"""Execution engine of the B200 SVD-UNet step: a hand-rolled tape over the C-ABI kernels.

Design (B200-first, not a translation of diffusers' module-by-module autograd graph):
  * activations live as token-major channels-last bf16 matrices ``[B*T*H*W, C]`` for the WHOLE
    network — the (BT,C,H,W)<->(BT,HW,C)<->(B*HW,T,C) permutes of the reference
    (SURVEY.md K13) never happen: linears are row-permutation invariant, the temporal conv and
    temporal attention address frames through strides (TMA tensor maps);
  * every op is one or two kernel launches through ``raw`` (ctypes -> extern "C"); the forward
    pushes a backward closure on a tape, the backward pops them — no torch autograd graph, no
    torch kernels on the path, so the whole step can be captured in one CUDA graph;
  * fan-out gradient accumulation, parameter-gradient accumulation (fp32) and the weight-operand
    cache (fp32 master -> bf16 forward / transposed dgrad layouts) are explicit.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence, Tuple

import os

import torch

from . import raw
from .raw import A_CONV2D, A_ROWS, OUT_F32_ATOMIC, bf16

F32 = torch.float32


class Var:
    """An activation on the tape: bf16 ``[rows, C]`` data plus (lazily) its gradient."""

    __slots__ = ("data", "grad", "needs_grad", "owned", "csum", "gnb", "gnb_sums")

    def __init__(self, data: torch.Tensor, needs_grad: bool = False):
        self.data = data
        self.grad: Optional[torch.Tensor] = None
        self.needs_grad = needs_grad
        self.owned = False  # True when .grad is a tensor no other Var can see (safe to accumulate in place)
        # fused GroupNorm statistics of this tensor, produced by the GEMM / conv epilogue that wrote it:
        # (rows per statistics slab, [(fp32 [slabs, 2, C_i] channel sums, C_i), ...]) — several parts after a channel concat
        self.csum = None
        # set on a GroupNorm OUTPUT: what the dgrad epilogue of its consumer needs to accumulate the GroupNorm-backward sums
        # (dict x / x2 / ab / rows / silu); gnb_sums = (fp32 [slabs, 2, C] sums, the gradient tensor they were computed on)
        self.gnb = None
        self.gnb_sums = None

    def take_grad(self) -> Optional[torch.Tensor]:
        g, self.grad, self.owned = self.grad, None, False
        return g

    @property
    def rows(self) -> int:
        return self.data.shape[0]

    @property
    def cols(self) -> int:
        return self.data.shape[1]


class Geom:
    """Clip geometry of the token matrix: rows = B*T*H*W in (b, t, h, w) order."""

    __slots__ = ("B", "T", "H", "W")

    def __init__(self, B, T, H, W):
        self.B, self.T, self.H, self.W = B, T, H, W

    @property
    def HW(self):
        return self.H * self.W

    @property
    def M(self):
        return self.B * self.T * self.H * self.W

    def down(self):
        return Geom(self.B, self.T, self.H // 2, self.W // 2)

    def up(self):
        return Geom(self.B, self.T, self.H * 2, self.W * 2)


CONV3x3_TAPS = tuple((kw - 1, kh - 1, 0) for kh in range(3) for kw in range(3))


def _neg_taps(taps):
    return tuple((-a, -b, -c) for a, b, c in taps)


class WeightCache:
    """bf16 operand layouts of the (fp32 or bf16) master parameters.

    kinds: 'lin' [N,K]; 'linT' [K,N]; 'conv' [O,taps,Ipad]; 'convT' [I,taps,O];
           'cat:<kind>' for fused projections (q|k|v); 'f32' fp32 copy of a bf16 vector.
    Entries are refreshed when the source parameter's version counter changes (optimizer step,
    load_state_dict), or unconditionally for trainable parameters when ``refresh_trainable`` is
    called (CUDA-graph capture of a full train step re-prepares them inside the graph)."""

    def __init__(self):
        self._store: Dict[Tuple, Tuple[torch.Tensor, Tuple, Callable[[], None], bool]] = {}

    @staticmethod
    def _ver(params):
        return tuple((p._version, p.data_ptr()) for p in params)

    def get(self, key, params: Sequence[torch.Tensor], shape, build: Callable[[torch.Tensor], None], dtype=bf16):
        ent = self._store.get(key)
        ver = self._ver(params)
        if ent is None or ent[0].shape != torch.Size(shape) or ent[0].device != params[0].device:
            buf = torch.empty(shape, device=params[0].device, dtype=dtype)
            fn = lambda buf=buf: build(buf)
            fn()
            self._store[key] = (buf, ver, fn, any(p.requires_grad for p in params))
            return buf
        if ent[1] != ver:
            ent[2]()
            self._store[key] = (ent[0], ver, ent[2], ent[3])
        return ent[0]

    def refresh_trainable(self):
        for key, (buf, ver, fn, trainable) in list(self._store.items()):
            if trainable:
                fn()

    def clear(self):
        self._store.clear()


class Engine:
    """Per-model execution state: weight cache, tape, parameter-gradient arena."""

    def __init__(self):
        self.wc = WeightCache()
        self.tape: List[Callable[[], None]] = []
        self.recording = False
        self.pgrads: Dict[torch.nn.Parameter, torch.Tensor] = {}
        self.launches = 0
        self.grad_views: Dict[torch.nn.Parameter, torch.Tensor] = {}   # optional flat gradient arena (train.ParamArena)
        self.arena = None   # train.ParamArena: bf16 shadow + batched transposes of the trainable linear weights
        self.keep: List[torch.Tensor] = []   # small device scalars referenced by in-flight launches
        self._consts: Dict[Tuple, torch.Tensor] = {}
        self.grad_ready_hook: Optional[Callable[[List[torch.nn.Parameter]], None]] = None
        # zeroed fp32 scratch for every fused-statistics / GroupNorm-backward accumulator of a step: ONE memset per
        # forward instead of one per GroupNorm (the buffers are consumed before the next forward zeroes them again)
        self._stat_arena: Optional[torch.Tensor] = None
        self._stat_ptr = 0
        self.fuse_gn_stats = True
        self.fuse_gn_bwd = os.environ.get("SVDX_GN_BWD_FUSE", "1") != "0"

    # ------------------------------------------------------------------ tape
    def begin(self, recording: bool):
        """start a forward: a fresh tape (the previous forward's tape, if any, stays with ITS autograd node — see
        `detach_tape`), so two forwards before a backward, or a no_grad forward in between, cannot clobber each other"""
        self.tape = []
        self.recording = recording
        if self._stat_arena is not None:
            self._stat_arena.zero_()
        self._stat_ptr = 0

    STAT_ARENA_FLOATS = 8 << 20      # 32 MB

    def stat_zeros(self, n: int, device) -> torch.Tensor:
        """n zeroed floats: a slice of the per-step arena (zeroed once at `begin`), or a fresh tensor when it is exhausted"""
        n_al = (n + 63) // 64 * 64
        if self._stat_arena is None or self._stat_arena.device != torch.device(device):
            self._stat_arena = torch.zeros(self.STAT_ARENA_FLOATS, device=device, dtype=F32)
            self._stat_ptr = 0
        if self._stat_ptr + n_al > self._stat_arena.numel():
            return torch.zeros(n, device=device, dtype=F32)
        t = self._stat_arena[self._stat_ptr:self._stat_ptr + n]
        self._stat_ptr += n_al
        return t

    def _gn_sink(self, gn_rows: Optional[int], M: int, N: int, K: int, ntaps: int, device, n_out: Optional[int] = None):
        """channel-sum buffer for the fused GroupNorm statistics of a GEMM / conv output, or None when the launch cannot
        carry them (split-K path, ragged widths) — the consumer then runs the stand-alone statistics kernel"""
        if gn_rows is None or not self.fuse_gn_stats or N % 32 or M % gn_rows:
            return None
        if raw.split_plan(True, M, N, K, ntaps) is not None:
            return None
        return self.stat_zeros((M // gn_rows) * 2 * N, device).view(M // gn_rows, 2, N)

    def _gnb_for(self, x: Var, M: int, N: int, K: int, ntaps: int, scales, device):
        """tapgemm(gnb=...) arguments when x is a GroupNorm output and the data-gradient launch about to run is the first
        writer of its gradient: the epilogue then also accumulates pass 1 of the GroupNorm backward (per-channel sums), and
        the GroupNorm's backward is ONE launch with one pass over x and dy. None when the launch cannot carry them."""
        ctx = x.gnb
        if ctx is None or not self.fuse_gn_bwd or scales is not None or x.grad is not None or N % 32 or M % ctx["rows"] or N != ctx["C"] or M <= 8:
            return None
        if raw.split_plan(True, M, N, K, ntaps) is not None:
            return None
        sums = self.stat_zeros((M // ctx["rows"]) * 2 * N, device).view(M // ctx["rows"], 2, N)
        return dict(x=ctx["x"], x2=ctx["x2"], ab=ctx["ab"], rows=ctx["rows"], silu=ctx["silu"], sum=sums)

    def detach_tape(self) -> List[Callable[[], None]]:
        """hand the recorded tape to the caller (the autograd node of this forward) and stop recording"""
        tape, self.tape = self.tape, []
        self.recording = False
        return tape

    def record(self, fn: Callable[[], None]):
        if self.recording:
            self.tape.append(fn)

    def run_backward(self, tape: Optional[List[Callable[[], None]]] = None):
        """replay a tape in reverse. Closures may record onto self.tape (gradient checkpointing re-runs forward pieces),
        so recording is on while the tape runs; parameter gradients of THIS backward collect in self.pgrads."""
        if tape is None:
            tape, self.tape = self.tape, []
        self.pgrads = {}
        was, self.recording = self.recording, True
        try:
            while tape:
                tape.pop()()
        finally:
            self.recording = was
        self.keep.clear()

    def checkpoint(self, fn: Callable[..., Var], *inputs: Var) -> Var:
        """Gradient checkpointing on the tape (the contract of src/unet_spatio_temporal_condition.py:323-325 and
        torch.utils.checkpoint in the diffusers blocks): run `fn` without recording, and re-run it with recording
        inside the backward to rebuild the saved activations just before they are consumed."""
        if not self.recording:
            return fn(*inputs)
        self.recording = False
        try:
            out = fn(*inputs)
        finally:
            self.recording = True
        if not out.needs_grad:
            return out

        def bwd():
            dy = out.take_grad()
            if dy is None:
                return
            outer, self.tape = self.tape, []
            ins2 = [Var(v.data, v.needs_grad) for v in inputs]
            out2 = fn(*ins2)
            self.add_grad(out2, dy, owned=False)
            sub, self.tape = self.tape, outer
            while sub:
                sub.pop()()
            for v, v2 in zip(inputs, ins2):
                g = v2.take_grad()
                if g is not None:
                    self.add_grad(v, g)
        self.record(bwd)
        return out

    def add_grad(self, v: Var, g: torch.Tensor, owned: bool = True):
        """Accumulate gradient g into v. `owned`: g is a fresh tensor nobody else references (it may be
        kept and later overwritten in place); pass owned=False when g aliases another Var's gradient."""
        if not v.needs_grad:
            return
        v.gnb_sums = None        # sums fused into an earlier producer of this gradient no longer describe it
        if v.grad is None:
            v.grad, v.owned = g, owned
        elif v.grad.dtype != bf16:
            v.grad = v.grad + g
            v.owned = True
        elif v.owned:
            raw.axpby(v.grad, g, v.grad)
        else:
            out = torch.empty_like(v.grad)
            raw.axpby(v.grad, g, out)
            v.grad, v.owned = out, True

    def pgrad(self, p: torch.nn.Parameter) -> torch.Tensor:
        """fp32 accumulation buffer for the gradient of p (zero-initialised once per backward)."""
        g = self.pgrads.get(p)
        if g is None:
            g = self.grad_views.get(p)
            if g is None:
                g = torch.zeros(p.shape, device=p.device, dtype=F32)
            self.pgrads[p] = g
        return g

    # ------------------------------------------------------------------ operand preparation
    def w_lin(self, p: torch.Tensor, transposed: bool) -> torch.Tensor:
        if self.arena is not None and p.dim() == 2:
            m = self.arena.transposed_matrix([p]) if transposed else self.arena.shadow_matrix([p])
            if m is not None:
                return m
        O, I = p.shape[0], p[0].numel()
        src = lambda: p.detach().reshape(O, I)      # re-read at build time: p.data may have been re-homed
        if transposed:
            return self.wc.get(("linT", id(p)), [p], (I, O), lambda buf: raw.prep_weight(src(), buf, 1, O, I))
        return self.wc.get(("lin", id(p)), [p], (O, I), lambda buf: raw.prep_weight(src(), buf, 0, O, I))

    def w_lin_cat(self, ps: Sequence[torch.Tensor], transposed: bool) -> torch.Tensor:
        """concatenated projection weights [sum O_i, I] (fused q|k|v)."""
        if self.arena is not None:
            m = self.arena.transposed_matrix(list(ps)) if transposed else self.arena.shadow_matrix(list(ps))
            if m is not None:
                return m
        I = ps[0].shape[1]
        Os = [p.shape[0] for p in ps]
        key = ("catT" if transposed else "cat",) + tuple(id(p) for p in ps)
        if transposed:
            def build(buf):
                tmp = torch.empty(sum(Os), I, device=buf.device, dtype=bf16)
                o0 = 0
                for p, O in zip(ps, Os):
                    raw.prep_weight(p.detach(), tmp[o0:o0 + O], 0, O, I)
                    o0 += O
                raw.prep_weight(tmp, buf, 1, sum(Os), I)
            return self.wc.get(key, list(ps), (I, sum(Os)), build)

        def build(buf):
            o0 = 0
            for p, O in zip(ps, Os):
                raw.prep_weight(p.detach(), buf[o0:o0 + O], 0, O, I)
                o0 += O
        return self.wc.get(key, list(ps), (sum(Os), I), build)

    def w_conv(self, p: torch.Tensor, transposed: bool, i_pad: Optional[int] = None) -> torch.Tensor:
        O, I = p.shape[0], p.shape[1]
        taps = p[0, 0].numel()
        if transposed:
            Op = (O + 7) // 8 * 8
            if Op != O:  # conv_out (O = 4): zero-pad the output-channel axis so rows stay 16-byte aligned
                def build(buf):
                    w = p.detach()
                    wp = torch.zeros(Op, I, taps, device=w.device, dtype=w.dtype)
                    wp[:O] = w.reshape(O, I, taps)
                    raw.prep_weight(wp, buf, 3, Op, I, taps)
                return self.wc.get(("convT", id(p)), [p], (I, taps * Op), build)
            return self.wc.get(("convT", id(p)), [p], (I, taps * O), lambda buf: raw.prep_weight(p.detach(), buf, 3, O, I, taps))
        ip = i_pad if i_pad is not None else I
        return self.wc.get(("conv", id(p), ip), [p], (O, taps * ip), lambda buf: raw.prep_weight(p.detach(), buf, 2, O, I, taps, ip))

    def vec_f32(self, p: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        if p is None:
            return None
        if p.dtype == F32:
            return p.detach()
        return self.wc.get(("f32", id(p)), [p], tuple(p.shape), lambda buf: raw.cast_to_f32(p.detach().contiguous(), buf), dtype=F32)

    # ------------------------------------------------------------------ small helpers
    @staticmethod
    def empty(rows, cols, like: torch.Tensor, dtype=bf16):
        return torch.empty(rows, cols, device=like.device, dtype=dtype)

    def _bias_grad(self, bias_p, dy: torch.Tensor, scale: Optional[torch.Tensor] = None):
        """bias gradient = column sums of dy (dy may carry zero-padded extra columns, e.g. conv_out's 4 -> 8)."""
        if bias_p is None or not bias_p.requires_grad:
            return
        g = self.pgrad(bias_p)
        n = g.numel()
        if scale is None and dy.shape[1] == n:
            raw.colsum(dy, g, accumulate=True)
        else:
            tmp = torch.empty(dy.shape[1], device=dy.device, dtype=F32)
            raw.colsum(dy, tmp)
            g.add_(tmp[:n] if scale is None else tmp[:n] * scale)

    # ------------------------------------------------------------------ linear family
    def _res_grad(self, r: Optional[Var], dy: torch.Tensor, scale: Optional[torch.Tensor]):
        """gradient of a residual epilogue operand: scale * dy (scale None = 1: dy is passed on by alias)."""
        if r is None or not r.needs_grad:
            return
        if scale is None:
            self.add_grad(r, dy, owned=False)
        else:
            self.add_grad(r, self._scaled(dy, scale))

    def _rowbias_grad(self, rb: Optional[Var], dy: torch.Tensor, div: int, scale: Optional[torch.Tensor]):
        """rowbias[b] is added to rows [b*div, (b+1)*div): its gradient is the per-block column sum of dy."""
        if rb is None or not rb.needs_grad:
            return
        nb = rb.rows
        g = torch.empty(nb, dy.shape[1], device=dy.device, dtype=F32)
        for b in range(nb):
            raw.colsum(dy[b * div:(b + 1) * div], g[b])
        if scale is not None:
            g = g * scale
        self.add_grad(rb, g)

    def linear(self, x: Var, weight, bias=None, *, res1: Optional[Var] = None, res2: Optional[Var] = None,
               scales: Optional[torch.Tensor] = None, res1_unit: bool = False, geglu: bool = False,
               rowbias: Optional[Var] = None, rowbias_div: int = 1, out_f32: bool = False,
               fused: Optional[Sequence] = None, blend=None, lora: Optional[Sequence] = None, gn_rows: Optional[int] = None,
               act: int = raw.ACT_NONE) -> Var:
        """y = epilogue(x @ W^T). `weight` is a parameter [N,K] (or conv 1x1 [N,K,1,1]); `fused` = list of
        parameters whose rows are concatenated (q|k|v). scales (device float[>=3]) = {acc, res1, res2};
        res1_unit: scales[1] is known to be exactly 1. rowbias: Var with fp32 data [ceil(M/div), N].
        act (raw.ACT_GELU): activation of acc + bias before the residual step; forward-only (no backward is recorded)."""
        ws = list(fused) if fused is not None else [weight]
        wf = self.w_lin_cat(ws, False) if fused is not None else self.w_lin(weight, False)
        N, K = wf.shape
        M = x.rows
        n_out = N // 2 if geglu else N
        out = self.empty(M, n_out, x.data, F32 if out_f32 else bf16)
        pre = self.empty(M, N, x.data) if (geglu and self.recording) else None
        b32 = self.vec_f32(bias)
        lora = [l for l in (lora or []) if l is not None]
        if act and (geglu or out_f32 or lora):
            raise ValueError("Engine.linear: act needs a plain bf16 linear (no GEGLU, fp32 output or LoRA)")
        sink = None if (geglu or out_f32 or lora or act) else self._gn_sink(gn_rows, M, N, K, 1, out.device)
        raw.tapgemm_auto(x.data, wf, out, M=M, N=N, K=K, bias=b32, res1=None if res1 is None else res1.data,
                         res2=None if res2 is None else res2.data, scales=scales, geglu=geglu, pre=pre,
                         rowbias=None if rowbias is None else rowbias.data, rowbias_div=rowbias_div, gn_sum=sink, gn_rows=gn_rows or 0,
                         act=act)
        lora_t = []
        for (off, n, A, Bm, sc) in lora:
            # LoRA side path (train_svd_lora.py:659-671): out[:, off:off+n] += scale * (x A^T) B^T, accumulated in place.
            # The rank axis is padded to a multiple of 8 in the OPERAND copies (16-byte rows for TMA); parameter and
            # gradient shapes stay [r, in] / [out, r] (the reference default is --rank 4, train_svd_lora.py:551-553).
            rp = (A.shape[0] + 7) // 8 * 8
            t = self.empty(M, rp, x.data)
            ov = out[:, off:off + n]
            if M <= 8:      # the [B, C] cross-attention vectors: skinny products, not 128-row tiles
                raw.gemv(x.data, self.w_lora(A, "A", False), t, M=M, N=rp, K=K)
                raw.gemv(t, self.w_lora(Bm, "B", False), ov, M=M, N=n, K=rp, scale=sc, accumulate=True)
            else:
                raw.tapgemm(x.data, self.w_lora(A, "A", False), t, M=M, N=rp, K=K)
                raw.tapgemm(t, self.w_lora(Bm, "B", False), ov, M=M, N=n, K=rp, res1=ov, scales=self._lora_scales(sc, out.device))
            lora_t.append(t)
        w_train = any(p.requires_grad for p in ws) or (bias is not None and bias.requires_grad) \
            or (blend is not None and blend[0].requires_grad) or any(l[2].requires_grad or l[3].requires_grad for l in lora)
        need = x.needs_grad or w_train or any(v is not None and v.needs_grad for v in (res1, res2, rowbias))
        if act and need and self.recording:
            raise RuntimeError("Engine.linear: the activation epilogue is forward-only; it cannot record a backward")
        y = Var(out, need)
        if sink is not None:
            y.csum = (gn_rows, [(sink, N)])
        if need and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                if dy.dtype != bf16:
                    dy = raw.cast_f32_bf16(dy.contiguous(), torch.empty(dy.shape, device=dy.device, dtype=bf16))
                s_acc = None if scales is None else scales[0:1]
                self._mix_grad(blend, dy, res1, out)
                self._res_grad(res1, dy, None if (scales is None or res1_unit) else scales[1:2])
                self._res_grad(res2, dy, None if scales is None else scales[2:3])
                bias_done = False
                if geglu:
                    # the projection's bias gradient (column sums of dpre) rides in the same pass
                    fuse_b = bias is not None and bias.requires_grad and scales is None and self.pgrad(bias).numel() == pre.shape[1]
                    dyl = raw.geglu_bwd(pre, dy, torch.empty_like(pre), bias_grad=self.pgrad(bias) if fuse_b else None)
                    bias_done = fuse_b
                else:
                    dyl = dy
                self._rowbias_grad(rowbias, dyl, rowbias_div, s_acc)
                sc3 = self._acc_only(s_acc)
                if x.needs_grad:
                    wt = self.w_lin_cat(ws, True) if fused is not None else self.w_lin(weight, True)
                    dx = self.empty(M, K, x.data)
                    # x a GroupNorm output (the transformers' proj_in): pass 1 of its backward rides in this epilogue
                    gnb = None if lora else self._gnb_for(x, M, K, N, 1, sc3, dyl.device)
                    raw.tapgemm_auto(dyl, wt, dx, M=M, N=K, K=N, scales=sc3, **({} if gnb is None else {"gnb": gnb}))
                    self.add_grad(x, dx)
                    if gnb is not None:
                        x.gnb_sums = (gnb["sum"], dx)
                if any(p.requires_grad for p in ws):
                    self._wgrad(dyl, x.data, ws, N, K, M, sc3)
                if bias is not None and bias.requires_grad and not bias_done:
                    self._bias_grad(bias, dyl, s_acc)
                for (off, n, A, Bm, sc), t in zip(lora, lora_t):
                    r = A.shape[0]
                    rp = (r + 7) // 8 * 8
                    dys = dyl[:, off:off + n]
                    s3 = self._lora_scales(sc, dyl.device, acc_only=True)
                    dt = self.empty(M, rp, x.data)
                    if M <= 8:
                        raw.gemv(dys, self.w_lora(Bm, "B", True), dt, M=M, N=rp, K=n, scale=sc)       # dt = scale * dy B
                    else:
                        raw.tapgemm(dys, self.w_lora(Bm, "B", True), dt, M=M, N=rp, K=n, scales=s3)   # dt = scale * dy B
                    if Bm.requires_grad:
                        self._wgrad(dys, t, [Bm], n, rp, M, s3, pad_to=(n, rp))                  # dB += scale * dy^T t
                    if A.requires_grad:
                        self._wgrad(dt, x.data, [A], rp, K, M, None, pad_to=(rp, K))             # dA += dt^T x
                    if x.needs_grad:
                        dxl = self.empty(M, K, x.data)
                        if M <= 8:
                            raw.gemv(dt, self.w_lora(A, "A", True), dxl, M=M, N=K, K=rp)
                        else:
                            raw.tapgemm(dt, self.w_lora(A, "A", True), dxl, M=M, N=K, K=rp)
                        self.add_grad(x, dxl)
            self.record(bwd)
        return y

    def _lora_scales(self, scale: float, device, acc_only: bool = False) -> torch.Tensor:
        key = ("lora_scale", float(scale), acc_only, str(device))
        t = self._consts.get(key)
        if t is None:
            t = torch.tensor([float(scale), 0.0 if acc_only else 1.0, 0.0], device=device, dtype=F32)
            self._consts[key] = t
        return t

    @staticmethod
    def _blend_base(view: torch.Tensor):
        """(16-float svdx_blend_scales buffer, element offset of `view` in it) when `view` is a slice of one, else (None, 0)"""
        base = view._base
        if base is not None and base.numel() == 16 and base.dtype == F32:
            return base, (view.data_ptr() - base.data_ptr()) // 4
        return None, 0

    def _acc_only(self, s3):
        """scales triple {s_acc, 0, 0} for gradient GEMMs of a scaled forward (precomputed by svdx_blend_scales)."""
        if s3 is None:
            return None
        base, _ = self._blend_base(s3)
        if base is not None:
            return base[8:11]
        t = torch.zeros(3, device=s3.device, dtype=F32)
        t[0:1].copy_(s3[0:1])
        self.keep.append(t)
        return t

    def _scaled(self, t: torch.Tensor, s: torch.Tensor) -> torch.Tensor:
        """fresh tensor s*t (s: device scalar tensor [1])."""
        out = torch.empty_like(t)
        base, off = self._blend_base(s)
        if base is not None and off in (1, 2):          # alpha / (1 - alpha) of the transformer blend
            sc = base[12:14] if off == 1 else base[14:16]
        else:
            sc = torch.zeros(2, device=t.device, dtype=F32)
            sc[0:1].copy_(s)
            self.keep.append(sc)
        raw.axpby(t.reshape(-1), t.reshape(-1), out.reshape(-1), sc)
        return out

    def w_lora(self, p: torch.Tensor, which: str, transposed: bool) -> torch.Tensor:
        """bf16 operand of a LoRA factor with the rank axis zero-padded to a multiple of 8: A [r,in] -> [rp,in] (or its
        transpose [in,rp]); B [out,r] -> [out,rp] (or [rp,out]). rp == r: the plain (cached / arena) operand."""
        r = p.shape[0] if which == "A" else p.shape[1]
        rp = (r + 7) // 8 * 8
        if rp == r:
            return self.w_lin(p, transposed)
        O, I = p.shape
        Op, Ip = (rp, I) if which == "A" else (O, rp)
        shape = (Ip, Op) if transposed else (Op, Ip)

        def build(buf):
            buf.zero_()
            src = p.detach().t() if transposed else p.detach()
            buf[:src.shape[0], :src.shape[1]].copy_(src)
        return self.wc.get(("lora", id(p), transposed), [p], shape, build)

    def _wgrad(self, dy: torch.Tensor, x: torch.Tensor, ws, N, K, M, scales3, pad_to=None):
        """dW[N,K] += dy[M,N]^T @ x[M,K] — both operands MN-major, split-K over tokens, fp32 atomics.
        pad_to=(N, K): the operands carry zero-padded rank columns (LoRA, r % 8 != 0); the product is formed in a padded
        fp32 scratch and its valid block is added to the parameter gradient."""
        if pad_to is not None and tuple(pad_to) != tuple(ws[0].shape):
            p = ws[0]
            if not p.requires_grad:
                return
            tmp = torch.zeros(pad_to, device=dy.device, dtype=F32)
            bn = raw.choose_block_n(pad_to[0], pad_to[1], mn_major=True)
            raw.tapgemm(dy, x, tmp, M=pad_to[0], N=pad_to[1], K=M, a_mn=True, b_mn=True, split_k=1, out_dtype=OUT_F32_ATOMIC,
                        block_n=bn, lda=dy.stride(0), ldb=x.stride(0), scales=scales3)
            self.pgrad(p).add_(tmp[:p.shape[0], :p.shape[1]])
            return
        if M <= 8 and (pad_to is None or tuple(pad_to) == tuple(ws[0].shape)) and K % 4 == 0 and dy.shape[1] >= sum(p.shape[0] for p in ws):
            # conditioning vectors (B token rows): an outer-product accumulation, not a split-K tensor-core launch
            o0 = 0
            for p in ws:
                O = p.shape[0]
                if p.requires_grad:
                    raw.outer_accum(dy[:, o0:o0 + O], x, self.pgrad(p).view(O, -1), None if scales3 is None else scales3[0:1])
                o0 += O
            return
        fused_g = None
        if len(ws) > 1 and self.arena is not None and all(p.requires_grad for p in ws):
            fused_g = self.arena.grad_matrix(list(ws))     # q|k|v are adjacent in the arena: ONE [3C, C] weight-gradient GEMM
        if fused_g is not None:
            for p in ws:
                self.pgrads.setdefault(p, self.grad_views[p])
            targets = [(None, 0, N)]
        elif len(ws) == 1:
            targets = [(ws[0], 0, N)]
        else:
            targets, o0 = [], 0
            for p in ws:
                targets.append((p, o0, p.shape[0]))
                o0 += p.shape[0]
        for p, o0, O in targets:
            if p is not None and not p.requires_grad:
                continue
            g = fused_g if p is None else self.pgrad(p).view(O, -1)
            dyp = dy[:, o0:o0 + O]
            bn, split = raw.wgrad_plan(O, K, M)       # tile width and token split chosen together (L2 -> SM traffic model)
            raw.tapgemm(dyp, x, g, M=O, N=K, K=M, a_mn=True, b_mn=True, split_k=split, out_dtype=OUT_F32_ATOMIC,
                        block_n=bn, lda=dy.stride(0), ldb=x.stride(0), scales=scales3)

    # ------------------------------------------------------------------ convolutions
    def _conv_wgrad(self, dy: torch.Tensor, x: torch.Tensor, w: torch.nn.Parameter, taps, *, b_mode: int, Opad: int, ip: int,
                    K: int, conv_whn=None, rows_per_group=None, groups=1, scales3=None):
        """dW[o][tap][i] = sum_p dy[p, o] * x[p + tap, i]: one MN-major split-K launch per tap (fp32 atomics into a
        [O][taps][ip] workspace), then the adjoint of the weight re-layout accumulates into the OIHW gradient."""
        O, I = w.shape[0], w.shape[1]
        nt = len(taps)
        ws = torch.zeros(Opad, nt * ip, device=dy.device, dtype=F32)
        bn = raw.choose_block_n(Opad, ip, mn_major=True)
        tiles = ((Opad + 127) // 128) * ((ip + bn - 1) // bn)
        kb = (K + 63) // 64
        split = max(1, min(kb // 32, raw.num_sms() // max(tiles, 1)))
        for t, tap in enumerate(taps):
            raw.tapgemm(dy, x, ws[:, t * ip:(t + 1) * ip], M=Opad, N=ip, K=K, a_mn=True, b_mn=True, b_mode=b_mode, taps=(tap,),
                        conv_whn=conv_whn, rows_per_group=rows_per_group if rows_per_group is not None else K, groups=groups,
                        split_k=split, out_dtype=OUT_F32_ATOMIC, block_n=bn, lda=dy.stride(0), ldb=x.stride(0), ldo=nt * ip,
                        scales=scales3)
        raw.unprep_conv_grad(ws, self.pgrad(w).view(O, I, nt), O, I, nt, ip)

    def _mix_grad(self, blend, dy: torch.Tensor, res1: Var, out: torch.Tensor):
        """AlphaBlender.mix_factor gradient: d mix = alpha * sum(dy * (x_spatial - out))  (see DESIGN.md)."""
        if blend is None or not blend[0].requires_grad:
            return
        mix, alpha = blend
        acc = torch.zeros(1, device=dy.device, dtype=F32)
        raw.dot_diff(dy.reshape(-1), res1.data.reshape(-1), out.reshape(-1), acc)
        self.pgrad(mix).add_((acc * alpha).to(F32).view(mix.shape))

    def conv2d_3x3(self, x: Var, g: Geom, conv, *, rowbias: Optional[Var] = None, rowbias_div=1, res1: Optional[Var] = None,
                   scales=None, res1_unit: bool = False, i_pad=None, n_pad=None, planes: bool = False, gn_rows: Optional[int] = None,
                   planes_pad0: bool = False) -> Var:
        """3x3 conv, padding 1, on channels-last [N*H*W, Cin]. planes=True: x holds the 4 stride-2 parity planes
        of a [N,2H,2W] image and the result is the stride-2 conv at geometry g (= output geometry): padding 1 on all sides
        (the UNet's Downsample2D), or with planes_pad0 the VAE encoder's form, F.pad(x, (0,1,0,1)) + conv(stride 2, padding 0)."""
        w = conv.weight
        O, I = w.shape[0], w.shape[1]
        ip = i_pad if i_pad is not None else I
        wf = self.w_conv(w, False, ip)
        nimg = g.B * g.T
        M = nimg * g.H * g.W
        n_alloc = n_pad if n_pad is not None else O
        out = self.empty(M, n_alloc, x.data)
        if planes:
            taps = []
            # input row 2h + kh - pad = parity plane (kh - pad) & 1 at row h + (kh - pad) // 2 — out-of-image rows read as zero
            table = ((0, 0), (1, 0), (0, 1)) if planes_pad0 else ((1, -1), (0, 0), (1, 0))
            for kh in range(3):
                for kw in range(3):
                    ph, dh = table[kh]
                    pw, dw = table[kw]
                    taps.append((dw, dh, (ph * 2 + pw) * nimg))
            taps = tuple(taps)
            whn = (g.W, g.H, 4 * nimg)
        else:
            taps = CONV3x3_TAPS
            whn = (g.W, g.H, nimg)
        sink = None if (n_alloc != O or O < 32) else self._gn_sink(gn_rows, M, O, ip, len(taps), out.device)
        raw.tapgemm_auto(x.data, wf, out, M=M, N=O, K=ip, mode=A_CONV2D, taps=taps, conv_whn=whn, bias=self.vec_f32(conv.bias),
                         rowbias=None if rowbias is None else rowbias.data, rowbias_div=rowbias_div,
                         res1=None if res1 is None else res1.data, scales=scales,
                         block_n=None if O >= 32 else 32, gn_sum=sink, gn_rows=gn_rows or 0)
        w_train = w.requires_grad or (conv.bias is not None and conv.bias.requires_grad)
        need = x.needs_grad or w_train or any(v is not None and v.needs_grad for v in (res1, rowbias))
        y = Var(out, need)
        if sink is not None:
            y.csum = (gn_rows, [(sink, O)])
        if need and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                s_acc = None if scales is None else scales[0:1]
                self._res_grad(res1, dy, None if (scales is None or res1_unit) else scales[1:2])
                if conv.bias is not None and conv.bias.requires_grad:
                    self._bias_grad(conv.bias, dy, s_acc)
                self._rowbias_grad(rowbias, dy, rowbias_div, s_acc)
                sc = self._acc_only(s_acc)
                if w.requires_grad:
                    self._conv_wgrad(dy, x.data, w, taps, b_mode=1, Opad=dy.shape[1], ip=ip, K=M, conv_whn=whn, scales3=sc)
                if x.needs_grad:
                    wt = self.w_conv(w, True)  # [I, 9*Opad]
                    Op = wt.shape[1] // 9
                    gnb = None
                    if not planes:
                        dx = self.empty(M, I, x.data)
                        gnb = self._gnb_for(x, M, I, Op, 9, sc, dy.device)
                        raw.tapgemm_auto(dy, wt, dx, M=M, N=I, K=Op, mode=A_CONV2D, taps=_neg_taps(CONV3x3_TAPS),
                                         conv_whn=(g.W, g.H, nimg), scales=sc, **({} if gnb is None else {"gnb": gnb}))
                    else:
                        # gradient w.r.t. each parity plane: the taps that read that plane, shifts negated
                        dx = self.empty(4 * M, I, x.data)
                        wt3 = wt.view(I, 9, O)
                        for pl in range(4):
                            sel = [t for t in range(9) if taps[t][2] == pl * nimg]
                            wsub = self.wc.get(("convT_plane", id(w), pl), [w], (I, len(sel) * O),
                                               lambda buf, sel=sel: buf.view(I, len(sel), O).copy_(wt3[:, sel, :]))
                            tp = tuple((-taps[t][0], -taps[t][1], 0) for t in sel)
                            raw.tapgemm(dy, wsub, dx[pl * M:(pl + 1) * M], M=M, N=I, K=O, mode=A_CONV2D, taps=tp,
                                        conv_whn=(g.W, g.H, nimg), scales=sc)
                    self.add_grad(x, dx)
                    if gnb is not None:
                        x.gnb_sums = (gnb["sum"], dx)
            self.record(bwd)
        return y

    def conv_temporal(self, x: Var, g: Geom, conv, *, rowbias: Optional[Var] = None, rowbias_div=1, res1: Optional[Var] = None,
                      scales=None, res1_unit: bool = False, blend=None, gn_rows: Optional[int] = None) -> Var:
        """Conv3d kernel (3,1,1), padding (1,0,0): frames are HW rows apart in the token matrix.
        blend = (mix_factor parameter, device alpha[1]) when this conv carries the AlphaBlender epilogue."""
        w = conv.weight
        O, I = w.shape[0], w.shape[1]
        wf = self.w_conv(w, False)
        M = g.M
        HW = g.HW
        taps = ((-HW, 0, 0), (0, 0, 0), (HW, 0, 0))
        out = self.empty(M, O, x.data)
        sink = self._gn_sink(gn_rows, M, O, I, 3, out.device)
        raw.tapgemm_auto(x.data, wf, out, M=M, N=O, K=I, taps=taps, rows_per_group=g.T * HW, groups=g.B, bias=self.vec_f32(conv.bias),
                         rowbias=None if rowbias is None else rowbias.data, rowbias_div=rowbias_div,
                         res1=None if res1 is None else res1.data, scales=scales, gn_sum=sink, gn_rows=gn_rows or 0)
        w_train = w.requires_grad or (conv.bias is not None and conv.bias.requires_grad) or (blend is not None and blend[0].requires_grad)
        need = x.needs_grad or w_train or any(v is not None and v.needs_grad for v in (res1, rowbias))
        y = Var(out, need)
        if sink is not None:
            y.csum = (gn_rows, [(sink, O)])
        if need and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                s_acc = None if scales is None else scales[0:1]
                self._mix_grad(blend, dy, res1, out)
                self._res_grad(res1, dy, None if (scales is None or res1_unit) else scales[1:2])
                if conv.bias is not None and conv.bias.requires_grad:
                    self._bias_grad(conv.bias, dy, s_acc)
                self._rowbias_grad(rowbias, dy, rowbias_div, s_acc)
                sc = self._acc_only(s_acc)
                if w.requires_grad:
                    self._conv_wgrad(dy, x.data, w, taps, b_mode=2, Opad=O, ip=I, K=M, rows_per_group=g.T * HW, groups=g.B, scales3=sc)
                if x.needs_grad:
                    wt = self.w_conv(w, True)
                    dx = self.empty(M, I, x.data)
                    gnb = self._gnb_for(x, M, I, O, 3, sc, dy.device)
                    raw.tapgemm_auto(dy, wt, dx, M=M, N=I, K=O, taps=_neg_taps(taps), rows_per_group=g.T * HW, groups=g.B, scales=sc,
                                     **({} if gnb is None else {"gnb": gnb}))
                    self.add_grad(x, dx)
                    if gnb is not None:
                        x.gnb_sums = (gnb["sum"], dx)
            self.record(bwd)
        return y

    # ------------------------------------------------------------------ small fp32 ops of the embedding MLPs
    def silu_cast(self, x: Var) -> Var:
        """bf16(silu(x)) for an fp32 Var (TimestepEmbedding.act / nonlinearity(temb) feeding a GEMM)."""
        h = raw.silu_f32(x.data, torch.empty_like(x.data))
        y = Var(raw.cast_f32_bf16(h, torch.empty(h.shape, device=h.device, dtype=bf16)), x.needs_grad)
        if x.needs_grad and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                d32 = raw.cast_bf16_f32(dy.contiguous(), torch.empty(dy.shape, device=dy.device, dtype=F32)) if dy.dtype == bf16 else dy
                self.add_grad(x, raw.silu_bwd_f32(x.data, d32.contiguous(), torch.empty_like(x.data)))
            self.record(bwd)
        return y

    def cast_to_f32(self, x: Var) -> Var:
        y = Var(raw.cast_bf16_f32(x.data.contiguous(), torch.empty(x.data.shape, device=x.data.device, dtype=F32)), x.needs_grad)
        if x.needs_grad and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                self.add_grad(x, raw.cast_f32_bf16(dy.contiguous(), torch.empty(dy.shape, device=dy.device, dtype=bf16)))
            self.record(bwd)
        return y

    def add_f32(self, a: Var, b: Var) -> Var:
        y = Var(a.data + b.data, a.needs_grad or b.needs_grad)
        if y.needs_grad and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                self.add_grad(a, dy, owned=False)
                self.add_grad(b, dy, owned=False)
            self.record(bwd)
        return y

    # ------------------------------------------------------------------ normalisation
    def groupnorm(self, x: Var, gn, outer: int, rows: int, silu: bool) -> Var:
        """GroupNorm(32) (+SiLU); one statistics group spans `rows` rows (H*W per frame, or T*H*W per clip).
        When the producer(s) of x accumulated per-channel sums in their epilogues (x.csum, slab = `rows` rows), the group
        statistics are folded from them inside the apply kernel: ONE launch, no pass over x for the statistics."""
        C = x.cols
        gamma, beta = self.vec_f32(gn.weight), self.vec_f32(gn.bias)
        out = self.empty(x.rows, C, x.data)
        cs = x.csum
        p_train = gn.weight.requires_grad
        need = x.needs_grad or p_train
        # per-channel scale / shift table for the backward sums fused into the consumer's dgrad epilogue (see _gnb_for)
        ab = torch.empty(outer, 2, C, device=out.device, dtype=F32) if (need and self.recording and self.fuse_gn_bwd) else None
        if cs is not None and cs[0] == rows and len(cs[1]) <= 2 and sum(c for _, c in cs[1]) == C and all(t.shape[0] == outer for t, _ in cs[1]):
            parts = cs[1]
            C1 = parts[0][1]
            x1 = x.data if len(parts) == 1 else x.data[:, :C1]
            x2 = None if len(parts) == 1 else x.data[:, C1:]
            mean, rstd = raw.groupnorm_apply_fused(x1, x2, outer, rows, gn.eps, parts[0][0], None if len(parts) == 1 else parts[1][0],
                                                   gamma, beta, silu, out, gn.num_groups, ab=ab)
        else:
            mean, rstd = raw.groupnorm_stats(x.data, None, outer, rows, gn.eps, gn.num_groups)
            raw.groupnorm_apply(x.data, None, outer, rows, mean, rstd, gamma, beta, silu, out, gn.num_groups, ab=ab)
        y = Var(out, need)
        if ab is not None:
            y.gnb = dict(x=x.data, x2=None, ab=ab, rows=rows, silu=silu, C=C)   # x.data is the (already concatenated) [M, C] tensor
        if need and self.recording:
            def bwd():
                fused = y.gnb_sums
                dy = y.take_grad()
                y.gnb_sums = None
                if dy is None:
                    return
                dx = self.empty(x.rows, C, x.data)
                dg = self.pgrad(gn.weight) if p_train else None
                db = self.pgrad(gn.bias) if p_train else None
                # x usually already carries the gradient of its residual use (conv2 / proj_out `res1`): folded into this pass
                dres = x.grad if (x.needs_grad and x.grad is not None and x.grad.dtype == bf16 and x.grad.shape == dx.shape
                                  and x.grad.stride(-1) == 1) else None
                if fused is not None and fused[1] is dy:
                    # pass 1 ran inside the dgrad epilogue that wrote dy: one launch, one pass over x and dy
                    raw.groupnorm_bwd_fused(x.data, None, dy, outer, rows, mean, rstd, gamma, beta, silu, fused[0], dx, None, dg, db,
                                            gn.num_groups, dres=dres)
                else:
                    ws = self.stat_zeros(2 * outer * gn.num_groups, dy.device)
                    raw.groupnorm_bwd(x.data, None, dy, outer, rows, mean, rstd, gamma, beta, silu, dx, None, dg, db, gn.num_groups, ws=ws, dres=dres)
                if dres is not None:
                    x.grad, x.owned = dx, True
                else:
                    self.add_grad(x, dx)
            self.record(bwd)
        return y

    def layernorm(self, x: Var, ln, *, addvec: Optional[torch.Tensor] = None, add_div: int = 1,
                  addvec_var: Optional[Var] = None) -> Tuple[Var, Var]:
        """returns (xs, LN(xs)) with xs = x + addvec[row / add_div] (xs is x itself when addvec is None).
        Backward folds the gradient already accumulated on xs (its residual uses) into dx."""
        C = x.cols
        gamma, beta = self.vec_f32(ln.weight), self.vec_f32(ln.bias)
        out = self.empty(x.rows, C, x.data)
        if addvec is not None:
            xs_data = self.empty(x.rows, C, x.data)
            mean, rstd = raw.layernorm_fwd(x.data, gamma, beta, ln.eps, out, addvec, add_div, xs_data)
        else:
            xs_data = x.data
            mean, rstd = raw.layernorm_fwd(x.data, gamma, beta, ln.eps, out)
        p_train = ln.weight.requires_grad
        need = x.needs_grad or p_train
        xs = x if addvec is None else Var(xs_data, x.needs_grad)
        y = Var(out, need)
        if need and self.recording:
            def bwd():
                dy = y.take_grad()
                dres = xs.grad
                if dy is None:
                    if addvec is not None and dres is not None:
                        self.add_grad(x, xs.take_grad(), owned=False)
                    return
                dg = self.pgrad(ln.weight) if p_train else None
                db = self.pgrad(ln.bias) if p_train else None
                if x.needs_grad:
                    dx = self.empty(x.rows, C, x.data)
                    raw.layernorm_bwd(xs_data, dy, gamma, mean, rstd, dx, dres, dg, db)
                    xs.take_grad()
                    if addvec is None:
                        x.grad, x.owned = dx, True   # dres (the old x.grad) is folded in
                    else:
                        self._rowbias_grad(addvec_var, dx, add_div, None)   # d(frame embedding) = per-frame sums of d(x + emb)
                        self.add_grad(x, dx)
                elif p_train:
                    dx = self.empty(x.rows, C, x.data)  # still needed to produce dgamma/dbeta
                    raw.layernorm_bwd(xs_data, dy, gamma, mean, rstd, dx, None, dg, db)
            self.record(bwd)
        return xs, y

    # ------------------------------------------------------------------ attention
    def attention(self, qkv: Var, heads: int, g: Geom, temporal: bool) -> Var:
        """self-attention over H*W per frame (spatial) or over T per pixel (temporal) on a fused q|k|v matrix."""
        C = heads * 64
        M = qkv.rows
        q, k, v = qkv.data[:, :C], qkv.data[:, C:2 * C], qkv.data[:, 2 * C:3 * C]
        out = self.empty(M, C, qkv.data)
        need = qkv.needs_grad
        lse = torch.empty(M, heads, device=out.device, dtype=F32) if (need and self.recording) else None
        if temporal:
            geo = dict(heads=heads, S=g.T, nseq=g.B * g.HW, inner=g.HW, outer_stride=g.T * g.HW, inner_stride=1, tok_stride=g.HW)
        else:
            geo = dict(heads=heads, S=g.HW, nseq=g.B * g.T, inner=1, outer_stride=g.HW, inner_stride=0, tok_stride=1)
        raw.attention_fwd(q, k, v, out, lse=lse, **geo)
        y = Var(out, need)
        if need and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                dqkv = self.empty(M, 3 * C, out)
                delta = torch.empty_like(lse)
                raw.attention_bwd(q, k, v, out, dy, dqkv[:, :C], dqkv[:, C:2 * C], dqkv[:, 2 * C:], lse, delta, **geo)
                self.add_grad(qkv, dqkv)
            self.record(bwd)
        return y

    # ------------------------------------------------------------------ layout ops
    def concat(self, a: Var, b: Var) -> Var:
        out = self.empty(a.rows, a.cols + b.cols, a.data)
        raw.concat_channels(a.data, b.data, out)
        need = a.needs_grad or b.needs_grad
        y = Var(out, need)
        if a.csum is not None and b.csum is not None and a.csum[0] == b.csum[0] and len(a.csum[1]) == 1 and len(b.csum[1]) == 1:
            y.csum = (a.csum[0], [a.csum[1][0], b.csum[1][0]])      # GroupNorm over the concatenation folds both producers' sums
        if need and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                da = torch.empty_like(a.data)
                db = torch.empty_like(b.data)
                raw.split_channels(dy, da, db)
                self.add_grad(a, da)
                self.add_grad(b, db)
            self.record(bwd)
        return y

    def upsample2x(self, x: Var, g: Geom) -> Var:
        N = g.B * g.T
        out = self.empty(4 * x.rows, x.cols, x.data)
        raw.upsample2x(x.data, out, N, g.H, g.W, x.cols)
        y = Var(out, x.needs_grad)
        if x.needs_grad and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                dx = torch.empty_like(x.data)
                raw.upsample2x_bwd(dy, dx, N, g.H, g.W, x.cols)
                self.add_grad(x, dx)
            self.record(bwd)
        return y

    def space_to_planes(self, x: Var, g: Geom) -> Var:
        N = g.B * g.T
        out = torch.empty_like(x.data)
        raw.space_to_planes(x.data, out, N, g.H, g.W, x.cols)
        y = Var(out, x.needs_grad)
        if x.needs_grad and self.recording:
            def bwd():
                dy = y.take_grad()
                if dy is None:
                    return
                dx = torch.empty_like(x.data)
                raw.planes_to_space(dy, dx, N, g.H, g.W, x.cols)
                self.add_grad(x, dx)
            self.record(bwd)
        return y
