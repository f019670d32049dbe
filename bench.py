#!/usr/bin/env python
"""bench.py — SVD UNet train-step frames/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|4|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" = one pass of the hot path over one synthetic batch: UNet forward + EDM loss + backward +
(N>1) gradient all-reduce + AdamW update, exactly what train_svd.py:934-1049 loops over, on
config 2 of BASELINE.json (bs=1/GPU, 14 frames, latents 8x40x64, bf16 compute, fp32 master weights,
trainable set as scripted at train_svd.py:761-766). value = whole-job frames/s with inputs resident in
HBM; e2e = the same step driven from pinned HOST buffers through the public
`UNetSpatioTemporalConditionModel.forward` (H2D of the inputs + D2H of the loss inside the timed region).

--impl reference times the reference's CPU path: the oracle restatement of the diffusers blocks under the
reference's own wiring (diffusers itself is not installable offline), fp32, all host threads, on a bounded
sample of the same workload (fewer frames of the same 40x64 latents per step).

--config selects the BASELINE.json configuration (default 2, the one the metric is quoted on; 4 = 25 frames 576x1024 with
gradient checkpointing, 5 = rank-64 LoRA): same step, same JSON line, `config.workload` names it.

Only the baseline legs (`cpu_baseline`, `--impl reference`, `gpu_eager_baseline`) import `oracle/`; the product arm takes
its synthetic batches and the EDM loss from svd_xtend_b200.workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_FRAMES, LAT_H, LAT_W = 14, 40, 64
METRIC = "SVD UNet train-step frames/sec @ 14x320x512 bf16"
WORKLOAD = ("train_svd.py full-finetune step as scripted (trainable = *temporal_transformer_block* params, "
            "train_svd.py:761-766), bs=1/GPU, 14 frames 320x512 (latents 14x8x40x64), bf16 compute, fp32 master weights, AdamW")
CPU_ARM_NOTE = ("CPU arm = oracle port (diffusers not installable offline), fp32, on a BOUNDED SAMPLE of the workload: fewer frames per "
                "step than the 14 of the GPU arm (same_config: false; a short clip shortens the temporal convolution / attention axis), "
                "scaled to frames/s by frame-equivalents")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5], help="BASELINE.json configuration")
    ap.add_argument("--ddp", default="p2p", choices=["p2p", "sharded", "allreduce"],
                    help="N > 1: p2p (default) = sharded AdamW with reduce-scatter + update + all-gather as ONE kernel over NVLink peer "
                         "memory (falls back to 'sharded' if the peer mapping cannot be set up); sharded = the same through NCCL "
                         "reduce-scatter / all-gather; allreduce = bucketed all-reduce + replicated AdamW")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the torch-eager bf16-autocast oracle timing on the GPU")
    ap.add_argument("--no-families", action="store_true", help="skip the per-family ablation rooflines")
    ap.add_argument("--no-script-path", action="store_true", help="skip the unchanged-script (eager, torch.optim.AdamW) timing")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step in a CUDA graph")
    ap.add_argument("--profile-one", action="store_true", help="run warm-up + one eager step only (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy: the UNet prediction, "
                         "the loss, and a fixed seeded sample of the updated trainable weights and of their gradients (float32), "
                         "with the sample positions (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 1400.0, 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- CPU reference arm
def build_oracle_cpu():
    from oracle.svd_unet_oracle import SVD_CONFIG, UNetSpatioTemporalConditionModel as Oracle
    with torch.device("meta"):
        m = Oracle(**SVD_CONFIG)
    m = m.to_empty(device="cpu")
    g = torch.Generator().manual_seed(1234)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("mix_factor"):
                p.fill_(0.5)
            elif "norm" in n and n.endswith("weight"):
                p.fill_(1.0)
            elif n.endswith("bias"):
                p.zero_()
            else:
                fan_in = p[0].numel()
                p.uniform_(-(fan_in ** -0.5), fan_in ** -0.5, generator=g)
    m.requires_grad_(False)
    for n, p in m.named_parameters():
        if "temporal_transformer_block" in n:   # train_svd.py:761-766
            p.requires_grad_(True)
    m.train()
    return m


def usable_cores():
    """Threads this process can really use: affinity mask and cgroup CPU quota, not the host's core count."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, (q + per // 2) // per))
        except Exception:
            pass
    return n


# (frames, latent H, latent W, frame-equivalents) samples of the BASELINE workload, largest first
CPU_SAMPLES = [(2, LAT_H, LAT_W, 2.0), (1, LAT_H, LAT_W, 1.0), (1, LAT_H, LAT_W // 4, 0.25)]


def cpu_step(model, frames, seed=1234, h=LAT_H, w=LAT_W):
    from oracle.svd_unet_oracle import edm_loss, synthetic_batch
    b = synthetic_batch(1, frames, h, w, seed=seed)
    t0 = time.perf_counter()
    pred = model(b["sample"], b["timestep"], b["encoder_hidden_states"], b["added_time_ids"]).sample
    loss = edm_loss(pred, b["noisy"], b["latents"], b["sigmas"])
    loss.backward()
    for p in model.parameters():
        p.grad = None
    return time.perf_counter() - t0


def pick_cpu_sample(model, n_steps, budget_s):
    """One quarter-frame probe step, then the largest sample whose n_steps fit the time budget."""
    f, h, w, eq = CPU_SAMPLES[-1]
    cpu_step(model, f, h=h, w=w)               # first touch of the weights
    tq = cpu_step(model, f, h=h, w=w)
    for s in CPU_SAMPLES:
        if tq * (s[3] / eq) * n_steps <= budget_s:
            return s, tq
    return CPU_SAMPLES[-1], tq


def _sample_text(s):
    return (f"{s[0]} of {T_FRAMES} frames at {s[1]}x{s[2]} latents (= {s[3]} frame-equivalents of the {LAT_H}x{LAT_W} workload)")


def cpu_baseline(budget_s=25.0):
    cores = usable_cores()
    torch.set_num_threads(cores)
    model = build_oracle_cpu()
    s, _ = pick_cpu_sample(model, 1, budget_s)
    t = cpu_step(model, s[0], h=s[1], w=s[2])
    return {"value": s[3] / t, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"1 x train step (fwd + EDM loss + bwd, fp32, as-scripted trainable set) on {_sample_text(s)}, "
                      f"full 1.52 B-param topology, torch CPU fp32, {cores} threads",
            "seconds": t}


def run_reference(args, out_fd):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = usable_cores()
    torch.set_num_threads(cores)
    model = build_oracle_cpu()
    # size the per-step sample so that the whole run stays within a few minutes
    s, _ = pick_cpu_sample(model, args.steps + args.warmup, 150.0)
    for _ in range(args.warmup):
        cpu_step(model, s[0], h=s[1], w=s[2])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(model, s[0], h=s[1], w=s[2])
    t = time.perf_counter() - t0
    val = s[3] * args.steps / t
    frames = s[3]
    sample = (f"each step = one train step (fwd + EDM loss + bwd, fp32, as-scripted trainable set) on {_sample_text(s)}, "
              f"full topology; oracle restatement of the diffusers path (diffusers not installable offline)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_sample": frames, "per_gpu_batch": 1},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(out_fd, line)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def count(self):
        """samples written so far (used to bracket the timed region)"""
        try:
            return sum(1 for r in open(self.f.name) if r.strip())
        except Exception:
            return 0

    def stop(self, first=0, last=None):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        if last is not None:
            # samples taken inside the timed region; a region shorter than the 100 ms period keeps its two neighbours
            # (the GPU runs the same replays right before and after the region)
            sel = rows[first:last]
            if not sel:
                sel = rows[max(first - 1, 0):last + 1]
            rows = sel
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


# ----------------------------------------------------------------------------- GPU torch-eager baseline (the "bar to beat")
def gpu_eager_baseline(dev, cfg, steps=3, warmup=2):
    """What the reference's script really executes on a GPU (SURVEY.md §2.3 K1/K5/K6): the diffusers-style module graph
    (here: the oracle restatement of it) under torch bf16 autocast — cuDNN convolutions, cuBLASLt linears, SDPA flash
    attention, eager elementwise kernels — with fp32 master weights, torch.optim.AdamW over the as-scripted trainable set.
    Baseline leg only (imports oracle/); informational: it is NOT the reference arm the driver computes its ratio with."""
    from oracle.svd_unet_oracle import SVD_CONFIG, UNetSpatioTemporalConditionModel as Oracle, edm_loss, synthetic_batch
    torch.manual_seed(1234)
    with torch.device(dev):
        m = Oracle(**SVD_CONFIG)
    m.to(dev)      # AlphaBlender.mix_factor is built with the legacy torch.Tensor([..]) constructor, which ignores the device context
    m.requires_grad_(False)
    for n, p in m.named_parameters():
        if "temporal_transformer_block" in n:
            p.requires_grad_(True)
    m.train()
    if cfg["grad_ckpt"]:
        m.enable_gradient_checkpointing()
    opt = torch.optim.AdamW([p for p in m.parameters() if p.requires_grad], lr=1e-5, weight_decay=1e-2)
    b = synthetic_batch(1, cfg["frames"], cfg["h"], cfg["w"], seed=1234, device=dev)

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            pred = m(b["sample"], b["timestep"], b["encoder_hidden_states"], b["added_time_ids"]).sample
        loss = edm_loss(pred.float(), b["noisy"], b["latents"], b["sigmas"])
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    out = {"value": cfg["frames"] / (ms / 1e3), "unit": "frames/s", "ms_per_step": ms, "steps": steps,
           "what": "oracle restatement of the diffusers modules under torch.autocast(bf16) on this GPU (cuDNN / cuBLASLt / SDPA / ATen eager), "
                   "fp32 masters, torch.optim.AdamW, as-scripted trainable set; informational"}
    del m, opt
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------- our arm
FAMILY_BOUND = {"linear": "tensor", "conv": "tensor", "attention": "tensor", "groupnorm": "hbm", "layernorm": "hbm", "adamw": "hbm",
                "elementwise": "hbm"}


def _protect_stdout():
    """The driver reads ONE JSON line from stdout. Libraries print there at C level (NCCL's version banner with NCCL_DEBUG set):
    fd 1 is pointed at stderr for the whole run and the line is written to the saved descriptor at the end."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(saved_fd, line):
    sys.stdout.flush()
    os.write(saved_fd, (json.dumps(line) + "\n").encode())


DUMP_SAMPLE = 1 << 20      # sampled elements of the trainable weights and of their gradients (4 MB each in float32)


def dump_outputs(out_dir, pred, loss, params):
    """What the last timed step hands its caller, as out_dir/<name>.npy in float32: `pred` (the UNet output), `loss`, and
    the updated weights and the gradients of the trainable parameters, flattened in parameter order, at DUMP_SAMPLE
    positions drawn with a fixed seed (`weights_sample`, `grads_sample`; the positions in `sample_index`, float64).
    Two runs with the same arguments agree to the bf16 noise floor, not bitwise: the GroupNorm statistics use fp32 atomics
    (DESIGN.md, run-to-run reproducibility)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(p.numel() for p in params)
    if total > DUMP_SAMPLE:
        idx = torch.randint(total, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).unique()
    else:
        idx = torch.arange(total)
    dev_idx = idx.to(params[0].device)
    weights = torch.cat([p.detach().reshape(-1) for p in params])[dev_idx]
    grads = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])[dev_idx]
    for name, t in (("pred", pred), ("loss", loss), ("weights_sample", weights), ("grads_sample", grads)):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "sample_index.npy"), idx.double().numpy())


def main():
    args = parse()
    out_fd = _protect_stdout()
    if args.impl == "reference":
        run_reference(args, out_fd)
        return

    import torch.distributed as dist
    from svd_xtend_b200 import raw
    from svd_xtend_b200.train import FusedAdamW, GradReducer, GraphedStep, P2PShardedAdamW, ParamArena, ShardedAdamW
    from svd_xtend_b200.unet import UNetSpatioTemporalConditionModel
    from svd_xtend_b200.workload import BENCH_CONFIGS, SVD_CONFIG, edm_loss, synthetic_batch   # train_svd.py:951-1036

    cfg = BENCH_CONFIGS[args.config]
    frames, lat_h, lat_w = cfg["frames"], cfg["h"], cfg["w"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (ours) needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- model: SVD topology, seeded default init (no checkpoints offline)
    torch.manual_seed(1234)
    with torch.device(dev):
        unet = UNetSpatioTemporalConditionModel(**SVD_CONFIG)
    unet.to(dev)
    unet.requires_grad_(False)
    if cfg["lora_rank"]:
        # train_svd_lora.py:645-675: frozen base in the mixed-precision dtype, LoRA on q/k/v/out of every Attention; the LoRA
        # parameters are kept in fp32 here (>= the reference's precision: its bf16 run keeps them in bf16)
        from types import SimpleNamespace
        unet.to(torch.bfloat16)
        r = cfg["lora_rank"]
        unet.add_adapter(SimpleNamespace(r=r, lora_alpha=r, init_lora_weights="gaussian", target_modules=["to_k", "to_q", "to_v", "to_out.0"]))
        for p in unet.parameters():
            if p.requires_grad:
                p.data = p.data.float()
    else:
        for n, p in unet.named_parameters():
            if "temporal_transformer_block" in n:   # train_svd.py:761-766
                p.requires_grad_(True)
    n_train = sum(p.numel() for p in unet.parameters() if p.requires_grad)
    n_total = sum(p.numel() for p in unet.parameters())
    unet.train()
    if cfg["grad_ckpt"]:
        unet.enable_gradient_checkpointing()     # train_svd.py:731-732
    sharded = world > 1 and args.ddp in ("sharded", "p2p")
    arena = ParamArena(unet, pad_to=world * 64)
    unet.attach_arena(arena)
    hyper = dict(lr=1e-5, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)             # train_svd.py:384-418 defaults
    # N > 1 (default): reduce-scatter of the gradient arena + AdamW on this rank's 1/N slice + all-gather of the bf16 operand
    # weights (0.75x the NVLink bytes of an all-reduce, 1/N of the optimizer traffic); --ddp allreduce keeps replicated AdamW
    ddp_mode = args.ddp if world > 1 else None
    if sharded and args.ddp == "p2p":
        # the fused exchange needs every rank's arenas mapped into every process (CUDA IPC, one node): all ranks agree on
        # whether that worked before anyone builds a graph on it
        try:
            opt = P2PShardedAdamW(arena, **hyper)
            ok = torch.ones(1, device=dev)
        except Exception as e:      # noqa: BLE001
            print(f"[bench] rank {rank}: peer mapping failed ({type(e).__name__}: {e}); using the NCCL sharded exchange", file=sys.stderr, flush=True)
            opt, ok = None, torch.zeros(1, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() < 1:
            opt = ShardedAdamW(arena, **hyper)
            ddp_mode = "sharded (p2p mapping unavailable)"
    elif sharded:
        opt = ShardedAdamW(arena, **hyper)
    else:
        opt = FusedAdamW(arena, **hyper)
    opt.on_updated = lambda: unet.refresh_trainable_operands(shadow_current=True)   # the optimizer rewrites the bf16 shadow itself
    reducer = GradReducer(arena) if (world > 1 and not sharded) else None
    if reducer is not None:
        unet.grad_hook = lambda ps: reducer.on_grads_ready(ps) if ps is not None else None

    host = synthetic_batch(1, frames, lat_h, lat_w, seed=1234 + rank)
    host = {k: v.pin_memory() for k, v in host.items()}
    devb = {k: v.to(dev) for k, v in host.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())

    def step(b):
        arena.zero_grad()
        pred = unet(b["sample"], b["timestep"], b["encoder_hidden_states"], added_time_ids=b["added_time_ids"]).sample
        loss = edm_loss(pred.float(), b["noisy"], b["latents"], b["sigmas"])
        loss.backward()
        if reducer is not None:
            reducer.finish()
        opt.step()
        return loss, pred

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also fills the weight-operand cache); with graphs the warm-up happens inside GraphedStep
    # world > 1: the bucketed NCCL all-reduces of GradReducer are captured into the same graph (side-stream fork/join)
    use_graph = (not args.no_graph) and not args.profile_one and (world == 1 or os.environ.get("SVDX_DDP_GRAPH", "1") != "0")
    lps = 0
    account = {}

    def acc(fam, flops, nbytes):
        a = account.setdefault(fam, [0, 0.0, 0.0])
        a[0] += 1
        a[1] += flops
        a[2] += nbytes

    for i in range(1 if use_graph else max(args.warmup, 3)):
        l_before = raw.LAUNCHES[0]
        if i == 0:
            raw.ACCOUNT = acc           # algorithmic FLOPs / bytes of every launch of ONE step, by kernel family
        step(devb)
        raw.ACCOUNT = None
        lps = raw.LAUNCHES[0] - l_before      # kernels of OUR library launched by one step
    barrier()
    if args.profile_one:
        if os.environ.get("SVDX_SHAPE_LOG"):
            raw.SHAPE_LOG = []
        step(devb)
        torch.cuda.synchronize()
        if raw.SHAPE_LOG is not None:     # the tapgemm launches of the LAST step, in launch order (scripts/join_shapes.py)
            with open(os.environ["SVDX_SHAPE_LOG"], "w") as fh:
                json.dump(raw.SHAPE_LOG, fh)
        return

    # ---- CUDA-graph capture of the whole step through the public helper (svd_xtend_b200.train.GraphedStep)
    graphed = None
    if use_graph:
        try:
            l_before = raw.LAUNCHES[0]
            graphed = GraphedStep(step, devb, warmup=max(args.warmup, 3))
            lps = (raw.LAUNCHES[0] - l_before) // (max(args.warmup, 3) + 1)
        except Exception as e:  # fall back to eager launches, say so
            import traceback
            traceback.print_exc()
            print(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); timing eager launches", file=sys.stderr)
            graphed = None
            torch.cuda.synchronize()
    graph_captured = graphed is not None

    def run_step():
        if graphed is not None:
            return graphed.replay()
        return step(devb)

    for _ in range(2):
        run_step()
    barrier()

    # ---- timed region: K steps, device events, max over ranks
    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(8):          # nvidia-smi needs a few hundred ms to emit its first sample: keep the GPU under the same load
        run_step()
    l0 = raw.LAUNCHES[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    c0 = clocks.count() if clocks is not None else 0
    e0.record()
    for _ in range(args.steps):
        loss, pred = run_step()
    e1.record()
    barrier()
    c1 = clocks.count() if clocks is not None else 0
    ms = e0.elapsed_time(e1)
    launches = raw.LAUNCHES[0] - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pred, loss, [p for p in unet.parameters() if p.requires_grad])
    for _ in range(2):          # one more sampling period under load before the sampler stops
        run_step()
    torch.cuda.synchronize()
    clk = clocks.stop(c0, c1) if clocks is not None else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = frames * world * args.steps / (ms / 1e3)
    final_loss = float(loss.item())

    # ---- e2e: public API from pinned host buffers, H2D inside, loss read back every step
    def e2e_step():
        if graphed is not None:     # pinned host -> static device buffers -> one graph launch -> loss back to the host
            return float(graphed(host)[0].item())
        b = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        return float(step(b)[0].item())

    e2e_step()
    barrier()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = frames * world * args.steps / (float(t.item()) / 1e3)

    # ---- rooflines. In eager mode the CPU (descriptor build + cuLaunchKernel, ~10 us) trails the GPU, so an event pair around one
    # launch also times host work whenever the stream is idle. With the whole step in a CUDA graph the in-step cost of a kernel
    # FAMILY is measured by ablation instead: capture the same step with every launch of that family skipped (raw.ABLATE) and
    # take the difference of the two replay times (CUDA events, the same K replays, max over ranks). Same method at every N.
    # Algorithmic work per family comes from raw.ACCOUNT over one step. Done last: the ablated steps compute garbage.
    sustained, burst, hbm, src = peaks()

    def ablated_ms(fams):
        raw.ABLATE = set(fams)
        try:
            g = GraphedStep(step, devb, warmup=2)
            for _ in range(2):
                g.replay()
            barrier()
            e0.record()
            for _ in range(args.steps):
                g.replay()
            e1.record()
            barrier()
            tt = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            del g
            return float(tt.item())
        finally:
            raw.ABLATE = set()

    fam_ms = {}
    method = None
    if graph_captured and args.config == 4:
        graphed = None              # one captured step of config 4 holds > 60 GB of activations: release it before re-capturing
        torch.cuda.empty_cache()
    if graph_captured:
        todo = [("tapgemm", ["linear", "conv"])]
        if not args.no_families and world == 1:
            todo += [(f, [f]) for f in ("linear", "conv", "attention", "groupnorm", "layernorm", "adamw", "elementwise") if f in account]
        for name, fams in todo:
            try:
                wo = ablated_ms(fams)
                if 0.0 < wo < ms_per_step:
                    fam_ms[name] = ms_per_step - wo
            except Exception as e:
                print(f"[bench] ablation of {name} failed ({type(e).__name__}: {e})", file=sys.stderr)
        method = ("graph-replay ablation: ms_per_step minus the replay time of the same captured step with every launch of the kernel "
                  f"family skipped, CUDA events over {args.steps} replays each")
    gemm_flops = sum(account.get(f, [0, 0.0, 0.0])[1] for f in ("linear", "conv"))
    gemm_launches = sum(account.get(f, [0, 0.0, 0.0])[0] for f in ("linear", "conv"))
    gemm_ms = fam_ms.get("tapgemm")
    if gemm_ms is None:       # no graph: events around every tapgemm launch of one eager step (includes host launch gaps)
        recs = []
        orig = raw.tapgemm

        def timed_tapgemm(a, b, out, **kw):
            s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s_.record()
            r_ = orig(a, b, out, **kw)
            e_.record()
            recs.append((s_, e_))
            return r_

        raw.tapgemm = timed_tapgemm
        try:
            step(devb)
            torch.cuda.synchronize()
        finally:
            raw.tapgemm = orig
        gemm_ms = sum(s_.elapsed_time(e_) for s_, e_ in recs)
        method = "sum of CUDA-event pairs around every svdx_tapgemm launch of one eager step (host launch gaps included)"
    traffic, traffic_src = None, None
    pdir = os.path.join(ROOT, "profiles")
    for tp in sorted([f for f in os.listdir(pdir) if f.endswith("_traffic.json")] if os.path.isdir(pdir) else [], reverse=True):
        try:
            tj = json.load(open(os.path.join(pdir, tp)))
            traffic, traffic_src = tj["traffic_bytes_per_launch"], f"profiles/{tp} (ncu dram__bytes_read+write summed over the {tj['launches_per_step']} tapgemm launches of one step, per launch)"
            break
        except Exception:
            pass
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms and gemm_ms > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "svdx::tapgemm2_kernel / tapgemm_kernel (tcgen05)", "achieved": achieved, "peak": sustained, "unit": "TFLOP/s",
                "frac": achieved / sustained, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_note": "tensor-bound kernel: algorithmic work is FLOPs (2*M*N*K*taps per launch, summed); see DESIGN.md §3",
                "peak_source": src + ", bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_per_step": gemm_launches, "algorithmic_tflop_per_step": gemm_flops / 1e12, "kernel_ms_per_step": gemm_ms,
                "avg_launch_us": 1e3 * gemm_ms / max(gemm_launches, 1), "timing_method": method,
                "share_of_step": gemm_ms / ms_per_step}
    by_family = {}
    for fam, (n_l, fl, by) in account.items():
        if fam not in fam_ms:
            continue
        t_ms = fam_ms[fam]
        if FAMILY_BOUND[fam] == "tensor":
            ach = fl / (t_ms / 1e3) / 1e12
            by_family[fam] = {"bound": "tensor", "achieved": ach, "peak": sustained, "unit": "TFLOP/s", "frac": ach / sustained,
                              "ms_per_step": t_ms, "launches_per_step": n_l, "algorithmic_tflop_per_step": fl / 1e12}
        else:
            ach = by / (t_ms / 1e3) / 1e9
            by_family[fam] = {"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                              "ms_per_step": t_ms, "launches_per_step": n_l, "algorithmic_gb_per_step": by / 1e9}

    # ---- the unchanged-script calling pattern (train_svd.py:1021-1049): eager launches from Python, forward inside an autocast
    # region, torch.optim.AdamW over p.grad, zero_grad(set_to_none=True); no GraphedStep, no FusedAdamW.
    script_path = None
    if world == 1 and not args.no_script_path:
        try:
            topt = torch.optim.AdamW([p for p in unet.parameters() if p.requires_grad], lr=1e-5, weight_decay=1e-2)

            def script_step():
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    pred = unet(devb["sample"], devb["timestep"], devb["encoder_hidden_states"], added_time_ids=devb["added_time_ids"]).sample
                loss_ = edm_loss(pred.float(), devb["noisy"], devb["latents"], devb["sigmas"])
                loss_.backward()
                topt.step()
                topt.zero_grad(set_to_none=True)
                return loss_

            for _ in range(2):
                script_step()
            torch.cuda.synchronize()
            n_s = max(3, min(args.steps, 10))
            e0.record()
            for _ in range(n_s):
                script_step()
            e1.record()
            torch.cuda.synchronize()
            sp_ms = e0.elapsed_time(e1) / n_s
            script_path = {"ms_per_step": sp_ms, "value": frames / (sp_ms / 1e3), "unit": "frames/s", "steps": n_s,
                           "what": "unet(...) inside torch.autocast + loss.backward() + torch.optim.AdamW.step() + zero_grad(set_to_none=True), "
                                   "every kernel launched eagerly from Python through the C ABI (train_svd.py:1021-1049 pattern)"}
            # the same loop with unet.enable_cuda_graphs(): forward and backward of the autograd node replay captured graphs
            try:
                unet.enable_cuda_graphs(warmup=2)
                for _ in range(5):
                    script_step()
                torch.cuda.synchronize()
                e0.record()
                for _ in range(n_s):
                    script_step()
                e1.record()
                torch.cuda.synchronize()
                spg_ms = e0.elapsed_time(e1) / n_s
                script_path["graphed_ms_per_step"] = spg_ms
                script_path["graphed_value"] = frames / (spg_ms / 1e3)
                script_path["graphed_what"] = ("same script loop after unet.enable_cuda_graphs(): two shape-keyed graph launches (forward, backward) "
                                               "per step + the script's own torch.optim.AdamW")
            except Exception as e:
                script_path["graphed_failed"] = f"{type(e).__name__}: {e}"
            finally:
                unet.disable_cuda_graphs()
            del topt
        except Exception as e:
            script_path = {"failed": f"{type(e).__name__}: {e}"}

    # ---- the data-parallel exchange alone (N > 1): the same collectives captured without the step around them
    exchange = None
    if world > 1:
        try:
            p2p = isinstance(opt, P2PShardedAdamW)

            def ex():
                if p2p:
                    opt._fence()
                    raw.adamw_p2p(arena.data[opt.lo:opt.hi], opt.m, opt.v, opt.peer_grad, opt.peer_shadow, opt.lo, ex_state, 1.0 / world, tick=False)
                    opt._fence()
                elif sharded:
                    opt.reduce_scatter_grads()
                    opt.all_gather_(arena.shadow)
                else:
                    dist.all_reduce(arena.grad)
            # (p2p: the timed kernel includes the optimizer arithmetic; lr = 0 and weight decay 0 in this copy of the state so
            # the replays leave the weights alone)
            ex_state = opt.state.clone() if p2p else None
            if p2p:
                ex_state[0] = 0.0
                ex_state[4] = 0.0
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                ex()
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            gx = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gx):
                ex()
            gx.replay()
            barrier()
            e0.record()
            for _ in range(5):
                gx.replay()
            e1.record()
            barrier()
            tx = torch.tensor([e0.elapsed_time(e1) / 5], device=dev)
            dist.all_reduce(tx, op=dist.ReduceOp.MAX)
            nb = arena.numel * 4
            exchange = {"ms": float(tx.item()), "mode": ddp_mode,
                        "payload_bytes": nb if not sharded else nb + arena.numel * 2,
                        "what": ("fence + svdx_adamw_p2p (peer loads of the gradient slices, AdamW on 1/N, peer stores of the bf16 operands) + fence" if p2p
                                 else "reduce-scatter(fp32 gradient arena) + all-gather(bf16 operand weights)" if sharded else "all-reduce(fp32 gradient arena)")
                                + " alone in a CUDA graph, max over ranks; in the step it runs after the backward (not overlapped)"}
            del gx
        except Exception as e:
            exchange = {"failed": f"{type(e).__name__}: {e}"}

    def finish():
        """leave without tearing NCCL down: communicators referenced by live CUDA graphs block destroy_process_group()"""
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            import threading
            threading.Timer(30.0, lambda: os._exit(0)).start()   # the result line is out: never hang in teardown
            try:
                dist.barrier()
                torch.cuda.synchronize()
            except Exception:
                pass
            os._exit(0)

    if rank != 0:
        finish()
        return

    # ---- the VAE encode that precedes the UNet in every step of train_svd.py (:948, :959): frames + 1 conditioning frame
    vae_encode = None
    if world == 1 and args.config == 2 and not args.no_script_path:
        try:
            from svd_xtend_b200.vae import AutoencoderKLTemporalDecoder, tensor_to_vae_latent
            graphed = None
            torch.cuda.empty_cache()
            torch.manual_seed(7)
            with torch.device(dev):
                vae = AutoencoderKLTemporalDecoder()
            vae.to(dev).requires_grad_(False).eval()
            px = (torch.randn(1, frames + 1, 3, 8 * lat_h, 8 * lat_w, device=dev) * 0.5).clamp(-1, 1)
            for _ in range(2):
                tensor_to_vae_latent(px, vae)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                lat = tensor_to_vae_latent(px, vae)
            e1.record()
            torch.cuda.synchronize()
            v_ms = e0.elapsed_time(e1) / 3
            vae_encode = {"ms": v_ms, "frames": frames + 1, "pixels": [8 * lat_h, 8 * lat_w], "finite": bool(torch.isfinite(lat).all()),
                          "what": "svd_xtend_b200.vae.tensor_to_vae_latent on the clip + conditioning frame (train_svd.py:283-291, :948, :959), eager launches, "
                                  "random-init weights; informational (SURVEY.md §8f-1)"}
            del vae, px, lat
            torch.cuda.empty_cache()
        except Exception as e:
            vae_encode = {"failed": f"{type(e).__name__}: {e}"}

    gpu_base = None
    if world == 1 and not args.no_gpu_baseline:
        try:
            graphed = None
            torch.cuda.empty_cache()
            gpu_base = gpu_eager_baseline(dev, cfg)
        except Exception as e:
            gpu_base = {"failed": f"{type(e).__name__}: {e}"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline()
        except Exception as e:
            cpu = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (seeded default-init weights, randn latents per train_svd.py:951-1017)",
        "config": {"workload": cfg["name"], "baseline_config": args.config, "frames": frames, "latent_hw": [lat_h, lat_w], "per_gpu_batch": 1,
                   "global_batch": world, "trainable_params": n_train, "total_params": n_total, "parallelism": f"dp{world}" + ("" if world == 1 else "-zero1-p2p" if isinstance(opt, P2PShardedAdamW) else "-zero1" if sharded else "-allreduce"),
                   "cuda_graph": graph_captured, "gradient_checkpointing": bool(cfg["grad_ckpt"]), "lora_rank": cfg["lora_rank"],
                   "l2": "no explicit flush: the per-step working set (3 GB bf16 operand weights + >10 GB activations) is >> 126 MB L2",
                   "final_loss": final_loss, "cpu_arm": CPU_ARM_NOTE},
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
        "gpu_launches": launches if not graph_captured else lps * args.steps,   # graph replay re-launches the captured kernels
        "roofline": roofline,
        "roofline_by_family": by_family,
        "exchange": exchange,
        "script_path": script_path,
        "vae_encode": vae_encode,
        "gpu_eager_baseline": gpu_base,
        "cpu_baseline": cpu,
    }
    _emit(out_fd, line)
    finish()


if __name__ == "__main__":
    main()
