"""Forward-only UNet sampling on B200: the UNet-facing part of the reference's validation / inference path
(`StableVideoDiffusionPipeline(...)(image, num_frames=…, motion_bucket_id=127, fps=7, noise_aug_strength=0.02)`,
/root/reference/train_svd.py:1106-1140, infer_svd.ipynb cell 3).

One denoising step = scale the latents, append the conditioning latents on the channel axis, run the spatio-temporal UNet
on the classifier-free-guidance batch (2 x B clips), combine the two branches with the per-frame guidance scale and take the
Euler step (v-prediction). Every per-step scalar (sigma, sigma_next, timestep) lives in a small device buffer, so ONE captured
CUDA graph replays all `num_inference_steps` steps; between replays the host only writes three floats.

Scheduler constants follow diffusers' EulerDiscreteScheduler in the SVD configuration [D] (Karras sigmas, rho 7, sigma in
[0.002, 700], timesteps 0.25 ln sigma, init_noise_sigma sqrt(sigma_max^2 + 1)); tests/test_sampling_gpu.py checks the loop
against oracle/svd_sampling_oracle.py. Out of scope here: VAE encode / decode and the CLIP image encoder (SURVEY.md §8f-1/-4) —
`image_latents` and `image_embeddings` are inputs, denoised latents are the output. `image_embeddings` come from
`svd_xtend_b200.clip.encode_image(frame, image_encoder)` (the conditioning frame in [-1, 1]), the VAE latents from
`svd_xtend_b200.vae`.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

F32 = torch.float32


def karras_sigmas(num_inference_steps: int, sigma_min: float = 0.002, sigma_max: float = 700.0, rho: float = 7.0) -> torch.Tensor:
    ramp = torch.linspace(0, 1, num_inference_steps, dtype=torch.float64)
    lo, hi = sigma_min ** (1 / rho), sigma_max ** (1 / rho)
    return torch.cat([(hi + ramp * (lo - hi)) ** rho, torch.zeros(1, dtype=torch.float64)]).float()


class VideoLatentSampler:
    """Euler / classifier-free-guidance sampling loop around `UNetSpatioTemporalConditionModel.forward` (no_grad)."""

    def __init__(self, unet, use_cuda_graph: bool = True):
        self.unet = unet
        self.use_cuda_graph = use_cuda_graph
        self._graph = None
        self._key = None

    def _step(self, st):
        """one denoising step on the static buffers `st` (all device tensors; scal = [sigma, sigma_next, timestep])"""
        sigma, sigma_next, t = st["scal"][0], st["scal"][1], st["scal"][2]
        lat = st["latents"]
        inv = torch.rsqrt(sigma * sigma + 1.0)
        x = lat * inv
        if st["cfg"]:
            x = torch.cat([x, x])
        x = torch.cat([x, st["cond"]], dim=2)
        v = self.unet(x, t.expand(x.shape[0]), st["emb"], added_time_ids=st["ids"]).sample.float()
        if st["cfg"]:
            v_u, v_c = v.chunk(2)
            v = v_u + st["gs"] * (v_c - v_u)
        pred_x0 = v * (-sigma * inv) + lat * (inv * inv)
        lat.add_((lat - pred_x0) / sigma * (sigma_next - sigma))

    @torch.no_grad()
    def __call__(self, image_latents: torch.Tensor, image_embeddings: torch.Tensor, *, num_frames: int, fps: int = 7,
                 motion_bucket_id: int = 127, noise_aug_strength: float = 0.02, num_inference_steps: int = 25,
                 min_guidance_scale: float = 1.0, max_guidance_scale: float = 3.0, noise: Optional[torch.Tensor] = None,
                 generator: Optional[torch.Generator] = None) -> torch.Tensor:
        B, _, h, w = image_latents.shape
        dev = image_latents.device
        cfg = max_guidance_scale > 1.0
        emb = image_embeddings.float()
        cond = image_latents.float()
        if cfg:
            emb = torch.cat([torch.zeros_like(emb), emb])
            cond = torch.cat([torch.zeros_like(cond), cond])
        cond = cond.unsqueeze(1).repeat(1, num_frames, 1, 1, 1).contiguous()
        ids = torch.tensor([[float(fps - 1), float(motion_bucket_id), float(noise_aug_strength)]], device=dev, dtype=F32).repeat(B, 1)
        if cfg:
            ids = torch.cat([ids, ids])
        sigmas = karras_sigmas(num_inference_steps)
        if noise is None:
            noise = torch.randn(B, num_frames, 4, h, w, generator=generator, device=dev, dtype=F32)
        key = (B, num_frames, h, w, cfg, str(dev))
        if self._key != key:
            self._graph, self._key = None, key
            self._st = dict(latents=torch.empty(B, num_frames, 4, h, w, device=dev, dtype=F32), cond=torch.empty_like(cond),
                            emb=torch.empty_like(emb), ids=torch.empty_like(ids), scal=torch.zeros(3, device=dev, dtype=F32),
                            gs=torch.empty(1, num_frames, 1, 1, 1, device=dev, dtype=F32), cfg=cfg)
        st = self._st
        st["latents"].copy_(noise.float() * math.sqrt(float(sigmas[0]) ** 2 + 1.0))
        st["cond"].copy_(cond)
        st["emb"].copy_(emb)
        st["ids"].copy_(ids)
        st["gs"].copy_(torch.linspace(min_guidance_scale, max_guidance_scale, num_frames, device=dev, dtype=F32).view(1, -1, 1, 1, 1))
        # per-step scalars of ALL steps in one pinned buffer: row i is copied to the device right before step i (an async copy
        # from a re-used 3-float buffer would race with the host writing the next step's values)
        host = torch.empty(num_inference_steps, 3, dtype=F32).pin_memory()
        host[:, 0], host[:, 1] = sigmas[:-1], sigmas[1:]
        host[:, 2] = 0.25 * sigmas[:-1].log()
        was_training = self.unet.training
        self.unet.eval()
        try:
            for i in range(num_inference_steps):
                st["scal"].copy_(host[i], non_blocking=True)
                if not self.use_cuda_graph:
                    self._step(st)
                    continue
                if self._graph is None:
                    saved = st["latents"].clone()
                    side = torch.cuda.Stream()
                    side.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(side):
                        self._step(st)                     # warm-up: fills the weight-operand cache outside the capture
                    torch.cuda.current_stream().wait_stream(side)
                    st["latents"].copy_(saved)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._step(st)
                    st["latents"].copy_(saved)
                    self._graph = g
                self._graph.replay()
        finally:
            self.unet.train(was_training)
        out = st["latents"].clone()
        torch.cuda.current_stream().synchronize()      # `host` must outlive the queued copies
        return out
