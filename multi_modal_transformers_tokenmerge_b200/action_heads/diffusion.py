"""Mirror of multi_modal_transformers/action_heads/diffusion.py (training path) on csrc/diffusion_head.cu.

    cosine_beta_schedule(timesteps, s=0.008)                                                        diffusion.py:16-26
    DiffusionActionHead(diffusion_steps, attention_pooling, denoising_model, rng_collection)       :66-92
        .denoise_loss(variables, readouts, actions, rng)  -> loss                                  :114-143
        .predict_denoise_term(variables, readouts, time, noisy_actions) -> [B, A]                  :94-112

`denoising_model` is the OctoDenoise config node of model_configs/action_heads/diffusion.yaml (time_encoder =
FourierFeatures + MLPBlock, mlp_block = the denoiser MLPBlock, num_blocks = 1).  Parameter tree, Flax names:
    denoiser/FourierFeatures_0/{fourier_kernel [F/2, 1], MLPBlock_0/Dense_{0,1}/{kernel, bias}}
    denoiser/MLPBlock_0/Dense_{0,1}/{kernel, bias}
The sampling loop (`predict_action`, :145-213) runs as one call, tome_diffusion_head_sample.  Random draws: jax's threefry
cannot be reproduced, so `denoise_loss` and `predict_action` draw from a numpy Generator seeded by `rng` (or take them
explicitly) -- statistics, not bits, match the reference.
"""
from __future__ import annotations

from typing import Any, Dict, Optional

import numpy as np
import torch

from .. import _lib as L
from .. import ops
from ..attention_blocks._module import Module, as_rng, instantiate, make_init


def cosine_beta_schedule(timesteps: int, s: float = 0.008) -> np.ndarray:
    """Host arithmetic in fp32, as jnp computes it (diffusion.py:16-26)."""
    f = np.float32
    t = np.linspace(f(0), f(timesteps), timesteps + 1, dtype=np.float32) / f(timesteps)
    ac = np.cos((t + f(s)) / f(1 + s) * f(np.pi) * f(0.5)) ** 2
    ac = ac / ac[0]
    return np.clip(f(1) - ac[1:] / ac[:-1], 0, 0.999).astype(np.float32)


def ddpm_coefficients(betas: np.ndarray) -> np.ndarray:
    """f32 [steps, 3]: row t = (c1, c2, c3) = (1 / sqrt(alpha_t), (1 - alpha_t) / sqrt(1 - alpha_hat_t), sqrt(beta_t)) of the
    sampler's update (diffusion.py:183-186), in the precision the reference's host arithmetic gives."""
    betas = np.asarray(betas, np.float32)
    alphas = np.float32(1) - betas
    ah = np.array([np.prod(alphas[: i + 1]) for i in range(len(betas))], np.float32)
    return np.array([[1.0 / float(np.sqrt(alphas[t])), float((np.float32(1) - alphas[t]) / np.sqrt(np.float32(1) - ah[t])),
                      float(np.sqrt(betas[t]))] for t in range(len(betas))], np.float32)


class DiffusionActionHead(Module):
    def __init__(self, diffusion_steps: int, attention_pooling: Optional[Dict[str, Any]], denoising_model: Dict[str, Any],
                 rng_collection: str = "diffusion"):
        self.diffusion_steps, self.attention_pooling = diffusion_steps, attention_pooling
        self.denoising_model, self.rng_collection = denoising_model, rng_collection
        self.betas = cosine_beta_schedule(diffusion_steps)                                              # :86
        self.alphas = np.float32(1) - self.betas                                                        # :87
        self.alpha_hats = np.array([np.prod(self.alphas[: i + 1]) for i in range(diffusion_steps)], np.float32)   # :88-90
        dm = denoising_model
        if int(dm.get("num_blocks", 1)) != 1:
            raise NotImplementedError("OctoDenoise.num_blocks != 1 (diffusion.yaml uses 1)")
        te = dm["time_encoder"]
        self._F = int(te["output_dim"])
        self._t0, self._t1 = instantiate(te["mlp_block"]["dense"]), instantiate(te["mlp_block"]["dense_out"])
        self._d0, self._d1 = instantiate(dm["mlp_block"]["dense"]), instantiate(dm["mlp_block"]["dense_out"])
        self._fourier_init = te.get("kernel_init")

    # ---- parameters
    def _desc(self, readouts) -> "L.DiffusionDesc":
        B, n, C = readouts.shape
        return L.DiffusionDesc(B, n, C, n, self._d1.features, self._F, self._t0.features, self._t1.features, self._d0.features,
                               self.diffusion_steps)

    def _init(self, rng, readouts):
        C = readouts.shape[-1]
        A, F, Ht, To, H = self._d1.features, self._F, self._t0.features, self._t1.features, self._d0.features

        def dense(spec, fan_in):
            return {"kernel": make_init(spec.kernel_init)(rng, (fan_in, spec.features), fan_in, spec.features),
                    "bias": make_init(spec.bias_init)(rng, (spec.features,))}
        return {"denoiser": {
            "FourierFeatures_0": {"fourier_kernel": make_init("he_normal")(rng, (F // 2, 1), 1, F // 2),
                                  "MLPBlock_0": {"Dense_0": dense(self._t0, F), "Dense_1": dense(self._t1, Ht)}},
            "MLPBlock_0": {"Dense_0": dense(self._d0, A + To + C), "Dense_1": dense(self._d1, H)}}}

    def _flat(self, params, device) -> torch.Tensor:
        d = params["denoiser"]
        ff, tm, dm = d["FourierFeatures_0"], d["FourierFeatures_0"]["MLPBlock_0"], d["MLPBlock_0"]
        parts = [ff["fourier_kernel"], tm["Dense_0"]["kernel"], tm["Dense_0"]["bias"], tm["Dense_1"]["kernel"], tm["Dense_1"]["bias"],
                 dm["Dense_0"]["kernel"], dm["Dense_0"]["bias"], dm["Dense_1"]["kernel"], dm["Dense_1"]["bias"]]
        return torch.cat([torch.as_tensor(np.asarray(p, np.float32)).reshape(-1) for p in parts]).to(device)

    # ---- training path
    def _run(self, params, readouts, actions, time, noise):
        if readouts.dim() != 3:
            raise ValueError("readouts must be [batch, readout, embedding] (diffusion.py:107 reduces axis -2)")
        x = readouts.to(torch.bfloat16).contiguous()
        dev = x.device
        return ops.diffusion_head_fwd(x, self._flat(params, dev), self._desc(readouts), actions.float().contiguous(),
                                      noise.float().contiguous(), time.to(torch.int32).reshape(-1).contiguous(),
                                      torch.as_tensor(self.alpha_hats).to(dev))

    def denoise_loss(self, variables, readouts, actions, rng=0, time=None, noise=None, train=True):
        """:114-143.  time int [B] / [B, 1] and noise [B, A] may be given; otherwise drawn from `rng`."""
        g = as_rng(rng)
        B, A = actions.shape
        if time is None:
            time = torch.as_tensor(g.integers(0, self.diffusion_steps, size=(B, 1)).astype(np.int32)).to(actions.device)   # :125
        if noise is None:
            noise = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32)).to(actions.device)                        # :128
        _, loss, _ = self._run(variables["params"], readouts, actions, time, noise)
        return loss[0]

    def predict_denoise_term(self, variables, readouts, time, noisy_actions, train=True):
        """:94-112 -- the same kernels with alpha_hat = 1 (so noisy = the given actions) and the loss ignored."""
        x = readouts.to(torch.bfloat16).contiguous()
        desc = self._desc(readouts)
        ones = torch.ones(self.diffusion_steps, dtype=torch.float32, device=x.device)
        z = torch.zeros_like(noisy_actions, dtype=torch.float32)
        pred, _, _ = ops.diffusion_head_fwd(x, self._flat(variables["params"], x.device), desc, noisy_actions.float().contiguous(), z,
                                            time.to(torch.int32).reshape(-1).contiguous(), ones)
        return pred

    def predict_action(self, variables, readouts, rng=0, train=True, init=None, noise=None, clip: float = 5.0):
        """:146-213 -- the sampling loop (inference): start from Gaussian noise [B, A], and for time = steps - 1 .. 0 take the
        denoise term and apply algorithm 2 of arXiv:2006.11239 with the schedule's coefficients, clipping to [-5, 5] (:190).
        The reference draws its step noise from the SAME per-sample keys at every step (:179, "TODO: check keys here"), i.e. one
        noise tensor [B, A] reused by all steps; `noise` may also be [steps, B, A].  `init` / `noise` default to draws from `rng`
        (numpy's generator, not jax.random's stream).  All steps run in one call (tome_diffusion_head_sample)."""
        g = as_rng(rng)
        x = readouts.to(torch.bfloat16).contiguous()
        dev = x.device
        B, A = x.shape[0], self._d1.features
        if init is None:
            init = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32))
        if noise is None:
            noise = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32))
        init = init.to(dev).float().contiguous()
        noise = noise.to(dev).float().contiguous()
        coef = torch.as_tensor(ddpm_coefficients(self.betas)).to(dev)
        return ops.diffusion_head_sample(x, self._flat(variables["params"], dev), self._desc(readouts), init, noise, coef, clip)

    def _apply(self, params, readouts, time, noisy_actions, dropout_rng=None):
        return self.predict_denoise_term({"params": params}, readouts, time, noisy_actions)
