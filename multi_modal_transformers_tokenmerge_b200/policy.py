"""Camera frames to actions in one native call (tome_policy_predict, C ABI 18): what Octo.generate_readouts
(models/octo/octo.py:91-126) and predict_continuous_action / predict_diffusion_action on top of it do, for closed-loop control.

`PixelPolicy` runs the image front end, writes its tokens straight into their rows of the assembled sequence, copies the text
and readout embeddings into theirs, and runs the forward-only stack and the action head (or the diffusion sampler), all in one
call over one workspace.  It reads the training engine's parameter storage (`ToMeStackEngine.policy`), so it sees every AdamW
step without a reload.  With graph=True the call is captured once into a CUDA graph and replayed: at small batches a prediction
is a few hundred short kernels, and replaying them saves the host work between launches.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from .ops import _scratch
from .tokenizers.images.image_tokenizer import encode_patch_position
from .tokenizers.token_sequencer import TokenSequence


def placement(token_sequence: TokenSequence, n_image_tokens: int):
    """The grammar's layout of the assembled sequence, as TokenSequence.assemble_embeddings fills it: (image_rows int32
    [n_image_tokens], sets) where image token k (= n * n_patches + p) lands in row image_rows[k] and `sets` lists the non-image
    token sets as (modality, first token of the modality's input, tokens, first sequence row)."""
    image_rows = token_sequence.get_modality_idx("images")
    if image_rows.size != n_image_tokens:
        raise ValueError(f"the grammar holds {image_rows.size} image tokens, the frames give {n_image_tokens}")
    sets, cursor, row = [], {"text": 0, "readouts": 0}, 0
    for s in token_sequence.token_sequence:
        if s.modality != "images" and s.num_tokens > 0:
            sets.append((s.modality, cursor[s.modality], s.num_tokens, row))
            cursor[s.modality] += s.num_tokens
        row += s.num_tokens
    return image_rows.astype(np.int32), sets


class PixelPolicy:
    """Frames -> actions at a fixed batch (build with `ToMeStackEngine.policy`).  One CUDA graph per policy: another batch
    size needs another policy."""

    def __init__(self, engine, tokenizer, tokenizer_variables, token_sequence, batch: Optional[int] = None, graph: bool = False):
        self.lib = L.lib()
        self.cfg = engine.cfg if batch is None else dataclasses.replace(engine.cfg, batch=int(batch))
        cfg, dev = self.cfg, engine.dev
        self.dev = dev
        self.ccfg = cfg.c()
        self.params, self.params_bf16 = engine.params, engine.params_bf16   # the engine's storage, not a copy
        self.gid, self.pos, self.allow, self.readout_idx = engine.gid, engine.pos, engine.allow, engine.readout_idx
        self.layer_gid, self.layer_pos = engine.layer_gid, engine.layer_pos
        self.tokenizer = tokenizer
        ts = token_sequence if isinstance(token_sequence, TokenSequence) else TokenSequence(token_sequence)
        if ts.num_tokens != cfg.tokens:
            raise ValueError(f"the grammar holds {ts.num_tokens} tokens, the stack {cfg.tokens}")
        H, _, _ = tokenizer.image_size
        self.n_patches = (H // tokenizer.patch_size) ** 2
        n_img = ts.get_modality_idx("images").size
        if n_img == 0 or n_img % self.n_patches:
            raise ValueError(f"{n_img} image tokens in the grammar are not whole frames of {self.n_patches} patches")
        self.n_images = n_img // self.n_patches
        self.image_rows, self.sets = placement(ts, n_img)
        self.n_text = sum(n for m, _, n, _ in self.sets if m == "text")
        self.n_readouts = sum(n for m, _, n, _ in self.sets if m == "readouts")
        # the front end's parameters, packed once (what ImageTokenizer.apply packs); evaluation-mode position tokens
        self.image_params = tokenizer.pack_params(tokenizer_variables["params"], dev)
        self.image_params_bf16 = self.image_params.to(torch.bfloat16)
        row, col = encode_patch_position(H, tokenizer.patch_size, tokenizer.position_interval, False)
        self.row_tokens = torch.from_numpy(np.ascontiguousarray(row)).to(dev)
        self.col_tokens = torch.from_numpy(np.ascontiguousarray(col)).to(dev)
        self._zero_readouts = torch.zeros(1, self.n_readouts, cfg.channels, dtype=torch.bfloat16, device=dev)
        # outputs and (diffusion head) the DDPM coefficient table, uploaded once
        self.readout = (torch.empty(cfg.batch, cfg.n_readout, cfg.channels, dtype=torch.float32, device=dev) if cfg.n_readout else None)
        self.head_out = (torch.empty(cfg.batch, cfg.head_groups, cfg.head_features, dtype=torch.float32, device=dev)
                         if cfg.head != "none" else None)
        self.coef = None
        if cfg.head == "diffusion":
            from .action_heads.diffusion import cosine_beta_schedule, ddpm_coefficients
            self.coef = torch.as_tensor(ddpm_coefficients(cosine_beta_schedule(cfg.diffusion_steps))).to(dev)
        ws = max(self.workspace_bytes(torch.uint8), self.workspace_bytes(torch.float32))
        self.workspace = _scratch(ws, dev)
        self._ws_bytes = ws
        self.graph = bool(graph)
        self._graph = None
        self._static = None

    # ------------------------------------------------------------------ the native call
    def _inputs(self, dtype: torch.dtype, pixels=None, text=None, readouts=None) -> L.PolicyInputs:
        cfg = self.cfg
        d = self.tokenizer._desc(cfg.batch, self.n_images, dtype, 1)
        inp = L.PolicyInputs()
        inp.image = d
        inp.image_params_f32, inp.image_params_bf16 = self.image_params.data_ptr(), self.image_params_bf16.data_ptr()
        inp.pixels = None if pixels is None else pixels.data_ptr()
        inp.row_tokens, inp.col_tokens = self.row_tokens.data_ptr(), self.col_tokens.data_ptr()
        self._rows_keepalive = (C.c_int * len(self.image_rows))(*[int(r) for r in self.image_rows])
        inp.image_rows = self._rows_keepalive
        inp.n_sets = len(self.sets)
        for i, (m, a, n, row) in enumerate(self.sets):
            src = text if m == "text" else readouts
            inp.sets[i].n, inp.sets[i].first_row = n, row
            if src is not None:
                inp.sets[i].rows = src.data_ptr() + a * cfg.channels * 2
                inp.sets[i].batch_stride = 0 if src.shape[0] == 1 else src.shape[1] * cfg.channels
            else:   # sizing only: a dense [B, n, C] layout
                inp.sets[i].batch_stride = (self.n_text if m == "text" else self.n_readouts) * cfg.channels
        return inp

    def workspace_bytes(self, pixel_dtype: torch.dtype = torch.uint8) -> int:
        """Bytes of tome_policy_predict's workspace: the assembled sequence plus the larger of the front end's and the
        forward-only stack's scratch."""
        n = int(self.lib.tome_policy_predict_workspace_bytes(C.byref(self.ccfg), C.byref(self._inputs(pixel_dtype))))
        if n == 0:
            L.check(L.TOME_ERR_INVALID)   # raises with the library's message
        return n

    def _call(self, frames, text, readouts, init, noise) -> None:
        io = L.StackIO(self.params.data_ptr(), self.params_bf16.data_ptr(), None, L.TOME_BF16,
                       None if self.gid is None else self.gid.data_ptr(), None if self.pos is None else self.pos.data_ptr(),
                       None if self.allow is None else self.allow.data_ptr(),
                       None if self.readout_idx is None else self.readout_idx.data_ptr(), None,
                       self.workspace.data_ptr(), self._ws_bytes, None,
                       None if self.readout is None else self.readout.data_ptr(), None, None, None,
                       None if self.head_out is None else self.head_out.data_ptr(), None, None, None,
                       None if self.layer_gid is None else self.layer_gid.data_ptr(),
                       None if self.layer_pos is None else self.layer_pos.data_ptr())
        smp = None
        if self.cfg.head == "diffusion":
            smp = L.DdpmSample(init.data_ptr(), noise.data_ptr(), int(noise.dim() == 3), self.coef.data_ptr(), 5.0)
        inp = self._inputs(frames.dtype, frames, text, readouts)
        L.check(self.lib.tome_policy_predict(C.byref(self.ccfg), C.byref(inp), C.byref(io), None if smp is None else C.byref(smp),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))

    # ------------------------------------------------------------------ public API
    def predict(self, frames: torch.Tensor, text: Optional[torch.Tensor], readouts: Optional[torch.Tensor] = None, rng=0,
                init=None, noise=None):
        """frames: u8 or f32 [B, N, H, W, C_in] pixels; text: bf16 [B or 1, n_text, C] embeddings of the grammar's text sets
        in order (None when it has none); readouts: bf16 [B or 1, n_readout, C] or [n_readout, C] readout embeddings, one set
        for every batch row when its batch is 1 (None: zeros, so the readout rows carry the stack's position embedding only).
        The front end runs in evaluation mode (the interval midpoints as position tokens).  Diffusion head: init [B, A] and
        noise [B, A] or [steps, B, A] default to draws from `rng` as ToMeStackEngine.predict draws them.
        Returns what ToMeStackEngine.predict returns: (actions [B, A] | logits [B, groups, bins] | sampled actions [B, A] |
        None, readout f32 [B, n_readout, C] | None), copies a later call does not overwrite."""
        cfg = self.cfg
        B, C_ = cfg.batch, cfg.channels
        H, W, Ci = self.tokenizer.image_size
        if not (frames.is_cuda and frames.dtype in (torch.uint8, torch.float32)
                and tuple(frames.shape) == (B, self.n_images, H, W, Ci)):
            raise ValueError(f"frames must be u8 / f32 CUDA [{B}, {self.n_images}, {H}, {W}, {Ci}], got {frames.dtype} {tuple(frames.shape)}")
        frames = frames.contiguous()
        text = self._rows_arg(text, self.n_text, "text")
        if readouts is None:
            readouts = self._zero_readouts
        readouts = self._rows_arg(readouts, self.n_readouts, "readouts")
        init_t = noise_t = None
        if cfg.head == "diffusion":
            from .attention_blocks._module import as_rng
            g = as_rng(rng)
            A = cfg.head_features
            if init is None:
                init = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32))
            if noise is None:
                noise = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32))
            init_t = torch.as_tensor(init).to(self.dev).float().contiguous()
            noise_t = torch.as_tensor(noise).to(self.dev).float().contiguous()
            if tuple(init_t.shape) != (B, A) or tuple(noise_t.shape) not in ((B, A), (cfg.diffusion_steps, B, A)):
                raise ValueError(f"init must be [{B}, {A}] and noise [{B}, {A}] or [{cfg.diffusion_steps}, {B}, {A}]")
        if not self.graph:
            self._draws = (init_t, noise_t)   # alive until the kernels that read them have run
            self._call(frames, text, readouts, init_t, noise_t)
            return self._outputs()
        args = (frames, text, readouts, init_t, noise_t)
        if self._graph is None:
            # first call: eager on static buffers (sets kernel attributes, loads modules), then capture the same call
            self._static = tuple(None if a is None else a.clone() for a in args)
            self._call(*self._static)
            out = self._outputs()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._call(*self._static)
            self._graph = g
            return out
        for dst, src in zip(self._static, args):
            if dst is None:
                continue
            if src is None or src.shape != dst.shape or src.dtype != dst.dtype:
                raise ValueError("a graph policy replays the shapes and dtypes of its first call: build another policy for others")
            dst.copy_(src)
        self._graph.replay()
        return self._outputs()

    def _rows_arg(self, t, n, what):
        cfg = self.cfg
        if n == 0:
            return None
        if t is None:
            raise ValueError(f"the grammar has {n} {what} tokens: pass {what} [B or 1, {n}, {cfg.channels}]")
        if t.dim() == 2:
            t = t.unsqueeze(0)
        if not (t.is_cuda and t.dtype == torch.bfloat16 and t.dim() == 3 and t.shape[0] in (1, cfg.batch)
                and tuple(t.shape[1:]) == (n, cfg.channels)):
            raise ValueError(f"{what} must be bf16 CUDA [{cfg.batch} or 1, {n}, {cfg.channels}], got {t.dtype} {tuple(t.shape)}")
        return t.contiguous()

    def _outputs(self):
        cfg = self.cfg
        out = None
        if self.head_out is not None:
            out = (self.head_out if cfg.head == "categorical" else self.head_out.view(cfg.batch, cfg.head_features)).clone()
        return out, None if self.readout is None else self.readout.clone()
