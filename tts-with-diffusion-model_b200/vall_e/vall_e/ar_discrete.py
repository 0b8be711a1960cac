"""Checkpoint-compatibility mode for the reference's own D3PM class (SURVEY.md §8f.2).

The reference's ``vall_e/vall_e/ar_discrete.py`` ``AR`` is a level-0 diffusion model with K = 1025
classes (absorbing class 512), 100 timesteps and a small DiT denoiser: d = 32, 8 blocks of
self-attention + cross-attention over two conditioning sequences (prompt codes, phones) + a FiLM
MLP, 16 heads (head_dim 2) through ``nn.MultiheadAttention``, and two 2-layer
``nn.TransformerEncoder`` conditioning encoders (``ar_discrete.py:98-161, 205-256``).  This module
keeps that class importable under the same path with the same constructor, sub-module names and
state-dict keys, so a module pickle or state dict trained with the reference loads, and samples it:

* the denoiser is far too small for tensor cores (head_dim 2, d = 32) — it runs as the same
  PyTorch modules the reference uses, on the GPU;
* the part of the reference that costs time, the reverse step (``p_sample`` :401-420 with two
  dense (W, 1025) x (1025, 1025) fp16 products per step over 630 MB of tables), runs on
  ``vb200_posterior_sample_from_logits`` (closed form, arbitrary K) through ``D3PMOps``.

The reference forward has batch-1 semantics baked in (``[0]`` indexing, one mask for the batch,
x_T built as one row; ``ar_discrete.py:696-712``); ``generate_audio`` therefore takes one
utterance, like the reference, and returns the same ``(448,)`` tensor.  Known reference quirks are
kept because trained weights depend on them: ``cross_attn`` is applied to both conditioning
sequences while ``cross_attn2`` is never used (:141-147), and the fixed window sizes 448 / 398 / 50.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F
from torch import Tensor, nn
from torch.nn import TransformerEncoder, TransformerEncoderLayer

from .base import MultiEmbedding
from .diffusion import D3PMOps

RESP_WINDOW, PROM_WINDOW, TEXT_WINDOW = 448, 398, 50      # ar_discrete.py:701-733


class Mlp(nn.Module):
    """Layout of ``timm.models.vision_transformer.Mlp`` (fc1, act, drop1, norm, fc2, drop2), which the
    reference instantiates (:16, :124, :227, :235); timm itself is not needed to load its weights."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.0):
        super().__init__()
        hidden_features = hidden_features or in_features
        out_features = out_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop)
        self.norm = nn.Identity()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop2 = nn.Dropout(drop)

    def forward(self, x):
        return self.drop2(self.fc2(self.norm(self.drop1(self.act(self.fc1(x))))))


class SinusodialEmbedding(nn.Module):
    """``ar_discrete.py:42-92``: frequencies held in fp16, [sin | cos] halves, added per position."""

    def __init__(self, d_model):
        super().__init__()
        half = d_model // 2
        omega = torch.exp(-math.log(1e4) * (torch.arange(half, dtype=torch.float16) / half))
        self.register_buffer("omega", omega, persistent=False)

    def add_pe(self, x: Tensor) -> Tensor:
        """x (t, c) -> (1, t, c): positions 0..t-1 along the FIRST axis, as the reference (:85-92)."""
        ang = self.omega[None, :] * torch.arange(x.shape[0], device=self.omega.device)[:, None]
        return x + torch.cat([ang.sin(), ang.cos()], dim=-1)[None]


class DiTBlock(nn.Module):
    """One denoiser block (``ar_discrete.py:98-147``): self-attention, cross-attention over the
    phones and over the prompt — both through ``cross_attn`` — and a FiLM-modulated MLP."""

    def __init__(self, hidden_size, num_heads, mlp_ratio=4.0):
        super().__init__()
        self.hidden_size = hidden_size
        self.norm1 = nn.LayerNorm(hidden_size, eps=1e-6)
        self.attn = nn.MultiheadAttention(hidden_size, num_heads=num_heads)
        self.norm2 = nn.LayerNorm(hidden_size, eps=1e-6)
        self.cross_attn = nn.MultiheadAttention(hidden_size, num_heads=num_heads)
        self.norm22 = nn.LayerNorm(hidden_size, eps=1e-6)
        self.cross_attn2 = nn.MultiheadAttention(hidden_size, num_heads=num_heads)   # weights only
        self.norm3 = nn.LayerNorm(hidden_size, eps=1e-6)
        self.mlp = Mlp(hidden_size, int(hidden_size * mlp_ratio), act_layer=nn.GELU, drop=0)
        self.timestep_fc = nn.Linear(hidden_size, hidden_size * 2)

    def forward(self, x, speaker_emb, text_phonemes, timestep_emb, mask):
        keep = mask[None, :, None]
        h = (x * keep).transpose(0, 1)                       # (t, 1, c): MultiheadAttention is sequence-first
        n = self.norm1(h)
        h = h + self.attn(n, n, n)[0]
        phones, spk = text_phonemes.transpose(0, 1), speaker_emb.transpose(0, 1)
        h = h + self.cross_attn(self.norm2(h), phones, phones)[0] + self.cross_attn(self.norm22(h), spk, spk)[0]
        scale, shift = self.timestep_fc(timestep_emb).split(self.hidden_size, dim=-1)
        h = h + self.mlp(self.norm3(h) * (1 + scale[None]) + shift[None])
        return h.transpose(0, 1) * keep


class AR(D3PMOps, nn.Module):
    """Drop-in for ``vall_e.vall_e.ar_discrete.AR``: same constructor signature (all sizes are
    fixed by the reference: d = 32, 8 blocks, 16 heads, 100 timesteps, K = 1025) and state dict."""

    n_resp_levels = 1
    casual = True
    use_stop_token = True
    norm_type = "ln"
    resp_loss_only = False
    transition = "absorbing"

    def __init__(self, d_model=32, n_steps=100, n_tokens=1025, max_n_levels=8, n_heads=16, num_layers=8):
        super().__init__()
        d = 32                                               # the reference overrides its argument (:208)
        self.timesteps = 100
        self.num_classes = 1025
        self.eps = 1.0e-6
        self.text_emb = nn.Embedding(1025, d, padding_idx=0)
        self.proms_emb = MultiEmbedding(max_n_levels, 1025, d)
        self.resps_emb = nn.Embedding(1025, d, padding_idx=0)
        self.time_emb = nn.Embedding(self.timesteps + 1, d)
        self.encodertext = nn.Sequential(TransformerEncoder(TransformerEncoderLayer(d_model=d, nhead=16), num_layers=2,
                                                            enable_nested_tensor=False),
                                         Mlp(d, d * 2, d, act_layer=nn.SiLU, drop=0.01))
        self.encoder2 = nn.Sequential(TransformerEncoder(TransformerEncoderLayer(d_model=d, nhead=16), num_layers=2,
                                                            enable_nested_tensor=False),
                                      Mlp(d, d * 3, d, act_layer=nn.SiLU, drop=0.01))
        self.sin_emb = SinusodialEmbedding(d)
        self.sin_emb2 = SinusodialEmbedding(d)
        self.token_emb = nn.Embedding(num_embeddings=1025, embedding_dim=d)
        self.blocks = nn.ModuleList([DiTBlock(d, 16, mlp_ratio=4.0) for _ in range(8)])
        self.final = nn.Linear(d, 1025)

    # ------------------------------------------------------------------ conditioning (computed once, :735-746)
    @staticmethod
    def _window(x: Tensor, n: int) -> Tensor:
        """zero-pad or cut the first axis to n (ar_discrete.py:703-733)."""
        return x[:n] if x.shape[0] >= n else F.pad(x, (0, 0) * (x.dim() - 1) + (0, n - x.shape[0]))

    def conditioning(self, text: Tensor, proms: Tensor):
        """text (t,) phone ids, proms (t', l) prompt codes -> (cond1 (1, 398, d), cond2 (1, 50, d))."""
        text, proms = self._window(text, TEXT_WINDOW), self._window(proms, PROM_WINDOW)
        w = self.proms_emb.weight                             # (max_n_levels, 1025, d): sum over the given levels
        prom_rows = sum(w[l][proms[:, l]] for l in range(proms.shape[1]))
        cond1 = self.encoder2(self.sin_emb.add_pe(prom_rows)[0])[None]
        cond2 = self.encodertext(self.sin_emb.add_pe(self.text_emb(text)[None])[0])[None]   # 3-D input: position 0 for every row (:739-741)
        return cond1, cond2

    def denoise_logits(self, x_t: Tensor, t: Tensor, cond1: Tensor, cond2: Tensor, mask: Tensor) -> Tensor:
        """x_t (1, 448) ints, t (1,) -> logits of p(x_0 | x_t) (1, 448, 1025) (ar_discrete.py:751-776)."""
        t_emb = self.time_emb(t)
        x = self.resps_emb(x_t)[0][None]
        for block in self.blocks:
            x = block(x, cond1, cond2, t_emb, mask)
        return self.final(x * mask[:, None])

    # ------------------------------------------------------------------ reverse loop (:696-780)
    @torch.no_grad()
    def generate_audio(self, text_list, proms_list, resps_list=None, *, seed: int | None = None,
                       greedy: bool = False, noise_fn=None, temperature: float = 1.0) -> Tensor:
        """x_T = 350 frames of the absorbing class in a 448 window, t = 99 .. 1, returns the (448,)
        level-0 codes like the reference.  Noise: ``torch.rand`` uniforms on the CPU generator as the
        reference (default), ``noise_fn(t) -> (1, 448, 1025)`` supplied uniforms, in-kernel Philox when
        ``seed`` is given, or none (``greedy``).  ``temperature``: p̂(x0) = softmax(logits / temperature) in every
        reverse step (``D3PMOps.p_sample``); ValueError unless it is a finite number > 0."""
        temperature = self._temperature(temperature)
        if len(text_list) != 1 or len(proms_list) != 1:
            raise ValueError("the reference's D3PM sampler handles one utterance per call (ar_discrete.py:699-712)")
        dev = self.final.weight.device
        x = torch.zeros(1, RESP_WINDOW, dtype=torch.int32, device=dev)
        x[:, :350] = self.mask_id
        mask = x[0] != 0
        cond1, cond2 = self.conditioning(text_list[0].to(dev), proms_list[0].to(dev))
        for step in range(self.timesteps - 1, 0, -1):
            t = torch.full((1,), step, dtype=torch.long, device=dev)
            logits = self.denoise_logits(x, t, cond1, cond2, mask)
            noise = noise_fn(step) if noise_fn is not None else None
            x, _ = self.p_sample(logits, t, x, noise=noise, greedy=greedy, seed=seed, temperature=temperature)
            x = x.to(torch.int32)
        return x.squeeze().long()
