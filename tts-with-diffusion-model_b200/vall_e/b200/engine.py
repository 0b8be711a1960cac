"""Denoiser engine: packs a reference-layout state dict for the sm_100a kernels and runs the
denoiser forward (``base.py:403-443``) and the D3PM reverse loop (``ar_discrete.py:696-780``)
as a fixed sequence of libvalle_b200 launches on torch's current CUDA stream.

HBM layout
  * weights: bf16, nn.Linear layout (N, K) == K-major operands for tcgen05; biases / AdaLN tables
    fp32 (AdaLN table stores exp(log gamma) | beta so the kernel has no transcendental);
  * activations: utterances packed back to back, M = sum_b T_b rows, no padding rows, so the
    reference's mask multiplies (base.py:131,193-194,440) have nothing left to zero;
  * residual stream fp32 (M, d); GEMM inputs bf16; logits fp16 (M_resp, n_out).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field

import numpy as np
import torch

from . import lib as L


def sinusoidal_table(n: int, d_model: int) -> torch.Tensor:
    """pe[p] = [sin(p w_i) || cos(p w_i)], w_i = exp(-ln(1e4) i / (d/2)) — computed with the same
    torch ops as the reference (base.py:38-89) so the table is bit-identical to its add_pe."""
    d_half = d_model // 2
    omega = torch.exp(-math.log(1e4) * (torch.arange(d_half, dtype=torch.float32) / d_half))
    ang = omega[None, :] * torch.arange(n)[:, None]
    return torch.cat([ang.sin(), ang.cos()], dim=-1).contiguous()


# 16-bit format of the GEMM operands whose range is safe in fp16 — the normalised rows (h), the FFN hidden (ff),
# the classifier input (head), each with the weights it meets (tcgen05 takes both operands in ONE format): 11
# significand bits against bf16's 8.  Measured on the full model (DESIGN.md §2), logits max-abs error against the
# fp32 reference / reverse-loop time on one box:  none 2.2e-2 (over the 2e-2 bar) / 1302 ms;  head 1.4e-2 / 1306;
# head,ff 1.2e-2 / 1319;  head,h 1.1e-2 / 1331;  all 7.6e-3 / 1343 — fp16 MMAs cost power, and the step is
# power-capped, so each GEMM moved to fp16 is paid for in clocks.  Default: the classifier input alone (the
# largest single error source, 3 % of the FLOPs).  VB200_ACT picks another set: "f16" = all three, "bf16" = none,
# or a comma list such as "head,ff".  qkv, the attention output and the to_out weights are always bf16.
def _act_dtypes():
    v = os.environ.get("VB200_ACT", "head")
    on = {"h", "ff", "head"} if v == "f16" else (set() if v == "bf16" else {x.strip() for x in v.split(",")})
    if not on <= {"h", "ff", "head"}:
        raise ValueError(f"VB200_ACT={v!r}: expected f16, bf16 or a comma list of h, ff, head")
    return {k: (torch.float16 if k in on else torch.bfloat16) for k in ("h", "ff", "head")}


ACT = _act_dtypes()


class PackedWeights:
    """Device-resident weights in kernel layout, built from a state dict with base.py's keys."""

    def __init__(self, sd: dict, n_heads: int, n_layers: int, norm_type: str, device, max_rows: int = 4096):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise L.VB200Error("PackedWeights needs a CUDA device (no CPU fallback)")
        bf = lambda t: t.detach().to(dev, torch.bfloat16).contiguous()
        as_ = lambda t, k: t.detach().to(dev, ACT[k]).contiguous()      # weights in the format of the rows they meet
        f32 = lambda t: t.detach().to(dev, torch.float32).contiguous()
        self.device = dev
        self.n_heads, self.n_layers, self.norm_type = n_heads, n_layers, norm_type
        self.d = int(sd["sep"].shape[0])
        if self.d % n_heads or self.d // n_heads != 64:
            raise L.VB200Error(f"head_dim must be 64 (d_model={self.d}, n_heads={n_heads})")
        self.text_w = bf(sd["text_emb.weight"])
        self.prom_w = bf(sd["proms_emb.weight"])
        self.resp_w = bf(sd["resps_emb.weight"])
        self.K = int(self.prom_w.shape[1])
        if int(self.resp_w.shape[1]) != self.K:
            # Kernels index both tables with one class count; AR-style stop tokens are out of scope.
            raise L.VB200Error("resps_emb and proms_emb must have the same number of classes")
        self.sep = bf(sd["sep"])
        self.time_w = bf(sd["time_emb.weight"]) if "time_emb.weight" in sd else None
        self.layers = []
        for i in range(n_layers):
            p = f"blocks.{i}"
            ly = dict(
                w_qkv=as_(sd[f"{p}.attn.block.to_qkv.weight"], "h"),
                w_out=bf(sd[f"{p}.attn.block.to_out.weight"]),
                b_out=f32(sd[f"{p}.attn.block.to_out.bias"]),
                w_ff1=as_(sd[f"{p}.ffn.block.0.weight"], "h"), b_ff1=f32(sd[f"{p}.ffn.block.0.bias"]),
                w_ff2=as_(sd[f"{p}.ffn.block.3.weight"], "ff"), b_ff2=f32(sd[f"{p}.ffn.block.3.bias"]),
            )
            for which in ("attn", "ffn"):
                if norm_type == "adaln":
                    emb = sd[f"{p}.{which}.norm.emb.weight"].detach().float()
                    logg, beta = emb.chunk(2, dim=-1)
                    ly[f"norm_{which}"] = f32(torch.cat([logg.exp(), beta], dim=-1))
                else:
                    ly[f"norm_{which}"] = (f32(sd[f"{p}.{which}.norm.weight"]), f32(sd[f"{p}.{which}.norm.bias"]))
            self.layers.append(ly)
        self.w_cls = as_(sd["classifier.weight"], "head")
        self.b_cls = f32(sd["classifier.bias"])
        self.n_out = int(self.w_cls.shape[0])
        self._pe, self._pe_retired = None, []
        self.ensure_pe(max_rows)

    def ensure_pe(self, n: int) -> torch.Tensor:
        """Positional table with at least ``n`` rows.  A table that has been handed out is never freed:
        CUDA graphs captured by cached Sessions keep its address, and the caching allocator would hand
        the block to someone else."""
        if self._pe is None or self._pe.shape[0] < n:
            if self._pe is not None:
                self._pe_retired.append(self._pe)
            self._pe = sinusoidal_table(max(n, 1), self.d).to(self.device)
        return self._pe


def check_ids(ids: torch.Tensor, n: int, what: str, lo: int = 0) -> None:
    """Token ids index embedding tables and logits rows with no bounds check in the kernels; the
    reference raises IndexError for an id outside its table (F.one_hot / nn.Embedding), so does this.
    Host tensors are checked on the host; device tensors cost one synchronising reduction per batch
    (never per denoise step).  VB200_CHECK_IDS=0 skips it."""
    if ids.numel() == 0 or os.environ.get("VB200_CHECK_IDS", "1")[:1] == "0":
        return
    mn, mx = torch.aminmax(ids)
    mn, mx = int(mn), int(mx)
    if mn < lo or mx >= n:
        raise IndexError(f"{what}: ids must lie in [{lo}, {n}), got [{mn}, {mx}]")


class BatchLayout:
    """Packed-row layout of one batch of utterances (host-built once, constant across steps)."""

    def __init__(self, text_list, proms_list, resp_lens, device, gids=None, n_text: int | None = None,
                 n_codes: int | None = None):
        dev = torch.device(device)
        B = len(text_list)
        if B == 0:
            raise ValueError("empty batch")
        if not (len(proms_list) == B and len(resp_lens) == B):
            raise ValueError("text_list, proms_list and resps must have the same length")
        t_txt = [int(t.shape[0]) for t in text_list]
        t_prom = [int(p.shape[0]) for p in proms_list]
        t_resp = [int(r) for r in resp_lens]
        for p in proms_list:
            if p.dim() != 2 or p.shape[1] != 8:
                raise ValueError(f"prompts must be (t, 8) code grids, got {tuple(p.shape)}")
        rows = [a + 1 + b + 1 + c for a, b, c in zip(t_txt, t_prom, t_resp)]
        cu = np.zeros(B + 1, dtype=np.int64)
        cu[1:] = np.cumsum(rows)
        if cu[-1] >= 2 ** 31:
            raise ValueError("batch too large for int32 row indices")
        self.B, self.M, self.max_T = B, int(cu[-1]), int(max(rows))
        self.t_txt, self.t_prom, self.t_resp, self.rows = t_txt, t_prom, t_resp, rows
        self.M_resp = int(sum(t_resp))
        utt = np.zeros((B, L.U_STRIDE), dtype=np.int32)
        utt[:, L.U_ROW0] = cu[:-1]
        utt[:, L.U_TTXT], utt[:, L.U_TPROM], utt[:, L.U_TRESP] = t_txt, t_prom, t_resp
        utt[:, L.U_TXT0] = np.concatenate([[0], np.cumsum(t_txt)[:-1]])
        utt[:, L.U_PROM0] = np.concatenate([[0], np.cumsum(t_prom)[:-1]])
        resp0 = np.concatenate([[0], np.cumsum(t_resp)[:-1]])
        utt[:, L.U_RESP0] = resp0
        utt[:, L.U_GID] = np.arange(B) if gids is None else np.asarray(gids)
        row_utt = np.repeat(np.arange(B, dtype=np.int32), rows)
        resp_row_utt = np.repeat(np.arange(B, dtype=np.int32), t_resp)
        resp_row_index = np.concatenate(
            [np.arange(cu[b + 1] - t_resp[b], cu[b + 1], dtype=np.int32) for b in range(B)]
        ) if self.M_resp else np.zeros(0, dtype=np.int32)
        self.resp_offsets = resp0.tolist()

        def up(a):
            return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().to(dev, non_blocking=True)

        self.utt, self.row_utt, self.cu_rows = up(utt), up(row_utt), up(cu.astype(np.int32))
        self.resp_row_utt, self.resp_row_index = up(resp_row_utt), up(resp_row_index)
        text = torch.cat([t.reshape(-1) for t in text_list]).to(torch.int32)
        proms = torch.cat([p.reshape(-1, 8) for p in proms_list]).to(torch.int32)
        self.n_text, self.n_codes = n_text, n_codes
        if n_text is not None:
            check_ids(text, n_text, "text_list")
        if n_codes is not None:
            check_ids(proms, n_codes, "proms_list")
        self.text_ids = text.contiguous().to(dev, non_blocking=True)
        self.prom_ids = proms.contiguous().to(dev, non_blocking=True)
        self.h2d_bytes = int(utt.nbytes + row_utt.nbytes + (B + 1) * 4 + resp_row_utt.nbytes +
                             resp_row_index.nbytes + text.numel() * 4 + proms.numel() * 4)
        self.device = dev

    def split_resp(self, packed: torch.Tensor):
        """(M_resp, ...) packed response rows -> list of per-utterance tensors."""
        return list(packed.split(self.t_resp, dim=0))


@dataclass
class Workspace:
    x: torch.Tensor
    h: torch.Tensor
    qkv: torch.Tensor
    att: torch.Tensor
    ff: torch.Tensor
    head_in: torch.Tensor
    logits: torch.Tensor
    extra: dict = field(default_factory=dict)


class DenoiserEngine:
    """Runs the packed denoiser forward and the reverse loop for one PackedWeights."""

    def __init__(self, weights: PackedWeights, logits_dtype=torch.float16, attn_variant="tmem", simt=False):
        self.w = weights
        self.logits_dtype = logits_dtype
        self.attn_variant = attn_variant
        self.simt = simt      # validation only: route GEMM/attention through the CUDA-core kernels
        self.launches = 0     # kernels launched by this engine (bench.py reports it)
        self.profile = None   # bench.py: list collecting (kind, flops, start_event, end_event) per GEMM/attention launch

    # ------------------------------------------------------------------ buffers
    def workspace(self, lay: BatchLayout, logits_dtype=None) -> Workspace:
        w, dev = self.w, self.w.device
        d, M, Mr = w.d, lay.M, lay.M_resp
        e = lambda *s, dt: torch.empty(*s, dtype=dt, device=dev)
        w.ensure_pe(lay.max_T)
        # one allocation, carved up the way the C ABI sizes it (vb200_workspace_bytes)
        ldt = logits_dtype or self.logits_dtype
        total, sizes = L.workspace_bytes(M, Mr, d, w.n_out, ldt)
        flat = e(max(total, 1), dt=torch.uint8)
        shapes = {"x": ((M, d), torch.float32), "h": ((M, d), ACT["h"]), "qkv": ((M, 3 * d), torch.bfloat16),
                  "att": ((M, d), torch.bfloat16), "ff": ((M, 4 * d), ACT["ff"]),
                  "head_in": ((Mr, d), ACT["head"]), "logits": ((Mr, w.n_out), ldt)}
        views, off = {}, 0
        for name, size in zip(L.WS_FIELDS, sizes):
            shape, dt = shapes[name]
            n = shape[0] * shape[1] * torch.empty((), dtype=dt).element_size()
            views[name] = flat[off:off + n].view(dt).view(shape)
            off += size
        return Workspace(extra={"flat": flat}, **views)

    # ------------------------------------------------------------------ one denoiser forward
    def forward(self, lay: BatchLayout, ws: Workspace, resp_ids: torch.Tensor, level_utt: torch.Tensor,
                use_time: bool, hidden_out: list | None = None, head: bool = True) -> torch.Tensor:
        """resp_ids int32 (M_resp, levels_in); level_utt int32 (B) = AdaLN row (and time_emb row when
        use_time).  Returns ws.logits (M_resp, n_out): classifier(x) on the response rows."""
        with torch.cuda.device(self.w.device):      # launches go to the CURRENT device's stream (lib.stream)
            return self._forward(lay, ws, resp_ids, level_utt, use_time, hidden_out, head)

    def _forward(self, lay, ws, resp_ids, level_utt, use_time, hidden_out, head):
        w = self.w
        sv = self.simt
        levels_in = int(resp_ids.shape[1])
        L.embed_gather(ws.x, w.text_w, w.prom_w, w.resp_w, w.sep, w.time_w if use_time else None,
                       w.ensure_pe(lay.max_T), lay.text_ids, lay.prom_ids, resp_ids, lay.utt, lay.row_utt,
                       level_utt, w.K, levels_in)
        scale = 64 ** -0.5
        gemm, attn_flops = self._gemm, sum(4 * T * T * w.d for T in lay.rows)
        for ly in w.layers:
            self._norm(ws.h, ws.x, ly["norm_attn"], level_utt, lay)
            gemm(ws.qkv, ws.h, ly["w_qkv"], epi=L.EPI_NONE)
            ev = self._prof_begin()
            L.flash_attn_varlen(ws.att, ws.qkv, lay.cu_rows, lay.max_T, w.n_heads, scale,
                                variant="simt" if sv else self.attn_variant)
            self._prof_end(ev, "attn", attn_flops)
            gemm(ws.x, ws.att, ly["w_out"], ly["b_out"], residual=ws.x, epi=L.EPI_BIAS_RESIDUAL)
            self._norm(ws.h, ws.x, ly["norm_ffn"], level_utt, lay)
            gemm(ws.ff, ws.h, ly["w_ff1"], ly["b_ff1"], epi=L.EPI_BIAS_GELU)
            gemm(ws.x, ws.ff, ly["w_ff2"], ly["b_ff2"], residual=ws.x, epi=L.EPI_BIAS_RESIDUAL)
            if hidden_out is not None:
                hidden_out.append(ws.x.clone())
        L.gather_rows_bf16(ws.head_in, ws.x, lay.resp_row_index)
        self.launches += 1 + 7 * len(w.layers) + 1
        if not head:              # the caller runs classifier + reverse step as one C call
            return ws.head_in
        gemm(ws.logits, ws.head_in, w.w_cls, w.b_cls, epi=L.EPI_BIAS)
        self.launches += 1
        return ws.logits

    def _gemm(self, out, A, W, bias=None, residual=None, epi=L.EPI_NONE):
        ev = self._prof_begin()
        L.gemm_bf16(out, A, W, bias, residual=residual, epi=epi, simt=self.simt)
        self._prof_end(ev, "gemm", 2 * A.shape[0] * A.shape[1] * W.shape[0])

    def _prof_begin(self):
        if self.profile is None:
            return None
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        return ev

    def _prof_end(self, ev, kind, flops):
        if ev is None:
            return
        end = torch.cuda.Event(enable_timing=True)
        end.record()
        self.profile.append((kind, flops, ev, end))

    def _norm(self, out, x, params, level_utt, lay):
        ev = self._prof_begin()
        if self.w.norm_type == "adaln":
            L.adaln(out, x, params, level_utt, lay.row_utt)
        else:
            L.layernorm(out, x, params[0], params[1])
        self._prof_end(ev, "norm", x.numel() * 6)      # bytes: fp32 in, bf16 out

    # ------------------------------------------------------------------ reverse loop
    def session(self, lay: BatchLayout) -> "Session":
        return Session(self, lay)

    def reverse_loop(self, lay: BatchLayout, ws: Workspace, x_t: torch.Tensor, table: torch.Tensor,
                     timesteps: int, transition: int, noise: int = L.NOISE_PHILOX, seed: int = 0,
                     uniforms_fn=None, use_graph: bool = True, n_levels: int = 8, trace: list | None = None,
                     schedule=None, next_t: torch.Tensor | None = None, known: torch.Tensor | None = None,
                     temperature: float = 1.0):
        """One-shot form (tests): x_T -> x_0 in place on x_t int32 (M_resp, n_levels)."""
        ses = Session(self, lay, ws=ws, x_t=x_t)
        ses.run(table, timesteps, transition, noise=noise, seed=seed, uniforms_fn=uniforms_fn,
                use_graph=use_graph, n_levels=n_levels, trace=trace, schedule=schedule, next_t=next_t, known=known,
                temperature=temperature)
        return x_t


def successor_tensor(timesteps: int, schedule, device) -> torch.Tensor:
    """int32 (S,) next_t of ``schedule`` on ``device`` for ``vb200_step_timesteps_to``."""
    from ..vall_e import d3pm
    return torch.tensor(d3pm.successors(timesteps, schedule), dtype=torch.int32).to(device)


class Session:
    """Persistent device state for batches of one shape signature: layout arrays, workspace, x_t,
    the per-utterance timestep vector and (after the first run) a CUDA graph of one denoise step.
    A new batch with the same per-utterance lengths is ``load``-ed into the same buffers, so the
    captured graph is replayed unchanged."""

    def __init__(self, engine: DenoiserEngine, lay: BatchLayout, ws: Workspace | None = None,
                 x_t: torch.Tensor | None = None, n_levels: int = 8):
        self.eng, self.lay = engine, lay
        dev = engine.w.device
        self.ws = ws if ws is not None else engine.workspace(lay)
        self.x_t = x_t if x_t is not None else torch.empty(lay.M_resp, n_levels, dtype=torch.int32, device=dev)
        self.t_utt = torch.zeros(lay.B, dtype=torch.int32, device=dev)
        self.graph = None
        self.graph_key = None
        self.per_step_launches = 0
        self._next_t = {}
        self._known = None

    def known_buffer(self) -> torch.Tensor:
        """The session's int32 (M_resp, n_levels) buffer of given codes (-1 = generate), allocated on first use.
        Callers fill it per call; its address stays, so a captured step graph that reads it replays."""
        if self._known is None:
            self._known = torch.empty_like(self.x_t)
        return self._known

    def signature(self):
        return (tuple(self.lay.t_txt), tuple(self.lay.t_prom), tuple(self.lay.t_resp))

    def load(self, text_list, proms_list, gids=None) -> int:
        """Copies a new same-shape batch (host or device tensors) into the session's buffers.
        Returns the bytes moved host->device."""
        lay = self.lay
        if [len(t) for t in text_list] != lay.t_txt or [len(p) for p in proms_list] != lay.t_prom:
            raise ValueError("batch shape does not match this session")
        text = torch.cat([t.reshape(-1) for t in text_list]).to(torch.int32)
        proms = torch.cat([p.reshape(-1, 8) for p in proms_list]).to(torch.int32)
        if lay.n_text is not None:
            check_ids(text, lay.n_text, "text_list")
        if lay.n_codes is not None:
            check_ids(proms, lay.n_codes, "proms_list")
        lay.text_ids.copy_(text, non_blocking=True)
        lay.prom_ids.copy_(proms, non_blocking=True)
        moved = (text.numel() + proms.numel()) * 4
        if gids is not None:
            g = torch.as_tensor(gids, dtype=torch.int32)
            lay.utt[:, L.U_GID].copy_(g, non_blocking=True)
            moved += g.numel() * 4
        return moved

    def run(self, table: torch.Tensor, timesteps: int, transition: int, noise: int = L.NOISE_PHILOX,
            seed: int = 0, uniforms_fn=None, use_graph: bool = True, n_levels: int = 8,
            trace: list | None = None, schedule=None, next_t: torch.Tensor | None = None,
            known: torch.Tensor | None = None, temperature: float = 1.0) -> torch.Tensor:
        """for t in schedule (default S-1 .. 1; never t = 0, as the reference, ar_discrete.py:750):
        logits = denoiser(x_t, t); x_{sigma(t)} = p_sample(logits, t, x_t), in place on self.x_t, where
        sigma(t) is the next timestep of the schedule (0 after the last).  ``table`` must be the schedule's
        (``d3pm.schedule_table``; ``d3pm.scalar_table`` for the default) and ``next_t`` its int32 (S,)
        successor vector on the device (``successor_tensor``; built here when omitted).
        uniforms_fn(t) -> float32 (M_resp*n_levels, K) supplies the reference's torch.rand (parity).
        ``known``: int32 (M_resp, n_levels) device tensor (``known_buffer``) or None.  A token with known[r, l] = k
        >= 0 draws every step from q(x_s | x_t, x0 = k) and is set to k once after the last step; -1 draws as
        usual (vb200_head_posterior_sample_known).  ``temperature``: every step draws with p̂(x0) =
        softmax(logits / temperature) (vb200_head_posterior_sample_temp; 1.0 is the unscaled step bit for bit)."""
        from ..vall_e import d3pm
        if schedule is None:
            schedule = range(timesteps - 1, 0, -1)
        schedule = d3pm.check_schedule(timesteps, schedule)
        if next_t is None:
            next_t = self._next_t.get(schedule)
            if next_t is None:
                next_t = self._next_t[schedule] = successor_tensor(timesteps, schedule, self.eng.w.device)
        elif next_t.numel() != timesteps:
            raise ValueError(f"next_t has {next_t.numel()} entries, the table {timesteps} timesteps")
        with torch.cuda.device(self.eng.w.device):
            self._run(table, schedule, next_t, transition, noise, seed, uniforms_fn, use_graph, n_levels, trace,
                      known, float(temperature))
            if known is not None:      # the given codes come back exactly: once per generation, not per step
                self.x_t.copy_(torch.where(known >= 0, known, self.x_t))
            return self.x_t

    def _run(self, table, schedule, next_t, transition, noise, seed, uniforms_fn, use_graph, n_levels, trace, known,
             temperature):
        eng, lay, ws, x_t, t_utt = self.eng, self.lay, self.ws, self.x_t, self.t_utt
        w, dev = eng.w, eng.w.device
        K = w.n_out // n_levels
        t_utt.fill_(schedule[0])

        def one_step(uniforms=None):
            if eng.profile is None and not eng.simt:
                head_in = eng._forward(lay, ws, x_t, t_utt, True, None, False)
                L.head_posterior_sample(x_t, ws.logits, head_in, w.w_cls, w.b_cls, x_t, lay.resp_row_utt, t_utt,
                                        lay.utt, table, n_levels, K, transition, noise, uniforms, seed, known,
                                        temperature)
                eng.launches += 0 if L.head_fused(w.d, K, noise) else 1   # the `+= 2` below counts one of them
            else:                 # per-launch timing hooks / CUDA-core validation path: separate calls
                logits = eng._forward(lay, ws, x_t, t_utt, True, None, True)
                L.posterior_sample_from_logits(x_t, None, logits, w.n_out, x_t, lay.resp_row_utt, t_utt, lay.utt,
                                               table, lay.M_resp, n_levels, K, transition, noise, uniforms, seed,
                                               known, temperature)
            L.step_timesteps_to(t_utt, next_t)
            eng.launches += 2

        n_steps = len(schedule)
        graph_ok = (use_graph and noise != L.NOISE_UNIFORMS and trace is None and n_steps > 2
                    and eng.profile is None)
        if not graph_ok:
            for t in schedule:
                one_step(uniforms_fn(t) if noise == L.NOISE_UNIFORMS else None)
                if trace is not None:
                    trace.append(x_t.clone())
            return x_t
        # the temperature is a kernel argument baked into the captured step: a new one needs a new capture
        key = (table.data_ptr(), next_t.data_ptr(), transition, noise, seed, n_levels,
               known.data_ptr() if known is not None else None, temperature)
        first = 0
        if self.graph is None or self.graph_key != key:
            # First step eagerly (also warms tensor-map caches and function attributes), then capture
            # one step: the timestep lives in device memory, so the graph is step-invariant.
            one_step()
            first = 1
            g = torch.cuda.CUDAGraph()
            cap_stream = torch.cuda.Stream(device=dev)
            cap_stream.wait_stream(torch.cuda.current_stream(dev))
            before = eng.launches
            with torch.cuda.stream(cap_stream):
                with torch.cuda.graph(g, stream=cap_stream):
                    one_step()
            self.per_step_launches = eng.launches - before
            eng.launches = before
            torch.cuda.current_stream(dev).wait_stream(cap_stream)
            self.graph, self.graph_key = g, key
        for _ in range(n_steps - first):
            self.graph.replay()
            eng.launches += self.per_step_launches
        return x_t
