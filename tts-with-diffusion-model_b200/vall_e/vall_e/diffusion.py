"""D3PM denoising sampler: the glue class of SURVEY.md §7.1.

Denoiser  = the reference's non-causal AdaLN transformer (``base.py``) at the factory sizes, fed
            ``text + sep + prompt(8 levels) + sep + x_t(8 levels)``, with the AdaLN "level" slot
            (base.py:140,146) indexed by the timestep and ``time_emb`` (name from
            ar_discrete.py:213) added to the x_t rows; ``classifier`` carries 8 K-way heads.
Sampler   = the D3PM algebra of ``ar_discrete.py``: cosine schedule (:286-304), absorbing (:315-334)
            or uniform (:308-313) transitions, ``q_sample`` (:467-487), ``q_posterior_logits`` +
            ``p_sample`` (:347-375, :401-420) and the reverse loop of ``generate_audio`` (:696-780),
            with the dense (K, K) fp16 tables replaced by per-timestep scalars (``d3pm.py``).
Method names, argument order and tensor shapes follow the reference so parity tests read like it.
"""
from __future__ import annotations

import math
import numbers

import torch
import torch.nn.functional as F
from torch import Tensor, nn

from ..b200 import lib as L
from ..b200.engine import BatchLayout, check_ids, successor_tensor
from . import d3pm
from .base import Base

_TRANSITIONS = {"absorbing": L.ABSORBING, "uniform": L.UNIFORM}


class D3PMOps:
    """The D3PM algebra of ``ar_discrete.py`` on the B200 kernels, for any module that defines
    ``num_classes``, ``timesteps`` and ``transition``: schedule / table access, ``q_sample``,
    ``q_posterior_logits`` and ``p_sample`` with the reference's signatures and shapes."""

    # ------------------------------------------------------------------ D3PM constants
    @property
    def mask_id(self) -> int:
        """absorbing class = K // 2, an ordinary codec token (ar_discrete.py:332,699)."""
        return self.num_classes // 2

    @property
    def betas(self) -> Tensor:
        return d3pm.betas_fp16(self.timesteps)

    def _table(self, device) -> Tensor:
        cache = self.__dict__.setdefault("_tables", {})
        key = (str(device), self.timesteps, self.num_classes, self.transition)
        if key not in cache:
            cache[key] = d3pm.scalar_table(self.timesteps, self.num_classes, self.transition).to(device)
        return cache[key]

    def _sample_steps(self, sample_steps) -> int:
        """The number of denoise steps: ``sample_steps`` (None: S-1, every timestep), or ValueError for
        anything but an integer in [1, S-1]."""
        S = self.timesteps
        n = S - 1 if sample_steps is None else sample_steps
        if isinstance(n, bool) or not isinstance(n, numbers.Integral) or not 1 <= n <= S - 1:
            raise ValueError(f"sample_steps must be an integer in [1, {S - 1}] for a model with {S} timesteps, "
                             f"got {sample_steps!r}")
        return int(n)

    @staticmethod
    def _temperature(temperature) -> float:
        """``temperature`` as a float, or ValueError for anything but a finite real number > 0 (bool refused)."""
        ok = isinstance(temperature, numbers.Real) and not isinstance(temperature, bool)
        if not ok or not math.isfinite(float(temperature)) or not float(temperature) > 0:
            raise ValueError(f"temperature must be a finite number > 0, got {temperature!r}")
        return float(temperature)

    def _sampling(self, device, n: int) -> tuple:
        """(schedule, its table, its int32 (S,) successor vector) of a reverse loop of n denoise steps."""
        cache = self.__dict__.setdefault("_tables", {})
        key = ("schedule", str(device), self.timesteps, self.num_classes, self.transition, n)
        if key not in cache:
            sch = d3pm.sample_schedule(self.timesteps, n)
            cache[key] = (sch, d3pm.schedule_table(self.timesteps, self.num_classes, self.transition, sch).to(device),
                          successor_tensor(self.timesteps, sch, device))
        return cache[key]

    def _dense_log_qbar(self, device) -> Tensor:
        cache = self.__dict__.setdefault("_tables", {})
        key = ("dense", str(device), self.timesteps, self.num_classes, self.transition)
        if key not in cache:
            cache[key] = d3pm.dense_log_qbar(self.timesteps, self.num_classes, self.transition).to(device)
        return cache[key]

    def __getstate__(self):
        state = super().__getstate__()
        state.pop("_tables", None)
        return state

    # ------------------------------------------------------------------ forward noising (row Q)
    def q_sample(self, x_start: Tensor, t: Tensor, mask: Tensor, noise: Tensor | None = None) -> Tensor:
        """x_start (B, W) ints, t (B,), mask (W,) or (B, W); noise: U[0,1) (B, W, K) float32 — drawn
        with torch.rand on the CPU generator like the reference (ar_discrete.py:480) when omitted."""
        B, W = x_start.shape
        K = self.num_classes
        dev = x_start.device
        if noise is None:
            noise = torch.rand(size=x_start.shape + (K,)).to(dev)
        x0 = x_start.to(torch.int32).contiguous().view(-1)
        check_ids(x0, K, "q_sample: x_start")
        t_tok = t.to(dev, torch.int32).view(B, 1).expand(B, W).contiguous().view(-1)
        m = mask.to(dev, torch.int32).expand(B, W).contiguous().view(-1)
        out = torch.empty_like(x0)
        u = noise.to(dev, torch.float32).contiguous()
        with torch.cuda.device(dev):
            if self.transition == "uniform":  # bit-exact needs the dense fp16 chain product (d3pm.dense_log_qbar)
                L.q_sample_dense(out, x0, t_tok, m, u, self._dense_log_qbar(dev))
            else:
                L.q_sample(out, x0, t_tok, m, u, self._table(dev), K, _TRANSITIONS[self.transition])
        return out.view(B, W).long()

    # ------------------------------------------------------------------ reverse step (row P)
    def _posterior(self, model_logits: Tensor, t: Tensor, x: Tensor, noise_mode: int, noise, want_post: bool,
                   seed: int = 0, known: Tensor | None = None, temperature: float = 1.0):
        B, W, K = model_logits.shape
        if K != self.num_classes:
            raise ValueError(f"logits have {K} classes, model has {self.num_classes}")
        dev = model_logits.device
        logits = model_logits.contiguous().view(B * W, K)
        if logits.dtype not in (torch.float32, torch.float16, torch.bfloat16):
            logits = logits.float()
        x_t = x.to(torch.int32).contiguous().view(-1)
        check_ids(x_t, K, "p_sample: x")
        row_utt = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(W)
        t_utt = t.to(dev, torch.int32).contiguous()
        utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=dev)
        utt[:, L.U_RESP0] = torch.arange(B, device=dev, dtype=torch.int32) * W
        utt[:, L.U_GID] = torch.arange(B, device=dev, dtype=torch.int32)
        out = torch.empty_like(x_t)
        post = torch.empty(B * W, K, dtype=torch.float32, device=dev) if want_post else None
        uni = noise.to(dev, torch.float32).contiguous() if noise is not None else None
        with torch.cuda.device(dev):
            L.posterior_sample_from_logits(out, post, logits, K, x_t, row_utt, t_utt, utt, self._table(dev),
                                           B * W, 1, K, _TRANSITIONS[self.transition], noise_mode, uni, seed,
                                           known.to(dev) if known is not None else None, temperature)
        return out.view(B, W).long(), (post.view(B, W, K) if want_post else None)

    def q_posterior_logits(self, x_start: Tensor, x_t: Tensor, t: Tensor, x_start_logits: bool = True,
                           temperature: float = 1.0) -> Tensor:
        """logits of q(x_{t-1} | x_t, p(x_0)) (ar_discrete.py:347-375), fp32 closed form.  ``x_start_logits=False``:
        x_start holds the ids of x0 (B, W) and this is q(x_{t-1} | x_t, x0) — the reference's ids branch, through
        vb200_posterior_sample_from_logits_known with every token known (0 at t == 0, as the reference returns).
        ``temperature`` (logits form): p(x_0) = softmax(x_start / temperature); t == 0 returns the raw logits."""
        temperature = self._temperature(temperature)
        if x_start_logits:
            return self._posterior(x_start, t, x_t, L.NOISE_GREEDY, None, want_post=True, temperature=temperature)[1]
        if temperature != 1.0:
            raise ValueError("temperature applies to the logits form only (x_start_logits=True)")
        B, W = x_start.shape
        K = self.num_classes
        known = x_start.to(torch.int32).contiguous().view(-1)
        check_ids(known, K, "q_posterior_logits: x_start")
        # the logit rows of known tokens are never read: an uninitialised (B, W, K) placeholder fills the argument
        placeholder = torch.empty(B, W, K, dtype=torch.float16, device=x_start.device)
        return self._posterior(placeholder, t, x_t, L.NOISE_GREEDY, None, want_post=True, known=known)[1]

    def p_sample(self, model_logits: Tensor, t: Tensor, x: Tensor, noise: Tensor | None = None,
                 greedy: bool = False, seed: int | None = None, temperature: float = 1.0):
        """(sample (B, W) int64, softmax(model_logits)) like ar_discrete.py:401-420.  ``noise``:
        supplied uniforms (B, W, K); omitted -> torch.rand on the CPU generator as the reference,
        unless ``seed`` is given (in-kernel Philox) or ``greedy``.  ``temperature``: the posterior is formed
        from p̂(x0) = softmax(model_logits / temperature) (t == 0 still returns the arg max of the raw logits);
        ValueError unless it is a finite number > 0."""
        temperature = self._temperature(temperature)
        if greedy:
            mode, noise = L.NOISE_GREEDY, None
        elif noise is None and seed is not None:
            mode = L.NOISE_PHILOX
        else:
            mode = L.NOISE_UNIFORMS
            if noise is None:
                noise = torch.rand(size=x.shape + (self.num_classes,)).to(x.device)
        sample, _ = self._posterior(model_logits, t, x, mode, noise, want_post=False, seed=seed or 0,
                                    temperature=temperature)
        return sample, F.softmax(model_logits, dim=-1)


class Diffusion(D3PMOps, Base):
    n_levels = 8  # codebooks diffused jointly (EnCodec 6 kbps, emb/qnt.py:21-23)

    @property
    def n_resp_levels(self):
        return 8

    @property
    def casual(self):
        return False

    @property
    def use_stop_token(self):
        return False

    @property
    def norm_type(self):
        return "adaln"

    @property
    def resp_loss_only(self):
        return True

    @property
    def n_norm_levels(self):
        return self.timesteps + 1

    def _n_classifier_out(self, n_resp_tokens):
        return self.n_levels * n_resp_tokens

    def __init__(self, n_tokens: int = 1024, d_model: int = 1024, n_heads: int = 16, n_layers: int = 12,
                 p_dropout: float = 0.1, n_steps: int = 50, transition: str = "absorbing"):
        if transition not in _TRANSITIONS:
            raise ValueError(f"transition must be 'absorbing' or 'uniform', got {transition!r}")
        # attributes the constructor of Base reads through the properties above
        nn.Module.__init__(self)
        self.timesteps = int(n_steps)
        self.transition = transition
        super().__init__(n_tokens, d_model=d_model, n_heads=n_heads, n_layers=n_layers, p_dropout=p_dropout)
        self.time_emb = nn.Embedding(self.timesteps + 1, d_model)
        self.num_classes = n_tokens
        self.eps = d3pm.EPS

    # ------------------------------------------------------------------ denoiser logits
    def denoise_logits(self, text_list, proms_list, xt_list, t: Tensor, logits_dtype=torch.float32):
        """list of (t'', 8, K) logits of p(x_0 | x_t) for x_t = xt_list[i] (t'', 8) at timestep t[i]."""
        rows = self._logits(text_list, proms_list, xt_list, t, use_time=True, logits_dtype=logits_dtype)
        return [r.view(len(r), self.n_levels, self.num_classes) for r in rows]

    # ------------------------------------------------------------------ reverse loop (row R)
    @torch.no_grad()
    def generate_audio(self, text_list: list[Tensor], proms_list: list[Tensor], resps_list=None, *,
                       resp_lens: list[int] | None = None, seed: int = 0, greedy: bool = False,
                       uniforms_fn=None, gids=None, use_graph: bool = True, trace: list | None = None,
                       to_host: bool = False, as_bqt: bool = False, sample_steps: int | None = None,
                       known_list: list[Tensor] | None = None, temperature: float = 1.0):
        """x_T -> x_0 for a batch of utterances; returns [LongTensor (t'', 8)].

        x_T is all ``mask_id`` for the absorbing transition (ar_discrete.py:699) and uniform random
        codes for the uniform one; the loop runs t = S-1 .. 1 (ar_discrete.py:750).  ``sample_steps``
        = n in [1, S-1] runs n denoise steps instead, at t_i = (S-1) - floor(i (S-1) / n), each drawing
        from the exact jump posterior q(x_{t_{i+1}} | x_{t_i}, x̂0) (``d3pm.schedule_table``); None is
        S-1, the full loop.  ``resp_lens``
        gives the number of frames to generate per utterance (reference: fixed 350, :699);
        ``resps_list`` (optional) supplies x_T explicitly.  ``uniforms_fn(t)`` switches to the
        reference's noise convention (supplied U[0,1) of shape (sum t'' * 8, K)) for parity runs.
        ``to_host`` returns CPU tensors (one device->host copy of the int32 codes).
        ``as_bqt`` returns ``(LongTensor (B, 8, T_max), [t''])`` instead: the whole batch in the layout
        ``emb/qnt.py:32-49 decode(codes (b q t))`` takes, zero-padded, so the EnCodec stage decodes
        the batch in one call instead of one ``t q -> 1 q t`` utterance at a time (SURVEY §8f.4).
        ``known_list``: per utterance an integer (t'', 8) tensor of given codes, -1 where a code is to be
        generated (continuation: a known prefix; span editing: known frames around a span; level-conditional:
        known levels).  Its lengths define ``resp_lens``.  Known tokens start from the same x_T as the others and
        draw every step from the exact posterior q(x_s | x_t, x0 = k); the returned codes equal the given ones at
        every known position (DESIGN.md §5).
        ``temperature`` τ: every reverse step draws from the posterior on p̂(x0) = softmax(logits / τ); τ < 1
        sharpens p̂(x0), τ = 1 (default) is the unscaled loop bit for bit.  Known tokens do not read their logits and
        are unaffected.  ValueError unless τ is a finite number > 0 (DESIGN.md §5).
        """
        n_steps = self._sample_steps(sample_steps)
        temperature = self._temperature(temperature)
        known = None
        if known_list is not None:      # checked before the device is touched, like sample_steps
            known, resp_lens = self._known(known_list, resp_lens, resps_list, len(text_list))
        eng = self.engine()
        dev = eng.w.device
        schedule, table, next_t = self._sampling(dev, n_steps)
        if resps_list is not None:
            resp_lens = [len(r) for r in resps_list]
        elif resp_lens is None:
            resp_lens = [350] * len(text_list)
        ses = self._session(text_list, proms_list, resp_lens, gids)
        lay, x_t = ses.lay, ses.x_t
        if known is not None:
            known = ses.known_buffer().copy_(known, non_blocking=True)
        if resps_list is not None:
            x_T = torch.cat([r.reshape(len(r), self.n_levels) for r in resps_list]).to(torch.int32)
            check_ids(x_T, self.num_classes, "resps_list (x_T)")
            x_t.copy_(x_T, non_blocking=True)
        elif self.transition == "absorbing":
            x_t.fill_(self.mask_id)
        else:
            # uniform start state, one stream per utterance keyed by (seed, GLOBAL utterance id) like the Philox
            # step noise: an utterance's x_T does not depend on which rank or batch it landed in
            ids = gids if gids is not None else range(lay.B)
            parts = []
            for gid, n in zip(ids, lay.t_resp):
                g = torch.Generator().manual_seed((int(seed) * 0x9E3779B1 + int(gid) * 0x85EBCA77 + 0x5D3B) % (1 << 63))
                parts.append(torch.randint(0, self.num_classes, (n, self.n_levels), generator=g, dtype=torch.int32))
            x_t.copy_(torch.cat(parts), non_blocking=True)
        noise = L.NOISE_GREEDY if greedy else (L.NOISE_UNIFORMS if uniforms_fn is not None else L.NOISE_PHILOX)
        ses.run(table, self.timesteps, _TRANSITIONS[self.transition], noise=noise, seed=seed,
                uniforms_fn=uniforms_fn, use_graph=use_graph, n_levels=self.n_levels, trace=trace,
                schedule=schedule, next_t=next_t, known=known, temperature=temperature)
        if as_bqt:        # one (B, 8, T_max) int64 tensor in the EnCodec decoder's layout + the frame counts
            bqt = torch.empty(lay.B, self.n_levels, max(lay.t_resp), dtype=torch.int64, device=dev)
            with torch.cuda.device(dev):
                L.codes_to_bqt(bqt, x_t, lay.utt, pad=0)
            return (bqt.cpu() if to_host else bqt), list(lay.t_resp)
        out = x_t.to("cpu", non_blocking=False) if to_host else x_t
        return [r.long() for r in out.split(lay.t_resp, dim=0)]

    def _known(self, known_list, resp_lens, resps_list, B):
        """(int32 (sum t'', 8) packed given codes, resp_lens) of ``known_list``; ValueError for a wrong count or
        shape, or lengths that disagree with ``resp_lens`` / ``resps_list``; IndexError for ids outside [-1, K)."""
        if len(known_list) != B:
            raise ValueError(f"known_list has {len(known_list)} entries for {B} utterances")
        for i, k in enumerate(known_list):
            if not isinstance(k, Tensor) or k.dim() != 2 or k.shape[1] != self.n_levels:
                raise ValueError(f"known_list[{i}] must be a ({{frames}}, {self.n_levels}) tensor, "
                                 f"got {tuple(k.shape) if isinstance(k, Tensor) else type(k).__name__}")
            if k.dtype.is_floating_point or k.dtype == torch.bool or k.dtype.is_complex:
                raise ValueError(f"known_list[{i}] must hold integer codes, got {k.dtype}")
        lens = [int(k.shape[0]) for k in known_list]
        if resp_lens is not None and [int(n) for n in resp_lens] != lens:
            raise ValueError(f"resp_lens {list(resp_lens)} disagree with the lengths of known_list {lens}")
        if resps_list is not None and [len(r) for r in resps_list] != lens:
            raise ValueError(f"resps_list lengths {[len(r) for r in resps_list]} disagree with known_list {lens}")
        known = torch.cat([k.to(torch.int32) for k in known_list]) if lens else torch.zeros(0, self.n_levels,
                                                                                            dtype=torch.int32)
        check_ids(known, self.num_classes, "known_list", lo=-1)
        return known, lens

    # ------------------------------------------------------------------ training forward (SURVEY §8f.3)
    @torch.no_grad()
    def d3pm_loss(self, text_list: list[Tensor], proms_list: list[Tensor], resps_list: list[Tensor],
                  t: Tensor | int | None = None, *, seed: int = 0, return_per_token: bool = False):
        """The loss of the reference's training forward (ar_discrete.py:651-688) on the GPU, forward
        only: x_t ~ q(x_t | x_0) with in-kernel noise (no K uniforms per token from the host),
        logits = denoiser(x_t, t), cross-entropy against x_0 averaged over all response tokens.

        ``t``: one timestep for the whole batch, a (B,) tensor of per-utterance timesteps, or None for
        the reference's sweep t = 1 .. S-1 (loss averaged over the sweep).  The cross-entropy runs as
        the classifier GEMM's epilogue, so no logits are materialised.  Returns a 0-dim float tensor
        (and the (sum t'', 8) per-token losses of the last timestep when ``return_per_token``)."""
        eng = self.engine()
        dev = eng.w.device
        ses = self._session(text_list, proms_list, [len(r) for r in resps_list], None)
        lay, ws = ses.lay, ses.ws
        x0 = torch.cat([r.reshape(len(r), self.n_levels) for r in resps_list]).to(device=dev, dtype=torch.int32)
        table, tr = self._table(dev), _TRANSITIONS[self.transition]
        if t is None:
            sweep = [torch.full((lay.B,), ti, dtype=torch.int32, device=dev) for ti in range(1, self.timesteps)]
        else:
            tt = torch.as_tensor(t, dtype=torch.int32, device=dev)
            sweep = [tt.expand(lay.B).contiguous() if tt.dim() == 0 else tt.contiguous()]
        check_ids(x0, self.num_classes, "resps_list (x_0)")
        x_t = torch.empty_like(x0)
        loss = torch.empty(lay.M_resp, self.n_levels, dtype=torch.float32, device=dev)
        total = torch.zeros((), dtype=torch.float32, device=dev)
        for i, t_utt in enumerate(sweep):
            t_tok = t_utt[lay.resp_row_utt.long()].repeat_interleave(self.n_levels).contiguous()
            with torch.cuda.device(dev):
                L.q_sample_philox(x_t.view(-1), x0.view(-1), t_tok, None, table, self.num_classes, tr, seed=seed + i)
                head_in = eng.forward(lay, ws, x_t, t_utt, use_time=True, head=False)
                L.head_ce_loss(loss, head_in, eng.w.w_cls, eng.w.b_cls, x0, self.n_levels, self.num_classes)
            total += loss.mean()
        total /= len(sweep)
        return (total, loss, x_t) if return_per_token else total

    def _session(self, text_list, proms_list, resp_lens, gids):
        """Sessions (buffers + captured step graph) are cached per shape signature, so a stream of
        same-shape batches pays layout upload and graph capture once."""
        eng = self.engine()
        cache = eng.__dict__.setdefault("_sessions", {})
        sig = (tuple(len(t) for t in text_list), tuple(len(p) for p in proms_list), tuple(resp_lens))
        ses = cache.get(sig)
        if ses is None:
            if len(cache) >= 4:
                cache.pop(next(iter(cache)))
            lay = BatchLayout(text_list, proms_list, resp_lens, eng.w.device, gids=gids,
                              n_text=eng.w.text_w.shape[0], n_codes=eng.w.K)
            ses = cache[sig] = eng.session(lay)
            self.last_h2d_bytes = lay.h2d_bytes
        else:
            self.last_h2d_bytes = ses.load(text_list, proms_list,
                                           gids if gids is not None else list(range(len(text_list))))
        return ses
