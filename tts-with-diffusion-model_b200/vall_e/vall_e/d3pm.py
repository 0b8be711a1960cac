"""Host-side D3PM constants for the CUDA reverse step.

The reference keeps three dense (S, K, K) fp16 tensors (``ar_discrete.py:257-277``: one-step
matrices, their fp16 chain product ``q_mats`` and the transposes, 3 x 210 MB at S=100, K=1025) and
indexes them with one-hot matmuls.  Both transition families have rank-structured matrices, so the
kernels only need a few scalars per timestep.  To keep those scalars equal to what the reference
holds (the fp16 chain product drifts from the analytic value — row sums reach 1.002 — and
``eps=1e-6`` makes that drift observable), they are read out of the same fp16 chain product,
computed here once with a running (K, K) matrix instead of being re-derived from alpha-bar.
Absorbing: every entry of the product has at most two non-zero terms, so the product is exactly
rank-structured and the scalars are bit-identical to the dense entries.  Uniform: K-term sums, so
the dense product carries up to 2 diagonal / 3 off-diagonal values per t that differ by one fp16
ulp; the scalars are representative entries (``tests/test_host_cpu.py`` bounds the gap), and the
bit-exact parity path reads the dense table instead (``dense_log_qbar``).
"""
from __future__ import annotations

import functools

import numpy as np
import torch

from ..b200 import lib as L

EPS = 1.0e-6  # ar_discrete.py:276


def cosine_beta_schedule(timesteps: int, s: float = 0.008) -> torch.Tensor:
    """Cosine schedule with the reference's grid: ``steps`` points spread over [0, steps]
    (not [0, 1]) before normalising by ``steps`` (ar_discrete.py:286-304)."""
    steps = timesteps + 1
    grid = np.linspace(0, steps, steps)
    abar = np.cos(((grid / steps) + s) / (1 + s) * np.pi * 0.5) ** 2
    abar = abar / abar[0]
    betas = np.clip(1 - (abar[1:] / abar[:-1]), a_min=0, a_max=0.999)
    return torch.from_numpy(betas)


def _onestep(beta_t: torch.Tensor, K: int, transition: str) -> torch.Tensor:
    if transition == "absorbing":      # (1-b) I + b 1 e_m^T, float64 then fp16 (ar_discrete.py:315-334,269)
        b = float(beta_t.numpy())
        q = torch.zeros(K, K, dtype=torch.float64)
        q.fill_diagonal_(1.0 - b)
        q[:, K // 2] += b
        return q.to(torch.float16)
    if transition == "uniform":        # fp16 from the start (ar_discrete.py:308-313)
        q = torch.full((K, K), beta_t / K).to(torch.float16)
        q.fill_diagonal_(1.0 - beta_t * (K - 1) / K)
        return q
    raise ValueError(f"unknown transition {transition!r} (expected 'absorbing' or 'uniform')")


@functools.lru_cache(maxsize=16)
def scalar_table(timesteps: int, K: int, transition: str) -> torch.Tensor:
    """float32 (S, TAB_STRIDE) table for vb200_q_sample / vb200_posterior_sample_from_logits (the reverse
    step at every t = S-1 .. 1; ``schedule_table`` for fewer steps)."""
    betas = cosine_beta_schedule(timesteps + 1).to(torch.float16)     # ar_discrete.py:257
    m = K // 2
    a = 0 if m != 0 else 1
    b = 1 if m != 1 else 2
    tab = torch.zeros(timesteps, L.TAB_STRIDE, dtype=torch.float32)
    cum = None
    for t in range(timesteps):
        one = _onestep(betas[t], K, transition)
        cum = one if cum is None else torch.tensordot(cum, one, dims=[[1], [0]])  # fp16, :270-274
        tab[t, L.TAB_ONE_KEEP] = one[a, a]
        tab[t, L.TAB_ONE_OFF] = one[a, b]
        tab[t, L.TAB_ONE_ABSORB] = one[a, m]
        tab[t, L.TAB_ONE_BOTH] = one[m, m]
        picks = torch.stack([cum[a, a], cum[a, b], cum[a, m], cum[m, m]])
        tab[t, L.TAB_CUM_KEEP:L.TAB_CUM_BOTH + 1] = picks.float()
        # q_sample logits are formed in fp16: log(fp16(q) + eps) (ar_discrete.py:482)
        tab[t, L.TAB_LOG_KEEP:L.TAB_LOG_BOTH + 1] = torch.log(picks + EPS).float()
    return tab


@functools.lru_cache(maxsize=64)
def sample_schedule(timesteps: int, n: int) -> tuple[int, ...]:
    """The ``n`` timesteps a reverse loop of ``n`` denoise steps visits: t_i = (S-1) - floor(i (S-1) / n),
    i = 0 .. n-1, strictly decreasing from S-1; the step at t_i draws x_{t_{i+1}} (x_0 after the last).
    ``n = S-1`` is the full loop S-1, ..., 1."""
    S, n = int(timesteps), int(n)
    if not 1 <= n <= S - 1:
        raise ValueError(f"sample_steps must lie in [1, {S - 1}] for a model with {S} timesteps, got {n}")
    return tuple((S - 1) - (i * (S - 1)) // n for i in range(n))


def check_schedule(timesteps: int, schedule) -> tuple[int, ...]:
    """``schedule`` as a tuple, or ValueError unless it is a non-empty, strictly decreasing list of
    timesteps in [1, S-1]."""
    sch = tuple(int(t) for t in schedule)
    if not sch or not all(1 <= t <= timesteps - 1 for t in sch) or any(a <= b for a, b in zip(sch, sch[1:])):
        raise ValueError(f"a schedule is a strictly decreasing list of timesteps in [1, {timesteps - 1}], got {sch}")
    return sch


def successors(timesteps: int, schedule) -> list[int]:
    """next_t for ``vb200_step_timesteps_to``: next_t[t] = the timestep after t in ``schedule`` (0 after
    the last), and t-1 (0 at t = 0) at every timestep the schedule does not visit."""
    sch = check_schedule(timesteps, schedule)
    nxt = [max(t - 1, 0) for t in range(timesteps)]
    for t, s in zip(sch, sch[1:] + (0,)):
        nxt[t] = s
    return nxt


@functools.lru_cache(maxsize=16)
def _schedule_table(timesteps: int, K: int, transition: str, schedule: tuple) -> torch.Tensor:
    plain = scalar_table(timesteps, K, transition)
    tab = plain.clone()
    betas = cosine_beta_schedule(timesteps + 1).to(torch.float16)
    m = K // 2
    a = 0 if m != 0 else 1
    b = 1 if m != 1 else 2
    for t, s in zip(schedule, schedule[1:] + (0,)):
        if s == t - 1:
            continue
        jump = _onestep(betas[s + 1], K, transition)          # Q_{t|s} = Q_{s+1} ... Q_t, fp16 as scalar_table's Qbar
        for u in range(s + 2, t + 1):
            jump = torch.tensordot(jump, _onestep(betas[u], K, transition), dims=[[1], [0]])
        tab[t, L.TAB_ONE_KEEP] = jump[a, a]
        tab[t, L.TAB_ONE_OFF] = jump[a, b]
        tab[t, L.TAB_ONE_ABSORB] = jump[a, m]
        tab[t, L.TAB_ONE_BOTH] = jump[m, m]
        tab[t - 1, L.TAB_CUM_KEEP:L.TAB_CUM_BOTH + 1] = plain[s, L.TAB_CUM_KEEP:L.TAB_CUM_BOTH + 1]
    return tab


def schedule_table(timesteps: int, K: int, transition: str, schedule) -> torch.Tensor:
    """The scalar table of a reverse loop that visits ``schedule`` (``sample_schedule``, or any strictly
    decreasing list in [1, S-1]), for the reverse-step kernels only.

    The reverse step at t reads the Q entries of row t and the Qbar entries of row t-1 (``post_scalars``
    in csrc/posterior.cuh).  For every visited t whose successor s = sigma(t) is not t-1, row t's ONE_*
    fields hold Q_{t|s} = Q_{s+1} ... Q_t (the fp16 chain product, formed as ``scalar_table`` forms Qbar)
    and row t-1's CUM_* fields hold Qbar_s, so the same closed form draws from the jump posterior
    q(x_s | x_t, x̂0).  Every other entry is ``scalar_table``'s: for the full schedule the two tables are
    equal.  A row's CUM_* fields no longer need to hold that row's own Qbar_t, so the table is for the
    reverse step only: ``q_sample`` and the training forward keep getting ``scalar_table``.  This
    function is the one place that knows that row layout.  Cached: do not modify the returned tensor."""
    return _schedule_table(int(timesteps), int(K), transition, check_schedule(timesteps, schedule))


@functools.lru_cache(maxsize=2)
def dense_log_qbar(timesteps: int, K: int, transition: str) -> torch.Tensor:
    """fp16 (S, K, K) ``log(Qbar_t + eps)`` — the logits ``q_sample`` forms (ar_discrete.py:482) from
    the fp16 chain product (:270-275), for ``vb200_q_sample_dense``.  Only the *uniform* transition
    needs it, and only for bit-exact parity runs with supplied uniforms: its K-term fp16 sums are not
    rank-structured to the last bit (up to 2 diagonal and 3 off-diagonal values per t, placed by the
    summation order of the GEMM), so `scalar_table` holds representative values there, exact ones
    for absorbing (<= 2 non-zero terms per entry)."""
    betas = cosine_beta_schedule(timesteps + 1).to(torch.float16)
    out = torch.empty(timesteps, K, K, dtype=torch.float16)
    cum = None
    for t in range(timesteps):
        one = _onestep(betas[t], K, transition)
        cum = one if cum is None else torch.tensordot(cum, one, dims=[[1], [0]])
        out[t] = torch.log(cum + EPS)
    return out


def betas_fp16(timesteps: int) -> torch.Tensor:
    return cosine_beta_schedule(timesteps + 1).to(torch.float16)
