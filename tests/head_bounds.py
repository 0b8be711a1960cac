"""float64 references and error bounds of the fused classifier head (head_sample_kernel,
csrc/head_sample_tcgen05.cu): its greedy codes, its Philox draws and its cross-entropy.

The kernel's logits are the fp32 accumulator plus the fp32 bias, so their float64 reference and per-element
bound come from error_bounds.gemm_reference (bound rest + C_ACC unit); delta is the largest bound over the K
columns of a token's level.  From there:

* greedy: a logit error of at most delta moves log p_j by at most 2 delta, and log(f2_j + eps) by no more,
  because a > c in every table.  On top come the fp32 sum of Z, exp2f_fast and the rounding of the exponent's
  argument, eps_math = (K + 64 + 4 max|l|) 2^-24.  A token is clear when every class within
  2 (2 delta + eps_math) of its float64 top posterior weight has exactly that weight (planted ties), and then
  the kernel must pick the lowest of those classes.
* cross-entropy: LSE is 1-Lipschitz in the max-norm, so |loss - ref| <= 2 delta + the fp32 rounding of
  m + ln Z - l_x + C_CE (K 2^-24 + 2^-21) for the online Z and __logf.
* Philox draws: a randomised probability integral transform u = F(c - 1) + V p_c, V ~ U(0, 1) from a seeded
  CPU generator, is iid U(0, 1) under the float64 posterior; the Kolmogorov-Smirnov statistic must stay below
  1.95 / sqrt(n) (about the 0.1 % level; the seeds are fixed, so the test is deterministic).

tests/test_head_bounds_teeth.py shows on the CPU that these checks reject plausible defects of the kernel's
streaming epilogue and accept an emulation of its fp32 arithmetic; tests/test_gpu_head_bounds.py applies them
to the kernel at multi-item scale.
"""
from __future__ import annotations

import math

import numpy as np
import torch

import error_bounds as eb

U32 = 2.0 ** -24
EPS = 1.0e-6            # kEps (csrc/common.cuh), ar_discrete.py:276
TILE, HALF = 256, 128   # column tile of one work item step and the columns one epilogue thread streams of it
# fp32 arithmetic of the cross-entropy epilogue (online max and Z, exp2f_fast, __logf), in units of
# K 2^-24 + 2^-21.  Largest observed ratio: not yet measured (provisional value, not calibrated).
C_CE = 8.0
S_STEPS = 50


# ---------------------------------------------------------------- the reverse step in float64
def kernel_weights(tab, t, x_t, p, tr, eps=EPS):
    """Restatement of post_scalars + post_special (csrc/posterior.cuh), vectorised over tokens: the unnormalised
    weights (N, K) the reverse-step kernels give every class, reading row t's Q and row t-1's Qbar entries of the
    scalar table ``tab`` (S, TAB_STRIDE).  t, x_t: (N,) integer tensors; p: (N, K) softmax of the logits."""
    from vall_e.b200 import lib as L
    N, K = p.shape
    t, x_t = t.long().to(p.device), x_t.long().to(p.device)
    tab = tab.to(device=p.device, dtype=p.dtype)
    one, cum = tab[t], tab[(t - 1).clamp_min(0)]
    absorbing = tr == "absorbing"
    m = K // 2 if absorbing else -1
    at_m = x_t == m
    f1_self = torch.where(at_m, one[:, L.TAB_ONE_BOTH], one[:, L.TAB_ONE_KEEP]) + eps
    f1_oth = torch.where(at_m, one[:, L.TAB_ONE_ABSORB], one[:, L.TAB_ONE_OFF]) + eps
    a_gen, c_gen = cum[:, L.TAB_CUM_KEEP], cum[:, L.TAB_CUM_OFF]
    a_m = cum[:, L.TAB_CUM_BOTH] if absorbing else a_gen
    c_m = cum[:, L.TAB_CUM_ABSORB] if absorbing else c_gen
    w = f1_oth[:, None] * (p * (a_gen - c_gen)[:, None] + (c_gen + eps)[:, None])
    rows = torch.arange(N, device=p.device)
    if absorbing:
        h = ~at_m
        w[rows[h], m] = f1_oth[h] * (p[h, m] * (a_m - c_m)[h] + c_m[h] + eps)
    a_x, c_x = torch.where(at_m, a_m, a_gen), torch.where(at_m, c_m, c_gen)
    w[rows, x_t] = f1_self * (p[rows, x_t] * (a_x - c_x) + c_x + eps)
    return w


def log_posterior(logits64, tab, t, x_t, tr):
    """float64 log of the reverse step's weights (N, K), unnormalised; the raw logits where t == 0."""
    lw = torch.log(kernel_weights(tab, t, x_t, torch.softmax(logits64, -1), tr))
    return torch.where((t.to(logits64.device) == 0)[:, None], logits64, lw)


def level_references(head_in, W, bias, n_levels, K, c_acc=eb.C_ACC):
    """Yields (level, logits64 (rows, K), bound (rows, K)) of the kernel's fp32 logits, one level at a time."""
    for lv in range(n_levels):
        cols = slice(lv * K, (lv + 1) * K)
        ref, rest, unit = eb.gemm_reference(head_in, W[cols], torch.float32, eb.EPI_BIAS, bias[cols])
        yield lv, ref, rest + c_acc * unit


def eps_math(K, lmax):
    return (K + 64 + 4 * lmax) * U32


def greedy_expected(logpost, margin):
    """(expected code, clear, tied) per token: clear when the classes within ``margin`` of the top log-weight are
    exactly those at the top; the expected code is the lowest of them, tied marks more than one."""
    K = logpost.shape[-1]
    top = logpost.max(-1, keepdim=True).values
    exact = logpost == top
    clear = ((logpost > top - margin[:, None]) == exact).all(-1)
    cls = torch.arange(K, device=logpost.device).expand_as(logpost)
    expected = torch.where(exact, cls, K).min(-1).values
    return expected, clear, exact.sum(-1) > 1


def greedy_reference(logits64, bound, tab, t, x_t, tr):
    """(expected, clear, tied) of one level's tokens for the greedy codes (see greedy_expected)."""
    delta = bound.max(-1).values
    margin = 2 * (2 * delta + eps_math(logits64.shape[-1], logits64.abs().max(-1).values))
    return greedy_expected(log_posterior(logits64, tab, t, x_t, tr), margin)


def ce_reference(logits64, bound, target):
    """(ref, rest, unit) of -log softmax(logits)[target]; the bound is rest + C_CE unit."""
    K = logits64.shape[-1]
    tgt = target.long().to(logits64.device)[:, None]
    m = logits64.max(-1).values
    lnZ = torch.log(torch.exp(logits64 - m[:, None]).sum(-1))
    lx = logits64.gather(-1, tgt)[:, 0]
    ref = m + lnZ - lx
    rest = 2 * bound.max(-1).values + 4 * U32 * (m.abs() + lnZ + lx.abs())
    return ref, rest, torch.full_like(ref, K * U32 + 2.0 ** -21)


def law(logits64, tab, t, x_t, tr):
    """float64 probabilities (N, K) of the reverse step's draw (t > 0)."""
    w = kernel_weights(tab, t, x_t, torch.softmax(logits64, -1), tr)
    return w / w.sum(-1, keepdim=True)


def pit(prob, codes, v):
    """Randomised probability integral transform of draws ``codes`` under ``prob`` (N, K): u = F(c - 1) + V p_c."""
    c = codes.long().to(prob.device)[:, None]
    pc = prob.gather(-1, c)[:, 0]
    below = prob.cumsum(-1).gather(-1, c)[:, 0] - pc
    return (below + v.to(prob.device) * pc).clamp(0.0, 1.0)


def ks_statistic(u):
    u = np.sort(np.asarray(u, dtype=np.float64))
    n = u.size
    i = np.arange(1, n + 1)
    return float(max((i / n - u).max(), (u - (i - 1) / n).max()))


def check_law(u, ctx=""):
    n = int(np.asarray(u).size)
    D = ks_statistic(u)
    assert D < 1.95 / math.sqrt(n), f"{ctx}: KS statistic {D:.4g} >= 1.95 / sqrt({n}) = {1.95 / math.sqrt(n):.4g}"
    return D


def check_greedy(got, expected, clear, ctx=""):
    got, expected, clear = got.long().cpu(), expected.long().cpu(), clear.cpu()
    frac = clear.float().mean().item()
    assert frac >= 0.7, f"{ctx}: only {frac:.3f} of the tokens are clear"
    bad = clear & (got != expected)
    nbad = int(bad.sum())
    if nbad:
        idx = bad.nonzero()[:5].view(-1).tolist()
        raise AssertionError(f"{ctx}: {nbad} of {int(clear.sum())} clear greedy codes differ; "
                             f"(token, got, expected): {[(i, int(got[i]), int(expected[i])) for i in idx]}")
    return frac


# ---------------------------------------------------------------- inputs shared by the GPU tests and the CPU teeth
def special_classes(K):
    """Class 0, both sides of the half and tile edges, the absorbing class K/2 and K - 1."""
    return sorted({0, 127, 128, 255, 256, K // 2, K - 1} & set(range(K)))


def tie_pairs(K):
    """Duplicated W rows with equal bias, in different tiles (K > 256) and halves; none is special."""
    return [(5, K - 100), (200, K // 2 + 60 if K > TILE else 60)]


def last_tile_classes(K):
    return [K - 250, K - 40]


class Case:
    """A multi-item launch of the fused head: rows chosen so that every CTA pair runs at least ``items_per_pair``
    work items (256-row block, level) on a device with ``sms`` SMs; ``rows_mod`` = rows % 256 (or 256) leaves the
    rank-1 CTA of the last block partial (> 128) or empty (<= 128).

    Rows cycle through kinds (row % 8): 0 logits scaled to about +-80..100, 1 maximum only in the last column
    tile, 2 the planted ties at the top, other plain.  Utterances of 100..900 rows take t = 0, 1, S/2, S-1 in
    turn; x_t is masked (K/2), a special class, or random, a third each."""

    def __init__(self, K, d, n_levels, dtype, sms, seed, rows_mod, items_per_pair=3, S=S_STEPS):
        from vall_e.b200 import lib as L
        self.K, self.d, self.n_levels, self.dtype, self.S = K, d, n_levels, dtype, S
        self.pairs = sms // 2
        blocks = -(-items_per_pair * self.pairs // n_levels)
        self.rows = rows = (blocks - 1) * TILE + rows_mod
        self.items = blocks * n_levels
        g = torch.Generator().manual_seed(seed)
        x = torch.randn(rows, d, generator=g)
        W = torch.randn(n_levels * K, d, generator=g) * d ** -0.5
        bias = torch.randn(n_levels * K, generator=g)
        self.kind = kind = torch.arange(rows) % 8
        x[:, :2] = 0.0
        W[:, :2] = 0.0
        x[kind == 0] *= 24.0
        x[kind == 1, 0] = 10.0
        x[kind == 2, 1] = 10.0
        for lv in range(n_levels):
            o = lv * K
            for c in last_tile_classes(K):
                W[o + c, 0] = 1.0
            for j1, j2 in tie_pairs(K):
                W[o + j1, 1] = 1.0
                W[o + j2] = W[o + j1]
                bias[o + j2] = bias[o + j1]
        self.head_in, self.W, self.bias = x.to(dtype), W.to(dtype), bias
        lens, r = [], 0
        while r < rows:
            n = min(int(torch.randint(100, 900, (1,), generator=g)), rows - r)
            lens.append(n)
            r += n
        B = len(lens)
        self.lens = lens
        starts = torch.tensor([0] + lens[:-1]).cumsum(0)
        self.row_utt = torch.repeat_interleave(torch.arange(B, dtype=torch.int32), torch.tensor(lens))
        self.t_utt = torch.tensor([0, 1, S // 2, S - 1], dtype=torch.int32)[torch.arange(B) % 4]
        self.utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32)
        self.utt[:, L.U_RESP0] = starts.int()
        self.utt[:, L.U_GID] = 1000 + 7 * torch.arange(B, dtype=torch.int32)
        tok = torch.arange(rows * n_levels).view(rows, n_levels)
        x_t = torch.randint(0, K, (rows, n_levels), generator=g, dtype=torch.int32)
        sp = torch.tensor(special_classes(K), dtype=torch.int32)
        x_t = torch.where(tok % 3 == 0, K // 2, torch.where(tok % 3 == 1, sp[(tok // 3) % len(sp)], x_t))
        self.x_t = x_t.int()
        # cross-entropy targets: the row's arg max (loss ~ 0), edges of tiles / halves, or random
        tgt = torch.randint(0, K, (rows, n_levels), generator=g, dtype=torch.int32)
        edge = torch.tensor([0, K - 1] + special_classes(K), dtype=torch.int32)
        tgt = torch.where(tok % 4 == 1, edge[(tok // 4) % len(edge)], tgt)
        self._tgt, self._tok = tgt, tok

    def t_rows(self):
        """(rows,) clamped timestep of every row."""
        return self.t_utt.long()[self.row_utt.long()]

    def targets(self, logits_fp32_levels):
        """CE targets, with every 4th token on its row's arg max, from fp32 logits (rows, n_levels, K)."""
        am = logits_fp32_levels.argmax(-1).int().cpu()
        return torch.where(self._tok % 4 == 0, am, self._tgt)

    def ctx(self):
        return (f"K={self.K} d={self.d} levels={self.n_levels} {str(self.dtype)[6:]} rows={self.rows} "
                f"items={self.items}")


F16, BF16 = torch.float16, torch.bfloat16
KS, DS = (256, 768, 1024, 4096), (72, 200, 1024)


def _matrix():
    """Every (K, d); the level count, operand type and ragged end rotate so that each K and each d sees all."""
    out = []
    for ki, K in enumerate(KS):
        for di, d in enumerate(DS):
            i = 3 * ki + di
            out.append((K, d, (1, 3, 8)[(ki + di) % 3], (BF16, F16)[i % 2], (200, 100)[(i // 2) % 2], 100 + i))
    return out


CASES = _matrix()           # (K, d, n_levels, dtype, rows_mod, seed); tpl = K / 256 is 1, 3, 4 and 16
# Philox law: pooled over these launches, with at least 6 work items per CTA pair (>= 200 k tokens at t > 0)
LAW_CASES = [(256, 200, 8, F16, 200, 301), (768, 72, 3, BF16, 100, 302), (1024, 136, 8, BF16, 60, 303)]
LAW_ITEMS_PER_PAIR = 6
