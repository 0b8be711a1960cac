"""float64 references and per-element error bounds of the GEMM and attention kernels.

Every check of those kernels asserts |out - ref| <= bound element by element, with the bound derived from
the arithmetic the kernel does (rounding of the output, fp32 accumulation, bf16 rounding of P, polynomial
approximations) rather than a flat tolerance.  tests/test_error_bounds_teeth.py shows on the CPU that the
same criteria reject plausible defects (a dropped key, a shifted bias column, ...) and accept a faithful
emulation of the kernels' rounding.

Calibration (B200, 148 SMs, the tests of tests/test_gpu_error_bounds.py and tests/test_gpu_kernels.py, both
the tcgen05 and the SIMT kernels): each constant is the smallest power of two that is at least 4 times the
largest ratio (err - other terms) / term observed over all cases.
"""
from __future__ import annotations

import math

import torch

EPI_NONE, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RESIDUAL = 0, 1, 2, 3     # vb200_epilogue (include/vb200.h)

# fp32 accumulation of the K products, in units of 2^-24 * sum_k |a_k w_k|.  Largest observed ratio: not yet
# measured (provisional value).
C_ACC = 16.0
# random-sign bf16 rounding of P, in units of 2^-8 * sqrt(sum_j p_j^2 v_j^2).  Largest observed ratio: not yet
# measured (provisional value).
C_P = 8.0
EPS_GELU = 5e-5      # gelu_erf_fast2 against erf-GELU: max |error| 4.4e-5 (from its coefficients)
EPS_EXP = 7.5e-5     # relative error of ex2_poly2 (the exponential polynomial of the attention softmax)
U_OUT = {torch.float32: 2.0 ** -24, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
FP16_MAX = 65504.0
ATTN_SCALE = 0.125   # 1 / sqrt(head_dim 64)


def gelu64(x: torch.Tensor) -> torch.Tensor:
    return 0.5 * x * (1.0 + torch.special.erf(x * (0.5 ** 0.5)))


def gemm_reference(A, W, out_dtype, epi=EPI_NONE, bias=None, residual=None):
    """(ref, rest, unit) of out = epilogue(A @ W^T) in float64 from the exact 16-bit operands.

    The bound is rest + C_ACC * unit: rest = u_out |ref| (+ 2^-24 (|acc| + |bias|) for the bias add,
    + EPS_GELU for GELU), unit = 2^-24 |A| @ |W|^T."""
    A64, W64 = A.double(), W.double()
    acc = A64 @ W64.t()
    unit = (A64.abs() @ W64.abs().t()) * 2.0 ** -24
    rest = torch.zeros_like(acc)
    ref = acc
    if epi != EPI_NONE:
        b = bias.double()
        rest = rest + 2.0 ** -24 * (acc.abs() + b.abs())
        ref = acc + b
        if epi == EPI_BIAS_GELU:
            ref = gelu64(ref)
            rest = rest + EPS_GELU
        elif epi == EPI_BIAS_RESIDUAL:
            ref = residual.double() + ref
    rest = rest + U_OUT[out_dtype] * ref.abs()
    return ref, rest, unit


def attention_reference(qkv, lens, n_heads, scale=ATTN_SCALE):
    """(ref, rest, unit) of varlen attention in float64 from the bf16 qkv rows, (rows, n_heads * 64) each.

    The bound is rest + C_P * unit: rest = 2^-8 |ref| + EPS_EXP sum_j p_j |v_j|,
    unit = 2^-8 sqrt(sum_j p_j^2 v_j^2)."""
    d = n_heads * 64
    x = qkv.double()
    ref = torch.empty(x.shape[0], d, dtype=torch.float64, device=x.device)
    sq, lin = torch.empty_like(ref), torch.empty_like(ref)
    r0 = 0
    for T in lens:
        for h in range(n_heads):
            c = slice(h * 64, (h + 1) * 64)
            q, k, v = x[r0:r0 + T, c], x[r0:r0 + T, d:][:, c], x[r0:r0 + T, 2 * d:][:, c]
            p = torch.softmax(q @ k.t() * scale, dim=-1)
            ref[r0:r0 + T, c] = p @ v
            sq[r0:r0 + T, c] = (p * p) @ (v * v)
            lin[r0:r0 + T, c] = p @ v.abs()
        r0 += T
    rest = 2.0 ** -8 * ref.abs() + EPS_EXP * lin
    return ref, rest, 2.0 ** -8 * sq.sqrt()


class Report:
    """What one check saw: max err / bound, and the calibration ratio max (err - rest) / unit."""

    def __init__(self, bound_ratio: float, calib_ratio: float):
        self.bound_ratio, self.calib_ratio = bound_ratio, calib_ratio

    def __repr__(self):
        return f"err/bound {self.bound_ratio:.3g}, (err-rest)/unit {self.calib_ratio:.3g}"


def within(out, ref, rest, unit, c, ctx="", saturate_at=None) -> Report:
    """Asserts |out - ref| <= rest + c * unit for every element (NaN fails).  With ``saturate_at`` (fp16 outputs of
    the tcgen05 GEMM, converted with satfinite), elements whose reference lies beyond +-saturate_at by more than
    the bound must equal +-saturate_at exactly, and the others are compared with the clamped reference."""
    o = out.double()
    bound = rest + c * unit
    if saturate_at is not None:
        sat = ref.abs() - bound > saturate_at
        exp = torch.sign(ref) * saturate_at
        nsat = int((sat & (o != exp)).sum())
        assert nsat == 0, f"{ctx}: {nsat} saturated elements are not +-{saturate_at}"
        ref = ref.clamp(-saturate_at, saturate_at)
        o = torch.where(sat, ref, o)
    err = (o - ref).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        idx = bad.nonzero()[:5].tolist()
        sample = [(i, float(o[tuple(i)]), float(ref[tuple(i)]), float(bound[tuple(i)])) for i in idx]
        raise AssertionError(f"{ctx}: {int(bad.sum())} of {bad.numel()} elements outside the bound; "
                             f"max err/bound {float((err / bound).max()):.3g}, max (err - rest)/unit "
                             f"{float(((err - rest) / unit.clamp_min(1e-300)).max()):.3g}; "
                             f"(index, out, ref, bound): {sample}")
    ratio = float((err / bound).max()) if err.numel() else 0.0
    calib = float(((err - rest) / unit.clamp_min(1e-300)).max()) if err.numel() else 0.0
    return Report(ratio, calib)


def check_gemm(out, A, W, epi=EPI_NONE, bias=None, residual=None, ctx="", saturating=False) -> Report:
    ref, rest, unit = gemm_reference(A, W, out.dtype, epi, bias, residual)
    sat = FP16_MAX if (saturating and out.dtype == torch.float16) else None
    return within(out, ref, rest, unit, C_ACC, ctx, sat)


def check_attention(out, qkv, lens, n_heads, ctx="") -> Report:
    ref, rest, unit = attention_reference(qkv, lens, n_heads)
    return within(out, ref, rest, unit, C_P, ctx)


# ---------------------------------------------------------------- inputs shared by the GPU tests and the CPU teeth
RESCALE_THRESHOLD = 8.0 / math.log2(math.e)   # score growth (natural units) past which the kernel moves its maximum
GAP_BELOW, GAP_ABOVE = 5.3125, 5.8125         # bf16-exact, either side of RESCALE_THRESHOLD (5.545)


def random_qkv(rows, n_heads, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(rows, 3 * n_heads * 64, generator=g) * scale).bfloat16()


def structured_qkv(lens, n_heads, seed, events=(), base=0.0):
    """q / k rows whose scores are set through coordinate 0, the other coordinates small (|score noise| < 0.01):
    even query rows have q[0] = 8, odd rows q[0] = 4, so with k[0] = c their score with that key is c resp. c / 2.
    Every key of every utterance has k[0] = ``base`` except ``events``: (utterance, key index, c) set k[0] = c.
    V is random.  With events of growing c, a row's maximum moves in a chosen key block by a chosen amount."""
    g = torch.Generator().manual_seed(seed)
    M, d = sum(lens), n_heads * 64
    qkv = torch.randn(M, 3 * d, generator=g) * 0.05
    qkv[:, 2 * d:] = torch.randn(M, d, generator=g)
    q0 = torch.where(torch.arange(M) % 2 == 0, 8.0, 4.0)
    starts = [sum(lens[:i]) for i in range(len(lens))]
    for h in range(n_heads):
        qkv[:, h * 64] = q0
        qkv[:, d + h * 64] = base
        for u, j, c in events:
            qkv[starts[u] + j, d + h * 64] = c
    return qkv.bfloat16()


def gemm_inputs(M, N, K, op_dtype, seed, a_scale=1.0, device="cpu"):
    """A (M, K), W (N, K) scaled by K^-1/2 (outputs of order a_scale), bias (N,) and residual (M, N), drawn from a
    generator on ``device`` (the CPU one for every shape the CPU teeth replay).  A stays within fp16's range."""
    g = torch.Generator(device=device).manual_seed(seed)
    A = (torch.randn(M, K, generator=g, device=device) * a_scale).clamp(-6e4, 6e4).to(op_dtype)
    W = (torch.randn(N, K, generator=g, device=device) * K ** -0.5).to(op_dtype)
    bias = torch.randn(N, generator=g, device=device)
    resid = torch.randn(M, N, generator=g, device=device)
    return A, W, bias, resid
