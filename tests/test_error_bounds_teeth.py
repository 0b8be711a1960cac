"""The error bounds of tests/error_bounds.py have teeth (CPU only, no GPU needed).

Each planted defect below is a plausible off-by-one of the GEMM or attention kernel, replayed on the CPU from the
same shapes and seeds the GPU tests use; the bound must reject it.  An emulation of the kernels' own rounding
(fp32 accumulation and epilogue, bf16 P with a lazily moved maximum, 16-bit outputs) must pass with 2x margin:
with the calibrated constant (C_ACC, C_P) halved.  The output-rounding term u_out |ref| has no margin to give —
a 16-bit output rounded from just past a midpoint at the bottom of a binade is off by u_out |ref| itself."""
import pytest
import torch

import error_bounds as eb

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


# ---------------------------------------------------------------- GEMM
def emulate_gemm(A, W, out_dtype, epi, bias=None, resid=None, defect=None):
    """fp32 accumulation and epilogue, rounded once to ``out_dtype``; ``defect`` plants one error."""
    A32, W32 = A.float().clone(), W.float()
    K = A.shape[1]
    if defect == "drop_k16":                     # one 16-wide k-slice of one MMA missing
        k0 = 16 * ((K // 16) // 2)
        A32[:, k0:k0 + 16] = 0
    elif defect == "drop_last_kblock":           # the partial last k-block of 64 missing
        A32[:, (K // 64) * 64:] = 0
    acc = A32 @ W32.t()
    if defect == "acc_bf16":                     # accumulator through bf16 before an fp32 epilogue
        acc = acc.bfloat16().float()
    x = acc
    if epi != eb.EPI_NONE:
        x = acc + (torch.roll(bias, -1) if defect == "bias_shift" else bias)
        if epi == eb.EPI_BIAS_GELU:
            x = torch.nn.functional.gelu(x, approximate="tanh" if defect == "tanh_gelu" else "none")
        elif epi == eb.EPI_BIAS_RESIDUAL:
            x = x + {"no_residual": 0.0, "residual_twice": 2 * resid}.get(defect, resid)
    return x.to(out_dtype)


# (M, N, K, seed, operands, epilogue, output dtype) as tests/test_gpu_error_bounds.py draws them
GEMM_FAITHFUL = [
    (1027, 1024, 4096, 1024, BF16, eb.EPI_BIAS_RESIDUAL, F32),     # FFN2 of one utterance
    (1027, 1024, 4096, 1024, BF16, eb.EPI_BIAS, F32),
    (129, 384, 200, 9, F16, eb.EPI_BIAS_GELU, F32),
    (257, 264, 1024, 5, BF16, eb.EPI_BIAS_GELU, BF16),
    (300, 200, 4104, 7, F16, eb.EPI_NONE, F16),
    (127, 72, 56, 3, BF16, eb.EPI_BIAS, F16),
]


def _gemm_case(M, N, K, seed, op):
    return eb.gemm_inputs(M, N, K, op, seed)


@pytest.mark.parametrize("M,N,K,seed,op,epi,out_dt", GEMM_FAITHFUL)
def test_gemm_bound_accepts_the_kernels_rounding(M, N, K, seed, op, epi, out_dt):
    A, W, bias, resid = _gemm_case(M, N, K, seed, op)
    out = emulate_gemm(A, W, out_dt, epi, bias, resid)
    ref, rest, unit = eb.gemm_reference(A, W, out_dt, epi, bias, resid)
    eb.within(out, ref, rest, unit, eb.C_ACC / 2, "emulation")


GEMM_DEFECTS = [
    ("drop_k16", (1027, 1024, 4096, 1024, BF16, eb.EPI_NONE, BF16)),
    ("drop_k16", (129, 384, 200, 9, F16, eb.EPI_BIAS, F16)),
    ("drop_k16", (127, 72, 56, 3, BF16, eb.EPI_NONE, F32)),
    ("drop_last_kblock", (300, 200, 4104, 7, F16, eb.EPI_NONE, BF16)),
    ("drop_last_kblock", (129, 200, 200, 4, BF16, eb.EPI_BIAS, F16)),
    ("acc_bf16", (1027, 1024, 4096, 1024, BF16, eb.EPI_BIAS, F32)),
    ("acc_bf16", (1027, 1024, 4096, 1024, BF16, eb.EPI_BIAS_RESIDUAL, F32)),
    ("bias_shift", (257, 264, 1024, 5, BF16, eb.EPI_BIAS, BF16)),
    ("bias_shift", (127, 72, 56, 3, BF16, eb.EPI_BIAS_GELU, F16)),
    ("no_residual", (1027, 1024, 4096, 1024, BF16, eb.EPI_BIAS_RESIDUAL, F32)),
    ("residual_twice", (257, 264, 1024, 5, BF16, eb.EPI_BIAS_RESIDUAL, F32)),
    ("tanh_gelu", (129, 384, 200, 9, F16, eb.EPI_BIAS_GELU, F32)),
    ("tanh_gelu", (1027, 4096, 1024, 1024, BF16, eb.EPI_BIAS_GELU, F32)),
]


@pytest.mark.parametrize("defect,case", GEMM_DEFECTS, ids=[f"{d}-{c[0]}x{c[1]}x{c[2]}" for d, c in GEMM_DEFECTS])
def test_gemm_bound_rejects_planted_defect(defect, case):
    M, N, K, seed, op, epi, out_dt = case
    A, W, bias, resid = _gemm_case(M, N, K, seed, op)
    out = emulate_gemm(A, W, out_dt, epi, bias, resid, defect)
    ref, rest, unit = eb.gemm_reference(A, W, out_dt, epi, bias, resid)
    with pytest.raises(AssertionError, match="outside the bound"):
        eb.within(out, ref, rest, unit, eb.C_ACC, defect)


def test_fp16_saturation_criterion():
    """Saturated fp16 outputs must be exactly +-65504: inf, or a value below the limit, is rejected."""
    A, W, bias, resid = eb.gemm_inputs(129, 200, 200, F16, 4, a_scale=3e4)
    ref, rest, unit = eb.gemm_reference(A, W, F16, eb.EPI_NONE)
    good = (A.float() @ W.float().t()).clamp(-eb.FP16_MAX, eb.FP16_MAX).half()
    assert (ref.abs() > 1.1 * eb.FP16_MAX).any()
    eb.within(good, ref, rest, unit, eb.C_ACC, "satfinite", saturate_at=eb.FP16_MAX)
    with pytest.raises(AssertionError, match="saturated"):
        eb.within((A.float() @ W.float().t()).half(), ref, rest, unit, eb.C_ACC, "inf", saturate_at=eb.FP16_MAX)


# ---------------------------------------------------------------- attention
def emulate_attention(qkv, lens, n_heads, scale=eb.ATTN_SCALE, defect=None):
    """The tcgen05 kernel's arithmetic: 128-key blocks, the reference maximum moved only when a block exceeds it by
    2^8 (O and l rescaled then), P rounded to bf16 for O += P V, l summed from the unrounded P, bf16 output.
    ``defect`` plants one error."""
    d = n_heads * 64
    x = qkv.double()
    out = torch.empty(x.shape[0], d, dtype=torch.bfloat16)
    r0 = 0
    for b, T in enumerate(lens):
        keys = torch.arange(r0, r0 + T)
        if defect == "drop_last_key":
            keys = keys[:-1]
        elif defect == "drop_short_block" and T % 128 and T % 128 <= 32:
            keys = keys[:T - T % 128]
        for h in range(n_heads):
            c = slice(h * 64, (h + 1) * 64)
            kc = slice(d + (h + 1) * 64, d + (h + 2) * 64) if defect == "next_head_k" else slice(d + h * 64, d + (h + 1) * 64)
            q = x[r0:r0 + T, c]
            k, v = x[keys, kc], x[keys, 2 * d + h * 64:2 * d + (h + 1) * 64]
            if defect == "key_past_end":          # the next utterance's first row, or the TMA's zero fill
                nxt = x[r0 + T:r0 + T + 1] if r0 + T < x.shape[0] else torch.zeros(1, 3 * d, dtype=x.dtype)
                k = torch.cat([k, nxt[:, kc]])
                v = torch.cat([v, nxt[:, 2 * d + h * 64:2 * d + (h + 1) * 64]])
            s = q @ k.t() * (d ** -0.5 if defect == "scale_dmodel" else scale)
            m = torch.full((T, 1), -float("inf"), dtype=torch.float64)
            l = torch.zeros(T, 1, dtype=torch.float64)
            o = torch.zeros(T, 64, dtype=torch.float64)
            for j0 in range(0, s.shape[1], 128):
                sb = s[:, j0:j0 + 128]
                bm = sb.max(dim=1, keepdim=True).values
                if j0 == 0:
                    m = bm
                else:
                    grow = (bm - m) * 1.4426950408889634 > 8.0
                    m_new = torch.where(grow, bm, m)
                    alpha = torch.exp(m - m_new)
                    l = l * alpha
                    if defect != "missed_rescale":
                        o = o * alpha
                    m = m_new
                p = torch.exp(sb - m).float()
                l = l + p.double().sum(dim=1, keepdim=True)
                o = o + p.bfloat16().double() @ v[j0:j0 + 128]
            out[r0:r0 + T, c] = (o / l).bfloat16()
        r0 += T
    return out


# (lens, heads, qkv) as tests/test_gpu_error_bounds.py and tests/test_gpu_kernels.py build them
def _random(lens, heads, seed):
    return lambda: eb.random_qkv(sum(lens), heads, seed)


ALL_LENS = [1, 2, 31, 32, 33, 127, 128, 129, 160, 161, 255, 256, 257, 1027, 2527]
ATTN_CASES = {
    "ragged-h2": (ALL_LENS, 2, _random(ALL_LENS, 2, 2)),            # seed = heads
    "c4-2527-h2": ([2527], 2, _random([2527], 2, 5)),                       # test_gpu_kernels.test_attention
    "c2-1027-h16": ([1027], 16, lambda: eb.random_qkv(sum(ALL_LENS), 16, 16)[sum(ALL_LENS[:13]):][:1027]),
    "negative-scores": ([300, 1027], 2, lambda: eb.structured_qkv([300, 1027], 2, 31, base=-10.0)),
    "rescale-full-block": ([1027], 2, lambda: eb.structured_qkv([1027], 2, 40, [(0, 300, eb.GAP_ABOVE)])),
    "rescale-masked-pass": ([328], 2, lambda: eb.structured_qkv([328], 2, 40, [(0, 300, eb.GAP_ABOVE)])),
    "rescale-short-block": ([1027], 2, lambda: eb.structured_qkv([1027], 2, 40, [(0, 1025, eb.GAP_ABOVE)])),
    "rescale-twice": ([1027], 2, lambda: eb.structured_qkv([1027], 2, 40, [(0, 300, eb.GAP_ABOVE),
                                                                           (0, 700, 2 * eb.GAP_ABOVE)])),
    "no-rescale-just-below": ([1027], 2, lambda: eb.structured_qkv([1027], 2, 40, [(0, 300, eb.GAP_BELOW)])),
}


@pytest.mark.parametrize("case", list(ATTN_CASES))
def test_attention_bound_accepts_the_kernels_rounding(case):
    lens, heads, make = ATTN_CASES[case]
    qkv = make()
    out = emulate_attention(qkv, lens, heads)
    ref, rest, unit = eb.attention_reference(qkv, lens, heads)
    eb.within(out, ref, rest, unit, eb.C_P / 2, case)


ATTN_DEFECTS = [
    ("drop_last_key", "ragged-h2"), ("drop_last_key", "c4-2527-h2"),
    ("drop_short_block", "c2-1027-h16"), ("drop_short_block", "rescale-short-block"),
    ("key_past_end", "ragged-h2"), ("key_past_end", "negative-scores"),
    ("next_head_k", "ragged-h2"), ("next_head_k", "c2-1027-h16"),
    ("scale_dmodel", "ragged-h2"), ("scale_dmodel", "c2-1027-h16"),
    ("missed_rescale", "rescale-full-block"), ("missed_rescale", "rescale-masked-pass"),
    ("missed_rescale", "rescale-short-block"), ("missed_rescale", "rescale-twice"),
]


@pytest.mark.parametrize("defect,case", ATTN_DEFECTS, ids=[f"{d}-{c}" for d, c in ATTN_DEFECTS])
def test_attention_bound_rejects_planted_defect(defect, case):
    lens, heads, make = ATTN_CASES[case]
    qkv = make()
    out = emulate_attention(qkv, lens, heads, defect=defect)
    ref, rest, unit = eb.attention_reference(qkv, lens, heads)
    with pytest.raises(AssertionError, match="outside the bound"):
        eb.within(out, ref, rest, unit, eb.C_P, defect)


def test_key_past_end_of_the_last_utterance_is_caught_only_with_negative_scores():
    """The zero row the TMA fills in past the last utterance scores 0: against random scores that is one more key
    of average weight, which no bound can tell from rounding, so the GPU tests include an utterance whose scores
    are all negative, where the same defect takes almost all the weight."""
    lens, heads, make = ATTN_CASES["negative-scores"]
    qkv = make()
    out = emulate_attention(qkv, lens, heads, defect="key_past_end")
    ref, rest, unit = eb.attention_reference(qkv, lens, heads)
    last = slice(lens[0], None)
    with pytest.raises(AssertionError, match="outside the bound"):
        eb.within(out[last], ref[last], rest[last], unit[last], eb.C_P, "last utterance")
