"""Quick kernel timing probe (CUDA events) for bring-up: GEMM shapes of the full denoiser,
attention at T=1027/2527, posterior kernel.  Prints TFLOP/s and GB/s."""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tts-with-diffusion-model_b200"))
from vall_e.b200 import lib as L  # noqa: E402

L.load()
dev = "cuda"


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def gemm(M, N, K, epi, dt):
    A = torch.randn(M, K, device=dev).bfloat16()
    W = torch.randn(N, K, device=dev).bfloat16()
    bias = torch.randn(N, device=dev)
    out = torch.empty(M, N, dtype=dt, device=dev)
    res = out if epi == L.EPI_BIAS_RESIDUAL else None
    ms = timeit(lambda: L.gemm_bf16(out, A, W, bias, res, epi))
    ref = timeit(lambda: torch.matmul(A, W.t()))
    print(f"gemm M={M} N={N} K={K} epi={epi}: {ms:.3f} ms {2*M*N*K/ms/1e9:.0f} TFLOP/s | cuBLAS {ref:.3f} ms {2*M*N*K/ref/1e9:.0f}", flush=True)


def attn(lens, heads, variant):
    M = sum(lens)
    d = heads * 64
    qkv = torch.randn(M, 3 * d, device=dev).bfloat16()
    cu = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), dtype=torch.int32, device=dev)
    out = torch.empty(M, d, dtype=torch.bfloat16, device=dev)
    ms = timeit(lambda: L.flash_attn_varlen(out, qkv, cu, max(lens), heads, 0.125, variant=variant))
    fl = sum(4 * T * T * d for T in lens)
    print(f"attn[{variant}] B={len(lens)} T={lens[0]} heads={heads}: {ms:.3f} ms {fl/ms/1e9:.0f} TFLOP/s", flush=True)


def small_kernels():
    sys.path.insert(0, str(ROOT / "tts-with-diffusion-model_b200"))
    from vall_e.vall_e import d3pm
    M, d = 262912, 1024
    x = torch.randn(M, d, device=dev)
    table = torch.randn(52, 2 * d, device=dev)
    out = torch.empty(M, d, dtype=torch.bfloat16, device=dev)
    lv = torch.full((256,), 7, dtype=torch.int32, device=dev)
    ru = torch.arange(256, dtype=torch.int32, device=dev).repeat_interleave(1027)
    ms = timeit(lambda: L.adaln(out, x, table, lv, ru))
    print(f"adaln M={M} d={d}: {ms:.3f} ms {M*d*6/ms/1e6:.0f} GB/s", flush=True)
    S, K, rows = 51, 1024, 192000
    tab = d3pm.scalar_table(S, K, "absorbing").to(dev)
    logits = torch.randn(rows, 8 * K, device=dev).half()
    x_t = torch.full((rows, 8), K // 2, dtype=torch.int32, device=dev)
    row_utt = torch.arange(256, dtype=torch.int32, device=dev).repeat_interleave(750)
    utt = torch.zeros(256, L.U_STRIDE, dtype=torch.int32, device=dev)
    utt[:, L.U_RESP0] = torch.arange(256, device=dev, dtype=torch.int32) * 750
    t_utt = torch.full((256,), 30, dtype=torch.int32, device=dev)
    o = torch.empty(rows, 8, dtype=torch.int32, device=dev)
    for name, mode in (("philox-icdf", L.NOISE_PHILOX), ("greedy", L.NOISE_GREEDY)):
        ms = timeit(lambda: L.posterior_sample_from_logits(o, None, logits, 8 * K, x_t, row_utt, t_utt, utt, tab, rows, 8,
                                                           K, L.ABSORBING, mode, seed=1), iters=5)
        print(f"posterior[{name}] tokens={rows*8}: {ms:.3f} ms {rows*8*(2*K+8)/ms/1e6:.0f} GB/s", flush=True)


def head():
    """classifier + reverse step: fused (vb200_head_posterior_sample) and as gemm_bf16 + posterior_sample_from_logits"""
    sys.path.insert(0, str(ROOT / "tts-with-diffusion-model_b200"))
    from vall_e.vall_e import d3pm
    S, K, d = 51, 1024, 1024
    tab = d3pm.scalar_table(S, K, "absorbing").to(dev)
    W = (torch.randn(8 * K, d, device=dev) * 0.03).bfloat16()
    bias = torch.randn(8 * K, device=dev)
    for B in (256, 1):
        rows = 750 * B
        head_in = torch.randn(rows, d, device=dev).bfloat16()
        scratch = torch.empty(rows, 8 * K, dtype=torch.float16, device=dev)
        x_t = torch.full((rows, 8), K // 2, dtype=torch.int32, device=dev)
        row_utt = torch.arange(B, dtype=torch.int32, device=dev).repeat_interleave(750)
        utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=dev)
        utt[:, L.U_RESP0] = torch.arange(B, device=dev, dtype=torch.int32) * 750
        t_utt = torch.full((B,), 30, dtype=torch.int32, device=dev)
        o = torch.empty(rows, 8, dtype=torch.int32, device=dev)
        def unfused():
            L.gemm_bf16(scratch, head_in, W, bias, None, L.EPI_BIAS)
            L.posterior_sample_from_logits(o, None, scratch, 8 * K, x_t, row_utt, t_utt, utt, tab, rows, 8, K,
                                           L.ABSORBING, L.NOISE_PHILOX, seed=1)
        for form, fn in (("fused", lambda: L.head_posterior_sample(o, None, head_in, W, bias, x_t, row_utt, t_utt, utt,
                                                                    tab, 8, K, L.ABSORBING, L.NOISE_PHILOX, seed=1)),
                         ("gemm+posterior", unfused)):
            ms = timeit(fn, iters=10)
            print(f"head+posterior[{form}] rows={rows}: {ms:.3f} ms "
                  f"({2*rows*8*K*d/ms/1e9:.0f} TFLOP/s of GEMM work)", flush=True)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what == "head":
        head()
    if what in ("all", "small"):
        small_kernels()
    if what in ("all", "gemm"):
        for B in (1, 32):
            M = 1027 * B
            gemm(M, 3072, 1024, L.EPI_NONE, torch.bfloat16)
            gemm(M, 1024, 1024, L.EPI_BIAS_RESIDUAL, torch.float32)
            gemm(M, 4096, 1024, L.EPI_BIAS_GELU, torch.bfloat16)
            gemm(M, 1024, 4096, L.EPI_BIAS_RESIDUAL, torch.float32)
        gemm(750 * 32, 8192, 1024, L.EPI_BIAS, torch.float16)
    if what in ("all", "attn"):
        import os
        print("VB200_ATTN_VARIANT", os.environ.get("VB200_ATTN_VARIANT"))
        attn([1027] * 32, 16, "tmem")
        attn([2527] * 8, 16, "tmem")
        attn([1027] * 256, 16, "tmem")
