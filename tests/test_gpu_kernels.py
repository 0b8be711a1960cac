"""GPU parity tests, kernel level: every entry point of libvalle_b200.so against the oracle /
a plain torch fp32 evaluation of the same op.  Run on the B200 box: pytest -m gpu."""
import math

import numpy as np
import pytest
import torch

import error_bounds as eb
import head_bounds as hb

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


def _oracle_law(orc, logits16_row, x_t, t):
    """softmax of the ORACLE's posterior logits (reference q_posterior_logits, dense fp16 tables) for one
    token: the law every sampler of this library is tested against."""
    lg = logits16_row.view(1, 1, -1).to(torch.float16)
    post = orc.q_posterior_logits(lg, torch.tensor([[x_t]], dtype=torch.int32), torch.tensor([t]))
    return torch.softmax(post.double(), -1).view(-1)


def _assert_draws_follow(draws, law, ctx):
    """chi-square of the observed class counts against ``law`` (cells with expectation <= 5 pooled)."""
    n, K = draws.numel(), law.numel()
    counts = torch.bincount(draws.view(-1).cpu().long(), minlength=K).double()
    expected = law * n
    keep = expected > 5
    chi2 = (((counts - expected) ** 2) / expected)[keep].sum().item()
    cells = int(keep.sum().item())
    rest_obs, rest_exp = counts[~keep].sum().item(), expected[~keep].sum().item()
    if rest_exp > 5:
        chi2 += (rest_obs - rest_exp) ** 2 / rest_exp
        cells += 1
    dof = max(cells - 1, 1)
    assert chi2 < dof + 6 * math.sqrt(2 * dof), (ctx, chi2, dof)


def _rand_bf16(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16).to(DEV)


# ---------------------------------------------------------------- GEMM
GEMM_SHAPES = [(128, 256, 64), (300, 256, 128), (1027, 3072, 1024), (1027, 1024, 4096),
               (77, 8200, 256), (4096, 4096, 1024), (1, 64, 64), (257, 72, 200),
               (300, 384, 128), (130, 192, 64)]          # N % 192 == 0, one wave: the 128x192 tiling (16-bit outputs)


@pytest.mark.parametrize("simt", [False, True], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_gemm_plain(L, M, N, K, simt):
    A, W = _rand_bf16((M, K), 1), _rand_bf16((N, K), 2, K ** -0.5)
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        out = torch.full((M, N), float("nan"), dtype=dt, device=DEV)
        L.gemm_bf16(out, A, W, epi=L.EPI_NONE, simt=simt)
        torch.cuda.synchronize()
        eb.check_gemm(out, A, W, ctx=str(dt))


@pytest.mark.parametrize("simt", [False, True], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("M,N,K", [(515, 1024, 512), (515, 768, 512),
                                   (1027, 3072, 256)])     # the last: 144 tiles of 128x192 (16-bit outputs), one wave
def test_gemm_epilogues(L, simt, M, N, K):
    A, W = _rand_bf16((M, K), 3), _rand_bf16((N, K), 4, K ** -0.5)
    g = torch.Generator().manual_seed(5)
    bias = torch.randn(N, generator=g).to(DEV)
    resid = torch.randn(M, N, generator=g).to(DEV)
    out = torch.empty(M, N, dtype=torch.float16, device=DEV)
    L.gemm_bf16(out, A, W, bias, epi=L.EPI_BIAS, simt=simt)
    eb.check_gemm(out, A, W, L.EPI_BIAS, bias, ctx="bias")
    out = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
    L.gemm_bf16(out, A, W, bias, epi=L.EPI_BIAS_GELU, simt=simt)
    eb.check_gemm(out, A, W, L.EPI_BIAS_GELU, bias, ctx="gelu")
    x = resid.clone()
    L.gemm_bf16(x, A, W, bias, residual=x, epi=L.EPI_BIAS_RESIDUAL, simt=simt)   # in place, as the model uses it
    eb.check_gemm(x, A, W, L.EPI_BIAS_RESIDUAL, bias, resid, ctx="residual")


def test_gemm_rejects_bad_arguments(L):
    A, W = _rand_bf16((8, 12), 1), _rand_bf16((16, 12), 2)
    out = torch.empty(8, 16, dtype=torch.float32, device=DEV)
    with pytest.raises(L.VB200Error):
        L.gemm_bf16(out, A, W)                       # K % 8 != 0
    A, W = _rand_bf16((8, 16), 1), _rand_bf16((16, 16), 2)
    with pytest.raises(L.VB200Error):
        L.gemm_bf16(out, A, W, epi=L.EPI_BIAS)       # bias missing


def test_misaligned_bias_is_refused(L):
    """The GEMM epilogues read bias with float4 loads: a bias that is not 16-byte aligned is refused before any
    launch, by the GEMM, the fused classifier + reverse step and the fused cross-entropy."""
    rows, d, K = 64, 64, 256
    head_in, W = _rand_bf16((rows, d), 1), _rand_bf16((K, d), 2)
    bias = torch.zeros(K + 1, device=DEV)[1:]
    with pytest.raises(L.VB200Error, match="aligned"):
        L.gemm_bf16(torch.empty(rows, K, device=DEV), head_in, W, bias, epi=L.EPI_BIAS)
    from vall_e.vall_e import d3pm as pd
    table = pd.scalar_table(10, K, "absorbing").to(DEV)
    x_t = torch.zeros(rows, 1, dtype=torch.int32, device=DEV)
    row_utt = torch.zeros(rows, dtype=torch.int32, device=DEV)
    t_utt = torch.tensor([3], dtype=torch.int32, device=DEV)
    utt = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    assert L.head_fused(d, K, L.NOISE_GREEDY)
    with pytest.raises(L.VB200Error, match="aligned"):
        L.head_posterior_sample(torch.empty(rows, 1, dtype=torch.int32, device=DEV), None, head_in, W, bias, x_t,
                                row_utt, t_utt, utt, table, 1, K, L.ABSORBING, L.NOISE_GREEDY)
    with pytest.raises(L.VB200Error, match="aligned"):
        L.head_ce_loss(torch.empty(rows, 1, device=DEV), head_in, W, bias, x_t, 1, K)


# ---------------------------------------------------------------- attention
@pytest.mark.parametrize("variant", ["tmem", "simt"])
@pytest.mark.parametrize("lens,heads", [([5], 1), ([128], 2), ([129, 64, 300], 2), ([1027], 4), ([257, 1, 640], 3), ([256, 255, 385, 16, 17], 2), ([2527], 2)])
def test_attention(L, variant, lens, heads):
    M, d = sum(lens), heads * 64
    qkv = _rand_bf16((M, 3 * d), 5)
    cu = torch.tensor([0] + list(np.cumsum(lens)), dtype=torch.int32, device=DEV)
    out = torch.full((M, d), float("nan"), dtype=torch.bfloat16, device=DEV)
    L.flash_attn_varlen(out, qkv, cu, max(lens), heads, 64 ** -0.5, variant=variant)
    torch.cuda.synchronize()
    eb.check_attention(out, qkv, lens, heads)


@pytest.mark.parametrize("amp", [1.0, 5.0])
def test_attention_last_block_lengths(L, amp):
    """Every shape of the ragged end: a last key block of 1 .. 32 keys takes the one-chunk path (also as the
    ONLY block, T <= 32), 33 .. 127 the masked 128-key pass, 128 none; with amp = 5 the scores spread over
    ~2^60, so the row maximum moves in late blocks too (rescale of O in TMEM from the short block)."""
    lens = [1, 15, 16, 17, 31, 32, 33, 128 + 1, 128 + 16, 128 + 17, 128 + 32, 128 + 33, 256 + 3, 128 + 95, 128 + 127, 384]
    heads = 2
    M, d = sum(lens), heads * 64
    qkv = (_rand_bf16((M, 3 * d), 11).float() * amp).bfloat16()
    cu = torch.tensor([0] + list(np.cumsum(lens)), dtype=torch.int32, device=DEV)
    out = torch.full((M, d), float("nan"), dtype=torch.bfloat16, device=DEV)
    L.flash_attn_varlen(out, qkv, cu, max(lens), heads, 64 ** -0.5)
    torch.cuda.synchronize()
    eb.check_attention(out, qkv, lens, heads, f"amp {amp}")


def test_attention_output_does_not_depend_on_the_batch(L):
    """An utterance's attention output is the same bits whether it is launched alone (a one-wave grid: padded to one
    CTA per SM and launched with PDL) or inside a batch that fills the GPU several times over — what the
    batch-composition invariance of the generated codes rests on."""
    heads, d = 2, 128
    lens = [300, 1027, 17, 131, 64, 200] * 5                 # 30 utterances: 9 x 2 x 30 CTAs
    M = sum(lens)
    qkv = _rand_bf16((M, 3 * d), 21)
    cu = torch.tensor([0] + list(np.cumsum(lens)), dtype=torch.int32, device=DEV)
    big = torch.empty(M, d, dtype=torch.bfloat16, device=DEV)
    L.flash_attn_varlen(big, qkv, cu, max(lens), heads, 64 ** -0.5)
    eb.check_attention(big, qkv, lens, heads)
    r0 = 0
    for T in lens[:6]:                                       # each utterance alone
        one = torch.empty(T, d, dtype=torch.bfloat16, device=DEV)
        L.flash_attn_varlen(one, qkv[r0:r0 + T].contiguous(), torch.tensor([0, T], dtype=torch.int32, device=DEV), T, heads, 64 ** -0.5)
        assert torch.equal(one, big[r0:r0 + T]), T
        r0 += T


# ---------------------------------------------------------------- elementwise
def test_adaln_layernorm_gather(L):
    from oracle import denoiser as on
    M, d, B = 333, 1024, 3
    g = torch.Generator().manual_seed(6)
    x = (torch.randn(M, d, generator=g) * 3 + 0.5)
    emb = torch.randn(7, 2 * d, generator=g) * 0.1
    row_utt = torch.sort(torch.randint(0, B, (M,), generator=g)).values.to(torch.int32)
    lv = torch.tensor([3, 0, 6], dtype=torch.int32)
    ref = on.adaln(x[:, None, :], emb, lv[row_utt.long()].long())[:, 0]
    table = torch.cat([emb[:, :d].exp(), emb[:, d:]], dim=-1).to(DEV)
    out = torch.empty(M, d, dtype=torch.bfloat16, device=DEV)
    L.adaln(out, x.to(DEV), table, lv.to(DEV), row_utt.to(DEV))
    # output is bf16: allow one bf16 ulp (2^-7 relative) on top of fp32 round-off
    assert ((out.float().cpu() - ref).abs() <= ref.abs() * 2 ** -7 + 1e-3).all()
    w, b = torch.randn(d, generator=g), torch.randn(d, generator=g)
    ref = torch.nn.functional.layer_norm(x, (d,), w, b, 1e-5)
    L.layernorm(out, x.to(DEV), w.to(DEV), b.to(DEV))
    assert ((out.float().cpu() - ref).abs() <= ref.abs() * 2 ** -7 + 1e-3).all()
    idx = torch.tensor([5, 0, 332, 17], dtype=torch.int32)
    o2 = torch.empty(4, d, dtype=torch.bfloat16, device=DEV)
    L.gather_rows_bf16(o2, x.to(DEV), idx.to(DEV))
    assert torch.equal(o2.cpu(), x[idx.long()].bfloat16())


# ---------------------------------------------------------------- D3PM: q_sample / posterior
@pytest.fixture(scope="module", params=["absorbing", "uniform"])
def d3pm_pair(request):
    from oracle.d3pm import D3PM
    from vall_e.vall_e import d3pm as pd
    S, K = 100, 1025
    return request.param, D3PM(S, K, request.param), pd.scalar_table(S, K, request.param).to(DEV), S, K


def test_q_sample_bit_exact_vs_oracle(L, d3pm_pair):
    import detrand
    tr, orc, table, S, K = d3pm_pair
    B, W = 12, 64
    t = torch.tensor([0, 1, 5, 10, 25, 50, 75, 90, 97, 98, 99, 99])
    x0 = torch.from_numpy(detrand.integers(11, 0, K, (B, W)))
    x0[:, 0] = K // 2
    mask = torch.ones(W, dtype=torch.int64)
    mask[-5:] = 0
    noise = torch.from_numpy(detrand.uniform(12, (B, W, K)))
    ref = orc.q_sample(x0, t, mask, noise)
    got = _q_sample_cuda(L, tr, table, S, K, x0, t, mask, noise)
    mism = (got != ref).sum().item()
    assert mism == 0, f"{tr}: {mism} of {B * W} tokens differ"


def _q_sample_cuda(L, tr, table, S, K, x0, t, mask, noise):
    """absorbing: per-timestep scalars (the fp16 chain product is exactly rank-structured);
    uniform: the dense fp16 log(Qbar + eps) table (its K-term sums are not — DESIGN.md §2)."""
    from vall_e.vall_e import d3pm as pd
    B, W = x0.shape
    out = torch.empty(B * W, dtype=torch.int32, device=DEV)
    args = (out, x0.to(DEV, torch.int32).view(-1).contiguous(), t.to(DEV, torch.int32).repeat_interleave(W),
            mask.to(DEV, torch.int32).expand(B, W).contiguous().view(-1), noise.to(DEV).contiguous())
    if tr == "absorbing":
        L.q_sample(*args, table, K, L.ABSORBING)
    else:
        L.q_sample_dense(*args, pd.dense_log_qbar(S, K, "uniform").to(DEV))
    return out.cpu().view(B, W).long()


def test_q_sample_bit_exact_sweep_100k_tokens(L, d3pm_pair):
    """north_star: forward noising from supplied uniforms is bit-exact.  128 000 tokens, every timestep
    0..S-1, both transitions: ZERO tokens may differ from the oracle (reference ar_discrete.py:467-487)."""
    import detrand
    tr, orc, table, S, K = d3pm_pair
    W, total = 160, 0
    t = torch.arange(S)
    mask = torch.ones(W, dtype=torch.int64)
    for rep in range(8):
        x0 = torch.from_numpy(detrand.integers(300 + rep, 0, K, (S, W)))
        x0[:, rep] = K // 2
        noise = torch.from_numpy(detrand.uniform(400 + rep, (S, W, K)))
        ref = orc.q_sample(x0, t, mask, noise)
        got = _q_sample_cuda(L, tr, table, S, K, x0, t, mask, noise)
        mism = int((got != ref).sum())
        assert mism == 0, f"{tr}: {mism} of {S * W} tokens differ (rep {rep})"
        total += S * W
    assert total >= 100_000


def test_posterior_vs_oracle(L, d3pm_pair):
    import detrand
    from oracle.d3pm import posterior_fp32
    tr, orc, table, S, K = d3pm_pair
    B, W = 10, 48
    t = torch.tensor([0, 1, 2, 10, 30, 50, 70, 90, 98, 99])
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    x0 = torch.from_numpy(detrand.integers(21, 0, K, (B, W)))
    x_t = orc.q_sample(x0, t, torch.ones(W, dtype=torch.int64), torch.from_numpy(detrand.uniform(22, (B, W, K))))
    logits16 = torch.from_numpy(detrand.normal(23, (B, W, K)) * 2.5).to(torch.float16)
    noise = torch.from_numpy(detrand.uniform(24, (B, W, K)))
    ref_samp, ref_post16 = orc.p_sample(logits16, t, x_t.to(torch.int32), noise)
    ref_greedy, _ = orc.p_sample(logits16, t, x_t.to(torch.int32), greedy=True)
    ref_post32 = posterior_fp32(logits16, x_t, t, orc)

    row_utt = torch.arange(B, dtype=torch.int32, device=DEV).repeat_interleave(W)
    utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV)
    common = dict(ld_logits=K, x_t=x_t.to(DEV, torch.int32).view(-1).contiguous(), row_utt=row_utt,
                  t_utt=t.to(DEV, torch.int32), utt=utt, table=table, n_rows=B * W, n_levels=1, K=K,
                  transition=code)
    lg = logits16.to(DEV).view(B * W, K).contiguous()
    post = torch.empty(B * W, K, dtype=torch.float32, device=DEV)
    out = torch.empty(B * W, dtype=torch.int32, device=DEV)
    L.posterior_sample_from_logits(out, post, lg, noise=L.NOISE_GREEDY, **common)
    post = post.cpu().view(B, W, K)
    greedy = out.cpu().view(B, W).long()
    # posterior: KL(reference || ours) <= 1e-3 per token, against the reference's fp16 pipeline
    p_ref = torch.softmax(ref_post16.float(), -1)
    kl = (p_ref * (torch.log_softmax(ref_post16.float(), -1) - torch.log_softmax(post, -1))).sum(-1)
    assert kl.max().item() <= 1e-3, kl.max().item()
    # and tightly against the same dense algorithm evaluated in fp32 (rows with t == 0 are raw logits)
    nz = t != 0
    assert (post[nz] - ref_post32[nz]).abs().max().item() < 2e-3
    assert torch.equal(post[~nz], logits16[~nz].float())
    # greedy codes: bit-exact wherever the reference's top-2 margin exceeds the fp16 resolution
    top2 = ref_post16.float().topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05
    assert clear.float().mean().item() > 0.5
    assert torch.equal(greedy[clear], ref_greedy[clear])
    # supplied uniforms: same argmax wherever the noisy top-2 margin is clear
    L.posterior_sample_from_logits(out, None, lg, noise=L.NOISE_UNIFORMS, uniforms=noise.to(DEV).view(B * W, K).contiguous(), **common)
    samp = out.cpu().view(B, W).long()
    gn = -torch.log(-torch.log(noise.clamp(min=torch.finfo(torch.float32).tiny)))
    noisy = ref_post16.float() + (t != 0).float().view(B, 1, 1) * gn
    top2 = noisy.topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05
    assert torch.equal(samp[clear], ref_samp[clear])
    assert (samp != ref_samp).float().mean().item() < 0.05


def test_posterior_golden_fixture(L, golden_dir):
    """Against outputs of the reference's own p_sample / q_posterior_logits (make_golden.py)."""
    import detrand
    from vall_e.vall_e import d3pm as pd
    for tr, code in (("absorbing", L.ABSORBING), ("uniform", L.UNIFORM)):
        z = np.load(golden_dir / f"d3pm_{tr}_k1025.npz")
        S, K, W, seed = int(z["S"]), int(z["K"]), int(z["W"]), int(z["seed"])
        t = torch.from_numpy(z["q_t"])
        B = len(t)
        table = pd.scalar_table(S, K, tr).to(DEV)
        logits = torch.from_numpy(detrand.normal(seed + 2, (B, W, K)) * 2.0).to(torch.float16)
        x_in = torch.from_numpy(z["q_xt"])
        out = torch.empty(B * W, dtype=torch.int32, device=DEV)
        post = torch.empty(B * W, K, dtype=torch.float32, device=DEV)
        L.posterior_sample_from_logits(
            out, post, logits.to(DEV).view(B * W, K).contiguous(), K, x_in.to(DEV, torch.int32).view(-1).contiguous(),
            torch.arange(B, dtype=torch.int32, device=DEV).repeat_interleave(W), t.to(DEV, torch.int32),
            torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV), table, B * W, 1, K, code, L.NOISE_GREEDY)
        post = post.cpu().view(B, W, K)[:, :6]
        ref = torch.from_numpy(z["p_post_head"]).float()
        p_ref = torch.softmax(ref, -1)
        kl = (p_ref * (torch.log_softmax(ref, -1) - torch.log_softmax(post, -1))).sum(-1)
        assert kl.max().item() <= 1e-3
        greedy = out.cpu().view(B, W)
        same = (greedy == torch.from_numpy(z["p_greedy"])).float().mean().item()
        assert same > 0.97, same
        # q_sample golden (reference uniforms regenerated from the seed)
        x0 = torch.from_numpy(detrand.integers(seed, 0, 1024, (B, W)))
        x0[:, 0] = K // 2
        x0[:, 1] = 1024
        mask = torch.ones(W, dtype=torch.int32)
        mask[-3:] = 0
        nq = torch.from_numpy(detrand.uniform(seed + 1, (B, W, K)))
        xo = _q_sample_cuda(L, tr, table, S, K, x0, t, mask, nq)
        mism = (xo != torch.from_numpy(z["q_xt"]).long()).sum().item()
        if mism and tr == "uniform":
            # The fixture was made where the reference ran; the uniform chain product's last bit depends on
            # that CPU's fp16 GEMM summation order.  Only if THIS box's oracle does not reproduce the fixture
            # either may the kernel differ from it — and then it must equal the oracle on this box's tables.
            from oracle.d3pm import D3PM
            here = D3PM(S, K, tr).q_sample(x0, t, mask.long(), nq)
            assert not torch.equal(here, torch.from_numpy(z["q_xt"]).long()), "oracle matches the fixture, kernel does not"
            assert torch.equal(xo, here)
        else:
            assert mism == 0, (tr, mism)                # the reference's own q_sample output, bit for bit


def test_philox_sampling_matches_posterior_distribution(L):
    """Stochastic samples must match in distribution: chi-square of Philox Gumbel-max draws."""
    from vall_e.vall_e import d3pm as pd
    S, K, n = 50, 64, 40000
    table = pd.scalar_table(S, K, "absorbing").to(DEV)
    from oracle.d3pm import D3PM
    g = torch.Generator().manual_seed(3)
    row = (torch.randn(K, generator=g) * 1.5).half().float()          # fp16-representable: the oracle takes fp16 logits
    logits = row.repeat(n, 1).to(DEV)
    x_t = torch.full((n,), K // 2, dtype=torch.int32, device=DEV)
    utt = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    row_utt = torch.zeros(n, dtype=torch.int32, device=DEV)
    t_utt = torch.tensor([20], dtype=torch.int32, device=DEV)
    out = torch.empty(n, dtype=torch.int32, device=DEV)
    post = torch.empty(n, K, dtype=torch.float32, device=DEV)
    L.posterior_sample_from_logits(out, post, logits, K, x_t, row_utt, t_utt, utt, table, n, 1, K, L.ABSORBING,
                                   L.NOISE_PHILOX, seed=77)
    _assert_draws_follow(out, _oracle_law(D3PM(S, K, "absorbing"), row, K // 2, 20), "generic kernel, K=64")
    out2 = torch.empty_like(out)
    L.posterior_sample_from_logits(out2, None, logits, K, x_t, row_utt, t_utt, utt, table, n, 1, K, L.ABSORBING,
                                   L.NOISE_PHILOX, seed=77)
    assert torch.equal(out, out2)           # counter-based: reproducible


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
@pytest.mark.parametrize("K", [256, 1024])
def test_fast_posterior_kernel_matches_generic(L, transition, K):
    """The register-resident production kernel (K % 256 == 0) against the generic log-domain kernel:
    identical greedy codes, and inverse-CDF draws distributed as the posterior (chi-square)."""
    from vall_e.vall_e import d3pm as pd
    S = 40
    code = L.ABSORBING if transition == "absorbing" else L.UNIFORM
    table = pd.scalar_table(S, K, transition).to(DEV)
    g = torch.Generator().manual_seed(K)
    # (a) greedy equality on varied rows / timesteps / x_t (masked and unmasked)
    rows, levels = 300, 2
    logits = (torch.randn(rows, levels * K, generator=g) * 3).half().to(DEV)
    x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
    x_t[::3] = K // 2
    x_t = x_t.to(DEV)
    B = 6
    row_utt = (torch.arange(rows, dtype=torch.int32) % B).sort().values.to(DEV)
    t_utt = torch.tensor([0, 1, 5, 20, 38, 39], dtype=torch.int32, device=DEV)
    utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV)
    fast = torch.empty(rows, levels, dtype=torch.int32, device=DEV)
    slow = torch.empty_like(fast)
    post = torch.empty(rows * levels, K, dtype=torch.float32, device=DEV)
    args = (levels * K, x_t, row_utt, t_utt, utt, table, rows, levels, K, code)
    L.posterior_sample_from_logits(fast, None, logits, *args, L.NOISE_GREEDY)
    L.posterior_sample_from_logits(slow, post, logits, *args, L.NOISE_GREEDY)
    top2 = post.topk(2, dim=-1).values
    clear = ((top2[:, 0] - top2[:, 1]) > 1e-3).view(rows, levels)
    assert clear.float().mean().item() > 0.9
    assert torch.equal(fast[clear], slow[clear])
    # (b) distribution of the inverse-CDF sampler against the ORACLE's posterior law, masked and unmasked
    # current token, early / middle / last timestep
    from oracle.d3pm import D3PM
    orc = D3PM(S, K, transition)
    n = 40000
    row = (torch.randn(K, generator=g) * 2.0).half()
    lg = row.repeat(n, 1).to(DEV)
    for t_val in (1, 17, S - 1):
        for xt_val in (K // 2, 3):
            xt = torch.full((n, 1), xt_val, dtype=torch.int32, device=DEV)
            ru = torch.zeros(n, dtype=torch.int32, device=DEV)
            tu = torch.tensor([t_val], dtype=torch.int32, device=DEV)
            u1 = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
            out = torch.empty(n, 1, dtype=torch.int32, device=DEV)
            L.posterior_sample_from_logits(out, None, lg, K, xt, ru, tu, u1, table, n, 1, K, code, L.NOISE_PHILOX, seed=5)
            _assert_draws_follow(out, _oracle_law(orc, row, xt_val, t_val), (transition, K, t_val, xt_val))


def test_head_posterior_sample_fused_vs_separate_kernels(L):
    """vb200_head_posterior_sample (SURVEY §8a rows H1 + P; the reverse step as the classifier GEMM's
    epilogue, streaming reservoir sampling) against classifier GEMM + vb200_posterior_sample_from_logits:
    greedy codes agree wherever the posterior's top-2 margin is clear, the call is reproducible, and
    sampled codes are distributed as the posterior the generic kernel reports (chi-square)."""
    from vall_e.vall_e import d3pm as pd
    S, B = 30, 5
    g = torch.Generator().manual_seed(11)
    for transition, code in (("absorbing", L.ABSORBING), ("uniform", L.UNIFORM)):
        for K, levels, d, rows in ((256, 8, 128, 333), (1024, 2, 64, 600)):
            table = pd.scalar_table(S, K, transition).to(DEV)
            head_in = torch.randn(rows, d, generator=g).bfloat16().to(DEV)
            W = (torch.randn(levels * K, d, generator=g) * 0.3).bfloat16().to(DEV)
            bias = torch.randn(levels * K, generator=g).to(DEV)
            x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
            x_t[::2] = K // 2
            x_t = x_t.to(DEV)
            row_utt = (torch.arange(rows, dtype=torch.int32) % B).sort().values.to(DEV)
            t_utt = torch.tensor([0, 7, 15, 28, 29], dtype=torch.int32, device=DEV)
            utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV)
            utt[:, L.U_GID] = torch.arange(B, dtype=torch.int32, device=DEV) + 100
            scratch = torch.empty(rows, levels * K, dtype=torch.float16, device=DEV)
            lg = torch.empty_like(scratch)
            L.gemm_bf16(lg, head_in, W, bias, None, L.EPI_BIAS)
            post = torch.empty(rows * levels, K, dtype=torch.float32, device=DEV)
            ref = torch.empty(rows, levels, dtype=torch.int32, device=DEV)
            L.posterior_sample_from_logits(ref, post, lg, levels * K, x_t, row_utt, t_utt, utt, table, rows,
                                           levels, K, code, L.NOISE_GREEDY)
            out = torch.empty_like(ref)
            L.head_posterior_sample(out, scratch, head_in, W, bias, x_t, row_utt, t_utt, utt, table, levels, K,
                                    code, L.NOISE_GREEDY)
            top2 = post.topk(2, dim=-1).values
            clear = ((top2[:, 0] - top2[:, 1]) > 2e-2).view(rows, levels)      # logits differ by fp16 rounding
            assert clear.float().mean().item() > 0.8
            assert torch.equal(out[clear], ref[clear]), (transition, K)
            a = torch.empty_like(ref)
            b = torch.empty_like(ref)
            for dst, seed in ((a, 3), (b, 3)):
                L.head_posterior_sample(dst, scratch, head_in, W, bias, x_t, row_utt, t_utt, utt, table, levels, K,
                                        code, L.NOISE_PHILOX, seed=seed)
            assert torch.equal(a, b)                                           # counter-based: reproducible
            assert 0 <= int(a.min()) and int(a.max()) < K
            t0 = (row_utt == 0)                                                # t == 0: argmax of the raw logits
            assert torch.equal(a[t0][clear[t0]], ref[t0][clear[t0]])
    # distribution: n tokens with the same logits row (same head_in row), masked and unmasked x_t
    n, K, d = 30000, 1024, 64
    table = pd.scalar_table(S, K, "absorbing").to(DEV)
    row = torch.randn(1, d, generator=g).bfloat16()
    head_in = row.repeat(n, 1).to(DEV)
    W = (torch.randn(K, d, generator=g) * 0.35).bfloat16().to(DEV)
    bias = torch.randn(K, generator=g).to(DEV)
    ru = torch.zeros(n, dtype=torch.int32, device=DEV)
    tu = torch.tensor([17], dtype=torch.int32, device=DEV)
    u1 = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    scratch = torch.empty(n, K, dtype=torch.float16, device=DEV)
    from oracle.d3pm import D3PM
    orc = D3PM(S, K, "absorbing")
    row16 = (row.float() @ W.float().cpu().t() + bias.cpu()).view(-1).to(torch.float16)    # the token's logits, as the oracle takes them
    for xt_val in (K // 2, 3):
        xt = torch.full((n, 1), xt_val, dtype=torch.int32, device=DEV)
        out = torch.empty(n, 1, dtype=torch.int32, device=DEV)
        L.head_posterior_sample(out, scratch, head_in, W, bias, xt, ru, tu, u1, table, 1, K, L.ABSORBING,
                                L.NOISE_PHILOX, seed=5)
        _assert_draws_follow(out, _oracle_law(orc, row16, xt_val, 17), ("fused head", xt_val))


@pytest.mark.parametrize("act", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
@pytest.mark.parametrize("rows,K,levels,d", [(77, 1024, 8, 128), (600, 512, 3, 64), (1000, 256, 1, 256)])
def test_head_ce_loss_matches_torch(L, rows, K, levels, d, act):
    """vb200_head_ce_loss (cross-entropy as the classifier GEMM's epilogue, no logits in memory) against the
    float64 cross-entropy of the same 16-bit operands (both bf16 or both fp16), within the bound of
    tests/head_bounds.py."""
    g = torch.Generator().manual_seed(rows)
    head_in = torch.randn(rows, d, generator=g).to(act).to(DEV)
    W = (torch.randn(levels * K, d, generator=g) * 0.4).bfloat16().to(act).to(DEV)
    bias = torch.randn(levels * K, generator=g).to(DEV)
    tgt = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32).to(DEV)
    tgt[0, 0], tgt[-1, -1] = 0, K - 1                    # first / last class of a level
    loss = torch.full((rows, levels), float("nan"), device=DEV)
    L.head_ce_loss(loss, head_in, W, bias, tgt, levels, K)
    for lv, ref, bound in hb.level_references(head_in, W, bias, levels, K):
        r, rest, unit = hb.ce_reference(ref, bound, tgt[:, lv])
        eb.within(loss[:, lv], r, rest, unit, hb.C_CE, f"CE rows={rows} K={K} level {lv}")


def test_q_sample_philox_uniform_transition_law(L):
    """O(1) Philox q_sample, uniform transition: P(keep) and the spread over the other classes."""
    from vall_e.vall_e import d3pm as pd
    K, S, n, t0, x0 = 64, 20, 400000, 9, 17
    table = pd.scalar_table(S, K, "uniform").to(DEV)
    out = torch.empty(n, dtype=torch.int32, device=DEV)
    L.q_sample_philox(out, torch.full((n,), x0, dtype=torch.int32, device=DEV),
                      torch.full((n,), t0, dtype=torch.int32, device=DEV), None, table, K, L.UNIFORM, seed=4)
    row = table[t0].cpu().double()
    w_keep, w_off = math.exp(row[L.TAB_LOG_KEEP].item()), math.exp(row[L.TAB_LOG_OFF].item())
    p_keep = w_keep / (w_keep + (K - 1) * w_off)
    counts = torch.bincount(out.cpu().long(), minlength=K).double()
    assert abs(counts[x0].item() - p_keep * n) < 6 * math.sqrt(n * p_keep * (1 - p_keep)) + 1
    others = torch.cat([counts[:x0], counts[x0 + 1:]])
    exp_o = (n - p_keep * n) / (K - 1)
    chi2 = (((others - exp_o) ** 2) / exp_o).sum().item()
    assert chi2 < (K - 2) + 6 * math.sqrt(2 * (K - 2)), chi2
    assert int(out.min()) >= 0 and int(out.max()) < K


# ---------------------------------------------------------------- fp16 activations next to bf16 weights
def test_fp16_activations(L):
    """The GEMM operands may both be fp16 instead of bf16 (tcgen05 kind::f16 wants rows and weights in ONE
    format), and the norm / gather kernels write fp16 rows for them.  Same references as the bf16 cases,
    with fp16's tolerance; conversions saturate instead of producing inf; mixed formats are refused."""
    from oracle import denoiser as on
    # GEMM with an fp16 A operand, every tiling the launcher may pick, both kernels
    for (M, N, K), epi, dt in (((1027, 3072, 1024), L.EPI_NONE, torch.bfloat16), ((1027, 1024, 4096), L.EPI_BIAS_RESIDUAL, torch.float32),
                               ((4200, 4096, 1024), L.EPI_BIAS_GELU, torch.float16), ((257, 72, 200), L.EPI_BIAS, torch.float32)):
        g = torch.Generator().manual_seed(M)
        A = (torch.randn(M, K, generator=g)).to(torch.float16).to(DEV)
        W = _rand_bf16((N, K), 2, K ** -0.5).to(torch.float16)
        bias = torch.randn(N, generator=g).to(DEV)
        resid = torch.randn(M, N, generator=g).to(DEV)
        for simt in (False, True):
            out = resid.clone() if epi == L.EPI_BIAS_RESIDUAL else torch.full((M, N), float("nan"), dtype=dt, device=DEV)
            L.gemm_bf16(out, A, W, None if epi == L.EPI_NONE else bias, residual=out if epi == L.EPI_BIAS_RESIDUAL else None,
                        epi=epi, simt=simt)
            eb.check_gemm(out, A, W, epi, bias, resid, ctx=f"{(M, N, K)} simt={simt}")
    # AdaLN / LayerNorm / gather with fp16 outputs: one fp16 ulp (2^-10 relative)
    M, d, B = 333, 1024, 3
    g = torch.Generator().manual_seed(6)
    x = (torch.randn(M, d, generator=g) * 3 + 0.5)
    emb = torch.randn(7, 2 * d, generator=g) * 0.1
    row_utt = torch.sort(torch.randint(0, B, (M,), generator=g)).values.to(torch.int32)
    lv = torch.tensor([3, 0, 6], dtype=torch.int32)
    ref = on.adaln(x[:, None, :], emb, lv[row_utt.long()].long())[:, 0]
    table = torch.cat([emb[:, :d].exp(), emb[:, d:]], dim=-1).to(DEV)
    out = torch.empty(M, d, dtype=torch.float16, device=DEV)
    L.adaln(out, x.to(DEV), table, lv.to(DEV), row_utt.to(DEV))
    assert ((out.float().cpu() - ref).abs() <= ref.abs() * 2 ** -10 + 2e-4).all()
    w, b = torch.randn(d, generator=g), torch.randn(d, generator=g)
    ref = torch.nn.functional.layer_norm(x, (d,), w, b, 1e-5)
    L.layernorm(out, x.to(DEV), w.to(DEV), b.to(DEV))
    assert ((out.float().cpu() - ref).abs() <= ref.abs() * 2 ** -10 + 2e-4).all()
    xs = x.clone()
    xs[0, :4] = torch.tensor([1e6, -1e6, 65504.0, 70000.0])            # beyond fp16: saturate, never inf
    idx = torch.tensor([5, 0, 332, 17], dtype=torch.int32)
    o2 = torch.empty(4, d, dtype=torch.float16, device=DEV)
    L.gather_rows_bf16(o2, xs.to(DEV), idx.to(DEV))
    exp = xs[idx.long()].clamp(-65504, 65504).half()
    assert torch.equal(o2.cpu(), exp) and torch.isfinite(o2).all()
    with pytest.raises(L.VB200Error):
        L.adaln(torch.empty(M, d, dtype=torch.float32, device=DEV), x.to(DEV), table, lv.to(DEV), row_utt.to(DEV))
    with pytest.raises(AssertionError):          # fp16 rows against bf16 weights: the hardware faults on it
        L.gemm_bf16(torch.empty(8, 16, device=DEV), torch.zeros(8, 16, dtype=torch.float16, device=DEV),
                    torch.zeros(16, 16, dtype=torch.bfloat16, device=DEV))
