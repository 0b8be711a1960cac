"""GPU tests of sampling temperature on the three reverse-step kernels (fused classifier head, posterior_fast_kernel,
posterior_sample_kernel): tau = 1 gives today's codes bit for bit; Philox draws follow the ORACLE's posterior on
logits / tau; with supplied uniforms post_out is that posterior's logits; greedy codes are its arg max and t == 0
stays the arg max of the raw logits; the captured step graph is keyed on tau."""
import pytest
import torch

from test_gpu_sample_steps import _batch, _chi2_ok, _make

pytestmark = pytest.mark.gpu

DEV = "cuda"
S = 50
TAUS = (0.5, 2.0)


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


def _law(orc, logits32, x_t, t, tau):
    """softmax of the oracle's fp32 posterior on logits / tau, (rows, levels, K) float64."""
    from oracle.d3pm import posterior_fp32
    rows, levels, K = logits32.shape
    post = posterior_fp32((logits32 / tau).reshape(rows * levels, 1, K), x_t.reshape(-1, 1),
                          torch.full((rows * levels,), t), orc)
    return torch.softmax(post.double(), -1).view(rows, levels, K)


# ---------------------------------------------------------------- tau = 1 is today
@pytest.mark.parametrize("K", [64, 256])
def test_temperature_one_gives_the_default_codes(L, K):
    """K = 256: fused head; K = 64: GEMM + standalone kernel; profiling hooks: separate calls on every K."""
    m, _ = _make(K, 128, 2, 2, 12, "absorbing", seed=11)
    text, proms = _batch(K, [(4, 10), (6, 7)], 13)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    known = [torch.full((40, 8), -1, dtype=torch.long), torch.full((150, 8), -1, dtype=torch.long)]
    known[0][:10] = torch.randint(0, K, (10, 8))
    known[1][:, 0] = torch.randint(0, K, (150,))
    eng = m.engine()
    for kw in (dict(seed=5), dict(greedy=True), dict(seed=6, sample_steps=4), dict(seed=7, known_list=known),
               dict(greedy=True, known_list=known, sample_steps=3)):
        for profile in (None, []):
            eng.profile = profile
            a = m.generate_audio(text, proms, resp_lens=[40, 150], **kw)
            a = [x.clone() for x in a]
            b = m.generate_audio(text, proms, resp_lens=[40, 150], temperature=1.0, **kw)
            eng.profile = None
            assert all(torch.equal(x, y) for x, y in zip(a, b)), (K, kw, profile)


@pytest.mark.parametrize("K", [1024, 1025])
def test_temperature_one_p_sample_with_supplied_uniforms(L, K):
    from vall_e.vall_e.diffusion import D3PMOps

    class Ops(D3PMOps):
        num_classes, timesteps, transition = K, S, "absorbing"

    ops = Ops()
    g = torch.Generator().manual_seed(K)
    logits = (torch.randn(3, 40, K, generator=g) * 2.5).to(torch.float16).to(DEV)
    x = torch.randint(0, K, (3, 40), generator=g).to(DEV)
    t = torch.tensor([S - 1, 20, 0], device=DEV)
    u = torch.rand(3, 40, K, generator=g).to(DEV)
    a, _ = ops.p_sample(logits, t, x, noise=u)
    b, _ = ops.p_sample(logits, t, x, noise=u, temperature=1.0)
    assert torch.equal(a, b)
    for kw in (dict(seed=3), dict(greedy=True)):
        assert torch.equal(ops.p_sample(logits, t, x, **kw)[0], ops.p_sample(logits, t, x, temperature=1.0, **kw)[0])


# ---------------------------------------------------------------- law
@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fused_head_philox_law_at_temperature(L, tr, tau):
    """40 960 draws per case of one token against softmax(oracle posterior(logits / tau)), the bar and structure of
    test_fused_head_philox_law_vs_oracle_posterior."""
    from oracle.d3pm import D3PM
    from vall_e.vall_e import d3pm as pd
    K, n, d, levels = 1024, 40960, 128, 2
    orc = D3PM(S, K, tr)
    table = pd.scalar_table(S, K, tr).to(DEV)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(29)
    row = torch.randn(1, d, generator=g).to(torch.float16)
    W = (torch.randn(levels * K, d, generator=g) * 0.22).to(torch.float16)
    bias = torch.randn(levels * K, generator=g)
    logits32 = (row.float() @ W.float().t() + bias).view(1, levels, K)
    head_in = row.repeat(n, 1).to(DEV)
    ru = torch.zeros(n, dtype=torch.int32, device=DEV)
    u1 = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    assert L.head_fused(d, K, L.NOISE_PHILOX)
    for t in (1, S // 2, S - 1):
        for xt_val in (K // 2, 3):
            law = _law(orc, logits32, torch.full((1, levels), xt_val), t, tau)[0]
            xt = torch.full((n, levels), xt_val, dtype=torch.int32, device=DEV)
            out = torch.empty(n, levels, dtype=torch.int32, device=DEV)
            L.head_posterior_sample(out, None, head_in, W.to(DEV), bias.to(DEV), xt, ru,
                                    torch.tensor([t], dtype=torch.int32, device=DEV), u1, table, levels, K, code,
                                    L.NOISE_PHILOX, seed=1000 + t, temperature=tau)
            for lv in range(levels):
                ok, stat = _chi2_ok(out[:, lv], law[lv])
                assert ok, (tr, tau, t, xt_val, lv, stat)


@pytest.mark.parametrize("K", [1024, 1025])
@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_standalone_kernels_philox_law_at_temperature(L, tr, tau, K):
    """K = 1024: posterior_fast_kernel; K = 1025 (the ar_discrete drop-in): posterior_sample_kernel."""
    from oracle.d3pm import D3PM
    from vall_e.vall_e import d3pm as pd
    n = 40960
    orc = D3PM(S, K, tr)
    table = pd.scalar_table(S, K, tr).to(DEV)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(K + 17)
    logits16 = (torch.randn(1, 1, K, generator=g) * 2.5).to(torch.float16)
    lg = logits16.view(1, K).to(DEV).repeat(n, 1).contiguous()
    ru = torch.zeros(n, dtype=torch.int32, device=DEV)
    utt = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    for t in (1, S // 2, S - 1):
        for xt_val in (K // 2, 3):
            law = _law(orc, logits16.float(), torch.full((1, 1), xt_val), t, tau)[0, 0]
            xt = torch.full((n,), xt_val, dtype=torch.int32, device=DEV)
            out = torch.empty(n, dtype=torch.int32, device=DEV)
            L.posterior_sample_from_logits(out, None, lg, K, xt, ru, torch.tensor([t], dtype=torch.int32, device=DEV),
                                           utt, table, n, 1, K, code, L.NOISE_PHILOX, seed=77 + t, temperature=tau)
            ok, stat = _chi2_ok(out, law)
            assert ok, (tr, tau, K, t, xt_val, stat)


# ---------------------------------------------------------------- parity mode and greedy
@pytest.mark.parametrize("K", [1024, 1025])
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_post_out_and_greedy_at_temperature_vs_oracle(L, tr, K):
    """Supplied uniforms: post_out is the oracle's fp32 posterior on logits / tau (the bar of test_posterior_vs_oracle)
    and the raw logits at t == 0; greedy codes are its arg max wherever the top-2 margin is clear, and the arg max of
    the raw logits at t == 0."""
    from oracle.d3pm import D3PM, posterior_fp32
    from vall_e.vall_e import d3pm as pd
    orc = D3PM(S, K, tr)
    table = pd.scalar_table(S, K, tr).to(DEV)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    B, W = 6, 48
    g = torch.Generator().manual_seed(K + 3)
    t = torch.tensor([0, 1, 2, 20, 40, S - 1])
    x_t = torch.randint(0, K, (B, W), generator=g)
    x_t[:, ::2] = K // 2
    logits16 = (torch.randn(B, W, K, generator=g) * 2.5).to(torch.float16)
    u = torch.rand(B * W, K, generator=g)
    row_utt = torch.arange(B, dtype=torch.int32, device=DEV).repeat_interleave(W)
    utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV)
    lg = logits16.to(DEV).view(B * W, K).contiguous()
    nz = t != 0
    for tau in TAUS:
        ref = posterior_fp32(logits16.float() / tau, x_t, t, orc)
        common = dict(ld_logits=K, x_t=x_t.to(DEV, torch.int32).view(-1).contiguous(), row_utt=row_utt,
                      t_utt=t.to(DEV, torch.int32), utt=utt, table=table, n_rows=B * W, n_levels=1, K=K,
                      transition=code, temperature=tau)
        post = torch.empty(B * W, K, dtype=torch.float32, device=DEV)
        out = torch.empty(B * W, dtype=torch.int32, device=DEV)
        L.posterior_sample_from_logits(out, post, lg, noise=L.NOISE_UNIFORMS, uniforms=u.to(DEV), **common)
        post = post.cpu().view(B, W, K)
        assert (post[nz] - ref[nz]).abs().max().item() < 2e-3, tau
        assert torch.equal(post[~nz], logits16[~nz].float())
        L.posterior_sample_from_logits(out, None, lg, noise=L.NOISE_GREEDY, **common)
        greedy = out.cpu().view(B, W).long()
        top2 = ref.topk(2, dim=-1).values
        clear = ((top2[..., 0] - top2[..., 1]) > 0.05) & nz[:, None]
        assert clear.sum() > 0.5 * nz.sum() * W
        assert torch.equal(greedy[clear], ref.argmax(-1)[clear]), tau
        assert torch.equal(greedy[~nz], logits16[~nz].float().argmax(-1))


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fused_head_greedy_at_temperature_vs_oracle(L, tr):
    from oracle.d3pm import D3PM
    from vall_e.vall_e import d3pm as pd
    K, levels, rows, d = 1024, 8, 192, 128
    orc = D3PM(S, K, tr)
    table = pd.scalar_table(S, K, tr).to(DEV)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(53)
    sch = [0, 1, 25, S - 1]
    B = len(sch)
    head_in = torch.randn(rows, d, generator=g).to(torch.float16)
    W = (torch.randn(levels * K, d, generator=g) * 0.25).to(torch.float16)
    bias = torch.randn(levels * K, generator=g)
    x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
    x_t[::2] = K // 2
    row_utt = (torch.arange(rows, dtype=torch.int32) % B).sort().values
    t_rows = torch.tensor(sch)[row_utt.long()]
    logits32 = (head_in.float() @ W.float().t() + bias).view(rows, levels, K)
    for tau in TAUS:
        out = torch.full((rows, levels), -1, dtype=torch.int32, device=DEV)
        L.head_posterior_sample(out, None, head_in.to(DEV), W.to(DEV), bias.to(DEV), x_t.to(DEV), row_utt.to(DEV),
                                torch.tensor(sch, dtype=torch.int32, device=DEV),
                                torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV), table, levels, K, code,
                                L.NOISE_GREEDY, temperature=tau)
        got = out.cpu().long()
        checked = 0
        for r in range(rows):
            t = int(t_rows[r])
            if t == 0:      # raw logits, no temperature (ar_discrete.py:407,413)
                top2 = logits32[r].topk(2, -1).values
                clear = (top2[:, 0] - top2[:, 1]) > 1e-2
                assert torch.equal(got[r][clear], logits32[r].argmax(-1)[clear])
                continue
            law = _law(orc, logits32[r:r + 1], x_t[r:r + 1].long(), t, tau)[0]
            lp = law.log()
            top2 = lp.topk(2, -1).values
            clear = (top2[:, 0] - top2[:, 1]) > 0.05
            assert torch.equal(got[r][clear], lp.argmax(-1)[clear]), (tr, tau, r)
            checked += int(clear.sum())
        assert checked > 0.3 * rows * levels * 3 / 4


# ---------------------------------------------------------------- graph key
def test_graph_is_keyed_on_temperature(L):
    """One cached session: tau = 0.5, 2.0, 0.5 again, each equal to its eager (use_graph=False) run."""
    K = 256
    m, _ = _make(K, 128, 2, 2, 12, "absorbing", seed=19)
    text, proms = _batch(K, [(4, 10), (6, 7)], 23)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    outs = {}
    for tau in (0.5, 2.0, 0.5):
        a = [x.clone() for x in m.generate_audio(text, proms, resp_lens=[40, 150], seed=9, temperature=tau)]
        b = [x.clone() for x in m.generate_audio(text, proms, resp_lens=[40, 150], seed=9, temperature=tau,
                                                  use_graph=False)]
        assert all(torch.equal(x, y) for x, y in zip(a, b)), tau
        outs.setdefault(tau, a)
        assert all(torch.equal(x, y) for x, y in zip(outs[tau], a))
    assert not all(torch.equal(x, y) for x, y in zip(outs[0.5], outs[2.0]))
