"""GPU tests of sampling with fewer denoise steps than timesteps: the three reverse-step kernels on a
schedule table (``d3pm.schedule_table``) against the ORACLE's jump posterior q(x_s | x_t, x0)
(``jump_oracle``: the oracle's dense fp16 tables and algorithm with ``s=``), and ``Diffusion.generate_audio(sample_steps=n)`` end to
end: the full schedule gives the codes of the default loop, a strided loop follows the oracle step by
step, replays as a graph, and keeps the seed and sharding properties of the default loop."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
S = 50
JUMPS = ((S - 1, 0), (S - 1, S // 2), (S // 2, S // 2 - 7), (3, 0))
SCHEDULES = ([S - 1], [S - 1, S // 2, S // 2 - 7, 3])      # between them, every jump of JUMPS


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


def _schedule_of(t, s):
    return next(sch for sch in SCHEDULES if (t, s) in zip(sch, sch[1:] + [0]))


def _table(K, tr, sch):
    from vall_e.vall_e import d3pm as pd
    return pd.schedule_table(S, K, tr, sch).to(DEV)


def _clear(post, margin):
    top2 = post.float().topk(2, dim=-1).values
    return (top2[..., 0] - top2[..., 1]) > margin


def _chi2_ok(draws, law):
    """chi-square of the class counts against ``law`` (cells with expectation <= 5 pooled), the statistic and
    threshold of the fused-head Philox test."""
    n = draws.numel()
    counts = torch.bincount(draws.view(-1).cpu().long(), minlength=law.numel()).double()
    expected = law * n
    keep = expected > 5
    chi2 = (((counts - expected) ** 2) / expected)[keep].sum().item()
    cells = int(keep.sum().item())
    rest_obs, rest_exp = counts[~keep].sum().item(), expected[~keep].sum().item()
    if rest_exp > 5:
        chi2 += (rest_obs - rest_exp) ** 2 / rest_exp
        cells += 1
    dof = max(cells - 1, 1)
    return chi2 < dof + 6 * math.sqrt(2 * dof), (chi2, dof)


# ---------------------------------------------------------------- fused head (production reverse step)
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fused_head_philox_law_vs_oracle_jump_posterior(L, tr):
    from jump_oracle import JumpD3PM
    K, n, d, levels = 1024, 40960, 128, 2
    orc = JumpD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(31)
    row = torch.randn(1, d, generator=g).to(torch.float16)
    W = (torch.randn(levels * K, d, generator=g) * 0.22).to(torch.float16)
    bias = torch.randn(levels * K, generator=g)
    logits16 = (row.float() @ W.float().t() + bias).view(1, levels, K).to(torch.float16)
    head_in = row.repeat(n, 1).to(DEV)
    ru = torch.zeros(n, dtype=torch.int32, device=DEV)
    u1 = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    assert L.head_fused(d, K, L.NOISE_PHILOX)
    for t, s in JUMPS:
        table = _table(K, tr, _schedule_of(t, s))
        for xt_val in (K // 2, 3):
            x1 = torch.full((1, levels), xt_val, dtype=torch.int32)
            law = torch.softmax(orc.q_posterior_logits(logits16, x1, torch.tensor([t]), torch.tensor([s])).double(),
                                -1)[0]
            xt = torch.full((n, levels), xt_val, dtype=torch.int32, device=DEV)
            out = torch.empty(n, levels, dtype=torch.int32, device=DEV)
            L.head_posterior_sample(out, None, head_in, W.to(DEV), bias.to(DEV), xt, ru,
                                    torch.tensor([t], dtype=torch.int32, device=DEV), u1, table, levels, K, code,
                                    L.NOISE_PHILOX, seed=2000 + t)
            for lv in range(levels):
                ok, stat = _chi2_ok(out[:, lv], law[lv])
                assert ok, (tr, t, s, xt_val, lv, stat)


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fused_head_greedy_codes_vs_oracle_jump(L, tr):
    from jump_oracle import JumpD3PM
    K, levels, rows, d = 1024, 8, 320, 128
    orc = JumpD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(37)
    assert L.head_fused(d, K, L.NOISE_GREEDY)
    checked = 0
    for sch in SCHEDULES:
        B = len(sch)
        succ = sch[1:] + [0]
        head_in = torch.randn(rows, d, generator=g).to(torch.float16)
        W = (torch.randn(levels * K, d, generator=g) * 0.25).to(torch.float16)
        bias = torch.randn(levels * K, generator=g)
        x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
        x_t[::2] = K // 2
        row_utt = (torch.arange(rows, dtype=torch.int32) % B).sort().values
        t_utt = torch.tensor(sch, dtype=torch.int32)
        utt = torch.zeros(B, L.U_STRIDE, dtype=torch.int32)
        logits16 = (head_in.float() @ W.float().t() + bias).view(rows, levels, K).to(torch.float16)
        t_rows, s_rows = t_utt[row_utt.long()].long(), torch.tensor(succ)[row_utt.long()]
        refs, posts = [], []
        for r0 in range(0, rows, 32):
            c, p = orc.p_sample(logits16[r0:r0 + 32], t_rows[r0:r0 + 32], x_t[r0:r0 + 32], greedy=True,
                                s=s_rows[r0:r0 + 32])
            refs.append(c)
            posts.append(p.float())
        ref, post = torch.cat(refs), torch.cat(posts)
        out = torch.full((rows, levels), -1, dtype=torch.int32, device=DEV)
        L.head_posterior_sample(out, None, head_in.to(DEV), W.to(DEV), bias.to(DEV), x_t.to(DEV), row_utt.to(DEV),
                                t_utt.to(DEV), utt.to(DEV), _table(K, tr, sch), levels, K, code, L.NOISE_GREEDY)
        got = out.cpu().long()
        clear = _clear(post, 0.05)
        assert clear.float().mean().item() > 0.7
        assert torch.equal(got[clear], ref[clear]), (sch, int((got[clear] != ref[clear]).sum()))
        checked += int(clear.sum())
    assert checked > 2000


# ---------------------------------------------------------------- standalone reverse-step kernels
@pytest.mark.parametrize("K", [1025, 1024])
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_generic_posterior_kernel_vs_oracle_jump(L, tr, K):
    """posterior_sample_kernel (post_out requested, or supplied uniforms): posterior logits within the KL bar
    of the oracle's jump posterior, greedy and Gumbel-argmax codes equal wherever the margin is clear."""
    from jump_oracle import JumpD3PM, posterior_fp32
    orc = JumpD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    sch = SCHEDULES[1]
    B, W = len(sch), 40
    g = torch.Generator().manual_seed(K + 3)
    t, s = torch.tensor(sch), torch.tensor(sch[1:] + [0])
    logits16 = (torch.randn(B, W, K, generator=g) * 2.5).to(torch.float16)
    x_t = torch.randint(0, K, (B, W), generator=g, dtype=torch.int32)
    x_t[:, ::3] = K // 2
    noise = torch.rand(B, W, K, generator=g)
    ref_samp, ref_post16 = orc.p_sample(logits16, t, x_t, noise, s=s)
    ref_greedy, _ = orc.p_sample(logits16, t, x_t, greedy=True, s=s)
    ref_post32 = posterior_fp32(logits16, x_t, t, orc, s)
    common = dict(ld_logits=K, x_t=x_t.to(DEV).view(-1).contiguous(),
                  row_utt=torch.arange(B, dtype=torch.int32, device=DEV).repeat_interleave(W),
                  t_utt=t.to(DEV, torch.int32), utt=torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV),
                  table=_table(K, tr, sch), n_rows=B * W, n_levels=1, K=K, transition=code)
    lg = logits16.to(DEV).view(B * W, K).contiguous()
    post = torch.empty(B * W, K, dtype=torch.float32, device=DEV)
    out = torch.empty(B * W, dtype=torch.int32, device=DEV)
    L.posterior_sample_from_logits(out, post, lg, noise=L.NOISE_GREEDY, **common)
    post = post.cpu().view(B, W, K)
    p_ref = torch.softmax(ref_post16.float(), -1)
    kl = (p_ref * (torch.log_softmax(ref_post16.float(), -1) - torch.log_softmax(post, -1))).sum(-1)
    assert kl.max().item() <= 1e-3, kl.max().item()
    assert (post - ref_post32).abs().max().item() < 2e-3
    clear = _clear(ref_post16, 0.05)
    assert clear.float().mean().item() > 0.5
    assert torch.equal(out.cpu().view(B, W).long()[clear], ref_greedy[clear])
    L.posterior_sample_from_logits(out, None, lg, noise=L.NOISE_UNIFORMS, uniforms=noise.to(DEV).view(B * W, K), **common)
    samp = out.cpu().view(B, W).long()
    gn = -torch.log(-torch.log(noise.clamp(min=torch.finfo(torch.float32).tiny)))
    clear = _clear(ref_post16.float() + gn, 0.05)
    assert clear.float().mean().item() > 0.5
    assert torch.equal(samp[clear], ref_samp[clear])


@pytest.mark.parametrize("K", [256, 1024])
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fast_posterior_kernel_matches_generic_on_a_schedule_table(L, tr, K):
    from jump_oracle import JumpD3PM
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(K + 11)
    rows, levels = 300, 2
    sch = SCHEDULES[1]
    table = _table(K, tr, sch)
    B = len(sch)
    logits = (torch.randn(rows, levels * K, generator=g) * 3).half().to(DEV)
    x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
    x_t[::3] = K // 2
    row_utt = (torch.arange(rows, dtype=torch.int32) % B).sort().values.to(DEV)
    args = (levels * K, x_t.to(DEV), row_utt, torch.tensor(sch, dtype=torch.int32, device=DEV),
            torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV), table, rows, levels, K, code)
    fast = torch.empty(rows, levels, dtype=torch.int32, device=DEV)
    slow = torch.empty_like(fast)
    post = torch.empty(rows * levels, K, dtype=torch.float32, device=DEV)
    L.posterior_sample_from_logits(fast, None, logits, *args, L.NOISE_GREEDY)
    L.posterior_sample_from_logits(slow, post, logits, *args, L.NOISE_GREEDY)
    clear = _clear(post, 1e-3).view(rows, levels)
    assert clear.float().mean().item() > 0.9
    assert torch.equal(fast[clear], slow[clear])
    # inverse-CDF draws of the fast kernel against the oracle's jump law
    orc = JumpD3PM(S, K, tr)
    n = 40000
    row = (torch.randn(K, generator=g) * 2.0).half()
    lg = row.repeat(n, 1).to(DEV)
    for t, s in JUMPS:
        tab = _table(K, tr, _schedule_of(t, s))
        for xt_val in (K // 2, 3):
            law = torch.softmax(orc.q_posterior_logits(row.view(1, 1, K), torch.tensor([[xt_val]], dtype=torch.int32),
                                                       torch.tensor([t]), torch.tensor([s])).double(), -1).view(-1)
            out = torch.empty(n, 1, dtype=torch.int32, device=DEV)
            L.posterior_sample_from_logits(out, None, lg, K, torch.full((n, 1), xt_val, dtype=torch.int32, device=DEV),
                                           torch.zeros(n, dtype=torch.int32, device=DEV),
                                           torch.tensor([t], dtype=torch.int32, device=DEV),
                                           torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV), tab, n, 1, K, code,
                                           L.NOISE_PHILOX, seed=5)
            ok, stat = _chi2_ok(out, law)
            assert ok, (tr, K, t, s, xt_val, stat)


# ---------------------------------------------------------------- generate_audio(sample_steps=n)
def _make(K, d, h, nl, S_, transition, seed):
    from oracle import denoiser as on
    from vall_e.vall_e.diffusion import Diffusion
    sd = on.random_state_dict(K, d, nl, S_ + 1, n_resp_levels=8, n_out=8 * K, seed=seed, time_rows=S_ + 1)
    m = Diffusion(K, d_model=d, n_heads=h, n_layers=nl, n_steps=S_, transition=transition)
    m.load_state_dict(sd)
    return m.to(DEV), sd


def _batch(K, lens, seed):
    g = torch.Generator().manual_seed(seed)
    text = [torch.randint(1, K, (a,), generator=g) for a, _ in lens]
    proms = [torch.randint(0, K, (b, 8), generator=g) for _, b in lens]
    return text, proms


@pytest.mark.parametrize("K", [64, 256])
def test_full_schedule_gives_the_codes_of_the_default_loop(L, K):
    m, _ = _make(K, 128, 2, 2, 12, "absorbing", seed=5)
    text, proms = _batch(K, [(4, 10), (6, 7)], 3)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    for kw in (dict(seed=5), dict(greedy=True)):
        for use_graph in (True, False):
            a = m.generate_audio(text, proms, resp_lens=[40, 150], use_graph=use_graph, **kw)
            b = m.generate_audio(text, proms, resp_lens=[40, 150], use_graph=use_graph, sample_steps=11, **kw)
            assert all(torch.equal(x, y) for x, y in zip(a, b)), (kw, use_graph)
    assert L.head_fused(128, K, L.NOISE_PHILOX) == (K == 256)


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_strided_loop_teacher_forced_vs_oracle(L, transition):
    """S = 12, sample_steps = 4 (t = 11, 9, 6, 3 -> 0) through the fused head: every step equals the oracle's
    jump step at (t, sigma(t)) from the CUDA trajectory's previous state, wherever the margin is clear."""
    from oracle import denoiser as on
    from jump_oracle import JumpD3PM
    K, d, h, nl, S_ = 256, 128, 2, 2, 12
    m, sd = _make(K, d, h, nl, S_, transition, seed=19)
    assert L.head_fused(d, K, L.NOISE_GREEDY)
    lens = [24, 33]
    text, proms = _batch(K, [(4, 10), (6, 7)], 13)
    g = torch.Generator().manual_seed(1)
    x_T = (torch.full((sum(lens), 8), K // 2, dtype=torch.long) if transition == "absorbing"
           else torch.randint(0, K, (sum(lens), 8), generator=g))
    trace = []
    out = m.generate_audio([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [r.to(DEV) for r in x_T.split(lens)],
                           greedy=True, trace=trace, use_graph=False, sample_steps=4)
    sch = [11, 9, 6, 3]
    assert len(trace) == 4
    orc = JumpD3PM(S_, K, transition)
    prev, checked, agree = x_T, 0, 0
    for step, (t, s) in enumerate(zip(sch, sch[1:] + [0])):
        lg = torch.cat(on.diffusion_logits(sd, text, proms, list(prev.split(lens)), torch.tensor([t, t]), h, nl))
        lg = lg.to(torch.float16)
        n = lg.shape[0]
        ref, post = orc.p_sample(lg, torch.full((n,), t), prev.to(torch.int32), greedy=True, s=torch.full((n,), s))
        clear = _clear(post, 0.08)
        got = trace[step].cpu().long()
        checked += int(clear.sum())
        agree += int((got[clear] == ref[clear]).sum())
        prev = got
    assert checked > 0.3 * prev.numel() * 4 and agree == checked, (agree, checked)
    assert torch.equal(torch.cat(out).cpu(), prev)


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_strided_loop_graph_seed_and_sharding(L, transition):
    K, S_ = 256, 12
    m, _ = _make(K, 128, 2, 2, S_, transition, seed=21)
    text, proms = _batch(K, [(4, 10), (6, 7)], 3)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    lens = [40, 150]
    a = m.generate_audio(text, proms, resp_lens=lens, seed=5, sample_steps=4)
    b = m.generate_audio(text, proms, resp_lens=lens, seed=5, sample_steps=4, use_graph=False)
    again = m.generate_audio(text, proms, resp_lens=lens, seed=5, sample_steps=4)
    c = m.generate_audio(text, proms, resp_lens=lens, seed=6, sample_steps=4)
    full = m.generate_audio(text, proms, resp_lens=lens, seed=5)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert all(torch.equal(x, y) for x, y in zip(a, again))
    assert any(not torch.equal(x, y) for x, y in zip(a, c))
    assert any(not torch.equal(x, y) for x, y in zip(a, full))
    assert all(int(x.min()) >= 0 and int(x.max()) < K for x in a)
    m.generate_audio(text, proms, resp_lens=lens, seed=5, sample_steps=4)
    ses = m._session(text, proms, lens, None)
    assert ses.t_utt.cpu().tolist() == [0, 0]          # the schedule ends at t = 0 on the device
    solo = m.generate_audio(text[1:], proms[1:], resp_lens=lens[1:], seed=5, gids=[1], sample_steps=4)
    assert torch.equal(solo[0], a[1])


def test_bad_sample_steps_raise_before_any_launch(L):
    m, _ = _make(64, 64, 1, 1, 6, "absorbing", seed=8)
    text, proms = _batch(64, [(3, 5)], 2)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    m.generate_audio(text, proms, resp_lens=[9], sample_steps=2)
    before = m.engine().launches
    for bad in (0, 6, 2.5):
        with pytest.raises(ValueError, match="sample_steps"):
            m.generate_audio(text, proms, resp_lens=[9], sample_steps=bad)
    torch.cuda.synchronize()
    assert m.engine().launches == before
    t = torch.full((3,), 5, dtype=torch.int32, device=DEV)
    with pytest.raises(L.VB200Error, match="step_timesteps_to"):
        L.step_timesteps_to(t, None)
    L.step_timesteps_to(t, torch.tensor([0, 0, 1, 2, 3, 1], dtype=torch.int32, device=DEV))
    assert t.cpu().tolist() == [1, 1, 1]
