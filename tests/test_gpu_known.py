"""GPU tests of generation around given codes (``generate_audio(known_list=...)``): the reverse-step kernels'
draws of known tokens against the oracle's ids-form posterior q(x_s | x_t, x0 = k) (``known_oracle``), the
unknown tokens of the same launches against the model posterior, bit-identity without known codes, and
``generate_audio`` end to end: given codes come back, a teacher-forced loop follows the oracle, graph replay, seed,
batch and sharding invariance, cached sessions and ``--continue-from``."""
import pytest
import torch

from test_gpu_sample_steps import JUMPS, S, _batch, _chi2_ok, _clear, _make, _schedule_of, _table

pytestmark = pytest.mark.gpu

DEV = "cuda"
FULL = (S - 1, 30, 1)                     # one-step posteriors on the plain table


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


def _steps():
    """(t, s, table schedule): one-step and jump steps."""
    full = list(range(S - 1, 0, -1))
    return [(t, None, full) for t in FULL] + [(t, s, _schedule_of(t, s)) for t, s in JUMPS]


def _cases(K):
    m = K // 2
    return [(m, m), (m, 7), (5, 5), (5, m), (5, 900 % K)]        # (x_t, k): every special case


def _law(orc, k, x_t, t, s):
    x0 = torch.tensor([[k]], dtype=torch.int32)
    xt = torch.tensor([[x_t]], dtype=torch.int32)
    return torch.softmax(orc.log_law_ids(x0, xt, torch.tensor([t]), None if s is None else torch.tensor([s])), -1)[0, 0]


# ---------------------------------------------------------------- fused head
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fused_head_philox_known_law_vs_oracle(L, tr):
    """Level 0 known, level 1 not, in one launch: level 0 draws follow the ids-form law, level 1 the model's."""
    from known_oracle import KnownD3PM
    K, n, d, levels = 1024, 40960, 128, 2
    orc = KnownD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(41)
    row = torch.randn(1, d, generator=g).to(torch.float16)
    W = (torch.randn(levels * K, d, generator=g) * 0.22).to(torch.float16)
    bias = torch.randn(levels * K, generator=g)
    logits16 = (row.float() @ W.float().t() + bias).view(1, levels, K).to(torch.float16)
    head_in = row.repeat(n, 1).to(DEV)
    ru = torch.zeros(n, dtype=torch.int32, device=DEV)
    u1 = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    assert L.head_fused(d, K, L.NOISE_PHILOX)
    for t, s, sch in _steps():
        table = _table(K, tr, sch)
        for x_t, k in _cases(K):
            law_k = _law(orc, k, x_t, t, s)
            x1 = torch.full((1, levels), x_t, dtype=torch.int32)
            sv = None if s is None else torch.tensor([s])
            law_m = torch.softmax(orc.q_posterior_logits(logits16, x1, torch.tensor([t]), sv).double(), -1)[0, 1]
            xt = torch.full((n, levels), x_t, dtype=torch.int32, device=DEV)
            known = torch.full((n, levels), -1, dtype=torch.int32, device=DEV)
            known[:, 0] = k
            out = torch.empty(n, levels, dtype=torch.int32, device=DEV)
            L.head_posterior_sample(out, None, head_in, W.to(DEV), bias.to(DEV), xt, ru,
                                    torch.tensor([t], dtype=torch.int32, device=DEV), u1, table, levels, K, code,
                                    L.NOISE_PHILOX, seed=3000 + t, known=known)
            ok, stat = _chi2_ok(out[:, 0], law_k)
            assert ok, ("known", tr, t, s, x_t, k, stat)
            ok, stat = _chi2_ok(out[:, 1], law_m)
            assert ok, ("unknown", tr, t, s, x_t, k, stat)


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fused_head_greedy_known_codes_vs_oracle(L, tr):
    from known_oracle import KnownD3PM
    K, levels, rows, d = 1024, 8, 320, 128
    orc = KnownD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    g = torch.Generator().manual_seed(43)
    checked = 0
    full_sch = list(range(S - 1, 0, -1))
    for sch, succ, tab_sch in (([S - 1, S // 2, S // 2 - 7, 3], [S // 2, S // 2 - 7, 3, 0], None),
                               ([49, 37, 25, 13, 1], [48, 36, 24, 12, 0], full_sch)):     # jumps; one-step
        B = len(sch)
        head_in = torch.randn(rows, d, generator=g).to(torch.float16)
        W = (torch.randn(levels * K, d, generator=g) * 0.25).to(torch.float16)
        bias = torch.randn(levels * K, generator=g)
        x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
        x_t[::2] = K // 2
        known = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32)
        known[::3] = K // 2
        known[1::5] = x_t[1::5]
        is_known = torch.rand(rows, levels, generator=g) < 0.5
        known[~is_known] = -1
        row_utt = (torch.arange(rows, dtype=torch.int32) % B).sort().values
        t_utt = torch.tensor(sch, dtype=torch.int32)
        t_rows, s_rows = t_utt[row_utt.long()].long(), torch.tensor(succ)[row_utt.long()]
        logits16 = (head_in.float() @ W.float().t() + bias).view(rows, levels, K).to(torch.float16)
        parts = [(orc.p_sample(logits16[r:r + 32], t_rows[r:r + 32], x_t[r:r + 32], greedy=True, s=s_rows[r:r + 32]),
                  orc.p_sample_ids(known[r:r + 32].clamp(min=0), t_rows[r:r + 32], x_t[r:r + 32], greedy=True,
                                   s=s_rows[r:r + 32])) for r in range(0, rows, 32)]
        ref_u, post_u = torch.cat([u[0] for u, _ in parts]), torch.cat([u[1].float() for u, _ in parts])
        ref_k, post_k = torch.cat([k[0] for _, k in parts]), torch.cat([k[1] for _, k in parts])
        out = torch.full((rows, levels), -2, dtype=torch.int32, device=DEV)
        L.head_posterior_sample(out, None, head_in.to(DEV), W.to(DEV), bias.to(DEV), x_t.to(DEV), row_utt.to(DEV),
                                t_utt.to(DEV), torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV),
                                _table(K, tr, tab_sch or sch), levels, K, code,
                                L.NOISE_GREEDY, known=known.to(DEV))
        got = out.cpu().long()
        ck = _clear(post_k, 1e-3) & is_known
        cu = _clear(post_u, 0.05) & ~is_known
        assert ck.sum() > 0.8 * is_known.sum() and cu.sum() > 0.3 * (~is_known).sum()
        assert torch.equal(got[ck], ref_k[ck]), (sch, int((got[ck] != ref_k[ck]).sum()))
        assert torch.equal(got[cu], ref_u[cu]), (sch, int((got[cu] != ref_u[cu]).sum()))
        checked += int(ck.sum())
    assert checked > 500


# ---------------------------------------------------------------- standalone reverse-step kernels
@pytest.mark.parametrize("K", [1025, 1024])
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_generic_kernel_known_tokens_vs_oracle(L, tr, K):
    """posterior_sample_kernel: supplied uniforms give the oracle's Gumbel-arg max, post_out and
    q_posterior_logits(x_start_logits=False) the oracle's ids-form logits; the fast kernel (K = 1024) draws the
    generic kernel's codes from the same Philox counter."""
    from known_oracle import KnownD3PM
    from vall_e.vall_e.diffusion import D3PMOps
    orc = KnownD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    sch = [S - 1, S // 2, S // 2 - 7, 3]
    B, W = len(sch), 48
    g = torch.Generator().manual_seed(K + 5)
    t, s = torch.tensor(sch), torch.tensor(sch[1:] + [0])
    logits16 = (torch.randn(B, W, K, generator=g) * 2.5).to(torch.float16)
    x_t = torch.randint(0, K, (B, W), generator=g, dtype=torch.int32)
    x_t[:, ::3] = K // 2
    x0 = torch.randint(0, K, (B, W), generator=g, dtype=torch.int32)
    x0[:, 1::4] = K // 2
    x0[:, 2::5] = x_t[:, 2::5]
    known = x0.clone()
    known[:, ::2] = -1                                         # mixed: even columns drawn from the logits
    is_known = known >= 0
    noise = torch.rand(B, W, K, generator=g)
    ref_samp_k, ref_post_k = orc.p_sample_ids(x0, t, x_t, noise, s=s)
    ref_samp_u, ref_post_u = orc.p_sample(logits16, t, x_t, noise, s=s)
    common = dict(ld_logits=K, x_t=x_t.to(DEV).view(-1).contiguous(),
                  row_utt=torch.arange(B, dtype=torch.int32, device=DEV).repeat_interleave(W),
                  t_utt=t.to(DEV, torch.int32), utt=torch.zeros(B, L.U_STRIDE, dtype=torch.int32, device=DEV),
                  table=_table(K, tr, sch), n_rows=B * W, n_levels=1, K=K, transition=code,
                  known=known.to(DEV).view(-1).contiguous())
    lg = logits16.to(DEV).view(B * W, K).contiguous()
    lg_junk = lg.clone()
    lg_junk.view(B, W, K)[is_known.to(DEV)] = float("nan")    # logit rows of known tokens are never read
    out = torch.empty(B * W, dtype=torch.int32, device=DEV)
    post = torch.empty(B * W, K, dtype=torch.float32, device=DEV)
    L.posterior_sample_from_logits(out, post, lg_junk, noise=L.NOISE_UNIFORMS, uniforms=noise.to(DEV).view(B * W, K),
                                   **common)
    samp, post = out.cpu().view(B, W).long(), post.cpu().view(B, W, K)
    assert (post[is_known].double() - ref_post_k[is_known]).abs().max().item() < 2e-3
    gn = -torch.log(-torch.log(noise.clamp(min=torch.finfo(torch.float32).tiny))).double()
    ck = _clear(ref_post_k + gn, 0.05) & is_known
    assert ck.sum() > 0.5 * is_known.sum()
    assert torch.equal(samp[ck], ref_samp_k[ck])
    L.posterior_sample_from_logits(out, None, lg, noise=L.NOISE_UNIFORMS, uniforms=noise.to(DEV).view(B * W, K),
                                   **common)
    samp = out.cpu().view(B, W).long()
    cu = _clear(ref_post_u.float() + gn.float(), 0.05) & ~is_known
    assert cu.sum() > 0.5 * (~is_known).sum()
    assert torch.equal(samp[cu], ref_samp_u[cu])
    # the ids form of q_posterior_logits (one-step, plain table) against the oracle's
    ops = type("Ops", (D3PMOps,), {})()
    ops.num_classes, ops.timesteps, ops.transition = K, S, tr
    tq = torch.tensor([1, 7, S - 1, 0])
    ql = ops.q_posterior_logits(x0.to(DEV), x_t.to(DEV), tq.to(DEV), x_start_logits=False).cpu()
    ref = orc.q_posterior_logits_ids(x0, x_t, tq)
    ref64 = orc.log_law_ids(x0, x_t, tq)
    assert (ql[:3].double() - ref64[:3]).abs().max().item() < 2e-3
    assert float(ql[3].abs().max()) == 0.0 and float(ref[3].abs().max()) == 0.0
    if K % 256 == 0:                                            # fast kernel: same codes from the same counter
        for noise_mode in (L.NOISE_PHILOX, L.NOISE_GREEDY):
            fast, slow = torch.empty_like(out), torch.empty_like(out)
            L.posterior_sample_from_logits(fast, None, lg_junk, noise=noise_mode, seed=9, **common)
            L.posterior_sample_from_logits(slow, torch.empty(B * W, K, device=DEV), lg_junk, noise=noise_mode, seed=9,
                                           **common)
            kd = is_known.to(DEV).view(-1)
            assert torch.equal(fast[kd], slow[kd]), noise_mode


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_fast_kernel_known_law_vs_oracle(L, tr):
    from known_oracle import KnownD3PM
    K, n = 1024, 40000
    orc = KnownD3PM(S, K, tr)
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    lg = (torch.randn(n, K) * 2.0).half().to(DEV)
    for t, s, sch in _steps()[::2]:
        tab = _table(K, tr, sch)
        for x_t, k in _cases(K):
            out = torch.empty(n, 1, dtype=torch.int32, device=DEV)
            L.posterior_sample_from_logits(out, None, lg, K, torch.full((n, 1), x_t, dtype=torch.int32, device=DEV),
                                           torch.zeros(n, dtype=torch.int32, device=DEV),
                                           torch.tensor([t], dtype=torch.int32, device=DEV),
                                           torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV), tab, n, 1, K,
                                           code, L.NOISE_PHILOX, seed=6,
                                           known=torch.full((n, 1), k, dtype=torch.int32, device=DEV))
            ok, stat = _chi2_ok(out, _law(orc, k, x_t, t, s))
            assert ok, (tr, t, s, x_t, k, stat)


def test_kernels_without_known_codes_are_bit_identical(L):
    """known all -1 through the _known entry points gives the codes of the plain ones (fused head, fast and
    generic kernels, Philox and greedy)."""
    K, d, levels, rows = 1024, 128, 8, 700
    g = torch.Generator().manual_seed(3)
    head_in = torch.randn(rows, d, generator=g).to(torch.float16).to(DEV)
    W = (torch.randn(levels * K, d, generator=g) * 0.25).to(torch.float16).to(DEV)
    bias = torch.randn(levels * K, generator=g).to(DEV)
    x_t = torch.randint(0, K, (rows, levels), generator=g, dtype=torch.int32).to(DEV)
    ru = (torch.arange(rows, dtype=torch.int32) % 3).sort().values.to(DEV)
    tu = torch.tensor([40, 12, 1], dtype=torch.int32, device=DEV)
    utt = torch.zeros(3, L.U_STRIDE, dtype=torch.int32, device=DEV)
    none = torch.full((rows, levels), -1, dtype=torch.int32, device=DEV)
    lg = (torch.randn(rows, levels * K, generator=g) * 3).half().to(DEV)
    for tr, code in (("absorbing", L.ABSORBING), ("uniform", L.UNIFORM)):
        table = _table(K, tr, list(range(S - 1, 0, -1)))
        for noise in (L.NOISE_PHILOX, L.NOISE_GREEDY):
            a, b = torch.empty_like(x_t), torch.empty_like(x_t)
            L.head_posterior_sample(a, None, head_in, W, bias, x_t, ru, tu, utt, table, levels, K, code, noise, seed=4)
            L.head_posterior_sample(b, None, head_in, W, bias, x_t, ru, tu, utt, table, levels, K, code, noise, seed=4,
                                    known=none)
            assert torch.equal(a, b), (tr, noise)
            for post in (None, torch.empty(rows * levels, K, device=DEV)):
                L.posterior_sample_from_logits(a, post, lg, levels * K, x_t, ru, tu, utt, table, rows, levels, K, code,
                                               noise, seed=4)
                L.posterior_sample_from_logits(b, post, lg, levels * K, x_t, ru, tu, utt, table, rows, levels, K, code,
                                               noise, seed=4, known=none)
                assert torch.equal(a, b), (tr, noise, post is None)


# ---------------------------------------------------------------- generate_audio(known_list=...)
LENS = [40, 150]


def _setup(transition, seed=21, K=256):
    m, sd = _make(K, 128, 2, 2, 12, transition, seed=seed)
    text, proms = _batch(K, [(4, 10), (6, 7)], 3)
    return m, sd, [x.to(DEV) for x in text], [x.to(DEV) for x in proms]


def _masks(lens, K, seed=0):
    """name -> known_list: prefix, middle span, level 0, random 30 %, all known."""
    g = torch.Generator().manual_seed(seed)
    codes = [torch.randint(0, K, (n, 8), generator=g) for n in lens]
    out = {}
    for name in ("prefix", "span", "level0", "random", "all"):
        ks = []
        for c in codes:
            k = torch.full_like(c, -1)
            n = len(c)
            if name == "prefix":
                k[: n * 3 // 10] = c[: n * 3 // 10]
            elif name == "span":
                k[: n // 3] = c[: n // 3]
                k[2 * n // 3:] = c[2 * n // 3:]
            elif name == "level0":
                k[:, 0] = c[:, 0]
            elif name == "random":
                sel = torch.rand(c.shape, generator=g) < 0.3
                k[sel] = c[sel]
            else:
                k = c.clone()
            ks.append(k)
        out[name] = ks
    return out


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_generate_without_known_codes_is_unchanged(L, transition):
    m, _, text, proms = _setup(transition)
    none = [torch.full((n, 8), -1) for n in LENS]
    for steps in (None, 10):
        for use_graph in (True, False):
            for kw in (dict(seed=5), dict(greedy=True)):
                a = m.generate_audio(text, proms, resp_lens=LENS, use_graph=use_graph, sample_steps=steps, **kw)
                b = m.generate_audio(text, proms, resp_lens=LENS, use_graph=use_graph, sample_steps=steps,
                                     known_list=None, **kw)
                c = m.generate_audio(text, proms, use_graph=use_graph, sample_steps=steps, known_list=none, **kw)
                assert all(torch.equal(x, y) for x, y in zip(a, b)), (steps, use_graph, kw)
                assert all(torch.equal(x, y) for x, y in zip(a, c)), (steps, use_graph, kw)


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_given_codes_come_back(L, transition):
    m, _, text, proms = _setup(transition)
    for name, kl in _masks(LENS, 256).items():
        for kw in (dict(seed=5), dict(greedy=True, sample_steps=4), dict(seed=2, sample_steps=10, use_graph=False)):
            out = m.generate_audio(text, proms, known_list=kl, **kw)
            for o, k in zip(out, kl):
                sel = k >= 0
                assert torch.equal(o.cpu()[sel], k[sel]), (name, kw)
                assert int(o.min()) >= 0 and int(o.max()) < 256
    bqt, frames = m.generate_audio(text, proms, known_list=_masks(LENS, 256)["prefix"], seed=5, as_bqt=True,
                                   to_host=True)
    assert frames == LENS and bqt.device.type == "cpu"


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_strided_loop_with_known_codes_teacher_forced_vs_oracle(L, transition):
    """S = 12, sample_steps = 4 through the fused head with a mixed mask: every step of every token equals the
    oracle's step — the model posterior for unknown tokens, the ids form for known ones — wherever the margin is
    clear; the output is the last step with the given codes put back."""
    from known_oracle import KnownD3PM
    from oracle import denoiser as on
    K, h, nl, S_ = 256, 2, 2, 12
    m, sd = _make(K, 128, h, nl, S_, transition, seed=19)
    lens = [24, 33]
    text, proms = _batch(K, [(4, 10), (6, 7)], 13)
    g = torch.Generator().manual_seed(1)
    x_T = (torch.full((sum(lens), 8), K // 2, dtype=torch.long) if transition == "absorbing"
           else torch.randint(0, K, (sum(lens), 8), generator=g))
    codes = torch.randint(0, K, (sum(lens), 8), generator=g)
    known = torch.where(torch.rand(sum(lens), 8, generator=g) < 0.4, codes, torch.full_like(codes, -1))
    known[:5] = codes[:5]
    known[:, 0] = codes[:, 0]
    trace = []
    out = m.generate_audio([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [r.to(DEV) for r in x_T.split(lens)],
                           greedy=True, trace=trace, use_graph=False, sample_steps=4,
                           known_list=[k.to(DEV) for k in known.split(lens)])
    sch = [11, 9, 6, 3]
    orc = KnownD3PM(S_, K, transition)
    is_known = known >= 0
    prev, checked, agree, checked_k = x_T, 0, 0, 0
    for step, (t, s) in enumerate(zip(sch, sch[1:] + [0])):
        lg = torch.cat(on.diffusion_logits(sd, text, proms, list(prev.split(lens)), torch.tensor([t, t]), h, nl))
        lg = lg.to(torch.float16)
        n = lg.shape[0]
        tt, ss = torch.full((n,), t), torch.full((n,), s)
        ref_u, post_u = orc.p_sample(lg, tt, prev.to(torch.int32), greedy=True, s=ss)
        ref_k, post_k = orc.p_sample_ids(known.clamp(min=0), tt, prev.to(torch.int32), greedy=True, s=ss)
        ref = torch.where(is_known, ref_k, ref_u)
        clear = torch.where(is_known, _clear(post_k, 1e-3), _clear(post_u, 0.08))
        got = trace[step].cpu().long()
        checked += int(clear.sum())
        checked_k += int((clear & is_known).sum())
        agree += int((got[clear] == ref[clear]).sum())
        prev = got
    assert checked > 0.3 * prev.numel() * 4 and checked_k > 0.5 * int(is_known.sum()) * 4 and agree == checked, \
        (agree, checked, checked_k)
    assert torch.equal(torch.cat(out).cpu(), torch.where(is_known, known, prev))


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_known_codes_graph_seed_batch_sharding_and_cached_sessions(L, transition):
    from vall_e.b200.shard import generate_sharded
    m, _, text, proms = _setup(transition)
    masks = _masks(LENS, 256, seed=4)
    kl = masks["random"]
    a = m.generate_audio(text, proms, known_list=kl, seed=5, sample_steps=4)
    b = m.generate_audio(text, proms, known_list=kl, seed=5, sample_steps=4, use_graph=False)
    again = m.generate_audio(text, proms, known_list=kl, seed=5, sample_steps=4)
    c = m.generate_audio(text, proms, known_list=kl, seed=6, sample_steps=4)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert all(torch.equal(x, y) for x, y in zip(a, again))
    assert any(not torch.equal(x, y) for x, y in zip(a, c))
    # alone and inside the batch
    solo = m.generate_audio(text[1:], proms[1:], known_list=kl[1:], seed=5, gids=[1], sample_steps=4)
    assert torch.equal(solo[0], a[1])
    # through generate_sharded: generate_fn indexes known_list by the global ids it receives
    gen = lambda tx, pr, lens, gids: m.generate_audio(tx, pr, resp_lens=lens, gids=gids, seed=5, sample_steps=4,
                                                      known_list=[kl[i] for i in gids])
    sh = generate_sharded(gen, text, proms, LENS)
    assert all(torch.equal(x, y) for x, y in zip(a, sh))
    for shard in ([0], [1]):                      # what each rank of a two-GPU run computes
        part = gen([text[i] for i in shard], [proms[i] for i in shard], [LENS[i] for i in shard], shard)
        assert torch.equal(part[0], a[shard[0]])
    # one cached session, alternating conditional / unconditional / other masks: each equals a fresh session
    eng = m.engine()
    calls = [None, kl, None, masks["level0"], kl]
    got = [m.generate_audio(text, proms, resp_lens=LENS, known_list=k, seed=7) for k in calls]
    for k, x in zip(calls, got):
        eng.__dict__.pop("_sessions", None)
        fresh = m.generate_audio(text, proms, resp_lens=LENS, known_list=k, seed=7)
        assert all(torch.equal(p, q) for p, q in zip(x, fresh)), k is None


def test_cli_continue_from_end_to_end(tmp_path, monkeypatch):
    """--continue-from PART.wav through the stand-in EnCodec: the written response starts with PART's codes."""
    import sys

    from cli_helpers import run_cli, standin_reference_emb
    ref = standin_reference_emb(tmp_path / "standin")
    main, calls, out = run_cli(tmp_path, monkeypatch, "cuda", ref)
    import vall_e.emb.qnt as qnt
    part = tmp_path / "part.wav"
    part.write_bytes(b"RIFF")
    prefix = qnt.encode_from_file(part)[0].t().cpu()                    # (12, 8)
    written = []
    real = qnt.decode_to_file
    monkeypatch.setattr(qnt, "decode_to_file", lambda resps, path: (written.append(resps.cpu()), real(resps, path)))
    monkeypatch.setattr(sys, "argv", sys.argv + ["--continue-from", str(part)])
    main()
    assert out.exists()
    (resps,) = written
    assert tuple(resps.shape) == (20, 8)
    assert torch.equal(resps[: prefix.shape[0]], prefix.long())
