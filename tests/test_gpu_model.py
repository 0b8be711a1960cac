"""GPU parity tests, model level: denoiser logits, NAR pass and the D3PM reverse loop through the
reference-facing API (lists of per-utterance tensors) against the oracle and the golden fixtures."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _sd(z):
    return {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}


def test_nar_logits_match_reference_golden(golden_dir):
    from vall_e.vall_e.nar import NAR
    z = np.load(golden_dir / "denoiser_nar_small.npz")
    sd = _sd(z)
    m = NAR(64, d_model=64, n_heads=int(z["n_heads"]), n_layers=int(z["n_layers"]))
    m.load_state_dict(sd)
    m = m.to(DEV)
    text = [torch.from_numpy(z[f"text{i}"]).to(DEV) for i in range(2)]
    proms = [torch.from_numpy(z[f"proms{i}"]).to(DEV) for i in range(2)]
    resps = [torch.from_numpy(z[f"resps{i}"]).to(DEV) for i in range(2)]
    logits = m._logits(text, proms, resps, torch.from_numpy(z["levels"]), use_time=False)
    for i in range(2):
        ref = torch.from_numpy(z[f"logits{i}"])[-len(resps[i]):]
        err = (logits[i].cpu() - ref).abs().max().item()
        assert err <= 2e-2, err          # BASELINE.json: max-abs <= 2e-2 on logits (bf16 compute)


def test_diffusion_logits_match_reference_golden(golden_dir):
    from vall_e.vall_e.diffusion import Diffusion
    z = np.load(golden_dir / "denoiser_diffusion_small.npz")
    sd = _sd(z)
    m = Diffusion(64, d_model=64, n_heads=int(z["n_heads"]), n_layers=int(z["n_layers"]), n_steps=int(z["S"]))
    m.load_state_dict(sd)
    m = m.to(DEV)
    text = [torch.from_numpy(z[f"text{i}"]).to(DEV) for i in range(2)]
    proms = [torch.from_numpy(z[f"proms{i}"]).to(DEV) for i in range(2)]
    xt = [torch.from_numpy(z[f"xt{i}"]).to(DEV) for i in range(2)]
    logits = m.denoise_logits(text, proms, xt, torch.from_numpy(z["t"]))
    for i in range(2):
        ref = torch.from_numpy(z[f"logits{i}"])[-len(xt[i]):].view(len(xt[i]), 8, 64)
        err = (logits[i].cpu() - ref).abs().max().item()
        assert err <= 2e-2, err


def _make(n_tokens, d, h, nl, S, transition, seed=0):
    from oracle import denoiser as on
    from vall_e.vall_e.diffusion import Diffusion
    sd = on.random_state_dict(n_tokens, d, nl, S + 1, n_resp_levels=8, n_out=8 * n_tokens, seed=seed,
                              time_rows=S + 1)
    m = Diffusion(n_tokens, d_model=d, n_heads=h, n_layers=nl, n_steps=S, transition=transition)
    m.load_state_dict(sd)
    return m.to(DEV), sd


def _batch(n_tokens, lens, seed):
    g = torch.Generator().manual_seed(seed)
    text = [torch.randint(1, n_tokens, (a,), generator=g) for a, _, _ in lens]
    proms = [torch.randint(0, n_tokens, (b, 8), generator=g) for _, b, _ in lens]
    xt = [torch.randint(0, n_tokens, (c, 8), generator=g) for _, _, c in lens]
    return text, proms, xt


@pytest.mark.parametrize("d,h", [(128, 2), (256, 4)])
def test_diffusion_logits_vs_oracle_ragged_batch(d, h):
    from oracle import denoiser as on
    K, nl, S = 256, 3, 30
    m, sd = _make(K, d, h, nl, S, "absorbing")
    lens = [(7, 40, 130), (30, 225, 225), (1, 3, 1), (50, 100, 260)]
    text, proms, xt = _batch(K, lens, 5)
    t = torch.tensor([29, 1, 7, 15])
    ref = on.diffusion_logits(sd, text, proms, xt, t, h, nl)
    got = m.denoise_logits([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [x.to(DEV) for x in xt], t)
    for r, g_ in zip(ref, got):
        err = (g_.cpu() - r).abs().max().item()
        assert err <= 2e-2, err


def test_hidden_states_vs_oracle_and_simt_path():
    """Layer-by-layer residual stream against the oracle; tcgen05 path against the CUDA-core path."""
    from oracle import denoiser as on
    from vall_e.b200.engine import BatchLayout, DenoiserEngine
    K, d, h, nl, S = 128, 128, 2, 2, 10
    m, sd = _make(K, d, h, nl, S, "absorbing", seed=3)
    lens = [(5, 20, 140), (9, 64, 190)]
    text, proms, xt = _batch(K, lens, 9)
    t = torch.tensor([4, 9])
    _, hid_ref = on.base_forward_logits(sd, text, proms, xt, t, h, nl, time_t=t, return_hidden=True)
    eng = m.engine()
    lay = BatchLayout(text, proms, [len(x) for x in xt], DEV)
    ws = eng.workspace(lay, logits_dtype=torch.float32)
    resp = torch.cat(xt).to(DEV, torch.int32)
    hid = []
    logits = eng.forward(lay, ws, resp, t.to(DEV, torch.int32), use_time=True, hidden_out=hid).clone()
    for li in range(nl):
        ref = torch.cat(hid_ref[li])
        err = (hid[li].cpu() - ref).abs().max().item()
        assert err < 5e-2, (li, err)
    simt = DenoiserEngine(eng.w, simt=True)
    ws2 = simt.workspace(lay, logits_dtype=torch.float32)
    logits2 = simt.forward(lay, ws2, resp, t.to(DEV, torch.int32), use_time=True)
    assert (logits - logits2).abs().max().item() < 3e-2     # two bf16 pipelines, different summation orders


@pytest.mark.parametrize("transition", ["absorbing", "uniform"])
def test_reverse_loop_teacher_forced_vs_oracle(transition):
    """Every step of generate_audio against the oracle step (oracle denoiser logits in fp16 ->
    oracle p_sample, greedy) on the trajectory the CUDA path produced."""
    from oracle import denoiser as on
    from oracle.d3pm import D3PM
    K, d, h, nl, S = 64, 64, 1, 2, 8
    m, sd = _make(K, d, h, nl, S, transition, seed=11)
    lens = [(4, 10, 24), (6, 7, 33)]
    text, proms, _ = _batch(K, lens, 13)
    orc = D3PM(S, K, transition)
    trace = []
    x0 = torch.full((24 + 33, 8), K // 2, dtype=torch.long)
    g = torch.Generator().manual_seed(1)
    if transition == "uniform":
        x0 = torch.randint(0, K, (24 + 33, 8), generator=g)
    resps = list(x0.split([24, 33]))
    out = m.generate_audio([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [r.to(DEV) for r in resps],
                           greedy=True, trace=trace, use_graph=False)
    assert [tuple(o.shape) for o in out] == [(24, 8), (33, 8)]
    prev = x0
    checked = agree = 0
    for step, t in enumerate(range(S - 1, 0, -1)):
        tt = torch.tensor([t, t])
        logits = on.diffusion_logits(sd, text, proms, list(prev.split([24, 33])), tt, h, nl)
        lg = torch.cat(logits).to(torch.float16)                       # (57, 8, K)
        tok_t = torch.full((lg.shape[0],), t)
        ref, post = orc.p_sample(lg, tok_t, prev.to(torch.int32), greedy=True)
        top2 = post.float().topk(2, dim=-1).values
        clear = (top2[..., 0] - top2[..., 1]) > 0.08
        got = trace[step].cpu().long()
        checked += int(clear.sum())
        agree += int((got[clear] == ref[clear]).sum())
        prev = got                                                      # teacher forcing on our trajectory
    assert checked > 100 and agree == checked, (agree, checked)
    assert torch.equal(torch.cat(out).cpu(), prev)


def test_generate_graph_equals_eager_and_is_seed_reproducible():
    K, d, h, nl, S = 64, 128, 2, 2, 12
    m, _ = _make(K, d, h, nl, S, "absorbing", seed=21)
    lens = [(4, 10, 40), (6, 7, 150)]
    text, proms, _ = _batch(K, lens, 3)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    a = m.generate_audio(text, proms, resp_lens=[40, 150], seed=5, use_graph=True)
    b = m.generate_audio(text, proms, resp_lens=[40, 150], seed=5, use_graph=False)
    c = m.generate_audio(text, proms, resp_lens=[40, 150], seed=6, use_graph=True)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert any(not torch.equal(x, y) for x, y in zip(a, c))
    assert all(int(x.min()) >= 0 and int(x.max()) < K for x in a)
    # sharding invariance: utterance 1 alone with its global id gives the same codes
    solo = m.generate_audio(text[1:], proms[1:], resp_lens=[150], seed=5, gids=[1])
    assert torch.equal(solo[0], a[1])


def test_d3pm_methods_reference_shapes():
    """q_sample / p_sample with the reference's (B, W) call shapes (ar_discrete.py:401-420,467-487)."""
    import detrand
    from oracle.d3pm import D3PM
    K, S = 64, 20
    m, _ = _make(K, 64, 1, 1, S, "absorbing", seed=2)
    orc = D3PM(S, K, "absorbing")
    B, W = 3, 17
    x0 = torch.from_numpy(detrand.integers(5, 0, K, (B, W)))
    t = torch.tensor([1, 10, 19])
    mask = torch.ones(W, dtype=torch.long)
    noise = torch.from_numpy(detrand.uniform(6, (B, W, K)))
    got = m.q_sample(x0.to(DEV), t.to(DEV), mask.to(DEV), noise.to(DEV))
    assert torch.equal(got.cpu(), orc.q_sample(x0, t, mask, noise))
    logits = torch.from_numpy(detrand.normal(7, (B, W, K))).to(torch.float16)
    samp, p0 = m.p_sample(logits.to(DEV), t.to(DEV), got, greedy=True)
    assert samp.shape == (B, W) and p0.shape == (B, W, K) and samp.dtype == torch.int64
    post = m.q_posterior_logits(logits.to(DEV), got, t.to(DEV))
    ref = orc.q_posterior_logits(logits, got.cpu().to(torch.int32), t)
    assert (torch.softmax(post.cpu(), -1) - torch.softmax(ref.float(), -1)).abs().max().item() < 5e-3


def test_cpu_tensors_fail_loudly():
    from vall_e.b200 import lib as L
    from vall_e.vall_e.nar import NAR
    m = NAR(64, d_model=64, n_heads=1, n_layers=1)
    with pytest.raises(L.VB200Error):
        m([torch.tensor([1, 2])], [torch.zeros(3, 8, dtype=torch.long)], [torch.zeros(4, 1, dtype=torch.long)])


def test_layernorm_variant_and_nar_level_loop():
    """norm_type == 'ln' (base.py:175-176) through the same kernels, and the NAR level loop API."""
    from oracle import denoiser as on
    from vall_e.vall_e.base import Base
    from vall_e.vall_e.nar import NAR

    class LnModel(Base):
        casual = False
        n_resp_levels = 7
        use_stop_token = False
        norm_type = "ln"
        resp_loss_only = True

    K, d, h, nl = 64, 128, 2, 2
    torch.manual_seed(0)
    m = LnModel(K, d_model=d, n_heads=h, n_layers=nl)
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(p.bfloat16().float())
        for blk in m.blocks:
            for sub in (blk.attn, blk.ffn):
                sub.norm.weight.copy_((1 + 0.1 * torch.randn(d)).bfloat16().float())
                sub.norm.bias.copy_((0.1 * torch.randn(d)).bfloat16().float())
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    lens = [(5, 9, 40), (8, 17, 140)]
    g = torch.Generator().manual_seed(4)
    text = [torch.randint(1, K, (a,), generator=g) for a, _, _ in lens]
    proms = [torch.randint(0, K, (b, 8), generator=g) for _, b, _ in lens]
    resps = [torch.randint(0, K, (c, 2), generator=g) for _, _, c in lens]
    ref = on.base_forward_logits(sd, text, proms, resps, torch.zeros(2, dtype=torch.long), h, nl, norm_type="ln")
    got = m._logits([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [x.to(DEV) for x in resps],
                    torch.zeros(2, dtype=torch.long), use_time=False)
    for r, g_, rs in zip(ref, got, resps):
        assert (g_.cpu() - r[-len(rs):]).abs().max().item() <= 2e-2

    nar = NAR(K, d_model=d, n_heads=h, n_layers=nl).to(DEV)
    out = nar([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [r[:, :1].to(DEV) for r in resps])
    assert [tuple(o.shape) for o in out] == [(40, 8), (140, 8)]
    assert all(torch.equal(o[:, 0].cpu(), r[:, 0]) for o, r in zip(out, resps))
    assert all(int(o.min()) >= 0 and int(o.max()) < K for o in out)
    with pytest.raises(ValueError):
        nar([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [resps[0][:, :1].to(DEV), resps[1][:, :2].to(DEV)])


def test_long_and_degenerate_utterances_tcgen05_vs_cuda_core_path():
    """30 s utterance (T = 2 527, the C4 shape) next to degenerate ones (1 phone / 1 prompt frame /
    1 response frame): tcgen05 path against the independent CUDA-core path, same packed layout."""
    from vall_e.b200.engine import BatchLayout, DenoiserEngine
    K, d, h, nl, S = 64, 128, 2, 2, 10
    m, _ = _make(K, d, h, nl, S, "absorbing", seed=5)
    lens = [(50, 225, 2250), (1, 1, 1), (2, 3, 255), (7, 120, 128)]
    text, proms, xt = _batch(K, lens, 17)
    t = torch.tensor([9, 0, 3, 5])
    eng = m.engine()
    lay = BatchLayout(text, proms, [len(x) for x in xt], DEV)
    assert lay.max_T == 2527 and lay.M == 2527 + 5 + 262 + 257
    resp = torch.cat(xt).to(DEV, torch.int32)
    ws = eng.workspace(lay, logits_dtype=torch.float32)
    a = eng.forward(lay, ws, resp, t.to(DEV, torch.int32), use_time=True).clone()
    simt = DenoiserEngine(eng.w, simt=True)
    ws2 = simt.workspace(lay, logits_dtype=torch.float32)
    b = simt.forward(lay, ws2, resp, t.to(DEV, torch.int32), use_time=True)
    assert torch.isfinite(a).all()
    assert (a - b).abs().max().item() < 3e-2


def test_generate_uniform_transition_graph_and_empty_edge_cases():
    from vall_e.b200 import lib as L
    K, d, h, nl, S = 64, 64, 1, 1, 6
    m, _ = _make(K, d, h, nl, S, "uniform", seed=8)
    g = torch.Generator().manual_seed(2)
    text = [torch.randint(1, K, (3,), generator=g).to(DEV)]
    proms = [torch.randint(0, K, (5, 8), generator=g).to(DEV)]
    a = m.generate_audio(text, proms, resp_lens=[33], seed=1)
    b = m.generate_audio(text, proms, resp_lens=[33], seed=1, use_graph=False)
    assert torch.equal(a[0], b[0]) and a[0].shape == (33, 8)
    with pytest.raises(ValueError):
        m.generate_audio([], [], resp_lens=[])
    # zero-row launches are accepted and do nothing
    e = torch.empty(0, 64, dtype=torch.bfloat16, device=DEV)
    w = torch.zeros(64, 64, dtype=torch.bfloat16, device=DEV)
    L.gemm_bf16(torch.empty(0, 64, dtype=torch.float32, device=DEV), e, w)
    L.gather_rows_bf16(e, torch.empty(0, 64, device=DEV), torch.empty(0, dtype=torch.int32, device=DEV))


def test_full_size_model_size_independent_properties():
    """BASELINE.json's full configuration (d=1024, 16 heads, 12 layers, K=1024, 8 levels) at the C2 /
    C4 utterance shapes, through properties that need no oracle at this size: the packed layout has
    no padding and the Philox stream is keyed by (seed, global utterance id, frame, level, t), so an
    utterance's codes must not depend on what else is in the batch, on graph replay versus eager
    launches, or on the run; every code is a valid class; a different seed changes the draw."""
    from vall_e.vall_e.diffusion import Diffusion
    torch.manual_seed(0)
    S = 6
    m = Diffusion(1024, d_model=1024, n_heads=16, n_layers=12, n_steps=S, transition="absorbing")
    for blk in m.blocks:
        for sub in (blk.attn, blk.ffn):
            torch.nn.init.normal_(sub.norm.emb.weight, std=0.02)
    m = m.to(DEV)
    lens = [(50, 225, 750), (37, 225, 2250), (3, 1, 130)]          # C2, C4 and a short ragged one
    text, proms, _ = _batch(1024, lens, 9)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    resp = [c for _, _, c in lens]
    a = m.generate_audio(text, proms, resp_lens=resp, seed=11, use_graph=True)
    b = m.generate_audio(text, proms, resp_lens=resp, seed=11, use_graph=False)
    c = m.generate_audio(text, proms, resp_lens=resp, seed=12, use_graph=True)
    assert [tuple(x.shape) for x in a] == [(r, 8) for r in resp]
    assert all(torch.equal(x, y) for x, y in zip(a, b))                    # graph replay == eager launches
    assert all(not torch.equal(x, y) for x, y in zip(a, c))                # the seed matters
    assert all(int(x.min()) >= 0 and int(x.max()) < 1024 for x in a)
    for i in (0, 1):                                                       # alone, with its global id
        solo = m.generate_audio(text[i:i + 1], proms[i:i + 1], resp_lens=resp[i:i + 1], seed=11, gids=[i])
        assert torch.equal(solo[0], a[i]), i
    rev = m.generate_audio(text[::-1], proms[::-1], resp_lens=resp[::-1], seed=11, gids=[2, 1, 0])
    assert all(torch.equal(x, y) for x, y in zip(rev[::-1], a))            # batch order does not matter


def test_training_forward_loss_vs_oracle_and_torch():
    """SURVEY §8f.3: q_sample with in-kernel noise + cross-entropy as the classifier GEMM's epilogue.
    (a) the loss of Diffusion.d3pm_loss equals the cross-entropy of the ORACLE's logits on the same
    x_t (tolerance: the 2e-2 logits bar); (b) the fused per-token losses equal torch's CE on this
    library's own logits; (c) the O(1) Philox q_sample follows the table's categorical law."""
    from oracle import denoiser as on
    from vall_e.b200 import lib as L
    from vall_e.vall_e import d3pm as pd
    K, d, h, nl, S = 256, 128, 2, 2, 12
    m, sd = _make(K, d, h, nl, S, "absorbing", seed=31)
    lens = [(5, 9, 33), (7, 4, 70)]
    text, proms, x0 = _batch(K, lens, 5)
    dtext, dproms, dx0 = [x.to(DEV) for x in text], [x.to(DEV) for x in proms], [x.to(DEV) for x in x0]
    t = torch.tensor([4, 9])
    total, per_tok, x_t = m.d3pm_loss(dtext, dproms, dx0, t, seed=3, return_per_token=True)
    xt_list = [r.cpu().long() for r in x_t.split([c for _, _, c in lens])]
    ref_logits = on.diffusion_logits(sd, text, proms, xt_list, t, h, nl)
    ce = []
    for lg, tgt in zip(ref_logits, x0):
        lg = torch.as_tensor(lg).double().reshape(len(tgt), 8, K)
        ce.append(torch.nn.functional.cross_entropy(lg.reshape(-1, K), tgt.reshape(-1), reduction="none"))
    ce = torch.cat(ce)
    assert abs(total.item() - ce.mean().item()) < 2e-2, (total.item(), ce.mean().item())
    assert (per_tok.cpu().double().view(-1) - ce).abs().max().item() < 6e-2
    # (b) against torch on this library's own fp32 logits
    own = m.denoise_logits(dtext, dproms, [x.to(DEV) for x in xt_list], t)
    own_ce = torch.cat([torch.nn.functional.cross_entropy(lg.reshape(-1, K).float(), tgt.to(DEV).reshape(-1),
                                                          reduction="none") for lg, tgt in zip(own, x0)])
    assert (per_tok.view(-1) - own_ce).abs().max().item() < 2e-3
    # sweep form runs and is reproducible
    a = m.d3pm_loss(dtext, dproms, dx0, None, seed=1)
    b = m.d3pm_loss(dtext, dproms, dx0, None, seed=1)
    assert torch.equal(a, b) and math.isfinite(a.item())
    # (c) law of the Philox q_sample: absorbing, x0 != m
    n, t0 = 200000, 7
    table = pd.scalar_table(S + 1, K, "absorbing").to(DEV)
    x0v = torch.full((n,), 5, dtype=torch.int32, device=DEV)
    tt = torch.full((n,), t0, dtype=torch.int32, device=DEV)
    out = torch.empty_like(x0v)
    L.q_sample_philox(out, x0v, tt, None, table, K, L.ABSORBING, seed=9)
    row = table[t0].cpu().double()
    w = torch.full((K,), math.exp(row[L.TAB_LOG_OFF].item()), dtype=torch.float64)
    w[5], w[K // 2] = math.exp(row[L.TAB_LOG_KEEP].item()), math.exp(row[L.TAB_LOG_ABSORB].item())
    p = w / w.sum()
    counts = torch.bincount(out.cpu().long(), minlength=K).double()
    for j in (5, K // 2):
        exp_j = p[j].item() * n
        assert abs(counts[j].item() - exp_j) < 6 * math.sqrt(exp_j * (1 - p[j].item())) + 1, (j, counts[j].item(), exp_j)
    rest_exp = n - (p[5] + p[K // 2]).item() * n
    rest_obs = n - counts[5].item() - counts[K // 2].item()
    assert abs(rest_obs - rest_exp) < 6 * math.sqrt(max(rest_exp, 1.0)) + 1


def test_encodec_handoff_bqt_layout_matches_reference_rearrange():
    """SURVEY §8f.4: the batch hand-off to the EnCodec decoder (emb/qnt.py:32-49).  The (B, 8, T_max)
    tensor must hold, per utterance, exactly what the reference builds one utterance at a time with
    rearrange(resps, "t q -> 1 q t") (emb/qnt.py:46), zero-padded past its length.  Bit-exact."""
    from vall_e.b200 import lib as L
    K, d, h, nl, S = 64, 128, 2, 2, 8
    m, _ = _make(K, d, h, nl, S, "absorbing", seed=4)
    lens = [(4, 10, 40), (6, 7, 301), (3, 5, 1)]
    text, proms, _ = _batch(K, lens, 9)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    rl = [x[2] for x in lens]
    codes = m.generate_audio(text, proms, resp_lens=rl, seed=3)
    bqt, frames = m.generate_audio(text, proms, resp_lens=rl, seed=3, as_bqt=True)
    assert frames == rl and bqt.shape == (3, 8, 301) and bqt.dtype == torch.int64
    for b, c in enumerate(codes):
        ref = c.t()[None]                                   # "t q -> 1 q t"
        assert torch.equal(bqt[b:b + 1, :, :rl[b]], ref)
        assert int(bqt[b, :, rl[b]:].abs().sum()) == 0
    host, _ = m.generate_audio(text, proms, resp_lens=rl, seed=3, as_bqt=True, to_host=True)
    assert not host.is_cuda and torch.equal(host, bqt.cpu())
    # the kernel on its own, other level counts and a non-zero pad value; empty batch is a no-op
    g = torch.Generator().manual_seed(0)
    for n_levels, tl in ((1, [5, 300, 17]), (3, [257, 256, 255, 1])):
        packed = torch.randint(0, 1024, (sum(tl), n_levels), generator=g, dtype=torch.int32)
        utt = torch.zeros(len(tl), L.U_STRIDE, dtype=torch.int32)
        utt[:, L.U_TRESP] = torch.tensor(tl, dtype=torch.int32)
        utt[:, L.U_RESP0] = torch.tensor([0] + list(np.cumsum(tl)[:-1]), dtype=torch.int32)
        out = torch.empty(len(tl), n_levels, max(tl), dtype=torch.int64, device=DEV)
        L.codes_to_bqt(out, packed.to(DEV), utt.to(DEV), pad=-7)
        ref = torch.full(out.shape, -7, dtype=torch.int64)
        for b, chunk in enumerate(packed.split(tl)):
            ref[b, :, :tl[b]] = chunk.t().long()
        assert torch.equal(out.cpu(), ref)
    L.codes_to_bqt(torch.empty(0, 8, 4, dtype=torch.int64, device=DEV), torch.empty(0, 8, dtype=torch.int32, device=DEV),
                   torch.empty(0, L.U_STRIDE, dtype=torch.int32, device=DEV))


def test_ar_discrete_compat_reverse_step_and_loop(golden_dir):
    """SURVEY §8f.2: the drop-in for the reference's own D3PM class (K = 1025, level 0, d = 32 DiT).
    Denoiser logits on the GPU agree with the reference fixture; one reverse step on those logits
    agrees with the oracle's dense fp16-table p_sample (supplied uniforms and greedy, wherever the
    reference's top-2 margin is clear); the 99-step loop runs, is seed-reproducible, and returns the
    reference's (448,) layout."""
    import detrand
    from oracle.d3pm import D3PM
    from test_host_cpu import _compat_dit
    m, z, _, text, proms, x_t = _compat_dit(golden_dir)
    m = m.to(DEV)
    t = torch.tensor([int(z["t"])], device=DEV)
    with torch.no_grad():
        cond1, cond2 = m.conditioning(text.to(DEV), proms.to(DEV))
        logits = m.denoise_logits(x_t.to(DEV), t, cond1, cond2, (x_t[0] != 0).to(DEV))
    err = np.abs(logits[0, torch.from_numpy(z["rows"]).to(DEV)].cpu().numpy() - z["logits_rows"]).max()
    assert err <= 2e-3, err                    # fp32 (TF32 off) PyTorch modules; fp16 sin/cos tables differ in the last bit
    orc = D3PM(100, 1025, "absorbing")
    noise = torch.from_numpy(detrand.uniform(5, (1, 448, 1025)))
    lg16 = logits.cpu().to(torch.float16)
    ref_samp, ref_post = orc.p_sample(lg16, t.cpu(), x_t, noise)
    ref_greedy, _ = orc.p_sample(lg16, t.cpu(), x_t, greedy=True)
    got, probs = m.p_sample(logits, t, x_t.to(DEV), noise=noise.to(DEV))
    greedy, _ = m.p_sample(logits, t, x_t.to(DEV), greedy=True)
    assert got.shape == (1, 448) and probs.shape == (1, 448, 1025)
    g = -torch.log(-torch.log(noise.clamp(min=torch.finfo(torch.float32).tiny)))
    top2 = (ref_post.float() + g).topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05
    assert clear.float().mean().item() > 0.8
    assert torch.equal(got.cpu()[clear], ref_samp[clear])
    top2 = ref_post.float().topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 0.05
    assert torch.equal(greedy.cpu()[clear], ref_greedy[clear])
    a = m.generate_audio([text.to(DEV)], [proms.to(DEV)], seed=7)
    b = m.generate_audio([text.to(DEV)], [proms.to(DEV)], seed=7)
    c = m.generate_audio([text.to(DEV)], [proms.to(DEV)], seed=8)
    assert a.shape == (448,) and a.dtype == torch.int64 and int(a.min()) >= 0 and int(a.max()) < 1025
    assert torch.equal(a, b) and not torch.equal(a, c)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_second_device_in_the_same_process():
    """Kernel attributes (dynamic shared memory limits) are per device: a process that drives two GPUs
    must get identical codes from both (one-process-per-GPU is the deployment, this is the guard)."""
    K, d, h, nl, S = 64, 128, 2, 2, 8
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        with torch.cuda.device(dev):
            m, _ = _make(K, d, h, nl, S, "absorbing", seed=4)
            m = m.to(dev)
            text, proms, _ = _batch(K, [(4, 10, 140), (6, 7, 301)], 9)
            outs.append([c.cpu() for c in m.generate_audio([x.to(dev) for x in text], [x.to(dev) for x in proms],
                                                            resp_lens=[140, 301], seed=3)])
    assert all(torch.equal(a, b) for a, b in zip(*outs))
    # a model on cuda:1 while the CURRENT device is cuda:0 (`python -m vall_e --device cuda:1`): the model
    # classes switch device themselves, so the codes are the same again ...
    assert torch.cuda.current_device() == 0
    m, _ = _make(K, d, h, nl, S, "absorbing", seed=4)
    m = m.to("cuda:1")
    text, proms, _ = _batch(K, [(4, 10, 140), (6, 7, 301)], 9)
    other = m.generate_audio([x.to("cuda:1") for x in text], [x.to("cuda:1") for x in proms], resp_lens=[140, 301], seed=3)
    assert all(torch.equal(a.cpu(), b) for a, b in zip(other, outs[0]))
    assert torch.cuda.current_device() == 0
    # ... and a raw kernel call with tensors of another device is refused instead of dereferencing them on cuda:0
    from vall_e.b200 import lib as L
    t1 = torch.zeros(4, dtype=torch.int32, device="cuda:1")
    with pytest.raises(L.VB200Error, match="current CUDA device"):
        L.step_timesteps(t1, -1)
    with pytest.raises(L.VB200Error, match="different devices"):
        L.gather_rows_bf16(torch.empty(1, 64, dtype=torch.bfloat16, device="cuda:0"), torch.zeros(2, 64, device="cuda:1"),
                           torch.zeros(1, dtype=torch.int32, device="cuda:0"))


def test_wrong_ids_are_refused_before_any_launch():
    """An id outside its table (e.g. the AR stop token 1024 in a K = 1024 model) raises IndexError, as the
    reference's F.one_hot / nn.Embedding do, instead of an out-of-bounds read in the gather kernel."""
    K, d, h, nl, S = 64, 64, 1, 1, 6
    m, _ = _make(K, d, h, nl, S, "absorbing", seed=8)
    text, proms, xt = _batch(K, [(3, 5, 9)], 2)
    bad = [xt[0].clone()]
    bad[0][2, 3] = m.num_classes           # K itself is the absorbing mask id, a legal x_T entry
    with pytest.raises(IndexError):
        m.generate_audio([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [x.to(DEV) for x in bad])
    neg = proms[0].clone()
    neg[1, 2] = -1
    with pytest.raises(IndexError):
        m.generate_audio([x.to(DEV) for x in text], [neg.to(DEV)], resp_lens=[9])
    with pytest.raises(IndexError):
        m.generate_audio([torch.full_like(text[0], K).to(DEV)], [x.to(DEV) for x in proms], resp_lens=[9])
    with pytest.raises(IndexError):
        m.p_sample(torch.zeros(1, 2, m.num_classes, device=DEV), torch.tensor([1]),
                   torch.tensor([[0, m.num_classes]], device=DEV), greedy=True)


def test_uniform_start_state_is_keyed_by_global_utterance_id():
    """x_T of the uniform transition is drawn per utterance from (seed, global id): an utterance generated
    alone, or in another batch order, gets the codes it gets inside the full batch (sharding invariance)."""
    K, d, h, nl, S = 256, 128, 2, 2, 7
    m, _ = _make(K, d, h, nl, S, "uniform", seed=4)
    text, proms, _ = _batch(K, [(4, 10, 40), (6, 7, 77), (3, 3, 21)], 9)
    text, proms = [x.to(DEV) for x in text], [x.to(DEV) for x in proms]
    full = m.generate_audio(text, proms, resp_lens=[40, 77, 21], seed=5, gids=[10, 11, 12])
    solo = m.generate_audio(text[1:2], proms[1:2], resp_lens=[77], seed=5, gids=[11])
    rev = m.generate_audio(text[::-1], proms[::-1], resp_lens=[21, 77, 40], seed=5, gids=[12, 11, 10])
    assert torch.equal(solo[0], full[1])
    assert all(torch.equal(a, b) for a, b in zip(rev[::-1], full))


def test_full_size_logits_vs_oracle():
    """BASELINE.json's full denoiser (d = 1024, 16 heads, 12 layers, K = 1024 x 8 levels) against the
    oracle's fp32 forward on the same weights and inputs: the C2 sequence (50 phones + 225 prompt frames +
    750 frames, T = 1 027) and a short ragged companion in one batch.  Bar: max-abs <= 2e-2 on the logits
    (bf16 compute), as BASELINE.json states; the observed error is printed."""
    from oracle import denoiser as on
    K, d, h, nl, S = 1024, 1024, 16, 12, 50
    m, sd = _make(K, d, h, nl, S, "absorbing", seed=2)
    lens = [(50, 225, 750), (9, 33, 77)]
    text, proms, xt = _batch(K, lens, 17)
    t = torch.tensor([37, 3])
    torch.set_num_threads(max(1, min(16, torch.get_num_threads())))
    ref = on.diffusion_logits(sd, text, proms, xt, t, h, nl)
    got = m.denoise_logits([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [x.to(DEV) for x in xt], t)
    errs = [(g_.cpu() - r).abs().max().item() for r, g_ in zip(ref, got)]
    rms = [(g_.cpu() - r).pow(2).mean().sqrt().item() for r, g_ in zip(ref, got)]
    print(f"full-size logits vs oracle: max-abs {errs}, rms {rms}, logit std {ref[0].std().item():.3f}")
    assert max(errs) <= 2e-2, errs
    # greedy x_0 prediction: identical wherever the oracle's top-2 margin exceeds the logits tolerance
    for r, g_ in zip(ref, got):
        top2 = r.topk(2, dim=-1).values
        clear = (top2[..., 0] - top2[..., 1]) > 4e-2
        assert torch.equal(g_.cpu().argmax(-1)[clear], r.argmax(-1)[clear])
    # the long-form sequence of BASELINE configs[3] (C4: 2 250 frames, T = 2 527) on its own
    text, proms, xt = _batch(K, [(50, 225, 2250)], 19)
    t = torch.tensor([21])
    ref = on.diffusion_logits(sd, text, proms, xt, t, h, nl)[0]
    got = m.denoise_logits([x.to(DEV) for x in text], [x.to(DEV) for x in proms], [x.to(DEV) for x in xt], t)[0].cpu()
    err = (got - ref).abs().max().item()
    print(f"full-size logits vs oracle, C4 sequence: max-abs {err:.4f}, rms {(got - ref).pow(2).mean().sqrt().item():.5f}")
    assert err <= 2e-2, err


def test_c1_config_reverse_loop_vs_oracle():
    """BASELINE.json configs[0] / SURVEY C1, literally: the quarter model (d = 256, 4 heads, 12 layers,
    K = 1024 x 8 levels), one utterance of 3 s (30 phones + 225 prompt frames + 225 frames, T = 482), 50
    denoise steps, uniform transition, the reference's noise convention (supplied uniforms).  Every seventh
    step of the CUDA trajectory is re-done by the oracle (fp32 denoiser -> fp16 logits -> dense fp16-table
    p_sample with the same uniforms): tokens must agree wherever the oracle's noisy top-2 margin is clear."""
    import detrand
    from oracle import denoiser as on
    from oracle.d3pm import D3PM
    K, d, h, nl, S = 1024, 256, 4, 12, 51
    m, sd = _make(K, d, h, nl, S, "uniform", seed=5)
    text, proms, _ = _batch(K, [(30, 225, 225)], 21)
    x_T = torch.from_numpy(detrand.integers(77, 0, K, (225, 8)))
    noise = {t: torch.from_numpy(detrand.uniform(1000 + t, (225 * 8, K))) for t in range(1, S)}
    trace = []
    out = m.generate_audio([text[0].to(DEV)], [proms[0].to(DEV)], [x_T.to(DEV)],
                           uniforms_fn=lambda t: noise[t].to(DEV), trace=trace, use_graph=False)
    assert out[0].shape == (225, 8) and len(trace) == S - 1
    assert int(out[0].min()) >= 0 and int(out[0].max()) < K
    orc = D3PM(S, K, "uniform")
    steps = list(range(S - 1, 0, -1))
    checked = agree = 0
    for i in range(0, len(steps), 7):
        t = steps[i]
        prev = x_T if i == 0 else trace[i - 1].cpu().long()
        lg = on.diffusion_logits(sd, text, proms, [prev], torch.tensor([t]), h, nl)[0].to(torch.float16)   # (225, 8, K)
        u = noise[t].view(225, 8, K)
        ref, post = orc.p_sample(lg, torch.full((225,), t), prev.to(torch.int32), u)
        g = -torch.log(-torch.log(u.clamp(min=torch.finfo(torch.float32).tiny)))
        top2 = (post.float() + g).topk(2, dim=-1).values
        clear = (top2[..., 0] - top2[..., 1]) > 0.08
        got = trace[i].cpu().long()
        checked += int(clear.sum())
        agree += int((got[clear] == ref[clear]).sum())
    assert checked > 0.8 * 8 * 225 * 8 and agree == checked, (agree, checked)


def test_cli_main_end_to_end(tmp_path, monkeypatch):
    """``python -m vall_e <text> <ref.wav> <out.wav> --ar-ckpt <Diffusion pickle>`` in-process, all the way to
    the written file: prompt through the (stubbed) EnCodec wrapper of ``vall_e.emb.qnt``, phones through
    ``vall_e.emb.g2p``, the reverse loop on the CUDA kernels, the codes back through ``qnt.decode_to_file``.
    ``vall_e.emb`` executes the files of a stand-in checkout of the reference, written by the test."""
    from cli_helpers import run_cli, standin_reference_emb
    ref = standin_reference_emb(tmp_path / "standin")
    main, calls, out = run_cli(tmp_path, monkeypatch, "cuda", ref)
    main()
    assert out.exists()
    dec = [c for c in calls if c[0] == "decode"]
    assert dec and dec[-1][1] == (1, 8, 20)                 # (b q t): 20 frames x 8 levels went to the decoder
    wr = [c for c in calls if c[0] == "write"]
    assert wr and wr[-1][1] == str(out) and wr[-1][3] == 24_000


def test_codes_do_not_depend_on_the_launch_order_mode():
    """Programmatic dependent launch (default: GEMMs, fused classifier, one-wave attention / AdaLN; loads of weights
    and AdaLN rows hoisted in front of the wait) only moves WHEN kernels start: the full-size model generates the
    same codes with it, without it (VB200_PDL=0) and with it on every launch (VB200_PDL=255), for one utterance
    (every kernel one wave) and for a ragged batch.  The mask is read once per process, hence subprocesses."""
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    child = r'''
import sys, hashlib, torch
sys.path.insert(0, %r); sys.path.insert(0, %r)
import bench
from vall_e.vall_e.diffusion import Diffusion
torch.manual_seed(0)
m = Diffusion(**bench.MODEL, n_steps=7, transition="absorbing")
for blk in m.blocks:
    for sub in (blk.attn, blk.ffn):
        torch.nn.init.normal_(sub.norm.emb.weight, std=0.02)
m = m.to("cuda")
h = hashlib.sha256()
for shapes in ([(50, 225, 750)], [(50, 225, 300), (7, 40, 130), (30, 100, 333)]):
    utts = [bench.synth_utterance(i, a, b) for i, (a, b, _) in enumerate(shapes)]
    out = m.generate_audio([u[0].cuda() for u in utts], [u[1].cuda() for u in utts], resp_lens=[c for _, _, c in shapes], seed=9)
    h.update(torch.cat(out).cpu().numpy().tobytes())
print("CODES", h.hexdigest())
''' % (str(root), str(root / "tts-with-diffusion-model_b200"))
    digests = {}
    for mask in (None, "0", "255"):
        env = dict(os.environ)
        env.pop("VB200_PDL", None)
        if mask is not None:
            env["VB200_PDL"] = mask
        r = subprocess.run([sys.executable, "-c", child], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        digests[mask] = [ln for ln in r.stdout.splitlines() if ln.startswith("CODES")][-1]
    assert digests[None] == digests["0"] == digests["255"], digests
