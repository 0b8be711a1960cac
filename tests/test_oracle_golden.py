"""Pins the oracle (oracle/*.py) against fixtures produced by the reference's own code
(tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

import detrand
from oracle import d3pm as od
from oracle import denoiser as on


@pytest.fixture(scope="module", params=["absorbing", "uniform"])
def d3pm_case(request, golden_dir):
    z = np.load(golden_dir / f"d3pm_{request.param}_k1025.npz")
    return request.param, z, od.D3PM(int(z["S"]), int(z["K"]), request.param)


def test_tables_bit_exact(d3pm_case):
    tr, z, d = d3pm_case
    m = d.K // 2
    assert np.array_equal(z["betas"], d.betas.numpy())
    one, cum = d.q_onestep_mats.float().numpy(), d.q_mats.float().numpy()
    for name, arr in (("one_aa", one[:, 0, 0]), ("one_ab", one[:, 0, 1]), ("one_am", one[:, 0, m]),
                      ("one_mm", one[:, m, m]), ("cum_aa", cum[:, 0, 0]), ("cum_ab", cum[:, 0, 1]),
                      ("cum_am", cum[:, 0, m]), ("cum_mm", cum[:, m, m]), ("cum_ma", cum[:, m, 0])):
        assert np.array_equal(z[name], arr), name


def _inputs(z):
    seed, W, K = int(z["seed"]), int(z["W"]), int(z["K"])
    t = torch.from_numpy(z["q_t"])
    x0 = torch.from_numpy(detrand.integers(seed, 0, 1024, (len(t), W)))
    x0[:, 0] = K // 2
    x0[:, 1] = 1024
    mask = torch.ones(W, dtype=torch.int64)
    mask[-3:] = 0
    nq = torch.from_numpy(detrand.uniform(seed + 1, (len(t), W, K)))
    logits = torch.from_numpy(detrand.normal(seed + 2, (len(t), W, K)) * 2.0).to(torch.float16)
    npn = torch.from_numpy(detrand.uniform(seed + 3, (len(t), W, K)))
    return t, x0, mask, nq, logits, npn


def test_q_sample_bit_exact(d3pm_case):
    _, z, d = d3pm_case
    t, x0, mask, nq, _, _ = _inputs(z)
    xt = d.q_sample(x0, t, mask, nq)
    assert np.array_equal(xt.numpy().astype(np.int32), z["q_xt"])


def test_p_sample_bit_exact(d3pm_case):
    _, z, d = d3pm_case
    t, _, _, _, logits, npn = _inputs(z)
    x_in = torch.from_numpy(z["q_xt"])
    samp, post = d.p_sample(logits, t, x_in, npn)
    assert np.array_equal(samp.numpy().astype(np.int32), z["p_sample"])
    assert np.array_equal(post[:, :6].numpy(), z["p_post_head"])
    greedy, _ = d.p_sample(logits, t, x_in, greedy=True)
    assert np.array_equal(greedy.numpy().astype(np.int32), z["p_greedy"])


def _sd(z):
    return {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}


def test_denoiser_nar_matches_reference(golden_dir):
    z = np.load(golden_dir / "denoiser_nar_small.npz")
    sd = _sd(z)
    text = [torch.from_numpy(z[f"text{i}"]) for i in range(2)]
    proms = [torch.from_numpy(z[f"proms{i}"]) for i in range(2)]
    resps = [torch.from_numpy(z[f"resps{i}"]) for i in range(2)]
    out, hid = on.base_forward_logits(sd, text, proms, resps, torch.from_numpy(z["levels"]),
                                      int(z["n_heads"]), int(z["n_layers"]), return_hidden=True)
    for i in range(2):
        assert np.abs(out[i].numpy() - z[f"logits{i}"]).max() < 2e-5
        assert np.abs(hid[0][i].numpy() - z[f"hidden_first{i}"]).max() < 2e-5
        assert np.abs(hid[-1][i].numpy() - z[f"hidden_last{i}"]).max() < 5e-5


def test_denoiser_diffusion_matches_reference(golden_dir):
    z = np.load(golden_dir / "denoiser_diffusion_small.npz")
    sd = _sd(z)
    text = [torch.from_numpy(z[f"text{i}"]) for i in range(2)]
    proms = [torch.from_numpy(z[f"proms{i}"]) for i in range(2)]
    xt = [torch.from_numpy(z[f"xt{i}"]) for i in range(2)]
    t = torch.from_numpy(z["t"])
    rows = on.base_forward_logits(sd, text, proms, xt, t, int(z["n_heads"]), int(z["n_layers"]), time_t=t)
    for i in range(2):
        assert np.abs(rows[i].numpy() - z[f"logits{i}"]).max() < 5e-5


def test_reference_arm_runs_the_staged_reference_modules():
    """oracle/refarm.py (the CPU arm of bench.py): the reference's own modules from oracle/_ref — staged by
    build() wherever a reference checkout can be read (refarm.reference_root) — run one denoise step, and the
    oracle port reproduces their logits on the same weights (fp32, <= 5e-5) and their posterior (bit-exact),
    live, not only through fixtures."""
    from oracle import denoiser as on
    from oracle import refarm
    from oracle.d3pm import D3PM
    if not refarm.stage():
        pytest.skip("oracle/_ref not staged: no readable reference checkout (VALL_E_REF, ../reference or "
                    "BASELINE.json reference_path)")
    g = torch.Generator().manual_seed(3)
    text, proms = torch.randint(1, 1025, (7,), generator=g), torch.randint(0, 1025, (11, 8), generator=g)
    S = 6
    ref = refarm.ReferenceStep(64, 1, 2, S, "absorbing", text, proms, t_resp=13, seed=5)
    x = torch.randint(0, 1025, (13, 8), generator=g)
    lg = ref.logits(x, 4)
    sd = {k: v.detach() for k, v in ref.gm.state_dict().items()}
    mine = on.diffusion_logits(sd, [text], [proms], [x], torch.tensor([4]), 1, 2)[0]
    assert (mine - lg).abs().max().item() <= 5e-5
    orc = D3PM(S, refarm.K_REF, "absorbing")
    assert torch.equal(orc.q_mats, ref.tab.q_mats) and torch.equal(orc.betas, ref.tab.betas)
    l16 = lg.to(torch.float16).view(1, -1, refarm.K_REF)
    xr = x.reshape(1, -1).to(torch.int32)
    assert torch.equal(orc.q_posterior_logits(l16, xr, torch.tensor([4])),
                       ref.tab.q_posterior_logits(l16, xr, torch.tensor([4]), x_start_logits=True))
    out = ref.step()
    assert out.shape == (13, 8) and 0 <= int(out.min()) and int(out.max()) < refarm.K_REF
