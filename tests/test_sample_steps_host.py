"""CPU tests of sampling with fewer denoise steps than timesteps (``generate_audio(sample_steps=n)``):
the schedule, the schedule table and the row invariant the reverse-step kernels rely on, the oracle's
jump posterior q(x_s | x_t, x0), argument checks and the ``--steps`` option of ``python -m vall_e``."""
import ctypes
import math
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "tts-with-diffusion-model_b200"


@pytest.mark.parametrize("S", [2, 8, 51, 101])
def test_sample_schedule(S):
    from vall_e.vall_e import d3pm as pd
    for n in range(1, S):
        sch = pd.sample_schedule(S, n)
        assert len(sch) == n and sch[0] == S - 1 and sch[-1] >= 1, (S, n, sch)
        assert all(a > b for a, b in zip(sch, sch[1:])), (S, n, sch)
        nxt = pd.successors(S, sch)
        assert [nxt[t] for t in sch] == list(sch[1:]) + [0]
    assert list(pd.sample_schedule(S, S - 1)) == list(range(S - 1, 0, -1))
    assert pd.successors(S, range(S - 1, 0, -1)) == [max(t - 1, 0) for t in range(S)]
    for bad in (0, -1, S, S + 5):
        with pytest.raises(ValueError):
            pd.sample_schedule(S, bad)


def test_sample_schedule_example_and_bad_schedules():
    from vall_e.vall_e import d3pm as pd
    assert pd.sample_schedule(51, 10) == (50, 45, 40, 35, 30, 25, 20, 15, 10, 5)
    for bad in ([], [10, 10], [5, 7], [12], [3, 0]):
        with pytest.raises(ValueError):
            pd.check_schedule(12, bad)


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_full_schedule_table_is_the_scalar_table(tr):
    from vall_e.vall_e import d3pm as pd
    for S, K in ((50, 1024), (30, 257), (2, 64)):
        full = pd.sample_schedule(S, S - 1)
        assert torch.equal(pd.schedule_table(S, K, tr, full), pd.scalar_table(S, K, tr)), (S, K)


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_jump_entries_are_the_dense_chain_product(tr):
    """Overwritten entries against the dense fp16 chain product Q_{s+1}...Q_t (and Qbar_s): exactly for
    absorbing (<= 2 non-zero terms per entry), within one fp16 ulp for uniform (K-term sums)."""
    from jump_oracle import JumpD3PM
    from vall_e.b200 import lib as L
    from vall_e.vall_e import d3pm as pd
    S, K = 50, 1024
    m = K // 2
    orc = JumpD3PM(S, K, tr)
    sch = pd.sample_schedule(S, 10)
    tab, plain = pd.schedule_table(S, K, tr, sch), pd.scalar_table(S, K, tr)
    eye = torch.eye(K, dtype=torch.bool)
    rows = torch.arange(K) != m
    changed = torch.zeros(S, dtype=torch.bool)
    worst = 0.0
    for t, s in zip(sch, sch[1:] + (0,)):
        assert s != t - 1
        changed[t] = changed[t - 1] = True
        for q, row, lo in ((orc.jump_mat(t, s).float(), t, L.TAB_ONE_KEEP), (orc.q_mats[s].float(), t - 1, L.TAB_CUM_KEEP)):
            keep, off, absorb, both = (tab[row, lo + i] for i in range(4))
            if tr == "absorbing":
                assert torch.equal(q[rows][:, rows][eye[rows][:, rows]], keep.expand(K - 1)), (t, s)
                assert torch.equal(q[rows][:, rows][~eye[rows][:, rows]], off.expand((K - 1) * (K - 2))), (t, s)
                assert torch.equal(q[rows, m], absorb.expand(K - 1)) and float(q[m, m]) == float(both), (t, s)
                assert float(q[m][rows].abs().max()) == 0.0
                continue
            for vals, ref in ((q[eye], keep), (q[~eye], off)):
                ulp = 2.0 ** (math.floor(math.log2(float(ref))) - 10)
                worst = max(worst, float((vals - ref).abs().max()) / ulp)
    assert worst <= 1.0, worst
    # every entry the schedule does not own is the plain table's
    assert torch.equal(tab[~changed], plain[~changed])
    assert torch.equal(tab[:, L.TAB_LOG_KEEP:], plain[:, L.TAB_LOG_KEEP:])


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_oracle_jump_to_t_minus_1_is_the_one_step_posterior(tr):
    from jump_oracle import JumpD3PM, posterior_fp32
    S, K, B, W = 20, 256, 6, 9
    orc = JumpD3PM(S, K, tr)
    g = torch.Generator().manual_seed(4)
    logits = (torch.randn(B, W, K, generator=g) * 2).to(torch.float16)
    x_t = torch.randint(0, K, (B, W), generator=g, dtype=torch.int32)
    x_t[:, ::2] = K // 2
    t = torch.tensor([1, 2, 7, 10, 18, 19])
    s = t - 1
    assert torch.equal(orc.q_posterior_logits(logits, x_t, t, s), orc.q_posterior_logits(logits, x_t, t))
    assert torch.equal(orc.p_sample(logits, t, x_t, greedy=True, s=s)[1], orc.p_sample(logits, t, x_t, greedy=True)[1])
    assert torch.equal(posterior_fp32(logits, x_t, t, orc, s), posterior_fp32(logits, x_t, t, orc))


def _analytic_oracle(S, K, tr):
    """The oracle with float64 analytic matrices (no fp16 rounding) and eps = 0."""
    from jump_oracle import JumpD3PM
    from oracle.d3pm import absorbing_onestep, cosine_beta_schedule
    orc = JumpD3PM(S, K, tr)
    betas = cosine_beta_schedule(S + 1).numpy()
    one = []
    for b in betas[:S]:
        if tr == "absorbing":
            one.append(absorbing_onestep(b, K))
        else:
            one.append(torch.full((K, K), b / K, dtype=torch.float64) + torch.eye(K, dtype=torch.float64) * (1 - b))
    orc.q_onestep_mats = torch.stack(one)
    cum = [one[0]]
    for q in one[1:]:
        cum.append(cum[-1] @ q)
    orc.q_mats = torch.stack(cum)
    orc.transpose_q_onestep_mats = orc.q_onestep_mats.transpose(1, 2).contiguous()
    orc.eps = 0.0
    return orc


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_oracle_jump_posterior_equals_chained_one_step_posteriors(tr):
    """q(x_s | x_t, x0) = sum over x_{t-1} .. x_{s+1} of the one-step posteriors, for every x0 and x_t
    that x0 can reach: checks the orientation of the oracle's Q_{t|s}."""
    S, K = 12, 6
    orc = _analytic_oracle(S, K, tr)
    Q, Qbar = orc.q_onestep_mats.numpy(), orc.q_mats.numpy()
    x0 = torch.arange(K).repeat_interleave(K)          # every (x0, x_t) pair
    xt = torch.arange(K).repeat(K)
    x0_logits = torch.full((1, K * K, K), -math.inf, dtype=torch.float64)
    x0_logits[0, torch.arange(K * K), x0] = 0.0
    for t, s in ((11, 0), (11, 6), (6, 2), (3, 0), (5, 4)):
        got = torch.softmax(orc.q_posterior_logits(x0_logits, xt.view(1, -1), torch.tensor([t]), torch.tensor([s])),
                            -1)[0].numpy()
        checked = 0
        for i, (a, b) in enumerate(zip(x0.tolist(), xt.tolist())):
            if Qbar[t][a, b] == 0.0:                   # x_t unreachable from x0: no posterior
                continue
            # one-step posteriors R_u[x_u, x_{u-1}] ∝ Q_u[x_{u-1}, x_u] Qbar_{u-1}[x0, x_{u-1}], chained t -> s
            P = np.eye(K)
            for u in range(t, s, -1):
                R = Q[u].T * Qbar[u - 1][a][None, :]
                z = R.sum(1, keepdims=True)
                P = P @ np.divide(R, z, out=np.zeros_like(R), where=z > 0)
            assert np.abs(got[i] - P[b]).max() <= 1e-12, (tr, t, s, a, b)
            checked += 1
        assert checked >= K


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_schedule_table_gives_the_jump_posterior_through_the_kernel_reads(tr):
    """The row invariant, before any GPU run: what the kernels compute from a schedule table's rows t and
    t-1 is the oracle's jump posterior (within the reverse step's 2e-3 bar on log-probabilities)."""
    from head_bounds import kernel_weights
    from jump_oracle import JumpD3PM, posterior_fp32
    from oracle.d3pm import EPS
    from vall_e.vall_e import d3pm as pd
    S, K, W = 50, 1024, 24
    orc = JumpD3PM(S, K, tr)
    g = torch.Generator().manual_seed(7)
    for sch in ([S - 1], [S - 1, S // 2, S // 2 - 7, 3]):        # jumps S-1 -> 0, S-1 -> S/2, mid -> mid-7, 3 -> 0
        tab = pd.schedule_table(S, K, tr, sch).double()
        for t, s in zip(sch, sch[1:] + [0]):
            logits = (torch.randn(1, W, K, generator=g) * 3).to(torch.float16)
            x_t = torch.randint(0, K, (1, W), generator=g, dtype=torch.int32)
            x_t[0, ::2] = K // 2                                  # masked and unmasked x_t
            ref = torch.log_softmax(posterior_fp32(logits, x_t, torch.tensor([t]), orc, torch.tensor([s])).double(), -1)
            p = torch.softmax(logits.double(), -1)[0]
            lw = torch.log_softmax(torch.log(kernel_weights(tab, torch.full((W,), t), x_t[0], p, tr, EPS)), -1)
            err = (lw - ref[0]).abs().max(-1).values
            assert float(err.max()) <= 2e-3, (tr, t, s, err.argmax().item(), float(err.max()))


def test_sample_steps_out_of_range_raise_before_the_device_is_touched():
    """On a CPU model generate_audio would raise VB200Error (no CPU fallback) once it reaches the engine:
    a bad sample_steps is refused before that."""
    from vall_e.b200 import lib as L
    from vall_e.vall_e import Diffusion
    m = Diffusion(64, d_model=64, n_heads=1, n_layers=1, n_steps=6)
    text, proms = [torch.tensor([1, 2, 3])], [torch.zeros(4, 8, dtype=torch.long)]
    for bad in (0, 6, -1, 2.5, "3", True):
        with pytest.raises(ValueError, match="sample_steps"):
            m.generate_audio(text, proms, resp_lens=[5], sample_steps=bad)
    for ok in (None, 1, 5, np.int64(3)):
        with pytest.raises(L.VB200Error, match="no CPU fallback"):
            m.generate_audio(text, proms, resp_lens=[5], sample_steps=ok)


def test_step_timesteps_to_refuses_bad_arguments():
    sys.path.insert(0, str(PKG))
    import build
    build.build()
    from vall_e.b200 import lib as L
    lib = L.load()
    t = (ctypes.c_int32 * 4)()
    nxt = (ctypes.c_int32 * 8)()
    for args in ((t, 4, None, 8), (None, 4, nxt, 8), (t, 4, nxt, 0), (t, -1, nxt, 8)):
        assert lib.vb200_step_timesteps_to(*[ctypes.cast(a, ctypes.c_void_p) if isinstance(a, ctypes.Array) else a
                                            for a in args], None) != L.OK, args
        assert "step_timesteps_to" in L.last_error()


def test_cli_steps_option_reaches_generate_audio(tmp_path, monkeypatch):
    from cli_helpers import run_cli, standin_reference_emb
    from vall_e.vall_e import Diffusion
    ref = standin_reference_emb(tmp_path / "standin")
    seen = []

    class Reached(Exception):
        pass

    def fake_generate_audio(self, *args, **kwargs):
        seen.append(kwargs)
        raise Reached

    for extra, want in ((["--steps", "7"], 7), ([], None)):
        main, calls, out = run_cli(tmp_path, monkeypatch, "cpu", ref)
        import vall_e.emb.qnt as qnt
        if qnt.encode_from_file.__defaults__ == ("cuda",):
            monkeypatch.setattr(qnt.encode_from_file, "__defaults__", ("cpu",))
        monkeypatch.setattr(Diffusion, "generate_audio", fake_generate_audio)
        monkeypatch.setattr(sys, "argv", sys.argv + extra)
        with pytest.raises(Reached):
            main()
        assert seen[-1]["sample_steps"] == want and seen[-1]["seed"] == 3
