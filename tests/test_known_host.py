"""CPU tests of generation around given codes (``generate_audio(known_list=...)``): the O(1) law of a known token
that the reverse-step kernels draw from (posterior.cuh ``known_pick``), restated in numpy from the table fields it
reads, against the oracle's dense ids-form posterior; argument checks; ``--continue-from`` of ``python -m vall_e``."""
import sys

import numpy as np
import pytest
import torch


def closed_form_law(tab, t, x_t, k, K, tr, eps):
    """posterior.cuh known_law in float64: f1 from row t's ONE_* fields (+ eps), f2 = Qbar_s[k, j] from row t-1's
    CUM_* fields; specials {x_t, k, m} get their own weight, every other class the generic one."""
    from vall_e.b200 import lib as L
    one, cum = tab[t].astype(np.float64), tab[max(t - 1, 0)].astype(np.float64)
    m = K // 2 if tr == "absorbing" else -1
    at_m = m >= 0 and x_t == m
    f1_self = (one[L.TAB_ONE_BOTH] if at_m else one[L.TAB_ONE_KEEP]) + eps
    f1_oth = (one[L.TAB_ONE_ABSORB] if at_m else one[L.TAB_ONE_OFF]) + eps
    a_gen, c_gen = cum[L.TAB_CUM_KEEP], cum[L.TAB_CUM_OFF]
    a_m, c_m = (cum[L.TAB_CUM_BOTH], cum[L.TAB_CUM_ABSORB]) if m >= 0 else (a_gen, c_gen)

    def weight(j):
        f1 = f1_self if j == x_t else f1_oth
        f2 = (a_m if j == m else a_gen) if j == k else (c_m if j == m else c_gen)
        return f1 * (f2 + eps)

    law = np.full(K, f1_oth * (c_gen + eps))
    specials = {x_t, k} | ({m} if m >= 0 else set())
    for j in specials:
        law[j] = weight(j)
    assert len(specials) <= 3
    return law / law.sum()


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_closed_form_known_law_matches_the_oracle_ids_posterior(tr):
    """Every special case: x_t in {m, other}, k in {m, x_t, other}; one-step (plain table) and jumps (schedule
    table); float64 against the oracle's dense law.  Exact tables for absorbing, one fp16 ulp for uniform."""
    from known_oracle import KnownD3PM
    from oracle.d3pm import EPS
    from vall_e.vall_e import d3pm as pd
    S, K = 50, 1024
    m = K // 2
    orc = KnownD3PM(S, K, tr)
    cases = [(m, m), (m, 7), (5, 5), (5, m), (5, 900)]              # (x_t, k)
    plain = pd.scalar_table(S, K, tr).numpy()
    sch = [S - 1, S // 2, S // 2 - 7, 3]
    jump_tab = pd.schedule_table(S, K, tr, sch).numpy()
    steps = [(t, None, plain) for t in (1, 2, 25, S - 1)] + [(t, s, jump_tab) for t, s in zip(sch, sch[1:] + [0])]
    tol = 1e-9 if tr == "absorbing" else 2e-3
    for t, s, tab in steps:
        x_t = torch.tensor([[c[0] for c in cases]], dtype=torch.int32)
        x0 = torch.tensor([[c[1] for c in cases]], dtype=torch.int32)
        ref = torch.log_softmax(orc.log_law_ids(x0, x_t, torch.tensor([t]), None if s is None else torch.tensor([s])),
                                -1)[0].numpy()
        for i, (xt, k) in enumerate(cases):
            got = np.log(closed_form_law(tab, t, xt, k, K, tr, EPS))
            err = np.abs(got - ref[i]).max()
            assert err <= tol, (tr, t, s, xt, k, err)
            if tr == "absorbing":        # the law is concentrated where the oracle puts it
                assert np.argmax(got) == np.argmax(ref[i])


def test_oracle_ids_form_is_the_logits_form_of_a_one_hot():
    """The ids form is the logits form at x0 logits = log one_hot(k) (up to the fp16 softmax), in float64."""
    from known_oracle import KnownD3PM
    S, K = 12, 64
    for tr in ("absorbing", "uniform"):
        orc = KnownD3PM(S, K, tr)
        g = torch.Generator().manual_seed(2)
        x0 = torch.randint(0, K, (3, 5), generator=g)
        xt = torch.randint(0, K, (3, 5), generator=g)
        xt[:, 0] = K // 2
        t = torch.tensor([1, 6, 11])
        for s in (None, torch.tensor([0, 2, 4])):
            ids = orc.q_posterior_logits_ids(x0, xt, t, s).double()
            onehot = torch.full((3, 5, K), -60.0, dtype=torch.float16)
            onehot.scatter_(-1, x0[..., None], 0.0)
            lg = orc.q_posterior_logits(onehot, xt, t, s).double()
            assert (ids - lg).abs().max().item() < 1e-2, (tr, s)


def _model():
    from vall_e.vall_e import Diffusion
    return Diffusion(64, d_model=64, n_heads=1, n_layers=1, n_steps=6)


def test_bad_known_list_raises_before_the_device_is_touched():
    """On a CPU model generate_audio raises VB200Error (no CPU fallback) once it reaches the engine: every bad
    known_list is refused before that."""
    from vall_e.b200 import lib as L
    m = _model()
    text, proms = [torch.tensor([1, 2, 3]), torch.tensor([4, 5])], [torch.zeros(4, 8, dtype=torch.long)] * 2
    ok = [torch.full((5, 8), -1), torch.randint(0, 64, (3, 8))]
    bad_value = [
        dict(known_list=ok[:1]),                                           # one entry for two utterances
        dict(known_list=[torch.full((5, 7), -1), ok[1]]),                  # wrong level count
        dict(known_list=[torch.full((5,), -1), ok[1]]),                    # not 2-D
        dict(known_list=[torch.full((5, 8), -1.0), ok[1]]),                # not integer codes
        dict(known_list=ok, resp_lens=[5, 4]),                             # disagrees with resp_lens
        dict(known_list=ok, resps_list=[torch.zeros(5, 8, dtype=torch.long), torch.zeros(2, 8, dtype=torch.long)]),
    ]
    for kw in bad_value:
        with pytest.raises(ValueError):
            m.generate_audio(text, proms, **kw)
    for v in (-2, 64, 1000):
        bad = ok[1].clone()
        bad[1, 3] = v
        with pytest.raises(IndexError, match="known_list"):
            m.generate_audio(text, proms, known_list=[ok[0], bad])
    with pytest.raises(ValueError, match="sample_steps"):
        m.generate_audio(text, proms, known_list=ok, sample_steps=9)
    for kw in (dict(), dict(resp_lens=[5, 3]), dict(sample_steps=2, greedy=True),
               dict(resps_list=[torch.zeros(5, 8, dtype=torch.long), torch.zeros(3, 8, dtype=torch.long)])):
        with pytest.raises(L.VB200Error, match="no CPU fallback"):
            m.generate_audio(text, proms, known_list=ok, **kw)


def test_q_posterior_logits_ids_form_checks_the_ids():
    """x_start_logits=False is implemented (on the GPU, test_gpu_known.py); ids outside [0, K) are refused first."""
    m = _model()
    x0 = torch.randint(0, 64, (2, 3))
    for bad in (x0 + 64, x0 - 65):
        with pytest.raises(IndexError, match="x_start"):
            m.q_posterior_logits(bad, x0, torch.tensor([1, 2]), x_start_logits=False)


def test_cli_continue_from_reaches_generate_audio_with_the_encoded_prefix(tmp_path, monkeypatch):
    from cli_helpers import run_cli, standin_reference_emb
    from vall_e.vall_e import Diffusion
    ref = standin_reference_emb(tmp_path / "standin")
    seen = []

    class Reached(Exception):
        pass

    def fake_generate_audio(self, *args, **kwargs):
        seen.append(kwargs)
        raise Reached

    part = tmp_path / "part.wav"
    part.write_bytes(b"RIFF")
    main, calls, out = run_cli(tmp_path, monkeypatch, "cpu", ref)
    import vall_e.emb.qnt as qnt
    if qnt.encode_from_file.__defaults__ == ("cuda",):
        monkeypatch.setattr(qnt.encode_from_file, "__defaults__", ("cpu",))
    monkeypatch.setattr(Diffusion, "generate_audio", fake_generate_audio)
    prefix = qnt.encode_from_file(part)[0].t()                       # (12, 8): the stand-in EnCodec's frames
    argv = list(sys.argv)
    monkeypatch.setattr(sys, "argv", argv + ["--continue-from", str(part)])
    with pytest.raises(Reached):
        main()
    (known,) = seen[-1]["known_list"]
    assert tuple(known.shape) == (20, 8) and seen[-1]["resp_lens"] == [20]
    assert torch.equal(known[: prefix.shape[0]].cpu(), prefix.long())
    assert bool((known[prefix.shape[0]:] == -1).all())
    for frames in ("12", "5"):                                        # a prefix of >= --frames frames exits
        monkeypatch.setattr(sys, "argv", argv + ["--continue-from", str(part), "--frames", frames])
        with pytest.raises(SystemExit, match="must exceed"):
            main()
    # without the option nothing is known
    monkeypatch.setattr(sys, "argv", argv)
    with pytest.raises(Reached):
        main()
    assert seen[-1]["known_list"] is None
