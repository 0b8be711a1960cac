"""CPU tests of sampling temperature: ``generate_audio(temperature=...)``, ``p_sample``, ``q_posterior_logits`` and the
seeded NAR level loop (``NAR.forward(seed=...)``) refuse a temperature that is not a finite number > 0 before any
CUDA call; the C entry points refuse it too (and supplied uniforms for the categorical draw) without touching a
device; ``--temperature`` and ``--nar-temperature`` of ``python -m vall_e`` reach the model calls."""
import math
import sys

import pytest
import torch

BAD = (0, 0.0, -1, -0.5, math.nan, math.inf, -math.inf, True, False, "1.0", None)


def _diffusion():
    from vall_e.vall_e import Diffusion
    torch.manual_seed(0)
    return Diffusion(64, d_model=64, n_heads=1, n_layers=1, n_steps=6)


def _batch():
    return [torch.tensor([1, 2, 3]), torch.tensor([4, 5])], [torch.zeros(4, 8, dtype=torch.long)] * 2


def test_generate_audio_refuses_a_bad_temperature_before_the_device_is_touched():
    """On a CPU model generate_audio raises VB200Error (no CPU fallback) once it reaches the engine: every bad
    temperature is refused with ValueError before that, alone and next to the other sampling options."""
    from vall_e.b200 import lib as L
    m = _diffusion()
    text, proms = _batch()
    for tau in BAD:
        with pytest.raises(ValueError, match="temperature"):
            m.generate_audio(text, proms, temperature=tau)
        with pytest.raises(ValueError, match="temperature"):
            m.generate_audio(text, proms, temperature=tau, sample_steps=2, greedy=True)
    for tau in (1.0, 1, 0.7, 2.5, 1e-3):
        with pytest.raises(L.VB200Error, match="no CPU fallback"):
            m.generate_audio(text, proms, resp_lens=[5, 3], temperature=tau)


def test_p_sample_and_q_posterior_logits_refuse_a_bad_temperature():
    m = _diffusion()
    logits = torch.randn(2, 3, 64)
    x = torch.full((2, 3), 32)
    t = torch.tensor([3, 1])
    for tau in BAD:
        for kw in (dict(seed=1), dict(greedy=True), dict(noise=torch.rand(2, 3, 64))):
            with pytest.raises(ValueError, match="temperature"):
                m.p_sample(logits, t, x, temperature=tau, **kw)
        with pytest.raises(ValueError, match="temperature"):
            m.q_posterior_logits(logits, x, t, temperature=tau)
    # the ids form reads no logits: a temperature there is refused rather than ignored
    with pytest.raises(ValueError, match="logits form"):
        m.q_posterior_logits(torch.randint(0, 64, (2, 3)), x, t, x_start_logits=False, temperature=0.5)
    with pytest.raises(Exception) as e:                                # a good one gets as far as the device
        m.p_sample(logits, t, x, seed=1, temperature=0.5)
    assert "temperature" not in str(e.value)


def test_ar_discrete_generate_audio_refuses_a_bad_temperature():
    from vall_e.vall_e.ar_discrete import AR
    m = AR()
    for tau in BAD:
        with pytest.raises(ValueError, match="temperature"):
            m.generate_audio([torch.tensor([1, 2])], [torch.zeros(3, 8, dtype=torch.long)], seed=0, temperature=tau)


def test_seeded_nar_refuses_a_bad_temperature_before_the_device_is_touched():
    from vall_e.b200 import lib as L
    from vall_e.vall_e import NAR
    torch.manual_seed(0)
    m = NAR(64, d_model=64, n_heads=1, n_layers=1)
    text, proms = _batch()
    resps = [torch.randint(0, 64, (5, 1)), torch.randint(0, 64, (3, 1))]
    for tau in BAD:
        with pytest.raises(ValueError, match="temperature"):
            m(text, proms, resps, sampling_temperature=tau, seed=3)
    with pytest.raises(L.VB200Error, match="no CPU fallback"):
        m(text, proms, resps, sampling_temperature=0.2, seed=3)


def test_c_entry_points_refuse_a_bad_temperature_without_a_device():
    """Argument checks run before any CUDA call: null pointers never get dereferenced here."""
    from vall_e.b200 import lib as L
    lib = L.load()
    for tau in (0.0, -1.0, math.nan, math.inf, -math.inf):
        assert lib.vb200_posterior_sample_from_logits_temp(
            None, None, None, L.F16, 64, None, None, None, None, None, 1, 1, 64, 6, L.ABSORBING, L.NOISE_PHILOX,
            None, 0, None, tau, None) == -1
        assert lib.vb200_head_posterior_sample_temp(
            None, None, L.F16, None, L.F16, None, None, 1, 64, 1, 256, None, None, None, None, None, 6, L.ABSORBING,
            L.NOISE_PHILOX, None, 0, None, tau, None) == -1
        assert lib.vb200_head_categorical_sample(None, 8, 1, None, L.F16, None, L.F16, None, None, 1, 64, 1024, None,
                                                 None, tau, L.NOISE_PHILOX, 0, None) == -1
        assert "temperature" in L.last_error()
    # supplied uniforms: there is no reference noise convention for the NAR's Categorical draw
    assert lib.vb200_head_categorical_sample(None, 8, 1, None, L.F16, None, L.F16, None, None, 1, 64, 1024, None,
                                             None, 1.0, L.NOISE_UNIFORMS, 0, None) == -3
    # the column must lie inside the row
    assert lib.vb200_head_categorical_sample(None, 8, 8, None, L.F16, None, L.F16, None, None, 1, 64, 1024, None,
                                             None, 1.0, L.NOISE_PHILOX, 0, None) == -1


def test_cli_temperature_reaches_generate_audio(tmp_path, monkeypatch):
    from cli_helpers import run_cli, standin_reference_emb
    from vall_e.vall_e import Diffusion
    ref = standin_reference_emb(tmp_path / "standin")
    seen = []

    class Reached(Exception):
        pass

    def fake_generate_audio(self, *args, **kwargs):
        seen.append(kwargs)
        raise Reached

    main, calls, out = run_cli(tmp_path, monkeypatch, "cpu", ref)
    monkeypatch.setattr(Diffusion, "generate_audio", fake_generate_audio)
    argv = list(sys.argv)
    with pytest.raises(Reached):
        main()
    assert seen[-1]["temperature"] == 1.0 and seen[-1]["seed"] == 3
    monkeypatch.setattr(sys, "argv", argv + ["--temperature", "0.7"])
    with pytest.raises(Reached):
        main()
    assert seen[-1]["temperature"] == 0.7


def test_cli_ar_discrete_and_nar_get_their_temperatures_and_the_seed(tmp_path, monkeypatch):
    """First stage = the reference's D3PM class: --temperature goes to it, --nar-temperature (default 0.2, reference
    nar.py:33) and --seed go to the NAR stage."""
    from cli_helpers import run_cli, standin_reference_emb
    from vall_e.vall_e import NAR
    from vall_e.vall_e.ar_discrete import AR
    ref = standin_reference_emb(tmp_path / "standin")
    main, calls, out = run_cli(tmp_path, monkeypatch, "cpu", ref)
    ar = AR()
    ar.phone_symmap = {ch: i + 1 for i, ch in enumerate("ABCDEFGHIJKLMNOPQRSTUVWXYZ_")}
    torch.save(ar, tmp_path / "ar.pt")
    torch.save(NAR(64, d_model=64, n_heads=1, n_layers=1), tmp_path / "nar.pt")
    seen = {}

    class Reached(Exception):
        pass

    def fake_ar(self, text_list, proms_list, **kwargs):
        seen["ar"] = kwargs
        return torch.zeros(448, dtype=torch.long)

    def fake_nar(self, text_list, proms_list, resps_list, **kwargs):
        seen["nar"] = kwargs
        raise Reached

    monkeypatch.setattr(AR, "generate_audio", fake_ar)
    monkeypatch.setattr(NAR, "forward", fake_nar)
    argv = [a for a in sys.argv]
    argv[argv.index("--ar-ckpt") + 1] = str(tmp_path / "ar.pt")
    monkeypatch.setattr(sys, "argv", argv + ["--nar-ckpt", str(tmp_path / "nar.pt")])
    with pytest.raises(Reached):
        main()
    assert seen["ar"] == dict(seed=3, temperature=1.0)
    assert seen["nar"] == dict(sampling_temperature=0.2, seed=3)
    monkeypatch.setattr(sys, "argv", argv + ["--nar-ckpt", str(tmp_path / "nar.pt"), "--temperature", "0.5",
                                             "--nar-temperature", "0.9"])
    with pytest.raises(Reached):
        main()
    assert seen["ar"] == dict(seed=3, temperature=0.5)
    assert seen["nar"] == dict(sampling_temperature=0.9, seed=3)
