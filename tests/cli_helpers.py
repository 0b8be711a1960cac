"""Shared by the CPU and GPU tests of the ``python -m vall_e`` entry point (reference __main__.py:44-73)."""
import sys
from pathlib import Path

import torch


def stub_audio_modules(monkeypatch, calls):
    """Stand-ins for the third-party packages the reference's emb/qnt.py and emb/g2p.py import (not installed
    in this image): an 'EnCodec' that returns fixed codes / silence and a 'G2p' that spells letters."""
    import types

    class FakeEncodec:
        sample_rate, channels = 24_000, 1

        @classmethod
        def encodec_model_24khz(cls):
            return cls()

        def set_target_bandwidth(self, bw):
            calls.append(("bandwidth", bw))

        def to(self, device):
            return self

        def encode(self, wav):
            calls.append(("encode", tuple(wav.shape)))
            g = torch.Generator().manual_seed(0)
            return [(torch.randint(0, 64, (1, 8, 12), generator=g), None)]

        def decode(self, frames):
            codes = frames[0][0]
            calls.append(("decode", tuple(codes.shape)))
            return torch.zeros(codes.shape[0], 1, codes.shape[-1] * 320)

    enc = types.ModuleType("encodec")
    enc.EncodecModel = FakeEncodec
    enc_utils = types.ModuleType("encodec.utils")
    enc_utils.convert_audio = lambda wav, sr, target_sr, target_channels: wav
    ta = types.ModuleType("torchaudio")
    ta.load = lambda path: (torch.zeros(2, 2400), 24_000)
    sf = types.ModuleType("soundfile")

    def write(path, data, sr):
        calls.append(("write", str(path), tuple(data.shape), sr))
        Path(path).write_bytes(b"RIFF")
    sf.write = write
    g2p_en = types.ModuleType("g2p_en")
    g2p_en.G2p = lambda: (lambda text: [ch.upper() if ch.isalpha() else ch for ch in text])
    for name, mod in (("encodec", enc), ("encodec.utils", enc_utils), ("torchaudio", ta), ("soundfile", sf),
                      ("g2p_en", g2p_en)):
        monkeypatch.setitem(sys.modules, name, mod)


def standin_reference_emb(root: Path):
    """A stand-in checkout of the reference: the two functions of emb/qnt.py and the one of
    emb/g2p.py that ``python -m vall_e`` calls (__main__.py:56-58,72), over the same third-party APIs."""
    emb = root / "vall_e" / "emb"
    emb.mkdir(parents=True)
    (emb / "qnt.py").write_text(
        "import soundfile, torch, torchaudio\nfrom encodec import EncodecModel\nfrom ..config import cfg\n"
        "def _m():\n    m = EncodecModel.encodec_model_24khz(); m.set_target_bandwidth(6.0); return m\n"
        "def encode_from_file(path, device='cuda'):\n    wav, sr = torchaudio.load(str(path))\n"
        "    assert cfg.sample_rate == 24_000\n    return torch.cat([e[0] for e in _m().encode(wav[:1].unsqueeze(0))], dim=-1)\n"
        "def decode_to_file(resps, path):\n    assert resps.dim() == 2\n"
        "    wavs = _m().decode([(resps.t().unsqueeze(0), None)])\n    soundfile.write(str(path), wavs.cpu()[0, 0], 24_000)\n")
    (emb / "g2p.py").write_text(
        "import string\nfrom g2p_en import G2p\n"
        "def encode(graphs):\n    ignored = {' ', *string.punctuation}\n"
        "    return ['_' if p in ignored else p for p in G2p()(graphs)]\n")
    return root


def run_cli(tmp_path, monkeypatch, device, ref_root):
    """python -m vall_e <text> <ref.wav> <out.wav> --ar-ckpt <pickled tiny Diffusion> in-process."""
    import importlib
    calls = []
    stub_audio_modules(monkeypatch, calls)
    monkeypatch.setenv("VALL_E_REF", str(ref_root))
    for name in [n for n in sys.modules if n == "vall_e.emb" or n.startswith("vall_e.emb.")]:
        monkeypatch.delitem(sys.modules, name)
    from vall_e.vall_e import Diffusion
    torch.manual_seed(0)
    m = Diffusion(64, d_model=64, n_heads=1, n_layers=1, n_steps=5)
    m.phone_symmap = {ch: i + 1 for i, ch in enumerate("ABCDEFGHIJKLMNOPQRSTUVWXYZ_")}
    ckpt = tmp_path / "diffusion.pt"
    torch.save(m, ckpt)
    out = tmp_path / "out.wav"
    monkeypatch.setattr(sys, "argv", ["vall_e", "hello, world", str(tmp_path / "ref.wav"), str(out), "--ar-ckpt", str(ckpt),
                                      "--device", device, "--frames", "20", "--seed", "3"])
    main = importlib.import_module("vall_e.__main__").main
    return main, calls, out
