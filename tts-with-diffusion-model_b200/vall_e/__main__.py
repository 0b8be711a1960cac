"""``python -m vall_e <text> <reference.wav> <out.wav>`` — the reference's inference entry point
(``vall_e/__main__.py:44-73``) with the non-autoregressive codec-token stage on the B200 kernels.

Stages, as in the reference: EnCodec-encode the prompt (reference ``emb/qnt.py``), phonemise the
text (``emb/g2p.py``), first-stage model -> codes, NAR / decode, write audio.  EnCodec and g2p stay
on the reference implementation (out of scope and excluded from timing, BASELINE.json): ``vall_e.emb``
executes the reference's own ``emb/qnt.py`` and ``emb/g2p.py`` from a checkout named by ``VALL_E_REF``
(see ``vall_e/emb/__init__.py``; they need encodec, torchaudio, soundfile and g2p_en installed).  The
model checkpoints are whole-module pickles (reference ``export.py``) resolved through this package's
``vall_e.vall_e.{ar,nar,diffusion}`` classes.

  --ar-ckpt may hold a ``Diffusion`` model (8 levels in one reverse loop; NAR is then skipped), the
  reference's own level-0 D3PM class (``vall_e.vall_e.ar_discrete.AR``: 350 frames by diffusion, then
  the NAR pass), or a reference causal AR model (unsupported here: raises).
"""
import argparse
from pathlib import Path

import torch
from einops import rearrange

from .utils import to_device
from .vall_e.ar_discrete import AR as DiscreteAR
from .vall_e.diffusion import Diffusion


def _load(path, device):
    # torch >= 2.6 defaults to weights_only=True, which rejects module pickles (SURVEY.md §5)
    return torch.load(path, weights_only=False).to(device)


def decode_batch_to_files(qnt, codes_bqt, frames, paths, hop: int = 320):
    """EnCodec hand-off for a batch (SURVEY §8f.4): ONE ``qnt.decode`` call (reference emb/qnt.py:32-41,
    which already takes ``(b q t)``) on the ``(B, 8, T_max)`` tensor ``Diffusion.generate_audio(...,
    as_bqt=True)`` returns, instead of the reference's one-utterance-at-a-time ``decode_to_file``
    (:44-48); each waveform is cut at its own length (``hop`` samples per frame: 24 kHz / 75 frames/s)."""
    import soundfile
    wavs, sr = qnt.decode(codes_bqt)
    for wav, n, path in zip(wavs.cpu(), frames, paths):
        soundfile.write(str(path), wav[0, : n * hop], sr)


def main():
    parser = argparse.ArgumentParser("VALL-E TTS")
    parser.add_argument("text")
    parser.add_argument("reference", type=Path)
    parser.add_argument("out_path", type=Path)
    parser.add_argument("--ar-ckpt", type=Path, default="zoo/ar.pt")
    parser.add_argument("--nar-ckpt", type=Path, default="zoo/nar.pt")
    parser.add_argument("--device", default="cuda")
    parser.add_argument("--frames", type=int, default=None, help="frames to generate (diffusion first stage)")
    parser.add_argument("--seed", type=int, default=0)
    parser.add_argument("--steps", type=int, default=None,
                        help="denoise steps of a diffusion first stage, 1 .. n_steps-1 (default: every timestep)")
    parser.add_argument("--continue-from", type=Path, default=None, metavar="PART.wav",
                        help="diffusion first stage: keep PART.wav's EnCodec frames as the start of the response and "
                             "generate the rest, up to --frames frames in all")
    args = parser.parse_args()

    try:
        from .emb import g2p, qnt  # reference front/back ends (EnCodec 24 kHz @ 6 kbps, g2p_en)
    except ImportError as e:  # pragma: no cover - depends on optional third-party packages
        raise SystemExit(f"python -m vall_e: audio I/O unavailable — {e}")

    first = _load(args.ar_ckpt, args.device)
    symmap = first.phone_symmap
    proms = rearrange(qnt.encode_from_file(args.reference), "1 l t -> t l")
    phns = torch.tensor([symmap[p] for p in g2p.encode(args.text)])
    proms = to_device(proms, args.device)
    phns = to_device(phns, args.device)

    known_list = None
    if args.continue_from is not None:
        if not isinstance(first, Diffusion):
            raise SystemExit("python -m vall_e: --continue-from needs a diffusion first stage (a Diffusion checkpoint)")
        prefix = rearrange(qnt.encode_from_file(args.continue_from), "1 l t -> t l")
        total = args.frames or 350
        if total <= prefix.shape[0]:
            raise SystemExit(f"python -m vall_e: --frames ({total}) must exceed the {prefix.shape[0]} frames of "
                             f"{args.continue_from}")
        known = torch.full((total, prefix.shape[1]), -1, dtype=torch.long)
        known[: prefix.shape[0]] = prefix.cpu()
        known_list = [to_device(known, args.device)]

    if isinstance(first, Diffusion):
        lens = [args.frames] if args.frames else None
        resps_list = first.generate_audio(text_list=[phns], proms_list=[proms], resp_lens=lens, seed=args.seed,
                                          sample_steps=args.steps, known_list=known_list)
    else:
        nar = _load(args.nar_ckpt, args.device)
        if isinstance(first, DiscreteAR):       # the reference's own D3PM class: level 0 by diffusion, 350 frames
            resp_list = [first.generate_audio([phns], [proms], seed=args.seed)[:350]]
        else:
            resp_list = first(text_list=[phns], proms_list=[proms])
        resps_list = [r.unsqueeze(-1) for r in resp_list]
        resps_list = nar(text_list=[phns], proms_list=[proms], resps_list=resps_list)
    qnt.decode_to_file(resps=resps_list[0], path=args.out_path)
    print(args.out_path, "saved.")


if __name__ == "__main__":
    main()
