"""Throughput of generate_audio(sample_steps=n) at the c3 shape: 256 utterances x (50 phones + 225 prompt
frames + 750 frames), the full model, S = 51 timesteps, absorbing, one GPU, n in {50, 25, 10, 5}.

Each point is warmed up (the first call of an n captures its step graph) and then timed over --reps calls,
each ending in a device synchronise; the order of the points is reversed on the second pass.  One JSON line
per point and pass, with the GPU's name, power limit and SM clock read right after it (nvidia-smi
--query-gpu, read-only), and a last line saying whether sample_steps=50 gave the codes of the default call.
    python tools/sample_steps_sweep.py [--reps 2] [--out FILE]"""
import argparse
import hashlib
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tts-with-diffusion-model_b200"))
sys.path.insert(0, str(ROOT))
from bench import MODEL, WORKLOADS, synth_utterance  # noqa: E402
from vall_e.b200 import lib as L  # noqa: E402
from vall_e.vall_e.diffusion import Diffusion  # noqa: E402


def gpu_state():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True, check=True).stdout
    name, power, sm, sm_max = [x.strip() for x in q.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}


def digest(codes):
    return hashlib.sha256(torch.cat(codes).to(torch.int32).cpu().numpy().tobytes()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    L.load()
    B, t_txt, t_prom, t_resp, S, tr = WORKLOADS["c3"]
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = Diffusion(**MODEL, n_steps=S, transition=tr)
    for blk in model.blocks:                 # AdaLN tables away from the identity, as a trained model's
        for sub in (blk.attn, blk.ffn):
            torch.nn.init.normal_(sub.norm.emb.weight, std=0.02)
    model = model.to(dev)
    utts = [synth_utterance(g, t_txt, t_prom) for g in range(B)]
    text, proms = [u[0].to(dev) for u in utts], [u[1].to(dev) for u in utts]
    lens = [t_resp] * B
    tokens = B * t_resp * model.n_levels
    lines = []

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        lines.append(line)

    points = [50, 25, 10, 5]
    for p, order in enumerate((points, points[::-1])):
        for n in order:
            model.generate_audio(text, proms, resp_lens=lens, seed=1, sample_steps=n)      # warm-up + graph capture
            torch.cuda.synchronize()
            times = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                model.generate_audio(text, proms, resp_lens=lens, seed=1, sample_steps=n)
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            s = min(times)
            emit({"pass": p, "sample_steps": n, "tokens_per_s": tokens / s, "ms_per_call": s * 1e3,
                  "ms_per_denoise_step": s * 1e3 / n, "calls_ms": [round(x * 1e3, 2) for x in times],
                  "workload": f"c3: {B} x ({t_txt} phones, {t_prom} prompt frames, {t_resp} frames), S={S}, {tr}",
                  **gpu_state()})
    a = model.generate_audio(text, proms, resp_lens=lens, seed=7)
    b = model.generate_audio(text, proms, resp_lens=lens, seed=7, sample_steps=S - 1)
    same = all(torch.equal(x, y) for x, y in zip(a, b))
    emit({"check": f"sample_steps={S - 1} equals the default call, seed 7", "equal": same,
          "codes_sha256": digest(a), "codes_sha256_sample_steps": digest(b)})
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text("\n".join(lines) + "\n")
    if not same:
        raise SystemExit("sample_steps=S-1 gave other codes than the default call")


if __name__ == "__main__":
    main()
