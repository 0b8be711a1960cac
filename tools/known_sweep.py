"""Cost of generating around given codes (generate_audio(known_list=...)) at the c3 shape: 256 utterances x (50 phones
+ 225 prompt frames + 750 frames), the full model, S = 51 timesteps (50 denoise steps), absorbing, one GPU, under four
conditions: no known_list, known_list all -1, the first 225 frames known (continuation) and level 0 known
(level-conditional).

Every condition is warmed up first (its first call captures the step graph).  Two passes run the conditions in
opposite order; each point is the best of --reps calls, each ending in a device synchronise.  One JSON line per point
and pass, with the GPU's name, power limit and SM clock read right after it (nvidia-smi --query-gpu, read-only), and
a last line saying whether known_list all -1 gave the codes of the call without it and whether the given codes
came back.
    python tools/known_sweep.py [--reps 2] [--out FILE]"""
import argparse
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
from sample_steps_sweep import MODEL, WORKLOADS, Diffusion, L, digest, gpu_state, synth_utterance  # noqa: E402


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
    g = torch.Generator().manual_seed(3)
    codes = [torch.randint(0, model.num_classes, (t_resp, 8), generator=g, dtype=torch.int32) for _ in range(B)]
    prefix = 225

    def masked(sel):
        out = []
        for c in codes:
            k = torch.full_like(c, -1)
            k[sel] = c[sel]
            out.append(k.to(dev))
        return out

    conditions = {
        "none": None,
        "all_minus_1": [torch.full((t_resp, 8), -1, dtype=torch.int32, device=dev) for _ in range(B)],
        "continuation_225": masked((slice(0, prefix),)),
        "level0": masked((slice(None), 0)),
    }
    lines = []

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        lines.append(line)

    def call(kl, seed=1):
        return model.generate_audio(text, proms, resp_lens=lens, seed=seed, known_list=kl)

    for kl in conditions.values():           # warm-up: graph capture of every condition
        call(kl)
    torch.cuda.synchronize()
    names = list(conditions)
    for p, order in enumerate((names, names[::-1])):
        for name in order:
            times = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                call(conditions[name])
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t0)
            s = min(times)
            emit({"pass": p, "condition": name, "tokens_per_s": tokens / s, "ms_per_call": s * 1e3,
                  "ms_per_denoise_step": s * 1e3 / (S - 1), "calls_ms": [round(x * 1e3, 2) for x in times],
                  "workload": f"c3: {B} x ({t_txt} phones, {t_prom} prompt frames, {t_resp} frames), S={S}, {tr}",
                  **gpu_state()})
    a, b = call(None, seed=7), call(conditions["all_minus_1"], seed=7)
    same = all(torch.equal(x, y) for x, y in zip(a, b))
    back = True
    for name in ("continuation_225", "level0"):
        out = call(conditions[name], seed=7)
        back &= all(torch.equal(o[k >= 0], k[k >= 0].long()) for o, k in zip(out, conditions[name]))
    emit({"check": "known_list all -1 equals no known_list (seed 7); given codes come back", "equal": same,
          "given_codes_back": bool(back), "codes_sha256": digest(a), "codes_sha256_all_minus_1": digest(b)})
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text("\n".join(lines) + "\n")
    if not (same and back):
        raise SystemExit("known_list check failed")


if __name__ == "__main__":
    main()
