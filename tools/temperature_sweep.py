"""Cost of sampling temperature.

1. generate_audio(temperature=...) at the c3 shape: 256 utterances x (50 phones + 225 prompt frames + 750 frames),
   the full model, S = 51 timesteps (50 denoise steps), absorbing, one GPU, with no temperature argument, 1.0 and 0.7.
2. The NAR level loop for one c2-shaped utterance (50 phones, 225 prompt frames, 750 frames, level 0 given, levels
   1-7 drawn) on the full-size NAR (K = 1024, one head): the reference's Categorical path (seed=None) against the
   seeded device path (one layout and workspace, draws in the classifier's epilogue).

Every point is warmed up first (the first diffusion call of a temperature captures its step graph).  Two passes
run the points in opposite order; each point is the best of --reps calls, each ending in a device synchronise.  One
JSON line per point and pass, with the GPU's name, power limit and SM clock read right after it (nvidia-smi
--query-gpu, read-only), and a last line saying whether temperature=1.0 gave the codes of the call without it.
    python tools/temperature_sweep.py [--reps 2] [--out FILE]"""
import argparse
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
from sample_steps_sweep import MODEL, WORKLOADS, Diffusion, L, digest, gpu_state, synth_utterance  # noqa: E402
from vall_e.vall_e import NAR  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    L.load()
    dev = torch.device("cuda")
    lines = []

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        lines.append(line)

    def best(fn):
        times = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        return min(times), times

    # ---- 1. diffusion, c3
    B, t_txt, t_prom, t_resp, S, tr = WORKLOADS["c3"]
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
    conditions = {"default": {}, "1.0": dict(temperature=1.0), "0.7": dict(temperature=0.7)}

    def call(kw, seed=1):
        return model.generate_audio(text, proms, resp_lens=lens, seed=seed, **kw)

    for kw in conditions.values():           # warm-up: graph capture of every temperature
        call(kw)
    torch.cuda.synchronize()
    names = list(conditions)
    for p, order in enumerate((names, names[::-1])):
        for name in order:
            s, times = best(lambda: call(conditions[name]))
            emit({"pass": p, "condition": f"temperature={name}", "tokens_per_s": tokens / s, "ms_per_call": s * 1e3,
                  "ms_per_denoise_step": s * 1e3 / (S - 1), "calls_ms": [round(x * 1e3, 2) for x in times],
                  "workload": f"c3: {B} x ({t_txt} phones, {t_prom} prompt frames, {t_resp} frames), S={S}, {tr}",
                  **gpu_state()})
    a, b, c = call({}, seed=7), call(dict(temperature=1.0), seed=7), call(dict(temperature=0.7), seed=7)
    same = all(torch.equal(x, y) for x, y in zip(a, b))
    emit({"check": "temperature=1.0 equals no temperature argument (seed 7)", "equal": same,
          "codes_sha256": digest(a), "codes_sha256_t1": digest(b), "codes_sha256_t07": digest(c)})
    del model
    torch.cuda.empty_cache()

    # ---- 2. NAR levels 1-7, one c2-shaped utterance
    _, t_txt, t_prom, t_resp, _, _ = WORKLOADS["c2"]
    torch.manual_seed(0)
    nar = NAR(MODEL["n_tokens"], d_model=MODEL["d_model"], n_heads=MODEL["n_heads"], n_layers=MODEL["n_layers"])
    for blk in nar.blocks:
        for sub in (blk.attn, blk.ffn):
            torch.nn.init.normal_(sub.norm.emb.weight, std=0.02)
    nar = nar.to(dev)
    u = synth_utterance(0, t_txt, t_prom)
    g = torch.Generator().manual_seed(5)
    level0 = torch.randint(0, MODEL["n_tokens"], (t_resp, 1), generator=g).to(dev)
    paths = {"categorical_seed_none": dict(), "device_seeded": dict(seed=3)}

    def nar_call(kw):
        return nar([u[0].to(dev)], [u[1].to(dev)], [level0], sampling_temperature=0.2, **kw)

    for kw in paths.values():
        nar_call(kw)
    torch.cuda.synchronize()
    names = list(paths)
    for p, order in enumerate((names, names[::-1])):
        for name in order:
            s, times = best(lambda: nar_call(paths[name]))
            emit({"pass": p, "nar_path": name, "ms_per_call": s * 1e3, "calls_ms": [round(x * 1e3, 2) for x in times],
                  "workload": f"NAR levels 1-7: 1 x ({t_txt} phones, {t_prom} prompt frames, {t_resp} frames), "
                              f"K={MODEL['n_tokens']}, d={MODEL['d_model']}, {MODEL['n_layers']} layers, tau=0.2",
                  **gpu_state()})
    r1, r2 = nar_call(paths["device_seeded"]), nar_call(paths["device_seeded"])
    emit({"check": "seeded NAR codes repeat", "equal": bool(torch.equal(r1[0], r2[0])), "codes_sha256": digest(r1)})
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text("\n".join(lines) + "\n")
    if not same:
        raise SystemExit("temperature=1.0 check failed")


if __name__ == "__main__":
    main()
