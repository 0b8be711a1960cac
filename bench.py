"""Benchmark of the D3PM denoising-sampler hot path (BASELINE.json metric: codec tokens/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c4|c5]
                    [--denoise-steps S] [--transition absorbing|uniform] [--dump-outputs DIR]

Workload (default c3 = BASELINE.json configs[2], the configuration the throughput metric is
quoted on; it fits one GPU): full denoiser (d=1024, 12 layers, 16 heads, K=1024, 8 levels), 256
utterances of 10 s (750 frames) + 3 s prompt (225 frames) + 50 phones, 50 denoise steps
(timesteps S=51, reverse loop t=50..1), absorbing transition, synthetic tokens, random-init
weights.  The 256 utterances are sharded by utterance over the N ranks (strong scaling: total
work fixed), no collective inside the loop, one all-gather of the codes at the end.

One "step" = one full pass of the hot path over one batch: all 50 denoise steps for every
utterance of the batch -> B * 750 * 8 codec tokens.  Both timed arms go through the product's own
multi-GPU entry point, ``vall_e.b200.shard.generate_sharded`` around ``Diffusion.generate_audio``:
`value` with the batch already resident in HBM, `e2e` from pinned host tensors with the gathered
codes read back to the host.  Every utterance is synthesised from its GLOBAL id, and the Philox
noise is keyed by it, so the generated codes — `codes_sha256` — do not depend on N.
One JSON line on stdout (rank 0).  ``--dump-outputs DIR`` also writes the codes of the last timed step
as ``DIR/codes.npy``, so two builds can be compared output for output; it applies to ``--impl ours``
only (the CPU reference arm times single denoise steps of one utterance, not a batch's codes).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
PKG = ROOT / "tts-with-diffusion-model_b200"
for p in (str(ROOT), str(PKG)):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

WORKLOADS = {
    #        B    T_txt T_prom T_resp timesteps transition
    "c1": (1, 30, 225, 225, 51, "uniform"),       # BASELINE configs[0]: the CPU-runnable case (quarter model)
    "c2": (1, 50, 225, 750, 51, "absorbing"),
    "c3": (256, 50, 225, 750, 51, "absorbing"),
    "c4": (16, 50, 225, 2250, 51, "absorbing"),
    "c5": (64, 50, 225, 300, 26, "uniform"),      # BASELINE configs[4], one point of its sweep: S = 25, uniform
}
MODEL = dict(n_tokens=1024, d_model=1024, n_heads=16, n_layers=12)
QUARTER = dict(n_tokens=1024, d_model=256, n_heads=4, n_layers=12)
METRIC, UNIT = "codec_tokens_per_sec", "tokens/s"


def synth_utterance(gid: int, t_txt: int, t_prom: int):
    """(text, prompt) of the utterance with GLOBAL id `gid` — independent of rank, batch and N."""
    g = torch.Generator().manual_seed(0x5EED0000 + gid)
    return (torch.randint(1, MODEL["n_tokens"], (t_txt,), generator=g),
            torch.randint(0, MODEL["n_tokens"], (t_prom, 8), generator=g))


def measured_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return d.get("bf16_tflops_sustained", 1378.2), d.get("hbm_gbs", 6450.3), "measured"
    return 1400.0, 6650.0, "fallback"   # B200_PROFILING.md fallback (sustained GEMM, copy)


def kernel_source_digest(*names):
    """sha256 over the named csrc files: ties a committed ncu capture to the kernel sources it was taken from."""
    h = hashlib.sha256()
    for n in names:
        h.update((PKG / "csrc" / n).read_bytes())
    return h.hexdigest()[:16]


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------- reference arm (CPU)
class CpuReference:
    """One utterance of a workload's shape on the host cores.  kind "reference": the reference's own modules
    staged in oracle/_ref (oracle/refarm.py: its Base stack + its p_sample with dense fp16 tables, its call
    convention, its hard-coded 1025 classes); kind "port": the oracle restatement, only where oracle/_ref is
    not staged."""

    def __init__(self, wl, quarter=False):
        from oracle import refarm
        B, t_txt, t_prom, t_resp, timesteps, transition = WORKLOADS[wl]
        torch.set_num_threads(os.cpu_count() or 1)
        self.wl, self.t_resp, self.n_den = wl, t_resp, timesteps - 1
        self.model = QUARTER if quarter else MODEL
        text, proms = synth_utterance(0, t_txt, t_prom)
        if refarm.available():
            self.kind = "reference"
            self.ref = refarm.ReferenceStep(self.model["d_model"], self.model["n_heads"], self.model["n_layers"],
                                            timesteps, transition, text, proms, t_resp)
            self.step = self.ref.step
        else:
            from oracle import denoiser as on
            from oracle.d3pm import D3PM
            self.kind = "port"
            K = self.model["n_tokens"]
            sd = on.random_state_dict(K, self.model["d_model"], self.model["n_layers"], timesteps + 1, n_resp_levels=8,
                                      n_out=8 * K, seed=0, time_rows=timesteps + 1, bf16_round=False)
            st = dict(x=torch.full((t_resp, 8), K // 2, dtype=torch.long), t=timesteps - 1)
            orc = D3PM(timesteps, K, transition)

            def step():
                lg = on.diffusion_logits(sd, [text], [proms], [st["x"]], torch.tensor([st["t"]]), self.model["n_heads"],
                                         self.model["n_layers"])[0].to(torch.float16).view(1, -1, K)
                samp, _ = orc.p_sample(lg, torch.tensor([st["t"]]), st["x"].reshape(1, -1).to(torch.int32),
                                       torch.rand(1, lg.shape[1], K))
                st["x"], st["t"] = samp.view(-1, 8), max(st["t"] - 1, 1)
            self.step = step
        self.cores = torch.get_num_threads()

    def time_steps(self, n, warmup=1):
        for _ in range(warmup):
            self.step()
        t0 = time.perf_counter()
        for _ in range(n):
            self.step()
        return (time.perf_counter() - t0) / n

    def tokens_per_s(self, step_s):
        return self.t_resp * 8 / (step_s * self.n_den)

    def sample_text(self, n, step_s):
        what = ("the reference's own modules (oracle/_ref: Base stack fp32 + p_sample with dense fp16 tables, 1025 classes)"
                if self.kind == "reference" else "oracle port of the reference (fp32 denoiser + dense fp16 p_sample)")
        size = "quarter model" if self.model is QUARTER else "full model"
        return (f"{what}; ONE utterance of the {self.wl} shape, {size}; {n} of its {self.n_den} denoise steps timed "
                f"({step_s:.3f} s each); tokens/s = {self.t_resp * 8} / ({self.n_den} x step time)")


def run_reference(args, wl):
    """`--impl reference`: each bench step = ONE denoise step of ONE utterance of the workload's shape on the host
    cores (a bounded sample: the whole batch would take hours), extrapolated to the utterance's full reverse loop;
    plus BASELINE configs[0] (C1: quarter model, 225 frames, 50 steps) run IN FULL, as BASELINE.md §5 promises."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, t_txt, t_prom, t_resp, timesteps, transition = WORKLOADS[wl]
    ref = CpuReference(wl)
    dt = ref.time_steps(args.steps, warmup=args.warmup)
    value = ref.tokens_per_s(dt)
    c1 = CpuReference("c1", quarter=True)
    t0 = time.perf_counter()
    for _ in range(c1.n_den):
        c1.step()
    c1_s = time.perf_counter() - t0
    cfg = config_dict(wl, args.gpus)
    cfg["reference_sample"] = ("ONE utterance of this shape, one denoise step per bench step (not the whole batch); "
                               "value = its tokens / (denoise steps x measured step time)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": ref.kind,
                             "sample": ref.sample_text(args.steps, dt)},
            "c1_full": {"workload": "c1: quarter model (d=256, 4 heads, 12 layers), 1 utterance x (30 phones + 225 prompt "
                                    "frames + 225 frames), 50 denoise steps, uniform — run in full",
                        "seconds": c1_s, "value": 225 * 8 / c1_s, "unit": UNIT, "kind": c1.kind, "cores": c1.cores},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, codes, resp_lens):
    """What a caller of the timed path receives for the last timed batch, ``generate_sharded(..., packed=True)``:
    the int16 codes (B, T_max, 8) in global utterance order and the frame counts, as float32 .npy (codes < 1024
    are exact in float32).  The largest workload, c3, writes 256 x 750 x 8 codes: 6 MB."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "codes.npy", codes.numpy().astype(np.float32))
    np.save(d / "resp_lens.npy", np.asarray(resp_lens, dtype=np.float32))


def config_dict(wl, n_gpus):
    B, t_txt, t_prom, t_resp, timesteps, transition = WORKLOADS[wl]
    return {"workload": f"{wl}: full D3PM denoiser d=1024 L=12 h=16 K=1024 x 8 levels, {B} utterances x "
                        f"({t_txt} phones + {t_prom} prompt frames + {t_resp} frames), {timesteps - 1} denoise steps, "
                        f"{transition}; sharded by utterance over {n_gpus} GPU(s)",
            "global_batch": B, "frames": t_resp, "denoise_steps": timesteps - 1, "transition": transition,
            "l2_policy": "per-step working set (activations > 1 GB per GPU at every N) exceeds the 126 MB L2; no flush needed",
            "operands": "16-bit tensor-core operands, fp32 accumulate: bf16 everywhere except the classifier GEMM "
                        "(fp16 rows and weights); fp32 residual stream",
            "parallelism": f"utterance-sharded x{n_gpus} (vall_e.b200.shard.generate_sharded), one final all-gather"}


# ----------------------------------------------------------------------------- our arm
def run_ours(args, wl):
    import torch.distributed as dist
    from vall_e.b200 import lib as L
    from vall_e.b200.shard import generate_sharded
    from vall_e.vall_e.diffusion import Diffusion

    B, t_txt, t_prom, t_resp, timesteps, transition = WORKLOADS[wl]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.load()

    torch.manual_seed(0)
    model = Diffusion(**MODEL, n_steps=timesteps, transition=transition)
    for blk in model.blocks:                      # AdaLN tables are zero-initialised; exercise the path
        for sub in (blk.attn, blk.ffn):
            torch.nn.init.normal_(sub.norm.emb.weight, std=0.02)
    model = model.to(dev)
    eng = model.engine()
    resp_lens = [t_resp] * B
    n_total = args.warmup + args.steps

    # Every rank holds the full (tiny) token lists of every step, built from GLOBAL utterance ids, in pinned
    # memory; generate_sharded picks this rank's shard.  gid of utterance i of step s = s * B + i.
    host, devb = [], []
    for s in range(n_total):
        utts = [synth_utterance(s * B + i, t_txt, t_prom) for i in range(B)]
        host.append(([u[0].pin_memory() for u in utts], [u[1].pin_memory() for u in utts]))

    def gen_fn(step):
        def fn(text_sub, proms_sub, lens_sub, mine):
            return model.generate_audio(text_sub, proms_sub, resp_lens=lens_sub, seed=args.seed,
                                        gids=[step * B + i for i in mine])
        return fn

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def reduce_ranks(ms, op):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def all_ranks(ms):
        if world == 1:
            return [ms]
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        out = torch.empty(world, device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(out, t)
        return [float(v) for v in out.tolist()]

    def timed_arm(batches, to_host):
        """W warm-up + K timed passes of generate_sharded; returns (mean step ms on this rank, mean local
        (pre-gather) ms on this rank, packed codes of the last step on the host, wall seconds)."""
        for i in range(args.warmup):
            generate_sharded(gen_fn(i), batches[i][0], batches[i][1], resp_lens, device=dev, packed=True)
        sync_all()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        tim = [dict() for _ in range(args.steps)]
        last = None
        t0 = time.perf_counter()
        for k in range(args.steps):
            i = args.warmup + k
            if to_host:
                sync_all()                       # e2e: every step starts from idle, like a fresh request
            ev[k][0].record()
            packed, _ = generate_sharded(gen_fn(i), batches[i][0], batches[i][1], resp_lens, device=dev, packed=True,
                                         timing=tim[k])
            if to_host:
                last = packed.to("cpu", non_blocking=False)      # the step's result, read back by the caller
            else:
                last = packed
            ev[k][1].record()
        sync_all()
        wall = time.perf_counter() - t0
        step_ms = [a.elapsed_time(b) for a, b in ev]
        local_ms = [t["local_start"].elapsed_time(t["local_end"]) for t in tim]
        return sum(step_ms) / len(step_ms), sum(local_ms) / len(local_ms), last.cpu(), wall

    # ---------------- device-resident arm: the batches are already in HBM when the clock starts
    for s in range(n_total):
        devb.append(([t.to(dev) for t in host[s][0]], [p.to(dev) for p in host[s][1]]))
    sync_all()
    launches0 = eng.launches
    with ClockSampler(local) as clocks:
        ms_rank, local_rank, codes_dev_arm, t_wall = timed_arm(devb, to_host=False)
    launches = eng.launches - launches0
    ms = reduce_ranks(ms_rank, dist.ReduceOp.MAX if world > 1 else None)
    rank_local_ms = all_ranks(local_rank)
    rank_step_ms = all_ranks(ms_rank)
    tokens_per_step = B * t_resp * 8
    value = tokens_per_step / (ms / 1e3)
    del devb

    # ---------------- end-to-end arm: pinned host inputs -> gathered codes on the host, every step
    e2e_rank, _, codes_host, _ = timed_arm(host, to_host=True)
    e2e = reduce_ranks(e2e_rank, dist.ReduceOp.MAX if world > 1 else None)
    h2d = int(model.last_h2d_bytes)
    d2h = int(codes_host.numel() * 2)                  # int16 codes of ALL utterances, read back on every rank
    sha = hashlib.sha256(codes_host.contiguous().numpy().tobytes()).hexdigest()
    same_codes = bool(torch.equal(codes_host, codes_dev_arm))       # the two arms generate the same batch

    # ---------------- roofline of the dominant kernel (tcgen05 GEMM), measured live: one eager
    # pass over this rank's shard of the last batch with CUDA events around every GEMM / attention launch
    ses = next(iter(eng._sessions.values()))
    table = model._table(dev)
    tr = L.ABSORBING if transition == "absorbing" else L.UNIFORM
    eng.profile = []
    ses.x_t.fill_(model.mask_id)
    prof_steps = 2
    ses.t_utt.fill_(timesteps - 1)
    K_cls = eng.w.n_out // 8
    for _ in range(prof_steps):
        head_in = eng.forward(ses.lay, ses.ws, ses.x_t, ses.t_utt, use_time=True, head=False)
        ev = eng._prof_begin()
        L.head_posterior_sample(ses.x_t, ses.ws.logits, head_in, eng.w.w_cls, eng.w.b_cls, ses.x_t,
                                ses.lay.resp_row_utt, ses.t_utt, ses.lay.utt, table, 8, K_cls, tr, L.NOISE_PHILOX,
                                None, args.seed)
        eng._prof_end(ev, "head_sample", 2 * ses.lay.M_resp * eng.w.n_out * eng.w.d)
    torch.cuda.synchronize(dev)
    prof, eng.profile = eng.profile, None
    agg = {}
    for kind, flops, s, e in prof:
        a = agg.setdefault(kind, [0.0, 0.0, 0])
        a[0] += flops
        a[1] += s.elapsed_time(e)
        a[2] += 1
    peak_tf, peak_hbm, peak_src = measured_peaks()
    g = list(agg.get("gemm", [0.0, 1.0, 1]))
    hsamp = agg.get("head_sample")
    if hsamp:                 # the classifier GEMM (with the reverse step as its epilogue) is a tcgen05 GEMM too
        g = [g[0] + hsamp[0], g[1] + hsamp[1], g[2] + hsamp[2]]
    at = agg.get("attn", [0.0, 1.0, 1])
    gemm_tf = g[0] / (g[1] * 1e-3) / 1e12
    attn_tf = at[0] / (at[1] * 1e-3) / 1e12
    step_total_ms = local_rank / (timesteps - 1)
    # dram bytes per launch of the largest GEMM (FFN1) from the committed `ncu --set full` capture — reported
    # only while the kernel sources are the ones the capture was taken from
    traffic, traffic_note = None, "no ncu capture committed for the current GEMM sources"
    tf = ROOT / "profiles" / "gemm_traffic.json"
    if tf.exists():
        tj = json.loads(tf.read_text())
        if tj.get("kernel_source_digest") == kernel_source_digest("gemm_tcgen05.cu", "common.cuh"):
            traffic = tj.get("bytes_per_launch")
            traffic_note = (f"dram bytes of one FFN1 launch (largest GEMM) from {tj.get('capture')}; algorithmic "
                            f"{tj.get('algorithmic_bytes')}; capture and build share kernel_source_digest "
                            f"{tj.get('kernel_source_digest')}")
        else:
            traffic_note = "profiles/gemm_traffic.json was captured from other GEMM sources (digest mismatch): not reported"
    roofline = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (QKV/out/FFN1/FFN2) + head_sample_kernel (classifier)",
                "achieved": gemm_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tf / peak_tf,
                "peak_source": f"{peak_src} bf16_tflops_sustained",
                "peak_note": "cuBLAS bf16 back to back for 4 s at the pool's power cap; the launches here are timed one by "
                             "one inside an eager pass of the step, so a lightly loaded box can exceed it (burst figure 1632)",
                "traffic": traffic, "traffic_note": traffic_note,
                "avg_launch_ms": g[1] / g[2], "launches_timed": g[2],
                "share_of_denoise_step": (g[1] / prof_steps) / step_total_ms,
                "attention": {"kernel": "flash_attn_kernel", "achieved": attn_tf, "unit": "TFLOP/s",
                              "frac": attn_tf / peak_tf, "avg_launch_ms": at[1] / at[2],
                              "share_of_denoise_step": (at[1] / prof_steps) / step_total_ms}}
    if hsamp:
        roofline["head_sample"] = {"kernel": "head_sample_kernel (classifier GEMM + D3PM reverse step, one launch)",
                                   "bound": "tensor", "achieved": hsamp[0] / (hsamp[1] * 1e-3) / 1e12,
                                   "unit": "TFLOP/s", "frac": hsamp[0] / (hsamp[1] * 1e-3) / 1e12 / peak_tf,
                                   "avg_launch_ms": hsamp[1] / hsamp[2],
                                   "share_of_denoise_step": (hsamp[1] / prof_steps) / step_total_ms}
    for kind, name in (("norm", "adaln_rows_kernel"),):
        if kind in agg:
            byt, t_ms, n = agg[kind]
            gbs = byt / (t_ms * 1e-3) / 1e9
            roofline[kind] = {"kernel": name, "bound": "hbm", "achieved": gbs, "peak": peak_hbm, "unit": "GB/s",
                              "frac": gbs / peak_hbm, "avg_launch_ms": t_ms / n,
                              "share_of_denoise_step": (t_ms / prof_steps) / step_total_ms}

    # ---------------- p50 denoise-step latency (BASELINE.json's second metric): C2 shape, batch 1,
    # one CUDA-graph replay = denoiser forward + posterior + sample, >= 20 warm iterations
    latency = None
    if rank == 0:
        b1, tt1, tp1, tr1, _, _ = WORKLOADS["c2"]
        text1, proms1 = synth_utterance(7, tt1, tp1)
        ses1 = model._session([text1.to(dev)], [proms1.to(dev)], [tr1], [0])
        ses1.x_t.fill_(model.mask_id)
        ses1.run(table, timesteps, tr, noise=L.NOISE_PHILOX, seed=args.seed, use_graph=True)   # captures the step graph
        lat = []
        for _ in range(60):
            ses1.t_utt.fill_(timesteps // 2)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ses1.graph.replay()
            b.record()
            torch.cuda.synchronize(dev)
            lat.append(a.elapsed_time(b))
        lat = sorted(lat[20:])
        T1 = tt1 + tp1 + tr1 + 2
        d_, nl_ = MODEL["d_model"], MODEL["n_layers"]
        flops1 = nl_ * (24 * T1 * d_ * d_ + 4 * T1 * T1 * d_) + 2 * tr1 * d_ * 8 * MODEL["n_tokens"]
        p50 = lat[len(lat) // 2]
        latency = {"p50_denoise_step_ms": p50, "p90_denoise_step_ms": lat[int(len(lat) * 0.9)],
                   "workload": f"c2: batch 1, T={T1} rows ({tr1} frames x 8 levels), one graph replay per step",
                   "tokens_per_sec_batch1": tr1 * 8 / (p50 * 1e-3 * (timesteps - 1)),
                   "roofline": {"bound": "tensor", "flop_per_step": flops1, "achieved": flops1 / (p50 * 1e-3) / 1e12,
                                "peak": measured_peaks()[0], "unit": "TFLOP/s",
                                "frac": flops1 / (p50 * 1e-3) / 1e12 / measured_peaks()[0],
                                "note": "single utterance: every kernel of the step is one partial wave; the floor is "
                                        "~0.27 ms of MMAs + 52 us of weight reads"}}

    # ---------------- CPU baseline beside it (rank 0, N=1 only): bounded sample on the host cores
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(wl)
        n = 2
        dt = ref.time_steps(n, warmup=1)
        cpu_baseline = {"value": ref.tokens_per_s(dt), "unit": UNIT, "cores": ref.cores, "kind": ref.kind,
                        "sample": ref.sample_text(n, dt)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config_dict(wl, world),
                "denoise_step_ms": step_total_ms, "wall_s_timed_region": t_wall,
                "clocks": clocks.summary(),
                "e2e": {"value": tokens_per_step / (e2e / 1e3), "unit": UNIT, "ms_per_step": e2e,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "codes_sha256": sha, "codes_note": "sha256 of the int16 codes of the LAST timed batch, all utterances in "
                                                   "global order; utterances and Philox noise are keyed by global id, so it "
                                                   "must be identical at N = 1, 2, 4, 8 for equal --steps/--warmup/--seed",
                "codes_equal_between_arms": same_codes,
                "per_rank": {"step_ms": rank_step_ms, "local_ms": rank_local_ms,
                             "local_ms_min": min(rank_local_ms), "local_ms_max": max(rank_local_ms),
                             "note": "step = generate_sharded incl. the all-gather; local = this rank's reverse loop only"},
                "gpu_launches": launches, "roofline": roofline, "latency": latency, "cpu_baseline": cpu_baseline}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, codes_dev_arm, resp_lens)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--denoise-steps", type=int, default=None,
                    help="override the workload's number of denoise steps (BASELINE configs[4] sweeps 10/25/50/100)")
    ap.add_argument("--transition", default=None, choices=["absorbing", "uniform"],
                    help="override the workload's transition (BASELINE configs[4] sweeps both)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the codes the last timed step generated to DIR/codes.npy (float32), with the frame "
                         "counts in DIR/resp_lens.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.denoise_steps is not None or args.transition is not None:
        B, t_txt, t_prom, t_resp, timesteps, transition = WORKLOADS[args.workload]
        WORKLOADS[args.workload] = (B, t_txt, t_prom, t_resp,
                                    timesteps if args.denoise_steps is None else args.denoise_steps + 1,
                                    transition if args.transition is None else args.transition)
    if args.impl == "reference":
        run_reference(args, args.workload)
    else:
        run_ours(args, args.workload)


if __name__ == "__main__":
    main()
