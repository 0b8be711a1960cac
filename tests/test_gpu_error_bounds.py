"""GEMM and attention kernels against float64 references, element by element within the bounds of
tests/error_bounds.py, on every GEMM tiling and every ragged edge.  Run on the B200 box: pytest -m gpu.

The GEMM launcher reads VB200_GEMM_TILE once per process, so each forced tiling (and the launcher's own choice)
runs in a child process of its own.  Each child checks its cases and writes their output bytes; the parent then
asserts that every case gives the same bytes on every tiling that ran it: the k-order of each output element is
the same in all of them, and an utterance's outputs must not depend on which tiling the batch size picks."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import error_bounds as eb

pytestmark = pytest.mark.gpu

DEV = "cuda"
HERE = Path(__file__).resolve().parent
TILINGS = ["pair", "wide", "narrow", "n64", "n192"]
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
EPIS = {"none": eb.EPI_NONE, "bias": eb.EPI_BIAS, "gelu": eb.EPI_BIAS_GELU, "resid": eb.EPI_BIAS_RESIDUAL}

# (M, N, K): M = 1, 127, 129; M leaving the pair's second CTA without rows (257, 4200); N tails below every tile
# (8, 72, 200, tile + 8); K < 64, K % 64 != 0 and 4096 + 8; N % 192 == 0 for the 128x192 tiling
SMALL_SHAPES = [(1, 64, 64), (1, 8, 8), (127, 72, 56), (129, 200, 200), (257, 264, 1024), (128, 136, 64),
                (300, 200, 4104), (129, 384, 200), (257, 192, 8), (513, 72, 8), (200, 8, 200), (255, 1032, 512),
                (1, 384, 1024), (4200, 192, 64)]
# multi-wave: on 148 SMs every persistent CTA of every tiling walks 3 or more tiles (both TMEM accumulators
# change phase); only some epilogues, to keep the output bytes small
MULTI_WAVE = [(4200, 4608, 128)]


def _combos(shape):
    out = []
    for op in ("bf16", "f16"):
        for epi in ("none", "bias", "gelu"):
            for dt in ("f32", "bf16", "f16"):
                out.append((epi, dt, op))
        out += [("resid", "f32", op), ("resid-distinct", "f32", op)]
    if shape in MULTI_WAVE:
        out = [("none", "bf16", "bf16"), ("gelu", "f16", "f16"), ("resid", "f32", "bf16"), ("bias", "f32", "f16")]
    return out


def gemm_cases():
    cases = []
    for i, shape in enumerate(SMALL_SHAPES + MULTI_WAVE):
        for epi, dt, op in _combos(shape):
            cases.append((shape, epi, dt, op, 100 + i, 1.0))
    for shape in ((129, 200, 200), (257, 384, 1024)):         # fp16 outputs beyond +-65504: satfinite
        cases.append((shape, "none", "f16", "f16", 7, 3e4))
        cases.append((shape, "bias", "f16", "bf16", 8, 3e4))
    return cases


def case_id(shape, epi, dt, op, seed, a_scale):
    return f"{shape[0]}x{shape[1]}x{shape[2]}-{epi}-{dt}-{op}-s{seed}" + ("-big" if a_scale != 1.0 else "")


def tiling_of(M, N, K, out_bytes, forced, sms):
    """Which tiling launch_gemm (csrc/gemm_tcgen05.cu) runs: the forced one where it applies, else 128x256; or its
    cost model's choice."""
    if forced:
        ok = {"pair": True, "wide": True, "narrow": N > 128, "n64": out_bytes == 4 and N > 64,
              "n192": out_bytes == 2 and N % 192 == 0}[forced]
        return forced if ok else "wide"
    big = 1 << 60
    mt, nn, ks = -(-M // 128), -(-N // 256), -(-K // 64) * 4
    waves = lambda tiles, units: -(-tiles // units)
    cost = {"pair": waves(-(-M // 256) * nn, sms // 2) * ks * 135 + 5000, "wide": waves(mt * nn, sms) * ks * 163}
    best = "pair" if cost["pair"] <= cost["wide"] else "wide"
    t = {"narrow": waves(mt * -(-N // 128), sms) * ks * 99 if N > 128 else big,
         "n64": waves(mt * -(-N // 64), sms) * ks * 75 if out_bytes == 4 and N > 64 else big,
         "n192": ks * 130 if out_bytes == 2 and N % 192 == 0 and mt * (N // 192) <= sms else big}
    best_cost = cost[best]
    for name in ("narrow", "n64", "n192"):
        if t[name] < best_cost:
            best, best_cost = name, t[name]
    return best


def _run_gemm_case(L, shape, epi, dt, op, seed, a_scale, simt=False, guard=True, device_inputs=False):
    """One GEMM into a guarded view of a larger buffer; returns (output, report)."""
    M, N, K = shape
    odt, opdt = DTYPES[dt], DTYPES[op]
    A, W, bias, resid = eb.gemm_inputs(M, N, K, opdt, seed, a_scale, device=DEV if device_inputs else "cpu")
    A, W, bias, resid = A.to(DEV), W.to(DEV), bias.to(DEV), resid.to(DEV)
    code = EPIS[epi.split("-")[0]]
    pre, post = (64, 64) if guard else (0, 0)                   # 64 elements: the view stays 16-byte aligned
    buf = torch.full((pre + M * N + post,), -777.0, dtype=odt, device=DEV)
    out = buf[pre:pre + M * N].view(M, N)
    out.fill_(float("nan"))
    if code == eb.EPI_BIAS_RESIDUAL and epi == "resid":
        out.copy_(resid)
    fences = buf[:pre].clone(), buf[pre + M * N:].clone()
    residual = None
    if code == eb.EPI_BIAS_RESIDUAL:
        residual = out if epi == "resid" else resid.clone()
    L.gemm_bf16(out, A, W, None if code == eb.EPI_NONE else bias, residual=residual, epi=code, simt=simt)
    torch.cuda.synchronize()
    ctx = f"{'simt' if simt else 'tcgen05'} {case_id(shape, epi, dt, op, seed, a_scale)}"
    assert torch.equal(buf[:pre], fences[0]) and torch.equal(buf[pre + M * N:], fences[1]), f"{ctx}: wrote outside out"
    if residual is not None and epi != "resid":
        assert torch.equal(residual, resid), f"{ctx}: the distinct residual was modified"
    rep = eb.check_gemm(out, A, W, code, bias, resid, ctx, saturating=not simt)
    return out, rep


# Production shapes at d = 1024: one C2 utterance and a C3-sized batch slice (M >= 32 768)
PRODUCTION = [((M, 3 * 1024, 1024), "bias", "bf16") for M in (1027, 32768)] + \
             [((M, 1024, 1024), "resid", "f32") for M in (1027, 32768)] + \
             [((M, 4 * 1024, 1024), "gelu", "bf16") for M in (1027, 32768)] + \
             [((M, 1024, 4 * 1024), "resid", "f32") for M in (1027, 32768)]


def child_main(tiling: str, out_dir: str) -> None:
    """Runs every GEMM case on one forced tiling ('' = the launcher's choice, which also runs the production shapes
    and the SIMT kernel); writes output bytes and a report next to them."""
    from vall_e.b200 import lib as L
    L.load()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    d = Path(out_dir) / (tiling or "default")
    d.mkdir(parents=True, exist_ok=True)
    report = {}

    def run(key, ran, *args, save=False, **kw):
        try:
            out, rep = _run_gemm_case(L, *args, **kw)
        except AssertionError as e:                      # recorded: the parent lists every failing case
            report[key] = {"tiling": ran, "epi": args[1], "error": str(e)}
            return
        if save:
            out.contiguous().view(torch.uint8).cpu().numpy().tofile(d / f"{key}.bin")
        report[key] = {"tiling": ran, "epi": args[1], "ratio": rep.bound_ratio, "calib": rep.calib_ratio}

    for shape, epi, dt, op, seed, a_scale in gemm_cases():
        cid = case_id(shape, epi, dt, op, seed, a_scale)
        run(cid, tiling_of(*shape, DTYPES[dt].itemsize, tiling, sms), shape, epi, dt, op, seed, a_scale, save=True)
        if not tiling and a_scale == 1.0:
            run("simt " + cid, "simt", shape, epi, dt, op, seed, a_scale, simt=True)
    if not tiling:
        for shape, epi, dt in PRODUCTION:
            cid = "production " + case_id(shape, epi, dt, "bf16", 3, 1.0)
            run(cid, tiling_of(*shape, DTYPES[dt].itemsize, "", sms), shape, epi, dt, "bf16", 3, 1.0, guard=False,
                device_inputs=True)
            run("simt " + cid, "simt", shape, epi, dt, "bf16", 3, 1.0, simt=True, guard=False, device_inputs=True)
            torch.cuda.empty_cache()
    (d / "report.json").write_text(json.dumps(report, indent=1))


def test_gemm_every_tiling_within_bound_and_bit_identical(tmp_path):
    env = dict(os.environ)
    flags = ["-s"] if sys.flags.no_user_site else []
    code = ("import sys; sys.path[:0] = {paths!r}; import test_gpu_error_bounds as t; t.child_main({tiling!r}, {out!r})")
    paths = [str(HERE), str(HERE.parent), str(HERE.parent / "tts-with-diffusion-model_b200")]
    for tiling in TILINGS + [""]:
        if tiling:
            env["VB200_GEMM_TILE"] = tiling
        else:
            env.pop("VB200_GEMM_TILE", None)
        r = subprocess.run([sys.executable, *flags, "-c", code.format(paths=paths, tiling=tiling, out=str(tmp_path))],
                           env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, f"tiling {tiling or 'default'}:\n{r.stdout[-3000:]}\n{r.stderr[-6000:]}"
    reports = {t or "default": json.loads((tmp_path / (t or "default") / "report.json").read_text())
               for t in TILINGS + [""]}
    errors = [f"{name}: {r['error']}" for name, rep in reports.items() for r in rep.values() if "error" in r]
    # the largest err / bound and calibration ratio per tiling (pytest -s shows them)
    summary = {}
    for rep in reports.values():
        for r in rep.values():
            if "error" not in r:
                s = summary.setdefault(r["tiling"], [0.0, 0.0])
                s[0], s[1] = max(s[0], r["ratio"]), max(s[1], r["calib"])
    print("\nGEMM max err/bound, max (err - rest)/unit per tiling:", json.dumps(summary))
    assert not errors, f"{len(errors)} cases outside the bound:\n" + "\n".join(errors[:40])
    # coverage: every tiling ran every epilogue
    ran = {}
    for rep in reports.values():
        for cid, r in rep.items():
            ran.setdefault(r["tiling"], set()).add(r["epi"].split("-")[0])
    for t in TILINGS + ["simt"]:
        assert ran.get(t, set()) >= set(EPIS) - ({"resid"} if t == "n192" else set()), (t, ran.get(t))
    # cross-tiling bit identity: every child's bytes of a case are the same
    diffs = []
    for shape, epi, dt, op, seed, a_scale in gemm_cases():
        cid = case_id(shape, epi, dt, op, seed, a_scale)
        blobs = {name: (tmp_path / name / f"{cid}.bin").read_bytes() for name in reports}
        base = blobs["default"]
        for name, blob in blobs.items():
            if blob != base:
                itype = np.int32 if DTYPES[dt].itemsize == 4 else np.int16
                a, b = np.frombuffer(base, itype).astype(np.int64), np.frombuffer(blob, itype).astype(np.int64)
                diffs.append(f"{cid}: {reports['default'][cid]['tiling']} (default) vs {reports[name][cid]['tiling']} "
                             f"({name}): {int((a != b).sum())} elements differ, up to {int(np.abs(a - b).max())} ulps")
    assert not diffs, "outputs differ between tilings:\n" + "\n".join(diffs[:40])


# ---------------------------------------------------------------- attention
ALL_LENS = [1, 2, 31, 32, 33, 127, 128, 129, 160, 161, 255, 256, 257, 1027, 2527]


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


def _attn(L, qkv, lens, heads, variant):
    qkv = qkv.to(DEV)
    cu = torch.tensor([0] + list(np.cumsum(lens)), dtype=torch.int32, device=DEV)
    out = torch.full((sum(lens), heads * 64), float("nan"), dtype=torch.bfloat16, device=DEV)
    L.flash_attn_varlen(out, qkv, cu, max(lens), heads, eb.ATTN_SCALE, variant=variant)
    torch.cuda.synchronize()
    return out, qkv


@pytest.mark.parametrize("variant", ["tmem", "simt"])
@pytest.mark.parametrize("heads", [1, 2, 16])
def test_attention_every_ragged_length_within_bound(L, heads, variant):
    """Every ragged class of the last key block, in one batch (grid > SMs) and each length alone (a one-wave,
    `solo` grid, except 2527 rows with 16 heads)."""
    qkv = eb.random_qkv(sum(ALL_LENS), heads, heads)
    out, qd = _attn(L, qkv, ALL_LENS, heads, variant)
    rep = eb.check_attention(out, qd, ALL_LENS, heads, f"{variant} h{heads} batch")
    print(f"\nattention {variant} h{heads} batch: {rep}")
    r0 = 0
    for T in ALL_LENS:
        one, q1 = _attn(L, qkv[r0:r0 + T].contiguous(), [T], heads, variant)
        rep = eb.check_attention(one, q1, [T], heads, f"{variant} h{heads} T={T} alone")
        if variant == "tmem":
            assert torch.equal(one, out[r0:r0 + T]), (heads, T)     # batch composition does not change the bits
        r0 += T
    print(f"attention {variant} h{heads} alone (last T): {rep}")


RESCALE_CASES = {          # (lens, events): (utterance, key, k[0]) — the score of even query rows is k[0]
    "full-block-above": ([1027], [(0, 300, eb.GAP_ABOVE)]),
    "full-block-below": ([1027], [(0, 300, eb.GAP_BELOW)]),
    "masked-pass-above": ([328], [(0, 300, eb.GAP_ABOVE)]),
    "masked-pass-below": ([328], [(0, 300, eb.GAP_BELOW)]),
    "short-block-above": ([1027], [(0, 1025, eb.GAP_ABOVE)]),
    "short-block-below": ([1027], [(0, 1025, eb.GAP_BELOW)]),
    "moves-twice": ([1027], [(0, 300, eb.GAP_ABOVE), (0, 700, 2 * eb.GAP_ABOVE)]),
    "two-utterances": ([328, 1027], [(0, 300, eb.GAP_ABOVE), (1, 1025, eb.GAP_ABOVE)]),
}


@pytest.mark.parametrize("variant", ["tmem", "simt"])
@pytest.mark.parametrize("case", list(RESCALE_CASES))
def test_attention_lazy_rescale_within_bound(L, case, variant):
    """A row's maximum grows in a later key block by just less / just more than the kernel's rescale threshold
    (8 / log2 e), in a full block, in the masked 33-127 key pass and in the <= 32 key short chunk, once or twice."""
    lens, events = RESCALE_CASES[case]
    qkv = eb.structured_qkv(lens, 2, 40, events)
    out, qd = _attn(L, qkv, lens, 2, variant)
    print(f"\nattention {variant} rescale {case}: {eb.check_attention(out, qd, lens, 2, f'{variant} {case}')}")


@pytest.mark.parametrize("variant", ["tmem", "simt"])
def test_attention_negative_scores_within_bound(L, variant):
    """Every score negative (-10 / -5): a key past the utterance end (the next rows, or the zero rows the TMA fills
    in past the last one) would take almost all of the weight."""
    lens = [300, 1027]
    qkv = eb.structured_qkv(lens, 2, 31, base=-10.0)
    out, qd = _attn(L, qkv, lens, 2, variant)
    print(f"\nattention {variant} negative scores: {eb.check_attention(out, qd, lens, 2, variant)}")
