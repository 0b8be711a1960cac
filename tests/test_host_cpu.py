"""CPU-only tests: C-ABI surface, host-side logic (tables, layout, config, factory, sharding)."""
import ctypes
import math
import os
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "tts-with-diffusion-model_b200"


@pytest.fixture(scope="module")
def built_lib():
    sys.path.insert(0, str(PKG))
    import build
    return build.build()


def test_workspace_bytes_matches_the_layout_the_engine_carves(built_lib):
    """vb200_workspace_bytes is a host-only call: sizes in WS_FIELDS order, 256-byte granules."""
    import torch
    from vall_e.b200 import lib as L
    M, Mr, d, n_out = 1027, 750, 1024, 8192
    total, sizes = L.workspace_bytes(M, Mr, d, n_out, torch.float16)
    raw = [M * d * 4, M * d * 2, M * 3 * d * 2, M * d * 2, M * 4 * d * 2, Mr * d * 2, Mr * n_out * 2]
    assert len(sizes) == len(L.WS_FIELDS) == 7
    assert all(s % 256 == 0 and 0 <= s - r < 256 for s, r in zip(sizes, raw))
    assert total == sum(sizes)
    assert L.workspace_bytes(0, 0, d, n_out, torch.float32) == (0, [0] * 7)
    assert L.workspace_bytes(M, Mr, d, n_out, torch.float32)[1][6] == (Mr * n_out * 4 + 255) // 256 * 256
    with pytest.raises(L.VB200Error):
        L.workspace_bytes(10, 11, d, n_out, torch.float16)      # more response rows than rows


def test_library_exports_every_declared_symbol(built_lib):
    header = (ROOT / "include" / "vb200.h").read_text()
    declared = set(re.findall(r"\b(vb200_[a-z0-9_]+)\s*\(", header)) - {"vb200_stream_t"}
    assert len(declared) >= 18
    lib = ctypes.CDLL(str(built_lib))
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/vb200.h but not exported"
    from vall_e.b200 import lib as L
    assert declared == set(L.PROTOTYPES), declared ^ set(L.PROTOTYPES)
    L.load()
    assert L.load().vb200_version() == 100


def test_library_contains_blackwell_instructions(built_lib):
    sass = subprocess.run(["cuobjdump", "-sass", str(built_lib)], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in sass, f"{mnemonic} missing from SASS: not a tcgen05/TMA build"


def test_enum_values_match_header():
    from vall_e.b200 import lib as L
    header = (ROOT / "include" / "vb200.h").read_text()
    for name, val in re.findall(r"\b(VB200_[A-Z0-9_]+)\s*=\s*(-?\d+)", header):
        py = name[len("VB200_"):]
        if hasattr(L, py):
            assert getattr(L, py) == int(val), name


def test_scalar_tables_match_reference_tables(golden_dir):
    from vall_e.b200 import lib as L
    from vall_e.vall_e import d3pm
    for tr in ("absorbing", "uniform"):
        z = np.load(golden_dir / f"d3pm_{tr}_k1025.npz")
        tab = d3pm.scalar_table(int(z["S"]), int(z["K"]), tr).numpy()
        pairs = [(L.TAB_ONE_KEEP, "one_aa"), (L.TAB_ONE_OFF, "one_ab"), (L.TAB_ONE_ABSORB, "one_am"),
                 (L.TAB_ONE_BOTH, "one_mm"), (L.TAB_CUM_KEEP, "cum_aa"), (L.TAB_CUM_OFF, "cum_ab"),
                 (L.TAB_CUM_ABSORB, "cum_am"), (L.TAB_CUM_BOTH, "cum_mm")]
        for col, name in pairs:
            if tr == "absorbing":
                assert np.array_equal(tab[:, col], z[name]), (tr, name)        # bit-exact
            else:   # uniform chain product: accumulation order may move one fp16 ulp across CPUs
                assert np.allclose(tab[:, col], z[name], rtol=2e-3, atol=1e-7), (tr, name)
        assert np.array_equal(d3pm.betas_fp16(int(z["S"])).numpy(), z["betas"])
    t50 = d3pm.scalar_table(100, 1025, "absorbing")[50]
    assert abs(t50[L.TAB_LOG_KEEP] + 0.7192) < 1e-3 and abs(t50[L.TAB_LOG_OFF] + 13.8047) < 1e-3


def test_state_dict_layout_and_factory():
    from vall_e.vall_e import Diffusion, NAR, get_model
    m = NAR(1024, d_model=256, n_heads=4, n_layers=12)
    keys = set(m.state_dict())
    for k in ("sep", "text_emb.weight", "proms_emb.weight", "resps_emb.weight", "classifier.weight",
              "classifier.bias", "blocks.0.attn.block.to_qkv.weight", "blocks.11.attn.block.to_out.bias",
              "blocks.3.attn.norm.emb.weight", "blocks.3.ffn.block.0.weight", "blocks.3.ffn.block.3.bias",
              "blocks.3.ffn.norm.emb.weight"):
        assert k in keys, k
    assert "sin_emb.omega" not in keys                     # non-persistent (base.py:46)
    assert m.resps_emb.weight.shape == (7, 1024, 256) and m.blocks[0].attn.norm.emb.weight.shape == (7, 512)
    d = Diffusion(1024, d_model=256, n_heads=4, n_layers=2, n_steps=50)
    assert d.time_emb.weight.shape == (51, 256) and d.classifier.weight.shape == (8192, 256)
    assert d.blocks[0].ffn.norm.emb.weight.shape == (51, 512) and d.mask_id == 512
    full = get_model("diffusion-quarter")
    assert isinstance(full, Diffusion) and full.sep.shape == (256,) and len(full.blocks) == 12
    with pytest.raises(ValueError):
        get_model("unet")
    with pytest.raises(NotImplementedError):
        get_model("nar-tiny")
    with pytest.raises(ValueError):
        Diffusion(64, d_model=64, n_heads=1, n_layers=1, transition="gaussian")


def test_checkpoint_pickle_roundtrip(tmp_path):
    """Whole-module pickles (reference export.py:14-20) load through this package's class paths."""
    from vall_e.vall_e import Diffusion
    m = Diffusion(64, d_model=64, n_heads=1, n_layers=1, n_steps=10)
    m.phone_symmap = {"AA": 1}
    torch.save(m, tmp_path / "m.pt")
    m2 = torch.load(tmp_path / "m.pt", weights_only=False)
    assert m2.phone_symmap == {"AA": 1} and m2.timesteps == 10
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))


def test_config_cli_convention(tmp_path, monkeypatch):
    from vall_e.config import Config
    y = tmp_path / "config" / "test" / "diffused.yml"
    y.parent.mkdir(parents=True)
    y.write_text("data_dirs: [data/train]\nmodel: diffusion\nbatch_size: 6\nmax_iter: 5_000_000\n"
                 "max_train_diffusion_steps: 1000\nspkr_name_getter: \"lambda p: p.parts[-1][:4]\"\n")
    monkeypatch.chdir(tmp_path)
    c = Config.from_words([f"yaml={y}", "n_steps=25", "transition=uniform", "sampling_temperature=0.2"])
    assert (c.model, c.batch_size, c.n_steps, c.transition, c.max_iter) == ("diffusion", 6, 25, "uniform", 5_000_000)
    assert c.cfg_name == "test/diffused" and c.max_train_diffusion_steps == 1000
    assert c.data_dirs == [Path("data/train")] and c.get_spkr(Path("a/p225_001")) == "p225"
    with pytest.raises(KeyError):
        Config.from_words(["not_a_key=1"])
    monkeypatch.setattr(sys, "argv", ["prog", "hello", "model=nar", "--device", "cuda"])
    c = Config.from_cli()
    assert c.model == "nar" and sys.argv == ["prog", "hello", "--device", "cuda"]
    # a host program's own name=value words (pytest -o ...) are not config words and stay in its argv
    monkeypatch.setattr(sys, "argv", ["pytest", "-o", "addopts=", "-o", "xfail_strict=true", "n_steps=7"])
    c = Config.from_cli()
    assert c.n_steps == 7 and sys.argv == ["pytest", "-o", "addopts=", "-o", "xfail_strict=true"]


def test_reference_yaml_configs_parse():
    """The YAMLs this repo ships for BASELINE configs C1-C5 (config/{test,LibriTTS,VCTK}/diffusion*.yml), every
    YAML of the reference checkout where one can be read (oracle.refarm.reference_root), and two of the
    reference's files restated inline (so the schema is exercised without a checkout too) are accepted by the
    schema; the factory builds the model each diffusion YAML names."""
    from vall_e.config import Config
    ours = sorted((PKG / "config").rglob("*.yml"))
    assert {p.parent.name for p in ours} == {"test", "LibriTTS", "VCTK"} and len(ours) >= 5
    for p in ours:
        c = Config.from_words([f"yaml={p}"])
        assert c.model.startswith("diffusion") and c.transition in ("absorbing", "uniform") and c.n_steps >= 2
    c = Config.from_words([f"yaml={PKG / 'config' / 'test' / 'diffusion.yml'}"])
    assert (c.model, c.n_steps, c.transition) == ("diffusion-quarter", 51, "uniform")          # C1
    c = Config.from_words([f"yaml={PKG / 'config' / 'VCTK' / 'diffusion.yml'}", "n_steps=11"])  # C5 sweep point
    assert (c.model, c.n_steps, c.transition) == ("diffusion", 11, "absorbing")
    from oracle.refarm import reference_root
    ref = reference_root()
    if ref is not None and (ref / "config").is_dir():
        n_ref = 0
        for p in sorted((ref / "config").rglob("*.yml")):
            c = Config.from_words([f"yaml={p}"])
            assert c.model.split("-")[0] in ("ar", "nar"), (p, c.model)
            n_ref += 1
        assert n_ref >= 9
    ref_cfgs = {
        "LibriTTS/nar.yml": "data_dirs: [data/LibriTTS/]\nspkr_name_getter: \"lambda p: p.parts[-3]\"\nmodel: nar\n"
                            "batch_size: 24\neval_batch_size: 24\neval_every: 1_000\nsampling_temperature: 0.2\n",
        "test/diffused.yml": "data_dirs: [data/train]\nmodel: ar\nspkr_name_getter: \"lambda p: p.parts[-1][:4]\"\n"
                             "batch_size: 6\neval_batch_size: 6\nsave_ckpt_every: 500\neval_every: 100000\n"
                             "max_iter: 5000000\nmax_train_diffusion_steps: 1000\n",
    }
    import tempfile
    for name, text in ref_cfgs.items():
        with tempfile.TemporaryDirectory() as d:
            p = Path(d) / name
            p.parent.mkdir(parents=True)
            p.write_text(text)
            c = Config.from_words([f"yaml={p}"])
            assert c.model in ("nar", "ar")


def test_cli_main_reaches_the_kernels_and_fails_loudly_without_cuda(tmp_path, monkeypatch):
    """The entry point (reference __main__.py:44-73) with a stand-in of the reference's emb/qnt.py and emb/g2p.py
    loaded through vall_e.emb (stub encodec / torchaudio / soundfile / g2p_en): checkpoint pickle, symmap, prompt
    encoding and phonemisation all run; on a CPU device the denoiser then refuses (no CPU fallback)."""
    from cli_helpers import run_cli, standin_reference_emb
    from vall_e.b200 import lib as L
    ref = standin_reference_emb(tmp_path / "standin")
    main, calls, out = run_cli(tmp_path, monkeypatch, "cpu", ref)
    import vall_e.emb.qnt as qnt
    if qnt.encode_from_file.__defaults__ == ("cuda",):   # the reference's EnCodec wrapper defaults to device="cuda"
        monkeypatch.setattr(qnt.encode_from_file, "__defaults__", ("cpu",))
    with pytest.raises(L.VB200Error, match="no CPU fallback"):
        main()
    assert ("bandwidth", 6.0) in calls and any(c[0] == "encode" for c in calls)
    assert not out.exists()
    import vall_e.emb as emb
    assert Path(emb.qnt.__file__).parent == (ref / "vall_e" / "emb")          # the reference's file, not a copy


def test_uniform_chain_product_is_structured_up_to_one_fp16_ulp():
    """d3pm.scalar_table reads 'the' diagonal / off-diagonal value of the fp16 chain product.  Absorbing: the
    dense product is exactly rank-structured.  Uniform: K-term sums, so entries differ from the scalars by at
    most one fp16 ulp — the bound the closed-form posterior (KL <= 1e-3 bar) rests on; the bit-exact q_sample
    path reads the dense table (dense_log_qbar), which must be the oracle's log(q_mats + eps) bit for bit."""
    from oracle.d3pm import D3PM, EPS
    from vall_e.b200 import lib as L
    from vall_e.vall_e import d3pm as pd
    S, K = 30, 257
    for tr in ("absorbing", "uniform"):
        orc, tab = D3PM(S, K, tr), pd.scalar_table(S, K, tr)
        q = orc.q_mats.float()
        m = K // 2
        eye = torch.eye(K, dtype=torch.bool)
        worst = 0.0
        for t in range(S):
            diag, off = q[t][eye], q[t][~eye]
            if tr == "absorbing":
                rows = torch.arange(K) != m
                assert torch.equal(q[t][rows, rows], tab[t, L.TAB_CUM_KEEP].expand(K - 1))
                assert torch.equal(q[t][rows, m], tab[t, L.TAB_CUM_ABSORB].expand(K - 1))
                assert float(q[t][m, m]) == float(tab[t, L.TAB_CUM_BOTH])
                continue
            for vals, ref in ((diag, tab[t, L.TAB_CUM_KEEP]), (off, tab[t, L.TAB_CUM_OFF])):
                ulp = 2.0 ** (math.floor(math.log2(float(ref))) - 10)
                worst = max(worst, float((vals - ref).abs().max()) / ulp)
        assert worst <= 1.0, worst
        dense = pd.dense_log_qbar(S, K, tr)
        assert dense.dtype == torch.float16 and torch.equal(dense, torch.log(orc.q_mats + EPS))


def test_token_ids_are_range_checked_on_the_host():
    """Kernels index embedding tables with raw ids; like the reference (IndexError from F.one_hot /
    nn.Embedding) an id outside its table is refused before any launch."""
    from vall_e.b200.engine import check_ids
    check_ids(torch.tensor([0, 5, 1023]), 1024, "ok")
    with pytest.raises(IndexError):
        check_ids(torch.tensor([0, 1024]), 1024, "AR stop token in a K=1024 model")
    with pytest.raises(IndexError):
        check_ids(torch.tensor([-1, 3]), 1024, "negative id")


def test_batch_layout_records():
    from vall_e.b200 import lib as L
    from vall_e.b200.engine import BatchLayout
    if not torch.cuda.is_available():
        dev = "cpu"
        # pin_memory needs CUDA; emulate by patching
        orig = torch.Tensor.pin_memory
        torch.Tensor.pin_memory = lambda self, *a, **k: self
    else:
        dev = "cuda"
    try:
        text = [torch.tensor([3, 4, 5]), torch.tensor([9])]
        proms = [torch.zeros(2, 8, dtype=torch.long), torch.ones(4, 8, dtype=torch.long)]
        lay = BatchLayout(text, proms, [5, 2], dev)
    finally:
        if dev == "cpu":
            torch.Tensor.pin_memory = orig
    assert lay.M == (3 + 1 + 2 + 1 + 5) + (1 + 1 + 4 + 1 + 2) and lay.max_T == 12 and lay.M_resp == 7
    utt = lay.utt.cpu().numpy()
    assert utt[1, L.U_ROW0] == 12 and utt[1, L.U_TXT0] == 3 and utt[1, L.U_PROM0] == 2 and utt[1, L.U_RESP0] == 5
    assert lay.cu_rows.cpu().tolist() == [0, 12, 21]
    assert lay.resp_row_index.cpu().tolist() == [7, 8, 9, 10, 11, 19, 20]
    assert lay.row_utt.cpu().tolist() == [0] * 12 + [1] * 9
    with pytest.raises(ValueError):
        BatchLayout(text, [torch.zeros(2, 7, dtype=torch.long)] * 2, [5, 2], dev)
    with pytest.raises(ValueError):
        BatchLayout([], [], [], dev)


def test_partition_balances_and_covers():
    from vall_e.b200.shard import partition
    costs = [100, 90, 80, 10, 10, 10, 5, 5]
    parts = partition(costs, 3)
    assert sorted(i for p in parts for i in p) == list(range(8))
    loads = [sum(costs[i] for i in p) for p in parts]
    assert max(loads) - min(loads) <= 15
    assert partition(costs, 1) == [list(range(8))]
    assert partition([], 4) == [[], [], [], []]
    assert partition([7], 2) == [[0], []]


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from vall_e.b200.shard import generate_sharded
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(0)
    lens = [5, 17, 3, 9, 12]
    text = [torch.randint(1, 50, (4 + i,), generator=g) for i in range(5)]
    proms = [torch.randint(0, 50, (6, 8), generator=g) for _ in range(5)]

    def fake_generate(t, p, rl, gids):      # codes depend only on (global id, length): sharding-invariant
        return [((torch.arange(n * 8).view(n, 8) * 7 + gid * 13) % 1024).long() for n, gid in zip(rl, gids)]

    out = generate_sharded(fake_generate, text, proms, lens, group=None, device=torch.device("cpu"))
    ref = fake_generate(None, None, lens, list(range(5)))
    q.put((rank, all(torch.equal(a, b) for a, b in zip(out, ref))))
    dist.destroy_process_group()


def test_sharded_generation_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 500)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _compat_dit(golden_dir):
    import detrand
    from vall_e.vall_e.ar_discrete import AR
    z = np.load(golden_dir / "ar_discrete_dit.npz")
    m = AR(32, 100, 1025, 8, 16, 8).eval()
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    sd = {}
    for i, (k, shape) in enumerate(sorted(shapes.items())):     # same recipe as make_golden.det_state_dict
        v = detrand.normal(4242 + 17 * i, tuple(shape)) * np.float32(0.1)
        if k.endswith("weight") and len(shape) == 1:
            v = v + np.float32(1.0)
        sd[k] = torch.from_numpy(v.astype(np.float32))
    m.load_state_dict(sd)
    seed = int(z["seed"])
    text = torch.from_numpy(detrand.integers(seed, 1, 1025, (37,)))
    proms = torch.from_numpy(detrand.integers(seed + 1, 0, 1025, (180, 8)))
    x_t = torch.zeros(1, 448, dtype=torch.int32)
    x_t[0, :350] = torch.from_numpy(detrand.integers(seed + 2, 1, 1025, (350,))).int()
    return m, z, shapes, text, proms, x_t


def test_ar_discrete_compat_matches_reference_module(golden_dir):
    """SURVEY §8f.2: the drop-in for the reference's own D3PM class (ar_discrete.py:205-256) has the
    reference's state-dict keys and shapes, and its conditioning encoders and DiT denoiser reproduce
    the reference modules' outputs (fixture written by make_golden.gen_ar_discrete_dit)."""
    m, z, shapes, text, proms, x_t = _compat_dit(golden_dir)
    assert sorted(shapes) == [str(k) for k in z["keys"]]
    assert [str(shapes[k]) for k in sorted(shapes)] == [str(s) for s in z["shapes"]]
    with torch.no_grad():
        cond1, cond2 = m.conditioning(text, proms)
        logits = m.denoise_logits(x_t, torch.tensor([int(z["t"])]), cond1, cond2, x_t[0] != 0)
    assert cond1.shape == (1, 398, 32) and cond2.shape == (1, 50, 32) and logits.shape == (1, 448, 1025)
    assert np.abs(cond1[0, :4].numpy() - z["cond1_head"]).max() <= 1e-5
    assert np.abs(cond2[0, :4].numpy() - z["cond2_head"]).max() <= 1e-5
    err = np.abs(logits[0, z["rows"]].numpy() - z["logits_rows"]).max()
    assert err <= 1e-4, err                               # fp32 PyTorch modules on both sides
    assert abs(float(logits.double().sum()) - float(z["logits_sum"])) <= 1e-2 * 448
    # D3PM constants of the class: K = 1025, absorbing class 512, 100 timesteps (ar_discrete.py:207,255,332)
    assert (m.num_classes, m.mask_id, m.timesteps, m.transition) == (1025, 512, 100, "absorbing")
    with pytest.raises(ValueError):
        m.generate_audio([text, text], [proms, proms])


def test_operand_format_selection(monkeypatch):
    """VB200_ACT picks which GEMM operand sets are fp16 (engine._act_dtypes): default = classifier only."""
    from vall_e.b200 import engine
    monkeypatch.delenv("VB200_ACT", raising=False)
    assert engine._act_dtypes() == {"h": torch.bfloat16, "ff": torch.bfloat16, "head": torch.float16}
    for v, want in (("bf16", set()), ("f16", {"h", "ff", "head"}), ("head,ff", {"head", "ff"}), ("h", {"h"})):
        monkeypatch.setenv("VB200_ACT", v)
        got = engine._act_dtypes()
        assert {k for k, dt in got.items() if dt == torch.float16} == want, v
    monkeypatch.setenv("VB200_ACT", "fp8")
    with pytest.raises(ValueError):
        engine._act_dtypes()
