"""ORACLE / REFERENCE ARM — TEST AND BENCH INFRASTRUCTURE ONLY.  Not product code.

The reference's OWN modules as the CPU arm of ``bench.py`` (``--impl reference`` and the
``cpu_baseline`` leg) and as a cross-check of the oracle port:

* ``stage()`` — the committed recipe: copies ``vall_e/vall_e/{base,nar,ar_discrete}.py`` verbatim from
  the reference checkout (``reference_root()``) into the git-ignored ``oracle/_ref/`` (it never enters the
  history).  Run by ``__graft_entry__.build()``; a no-op where no checkout can be read.
* ``load()`` — imports the staged files behind a shim package: the reference package itself cannot be
  imported (``vall_e/config.py:96`` needs omegaconf; ``ar_discrete.py:14,16`` import diffusers / timm, which
  are stubbed — only ``timm...Mlp`` is structurally needed and the benchmarked path never builds it).
* ``ReferenceStep`` — one denoise step of ONE utterance on the path BASELINE.json names, executed by the
  reference's classes and functions, unmodified:
    - denoiser: a subclass of the reference's ``Base`` (``base.py:289-499``; its Embedding, MultiEmbedding
      one-hot einsum, SinusodialEmbedding, Block / AdaLN / Attention, classifier) in the non-causal AdaLN
      configuration of ``nar.py:8-26``, with the glue of SURVEY.md §7.1 the reference never assembles
      (8 response levels, AdaLN rows = timesteps, ``time_emb``, 8 K-way heads);
    - sampler: ``AR.p_sample`` / ``q_posterior_logits`` / ``_at`` / ``_at_onehot`` of ``ar_discrete.py:337-420``
      bound to a namespace holding the fp16 tables the constructor builds (``:257-277``; the constructor
      itself hard-codes ``.to("cuda:0")``), in the reference's own call convention: one utterance is ONE
      row, ``x`` of shape (1, W) (``ar_discrete.py:699-712,750-776``), fp16 logits, ``torch.rand`` on the CPU.
"""
from __future__ import annotations

import importlib.util
import json
import os
import shutil
import sys
import types
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
STAGED = HERE / "_ref"
FILES = ("base.py", "nar.py", "ar_discrete.py")


def reference_root() -> Path | None:
    """The reference checkout: ``VALL_E_REF`` (its repository root), else ``reference`` next to this repository,
    else BASELINE.json's ``reference_path`` — the order of ``vall_e.emb``.  A location this user cannot read
    counts as absent (os.path.isdir returns False where pathlib would raise PermissionError)."""
    cands = [os.environ.get("VALL_E_REF"), str(HERE.parent.parent / "reference")]
    try:
        cands.append(json.loads((HERE.parent / "BASELINE.json").read_text()).get("reference_path"))
    except (OSError, ValueError):
        pass
    for c in cands:
        if c and os.path.isdir(os.path.join(c, "vall_e", "vall_e")):
            return Path(c)
    return None


def stage() -> bool:
    """Copies the three reference modules into oracle/_ref/ (verbatim).  True if they are staged."""
    root = reference_root()
    src = root / "vall_e" / "vall_e" if root else None
    if src is not None and all(os.path.isfile(src / f) for f in FILES):
        STAGED.mkdir(exist_ok=True)
        for f in FILES:
            shutil.copyfile(src / f, STAGED / f)
    return available()


def available() -> bool:
    return all((STAGED / f).is_file() for f in FILES)


_mods = None


def load():
    """{'base', 'nar', 'ar_discrete'} -> the reference's modules, executed from oracle/_ref/."""
    global _mods
    if _mods is not None:
        return _mods
    if not available():
        raise FileNotFoundError("oracle/_ref/ is not staged: run oracle.refarm.stage() where a checkout of the "
                                "reference can be read (see reference_root)")
    diffusers = types.ModuleType("diffusers")
    for n in ("UNet3DConditionModel", "UNet2DConditionModel", "DDPMScheduler",
              "CosineDPMSolverMultistepScheduler", "DDIMScheduler"):
        setattr(diffusers, n, object)
    tv = types.ModuleType("timm.models.vision_transformer")
    for n in ("PatchEmbed", "Attention", "Mlp"):
        setattr(tv, n, object)
    for name, mod in (("diffusers", diffusers), ("timm", types.ModuleType("timm")),
                      ("timm.models", types.ModuleType("timm.models")), ("timm.models.vision_transformer", tv)):
        sys.modules.setdefault(name, mod)
    pkg = types.ModuleType("vb200_refpkg")
    pkg.__path__ = [str(STAGED)]
    sys.modules["vb200_refpkg"] = pkg
    mods = {}
    for name in ("base", "nar", "ar_discrete"):
        spec = importlib.util.spec_from_file_location(f"vb200_refpkg.{name}", STAGED / f"{name}.py")
        m = importlib.util.module_from_spec(spec)
        sys.modules[f"vb200_refpkg.{name}"] = m
        spec.loader.exec_module(m)
        mods[name] = m
    _mods = mods
    return mods


K_REF = 1025      # the reference hard-codes its class count (ar_discrete.py:255,309,328-332,343-345,397,402)


def reference_tables(AR, S: int, transition: str):
    """The tensors of ar_discrete.py:257-277 on the CPU (the constructor hard-codes ``.to("cuda:0")``), built
    by the reference's own functions, with its D3PM methods bound to the namespace that holds them."""
    s = types.SimpleNamespace(timesteps=S, eps=1.0e-6, num_classes=K_REF, num_pixel_vals=K_REF)
    s.betas = AR.cosine_beta_schedule(s, S + 1).to(torch.float16)
    one = ([AR._get_absorbing_transition_mat(s, t) for t in range(S)] if transition == "absorbing"
           else [AR.create_transition_matrix(s, s.betas[t]) for t in range(S)])
    s.q_onestep_mats = torch.stack(one, dim=0).to(torch.float16)
    q = s.q_onestep_mats[0]
    qs = [q]
    for t in range(1, S):
        q = torch.tensordot(q, s.q_onestep_mats[t], dims=[[1], [0]])
        qs.append(q)
    s.q_mats = torch.stack(qs, dim=0).to(torch.float16)
    s.transpose_q_onestep_mats = torch.transpose(s.q_onestep_mats, 1, 2).to(torch.float16)
    for name in ("_at", "_at_onehot", "q_probs", "q_posterior_logits", "p_sample", "q_sample"):
        setattr(s, name, types.MethodType(getattr(AR, name), s))
    return s


class ReferenceStep:
    """One utterance; ``step()`` = reference denoiser forward (fp32) + reference ``p_sample`` (fp16 tables).
    The class count is the reference's hard-coded 1025 (its ``p_sample`` draws ``torch.rand(x.shape + (1025,))``),
    i.e. 0.1 % more classifier / sampler work than BASELINE's K = 1024 — the price of running it unmodified."""

    def __init__(self, d_model, n_heads, n_layers, timesteps, transition, text, proms, t_resp, seed=0):
        mods = load()
        base, AR = mods["base"], mods["ar_discrete"].AR
        K = K_REF
        torch.manual_seed(seed)

        class Glue(base.Base):
            casual = False
            n_resp_levels = 8
            use_stop_token = False
            norm_type = "adaln"
            resp_loss_only = True

        gm = Glue(K, d_model=d_model, n_heads=n_heads, n_layers=n_layers, p_dropout=0.1).eval()
        for blk in gm.blocks:
            for sub in (blk.attn, blk.ffn):
                sub.norm = base.AdaLN(d_model, timesteps + 1)
                torch.nn.init.normal_(sub.norm.emb.weight, std=0.02)
        gm.classifier = torch.nn.Linear(d_model, 8 * K)
        gm.time_emb = torch.nn.Embedding(timesteps + 1, d_model)
        self.base, self.gm, self.K, self.S = base, gm, K, timesteps
        self.tab = reference_tables(AR, timesteps, transition)
        self.text, self.proms = text, proms
        self.x = (torch.full((t_resp, 8), K // 2, dtype=torch.long) if transition == "absorbing"
                  else torch.randint(0, K, (t_resp, 8)))
        self.t = timesteps - 1

    @torch.no_grad()
    def logits(self, x, t):
        """(t'', 8, K) fp32: the reference's modules in the order of Base.forward (base.py:427-443)."""
        gm, base = self.gm, self.base
        tt = torch.tensor([t])
        resp = [r + gm.time_emb(tt[i])[None] for i, r in enumerate(gm.resps_emb([x]))]
        x_list = gm._samplewise_merge_tensors(gm.text_emb([self.text]), gm.proms_emb([self.proms]), resp, sep=gm.sep)
        h, m = base.list_to_tensor(x_list)
        h = gm.sin_emb.add_pe(h)
        for blk in gm.blocks:
            h = blk(h, m, tt)
        h = gm.classifier(h) * m
        return h[0, -len(x):].view(len(x), 8, self.K)

    @torch.no_grad()
    def step(self):
        lg = self.logits(self.x, self.t).to(torch.float16).view(1, -1, self.K)      # one utterance = one row
        x_row = self.x.reshape(1, -1).to(torch.int32)
        samp, _ = self.tab.p_sample(lg, torch.tensor([self.t]), x_row)              # torch.rand inside, CPU
        self.x = samp.view(-1, 8).long()
        self.t = max(self.t - 1, 1)
        return self.x
