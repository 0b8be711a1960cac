"""NAR: the non-causal AdaLN configuration of ``Base`` (reference ``vall_e/vall_e/nar.py:8-26``)
and its level-by-level inference loop (``nar.py:76-99``), running on the B200 kernels."""
from __future__ import annotations

import torch
from torch import Tensor

from ..b200 import lib as L
from ..b200.engine import BatchLayout, check_ids
from .base import Base
from .diffusion import D3PMOps


class NAR(Base):
    @property
    def n_resp_levels(self):
        return 7

    @property
    def casual(self):
        return False

    @property
    def use_stop_token(self):
        return False

    @property
    def norm_type(self):
        return "adaln"

    @property
    def resp_loss_only(self):
        return True

    def forward(self, text_list: list[Tensor], proms_list: list[Tensor], resps_list: list[Tensor],
                sampling_temperature: float = 0.2, seed: int | None = None, gids=None):
        """resps_list: [t'' l]; with l < 8 known levels, fills levels l .. 7 one forward pass per
        level (AdaLN row = level being predicted - 1) and returns [t'' 8].  Errors as the reference:
        ``ValueError`` when utterances carry different numbers of levels (nar.py:44-47).

        ``seed=None`` samples each level with ``Categorical(logits / sampling_temperature)`` on torch's global RNG,
        as the reference.  With a seed, every level is drawn on the device from softmax(logits /
        sampling_temperature) by ``vb200_head_categorical_sample``, keyed by (seed, global utterance id, frame * 8 +
        level): the codes are reproducible and do not depend on the batch an utterance is in.  ``gids`` give the
        global utterance ids (default 0 .. B-1), as in ``Diffusion.generate_audio``.  All levels then run on one
        packed layout and workspace; the given levels come back unchanged."""
        n_levels_set = {r.shape[-1] for r in resps_list}
        if len(n_levels_set) > 1:
            raise ValueError(f"Please give only one level, got {n_levels_set}.")
        n_levels = next(iter(n_levels_set))
        if n_levels == self.n_resp_levels + 1:
            raise NotImplementedError("NAR training step (8 given levels) is outside the B200 inference path")
        if seed is not None:
            return self._forward_seeded(text_list, proms_list, resps_list, D3PMOps._temperature(sampling_temperature),
                                        int(seed), gids)
        device = text_list[0].device
        prev_list = resps_list
        while True:
            level = prev_list[0].shape[-1] - 1
            if level >= self.n_resp_levels:
                break
            quant_levels = torch.full((len(text_list),), level, device=device)
            resp_list = super().forward(text_list, proms_list, prev_list, return_all_resp=True,
                                        shift_targ_list=False, quant_levels=quant_levels,
                                        sampling_temperature=sampling_temperature)
            prev_list = [torch.cat([rs, r.to(rs).unsqueeze(-1)], dim=-1) for rs, r in zip(prev_list, resp_list)]
        return prev_list

    @torch.no_grad()
    def _forward_seeded(self, text_list, proms_list, resps_list, temperature, seed, gids):
        eng = self.engine()
        w, dev = eng.w, eng.w.device
        n_given, n_all = int(resps_list[0].shape[-1]), self.n_resp_levels + 1
        lay = BatchLayout(text_list, proms_list, [len(r) for r in resps_list], dev, gids=gids,
                          n_text=w.text_w.shape[0], n_codes=w.K)
        ws = eng.workspace(lay)
        given = torch.cat([r.reshape(len(r), n_given) for r in resps_list]).to(dev, torch.int32)
        check_ids(given, w.K, "resps_list")
        codes = torch.zeros(lay.M_resp, n_all, dtype=torch.int32, device=dev)
        codes[:, :n_given] = given
        # AdaLN row of each pass (the reference's quant_levels), made once: the norm kernels read it before they
        # wait on the launch in front of them
        rows = torch.arange(n_all, dtype=torch.int32, device=dev).repeat_interleave(lay.B).view(n_all, lay.B)
        with torch.cuda.device(dev):
            for level in range(n_given - 1, self.n_resp_levels):
                head_in = eng.forward(lay, ws, codes[:, :level + 1].contiguous(), rows[level], use_time=False,
                                      head=False)
                L.head_categorical_sample(codes, level + 1, ws.logits, head_in, w.w_cls, w.b_cls, lay.resp_row_utt,
                                          lay.utt, temperature, L.NOISE_PHILOX, seed)
                eng.launches += 1
        out = codes.to(resps_list[0].device, resps_list[0].dtype)
        return list(out.split(lay.t_resp, dim=0))
