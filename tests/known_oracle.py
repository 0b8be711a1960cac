"""TEST INFRASTRUCTURE ONLY: the jump oracle (``jump_oracle.JumpD3PM``: the oracle's dense fp16 D3PM with the
jump posterior of ``sample_steps``) extended to the ids form of ``q_posterior_logits`` — the reference's
``x_start_logits=False`` branch (ar_discrete.py:347-375), where x0 is given as class ids:

    q(x_s | x_t, x0 = k)  ∝  (Q_{t|s}[j, x_t] + eps) · (Qbar_s[k, j] + eps),

fact2 = row k of Qbar_s taken as ``_at(q_mats, s, x_start)``; ``s=None`` is the one-step posterior, s = t-1.
This is the law of a known token of ``Diffusion.generate_audio(known_list=...)``."""
import torch

from jump_oracle import JumpD3PM


class KnownD3PM(JumpD3PM):
    def _fact1(self, t, s, x_t):
        if s is None:
            return self._at(self.transpose_q_onestep_mats, t, x_t), torch.where(t == 0, t, t - 1)
        return self._jump_fact1(t, s, x_t), s

    def q_posterior_logits_ids(self, x_start, x_t, t, s=None):
        """(B, W, K) logits of q(x_s | x_t, x0 = x_start) in the oracle's fp16 arithmetic; t == 0 rows are 0, as the
        reference's ``torch.where(t == 0, x_start_logits, out)`` gives with ``x_start_logits=False``."""
        fact1, s = self._fact1(t, s, x_t)
        fact2 = self._at(self.q_mats, s, x_start)
        out = torch.log(fact1 + self.eps) + torch.log(fact2 + self.eps)
        tb = torch.reshape(t, [out.shape[0]] + [1] * (out.dim() - 1))
        return torch.where(tb == 0, torch.zeros_like(out), out)

    def log_law_ids(self, x_start, x_t, t, s=None):
        """The same logits in float64 on the oracle's fp16 tables: log(fact1 + eps) + log(fact2 + eps), t >= 1."""
        fact1, s = self._fact1(t, s, x_t)
        fact2 = self.q_mats[s.long()[:, None], x_start.long()].double()   # row x0 of Qbar_s, (B, W, K)
        return torch.log(fact1.double() + self.eps) + torch.log(fact2 + self.eps)

    def p_sample_ids(self, x_start, t, x, noise=None, greedy=False, s=None):
        """(codes, float64 logits) of a known token's step: arg max of the law (greedy) or Gumbel-arg max with the
        reference's noise; t == 0 returns x_start."""
        post = self.log_law_ids(x_start, x, t, s)
        if greedy:
            code = torch.argmax(post, dim=-1)
        else:
            noise = torch.clamp(noise, min=torch.finfo(noise.dtype).tiny, max=1.0)
            code = torch.argmax(post + (-torch.log(-torch.log(noise))).double(), dim=-1)
        tb = torch.reshape(t, [x.shape[0]] + [1] * (x.dim() - 1))
        return torch.where(tb == 0, x_start.long(), code), post
