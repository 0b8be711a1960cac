"""TEST INFRASTRUCTURE ONLY: the oracle's dense fp16 D3PM (``oracle/d3pm.py``, the reference's tables and
algorithm, ar_discrete.py:257-277,347-375,401-420) extended to the jump posterior of a reverse loop that
skips from timestep t to s < t-1 (``Diffusion.generate_audio(sample_steps=n)``):

    q(x_s | x_t, x0)  ∝  (Q_{t|s}[j, x_t] + eps) · ((softmax(x0 logits) @ Qbar_s)_j + eps),
    Q_{t|s} = Q_{s+1} ... Q_t,

with Q_{t|s} the fp16 chain product of the reference's one-step matrices, formed as it forms ``q_mats``.
``s=None`` is the reference's own step (s = t-1) and runs the oracle's code unchanged."""
import torch
import torch.nn.functional as F

from oracle.d3pm import D3PM, EPS
from oracle.d3pm import posterior_fp32 as _posterior_fp32


class JumpD3PM(D3PM):
    def jump_mat(self, t: int, s: int) -> torch.Tensor:
        """Q_{t|s} = Q_{s+1} ... Q_t in the dtype of the one-step matrices (cached)."""
        cache = self.__dict__.setdefault("_jumps", {})
        if (t, s) not in cache:
            q = self.q_onestep_mats[s + 1]
            for u in range(s + 2, t + 1):
                q = torch.tensordot(q, self.q_onestep_mats[u], dims=[[1], [0]])
            cache[(t, s)] = q
        return cache[(t, s)]

    def _jump_fact1(self, t, s, x):
        """Q_{t|s}[j, x_t] for every token of x (B, W): row x_t of Q_{t|s}^T, per row b as ``_at`` does."""
        B, W = x.shape
        a_t = torch.stack([self.jump_mat(int(tb), int(sb)).t() for tb, sb in zip(t, s)])
        onehot = F.one_hot(x.view(B, -1).to(torch.int64), num_classes=self.K).to(a_t.dtype)
        return torch.matmul(onehot, a_t).view(B, W, self.K)

    def q_posterior_logits(self, x_start_logits, x_t, t, s=None):
        """``s`` (B,): logits of q(x_s | x_t, x0); None: the oracle's q(x_{t-1} | x_t, x0)."""
        if s is None:
            return super().q_posterior_logits(x_start_logits, x_t, t)
        fact1 = self._jump_fact1(t, s, x_t)
        fact2 = self._at_onehot(self.q_mats, s, F.softmax(x_start_logits, dim=-1))
        out = torch.log(fact1 + self.eps) + torch.log(fact2 + self.eps)
        tb = torch.reshape(t, [out.shape[0]] + [1] * (out.dim() - 1))
        return torch.where(tb == 0, x_start_logits, out)

    def p_sample(self, model_logits, t, x, noise=None, greedy=False, s=None):
        """The oracle's p_sample on the jump posterior (``s`` as above)."""
        if s is None:
            return super().p_sample(model_logits, t, x, noise, greedy)
        pred = model_logits
        tb = torch.reshape(t, [pred.shape[0]] + [1] * (pred.dim() - 1))
        post = torch.where(tb == 0, pred, self.q_posterior_logits(pred, x, t, s))
        if greedy:
            return torch.argmax(post, dim=-1), post
        nz = (t != 0).to(x.dtype).reshape(x.shape[0], *([1] * x.dim()))
        noise = torch.clamp(noise, min=torch.finfo(noise.dtype).tiny, max=1.0)
        g = -torch.log(-torch.log(noise))
        return torch.argmax(post + nz * g, dim=-1), post


def posterior_fp32(logits, x_t, t, d3pm: JumpD3PM, s=None):
    """``oracle.d3pm.posterior_fp32`` (the dense algorithm in fp32 on the upcast fp16 tables) for the jump from t
    to s (softmax @ Qbar_s, Q_{t|s} column); None: the oracle's function."""
    if s is None:
        return _posterior_fp32(logits, x_t, t, d3pm)
    p0 = torch.softmax(logits.float(), dim=-1)
    B, W = x_t.shape
    qt = torch.stack([d3pm.jump_mat(int(tb), int(sb)).t().float() for tb, sb in zip(t, s)])
    f2 = torch.matmul(p0, d3pm.q_mats.float()[s])
    f1 = qt[torch.arange(B)[:, None], x_t.long()]
    return torch.log(f1 + EPS) + torch.log(f2 + EPS)
