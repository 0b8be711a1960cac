"""GPU tests of the plain categorical draw (``vb200_head_categorical_sample``: the fused classifier head's categorical
mode at K = 1024, GEMM + one-warp-per-row kernel otherwise) against float64 softmax(logits / tau), and of the seeded
NAR level loop (``NAR.forward(seed=...)``): reproducible, independent of batch composition and utterance order, given
levels returned unchanged."""
import pytest
import torch

from test_gpu_sample_steps import _chi2_ok

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


def _head(K, d, seed, scale=0.22):
    g = torch.Generator().manual_seed(seed)
    W = (torch.randn(K, d, generator=g) * scale).to(torch.float16)
    bias = torch.randn(K, generator=g)
    return g, W, bias


@pytest.mark.parametrize("tau", [0.2, 1.0, 2.0])
@pytest.mark.parametrize("K", [1024, 64, 1000])
def test_categorical_law(L, K, tau):
    """n draws of one row (40 960 utterances of one frame) against float64 softmax((row W^T + b) / tau); K = 1024 is
    the fused mode, 64 and 1000 the standalone kernel (the classifier GEMM needs K % 8 == 0)."""
    n, d = 40960, 128
    g, W, bias = _head(K, d, 7 + K)
    row = torch.randn(1, d, generator=g).to(torch.float16)
    law = torch.softmax((row.double() @ W.double().t() + bias.double())[0] / tau, -1)
    head_in = row.repeat(n, 1).to(DEV)
    utt = torch.zeros(n, L.U_STRIDE, dtype=torch.int32)
    utt[:, L.U_RESP0] = torch.arange(n)
    utt[:, L.U_GID] = torch.arange(n)
    out = torch.full((n, 8), -7, dtype=torch.int32, device=DEV)
    logits = torch.empty(n, K, dtype=torch.float16, device=DEV)
    assert L.head_fused(d, K, L.NOISE_PHILOX) == (K == 1024)
    L.head_categorical_sample(out, 3, logits, head_in, W.to(DEV), bias.to(DEV),
                              torch.arange(n, dtype=torch.int32, device=DEV), utt.to(DEV), tau, L.NOISE_PHILOX, seed=5)
    got = out.cpu()
    ok, stat = _chi2_ok(got[:, 3], law)
    assert ok, (K, tau, stat)
    others = torch.cat([got[:, :3], got[:, 4:]], 1)
    assert bool((others == -7).all())                   # only column `col` is written


@pytest.mark.parametrize("K", [1024, 64])
def test_categorical_greedy_is_the_arg_max(L, K):
    rows, d = 600, 128
    g, W, bias = _head(K, d, 3 + K, scale=0.3)
    head_in = torch.randn(rows, d, generator=g).to(torch.float16)
    logits = (head_in.double() @ W.double().t() + bias.double())
    top2 = logits.topk(2, -1).values
    clear = (top2[:, 0] - top2[:, 1]) > 1e-2
    assert clear.float().mean() > 0.8
    utt = torch.zeros(1, L.U_STRIDE, dtype=torch.int32, device=DEV)
    out = torch.full((rows, 2), -7, dtype=torch.int32, device=DEV)
    scratch = torch.empty(rows, K, dtype=torch.float16, device=DEV)
    for tau in (0.3, 1.0, 4.0):                         # greedy: the raw arg max whatever the temperature
        L.head_categorical_sample(out, 0, scratch, head_in.to(DEV), W.to(DEV), bias.to(DEV),
                                  torch.zeros(rows, dtype=torch.int32, device=DEV), utt, tau, L.NOISE_GREEDY)
        got = out.cpu().long()
        assert torch.equal(got[clear, 0], logits.argmax(-1)[clear]), tau
        assert bool((got[:, 1] == -7).all())


def _nar(K, seed):
    from vall_e.vall_e import NAR
    torch.manual_seed(seed)
    m = NAR(K, d_model=128, n_heads=2, n_layers=2)
    with torch.no_grad():
        for blk in m.blocks:                             # exercise the AdaLN rows (zero-initialised)
            blk.attn.norm.emb.weight.normal_(0, 0.05)
            blk.ffn.norm.emb.weight.normal_(0, 0.05)
    return m.to(DEV)


def _utts(K, n, seed):
    g = torch.Generator().manual_seed(seed)
    lens = [(3 + 2 * i, 5 + i, 20 + 17 * i) for i in range(n)]
    text = [torch.randint(1, K, (a,), generator=g).to(DEV) for a, _, _ in lens]
    proms = [torch.randint(0, K, (b, 8), generator=g).to(DEV) for _, b, _ in lens]
    resps = [torch.randint(0, K, (c, 1), generator=g).to(DEV) for _, _, c in lens]
    return text, proms, resps


@pytest.mark.parametrize("K", [64, 1024])
def test_seeded_nar_loop_is_reproducible_and_batch_invariant(L, K):
    m = _nar(K, 31)
    text, proms, resps = _utts(K, 4, 37)
    a = m(text, proms, resps, seed=11)
    b = m(text, proms, resps, seed=11)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert [tuple(x.shape) for x in a] == [(len(r), 8) for r in resps]
    for x, r in zip(a, resps):
        assert torch.equal(x[:, :1], r)                 # the given level comes back unchanged
        assert 0 <= int(x.min()) and int(x.max()) < K
    c = m(text, proms, resps, seed=12)
    assert not all(torch.equal(x, y) for x, y in zip(a, c))
    # alone, inside the batch, and under a permutation of global ids split across two calls
    for i in range(4):
        (alone,) = m(text[i:i + 1], proms[i:i + 1], resps[i:i + 1], seed=11, gids=[i])
        assert torch.equal(alone, a[i]), i
    order = [2, 0, 3, 1]
    first, second = order[:2], order[2:]
    p1 = m([text[i] for i in first], [proms[i] for i in first], [resps[i] for i in first], seed=11, gids=first)
    p2 = m([text[i] for i in second], [proms[i] for i in second], [resps[i] for i in second], seed=11, gids=second)
    for i, x in zip(order, p1 + p2):
        assert torch.equal(x, a[i]), i
    # two given levels: both come back, levels 2-7 are drawn
    two = [torch.cat([x[:, :2]], 1) for x in a]
    d = m(text, proms, two, seed=11)
    for x, y in zip(d, a):
        assert torch.equal(x[:, :2], y[:, :2])
        assert torch.equal(x, y)                        # same keys, same earlier levels: the same draws
