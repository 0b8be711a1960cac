"""The fused classifier head (head_sample_kernel, csrc/head_sample_tcgen05.cu) against float64 references with
bounds derived from its arithmetic (tests/head_bounds.py), on launches where every CTA pair walks at least three
work items, over tile counts 1, 3, 4 and 16, reduction dims with a partial last k-block, 1 / 3 / 8 levels, bf16
and fp16 operands and both transitions:

  greedy codes equal the float64 posterior's arg max on every clear token, planted exact ties go to the lowest
  class; codes are bit-identical when one 256-row block runs alone and when whole utterances are permuted (the
  deterministic catch for state carried from one work item to the next); Philox draws follow the float64
  posterior (randomised PIT, Kolmogorov-Smirnov); the cross-entropy epilogue is within its bound everywhere.
Each test prints what calibration of C_ACC / C_CE uses and the work items per CTA pair."""
import numpy as np
import pytest
import torch

import error_bounds as eb
import head_bounds as hb

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def L():
    from vall_e.b200 import lib
    lib.load()
    return lib


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _table(K, tr):
    from vall_e.vall_e import d3pm as pd
    return pd.scalar_table(hb.S_STEPS, K, tr)


def _on_dev(c):
    return {k: getattr(c, k).to(DEV) for k in ("head_in", "W", "bias", "x_t", "row_utt", "t_utt", "utt")}


def _sample(L, c, dv, table, tr, noise, seed=0, rows=None, utt=None, perm=None):
    """Codes (rows, levels) of one launch; ``rows``: a slice run alone, ``perm``: (row order, utterance order) of
    a batch with whole utterances moved.  ``utt``: the utterance records for either (RESP0 moved along)."""
    code = L.ABSORBING if tr == "absorbing" else L.UNIFORM
    hi, xt, ru, tu, ut = dv["head_in"], dv["x_t"], dv["row_utt"], dv["t_utt"], dv["utt"] if utt is None else utt
    if rows is not None:
        hi, xt, ru = hi[rows], xt[rows], ru[rows]
    if perm is not None:
        order, uorder = perm
        hi, xt, tu = hi[order], xt[order], tu[uorder]
        inv = torch.empty_like(uorder)
        inv[uorder] = torch.arange(uorder.numel(), device=DEV)
        ru = inv[ru[order].long()].int()
    out = torch.full((hi.shape[0], c.n_levels), -1, dtype=torch.int32, device=DEV)
    L.head_posterior_sample(out, None, hi.contiguous(), dv["W"], dv["bias"], xt.contiguous(), ru.contiguous(),
                            tu.contiguous(), ut.contiguous(), table, c.n_levels, c.K, code, noise, seed=seed)
    return out


def _permuted(L, c):
    """Utterances in reverse order: (row order, utterance order, utt records with their new RESP0)."""
    B = len(c.lens)
    starts = c.utt[:, L.U_RESP0].long()
    uorder = torch.arange(B - 1, -1, -1)
    order = torch.cat([torch.arange(int(starts[b]), int(starts[b]) + c.lens[b]) for b in uorder.tolist()])
    new_utt = c.utt[uorder].clone()
    new_lens = torch.tensor([c.lens[b] for b in uorder.tolist()])
    new_utt[:, L.U_RESP0] = torch.cat([torch.zeros(1, dtype=torch.long), new_lens.cumsum(0)[:-1]]).int()
    inv_rows = torch.empty_like(order)
    inv_rows[order] = torch.arange(order.numel())
    return order.to(DEV), uorder.to(DEV), new_utt.to(DEV), inv_rows.to(DEV)


def _items_per_pair(c, sms):
    return c.items / min(c.items, sms // 2)


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
@pytest.mark.parametrize("K,d,n_levels,dtype,rows_mod,seed", hb.CASES,
                         ids=[f"K{k}-d{d}-l{n}-{str(t)[6:]}-r{r}" for k, d, n, t, r, _ in hb.CASES])
def test_head_greedy_codes_and_launch_shape_invariance(L, sms, K, d, n_levels, dtype, rows_mod, seed, tr):
    c = hb.Case(K, d, n_levels, dtype, sms, seed, rows_mod)
    ipp = _items_per_pair(c, sms)
    assert ipp >= 3, (c.ctx(), ipp)
    assert L.head_fused(d, K, L.NOISE_GREEDY) and L.head_fused(d, K, L.NOISE_PHILOX)
    dv = _on_dev(c)
    table = _table(K, tr).to(DEV)
    # planted ties: the GEMM with fp32 output must give bit-equal logits for the duplicated columns
    lg = torch.empty(c.rows, n_levels * K, dtype=torch.float32, device=DEV)
    L.gemm_bf16(lg, dv["head_in"], dv["W"], dv["bias"], None, L.EPI_BIAS)
    for lv in range(n_levels):
        for j1, j2 in hb.tie_pairs(K):
            assert torch.equal(lg[:, lv * K + j1], lg[:, lv * K + j2]), (c.ctx(), lv, j1, j2)
    del lg
    got = _sample(L, c, dv, table, tr, L.NOISE_GREEDY)
    t_rows = c.t_rows()
    n_clear = n_tied = n_tok = 0
    for lv, ref, bound in hb.level_references(dv["head_in"], dv["W"], dv["bias"], n_levels, K):
        exp, clear, tied = hb.greedy_reference(ref, bound, table.double(), t_rows, c.x_t[:, lv], tr)
        hb.check_greedy(got[:, lv], exp, clear, f"{c.ctx()} {tr} level {lv}")
        n_clear += int(clear.sum())
        n_tied += int((clear & tied).sum())
        n_tok += clear.numel()
        del ref, bound
    assert n_tied > 0, f"{c.ctx()}: no planted tie was decided"
    # launch-shape invariance, greedy and Philox: one 256-row block alone (the last, ragged one and one from the
    # middle), and the batch with its utterances in reverse order
    order, uorder, new_utt, inv_rows = _permuted(L, c)
    num_m = -(-c.rows // hb.TILE)
    for noise, seed_ in ((L.NOISE_GREEDY, 0), (L.NOISE_PHILOX, 77 + seed)):
        full = got if noise == L.NOISE_GREEDY else _sample(L, c, dv, table, tr, noise, seed_)
        for m_blk in (num_m - 1, num_m // 2):
            r0 = m_blk * hb.TILE
            rows = slice(r0, min(r0 + hb.TILE, c.rows))
            utt = dv["utt"].clone()
            utt[:, L.U_RESP0] -= r0
            alone = _sample(L, c, dv, table, tr, noise, seed_, rows=rows, utt=utt)
            assert torch.equal(alone, full[rows]), (c.ctx(), tr, noise, m_blk)
        perm = _sample(L, c, dv, table, tr, noise, seed_, utt=new_utt, perm=(order, uorder))
        assert torch.equal(perm[inv_rows], full), (c.ctx(), tr, noise, "permuted utterances")
    print(f"\n{c.ctx()} {tr}: {ipp:.2f} items per CTA pair, {n_clear / n_tok:.3f} of tokens clear, "
          f"{n_tied} planted ties decided")


@pytest.mark.parametrize("K,d,n_levels,dtype,rows_mod,seed", hb.CASES,
                         ids=[f"K{k}-d{d}-l{n}-{str(t)[6:]}-r{r}" for k, d, n, t, r, _ in hb.CASES])
def test_head_ce_loss_within_bound(L, sms, K, d, n_levels, dtype, rows_mod, seed):
    c = hb.Case(K, d, n_levels, dtype, sms, seed, rows_mod)
    ipp = _items_per_pair(c, sms)
    assert ipp >= 3, (c.ctx(), ipp)
    dv = _on_dev(c)
    lg = (dv["head_in"].float() @ dv["W"].float().t() + dv["bias"]).view(c.rows, n_levels, K)
    tgt = c.targets(lg)
    del lg
    loss = torch.full((c.rows, n_levels), float("nan"), device=DEV)
    L.head_ce_loss(loss, dv["head_in"], dv["W"], dv["bias"], tgt.to(DEV), n_levels, K)
    ratio = calib = 0.0
    for lv, ref, bound in hb.level_references(dv["head_in"], dv["W"], dv["bias"], n_levels, K):
        r, rest, unit = hb.ce_reference(ref, bound, tgt[:, lv])
        rep = eb.within(loss[:, lv], r, rest, unit, hb.C_CE, f"{c.ctx()} CE level {lv}")
        ratio, calib = max(ratio, rep.bound_ratio), max(calib, rep.calib_ratio)
        del ref, bound
    print(f"\n{c.ctx()} CE: {ipp:.2f} items per CTA pair, err/bound {ratio:.3g}, (err-rest)/unit {calib:.3g}")


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_head_philox_law_pit(L, sms, tr):
    """>= 200 k distinct tokens at t > 0, pooled over launches of >= 6 work items per CTA pair."""
    us = []
    for K, d, n_levels, dtype, rows_mod, seed in hb.LAW_CASES:
        c = hb.Case(K, d, n_levels, dtype, sms, seed, rows_mod, items_per_pair=hb.LAW_ITEMS_PER_PAIR)
        assert _items_per_pair(c, sms) >= hb.LAW_ITEMS_PER_PAIR
        dv = _on_dev(c)
        table = _table(K, tr).to(DEV)
        got = _sample(L, c, dv, table, tr, L.NOISE_PHILOX, seed=seed)
        t_rows = c.t_rows()
        live = t_rows > 0
        g = torch.Generator().manual_seed(seed)
        v = torch.rand(c.rows, n_levels, generator=g, dtype=torch.float64)
        for lv, ref, _ in hb.level_references(dv["head_in"], dv["W"], dv["bias"], n_levels, K):
            prob = hb.law(ref[live.to(DEV)], table.double(), t_rows[live], c.x_t[live, lv], tr)
            us.append(hb.pit(prob, got[live.to(DEV), lv], v[live, lv]).cpu().numpy())
            del prob, ref
    u = np.concatenate(us)
    assert u.size >= 200_000, u.size
    D = hb.check_law(u, tr)
    print(f"\n{tr}: KS D = {D:.4g} over {u.size} tokens (bound {1.95 / np.sqrt(u.size):.4g})")
