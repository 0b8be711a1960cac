"""The fused head's checks (tests/head_bounds.py) have teeth (CPU only, no GPU needed).

A numpy emulation of head_sample_kernel's streaming epilogue (256-column tiles split into two 128-column halves
and 32-class chunks, fp32 online max and Z, e_x / m_x and e_m / m_m, the merge of the two halves, the greedy
pick, the reservoir draw and the cross-entropy) walks the work items of the GPU tests' launches in the order a
148-SM B200 runs them.  It must pass every check, with the calibrated constants halved; each planted defect below
must be rejected at the GPU tests' shapes and token counts."""
import functools

import numpy as np
import pytest
import torch

import error_bounds as eb
import head_bounds as hb

SMS = 148               # B200: the GPU tests take the SM count from the device
F32 = np.float32
L2E = F32(1.4426950408889634)
EPS32 = F32(hb.EPS)


class _Half:
    """HsState of one thread: one accumulator row, one half of every tile's columns."""

    def __init__(self, N):
        self.m = np.full(N, -np.inf, F32)
        self.Z, self.e_x, self.m_x, self.e_m, self.m_m = (np.zeros(N, F32) for _ in range(5))
        self.best = np.full(N, -np.inf, F32)
        self.best_j = np.full(N, 0x7FFFFFFF, np.int64)
        self.win_col = np.zeros(N, np.int64)
        self.win = np.zeros((N, 32), F32)

    def take(self, n):
        h = _Half(0)
        for k, v in vars(self).items():
            setattr(h, k, v[:n].copy())
        return h


def _stream(st, X, xt, h, tpl, mode, m_abs, rng, defect):
    N = X.shape[0]
    ar = np.arange(N)
    for q in range(tpl - 1 if defect == "last_tile_dropped" else tpl):
        for c in range(4):
            col0 = q * hb.TILE + h * hb.HALF + c * 32
            v = X[:, col0:col0 + 32]
            cmax = v.max(1)
            up = cmax > st.best
            st.best_j = np.where(up, col0 + v.argmax(1), st.best_j)
            st.best = np.where(up, cmax, st.best)
            dxt = xt - col0
            inx = (dxt >= 0) & (dxt < 32)
            dxc = np.clip(dxt, 0, 31)
            if mode == "ce":
                st.e_x = np.where(inx, v[ar, dxc], st.e_x)
            m_new = np.maximum(st.m, cmax)
            if not (defect == "ce_no_max_rescale"):
                st.Z = st.Z * np.exp2((st.m - m_new) * L2E)
            st.m = m_new
            e = np.exp2(v * L2E + (-m_new * L2E)[:, None])
            s_c = e.sum(1, dtype=F32)
            st.Z = st.Z + s_c
            if mode != "ce":
                st.e_x = np.where(inx, e[ar, dxc], st.e_x)
                st.m_x = np.where(inx, m_new, st.m_x)
                if col0 == (m_abs & ~31):
                    st.e_m, st.m_m = e[:, 0].copy(), m_new
            if mode == "philox":
                take = rng.random(N, dtype=F32) * st.Z < s_c
                st.win_col = np.where(take, col0, st.win_col)
                st.win = np.where(take[:, None], e, st.win)
    if mode != "philox":
        return st.best_j
    target = rng.random(N, dtype=F32) * st.win.sum(1, dtype=F32)
    return st.win_col + (target[:, None] >= np.cumsum(st.win[:, :31], 1, dtype=F32)).sum(1)


def _finish(a, b, ca, cb, xt, t, tab, K, tr, mode, rng, defect):
    """The merge of the two halves and the reverse step (post_scalars, post_special, post_greedy), in fp32."""
    from vall_e.b200 import lib as L
    N = xt.shape[0]
    m_f = np.maximum(a.m, b.m)
    Za, Zb = a.Z * np.exp2((a.m - m_f) * L2E), b.Z * np.exp2((b.m - m_f) * L2E)
    Z = Za + Zb
    invZ = F32(1) / Z
    half1 = F32(0) if defect == "half1_special_ignored" else F32(1)
    if mode == "ce":
        return m_f + np.log(Z) - (a.e_x + half1 * b.e_x)

    def rescaled(e_a, m_a, e_b, m_b):
        if defect == "ex_rescaled_by_mf":
            return e_a + half1 * e_b
        return e_a * np.exp2((m_a - m_f) * L2E) + half1 * e_b * np.exp2((m_b - m_f) * L2E)

    e_x = rescaled(a.e_x, a.m_x, b.e_x, b.m_x)
    e_m = rescaled(a.e_m, a.m_m, b.e_m, b.m_m)
    j1 = b.best_j
    up = (b.best > a.best) | ((b.best == a.best) & (j1 < a.best_j))
    best, best_j = np.where(up, b.best, a.best), np.where(up, j1, a.best_j)
    absorbing = tr == "absorbing"
    m = K // 2 if absorbing else -1
    one, cum = tab[t], tab[np.maximum(t - 1, 0)]
    at_m = (xt == m) if absorbing else np.zeros(N, bool)
    has_m = absorbing & ~at_m
    f1_self = np.where(at_m, one[:, L.TAB_ONE_BOTH], one[:, L.TAB_ONE_KEEP]) + EPS32
    f1_oth = np.where(at_m, one[:, L.TAB_ONE_ABSORB], one[:, L.TAB_ONE_OFF]) + EPS32
    a_gen, c_gen = cum[:, L.TAB_CUM_KEEP], cum[:, L.TAB_CUM_OFF]
    a_m = cum[:, L.TAB_CUM_BOTH] if absorbing else a_gen
    c_m = cum[:, L.TAB_CUM_ABSORB] if absorbing else c_gen
    cA, cst = (a_gen - c_gen) * f1_oth, (c_gen + EPS32) * f1_oth
    coef = cA * invZ
    w_x = f1_self * (e_x * invZ * np.where(at_m, a_m - c_m, a_gen - c_gen) + np.where(at_m, c_m, c_gen) + EPS32)
    dx = np.maximum(w_x - (e_x * coef + cst), F32(0))
    w_m = np.where(has_m, f1_oth * (e_m * invZ * (a_m - c_m) + c_m + EPS32), F32(0))
    dm = np.where(has_m, np.maximum(w_m - (e_m * coef + cst), F32(0)), F32(0))
    if mode == "greedy":
        top_w = np.exp2((best - m_f) * L2E) * coef + cst
        best_w = np.where(best_j == xt, w_x, np.where(best_j == m, w_m, top_w))
        pick = best_j
        up = (w_x > best_w) | ((w_x == best_w) & (xt < pick))
        best_w, pick = np.where(up, w_x, best_w), np.where(up, xt, pick)
        pick = np.where(has_m & ((w_m > best_w) | ((w_m == best_w) & (m < pick))), m, pick)
    else:
        w_uni = F32(K) * cst
        u = rng.random((4, N), dtype=F32)
        target = u[0] * (cA + w_uni + dx + dm)
        uni = np.minimum((u[1] * F32(K)).astype(np.int64), K - 1)
        soft = np.where(u[2] * Z < Zb, cb, ca)
        pick = np.where(target < dx, xt, np.where(target < dx + dm, m, np.where(target < dx + dm + w_uni, uni, soft)))
    return np.where(t == 0, best_j, pick)


def kernel_logits(c, defect=None):
    """fp32 logits (rows, levels, K) as the kernel forms them: 16-bit products accumulated in fp32, plus the bias."""
    A, bias = c.head_in.float(), c.bias
    if defect == "partial_kblock_dropped":
        A = A.clone()
        A[:, (c.d // 64) * 64:] = 0
    if defect == "bias_wrong_level":
        bias = bias.view(c.n_levels, c.K).roll(1, 0).reshape(-1)
    return (A @ c.W.float().t() + bias).view(c.rows, c.n_levels, c.K).numpy()


def emulate(c, tr, mode, targets=None, defect=None, seed=0):
    """Codes (greedy / philox) or losses (ce), (rows, levels), over the work items in launch order."""
    K, nl, G = c.K, c.n_levels, SMS // 2
    tpl = K // hb.TILE
    lg = kernel_logits(c, defect)
    num_m = -(-c.rows // hb.TILE)
    pad = num_m * hb.TILE
    X_all = np.empty((pad, nl, K), F32)
    X_all[:c.rows] = lg
    X_all[c.rows:] = c.bias.view(nl, K).numpy()       # rows past the end: zero-filled A, logits = bias
    xt_all = np.zeros((pad, nl), np.int64)
    xt_all[:c.rows] = (targets if mode == "ce" else c.x_t).numpy()
    t_all = np.ones(pad, np.int64)
    t_all[:c.rows] = c.t_rows().numpy()
    tab = None
    if mode != "ce":
        from vall_e.vall_e import d3pm as pd
        tab = pd.scalar_table(c.S, K, tr).numpy()
    m_abs = K // 2 if (tr == "absorbing" and mode != "ce") else -1
    rng = np.random.default_rng(seed)
    out = np.zeros((pad, nl), F32 if mode == "ce" else np.int64)
    carried = None
    items = num_m * nl
    for i0 in range(0, items, G):                       # one round: each CTA pair's next work item
        its = np.arange(i0, min(i0 + G, items))
        rows = (its[:, None] // nl * hb.TILE + np.arange(hb.TILE)).ravel()
        lev = np.repeat(its % nl, hb.TILE)
        X, xt, t = X_all[rows, lev], xt_all[rows, lev], t_all[rows]
        N = rows.size
        if defect == "state_not_reset" and carried is not None:
            halves = [carried[0].take(N), carried[1].take(N)]
        else:
            halves = [_Half(N), _Half(N)]
        cands = [_stream(halves[h], X, xt, h, tpl, mode, m_abs, rng, defect) for h in (0, 1)]
        carried = halves
        res = _finish(halves[0], halves[1], cands[0], cands[1], xt, t, tab, K, tr, mode, rng, defect)
        out[rows, lev] = res
    return torch.from_numpy(out[:c.rows])


# ---------------------------------------------------------------- the checks, as the GPU tests apply them
def greedy_check(c, tr, codes, c_acc=eb.C_ACC):
    from vall_e.vall_e import d3pm as pd
    tab = pd.scalar_table(c.S, c.K, tr).double()
    for lv, ref, bound in hb.level_references(c.head_in, c.W, c.bias, c.n_levels, c.K, c_acc):
        exp, clear, _ = hb.greedy_reference(ref, bound, tab, c.t_rows(), c.x_t[:, lv], tr)
        hb.check_greedy(codes[:, lv], exp, clear, f"{c.ctx()} {tr} level {lv}")


def ce_check(c, targets, loss, c_acc=eb.C_ACC, c_ce=hb.C_CE):
    for lv, ref, bound in hb.level_references(c.head_in, c.W, c.bias, c.n_levels, c.K, c_acc):
        r, rest, unit = hb.ce_reference(ref, bound, targets[:, lv])
        eb.within(loss[:, lv], r, rest, unit, c_ce, f"{c.ctx()} CE level {lv}")


@functools.lru_cache(maxsize=None)
def case(i, items_per_pair=3):
    K, d, nl, dt, rows_mod, seed = (hb.CASES + hb.LAW_CASES)[i]
    return hb.Case(K, d, nl, dt, SMS, seed, rows_mod, items_per_pair)


def ce_targets(c):
    return c.targets(torch.from_numpy(kernel_logits(c)))


# CASES: 1 = K 256 d 200 3 levels, 3 = K 768 d 72 3 levels, 4 = K 768 d 200 8 levels, 6 = K 1024 d 72 8 levels
FAITHFUL = [1, 3, 4, 6]


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
@pytest.mark.parametrize("i", FAITHFUL)
def test_emulated_greedy_passes_with_halved_constants(i, tr):
    c = case(i)
    greedy_check(c, tr, emulate(c, tr, "greedy"), eb.C_ACC / 2)


@pytest.mark.parametrize("i", FAITHFUL)
def test_emulated_ce_passes_with_halved_constants(i):
    c = case(i)
    tgt = ce_targets(c)
    ce_check(c, tgt, emulate(c, None, "ce", tgt), eb.C_ACC / 2, hb.C_CE / 2)


# (defect, case index, transition or "ce"): each must be rejected by the greedy or the cross-entropy check
DEFECTS = [
    ("state_not_reset", 1, "absorbing"), ("state_not_reset", 3, "uniform"), ("state_not_reset", 4, "ce"),
    ("last_tile_dropped", 3, "absorbing"), ("last_tile_dropped", 6, "ce"),
    ("partial_kblock_dropped", 3, "uniform"), ("partial_kblock_dropped", 1, "ce"),
    ("ex_rescaled_by_mf", 3, "absorbing"), ("ex_rescaled_by_mf", 4, "absorbing"),
    ("half1_special_ignored", 3, "absorbing"), ("half1_special_ignored", 4, "ce"),
    ("bias_wrong_level", 1, "uniform"), ("bias_wrong_level", 4, "ce"),
    ("ce_no_max_rescale", 3, "ce"), ("ce_no_max_rescale", 6, "ce"),
]


@pytest.mark.parametrize("defect,i,tr", DEFECTS, ids=[f"{d}-{i}-{t}" for d, i, t in DEFECTS])
def test_planted_defect_is_rejected(defect, i, tr):
    c = case(i)
    if tr == "ce":
        tgt = ce_targets(c)
        loss = emulate(c, None, "ce", tgt, defect)
        with pytest.raises(AssertionError, match="outside the bound"):
            ce_check(c, tgt, loss)
    else:
        codes = emulate(c, tr, "greedy", defect=defect)
        with pytest.raises(AssertionError, match="greedy codes differ"):
            greedy_check(c, tr, codes)


# ---------------------------------------------------------------- the Philox law
def _inverse_cdf(prob, g):
    u = torch.rand(prob.shape[0], 1, generator=g, dtype=torch.float64)
    return torch.searchsorted(prob.cumsum(-1), u)[:, 0].clamp(max=prob.shape[1] - 1)


def pooled_pit(tr, source):
    """PIT values of the GPU law test's tokens (t > 0), drawn by the emulated reservoir sampler ("kernel"), from
    softmax(logits) or from the neighbouring token's law."""
    from vall_e.vall_e import d3pm as pd
    us = []
    for j, (K, _, nl, _, _, seed) in enumerate(hb.LAW_CASES):
        c = case(len(hb.CASES) + j, hb.LAW_ITEMS_PER_PAIR)
        tab = pd.scalar_table(c.S, K, tr).double()
        t_rows = c.t_rows()
        live = t_rows > 0
        codes = emulate(c, tr, "philox", seed=seed) if source == "kernel" else None
        v = torch.rand(c.rows, nl, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
        g = torch.Generator().manual_seed(seed + 1)
        for lv, ref, _ in hb.level_references(c.head_in, c.W, c.bias, nl, K):
            prob = hb.law(ref[live], tab, t_rows[live], c.x_t[live, lv], tr)
            if source == "kernel":
                drawn = codes[live, lv]
            elif source == "softmax":
                drawn = _inverse_cdf(torch.softmax(ref[live], -1), g)
            else:
                drawn = _inverse_cdf(prob.roll(1, 0), g)
            us.append(hb.pit(prob, drawn, v[live, lv]).numpy())
    return np.concatenate(us)


@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_emulated_reservoir_draws_pass_the_law_test(tr):
    u = pooled_pit(tr, "kernel")
    assert u.size >= 200_000
    hb.check_law(u, tr)


@pytest.mark.parametrize("source", ["softmax", "neighbour"])
@pytest.mark.parametrize("tr", ["absorbing", "uniform"])
def test_law_test_rejects_draws_from_the_wrong_law(tr, source):
    with pytest.raises(AssertionError, match="KS statistic"):
        hb.check_law(pooled_pit(tr, source), f"{tr} {source}")
