"""SGD epoch kernels held update by update to a float64 first-order restatement.

For a small learning rate one epoch equals the sum of the per-sample updates, each taken at the epoch-start values: what the
order of the updates, the samples in flight and the flush periods of item-run tiles change is second order.  That makes one
restatement cover every kernel variant (sgd_rating_epoch_kernel atomic / TRACK / Hogwild, general path and run tiles, the
BPR, RankSGD and GBPR kernels), with tolerances derived from the inputs rather than fitted:

- second order: a sample's step is a product of at most three of the values it reads (error or logistic derivative, a row, a
  regulariser).  While the epoch runs, every row it reads has moved by at most KAPPA times its first-order path length
  (the sum of |step| of the OTHER samples on that row); the change of the step follows from the product rule, component by
  component: e.g. |d(e p_k)| <= |de| |p_k| + (|e| + |de|) |dp|.
- fp32 rounding: the device rounds every reduction into a row to half an ulp (one ulp is allowed per RED), and every
  computed step carries a relative error of (k + 40) eps: a k-term dot product, up to 32 ratings summed in registers and
  a 5-level shuffle tree.

Every comparison prints its largest error / budget ratio.  The CPU tests pin the restatement to the oracle and show that
references with a known mistake (no reg_i, no reg_b, the q_j step of the wrong sign, the damping of the item step, rho = 1)
fail the same comparison, so the budgets are small enough to tell right from wrong."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

EPS32 = float(np.finfo(np.float32).eps)
KAPPA = 2.0              # a row's path length under the real dynamics exceeds its first-order path length by a second-order share (<< 1)
K_LAYOUTS = (3, 8, 16, 20, 64, 128, 200)       # G = 1, 2, 4, 8, 16, 32 and 32 x 2 (layout_for_k, lrk_api.cu)
RUN_DEGREES = (224, 704, 2048)                 # run-tile items: 8-rating, 16-rating and whole-tile flush periods
RUN_MIN_DEGREE, HOT_FLUSH_DEG = 128, 512       # staging.cuh, sgd_probes


def f32(a):
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def ulp32(a):
    return np.spacing(np.abs(np.asarray(a, np.float64)).astype(np.float32)).astype(np.float64)


def layout(k):
    """(G, V) of layout_for_k"""
    ld = 4
    while ld < k and ld < 128:
        ld <<= 1
    if k > 128:
        ld = (k + 127) // 128 * 128
    return (ld // 4, 1) if ld <= 128 else (32, ld // 128)


def norm(a):
    return np.linalg.norm(a, axis=-1)


def logistic(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


# ------------------------------------------------------------------------------------------------------------------------------
# the reference
# ------------------------------------------------------------------------------------------------------------------------------
class Epoch:
    """first-order epoch: `slots` = [(array, rows, steps, visible-displacement bound, rounding bound)], `loss` at the start values"""

    def __init__(self, shapes):
        self.shapes, self.slots, self.loss, self.loss_budget = shapes, [], 0.0, 0.0

    def add(self, name, rows, step, second=None, rnd=None):
        self.slots.append((name, rows, step, second, rnd))

    def delta(self):
        out = {n: np.zeros(s) for n, s in self.shapes.items()}
        for name, rows, step, _, _ in self.slots:
            np.add.at(out[name], rows, step)
        return out

    def path(self):
        """per row: sum of |step| (norm over the row) and the elementwise sum of |step|, and the number of updates"""
        ln, el, cnt = {}, {}, {}
        for n, s in self.shapes.items():
            ln[n] = np.zeros(s[0]); el[n] = np.zeros(s); cnt[n] = np.zeros(s[0])
        for name, rows, step, _, _ in self.slots:
            np.add.at(ln[name], rows, np.abs(step) if step.ndim == 1 else norm(step))
            np.add.at(el[name], rows, np.abs(step))
            np.add.at(cnt[name], rows, 1.0)
        return ln, el, cnt


def _visible(ln, rows, step):
    """displacement of a row that a sample can see: KAPPA x the path length of the other samples on it"""
    own = np.abs(step) if step.ndim == 1 else norm(step)
    return KAPPA * np.maximum(ln[rows] - own, 0.0)


def first_order_epoch(model, S, P, Q, bu=None, bi=None, mu=0.0, lr=0.0, reg_u=0.0, reg_i=0.0, reg_b=0.0, rho=1.5, damp=None,
                      perturb=(), ln=None):
    """Sum of the per-sample updates at the initial values, and the loss at the initial values (float64).

    BiasedMF BiasedMFRecommender.java:72-98, PMF PMFSimilarityRecommender.java:64-82, BPR BPRRecommender.java:54-93, RankSGD
    RankSGDRecommender.java:94-105, GBPR GBPRRecommender.java:127-168.  S: samples {u, i, r} (rating models, RankSGD also j) or
    {u, i, j} (BPR) or {u, i, j, grp} (GBPR, grp padded with -1); u = -1 or j = -1 is a skipped sample.  damp[i] scales the
    item-side steps (staleness-aware step of the kernels).  perturb: deliberate mistakes (no_reg_i, no_reg_b, flip_qj, damp1,
    rho1) for the tests that prove the budgets tight.  ln: first-order path lengths of the unperturbed epoch; when given, each
    slot also carries its second-order and rounding bounds (see the module docstring)."""
    k = P.shape[1]
    shapes = {"P": P.shape, "Q": Q.shape}
    if bu is not None:
        shapes["bu"] = bu.shape
    if bi is not None:
        shapes["bi"] = bi.shape
    E = Epoch(shapes)
    ri = 0.0 if "no_reg_i" in perturb else reg_i
    rb = 0.0 if "no_reg_b" in perturb else reg_b
    sgn_j = -1.0 if "flip_qj" in perturb else 1.0
    if "rho1" in perturb:
        rho = 1.0
    if damp is None or "damp1" in perturb:
        damp = np.ones(Q.shape[0])
    fp = EPS32 * (k + 40)
    A = np.abs
    u, i = S["u"], S["i"]
    ok = u >= 0
    if "j" in S:
        ok &= S["j"] >= 0
    u, i = u[ok], i[ok]
    p, qi = P[u], Q[i]
    if model in ("biasedmf", "pmf"):
        r = S["r"][ok]
        biased = model == "biasedmf"
        b = (bu[u] + bi[i] + mu) if biased else 0.0
        e = r - np.einsum("nk,nk->n", p, qi) - b
        c = damp[i]
        sp = lr * (e[:, None] * qi - reg_u * p)
        sq = c[:, None] * lr * (e[:, None] * p - ri * qi)
        ell = e * e + reg_u * (p * p).sum(1) + reg_i * (qi * qi).sum(1)
        if biased:
            sbu, sbi = lr * (e - rb * bu[u]), c * lr * (e - rb * bi[i])
            ell = ell + reg_b * (bu[u] ** 2 + bi[i] ** 2)
        E.loss = 0.5 * ell.sum()
        if ln is None:
            E.add("P", u, sp); E.add("Q", i, sq)
            if biased:
                E.add("bu", u, sbu); E.add("bi", i, sbi)
            return E
        Dp, Dq = _visible(ln["P"], u, sp), _visible(ln["Q"], i, sq)
        Dbu = _visible(ln["bu"], u, sbu) if biased else 0.0
        Dbi = _visible(ln["bi"], i, sbi) if biased else 0.0
        np_, nq = norm(p), norm(qi)
        de = nq * Dp + np_ * Dq + Dp * Dq + Dbu + Dbi
        xabs = A(S["r"][ok]) + np.einsum("nk,nk->n", A(p), A(qi)) + ((A(bu[u]) + A(bi[i]) + abs(mu)) if biased else 0.0)
        E.add("P", u, sp, lr * (de[:, None] * A(qi) + ((A(e) + de) * Dq + reg_u * Dp)[:, None]), fp * lr * (xabs[:, None] * A(qi) + reg_u * A(p)))
        E.add("Q", i, sq, (c * lr)[:, None] * (de[:, None] * A(p) + ((A(e) + de) * Dp + reg_i * Dq)[:, None]), fp * lr * (xabs[:, None] * A(p) + reg_i * A(qi)))
        l2 = (2 * A(e) + de) * de + reg_u * (2 * np_ * Dp + Dp * Dp) + reg_i * (2 * nq * Dq + Dq * Dq)
        if biased:
            E.add("bu", u, sbu, lr * (de + reg_b * Dbu), fp * lr * (xabs + reg_b * A(bu[u])))
            E.add("bi", i, sbi, c * lr * (de + reg_b * Dbi), fp * lr * (xabs + reg_b * A(bi[i])))
            l2 = l2 + reg_b * (2 * A(bu[u]) * Dbu + Dbu ** 2 + 2 * A(bi[i]) * Dbi + Dbi ** 2)
        E.loss_budget = 0.5 * (l2.sum() + fp * (xabs ** 2 + reg_u * (p * p).sum(1) + reg_i * (qi * qi).sum(1)).sum())
        return E
    j = S["j"][ok]
    qj = Q[j]
    if model in ("bpr", "ranksgd"):
        d = qi - qj
        x = np.einsum("nk,nk->n", p, d)
        if model == "bpr":
            g = logistic(-x)                                 # deri
            sp = lr * (g[:, None] * d - reg_u * p)
            si = lr * (g[:, None] * p - ri * qi)
            sj = lr * (-sgn_j * g[:, None] * p - ri * qj)
            E.loss = (np.logaddexp(0.0, -x) + reg_u * (p * p).sum(1) + reg_i * ((qi * qi).sum(1) + (qj * qj).sum(1))).sum()
        else:
            r = S["r"][ok]
            g = -(x - r)                                     # -error: the steps read like BPR's with deri = -error
            sp = lr * g[:, None] * d
            si = damp[i][:, None] * lr * g[:, None] * p
            sj = -sgn_j * damp[j][:, None] * lr * g[:, None] * p
            E.loss = 0.5 * ((x - r) ** 2).sum()
        if ln is None:
            E.add("P", u, sp); E.add("Q", i, si); E.add("Q", j, sj)
            return E
        Dp, Di, Dj = _visible(ln["P"], u, sp), _visible(ln["Q"], i, si), _visible(ln["Q"], j, sj)
        np_, nd = norm(p), norm(d)
        dx = nd * Dp + np_ * (Di + Dj) + Dp * (Di + Dj)
        dg = dx / 4 if model == "bpr" else dx               # |d logistic| <= 1/4
        ru, rq = (reg_u, reg_i) if model == "bpr" else (0.0, 0.0)
        xabs = np.einsum("nk,nk->n", A(p), A(qi) + A(qj)) + (0.0 if model == "bpr" else A(S["r"][ok]))
        ga = A(g) + xabs
        E.add("P", u, sp, lr * (dg[:, None] * A(d) + ((A(g) + dg) * (Di + Dj) + ru * Dp)[:, None]), fp * lr * (ga[:, None] * (A(qi) + A(qj)) + ru * A(p)))
        E.add("Q", i, si, lr * (dg[:, None] * A(p) + ((A(g) + dg) * Dp + rq * Di)[:, None]), fp * lr * (ga[:, None] * A(p) + rq * A(qi)))
        E.add("Q", j, sj, lr * (dg[:, None] * A(p) + ((A(g) + dg) * Dp + rq * Dj)[:, None]), fp * lr * (ga[:, None] * A(p) + rq * A(qj)))
        if model == "bpr":
            l2 = dx + reg_u * (2 * np_ * Dp + Dp ** 2) + reg_i * (2 * norm(qi) * Di + Di ** 2 + 2 * norm(qj) * Dj + Dj ** 2)
        else:
            l2 = 0.5 * (2 * A(g) * dx + dx * dx)
        E.loss_budget = l2.sum() + fp * (xabs + xabs ** 2 + A(E.loss) / max(len(u), 1)).sum()
        return E
    # GBPR: the factor steps go into accumulators (every sample reads the epoch-start factors); the item biases move at once
    grp = S["grp"][ok]
    gm = grp >= 0
    gn = gm.sum(1).astype(np.float64)
    pg = np.where(gm[:, :, None], P[np.maximum(grp, 0)], 0.0)           # [n, g, k]
    sumg = pg.sum(1)
    omr = float(np.float32(1.0) - np.float32(rho))                       # (1 - rho) in float, as the reference and the kernel
    b_i, b_j = bi[i], bi[j]
    pos = rho * (np.einsum("nk,nk->n", sumg, qi) / gn + b_i) + omr * (b_i + np.einsum("nk,nk->n", p, qi))
    x = pos - (b_j + np.einsum("nk,nk->n", p, qj))
    g = logistic(-x)
    delta = (grp == u[:, None]) & gm
    dgrp = (rho / gn)[:, None, None] * qi[:, None, :] + delta[:, :, None] * (omr * qi - qj)[:, None, :]
    sP = lr * (g[:, None, None] * dgrp - reg_u * pg)
    si = lr * (g[:, None] * (rho / gn[:, None] * sumg + omr * p) - ri * qi)
    sj = lr * (-sgn_j * g[:, None] * p - ri * qj)
    sbi, sbj = lr * (g - rb * b_i), lr * (-g - rb * b_j)
    E.loss = (np.logaddexp(0.0, -x) + reg_u * (pg * pg).sum((1, 2)) + reg_i * ((qi * qi).sum(1) + (qj * qj).sum(1))
              + reg_b * (b_i ** 2 + b_j ** 2)).sum()
    gi, gs = grp[gm], sP[gm]
    if ln is None:
        E.add("P", gi, gs); E.add("Q", i, si); E.add("Q", j, sj); E.add("bi", i, sbi); E.add("bi", j, sbj)
        return E
    Dbi, Dbj = _visible(ln["bi"], i, sbi), _visible(ln["bi"], j, sbj)
    dx = (abs(rho) + abs(omr)) * Dbi + Dbj
    dg = dx / 4
    xabs = (abs(rho) * (np.einsum("nk,nk->n", A(sumg), A(qi)) / gn + A(b_i)) + abs(omr) * (A(b_i) + np.einsum("nk,nk->n", A(p), A(qi)))
            + A(b_j) + np.einsum("nk,nk->n", A(p), A(qj)))
    ga = g + xabs
    dgrp_abs = (abs(rho) / gn)[:, None, None] * A(qi)[:, None, :] + delta[:, :, None] * (abs(omr) * A(qi) + A(qj))[:, None, :]
    E.add("P", gi, gs, (lr * dg[:, None, None] * A(dgrp))[gm], (fp * lr * (ga[:, None, None] * dgrp_abs + reg_u * A(pg)))[gm])
    E.add("Q", i, si, lr * dg[:, None] * A(rho / gn[:, None] * sumg + omr * p),
          fp * lr * (ga[:, None] * (abs(rho) / gn[:, None] * A(pg).sum(1) + abs(omr) * A(p)) + reg_i * A(qi)))
    E.add("Q", j, sj, lr * dg[:, None] * A(p), fp * lr * (ga[:, None] * A(p) + reg_i * A(qj)))
    E.add("bi", i, sbi, lr * (dg + reg_b * Dbi), fp * lr * (ga + reg_b * A(b_i)))
    E.add("bi", j, sbj, lr * (dg + reg_b * Dbj), fp * lr * (ga + reg_b * A(b_j)))
    E.loss_budget = (dx + reg_b * (2 * A(b_i) * Dbi + Dbi ** 2 + 2 * A(b_j) * Dbj + Dbj ** 2)).sum() + fp * (xabs + A(np.logaddexp(0.0, -x))).sum()
    return E


def reference(model, S, start, **kw):
    """(delta dict, loss, budget dict, loss budget) of the unperturbed first-order epoch"""
    P, Q, bu, bi = start
    E0 = first_order_epoch(model, S, P, Q, bu, bi, **kw)
    ln, _, _ = E0.path()
    E = first_order_epoch(model, S, P, Q, bu, bi, ln=ln, **kw)
    return E0.delta(), E0.loss, E, E.loss_budget


def budget(E, start, n_red=None):
    """per element: second-order bound + fp32 rounding of the steps + one ulp per reduction into the row; n_red[name]
    overrides the number of reductions into a row (default: one per sample, the item-run tiles flush less often)"""
    vals = dict(zip(("P", "Q", "bu", "bi"), start))
    _, el, cnt = E.path()
    B = {n: np.zeros(s) for n, s in E.shapes.items()}
    for name, rows, step, second, rnd in E.slots:
        np.add.at(B[name], rows, second + rnd)
    for name in B:
        nr = cnt[name] if n_red is None or name not in n_red else n_red[name]
        if B[name].ndim == 2:
            nr = nr[:, None]
        B[name] += (nr + 1) * ulp32(A_(vals[name]) + el[name])
    return B


def A_(a):
    return np.abs(np.asarray(a, np.float64))


def ratio(tag, got, want, bud, rows=None):
    """largest |got - want| / budget over the arrays (optionally only `rows` of each)"""
    worst = 0.0
    for n in want:
        g, w, b = got[n], want[n], bud[n]
        if rows is not None and n in rows:
            g, w, b = g[rows[n]], w[rows[n]], b[rows[n]]
        if w.size:
            worst = max(worst, float((np.abs(g - w) / b).max()))
    print("%s: error / budget %.3g" % (tag, worst))
    return worst


def loss_ratio(tag, got, want, bud):
    x = abs(got - want) / bud
    print("%s: loss error / budget %.3g" % (tag, x))
    return x


# ------------------------------------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------------------------------------
def rating_data(k, seed, run_degrees=RUN_DEGREES, n_general=1001, max_general_deg=40, p_scale=0.1, q_scale=0.1, biased=True):
    """one rating per user; items 0.. have the run degrees (multiples of 32: no remainder goes to the general path), then items
    of degree 1..max_general_deg (n_general ratings, odd: the last tile of the stream is partial).  Every p_u is a positive
    multiple of one direction plus a little noise, so an item's delta is coherent, not a random walk; ratings 2..5 lie above
    every prediction (mu = 0.5), so every error has the same sign."""
    rng = np.random.default_rng(seed)
    degs = list(run_degrees)
    left = n_general
    while left > 0:
        d = int(min(left, rng.integers(1, max_general_deg + 1)))
        degs.append(d)
        left -= d
    I = len(degs) + 3                                          # three items nobody rated
    items = np.repeat(np.arange(len(degs), dtype=np.int32), degs)
    rng.shuffle(items)
    n = items.shape[0]
    vals = rng.integers(2, 6, n).astype(np.float64)
    d = rng.normal(size=k); d /= np.linalg.norm(d)
    P = f32(np.outer(rng.uniform(0.8, 1.2, n) * p_scale, d) + rng.normal(0, 0.02 * p_scale, (n, k)))
    Q = f32(rng.normal(0, q_scale, (I, k)))
    bu = f32(rng.normal(0, 0.1, n)) if biased else None
    bi = f32(rng.normal(0, 0.1, I)) if biased else None
    return n, I, items, vals, (P, Q, bu, bi)


def csr_one_per_user(O, n, I, items, vals):
    return O.Csr(n, I, np.arange(n + 1, dtype=np.int64), items, vals)


def random_csr(O, U, I, density, seed, values=(1.0, 2.0, 3.0, 4.0, 5.0), full_users=()):
    """random CSR; full_users: {user: number of items it has NOT rated}"""
    rng = np.random.default_rng(seed)
    mask = rng.random((U, I)) < density
    for x, missing in dict(full_users).items():
        mask[x] = True
        mask[x, rng.choice(I, missing, replace=False)] = False
    rows, cols = np.nonzero(mask)
    rowptr = np.zeros(U + 1, np.int64)
    np.add.at(rowptr, rows + 1, 1)
    return O.Csr(U, I, np.cumsum(rowptr), cols.astype(np.int32), rng.choice(np.asarray(values), rows.shape[0]))


def factors(U, I, k, seed, scale=0.1):
    rng = np.random.default_rng(seed)
    return f32(rng.normal(0, scale, (U, k))), f32(rng.normal(0, scale, (I, k)))


def rating_of(tr, u, i):
    """value of entry (u, i) of a CSR (the pairs exist)"""
    key = tr.rows().astype(np.int64) * tr.I + tr.col
    return tr.val[np.searchsorted(key, u.astype(np.int64) * tr.I + i)]


def run_flush_steps(G, deg, lr, pn2=1.0):
    """flush period (warp steps) of a run tile of an item with `deg` ratings (sgd_rating_body.inc:51-61)"""
    steps, hot, rps = G, max(G // 4, 1), 32 // G
    lrc = np.float32(lr) * np.float32(pn2)
    if deg >= HOT_FLUSH_DEG:
        if deg >= 2 * HOT_FLUSH_DEG and lrc * 32 <= 0.125:
            return steps
        if steps >= 2 * hot and lrc * (2 * hot * rps) <= 0.125:
            return 2 * hot
    return hot


def inflight_frac_range(G, n):
    """inflight_frac of sgd_grid: grid * 8 * max(rps, 8) / n for a grid of at least 1 and at most the staleness cap of
    sgd_grid (the cap binds below ~37 k * rps ratings; it is <= 1/4 whenever it is >= 1)"""
    rps = 32 // G
    grid_hi = max(1, (n // 16) // (8 * rps * 2))
    f = lambda grid: grid * 8.0 * max(rps, 8) / n
    return f(1), f(grid_hi)


def damp_of(x):
    x = np.asarray(x, np.float64)
    return np.where(x > 1e-3, -np.expm1(-x) / np.where(x > 0, x, 1.0), 1.0)


def rating_n_red(G, I, items, lr):
    """reductions into each item row: one per rating on the general path, one per flush period in a run tile"""
    deg = np.bincount(items, minlength=I)
    nr = deg.astype(np.float64)
    for it in np.flatnonzero(deg >= RUN_MIN_DEGREE):
        tiles = deg[it] // 32
        nr[it] = tiles * (G // run_flush_steps(G, deg[it], lr)) + deg[it] % 32
    return nr


# ------------------------------------------------------------------------------------------------------------------------------
# CPU: the restatement against the oracle, and deliberate mistakes that the budgets catch
# ------------------------------------------------------------------------------------------------------------------------------
RATING_HYPER = dict(lr=4e-7, reg_u=0.05, reg_i=0.5, reg_b=0.5)      # lr * 2048 * max(1, |p|^2) <= 1e-3


def _pin(tag, E_ok, got_delta, got_loss, start, bad, n_red=None):
    """the oracle's epoch is inside the budget of the restatement; every perturbed restatement is outside it"""
    want, loss, E, lb = E_ok
    bud = budget(E, start, n_red)
    assert ratio(tag, got_delta, want, bud) < 1.0
    assert loss_ratio(tag, got_loss, loss, lb) < 1.0
    for name, Eb in bad.items():
        r = ratio("%s [%s]" % (tag, name), got_delta, Eb.delta(), bud)
        assert r > 3.0, "the budget does not tell the reference without %s from the right one" % name


@pytest.mark.parametrize("model", ["biasedmf", "pmf"])
def test_rating_restatement_pins_the_oracle(O, model):
    k = 20
    n, I, items, vals, start = rating_data(k, 1, biased=model == "biasedmf")
    P, Q, bu, bi = start
    tr = csr_one_per_user(O, n, I, items, vals)
    S = {"u": np.arange(n), "i": items, "r": vals}
    mu = 0.5 if model == "biasedmf" else 0.0
    h = RATING_HYPER
    kw = dict(mu=mu, **h)
    ref = reference(model, S, start, **kw)
    oP, oQ = P.copy(), Q.copy()
    if model == "biasedmf":
        obu, obi = bu.copy(), bi.copy()
        ol = O.lib().lro_biasedmf_epoch(n, tr.rowptr, tr.col, tr.val, k, oP, oQ, obu, obi, mu, h["lr"], h["reg_u"], h["reg_i"], h["reg_b"], None, None)
        got = {"P": oP - P, "Q": oQ - Q, "bu": obu - bu, "bi": obi - bi}
    else:
        ol = O.lib().lro_pmf_epoch(n, tr.rowptr, tr.col, tr.val, k, oP, oQ, h["lr"], h["reg_u"], h["reg_i"], None, None)
        got = {"P": oP - P, "Q": oQ - Q}
    bad = {"no_reg_i": first_order_epoch(model, S, *start, perturb=("no_reg_i",), **kw)}
    if model == "biasedmf":
        bad["no_reg_b"] = first_order_epoch(model, S, *start, perturb=("no_reg_b",), **kw)
    # the budget of the device comparison: reductions into the item rows as the k = 20 layout issues them
    nr = rating_n_red(layout(k)[0], I, items, h["lr"])
    _pin(model, ref, got, ol, start, bad, {"Q": nr, "bi": nr})


def _bpr_samples(tr, n, seed):
    """uniform users with a non-full row, positives from the row, negatives outside it"""
    rng = np.random.default_rng(seed)
    deg = np.diff(tr.rowptr)
    users = np.flatnonzero((deg > 0) & (deg < tr.I))
    u = rng.choice(users, n)
    i = tr.col[tr.rowptr[u] + (rng.random(n) * deg[u]).astype(np.int64)]
    rated = np.zeros((tr.U, tr.I), bool); rated[tr.rows(), tr.col] = True
    j = rng.integers(0, tr.I, n)
    while rated[u, j].any():
        bad = rated[u, j]
        j[bad] = rng.integers(0, tr.I, int(bad.sum()))
    return u.astype(np.int32), i.astype(np.int32), j.astype(np.int32)


@pytest.mark.parametrize("model", ["bpr", "ranksgd"])
def test_sampled_restatement_pins_the_oracle(O, model):
    k = 16
    tr = random_csr(O, 500, 400, 0.02, 3)
    P, Q = factors(tr.U, tr.I, k, 4)
    n = tr.nnz
    u, i, j = _bpr_samples(tr, n, 5)
    trip = np.ascontiguousarray(np.stack([u, i, j], 1).reshape(-1))
    oP, oQ = P.copy(), Q.copy()
    if model == "bpr":
        kw = dict(lr=2e-5, reg_u=0.05, reg_i=0.5)
        S = {"u": u, "i": i, "j": j}
        ol = O.lib().lro_bpr_epoch(tr.U, tr.I, tr.rowptr, tr.col, k, oP, oQ, kw["lr"], kw["reg_u"], kw["reg_i"], n, trip.ctypes.data, None)
        bad = {"no_reg_i": first_order_epoch(model, S, P, Q, perturb=("no_reg_i",), **kw)}
    else:
        kw = dict(lr=3e-5)
        S = {"u": u, "i": i, "j": j, "r": rating_of(tr, u, i)}
        ol = O.lib().lro_ranksgd_epoch(tr.U, tr.I, tr.rowptr, tr.col, tr.val, k, oP, oQ, kw["lr"], n, trip.ctypes.data, None)
        bad = {}
    bad["flip_qj"] = first_order_epoch(model, S, P, Q, perturb=("flip_qj",), **kw)
    _pin(model, reference(model, S, (P, Q, None, None), **kw), {"P": oP - P, "Q": oQ - Q}, ol, (P, Q, None, None), bad)


GBPR_HYPER = dict(lr=1e-5, reg_u=0.05, reg_i=0.05, reg_b=0.5)


@pytest.mark.parametrize("glen,rho", [(1, 0.0), (3, 0.0), (3, 1.5), (8, 1.5)])
def test_gbpr_restatement_pins_the_oracle(O, glen, rho):
    k = 12
    tr = random_csr(O, 400, 300, 0.03, 6, values=(1.0,))
    P, Q = factors(tr.U, tr.I, k, 7)
    bi = np.zeros(tr.I)
    n = tr.nnz
    trip, grp = np.zeros(3 * n, np.int32), np.zeros(n * glen, np.int32)
    oP, oQ, ob = P.copy(), Q.copy(), bi.copy()
    O.lib().lro_seed(13)
    h = GBPR_HYPER
    ol = O.lib().lro_gbpr_epoch(tr.U, tr.I, tr.rowptr, tr.col, k, oP, oQ, ob, h["lr"], h["reg_u"], h["reg_i"], h["reg_b"], rho, glen,
                                trip.ctypes.data, grp.ctypes.data)
    trip = trip.reshape(n, 3)
    S = {"u": trip[:, 0], "i": trip[:, 1], "j": trip[:, 2], "grp": grp.reshape(n, glen)}
    start = (P, Q, None, bi)
    kw = dict(rho=rho, **h)
    # (no reg_b is invisible here: it multiplies the start biases, which are zero as in the device test)
    bad = {m: first_order_epoch("gbpr", S, *start, perturb=(m,), **kw) for m in ("no_reg_i", "flip_qj", "rho1")}
    if glen == 1:
        del bad["rho1"]          # a group of one is {u}: the group term equals the user's own, whatever rho
    _pin("gbpr g%d rho %.1f" % (glen, rho), reference("gbpr", S, start, **kw), {"P": oP - P, "Q": oQ - Q, "bi": ob - bi}, ol, start, bad)


def test_layout_and_damping_helpers_follow_the_kernels():
    assert [layout(k) for k in K_LAYOUTS] == [(1, 1), (2, 1), (4, 1), (8, 1), (16, 1), (32, 1), (32, 2)]
    lr = RATING_HYPER["lr"]
    # G >= 4: 8 ratings below 512, 16 from 512, the whole tile from 1024 (while lr * pn2 * 32 <= 1/8)
    for G in (4, 8, 16, 32):
        rps = 32 // G
        assert [run_flush_steps(G, d, lr) * rps for d in RUN_DEGREES] == [8, 16, 32]
        assert run_flush_steps(G, 2048, 0.006) * rps == 16 and run_flush_steps(G, 2048, 0.02) * rps == 8
    assert [run_flush_steps(2, d, lr) * 16 for d in RUN_DEGREES] == [16, 32, 32]
    assert [run_flush_steps(1, d, lr) * 32 for d in RUN_DEGREES] == [32, 32, 32]
    for G in (1, 2, 4, 8, 16, 32):
        lo, hi = inflight_frac_range(G, 40000)
        assert 0 < lo <= hi <= 0.25
    assert np.allclose(damp_of([0.0, 1e-4, 0.5]), [1.0, 1.0, (1 - np.exp(-0.5)) / 0.5])


# ------------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------------
def _rating_cases():
    out = []
    for model in ("biasedmf", "pmf"):
        for k in K_LAYOUTS:
            G, V = layout(k)
            for variant in ("track", "nontrack", "hogwild"):
                if variant == "nontrack" and G * V >= 32:
                    continue                                  # the k > 64 layouts always run TRACK (sgd_want_track)
                out.append((model, k, variant))
    return out


def _run_rating(capi, model, k, tr, start, mu, hyper, mode, lr0_epochs):
    P, Q, bu, bi = start
    h_model = capi.MODEL_BIASEDMF if model == "biasedmf" else capi.MODEL_PMF
    regs = (hyper["reg_u"], hyper["reg_i"], hyper["reg_b"])
    with capi.Handle(h_model, k, update_mode=mode) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, mu)
        for e in range(lr0_epochs):          # lr = 0 leaves every value as it is and advances epochs_done (the variant choice)
            h.sgd_epoch(0.0, *regs, e + 1)
        if lr0_epochs:
            g0 = h.get_factors()
            assert all(a is None or np.array_equal(a, b) for a, b in zip(g0, start))
        loss = h.sgd_epoch(hyper["lr"], *regs, lr0_epochs + 1)
        got = h.get_factors()
        st = h.stage_stats()
    return got, loss, st


@pytest.mark.gpu
@pytest.mark.parametrize("model,k,variant", _rating_cases())
def test_rating_epoch_is_first_order(O, capi, model, k, variant):
    """sgd_rating_epoch_kernel<G, V, BIASED, ATOMIC, TRACK> at a learning rate where one epoch is first order: the user side
    to fp32 rounding, the item rows and biases (general path, run tiles of all three flush periods) and the loss within the
    derived budget.  At this lr the staleness-aware damping is exactly 1 (x < 1e-3)."""
    biased = model == "biasedmf"
    G, V = layout(k)
    if variant == "hogwild":          # plain stores: only conflict-free data has a defined result
        n, I, items, vals, start = rating_data(k, 11, run_degrees=(), n_general=3001, max_general_deg=1, biased=biased)
        mode, pre = capi.UPDATE_HOGWILD, 0
    else:
        n, I, items, vals, start = rating_data(k, 11, biased=biased)
        mode, pre = capi.UPDATE_ATOMIC, (2 if variant == "nontrack" else 0)
    assert n % 32 != 0
    tr = csr_one_per_user(O, n, I, items, vals)
    mu = 0.5 if biased else 0.0
    assert (start[0] ** 2).sum(1).mean() <= 0.02              # mean |p_u|^2: non-TRACK after two epochs (sgd_want_track)
    got, loss, st = _run_rating(capi, model, k, tr, start, mu, RATING_HYPER, mode, pre)
    if variant != "hogwild":
        assert st["run_tile_ratings"] == sum(RUN_DEGREES) and st["max_item_degree"] == max(RUN_DEGREES)
    S = {"u": np.arange(n), "i": items, "r": vals}
    want, wloss, E, lb = reference(model, S, start, mu=mu, **RATING_HYPER)
    bud = budget(E, start, {"Q": rating_n_red(G, I, items, RATING_HYPER["lr"]), "bi": rating_n_red(G, I, items, RATING_HYPER["lr"])})
    gd = {n_: g - s for n_, g, s in zip(("P", "Q", "bu", "bi"), got, start) if s is not None}
    tag = "%s k=%d %s" % (model, k, variant)
    assert ratio(tag + " users", gd, {"P": want["P"]} | ({"bu": want["bu"]} if biased else {}), bud) < 1.0
    assert ratio(tag + " items", gd, {"Q": want["Q"]} | ({"bi": want["bi"]} if biased else {}), bud) < 1.0
    assert loss_ratio(tag, loss, wloss, lb) < 1.0
    unrated = np.setdiff1d(np.arange(I), items)
    assert np.array_equal(got[1][unrated], start[1][unrated])


@pytest.mark.gpu
@pytest.mark.parametrize("k,variant", [(k, v) for k in K_LAYOUTS for v in ("track", "nontrack") if v == "track" or np.prod(layout(k)) < 32])
def test_run_tile_item_step_is_damped_by_the_staleness_factor(O, capi, k, variant):
    """PMF at a learning rate where the damping of run tiles is visible: the item delta of every item is ONE scalar c_i times
    its first-order delta, c_i = (1 - e^-x) / x with x inside the range sgd_rating_body.inc:52-66 allows (inflight_frac
    between its value for a one-block grid and the staleness cap of sgd_grid), c_i clearly below 1 for run-tile items
    and 1 for items below the run threshold.  |p_u|^2 ~ 1e-4 keeps the item rows first order although lr * degree is up to
    6 (the damping uses max(1, |p|^2) = 1); reg_i = 0, whose contraction lr * degree * reg_i would otherwise act like a
    second damping.  The user rows are checked by the first-order test above."""
    G, V = layout(k)
    lr = 3e-3
    hyper = dict(lr=lr, reg_u=0.002, reg_i=0.0, reg_b=0.0)     # reg_i is a curvature of its own: held by the first-order test
    n, I, items, vals, start = rating_data(k, 21, n_general=1001, max_general_deg=100, p_scale=0.01, biased=False)
    tr = csr_one_per_user(O, n, I, items, vals)
    got, loss, st = _run_rating(capi, "pmf", k, tr, start, 0.0, hyper, capi.UPDATE_ATOMIC, 2 if variant == "nontrack" else 0)
    S = {"u": np.arange(n), "i": items, "r": vals}
    want, _, E, _ = reference("pmf", S, start, **hyper)
    bud = budget(E, start, {"Q": rating_n_red(G, I, items, lr)})["Q"]
    gQ = got[1] - start[1]
    deg = np.bincount(items, minlength=I)
    f_lo, f_hi = inflight_frac_range(G, n)
    hot, rps = max(G // 4, 1), 32 // G
    worst = 0.0
    for it in np.flatnonzero(deg > 0):
        w, g, b = want["Q"][it], gQ[it], bud[it]
        c = float(g @ w / (w @ w))
        res = float((np.abs(g - c * w) / b).max())
        tol = float(b @ np.abs(w) / (w @ w))                    # what the budget allows the fitted c to be off by
        if deg[it] >= RUN_MIN_DEGREE:
            fs = run_flush_steps(G, deg[it], lr)
            x_lo = lr * fs * rps
            x_hi = lr * max(deg[it] * f_hi * (fs / hot), fs * rps)
            c_lo, c_hi = float(damp_of(x_hi)), float(damp_of(x_lo))
            print("k=%d item deg %d: c %.5f in [%.5f, %.5f] +- %.1e, residual / budget %.3g" % (k, deg[it], c, c_lo, c_hi, tol, res))
            assert c_lo - tol <= c <= c_hi + tol
            assert 1.0 - c > 3 * tol, "the damping is not visible: an undamped item step would pass"
        else:
            assert abs(c - 1.0) <= tol, (it, deg[it], c, tol)
        worst = max(worst, res)
    print("k=%d %s: item residual / budget %.3g" % (k, variant, worst))
    assert worst < 1.0


@pytest.mark.gpu
def test_variant_selection_seen_by_the_trace():
    """LRK_SGD_TRACE=1 (read once per process, so in a child): the epochs the tests above call TRACK, non-TRACK and Hogwild run
    those variants, on a stream whose run tiles reach all three flush periods"""
    child = r"""
import sys
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import numpy as np
from oracle import oracle as O
from librec_b200 import capi
import test_gpu_sgd_first_order as T
for k, mode, pre in ((20, capi.UPDATE_ATOMIC, 2), (128, capi.UPDATE_ATOMIC, 2), (20, capi.UPDATE_HOGWILD, 0)):
    n, I, items, vals, start = T.rating_data(k, 11)
    tr = T.csr_one_per_user(O, n, I, items, vals)
    print("case k=%%d mode=%%d" %% (k, mode), file=sys.stderr, flush=True)
    _, _, st = T._run_rating(capi, "biasedmf", k, tr, start, 0.5, T.RATING_HYPER, mode, pre)
    print("stage max_deg=%%d run=%%d" %% (st["max_item_degree"], st["run_tile_ratings"]), file=sys.stderr, flush=True)
""" % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", child], env=dict(os.environ, LRK_SGD_TRACE="1"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    cases, cur = [], None
    for line in r.stderr.splitlines():
        if line.startswith("case "):
            cur = []
            cases.append((line, cur))
        m = re.match(r"\[sgd\] epoch (\d+) .* track (\d)", line)
        if m and cur is not None:
            cur.append(int(m.group(2)))
        m = re.match(r"stage max_deg=(\d+) run=(\d+)", line)
        if m:
            assert int(m.group(1)) >= 2 * HOT_FLUSH_DEG and int(m.group(2)) == sum(RUN_DEGREES)
    print(r.stderr[-2000:])
    assert [c[1] for c in cases] == [[1, 1, 0], [1, 1, 1], [0]], cases


@pytest.mark.gpu
@pytest.mark.parametrize("k", K_LAYOUTS)
@pytest.mark.parametrize("mode", ["atomic", "hogwild"])
def test_bpr_epoch_is_first_order(O, capi, k, mode):
    """sgd_bpr_epoch_kernel<G, V, ATOMIC> on its own samples (lrk_bpr_peek_samples).  User 0 rated every item (never drawn);
    user 1 rated all but one, so many of its draws give up (u = -1) and must change nothing.  Hogwild stores race when two
    samples in flight share a row: there only the rows that exactly one sample touches are compared."""
    tr = random_csr(O, 3000, 3000, 0.0007, 8, values=(1.0,), full_users={0: 0, 1: 1})
    P, Q = factors(tr.U, tr.I, k, 9)
    hyper = dict(lr=2e-5, reg_u=0.05, reg_i=0.5)
    with capi.Handle(capi.MODEL_BPR, k, update_mode=capi.UPDATE_ATOMIC if mode == "atomic" else capi.UPDATE_HOGWILD, seed=4) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        s = h.bpr_peek_samples(1, 0, tr.nnz)
        loss = h.sgd_epoch(hyper["lr"], hyper["reg_u"], hyper["reg_i"], 0.0, 1)
        gP, gQ, _, _ = h.get_factors()
    u = s[:, 0]
    assert (u == -1).sum() > 0 and not (u == 0).any()
    assert ((u[u >= 0] == 1).sum()) > 0
    S = {"u": u, "i": s[:, 1], "j": s[:, 2]}
    start = (P, Q, None, None)
    want, wloss, E, lb = reference("bpr", S, start, **hyper)
    bud = budget(E, start)
    got = {"P": gP - P, "Q": gQ - Q}
    rows = None
    if mode == "hogwild":
        _, _, cnt = E.path()
        rows = {"P": cnt["P"] <= 1, "Q": cnt["Q"] <= 1}
        assert rows["P"].sum() > 100
    assert ratio("bpr k=%d %s" % (k, mode), got, want, bud, rows) < 1.0
    assert np.array_equal(gP[0], P[0])
    if mode == "atomic":
        assert loss_ratio("bpr k=%d" % k, loss, wloss, lb) < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("k", K_LAYOUTS)
def test_ranksgd_epoch_is_first_order(O, capi, k):
    """sgd_ranksgd_epoch_kernel<G, V, true> on its own samples.  At this lr the item damping x = 2 lr |p|^2 inflight_frac deg
    stays below 1e-3, where the kernel applies none.  (Where it is visible the item rows are not first order: x grows with the
    same |p_u|^2 that is the curvature of the row, so the damping of RankSGD is left to the C1 runs of test_gpu_ranksgd.py.)"""
    tr = random_csr(O, 1500, 1000, 0.01, 10)
    P, Q = factors(tr.U, tr.I, k, 11, scale=min(0.1, 0.5 / np.sqrt(k)))      # |p|^2 <= ~0.25 at every k
    lr = 3e-5
    with capi.Handle(capi.MODEL_RANKSGD, k, seed=6) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        s = h.bpr_peek_samples(1, 0, tr.nnz)
        loss = h.sgd_epoch(lr, 0.0, 0.0, 0.0, 1)
        gP, gQ, _, _ = h.get_factors()
    deg = np.bincount(tr.col, minlength=tr.I)
    assert 2 * lr * (P ** 2).sum(1).max() * inflight_frac_range(layout(k)[0], tr.nnz)[1] * deg.max() < 1e-3
    ok = s[:, 2] >= 0
    S = {"u": s[:, 0], "i": s[:, 1], "j": s[:, 2], "r": np.where(ok, rating_of(tr, s[:, 0], s[:, 1]), 0.0)}
    start = (P, Q, None, None)
    want, wloss, E, lb = reference("ranksgd", S, start, lr=lr)
    got = {"P": gP - P, "Q": gQ - Q}
    assert ratio("ranksgd k=%d" % k, got, want, budget(E, start)) < 1.0
    assert loss_ratio("ranksgd k=%d" % k, loss, wloss, lb) < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("k,glen,rho", [(k, g, r) for k in (3, 20) for g in (1, 3, 8) for r in (0.0, 1.5)] + [(200, 8, 1.5)])
def test_gbpr_epoch_is_first_order(O, capi, k, glen, rho):
    """sgd_gbpr_epoch_kernel<G, V>: every sample reads the epoch-start factors, so P and Q equal the first-order sum up to the
    fp32 accumulation; the item biases start at zero and move by O(lr), so their Hogwild interplay stays second order"""
    tr = random_csr(O, 1500, 1000, 0.01, 12, values=(1.0,))
    P, Q = factors(tr.U, tr.I, k, 13)
    bi = np.zeros(tr.I)
    h_ = GBPR_HYPER
    with capi.Handle(capi.MODEL_GBPR, k, seed=7) as h:
        h.set_param("gbpr.rho", rho)
        h.set_param("gbpr.gsize", glen)
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, None, bi)
        s = h.bpr_peek_samples(1, 0, tr.nnz)
        loss = h.sgd_epoch(h_["lr"], h_["reg_u"], h_["reg_i"], h_["reg_b"], 1)
        gP, gQ, _, gbi = h.get_factors()
    S = {"u": s[:, 0], "i": s[:, 1], "j": s[:, 2], "grp": s[:, 3:]}
    assert (S["grp"] >= 0).sum(1).max() == glen
    start = (P, Q, None, bi)
    kw = dict(rho=rho, **h_)
    want, wloss, E, lb = reference("gbpr", S, start, **kw)
    bud = budget(E, start)
    tag = "gbpr k=%d g%d rho %.1f" % (k, glen, rho)
    got = {"P": gP - P, "Q": gQ - Q, "bi": gbi - bi}
    assert ratio(tag, got, want, bud) < 1.0
    assert loss_ratio(tag, loss, wloss, lb) < 1.0
    for m in ("flip_qj", "no_reg_i") + (("rho1",) if glen > 1 else ()):
        assert ratio(tag + " [%s]" % m, got, first_order_epoch("gbpr", S, *start, perturb=(m,), **kw).delta(), bud) > 3.0
