"""CPU: the oracle's GBPR restatement (SURVEY 8f N3 groundwork) against an independent pure-Python replay of
recommender/cf/ranking/GBPRRecommender.java: own java.util.Random, a literal java.util.HashSet for the user group."""
import math

import numpy as np

from conftest import rng_csr
from test_oracle_aobpr import JavaRandom
from test_oracle_pins import _py_topk
from test_oracle_ranking_eval import JavaHashSet


def gbpr_replay(seed, U, I, rowptr, col, k, P, Q, bi, lr, reg_u, reg_i, reg_b, rho, g_len):
    rng = JavaRandom(seed)
    lr, reg_u, reg_i = float(np.float32(lr)), float(np.float32(reg_u)), float(np.float32(reg_i))
    rho32 = np.float32(rho)
    rho_d, omr = float(rho32), float(np.float32(1) - rho32)
    nnz = int(rowptr[-1])
    rows = [col[rowptr[u]:rowptr[u + 1]].tolist() for u in range(U)]
    cols = [[] for _ in range(I)]
    for u in range(U):
        for i in rows[u]:
            cols[i].append(u)
    tP, tQ = np.zeros_like(P), np.zeros_like(Q)
    loss = 0.0
    trips, groups = [], []

    def dot(a, b):
        s = 0.0
        for f in range(k):
            s += a[f] * b[f]
        return s
    for _ in range(nnz):
        while True:
            u = rng.next_int(U)
            if rows[u]:
                break
        i = rows[u][rng.next_int(len(rows[u]))]
        raters = cols[i]
        gset = JavaHashSet()
        if len(raters) <= g_len:
            for g in raters:
                gset.add(g)
        else:
            gset.add(u)
            while gset.size < g_len:
                t = raters[rng.next_int(len(raters))]
                if t not in gset:
                    gset.add(t)
        group = list(gset)
        pred = bi[i] + dot(P[u], Q[i])
        s = 0.0
        for g in group:
            s += dot(P[g], Q[i])
        pos = rho_d * (s / len(group) + bi[i]) + omr * pred
        while True:
            j = rng.next_int(I)
            if j not in rows[u]:
                break
        neg = bi[j] + dot(P[u], Q[j])
        trips.append((u, i, j)); groups.append(group)
        diff = pos - neg
        loss += -math.log(1.0 / (1.0 + math.exp(-diff)))
        deri = 1.0 / (1.0 + math.exp(diff))
        pb = bi[i]; bi[i] += lr * (deri - reg_b * pb); loss += reg_b * pb * pb
        nb = bi[j]; bi[j] += lr * (-deri - reg_b * nb); loss += reg_b * nb * nb
        avg = 1.0 / len(group)
        sum_group = [0.0] * k
        for g in group:
            delta = 1.0 if g == u else 0.0
            for f in range(k):
                gf, pf, nf = P[g, f], Q[i, f], Q[j, f]
                dg = rho_d * avg * pf + omr * delta * pf - delta * nf
                tP[g, f] += lr * (deri * dg - reg_u * gf)
                loss += reg_u * gf * gf
                sum_group[f] += gf
        for f in range(k):
            uf, pf, nf = P[u, f], Q[i, f], Q[j, f]
            pd = rho_d * avg * sum_group[f] + omr * uf
            tQ[i, f] += lr * (deri * pd - reg_i * pf)
            loss += reg_i * pf * pf
            loss += reg_i * nf * nf
            tQ[j, f] += lr * (deri * (-uf) - reg_i * nf)
    P += tP
    Q += tQ
    return loss, trips, groups


def test_gbpr_matches_python_replay(O):
    tr = rng_csr(O, 40, 25, 0.2, 6, values=(1.0,))
    k, g_len = 3, 3
    rng = np.random.default_rng(8)
    P0 = rng.normal(0, 0.1, (tr.U, k)); Q0 = rng.normal(0, 0.1, (tr.I, k)); b0 = rng.random(tr.I)
    P, Q, bi = P0.copy(), Q0.copy(), b0.copy()
    trip = np.zeros(3 * tr.nnz, np.int32); grp = np.zeros(g_len * tr.nnz, np.int32)
    O.lib().lro_seed(11)
    loss = O.lib().lro_gbpr_epoch(tr.U, tr.I, tr.rowptr, tr.col, k, P, Q, bi, 0.05, 0.01, 0.02, 0.03, 1.5, g_len,
                                  trip.ctypes.data, grp.ctypes.data)
    eP, eQ, eb = P0.copy(), Q0.copy(), b0.copy()
    eloss, etrips, egroups = gbpr_replay(11, tr.U, tr.I, tr.rowptr, tr.col, k, eP, eQ, eb, 0.05, 0.01, 0.02, 0.03, 1.5, g_len)
    assert trip.reshape(-1, 3).tolist() == [list(t) for t in etrips]
    got_groups = [[g for g in row if g >= 0] for row in grp.reshape(-1, g_len).tolist()]
    assert got_groups == egroups                                           # members AND HashSet iteration order
    assert np.array_equal(P, eP) and np.array_equal(Q, eQ) and np.array_equal(bi, eb)
    assert abs(loss - eloss) <= 1e-12 * abs(eloss)
    # factors are applied at the END of the epoch: a second epoch from the same state changes them again, the first sample
    # of this epoch saw the epoch-start factors (checked implicitly by the bit-equal replay); groups hold raters of i incl. u
    raters = {i: set(np.flatnonzero([(i in tr.col[tr.rowptr[u]:tr.rowptr[u + 1]]) for u in range(tr.U)]).tolist()) for i in range(tr.I)}
    for (u, i, j), g in zip(etrips, egroups):
        assert set(g) <= raters[i] and (u in g or len(raters[i]) <= g_len) and 1 <= len(g) <= g_len


def test_gbpr_ranking_is_biasedmf_with_zero_user_bias_and_mean(O):
    """GBPR's predict() is b_i + p_u.q_i (GBPRRecommender.java:194-196); the oracle and the device score it as BiasedMF does,
    ((d + b_u) + b_i) + mu with d the left-to-right dot product, given b_u = 0 and mu = 0.  The two agree bit for bit: the dot
    product starts from +0.0, and a round-to-nearest sum is -0.0 only when both terms are -0.0, so d is never -0.0.  Hence
    d + 0.0 == d, d + b_i is never -0.0 either, and ((d + 0) + b_i) + 0 == d + b_i == b_i + d.  This replays recommendRank
    with b_i + d in plain Python floats (sign-carrying zeros, exact ties) and compares the lists bit for bit."""
    U, I, k, N = 14, 60, 4, 8
    rng = np.random.default_rng(21)
    P, Q = rng.normal(size=(U, k)), rng.normal(size=(I, k))
    bi = rng.normal(size=I)
    P[0] = 0.0; P[1] = -0.0                               # d = +0.0 for every item: the score is b_i (or +0.0)
    Q[7] = -0.0; Q[8] = 0.0                               # d = +0.0 for every user
    bi[[7, 8, 9]] = -0.0; bi[[20, 21]] = bi[19]; Q[[20, 21]] = Q[19]   # -0.0 biases, exact ties
    tr = rng_csr(O, U, I, 0.2, 22)
    items, scores, counts = O.recommend_rank(O.BIASEDMF, U, I, k, P, Q, np.zeros(U), bi, 0.0, tr, N, nthreads=2)
    for u in range(U):
        row = set(tr.col[tr.rowptr[u]:tr.rowptr[u + 1]].tolist())
        cand = [i for i in range(I) if i not in row]
        vals = []
        for i in cand:
            d = 0.0
            for f in range(k):
                d += P[u, f] * Q[i, f]
            vals.append(float(bi[i]) + d)
        _, order = _py_topk(vals, N)
        assert counts[u] == len(order)
        assert items[u, :counts[u]].tolist() == [cand[t] for t in order]
        assert scores[u, :counts[u]].view(np.int64).tolist() == np.array([vals[t] for t in order]).view(np.int64).tolist()
