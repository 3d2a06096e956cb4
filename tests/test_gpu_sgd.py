"""GPU: SGD epoch parity through the C ABI against the oracle (same seeded inputs)."""
import numpy as np
import pytest

from conftest import rng_csr

pytestmark = pytest.mark.gpu


def _conflict_free(O, n, I, seed):
    """every user and item appears exactly once -> no concurrent updates, result is order-free"""
    rng = np.random.default_rng(seed)
    items = rng.permutation(I)[:n].astype(np.int32)
    vals = rng.integers(1, 11, n).astype(np.float64) / 2.0
    return O.Csr(n, I, np.arange(n + 1, dtype=np.int64), items, vals)


@pytest.mark.parametrize("model_name,k", [("biasedmf", 64), ("biasedmf", 20), ("pmf", 128), ("pmf", 6), ("biasedmf", 200), ("pmf", 1)])
@pytest.mark.parametrize("mode", ["atomic", "hogwild"])
def test_conflict_free_epoch_matches_oracle(O, capi, model_name, k, mode):
    n, I = 3000, 4000
    tr = _conflict_free(O, n, I, 3)
    rng = np.random.default_rng(1)
    P = rng.normal(0, 0.1, (n, k)); Q = rng.normal(0, 0.1, (I, k))
    biased = model_name == "biasedmf"
    bu = rng.normal(0, 0.1, n) if biased else None
    bi = rng.normal(0, 0.1, I) if biased else None
    mu = 3.0
    # the device works on fp32 copies: start the oracle from the same rounded values
    P, Q = P.astype(np.float32).astype(np.float64), Q.astype(np.float32).astype(np.float64)
    if biased:
        bu, bi = bu.astype(np.float32).astype(np.float64), bi.astype(np.float32).astype(np.float64)
    model = capi.MODEL_BIASEDMF if biased else capi.MODEL_PMF
    with capi.Handle(model, k, update_mode=capi.UPDATE_ATOMIC if mode == "atomic" else capi.UPDATE_HOGWILD) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, mu)
        loss = h.sgd_epoch(0.01, 0.02, 0.03, 0.04)
        gP, gQ, gbu, gbi = h.get_factors()
    oP, oQ = P.copy(), Q.copy()
    if biased:
        obu, obi = bu.copy(), bi.copy()
        oloss = O.lib().lro_biasedmf_epoch(tr.U, tr.rowptr, tr.col, tr.val, k, oP, oQ, obu, obi, mu, 0.01, 0.02, 0.03, 0.04, None, None)
    else:
        oloss = O.lib().lro_pmf_epoch(tr.U, tr.rowptr, tr.col, tr.val, k, oP, oQ, 0.01, 0.02, 0.03, None, None)
    # fp32 arithmetic vs fp64: tolerance = a few fp32 ulps of the operands (|values| <= ~5)
    assert np.allclose(gP, oP, rtol=0, atol=2e-6) and np.allclose(gQ, oQ, rtol=0, atol=2e-6)
    if biased:
        assert np.allclose(gbu, obu, rtol=0, atol=2e-6) and np.allclose(gbi, obi, rtol=0, atol=2e-6)
    assert abs(loss - oloss) <= 2e-5 * abs(oloss)
    # rows of users/items without ratings are untouched
    untouched = np.setdiff1d(np.arange(I), tr.col)
    assert np.array_equal(gQ[untouched], Q[untouched])


@pytest.mark.parametrize("model_name,k", [("biasedmf", 64), ("pmf", 128), ("biasedmf", 20), ("pmf", 3)])
def test_item_run_tiles_are_minibatches_for_the_item(O, capi, model_name, k):
    """Items with >= 512 ratings are staged as runs of 32 ratings (staging.cuh) and the kernel applies one item-row
    update per flush period (8, 16 or 32 ratings of a run, sgd.cuh): for users that rate a single item this is a mini-batch step on q_i / b_i.
    To first order in lr the epoch equals one step with every gradient taken at the initial q_i; which chunks see
    which earlier updates depends on scheduling and moves the result by O(lr^2 * degree) -- hence the tolerances.
    The item-side tolerances are loose on purpose: at lr * degree = 0.026 the item step also carries the staleness damping of
    run tiles (a few per cent) and second-order terms of the same size, which this test does not model.  The item side is held
    to derived budgets, and the damping to its formula, in test_gpu_sgd_first_order.py."""
    n_items, per_item = 6, 512
    n = n_items * per_item
    rng = np.random.default_rng(5)
    items = np.repeat(np.arange(n_items, dtype=np.int32), per_item)        # user u rates item u // 512 only
    vals = rng.integers(1, 6, n).astype(np.float64)
    I = 10
    tr = O.Csr(n, I, np.arange(n + 1, dtype=np.int64), items, vals)
    P = rng.normal(0, 0.1, (n, k)).astype(np.float32).astype(np.float64)
    Q = rng.normal(0, 0.1, (I, k)).astype(np.float32).astype(np.float64)
    biased = model_name == "biasedmf"
    bu = rng.normal(0, 0.1, n).astype(np.float32).astype(np.float64) if biased else None
    bi = rng.normal(0, 0.1, I).astype(np.float32).astype(np.float64) if biased else None
    mu, lr, ru, ri, rb = 3.0, 0.00005, 0.02, 0.03, 0.04     # small lr: the O(lr^2) interaction of the two runs stays tiny
    model = capi.MODEL_BIASEDMF if biased else capi.MODEL_PMF
    with capi.Handle(model, k) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, mu)
        loss = h.sgd_epoch(lr, ru, ri, rb)
        gP, gQ, gbu, gbi = h.get_factors()
    # mini-batch restatement of BiasedMFRecommender.java:77-98 / PMFSimilarityRecommender.java:64-82 per item
    q = Q[items]
    pred = np.einsum("ij,ij->i", P, q) + ((bu + bi[items] + mu) if biased else 0.0)
    err = vals - pred
    eP = P + lr * (err[:, None] * q - ru * P)
    dq = lr * (err[:, None] * P - ri * q)
    eQ = Q.copy()
    np.add.at(eQ, items, dq)
    assert np.allclose(gP, eP, rtol=0, atol=5e-6)                            # user side: one rating per user
    assert np.allclose(gQ, eQ, rtol=0, atol=1e-4) and np.abs(gQ - Q)[:n_items].max() > 2e-4
    assert np.array_equal(gQ[n_items:], Q[n_items:])
    eloss = np.sum(err ** 2) + np.sum(ru * P * P) + np.sum(ri * q * q)
    if biased:
        ebu = bu + lr * (err - rb * bu)
        ebi = bi.copy(); np.add.at(ebi, items, lr * (err - rb * bi[items]))
        assert np.allclose(gbu, ebu, rtol=0, atol=5e-6) and np.allclose(gbi, ebi, rtol=0, atol=1e-3)
        assert np.abs(gbi - bi)[:n_items].max() > 1e-3
        eloss += np.sum(rb * bu * bu) + np.sum(rb * bi[items] ** 2)
    assert abs(loss - 0.5 * eloss) <= 1e-3 * abs(0.5 * eloss)


def _train_gpu(capi, model, tr, k, P, Q, bu, bi, mu, lr, reg_u, reg_i, reg_b, iters, seed=1):
    with capi.Handle(model, k, seed=seed) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, mu)
        losses = [h.sgd_epoch(lr, reg_u, reg_i, reg_b, it) for it in range(1, iters + 1)]
        return h.get_factors(), losses


def test_c1_biasedmf_rmse_mae_within_1e3(O, capi, c1):
    """config C1 (biasedmf-test.properties on the seeded ml-100k split): RMSE / MAE within 1e-3 of the reference order"""
    tr, te, pins = c1["train"], c1["test"], c1["pins"]
    O.lib().lro_rng_set_state(*c1["rng_state"])
    P, Q, bu, bi = O.mf_setup(tr.U, tr.I, 20, True)
    (gP, gQ, gbu, gbi), losses = _train_gpu(capi, capi.MODEL_BIASEDMF, tr, 20, P, Q, bu, bi, pins["global_mean"],
                                            0.002, 0.01, 0.01, 0.01, 100)
    rmse, mae = O.eval_rating(O.BIASEDMF, te, 20, gP, gQ, gbu, gbi, pins["global_mean"], 1.0, 5.0)
    assert abs(rmse - pins["biasedmf"]["rmse"]) < 1e-3, (rmse, pins["biasedmf"]["rmse"])
    assert abs(mae - pins["biasedmf"]["mae"]) < 1e-3, (mae, pins["biasedmf"]["mae"])
    # loss curve: same definition as the reference, close to the sequential run, decreasing.  Epoch 1 is
    # looser: with thousands of ratings in flight the errors of one epoch are measured against slightly
    # older factors than in the sequential Gauss-Seidel walk (measured: +2.7 % on epoch 1, <1 % at the end).
    assert abs(losses[0] - pins["biasedmf"]["loss_1"]) < 0.05 * pins["biasedmf"]["loss_1"]
    assert abs(losses[-1] - pins["biasedmf"]["loss_100"]) < 0.01 * pins["biasedmf"]["loss_100"]
    assert all(b < a for a, b in zip(losses, losses[1:]))


def test_c1_pmf_fast_mode_tracks_reference(O, capi, c1):
    """PMF (pmf-test.properties hyper-parameters) on the C1 split, fast shuffled/atomic mode.
    At lr 0.01 / 70 iterations the result depends on the visiting ORDER at the 8e-3 level (a CPU
    simulation of the sequential loop over a shuffled order gives RMSE -7.8e-3 vs CSR order), so the
    fast mode is held to 1e-2 here; the reference-order mode below is held to bit-exactness."""
    tr, te, pins = c1["train"], c1["test"], c1["pins"]
    O.lib().lro_rng_set_state(*c1["rng_state"])
    P, Q, _, _ = O.mf_setup(tr.U, tr.I, 6, False)
    (gP, gQ, _, _), losses = _train_gpu(capi, capi.MODEL_PMF, tr, 6, P, Q, None, None, pins["global_mean"],
                                        0.01, 0.08, 0.08, 0.0, 70)
    rmse, mae = O.eval_rating(O.PMF, te, 6, gP, gQ, None, None, pins["global_mean"], 1.0, 5.0)
    assert abs(rmse - pins["pmf"]["rmse"]) < 1e-2, (rmse, pins["pmf"]["rmse"])
    assert abs(mae - pins["pmf"]["mae"]) < 1e-2, (mae, pins["pmf"]["mae"])
    assert abs(losses[-1] - pins["pmf"]["loss_70"]) < 0.03 * pins["pmf"]["loss_70"]


@pytest.mark.parametrize("model_name,k,iters,hyper", [
    ("biasedmf", 20, 100, (0.002, 0.01, 0.01, 0.01)),      # biasedmf-test.properties == config C1 in full
    ("pmf", 6, 70, (0.01, 0.08, 0.08, 0.0)),               # pmf-test.properties hyper-parameters
    ("biasedmf", 64, 3, (0.002, 0.01, 0.01, 0.01)),
    ("pmf", 128, 2, (0.01, 0.08, 0.08, 0.0)),
])
def test_reference_order_mode_is_bit_identical(O, capi, c1, model_name, k, iters, hyper):
    """LRK_UPDATE_REFERENCE_ORDER: the sequential CSR walk as a dependency wavefront in fp64 ->
    factors after `iters` epochs are bit-identical to the oracle; RMSE/MAE therefore identical."""
    tr, te, pins = c1["train"], c1["test"], c1["pins"]
    biased = model_name == "biasedmf"
    O.lib().lro_rng_set_state(*c1["rng_state"])
    P, Q, bu, bi = O.mf_setup(tr.U, tr.I, k, biased)
    mu = pins["global_mean"]
    model = capi.MODEL_BIASEDMF if biased else capi.MODEL_PMF
    with capi.Handle(model, k, update_mode=capi.UPDATE_REFERENCE_ORDER) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, mu)
        losses = [h.sgd_epoch(*hyper, it + 1) for it in range(iters)]
        gP, gQ, gbu, gbi = h.get_factors()
        rmse, mae = h.eval_rating(te.U, te.rowptr, te.col, te.val, 1.0, 5.0)
    oP, oQ = P.copy(), Q.copy()
    obu, obi = (bu.copy(), bi.copy()) if biased else (None, None)
    done, ol = O.train(O.BIASEDMF if biased else O.PMF, tr, k, oP, oQ, obu, obi, mu, hyper[0], 1000.0, hyper[1], hyper[2], hyper[3], iters)
    assert done == iters
    assert np.array_equal(gP.view(np.int64), oP.view(np.int64)) and np.array_equal(gQ.view(np.int64), oQ.view(np.int64))
    if biased:
        assert np.array_equal(gbu.view(np.int64), obu.view(np.int64)) and np.array_equal(gbi.view(np.int64), obi.view(np.int64))
    assert np.allclose(losses, ol, rtol=1e-11, atol=0)          # only the scalar loss is summed in another order
    ormse, omae = O.eval_rating(O.BIASEDMF if biased else O.PMF, te, k, oP, oQ, obu, obi, mu, 1.0, 5.0)
    assert abs(rmse - ormse) < 1e-12 and abs(mae - omae) < 1e-12
    if iters == 100:
        assert abs(ormse - pins["biasedmf"]["rmse"]) < 1e-12 and abs(omae - pins["biasedmf"]["mae"]) < 1e-12


def test_bpr_samples_are_valid_and_uniform(O, capi):
    tr = rng_csr(O, 400, 300, 0.05, 7, values=(1.0,))
    tr.rowptr[5:] -= (tr.rowptr[5] - tr.rowptr[4])       # make user 4 empty
    lo, hi = tr.rowptr[4], tr.rowptr[4] + (len(tr.col) - tr.rowptr[-1])
    keep = np.ones(len(tr.col), bool); keep[lo:hi] = False
    tr = O.Csr(tr.U, tr.I, tr.rowptr, tr.col[keep], tr.val[keep])
    with capi.Handle(capi.MODEL_BPR, 16, seed=5) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        s1 = h.bpr_peek_samples(1, 0, 60000)
        s1b = h.bpr_peek_samples(1, 0, 1000)
        s2 = h.bpr_peek_samples(2, 0, 1000)
    assert np.array_equal(s1[:1000], s1b) and not np.array_equal(s1b, s2)
    member = set((int(u) << 32) | int(i) for u, i in zip(tr.rows(), tr.col))
    u, i, j = s1[:, 0], s1[:, 1], s1[:, 2]
    assert u.min() >= 0 and u.max() < tr.U and 4 not in set(u.tolist())
    assert all(((int(a) << 32) | int(b)) in member for a, b in zip(u[:5000], i[:5000]))
    assert not any(((int(a) << 32) | int(b)) in member for a, b in zip(u[:5000], j[:5000]))
    # BPRRecommender.java:58 draws users uniformly (not by degree): chi-square over users
    cnt = np.bincount(u, minlength=tr.U).astype(np.float64)
    exp = len(u) / (tr.U - 1)
    chi2 = ((np.delete(cnt, 4) - exp) ** 2 / exp).sum()
    assert chi2 < 1.35 * (tr.U - 2)


def test_bpr_epoch_tracks_oracle_on_its_own_samples(O, capi):
    """feed the kernel's own (u,i,j) draws through the reference arithmetic: same loss, close factors"""
    tr = rng_csr(O, 3000, 2000, 0.01, 3, values=(1.0,))
    k = 32
    rng = np.random.default_rng(0)
    P = rng.normal(0, 0.1, (tr.U, k)).astype(np.float32).astype(np.float64)
    Q = rng.normal(0, 0.1, (tr.I, k)).astype(np.float32).astype(np.float64)
    n = tr.nnz
    with capi.Handle(capi.MODEL_BPR, k, seed=9) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        trip = h.bpr_peek_samples(1, 0, n)
        loss = h.sgd_epoch(0.01, 0.01, 0.01, 0.0, 1)
        gP, gQ, _, _ = h.get_factors()
    oP, oQ = P.copy(), Q.copy()
    trip = np.ascontiguousarray(trip.reshape(-1))
    oloss = O.lib().lro_bpr_epoch(tr.U, tr.I, tr.rowptr, tr.col, k, oP, oQ, 0.01, 0.01, 0.01, n, trip.ctypes.data, None)
    assert abs(loss - oloss) < 2e-3 * oloss
    # same samples, different interleaving: factor movement agrees to a small fraction of the step
    step = np.abs(oP - P).max()
    assert np.abs(gP - oP).max() < 0.1 * step + 1e-6
    assert np.abs(gQ - oQ).max() < 0.1 * np.abs(oQ - Q).max() + 1e-6


def test_diverged_loss_is_reported(O, capi):
    tr = rng_csr(O, 50, 40, 0.5, 1)
    P = np.full((50, 8), 1e18); Q = np.full((40, 8), 1e18)
    with capi.Handle(capi.MODEL_PMF, 8) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        with pytest.raises(capi.LibrecException) as e:
            for it in range(3):
                h.sgd_epoch(0.01, 0.01, 0.01, 0.0, it + 1)
        assert e.value.status == capi.ERR_DIVERGED and "NaN or Infinity" in str(e.value)
        # the safeguard re-ran the epoch with fewer ratings in flight before giving up
        assert h.sgd_safeguard()["rollbacks"] >= 1 and h.sgd_safeguard()["conc_div"] > 1


def test_argument_errors(O, capi):
    tr = rng_csr(O, 10, 12, 0.5, 1)
    with capi.Handle(capi.MODEL_BIASEDMF, 8) as h:
        with pytest.raises(capi.LibrecException):
            h.set_factors(np.zeros((10, 8)), np.zeros((12, 8)), np.zeros(10), np.zeros(12), 0.0)   # CSR first
        bad = tr.col.copy(); bad[0] = 99
        with pytest.raises(capi.LibrecException):
            h.set_train_csr(tr.U, tr.I, tr.rowptr, bad, tr.val)
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        with pytest.raises(capi.LibrecException):
            h.set_factors(np.zeros((10, 8)), np.zeros((12, 8)), None, None, 0.0)                   # biases required
        with pytest.raises(capi.LibrecException):
            h.sgd_epoch(0.01, 0.01, 0.01, 0.01)                                                    # no factors yet


def test_empty_and_ragged_inputs(O, capi):
    # users without ratings, items without ratings, and an all-empty matrix
    tr = O.Csr(5, 6, [0, 0, 3, 3, 4, 4], [0, 2, 5, 1], [1.0, 2.0, 3.0, 4.0])
    P = np.ones((5, 4)) * 0.1; Q = np.ones((6, 4)) * 0.1
    with capi.Handle(capi.MODEL_PMF, 4) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        loss = h.sgd_epoch(0.01, 0.01, 0.01)
        gP, gQ, _, _ = h.get_factors()
    assert np.array_equal(gP[[0, 2, 4]], P[[0, 2, 4]].astype(np.float32).astype(np.float64)) and loss > 0
    empty = O.Csr(3, 3, [0, 0, 0, 0], np.zeros(0, np.int32), np.zeros(0))
    with capi.Handle(capi.MODEL_PMF, 4) as h:
        h.set_train_csr(3, 3, empty.rowptr, empty.col, empty.val)
        h.set_factors(np.ones((3, 4)), np.ones((3, 4)))
        assert h.sgd_epoch(0.01, 0.01, 0.01) == 0.0


@pytest.mark.timeout(120)
def test_reference_order_mode_survives_restaging(O, capi):
    """ADVICE r01: a second lrk_set_train_csr on a reference-order handle rebuilds the wavefront schedule and its barrier counter;
    the epoch after it must not wait for arrivals counted on the old counter (it used to spin for ever -- e.g. cross-validation
    folds reusing one handle).  Both stagings must also stay bit-identical to the oracle."""
    k = 8
    rng = np.random.default_rng(5)
    with capi.Handle(capi.MODEL_PMF, k, update_mode=capi.UPDATE_REFERENCE_ORDER) as h:
        for fold in range(2):
            tr = rng_csr(O, 60, 50, 0.2, 100 + fold)
            P, Q = rng.normal(0, 0.1, (60, k)), rng.normal(0, 0.1, (50, k))
            h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
            h.set_factors(P, Q)
            for it in range(3):
                h.sgd_epoch(0.01, 0.05, 0.05, 0.0, it + 1)
            gP, gQ, _, _ = h.get_factors()
            oP, oQ = P.copy(), Q.copy()
            for it in range(3):
                O.lib().lro_pmf_epoch(tr.U, tr.rowptr, tr.col, tr.val, k, oP, oQ, 0.01, 0.05, 0.05, None, None)
            assert np.array_equal(gP, oP) and np.array_equal(gQ, oQ)


def test_peeking_samples_does_not_change_training(O, capi):
    """ADVICE r01: lrk_bpr_peek_samples is read-only -- training with and without peeks in between gives the same factors"""
    tr = rng_csr(O, 300, 200, 0.1, 9)
    rng = np.random.default_rng(2)
    P, Q = rng.normal(0, 0.1, (300, 16)), rng.normal(0, 0.1, (200, 16))
    outs = []
    for peek in (False, True):
        with capi.Handle(capi.MODEL_RANKSGD, 16, seed=3) as h:
            h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
            h.set_factors(P, Q)
            losses = []
            for it in range(4):
                if peek:
                    h.bpr_peek_samples(it + 1, 0, 64)
                    h.bpr_peek_samples(it + 1, 0, 64)
                losses.append(h.sgd_epoch(0.01, 0.0, 0.0, 0.0, it + 1))
            outs.append(losses)
    assert np.allclose(outs[0], outs[1], rtol=1e-3), outs    # atomics reorder fp32 sums; the kernel variant / grid must not change


def test_sgd_epochs_batches_the_iterations(O, capi):
    """lrk_sgd_epochs(n) == n x lrk_sgd_epoch with updateLRate's decay branch (MatrixFactorizationRecommender.java:131-138)"""
    n, I, k = 2000, 3000, 16
    tr = _conflict_free(O, n, I, 11)
    rng = np.random.default_rng(4)
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    P, Q = f32(rng.normal(0, 0.1, (n, k))), f32(rng.normal(0, 0.1, (I, k)))
    with capi.Handle(capi.MODEL_PMF, k) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        la = h.sgd_epochs(3, 0.02, 0.05, 0.05, 0.0, 1, decay=0.5, max_lr=0.015)
        A = h.get_factors()
        h.set_factors(P, Q)
        lb, lr = [], np.float32(0.02)
        for it in range(3):
            lb.append(h.sgd_epoch(float(lr), 0.05, 0.05, 0.0, it + 1))
            lr = min(np.float32(lr * np.float32(0.5)), np.float32(0.015))
        B = h.get_factors()
    assert np.allclose(la, lb, rtol=1e-6) and np.allclose(A[0], B[0], atol=1e-6) and np.allclose(A[1], B[1], atol=1e-6)
    st = None
    with capi.Handle(capi.MODEL_PMF, k) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        st = h.stage_stats()
    assert st["ratings"] == n and st["run_tile_ratings"] == 0


@pytest.mark.parametrize("shape,k", [("tiny", 64), ("small", 128), ("ml-1m", 20)])
def test_unit_ordered_stream_is_a_permutation_with_exclusive_units(O, capi, shape, k, monkeypatch):
    monkeypatch.setenv("LRK_SGD_GROUP", "1")
    _unit_stream_checks(O, capi, shape, k)


def _unit_stream_checks(O, capi, shape, k):
    """staging_group.cuh: the unit-ordered stream holds every train entry exactly once; the units partition it; a unit's ratings
    belong to its own users, users of units that store their rows (slices == 0) are disjoint, and inside a unit every item's
    ratings are adjacent (one item-row read + one RED per (unit, item) pair)"""
    from librec_b200 import synth
    d = synth.make_ratings(shape, cache=False)
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    with capi.Handle(capi.MODEL_PMF, k) as h:
        h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
        su, si, sr, units = h.debug_stream(nnz)
    assert units is not None and units.shape[0] > 0
    rows = np.repeat(np.arange(U, dtype=np.int64), np.diff(d["rowptr"]))
    want = np.sort(rows * I + d["col"])
    got = su.astype(np.int64) * I + si
    order = np.argsort(got, kind="stable")
    assert np.array_equal(got[order], want)
    ref_val = d["val"][np.argsort(rows * I + d["col"], kind="stable")].astype(np.float32)
    assert np.array_equal(sr[order], ref_val)
    start, count, first, w = units[:, 0].astype(np.int64) & 0xffffffff, units[:, 1], units[:, 2], units[:, 3]
    nus, slices = w & 0xffff, w >> 16
    assert count.sum() == nnz and np.array_equal(start, np.concatenate([[0], np.cumsum(count)[:-1]]))
    assert nus.max() <= 16 and (nus[slices > 0] == 1).all()
    owner = np.full(U, -1, np.int64)
    for t in range(units.shape[0]):
        a, b = start[t], start[t] + count[t]
        uu, ii = su[a:b], si[a:b]
        assert ((uu >= first[t]) & (uu < first[t] + nus[t])).all()
        if count[t]:
            change = np.flatnonzero(np.diff(ii) != 0)
            heads = ii[np.concatenate([[0], change + 1])]
            assert np.unique(heads).shape[0] == heads.shape[0], "an item's ratings are split inside a unit"
        if slices[t] == 0:
            assert (owner[first[t]:first[t] + nus[t]] == -1).all(), "two units store the same user's row"
            owner[first[t]:first[t] + nus[t]] = t


@pytest.mark.parametrize("model_name,k", [("biasedmf", 64), ("pmf", 128), ("biasedmf", 20)])
def test_group_kernel_conflict_free_epoch_matches_oracle(O, capi, model_name, k, monkeypatch):
    """LRK_SGD_GROUP=1 (sgd_group.cuh): with every user and item rated once nothing is concurrent -- one epoch of the user-group
    kernel equals the oracle's epoch up to fp32 rounding"""
    monkeypatch.setenv("LRK_SGD_GROUP", "1")
    n, I = 3000, 4000
    tr = _conflict_free(O, n, I, 3)
    rng = np.random.default_rng(1)
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    P, Q = f32(rng.normal(0, 0.1, (n, k))), f32(rng.normal(0, 0.1, (I, k)))
    biased = model_name == "biasedmf"
    bu = f32(rng.normal(0, 0.1, n)) if biased else None
    bi = f32(rng.normal(0, 0.1, I)) if biased else None
    with capi.Handle(capi.MODEL_BIASEDMF if biased else capi.MODEL_PMF, k) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        assert h.debug_stream(tr.nnz)[3] is not None          # the unit-ordered stream is in use
        h.set_factors(P, Q, bu, bi, 3.0)
        loss = h.sgd_epoch(0.01, 0.02, 0.03, 0.04)
        gP, gQ, gbu, gbi = h.get_factors()
    oP, oQ = P.copy(), Q.copy()
    if biased:
        obu, obi = bu.copy(), bi.copy()
        oloss = O.lib().lro_biasedmf_epoch(tr.U, tr.rowptr, tr.col, tr.val, k, oP, oQ, obu, obi, 3.0, 0.01, 0.02, 0.03, 0.04, None, None)
        assert np.allclose(gbu, obu, rtol=0, atol=2e-6) and np.allclose(gbi, obi, rtol=0, atol=2e-6)
    else:
        oloss = O.lib().lro_pmf_epoch(tr.U, tr.rowptr, tr.col, tr.val, k, oP, oQ, 0.01, 0.02, 0.03, None, None)
    assert np.allclose(gP, oP, rtol=0, atol=2e-6) and np.allclose(gQ, oQ, rtol=0, atol=2e-6)
    assert abs(loss - oloss) <= 2e-5 * abs(oloss)


def test_group_kernel_c1_biasedmf_rmse_mae_within_1e3(O, capi, c1, monkeypatch):
    """LRK_SGD_GROUP=1 on config C1 (k=20 -> the 8-lane layout): RMSE / MAE within 1e-3 of the oracle"""
    monkeypatch.setenv("LRK_SGD_GROUP", "1")
    tr, te, pins = c1["train"], c1["test"], c1["pins"]
    O.lib().lro_rng_set_state(*c1["rng_state"])
    P, Q, bu, bi = O.mf_setup(tr.U, tr.I, 20, True)
    mu = pins["global_mean"]
    with capi.Handle(capi.MODEL_BIASEDMF, 20) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        assert h.debug_stream(tr.nnz)[3] is not None
        h.set_factors(P, Q, bu, bi, mu)
        for it in range(100):
            h.sgd_epoch(0.002, 0.01, 0.01, 0.01, it + 1)
        rmse, mae = h.eval_rating(te.U, te.rowptr, te.col, te.val, 1.0, 5.0)
    print("group kernel C1: rmse %.6f (oracle %.6f) mae %.6f (oracle %.6f)" % (rmse, pins["biasedmf"]["rmse"], mae, pins["biasedmf"]["mae"]))
    assert abs(rmse - pins["biasedmf"]["rmse"]) < 1e-3 and abs(mae - pins["biasedmf"]["mae"]) < 1e-3


def test_group_kernel_c1_pmf_tracks_reference_order(O, capi, c1, monkeypatch):
    """PMF at lr 0.01 is sensitive to the visiting order (the shuffled stream kernel is held to 1e-2 above).  The user-group kernel
    walks user by user like the reference, every unit through its own rotation of the ascending item order (k=6 is padded to the
    8-lane layout).  r02 on a B200: RMSE -3.2e-3 / MAE -1.7e-3 from the reference -- 2-3x closer than the shuffled stream, still not
    the 1e-3 the reference-order mode delivers.  (Without the rotation, LRK_SGD_GROUP_ROTATE=0, all units start on the low item ids
    together and this configuration diverges: the rotation is what spreads the units over the catalogue.)"""
    monkeypatch.setenv("LRK_SGD_GROUP", "1")
    tr, te, pins = c1["train"], c1["test"], c1["pins"]
    O.lib().lro_rng_set_state(*c1["rng_state"])
    P, Q, _, _ = O.mf_setup(tr.U, tr.I, 6, False)
    with capi.Handle(capi.MODEL_PMF, 6) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        assert h.debug_stream(tr.nnz)[3] is not None
        h.set_factors(P, Q)
        losses = [h.sgd_epoch(0.01, 0.08, 0.08, 0.0, it + 1) for it in range(70)]
        gP, gQ, _, _ = h.get_factors()
    rmse, mae = O.eval_rating(O.PMF, te, 6, gP, gQ, None, None, pins["global_mean"], 1.0, 5.0)
    print("group kernel PMF C1: rmse %.6f (oracle %.6f, d %+.2e)  mae %.6f (oracle %.6f, d %+.2e)  loss_70 %.2f (oracle %.2f)" % (
        rmse, pins["pmf"]["rmse"], rmse - pins["pmf"]["rmse"], mae, pins["pmf"]["mae"], mae - pins["pmf"]["mae"], losses[-1], pins["pmf"]["loss_70"]))
    assert abs(rmse - pins["pmf"]["rmse"]) < 5e-3 and abs(mae - pins["pmf"]["mae"]) < 5e-3
