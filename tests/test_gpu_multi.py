"""GPU: the single-process multi-GPU handle (lrk_create_multi, rec.cuda.devices in the Java shim) -- full matrices in and out, sharding
inside.  With one device it must behave exactly like a plain handle; with two or more (skipped on a one-GPU lease) the DSGD epoch and
the sharded top-N must match the oracle / the single-device handle."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _conflict_free(O, n, I, seed):
    rng = np.random.default_rng(seed)
    items = rng.permutation(I)[:n].astype(np.int32)
    vals = rng.integers(1, 11, n).astype(np.float64) / 2.0
    return O.Csr(n, I, np.arange(n + 1, dtype=np.int64), items, vals)


def _devices(capi, n):
    if capi.device_count() < n:
        pytest.skip("needs %d GPUs" % n)
    return list(range(n))


@pytest.mark.parametrize("ndev", [1, 2, 4])
def test_multi_handle_conflict_free_epoch_and_topn(O, capi, ndev):
    devs = _devices(capi, ndev)
    n, I, k = 4000, 9000, 64
    tr = _conflict_free(O, n, I, 3)
    rng = np.random.default_rng(1)
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    P, Q = f32(rng.normal(0, 0.1, (n, k))), f32(rng.normal(0, 0.1, (I, k)))
    bu, bi = f32(rng.normal(0, 0.1, n)), f32(rng.normal(0, 0.1, I))
    with capi.Handle(capi.MODEL_BIASEDMF, k, devices=devs) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, 3.0)
        loss = h.sgd_epoch(0.01, 0.02, 0.03, 0.04)
        gP, gQ, gbu, gbi = h.get_factors()
        users = np.array([5, 3999, 17, 2000, 1999, 0, 3000], np.int32)
        items, scores, counts = h.topn(10, users=users)
        all_items, all_scores, all_counts = h.topn(10)
        assert h.launch_count() > 0 and h.stage_stats()["ratings"] == n
    oP, oQ, obu, obi = P.copy(), Q.copy(), bu.copy(), bi.copy()
    oloss = O.lib().lro_biasedmf_epoch(tr.U, tr.rowptr, tr.col, tr.val, k, oP, oQ, obu, obi, 3.0, 0.01, 0.02, 0.03, 0.04, None, None)
    assert np.allclose(gP, oP, rtol=0, atol=2e-6) and np.allclose(gQ, oQ, rtol=0, atol=2e-6)
    assert np.allclose(gbu, obu, rtol=0, atol=2e-6) and np.allclose(gbi, obi, rtol=0, atol=2e-6)
    assert abs(loss - oloss) <= 2e-5 * abs(oloss)
    # ranking for the trained factors: bit-identical to the oracle, whichever device served the user
    oi, os_, oc = O.recommend_rank(O.BIASEDMF, n, I, k, gP, gQ, gbu, gbi, 3.0, tr, 10, users=users)
    assert np.array_equal(items, oi) and np.array_equal(scores.view(np.int64), os_.view(np.int64)) and np.array_equal(counts, oc)
    assert np.array_equal(all_items[users], oi) and np.array_equal(all_counts[users], oc)


@pytest.mark.parametrize("ndev", [2])
def test_multi_handle_c1_rmse_within_1e3(O, capi, c1, ndev):
    devs = _devices(capi, ndev)
    tr, te, pins = c1["train"], c1["test"], c1["pins"]
    O.lib().lro_rng_set_state(*c1["rng_state"])
    P, Q, bu, bi = O.mf_setup(tr.U, tr.I, 20, True)
    mu = pins["global_mean"]
    with capi.Handle(capi.MODEL_BIASEDMF, 20, devices=devs) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q, bu, bi, mu)
        losses = h.sgd_epochs(100, 0.002, 0.01, 0.01, 0.01)
        gP, gQ, gbu, gbi = h.get_factors()
    rmse, mae = O.eval_rating(O.BIASEDMF, te, 20, gP, gQ, gbu, gbi, mu, 1.0, 5.0)
    assert abs(rmse - pins["biasedmf"]["rmse"]) < 1e-3 and abs(mae - pins["biasedmf"]["mae"]) < 1e-3
    assert np.isfinite(losses).all()


def test_multi_handle_rejects_what_it_does_not_shard(O, capi):
    devs = _devices(capi, 1)
    with capi.Handle(capi.MODEL_PMF, 8, devices=devs) as h:
        with pytest.raises(capi.LibrecException) as e:
            h.predict_pairs(np.zeros(1, np.int32), np.zeros(1, np.int32))
        assert e.value.status == capi.ERR_INVALID and "multi-device" in str(e.value)
    with pytest.raises(capi.LibrecException):
        capi.Handle(capi.MODEL_PMF, 8, devices=[0, 0])


def _sparse_csr(O, U, I, per_row, seed):
    """every user rates `per_row` distinct random items (values 1 .. 5)"""
    rng = np.random.default_rng(seed)
    col = np.concatenate([np.sort(rng.choice(I, per_row, replace=False)) for _ in range(U)]).astype(np.int32)
    return O.Csr(U, I, np.arange(U + 1, dtype=np.int64) * per_row, col, rng.integers(1, 6, U * per_row).astype(np.float64))


def _topn_users(capi, h):
    """(fast, fallback) users of the last top-N call, read without lrk_topn_phase_ms (a multi handle refuses that one)"""
    a, b = C.c_int64(), C.c_int64()
    assert capi.load().lrk_topn_stats(h._h, C.byref(a), C.byref(b), None) == capi.OK
    return a.value, b.value


@pytest.mark.parametrize("ndev,exclude_train", [(1, True), (2, True), (4, True), (2, False)])
def test_multi_handle_topn_after_training_and_set_factors(O, capi, ndev, exclude_train):
    """the children serve top-N from their own masters on the tensor-core path: after set_factors, after one more epoch (the ring
    gather refreshes the item side) and after set_factors with new factors, every list equals recommendRank on get_factors"""
    devs = _devices(capi, ndev)
    U, I, k, N = 600 * 4, 9000, 32, 10                 # >= 512 users per device, I >= 8192, k + 2 <= 128, N <= 26: tensor cores
    tr = _sparse_csr(O, U, I, 12, 5)
    rng = np.random.default_rng(6)
    fac = [(rng.normal(0, 0.1, (U, k)), rng.normal(0, 0.1, (I, k)), rng.normal(0, 0.1, U), rng.normal(0, 0.1, I)) for _ in range(2)]
    with capi.Handle(capi.MODEL_BIASEDMF, k, devices=devs) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        for step in ("set_factors", "epoch", "new_factors"):
            if step == "epoch":
                h.sgd_epoch(0.01, 0.02, 0.03, 0.04)
            else:
                h.set_factors(*fac[step == "new_factors"], 3.0)
            items, scores, counts = h.topn(N, exclude_train=exclude_train)
            fast, fallback = _topn_users(capi, h)
            gP, gQ, gbu, gbi = h.get_factors()
            oi, os_, oc = O.recommend_rank(O.BIASEDMF, U, I, k, gP, gQ, gbu, gbi, 3.0, tr if exclude_train else None, N)
            assert np.array_equal(items, oi) and np.array_equal(scores.view(np.int64), os_.view(np.int64)), step
            assert np.array_equal(counts, oc), step
            assert fast > 0 and fast + fallback == U, step


def test_one_device_multi_handle_topn_equals_plain_handle(O, capi):
    """same factors in, same lists and user counts out (no epoch: the atomic SGD epoch is not bit-reproducible across handles)"""
    devs = _devices(capi, 1)
    U, I, k, N = 1500, 9000, 32, 20
    tr = _sparse_csr(O, U, I, 15, 8)
    rng = np.random.default_rng(9)
    P, Q, bu, bi = rng.normal(0, 0.1, (U, k)), rng.normal(0, 0.1, (I, k)), rng.normal(0, 0.1, U), rng.normal(0, 0.1, I)
    users = rng.permutation(U)[:1200].astype(np.int32)
    out = []
    for devices in (None, devs):
        with capi.Handle(capi.MODEL_BIASEDMF, k, devices=devices) as h:
            h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
            h.set_factors(P, Q, bu, bi, 3.0)
            out.append((h.topn(N, users=users), _topn_users(capi, h)))
    (a, sa), (b, sb) = out
    assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))
    assert sa == sb and sa[0] > 0
