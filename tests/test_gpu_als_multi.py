"""GPU: WRMF on several devices through one multi-device handle (lrk_create_multi, rec.cuda.devices in the Java shim).  Every device
holds the full matrices, solves its own range of users and of items, and the devices exchange the new rows after each half-iteration
(multi_als_epoch in csrc/multi.cuh).  A row's solve reads only the full other side, so the split changes no
floating-point operation: the bar is BIT equality with the single-device handle and with the oracle, whatever the partition."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K_TILES = [1, 20, 40, 64, 70, 96, 112]       # every TILE instantiation of als_wrmf_solve_kernel (TILE = ceil(k / 16))


def _devices(capi, n):
    if capi.device_count() < n:
        pytest.skip("needs %d GPUs" % n)
    return list(range(n))


def _all_devices(capi):
    n = min(capi.device_count(), 8)
    if n < 2:
        pytest.skip("needs 2 GPUs")
    return list(range(n))


def _wrmf_weights(O, val, coef=4.0):
    lut = {float(v): O.lib().lro_wrmf_weight(float(v), coef) for v in np.unique(val)}
    return np.array([lut[float(v)] for v in val])


def _csr_from_mask(O, mask, seed):
    rng = np.random.default_rng(seed)
    rows, cols = np.nonzero(mask)
    rowptr = np.zeros(mask.shape[0] + 1, np.int64)
    np.add.at(rowptr, rows + 1, 1)
    val = rng.choice(np.array([1.0, 2.0, 3.0, 4.0, 5.0]), size=rows.shape[0])
    return O.Csr(mask.shape[0], mask.shape[1], np.cumsum(rowptr), cols.astype(np.int32), val)


def _csr_with_gaps(O, U, I, density, seed):
    """random CSR in which user 4 and item 3 have no entries"""
    mask = np.random.default_rng(seed).random((U, I)) < density
    mask[4, :] = False
    mask[:, 3] = False
    return _csr_from_mask(O, mask, seed + 1)


def _factors(tr, k, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(0, 0.1, (tr.U, k)), rng.normal(0, 0.1, (tr.I, k))


def _train(capi, tr, val, k, P, Q, reg_u, reg_i, iters, devices=None):
    with capi.Handle(capi.MODEL_WRMF, k, seed=1, devices=devices) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, val)
        h.set_factors(P, Q)
        losses = [h.sgd_epoch(0.0, reg_u, reg_i, 0.0, e + 1) for e in range(iters)]
        gP, gQ, _, _ = h.get_factors()
    assert losses == [0.0] * iters                       # trainModel never assigns `loss`
    return gP, gQ


def _oracle(O, tr, val, k, P, Q, reg_u, reg_i, iters):
    oP, oQ = P.copy(), Q.copy()
    for _ in range(iters):
        O.lib().lro_wrmf_epoch(tr.U, tr.I, tr.rowptr, tr.col, val, k, oP, oQ, reg_u, reg_i)
    return oP, oQ


def _check_three_ways(O, capi, tr, k, devs, reg_u=0.01, reg_i=0.02, iters=3, seed=5, equal_nan=False, P=None, Q=None):
    val = _wrmf_weights(O, tr.val)
    if P is None:
        P, Q = _factors(tr, k, seed)
    mP, mQ = _train(capi, tr, val, k, P, Q, reg_u, reg_i, iters, devices=devs)
    sP, sQ = _train(capi, tr, val, k, P, Q, reg_u, reg_i, iters)
    oP, oQ = _oracle(O, tr, val, k, P, Q, reg_u, reg_i, iters)
    for a, b in ((mP, sP), (mQ, sQ), (mP, oP), (mQ, oQ)):
        assert np.array_equal(a, b, equal_nan=equal_nan)
    return mP, mQ


@pytest.mark.parametrize("k", K_TILES)
@pytest.mark.parametrize("ndev", [2, 4, 8])
def test_wrmf_multi_bit_identical(O, capi, ndev, k):
    """an empty user row and an empty item column, rows with 0 .. ~20 entries, three iterations"""
    devs = _devices(capi, ndev)
    tr = _csr_with_gaps(O, 57, 41, 0.25, 3 + k)
    mP, mQ = _check_three_ways(O, capi, tr, k, devs, seed=k)
    assert np.isfinite(mP).all() and np.isfinite(mQ).all()


def _one_hot_item(O, seed):
    """item 0 is rated by every user but one; the rest is sparse"""
    rng = np.random.default_rng(seed)
    mask = rng.random((200, 30)) < 0.1
    mask[:, 0] = True
    mask[17, 0] = False
    return _csr_from_mask(O, mask, seed)


def _single_entry_users(O, seed):
    rng = np.random.default_rng(seed)
    mask = np.zeros((100, 40), bool)
    mask[np.arange(100), rng.integers(0, 40, 100)] = True
    return _csr_from_mask(O, mask, seed)


def _fewer_items_than_devices(O, seed, ndev):
    mask = np.random.default_rng(seed).random((60, ndev - 1)) < 0.5
    return _csr_from_mask(O, mask, seed)


@pytest.mark.parametrize("case", ["hot_item", "single_entry_users", "few_items"])
@pytest.mark.parametrize("ndev", [2, 4, 8])
def test_wrmf_multi_awkward_partitions(O, capi, ndev, case):
    """cost-balanced ranges around one very long item column, users of one entry each, and empty item ranges"""
    devs = _devices(capi, ndev)
    tr = {"hot_item": lambda: _one_hot_item(O, 11),
          "single_entry_users": lambda: _single_entry_users(O, 12),
          "few_items": lambda: _fewer_items_than_devices(O, 13, ndev)}[case]()
    _check_three_ways(O, capi, tr, 24, devs)


def test_wrmf_multi_singular_system(O, capi):
    """reg 0 and a zero factor column: every device returns the reference's half-built inverse, bit for bit"""
    devs = _devices(capi, 2)
    rng = np.random.default_rng(9)
    tr = _csr_from_mask(O, rng.random((31, 23)) < 0.3, 9)
    k = 4
    P, Q = _factors(tr, k, 1)
    Q[:, 2] = 0.0
    _check_three_ways(O, capi, tr, k, devs, reg_u=0.0, reg_i=0.0, iters=1, equal_nan=True, P=P, Q=Q)


def test_wrmf_multi_c1_factors_and_lists(O, capi, c1):
    """wrmf-test.properties (k=20, reg 0.01, coefficient 4) on the C1 train split over every device of the lease: two iterations
    through sgd_epochs, factors bit-identical to the oracle, and the top-10 list of every user equal to its recommendRank"""
    devs = _all_devices(capi)
    tr = c1["train"]
    k = 20
    val = _wrmf_weights(O, tr.val)
    P, Q = _factors(tr, k, 7)
    with capi.Handle(capi.MODEL_WRMF, k, seed=1, devices=devs) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, val)
        h.set_factors(P, Q)
        assert np.array_equal(h.sgd_epochs(2, 0.0, 0.01, 0.01), [0.0, 0.0])
        assert h.last_epoch_ms() > 0.0
        assert h.stage_stats()["ratings"] == tr.rowptr[-1]          # every device stages the matrix; it is counted once
        gP, gQ, _, _ = h.get_factors()
        items, scores, counts = h.topn(10, users=np.arange(tr.U, dtype=np.int32))
    oP, oQ = _oracle(O, tr, val, k, P, Q, 0.01, 0.01, 2)
    assert np.array_equal(gP, oP) and np.array_equal(gQ, oQ)
    oi, os_, oc = O.recommend_rank(1, tr.U, tr.I, k, oP, oQ, None, None, 0.0, tr, 10)
    assert np.array_equal(counts, oc) and np.array_equal(items, oi) and np.array_equal(scores, os_)


def test_wrmf_multi_handle_reuse(O, capi):
    """set_factors again restarts from the new factors; set_train_csr again with another matrix re-partitions it"""
    devs = _all_devices(capi)
    k = 16
    tr_a = _one_hot_item(O, 21)
    tr_b = _csr_with_gaps(O, 200, 30, 0.2, 22)
    val_a, val_b = _wrmf_weights(O, tr_a.val), _wrmf_weights(O, tr_b.val)
    P1, Q1 = _factors(tr_a, k, 1)
    P2, Q2 = _factors(tr_a, k, 2)
    with capi.Handle(capi.MODEL_WRMF, k, seed=1, devices=devs) as h:
        h.set_train_csr(tr_a.U, tr_a.I, tr_a.rowptr, tr_a.col, val_a)
        h.set_factors(P1, Q1)
        h.sgd_epoch(0.0, 0.01, 0.02, 0.0, 1)
        h.set_factors(P2, Q2)
        for e in range(2):
            h.sgd_epoch(0.0, 0.01, 0.02, 0.0, e + 1)
        aP, aQ, _, _ = h.get_factors()
        h.set_train_csr(tr_b.U, tr_b.I, tr_b.rowptr, tr_b.col, val_b)
        h.set_factors(P1, Q1)
        for e in range(2):
            h.sgd_epoch(0.0, 0.01, 0.02, 0.0, e + 1)
        bP, bQ, _, _ = h.get_factors()
        assert h.stage_stats()["ratings"] == tr_b.rowptr[-1]
    for (gP, gQ), tr, val, P, Q in (((aP, aQ), tr_a, val_a, P2, Q2), ((bP, bQ), tr_b, val_b, P1, Q1)):
        sP, sQ = _train(capi, tr, val, k, P, Q, 0.01, 0.02, 2)
        oP, oQ = _oracle(O, tr, val, k, P, Q, 0.01, 0.02, 2)
        assert np.array_equal(gP, sP) and np.array_equal(gQ, sQ)
        assert np.array_equal(gP, oP) and np.array_equal(gQ, oQ)


def test_wrmf_is_not_a_dsgd_rank(capi):
    """WRMF shards through the multi-device handle only: the process-per-GPU DSGD mode keeps refusing it"""
    with capi.Handle(capi.MODEL_WRMF, 8, seed=1) as h:
        with pytest.raises(capi.LibrecException) as e:
            h.comm_init(0, 2, bytes(128))
        assert e.value.status == capi.ERR_INVALID
    if capi.device_count() >= 2:
        with capi.Handle(capi.MODEL_WRMF, 8, seed=1, devices=[0, 1]) as h:
            with pytest.raises(capi.LibrecException) as e:
                h.comm_init(0, 2, bytes(128))
            assert e.value.status == capi.ERR_INVALID


def _topn_users(capi, h):
    """(fast, fallback) users of the last top-N call, read without lrk_topn_phase_ms (a multi handle refuses that one)"""
    a, b = C.c_int64(), C.c_int64()
    assert capi.load().lrk_topn_stats(h._h, C.byref(a), C.byref(b), None) == capi.OK
    return a.value, b.value


def test_wrmf_multi_topn_after_each_iteration(O, capi):
    """top-N of every user after iteration 1 and again after iteration 2, served by the children on the tensor-core path: each list
    equals recommendRank on the oracle's factors, so the iteration must have dropped each child's cached item operand"""
    devs = _all_devices(capi)
    U, I, k, N, per_row = 600 * len(devs), 8200, 16, 10, 10     # equal rows: >= 512 users per device; I >= 8192, N <= 26
    rng = np.random.default_rng(31)
    col = np.concatenate([np.sort(rng.choice(I, per_row, replace=False)) for _ in range(U)]).astype(np.int32)
    tr = O.Csr(U, I, np.arange(U + 1, dtype=np.int64) * per_row, col, rng.choice([1.0, 2.0, 3.0, 4.0, 5.0], U * per_row))
    val = _wrmf_weights(O, tr.val)
    P, Q = _factors(tr, k, 32)
    oP, oQ = P.copy(), Q.copy()
    with capi.Handle(capi.MODEL_WRMF, k, seed=1, devices=devs) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, val)
        h.set_factors(P, Q)
        for it in range(2):
            h.sgd_epoch(0.0, 0.01, 0.01, 0.0, it + 1)
            O.lib().lro_wrmf_epoch(tr.U, tr.I, tr.rowptr, tr.col, val, k, oP, oQ, 0.01, 0.01)
            items, scores, counts = h.topn(N)
            fast, fallback = _topn_users(capi, h)
            oi, os_, oc = O.recommend_rank(1, U, I, k, oP, oQ, None, None, 0.0, tr, N)
            assert np.array_equal(items, oi) and np.array_equal(scores.view(np.int64), os_.view(np.int64)), it
            assert np.array_equal(counts, oc), it
            assert fast > 0 and fast + fallback == U, it
