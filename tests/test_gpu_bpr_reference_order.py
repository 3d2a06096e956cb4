"""GPU: reference-order BPR (LRK_UPDATE_REFERENCE_ORDER with LRK_MODEL_BPR, csrc/sgd_bpr_exact.cuh) against the StrictMath BPR
epoch of tests/bpr_strict_reference.cpp: the drawn samples, the learned factors and the java.util.Random state after the epochs are bit-identical."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import rng_csr
import bpr_strict
from test_oracle_aobpr import JavaRandom
from test_oracle_bpr_strict import REJECTION_SEED, rejection_csr, seeded_state

pytestmark = pytest.mark.gpu

HYPER = (0.01, 0.01, 0.01)                  # bpr-test.properties: learnrate, user and item regularization


def _ones(O, tr):
    return O.Csr(tr.U, tr.I, tr.rowptr, tr.col, np.ones(tr.nnz))


def _handle(capi, k, seed=1):
    return capi.Handle(capi.MODEL_BPR, k, seed=seed, update_mode=capi.UPDATE_REFERENCE_ORDER)


def _oracle_samples(O, tr, state, n):
    L = bpr_strict.lib()
    L.lro_set_jrandom_state(state)
    trip = np.zeros(3 * n, np.int32)
    P, Q = np.zeros((tr.U, 1)), np.zeros((tr.I, 1))
    L.lro_bpr_epoch_strict(tr.U, tr.I, tr.rowptr, tr.col, 1, P, Q, 0.0, 0.0, 0.0, n, None, trip.ctypes.data)
    return trip.reshape(n, 3), L.lro_jrandom_state()


def _oracle_epochs(O, tr, k, P, Q, state, epochs, lr=HYPER[0], reg_u=HYPER[1], reg_i=HYPER[2], decay=1.0):
    L = bpr_strict.lib()
    L.lro_set_jrandom_state(state)
    P, Q = P.copy(), Q.copy()
    losses = []
    last_loss = C.c_double(0.0)
    rate = lr
    for it in range(1, epochs + 1):
        losses.append(L.lro_bpr_epoch_strict(tr.U, tr.I, tr.rowptr, tr.col, k, P, Q, rate, reg_u, reg_i, tr.nnz, None, None))
        rate = O.lib().lro_update_lrate(rate, 0.0, it, 0, decay, losses[-1], C.byref(last_loss))
    return P, Q, losses, L.lro_jrandom_state()


def _mixed_csr(O, U, I, seed, density=0.3):
    """random rows plus an empty row, a full row and a row whose length is a power of two"""
    tr = rng_csr(O, U, I, density, seed)
    rows = [tr.col[tr.rowptr[u]:tr.rowptr[u + 1]] for u in range(U)]
    rows[0] = np.zeros(0, np.int32)
    rows[1] = np.arange(I, dtype=np.int32)
    rows[2] = np.sort(np.random.default_rng(seed).choice(I, 8, replace=False)).astype(np.int32)
    rowptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col = np.concatenate(rows).astype(np.int32)
    return O.Csr(U, I, rowptr, col, np.ones(col.shape[0]))


def _init(U, I, k, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(0, 0.1, (U, k)), rng.normal(0, 0.1, (I, k))


def _same(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.int64), np.ascontiguousarray(b).view(np.int64))


def _state(h):
    return int(h.get_matrix("jdk.random.state", (1,))[0])


# ---- sampler -------------------------------------------------------------------------------------------------------------
def test_sampler_c1_equals_the_oracle(O, capi, c1):
    tr = _ones(O, c1["train"])
    with _handle(capi, 10, seed=1) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        assert _state(h) == seeded_state(1)                         # default: new Random(cfg.seed)
        got = h.bpr_peek_samples(1, 0, tr.nnz)
        window = h.bpr_peek_samples(99, 1234, 5000)                 # the epoch argument is ignored
        beyond = h.bpr_peek_samples(1, tr.nnz - 10, 30)            # past numRates: the stream continues
    want, _ = _oracle_samples(O, tr, seeded_state(1), tr.nnz + 20)
    assert np.array_equal(got, want[:tr.nnz])
    assert np.array_equal(window, want[1234:6234]) and np.array_equal(beyond, want[tr.nnz - 10:tr.nnz + 20])


@pytest.mark.parametrize("U,I,seed", [(64, 32, 1), (37, 29, 2), (50, 16, 3), (128, 100, 4), (33, 64, 5)])
def test_sampler_random_csr_equals_the_oracle(O, capi, U, I, seed):
    tr = _mixed_csr(O, U, I, seed)
    state = seeded_state(100 + seed)
    with _handle(capi, 4) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_matrix("jdk.random.state", np.array([float(state)]))
        got = h.bpr_peek_samples(1, 0, 3 * tr.nnz)
    want, _ = _oracle_samples(O, tr, state, 3 * tr.nnz)
    assert np.array_equal(got, want)


def test_sampler_with_a_nextint_rejection_equals_the_oracle(O, capi):
    """the CPU replay (test_oracle_bpr_strict) asserts this seed's first epoch reaches nextInt's rejection branch"""
    tr = rejection_csr(O)
    k = 2
    P, Q = _init(tr.U, tr.I, k, 1)
    with _handle(capi, k, seed=REJECTION_SEED) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        got = h.bpr_peek_samples(1, 0, tr.nnz)
        h.set_factors(P, Q)
        h.sgd_epoch(0.05, 0.01, 0.01, 0.0, 1)
        gP, gQ, _, _ = h.get_factors()
        gs = _state(h)
    want, _ = _oracle_samples(O, tr, seeded_state(REJECTION_SEED), tr.nnz)
    assert np.array_equal(got, want)
    oP, oQ, _, os_ = _oracle_epochs(O, tr, k, P, Q, seeded_state(REJECTION_SEED), 1, 0.05, 0.01, 0.01)
    assert _same(gP, oP) and _same(gQ, oQ) and gs == os_


def test_peeking_between_epochs_changes_nothing(O, capi, c1):
    tr = _ones(O, c1["train"])
    P, Q = _init(tr.U, tr.I, 8, 3)
    out = []
    for peek in (False, True):
        with _handle(capi, 8, seed=4) as h:
            h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
            h.set_factors(P, Q)
            h.sgd_epoch(*HYPER, 0.0, 1)
            s1 = _state(h)
            if peek:
                a = h.bpr_peek_samples(2, 0, 1000)
                assert _state(h) == s1
                assert np.array_equal(a, h.bpr_peek_samples(2, 0, 1000))
            h.sgd_epoch(*HYPER, 0.0, 2)
            out.append(h.get_factors()[:2] + (_state(h),))
    assert _same(out[0][0], out[1][0]) and _same(out[0][1], out[1][1]) and out[0][2] == out[1][2]


# ---- factors -------------------------------------------------------------------------------------------------------------
def test_c1_factors_and_state_equal_the_oracle_after_1_2_5_epochs(O, capi, c1):
    tr = _ones(O, c1["train"])
    k = 10
    P, Q = _init(tr.U, tr.I, k, 7)
    with _handle(capi, k, seed=1) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        got, losses = {}, []
        for it in range(1, 6):
            losses.append(h.sgd_epoch(*HYPER, 0.0, it))
            if it in (1, 2, 5):
                gP, gQ, _, _ = h.get_factors()
                got[it] = (gP, gQ, _state(h))
    for it in (1, 2, 5):
        oP, oQ, ol, os_ = _oracle_epochs(O, tr, k, P, Q, seeded_state(1), it)
        assert _same(got[it][0], oP) and _same(got[it][1], oQ) and got[it][2] == os_, it
    assert np.allclose(losses, ol, rtol=1e-12, atol=0)


@pytest.mark.parametrize("k", [1, 5, 32, 33, 64, 128, 256])
def test_random_csr_factors_equal_the_oracle(O, capi, k):
    tr = _mixed_csr(O, 300, 200, k, density=0.05)
    P, Q = _init(tr.U, tr.I, k, k)
    state = seeded_state(1000 + k)
    with _handle(capi, k) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        h.set_matrix("jdk.random.state", np.array([float(state)]))
        losses = [h.sgd_epoch(0.05, 0.01, 0.02, 0.0, it) for it in (1, 2)]
        gP, gQ, _, _ = h.get_factors()
        gs = _state(h)
    oP, oQ, ol, os_ = _oracle_epochs(O, tr, k, P, Q, state, 2, 0.05, 0.01, 0.02)
    assert _same(gP, oP) and _same(gQ, oQ) and gs == os_
    assert np.allclose(losses, ol, rtol=1e-12, atol=0)


def test_sgd_epochs_with_decay_equals_the_oracle_loop(O, capi, c1):
    tr = _ones(O, c1["train"])
    k = 16
    P, Q = _init(tr.U, tr.I, k, 11)
    with _handle(capi, k, seed=3) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        losses = h.sgd_epochs(3, 0.05, 0.01, 0.01, 0.0, 1, decay=0.9)
        gP, gQ, _, _ = h.get_factors()
        gs = _state(h)
    oP, oQ, ol, os_ = _oracle_epochs(O, tr, k, P, Q, seeded_state(3), 3, 0.05, 0.01, 0.01, decay=0.9)
    assert _same(gP, oP) and _same(gQ, oQ) and gs == os_
    assert np.allclose(losses, ol, rtol=1e-12, atol=0)


def test_topn_of_the_learned_factors_equals_the_oracle(O, capi, c1):
    tr = _ones(O, c1["train"])
    k = 10
    P, Q = _init(tr.U, tr.I, k, 5)
    with _handle(capi, k, seed=2) as h:
        h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
        h.set_factors(P, Q)
        for it in (1, 2):
            h.sgd_epoch(*HYPER, 0.0, it)
        items, scores, counts = h.topn(10)
        gP, gQ, _, _ = h.get_factors()
    oi, os_, oc = O.recommend_rank(O.BPR, tr.U, tr.I, k, gP, gQ, None, None, 0.0, tr, 10)
    assert np.array_equal(items, oi) and np.array_equal(counts, oc) and _same(scores, os_)


# ---- the job -------------------------------------------------------------------------------------------------------------
BPR_REF_PROPS = """
rec.recommender.class=bpr
rec.iterator.learnrate=0.01
rec.iterator.learnrate.maximum=0.01
rec.iterator.maximum=3
rec.user.regularization=0.01
rec.item.regularization=0.01
rec.factor.number=10
rec.recommender.isranking=true
rec.recommender.ranking.topn=10
rec.random.seed=1
rec.cuda.order=reference
"""


def test_job_equals_seed_gaussian_init_and_strict_epochs(O, capi, c1):
    from librec_b200.host import binding
    from librec_b200.host.binding import RecommenderJob
    H = binding.load()
    tr = _ones(O, c1["train"])
    job = RecommenderJob(BPR_REF_PROPS)
    job.set_data(tr.U, tr.I, tr, c1["test"])
    H.lrh_randoms_seed(1)                                     # set_data skips the splitter: the job starts right after the seed
    job.run_job()
    P, Q, _, _, _ = job.factors(10, False)
    O.lib().lro_seed(1)
    oP, oQ, _, _ = O.mf_setup(tr.U, tr.I, 10, False)          # MatrixFactorizationRecommender.setup's Gaussian init
    seed, have, nextg = C.c_uint64(), C.c_int32(), C.c_double()
    O.lib().lro_rng_get_state(C.byref(seed), C.byref(have), C.byref(nextg))
    L = bpr_strict.lib()
    L.lro_set_jrandom_state(seed.value)                       # the training continues the generator where the init left it
    for it in range(3):
        L.lro_bpr_epoch_strict(tr.U, tr.I, tr.rowptr, tr.col, 10, oP, oQ, 0.01, 0.01, 0.01, tr.nnz, None, None)
    assert _same(P, oP) and _same(Q, oQ)
    rng = JavaRandom(0)
    rng.s = L.lro_jrandom_state()
    assert H.lrh_randoms_uniform_int(1 << 30) == rng.next_int(1 << 30)       # the job handed the state back to Randoms


# ---- errors --------------------------------------------------------------------------------------------------------------
def test_no_drawable_user_is_an_error_not_a_hang(O, capi):
    U, I = 6, 4
    rowptr = np.array([0, 0, 4, 4, 8, 8, 8], np.int64)         # every row empty or full
    col = np.array([0, 1, 2, 3, 0, 1, 2, 3], np.int32)
    with _handle(capi, 4) as h:
        h.set_train_csr(U, I, rowptr, col, np.ones(8))
        with pytest.raises(capi.LibrecException):
            h.bpr_peek_samples(1, 0, 4)
        h.set_factors(np.zeros((U, 4)), np.zeros((I, 4)))
        with pytest.raises(capi.LibrecException):
            h.sgd_epoch(*HYPER, 0.0, 1)


def test_random_state_is_refused_elsewhere_and_out_of_range(O, capi):
    tr = rng_csr(O, 20, 10, 0.3, 1)
    for model, mode in ((capi.MODEL_BPR, capi.UPDATE_ATOMIC), (capi.MODEL_PMF, capi.UPDATE_REFERENCE_ORDER)):
        with capi.Handle(model, 4, update_mode=mode) as h:
            h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
            with pytest.raises(capi.LibrecException):
                h.set_matrix("jdk.random.state", np.array([5.0]))
            with pytest.raises(capi.LibrecException):
                h.get_matrix("jdk.random.state", (1,))
    with _handle(capi, 4) as h:
        for bad in (-1.0, 2.0 ** 48, 0.5, float("nan")):
            with pytest.raises(capi.LibrecException):
                h.set_matrix("jdk.random.state", np.array([bad]))
        h.set_matrix("jdk.random.state", np.array([2.0 ** 48 - 1]))
        assert _state(h) == 2 ** 48 - 1


# ---- SASS ----------------------------------------------------------------------------------------------------------------
def _functions(sass):
    out, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
        elif name and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            out[name].append(line)
    return out


def test_sass_has_dfma_only_inside_the_division_sequence(capi):
    """no FMA contraction: a DFMA appears only in the reciprocal refinement that follows MUFU.RCP64H (__ddiv_rn) or in the
    division's slow-path subroutine (the CALL.REL targets placed after the kernel's own code)"""
    from librec_b200 import _build
    cuobjdump = os.path.join(os.path.dirname(os.path.dirname(_build._nvcc())), "bin", "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", _build.LIB_PATH], stdout=subprocess.PIPE, text=True, check=True).stdout
    fns = {n: l for n, l in _functions(sass).items() if "bpr_ref_" in n}
    assert any("bpr_ref_update_kernel" in n for n in fns) and any("bpr_ref_parse_kernel" in n for n in fns)
    for name, lines in fns.items():
        addr = [int(re.search(r"/\*([0-9a-f]{4,})\*/", l).group(1), 16) for l in lines]
        calls = [int(m.group(1), 16) for l in lines for m in [re.search(r"CALL\.REL\S*\s+0x([0-9a-f]+)", l)] if m]
        sub_start = min(calls) if calls else None
        last_rcp = -10 ** 9
        for idx, (a, l) in enumerate(zip(addr, lines)):
            if "MUFU.RCP64H" in l:
                last_rcp = idx
            if re.search(r"\bDFMA\b", l):
                assert idx - last_rcp <= 12 or (sub_start is not None and a >= sub_start), (name, l)
        if "bpr_ref_update_kernel" not in name:
            assert not any(re.search(r"\bD(FMA|ADD|MUL)\b", l) for l in lines), name    # the draw stage is integer work
