"""GPU: an entry point called again on the same handle, with larger inputs, returns exactly what a fresh handle returns for
the larger call.  The device buffers behind these calls (staging arena, per-state buffers) are kept between calls and reused
when large enough: a buffer that is sized for the first call, or read before it is rewritten, shows up here."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _csr(U, I, density, seed):
    """random CSR with ascending columns per row and ratings 1..5"""
    rng = np.random.default_rng(seed)
    rows, cols = np.nonzero(rng.random((U, I)) < density)
    rowptr = np.zeros(U + 1, np.int64)
    np.add.at(rowptr, rows + 1, 1)
    return np.cumsum(rowptr), cols.astype(np.int32), rng.integers(1, 6, rows.shape[0]).astype(np.float64)


def _factors(U, I, k, seed, scale=0.1):
    rng = np.random.default_rng(seed)
    return rng.normal(0, scale, (U, k)), rng.normal(0, scale, (I, k)), rng.normal(0, scale, U), rng.normal(0, scale, I)


@pytest.fixture
def pair(capi):
    """pair(model, k, small, large, ...) -> (h, fresh): h is staged with the small and then the large train matrix, fresh with
    the large one only, and both get the same factors.  A matrix is (U, I, density, seed).  The handles close after the test."""
    made = []

    def make(model, k, small, large, Q=None, params=(), **kw):
        for shapes in ((small, large), (large,)):
            h = capi.Handle(model, k, **kw)
            made.append(h)
            for name, value in params:
                h.set_param(name, value)
            for U, I, density, seed in shapes:
                h.set_train_csr(U, I, *_csr(U, I, density, seed))
            P, Q0, bu, bi = _factors(large[0], large[1], k, 7)
            h.set_factors(P, Q0 if Q is None else Q, bu, bi, 3.5)
        return made[-2:]

    yield make
    for h in made:
        h.close()


def _same(a, b):
    a, b = np.atleast_1d(a), np.atleast_1d(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def test_eval_rating_reuse(capi, pair):
    U, I = 500, 800
    h, fresh = pair(capi.MODEL_BIASEDMF, 32, (200, 300, 0.02, 1), (U, I, 0.02, 2))
    small, large = _csr(U, I, 0.01, 11), _csr(U, I, 0.08, 12)
    h.eval_rating(U, *small, 1.0, 5.0, want_pred=True)
    got, want = h.eval_rating(U, *large, 1.0, 5.0, want_pred=True), fresh.eval_rating(U, *large, 1.0, 5.0, want_pred=True)
    assert all(_same(g, w) for g, w in zip(got, want))


@pytest.mark.parametrize("topn_path", [0, 1, 2])
def test_topn_reuse(capi, pair, topn_path):
    # I >= 32768 and at most 4 x SMs queried users: the automatic choice (0) takes the item-parallel exact path.
    # Duplicated item rows of an unbiased model give exact score ties, which the tensor-core path (2) hands to that same exact path.
    U, I, k = 2048, 32768, 32
    Q = _factors(U, I, k, 3)[1]
    Q[1::2] = Q[::2]
    h, fresh = pair(capi.MODEL_PMF, k, (300, 1000, 0.01, 3), (U, I, 0.002, 4), Q=Q, topn_path=topn_path)
    users = np.random.default_rng(4).permutation(U).astype(np.int32)
    h.topn(5, users=users[:64])
    assert all(_same(g, w) for g, w in zip(h.topn(10, users=users[:400]), fresh.topn(10, users=users[:400])))


def test_eval_ranking_reuse(capi, pair):
    U, I = 600, 2000
    h, fresh = pair(capi.MODEL_BPR, 32, (200, 300, 0.02, 1), (U, I, 0.02, 2))
    small, large = _csr(U, I, 0.002, 21), _csr(U, I, 0.02, 22)
    h.eval_ranking(5, *small, want_lists=True)
    got_m, got_l = h.eval_ranking(20, *large, want_lists=True)
    want_m, want_l = fresh.eval_ranking(20, *large, want_lists=True)
    assert all(_same(got_m[m], want_m[m]) for m in want_m) and all(_same(g, w) for g, w in zip(got_l, want_l))


@pytest.mark.parametrize("model", ["BPR", "GBPR", "RANKSGD", "AOBPR"])
def test_peek_samples_reuse(capi, pair, model):
    # AoBPR's draws read the factor rankings: sample draws are compared instead of its (atomically updated) factors
    params = (("aobpr.lambda", 0.1),) if model == "AOBPR" else ()
    h, fresh = pair(getattr(capi, "MODEL_" + model), 32, (200, 300, 0.02, 31), (700, 900, 0.03, 32), params=params)
    h.bpr_peek_samples(1, 0, 100)
    assert _same(h.bpr_peek_samples(2, 5, 4000), fresh.bpr_peek_samples(2, 5, 4000))


@pytest.mark.parametrize("model,update_mode", [("BIASEDMF", 2), ("WRMF", 0)])
def test_restage_then_epoch_reuse(capi, pair, model, update_mode):
    # reference-order BiasedMF and WRMF factors are bit-exact from run to run
    h, fresh = pair(getattr(capi, "MODEL_" + model), 16, (120, 90, 0.05, 41), (300, 200, 0.05, 42), update_mode=update_mode)
    for it in range(2):
        h.sgd_epoch(0.01, 0.05, 0.05, 0.05, it + 1)
        fresh.sgd_epoch(0.01, 0.05, 0.05, 0.05, it + 1)
    assert all(_same(g, w) for g, w in zip(h.get_factors(), fresh.get_factors()) if w is not None)


@pytest.mark.parametrize("group", [False, True])
def test_restage_stream_reuse(capi, pair, monkeypatch, group):
    # the staged stream of BiasedMF: item-run tiles by default; with LRK_SGD_GROUP=1 the unit-ordered stream of the user-group
    # kernel and its unit table
    if group:
        monkeypatch.setenv("LRK_SGD_GROUP", "1")
    h, fresh = pair(capi.MODEL_BIASEDMF, 64, (200, 300, 0.05, 51), (900, 1200, 0.05, 52))
    nnz = h.stage_stats()["ratings"]
    (su, si, sr, units), want = h.debug_stream(nnz), fresh.debug_stream(nnz)
    assert (units is not None) == group and (want[3] is not None) == group
    assert _same(su, want[0]) and _same(si, want[1]) and _same(sr, want[2]) and (not group or _same(units, want[3]))
