"""GPU: every exact top-N path of lrk_topn against the oracle, bit for bit, up to N = 512 and k = 256.

topn_to_device picks one of three paths (include/librec_b200.h, DESIGN.md section 4.4):
  warp-per-user heap replay   topn_exact_kernel: 1 launch
  item-parallel exact         topn_exact_parts_kernel + topn_exact_merge_kernel + the tie collector: 3 launches,
                              plus 2 (topn_exact_kernel + scatter) when some user has a tie among its first N+1 scores
  tensor-core sweep           topn_tc.cuh: reports fast_users > 0
The item-parallel path serves a users array of at most 4 x SMs users over a catalogue of 32768 items or more, as long as
its 3072 (N+1) + 8k + 128 bytes of lists fit a block's shared memory.  The warp-per-user kernel keeps its heaps in shared
memory while 512k + 256 + 384N bytes fit, in global memory beyond.  The cases sit on each side of each of these limits;
each asserts the path it exercises through the launch count."""
import numpy as np
import pytest

from conftest import rng_csr

pytestmark = pytest.mark.gpu

MU = 3.53


@pytest.fixture(scope="module")
def dev(capi):
    """(SM count, opt-in shared memory per block) of device 0"""
    import torch
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.shared_memory_per_block_optin


def _parts_smem(k, N):
    return 8 * (k + 256 * (N + 1) + 8) + 4 * (256 * (N + 1) + 16)


def _launches(dev, k, N, I, nq, explicit):
    """launches of an automatic (topn_path=0) exact call without ties"""
    sms, optin = dev
    return 3 if explicit and nq <= 4 * sms and I >= 32768 and _parts_smem(k, N) <= optin else 1


def _topn(h, N, **kw):
    n0 = h.launch_count()
    out = h.topn(N, **kw)
    return out, h.launch_count() - n0


def _train(O, U, I, density, seed, N):
    """random train CSR; user 1 rated all but N // 2 items (fewer candidates than N), user 2 rated every item"""
    rng = np.random.default_rng(seed)
    mask = rng.random((U, I)) < density
    mask[1] = True
    mask[1, rng.choice(I, N // 2, replace=False)] = False
    mask[2] = True
    rows, cols = np.nonzero(mask)
    rowptr = np.zeros(U + 1, np.int64)
    np.add.at(rowptr, rows + 1, 1)
    return O.Csr(U, I, np.cumsum(rowptr), cols.astype(np.int32), np.ones(rows.shape[0]))


def _users(U, nq, seed):
    """nq query slots with users 1 and 2 and a duplicate"""
    rng = np.random.default_rng(seed)
    return np.concatenate([[1, 2], rng.integers(0, U, nq - 3), [1]]).astype(np.int32)


def _factors(U, I, k, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(0, 0.1, (U, k)), rng.normal(0, 0.1, (I, k)), rng.normal(0, 0.1, U), rng.normal(0, 0.1, I)


def _handle(capi, name, k, tr, P, Q, bu, bi, mu=MU, **kw):
    """biases and a global mean go to every model, as the Java shim passes them: the unbiased ones must ignore them"""
    h = capi.Handle(getattr(capi, "MODEL_" + name.upper()), k, **kw)
    h.set_train_csr(tr.U, tr.I, tr.rowptr, tr.col, tr.val)
    h.set_factors(P, Q, bu, bi, mu)
    return h


def _reference(O, name, k, P, Q, bu, bi, tr, N, users, exclude_train=True):
    """recommendRank of the reference; GBPR predicts b_i + p.q (BiasedMF with b_u = mu = 0, pinned by
    tests/test_oracle_gbpr.py), WRMF scores like PMF"""
    U, I = P.shape[0], Q.shape[0]
    t = tr if exclude_train else None
    if name == "biasedmf":
        return O.recommend_rank(O.BIASEDMF, U, I, k, P, Q, bu, bi, MU, t, N, users=users)
    if name == "gbpr":
        return O.recommend_rank(O.BIASEDMF, U, I, k, P, Q, np.zeros(U), bi, 0.0, t, N, users=users)
    return O.recommend_rank(O.BPR if name == "bpr" else O.PMF, U, I, k, P, Q, None, None, 0.0, t, N, users=users)


def _assert_same(got, exp):
    (gi, gs, gc), (ei, es, ec) = got, exp
    assert np.array_equal(gc, ec)
    assert np.array_equal(gi, ei)
    assert np.array_equal(gs.view(np.int64), es.view(np.int64))


# (model, k, N, I, nq): both sides of the warp-per-user kernel's shared-memory limit 512k + 256 + 384N
# (k = 256: N <= 263; k = 128: N <= 434; N = 512: k <= 69)
WARP_CASES = [
    ("pmf", 1, 1, 700, 40),
    ("biasedmf", 20, 26, 1500, 60),
    ("bpr", 20, 27, 1500, 60),
    ("pmf", 128, 100, 1000, 40),
    ("wrmf", 112, 100, 1500, 40),
    ("biasedmf", 256, 263, 1200, 24),
    ("pmf", 256, 264, 1200, 24),
    ("gbpr", 256, 300, 1200, 16),
    ("bpr", 128, 434, 1500, 40),
    ("biasedmf", 128, 435, 1500, 40),
    ("pmf", 69, 512, 2000, 40),
    ("bpr", 70, 512, 2000, 40),
    ("biasedmf", 256, 512, 2000, 24),
]


@pytest.mark.parametrize("name,k,N,I,nq", WARP_CASES, ids=["%s-k%d-N%d" % c[:3] for c in WARP_CASES])
def test_warp_per_user_path(O, capi, name, k, N, I, nq):
    U = nq + 8
    tr = _train(O, U, I, 0.05, k + N, N)
    P, Q, bu, bi = _factors(U, I, k, k * N)
    users = _users(U, nq, N)
    with _handle(capi, name, k, tr, P, Q, bu, bi, topn_path=1) as h:
        first, n_first = _topn(h, N, nq=nq)
        listed, n_listed = _topn(h, N, users=users)
    assert n_first == 1 and n_listed == 1
    _assert_same(first, _reference(O, name, k, P, Q, bu, bi, tr, N, np.arange(nq)))
    _assert_same(listed, _reference(O, name, k, P, Q, bu, bi, tr, N, users))


# (model, k, N, I, nq) through the automatic choice with a users array over I >= 32768: both sides of the item-parallel
# path's shared-memory limit 3072 (N+1) + 8k + 128 (N <= 73; N = 74 for k <= 240), and beyond it the warp-per-user
# kernel on both sides of its own limit
AUTO_CASES = [
    ("pmf", 1, 1, 32768, 40),
    ("biasedmf", 20, 26, 40077, 100),      # 40077 = 156 x 256 + 141: the last item part is partial
    ("bpr", 20, 27, 32768, 60),
    ("wrmf", 64, 26, 32768, 40),
    ("biasedmf", 256, 73, 32768, 16),
    ("pmf", 256, 74, 32768, 16),
    ("bpr", 128, 74, 32768, 24),
    ("gbpr", 32, 74, 32768, 24),
    ("biasedmf", 69, 75, 32768, 24),
    ("pmf", 70, 100, 32768, 24),
    ("bpr", 128, 263, 32768, 16),
    ("biasedmf", 256, 264, 32768, 16),
    ("pmf", 128, 435, 32768, 16),
    ("pmf", 69, 512, 32768, 16),
    ("bpr", 70, 512, 32768, 16),
]


@pytest.mark.parametrize("name,k,N,I,nq", AUTO_CASES, ids=["%s-k%d-N%d-I%d" % c[:4] for c in AUTO_CASES])
def test_automatic_exact_path(O, capi, dev, name, k, N, I, nq):
    U = 200
    tr = _train(O, U, I, 0.002, k + N, N)
    P, Q, bu, bi = _factors(U, I, k, k * N + 1)
    users = _users(U, nq, N)
    with _handle(capi, name, k, tr, P, Q, bu, bi, topn_path=0) as h:
        got, n = _topn(h, N, users=users)
    assert n == _launches(dev, k, N, I, nq, True)
    _assert_same(got, _reference(O, name, k, P, Q, bu, bi, tr, N, users))


@pytest.mark.parametrize("I", [32767, 32768, 32845])
def test_catalogue_size_boundary(O, capi, dev, I):
    U, k, N, nq = 120, 20, 10, 50
    tr = _train(O, U, I, 0.003, I, N)
    P, Q, bu, bi = _factors(U, I, k, I)
    users = _users(U, nq, 3)
    with _handle(capi, "pmf", k, tr, P, Q, bu, bi) as h:
        got, n = _topn(h, N, users=users)
    assert n == (1 if I < 32768 else 3) == _launches(dev, k, N, I, nq, True)
    _assert_same(got, _reference(O, "pmf", k, P, Q, bu, bi, tr, N, users))


@pytest.mark.parametrize("extra", [0, 1])
def test_query_count_boundary(O, capi, dev, extra):
    """4 x SMs queried users take the item-parallel path, one more the warp-per-user kernel (N = 27 keeps the
    tensor-core path out of the choice)"""
    sms = dev[0]
    nq, U, I, k, N = 4 * sms + extra, 4 * sms + 16, 32768, 8, 27
    tr = _train(O, U, I, 0.001, 5 + extra, N)
    P, Q, bu, bi = _factors(U, I, k, 6)
    users = _users(U, nq, 7)
    with _handle(capi, "bpr", k, tr, P, Q, bu, bi) as h:
        got, n = _topn(h, N, users=users)
    assert n == (3 if extra == 0 else 1) == _launches(dev, k, N, I, nq, True)
    _assert_same(got, _reference(O, "bpr", k, P, Q, bu, bi, tr, N, users))


def test_users_array_or_none(O, capi, dev):
    """without a users array (the first nq users) the warp-per-user kernel serves the call; with one, duplicates
    included, the item-parallel path"""
    U, I, k, N, nq = 100, 32768, 16, 10, 40
    tr = _train(O, U, I, 0.002, 8, N)
    P, Q, bu, bi = _factors(U, I, k, 9)
    users = _users(U, nq, 10)
    with _handle(capi, "biasedmf", k, tr, P, Q, bu, bi) as h:
        first, n_first = _topn(h, N, nq=nq)
        listed, n_listed = _topn(h, N, users=users)
    assert n_first == 1 and n_listed == 3 == _launches(dev, k, N, I, nq, True)
    _assert_same(first, _reference(O, "biasedmf", k, P, Q, bu, bi, tr, N, np.arange(nq)))
    _assert_same(listed, _reference(O, "biasedmf", k, P, Q, bu, bi, tr, N, users))


def test_item_parallel_ties_nan_inf_and_short_rows(O, capi, dev):
    """equal item rows in different item parts (a tie across a part boundary), NaN rows (dropped), two +Inf items (a tie),
    a user with fewer candidates than N and one with none: the tie replay runs and the lists still match"""
    U, I, k, N, nq = 64, 32768 + 300, 16, 20, 40
    rng = np.random.default_rng(12)
    P, Q = rng.normal(0, 0.1, (U, k)), rng.normal(0, 0.1, (I, k))
    # nq = 40 on 148 SMs -> 8 parts of 4352 items (the last one 2604): items 100, 10000 and 33000 are in parts 0, 2 and 7
    Q[[100, 10000, 33000]] = 5.0                          # top of the list, tied, for every user whose row sums to > 0
    Q[[5000, 20000]] = np.nan
    Q[[15000, 25000]] = 0.0
    Q[[15000, 25000], 0] = np.inf                         # +Inf for users with p_0 > 0 (-Inf otherwise)
    open_items = np.array([3, 50, 400, 9000, 17000, 26000, I - 1])
    mask = rng.random((U, I)) < 0.002
    mask[1] = True
    mask[1, open_items] = False                           # user 1: 7 candidates < N
    mask[2] = True                                        # user 2: none
    rows, cols = np.nonzero(mask)
    rowptr = np.zeros(U + 1, np.int64)
    np.add.at(rowptr, rows + 1, 1)
    tr = O.Csr(U, I, np.cumsum(rowptr), cols.astype(np.int32), np.ones(rows.shape[0]))
    users = _users(U, nq, 13)
    assert _launches(dev, k, N, I, nq, True) == 3
    with _handle(capi, "pmf", k, tr, P, Q, None, None, 0.0) as h:
        got, n = _topn(h, N, users=users)
        noex, n_noex = _topn(h, N, users=users, exclude_train=False)
    assert n == 5 and n_noex == 5                          # parts, merge, tie collection + the replay and its scatter
    exp = _reference(O, "pmf", k, P, Q, None, None, tr, N, users)
    assert exp[2][0] == 7 and exp[2][1] == 0
    _assert_same(got, exp)
    _assert_same(noex, _reference(O, "pmf", k, P, Q, None, None, tr, N, users, exclude_train=False))


def test_multi_handle_matches_plain_handle(O, capi, dev):
    """a one-device multi-device handle serves top-N from its child, which chooses its path like a plain handle"""
    U, I, k, nq = 300, 32768 + 1000, 24, 50
    tr = _train(O, U, I, 0.002, 14, 100)
    P, Q, bu, bi = _factors(U, I, k, 15)
    users = _users(U, nq, 16)
    with _handle(capi, "biasedmf", k, tr, P, Q, bu, bi, devices=[0]) as m, _handle(capi, "biasedmf", k, tr, P, Q, bu, bi) as h:
        for N in (10, 100):
            m.topn(N, users=users)                       # the first call brings the child's masters up to date
            got, n = _topn(m, N, users=users)
            plain, n_plain = _topn(h, N, users=users)
            assert n == n_plain == _launches(dev, k, N, I, nq, True)
            _assert_same(got, plain)
            _assert_same(got, _reference(O, "biasedmf", k, P, Q, bu, bi, tr, N, users))


def test_gbpr_ignores_global_mean_and_user_biases(O, capi, dev):
    """GBPR predicts b_i + p_u.q_i (GBPRRecommender.java:194-196).  The Java shim passes the train mean to every model and
    lrk_set_factors takes user biases: a GBPR handle keeps neither, so top-N on all three paths, predict_pairs and
    eval_ranking equal the reference"""
    U, I, k, N = 600, 32768, 32, 10
    rng = np.random.default_rng(17)
    full = rng_csr(O, U, I, 0.003, 18)
    in_train = rng.random(full.nnz) < 0.8
    tr, te = full.select(in_train), full.select(~in_train)
    P, Q, bu, bi = _factors(U, I, k, 19)
    users = _users(U, 200, 20)
    ref = _reference(O, "gbpr", k, P, Q, bu, bi, tr, N, None)
    with _handle(capi, "gbpr", k, tr, P, Q, bu, bi, mu=3.7, topn_path=0) as h:
        first, n_first = _topn(h, N, nq=100)
        listed, n_listed = _topn(h, N, users=users)
        us, its = rng.integers(0, U, 4000).astype(np.int32), rng.integers(0, I, 4000).astype(np.int32)
        pred = h.predict_pairs(us, its)
        measures, lists = h.eval_ranking(N, te.rowptr, te.col, te.val, want_lists=True)
        gbu = h.get_factors()[2]
    with _handle(capi, "gbpr", k, tr, P, Q, bu, bi, mu=3.7, topn_path=2) as h2:
        tc = h2.topn(N)
        stats = h2.topn_stats()
    assert n_first == 1 and n_listed == 3 == _launches(dev, k, N, I, 200, True)
    _assert_same(first, tuple(a[:100] for a in ref))
    _assert_same(listed, tuple(a[users] for a in ref))
    assert stats["fast_users"] > 0, stats
    _assert_same(tc, ref)
    exp, zero_bu = np.zeros(4000), np.zeros(U)
    O.lib().lro_predict_pairs(O.BIASEDMF, k, P, Q, zero_bu.ctypes.data, bi.ctypes.data, 0.0, us, its, 4000, exp)
    assert np.array_equal(pred.view(np.int64), exp.view(np.int64))
    _assert_same(lists, ref)
    exp_m = O.eval_ranking(te, tr, N, ref[0], ref[2])
    for name in O.RANKING_MEASURES:
        assert abs(measures[name] - exp_m[name]) <= 1e-12 * max(1.0, abs(exp_m[name])), (name, measures[name], exp_m[name])
    assert np.all(gbu == 0.0)
