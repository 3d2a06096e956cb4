"""GPU: the staged COO stream of the SGD epoch equals its restatement (librec_b200/dsgd_plan.py, stream_order) bit for bit, and
lrk_stage_stats reports its run tiles and largest item degree, for every model whose epoch reads the stream.  The DSGD rank's
stream (block bits, block-local ids, seed + 977 * rank) is checked by tests/dsgd_gpu_check.py."""
import numpy as np
import pytest

from librec_b200.dsgd_plan import RUN_MIN_DEGREE, stream_order

pytestmark = pytest.mark.gpu

SEED = 5


def _csr(dense, seed):
    rows, cols = np.nonzero(dense)
    rowptr = np.zeros(dense.shape[0] + 1, np.int64)
    np.add.at(rowptr, rows + 1, 1)
    val = np.random.default_rng(seed).random(rows.shape[0]) * 5.0
    return np.cumsum(rowptr), cols.astype(np.int32), val


def _degrees(U, degs, extra_items, density, seed):
    """items 0..len(degs)-1 with exactly those degrees (random users), then extra_items random ones"""
    rng = np.random.default_rng(seed)
    dense = np.zeros((U, len(degs) + extra_items), bool)
    for i, d in enumerate(degs):
        dense[rng.choice(U, d, replace=False), i] = True
    dense[:, len(degs):] = rng.random((U, extra_items)) < density
    return dense


MATRICES = {
    # around the run threshold, a degree that is not a multiple of 32, an item rated by every user, items with no rating
    "degrees": lambda: _degrees(300, [RUN_MIN_DEGREE - 1, RUN_MIN_DEGREE, RUN_MIN_DEGREE + 1, 200, 300, 0, 31, 0], 40, 0.05, 1),
    "single_item": lambda: _degrees(260, [170], 0, 0.0, 2),
    "skewed": lambda: np.random.default_rng(3).random((1500, 700)) < np.linspace(0.4, 0.002, 700)[None, :],
    "empty": lambda: np.zeros((7, 5), bool),
}


def _stage(capi, model, dense, seed):
    U, I = dense.shape
    rowptr, col, val = _csr(dense, seed)
    h = capi.Handle(model, 16, seed=SEED)
    h.set_train_csr(U, I, rowptr, col, val)
    return h, (rowptr, col, val, I)


def _check(h, rowptr, col, val, I):
    su, si, sr, run_tiles, max_deg = stream_order(rowptr, col, val, I, SEED)
    n = col.shape[0]
    gu, gi, gr, units = h.debug_stream(n)
    assert units is None
    assert np.array_equal(gu, su) and np.array_equal(gi, si) and np.array_equal(gr.view(np.int32), sr.view(np.int32))
    st = h.stage_stats()
    assert (st["ratings"], st["run_tile_ratings"], st["max_item_degree"], st["run_min_degree"]) == (n, 32 * run_tiles, max_deg, RUN_MIN_DEGREE)


@pytest.mark.parametrize("name", sorted(MATRICES))
@pytest.mark.parametrize("model", ["MODEL_BIASEDMF", "MODEL_PMF", "MODEL_RANKSGD", "MODEL_AOBPR"])
def test_stream_order(capi, model, name):
    dense = MATRICES[name]()
    h, csr = _stage(capi, getattr(capi, model), dense, 11)
    with h:
        _check(h, *csr)
    if name == "degrees":        # the case exercises what it names: run tiles, and ratings outside them
        assert csr[0][-1] > 32 * stream_order(*csr, SEED)[3] > 0


def test_restage_empty(capi):
    """a handle restaged with an empty matrix reports what a fresh handle reports for it"""
    full, empty = MATRICES["degrees"](), np.zeros((300, 48), bool)
    h, csr = _stage(capi, capi.MODEL_BIASEDMF, full, 11)
    with h:
        assert h.stage_stats()["run_tile_ratings"] > 0
        h.set_train_csr(300, 48, *_csr(empty, 12))
        fresh, _ = _stage(capi, capi.MODEL_BIASEDMF, empty, 12)
        with fresh:
            assert h.stage_stats() == fresh.stage_stats()
            assert h.stage_stats()["max_item_degree"] == 0 and h.stage_stats()["run_tile_ratings"] == 0
