"""Seeded synthetic rating matrices with the shapes BASELINE.json names (SURVEY.md 8d).

ML-20M shape: 138 493 users x 26 744 items, 20 000 263 ratings; Netflix shape: 480 189 x 17 770,
100 480 507 ratings.  User activity is log-normal, item popularity Zipf(1.0), ratings come from a
planted rank-16 model + biases + noise rounded to half stars, rows are sorted by item (CSR, like
SequentialAccessSparseMatrix).  Everything is numpy on the host; results are cached under
$LRK_CACHE (default lrk_synth-<uid> in the system's temporary directory) because generation takes tens of seconds.
The default is per user: a machine's other users can neither block the cache nor hand this one their files.
"""
import os
import tempfile

import numpy as np

SHAPES = {
    "ml-20m": (138493, 26744, 20000263, 0x4C520001),
    "netflix": (480189, 17770, 100480507, 0x4C520002),
    "ml-1m": (6040, 3706, 1000209, 0x4C520003),
    # one tenth of the Netflix shape's users over the same 17 770-item catalogue and popularity law: the at-scale parity case
    # the CPU oracle finishes in seconds per epoch (tests/parity_scale.py)
    "netflix-10m": (48019, 17770, 10048050, 0x4C520002),
    "tiny": (2000, 1500, 60000, 0x4C520004),
    # smallest shape whose top-N takes the tensor-core path (>= 512 users, >= 8192 items): __graft_entry__.smoke()
    "small": (4096, 8192, 400000, 0x4C520006),
}


def _cache_dir():
    d = os.environ.get("LRK_CACHE") or os.path.join(tempfile.gettempdir(), "lrk_synth-%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    return d


def make_ratings(shape="ml-20m", binary=False, cache=True, shard=0, zipf=1.0):
    """-> dict(U, I, rowptr int64[U+1], col int32[nnz], val float64[nnz]) ; exactly SHAPES[shape] nnz.
    `shard` selects an independent block of users over the SAME item catalogue (same popularity and
    planted item factors) -- the per-rank user shard of the weak-scaling DSGD runs.  `zipf` is the exponent of the item
    popularity law (1.0 = the survey's generator; 0.5 gives the flatter head of real MovieLens data)."""
    U, I, nnz, seed = SHAPES[shape]
    tag = "" if zipf == 1.0 else "_z%g" % zipf
    path = os.path.join(_cache_dir(), "%s_%s_s%d%s.npz" % (shape, "bin" if binary else "rat", shard, tag))
    if cache and os.path.exists(path):
        z = np.load(path)
        return {"U": U, "I": I, "rowptr": z["rowptr"], "col": z["col"], "val": z["val"].astype(np.float64)}
    rng_items = np.random.default_rng(seed)               # shared by all shards
    rng = np.random.default_rng([seed, shard])            # user side of this shard
    # user activity: log-normal, clipped to [20, I/2], rescaled to the target total
    deg = np.exp(rng.normal(0.0, 1.0, U))
    deg = deg / deg.sum() * nnz
    deg = np.clip(deg, min(20, nnz / U), I / 2)
    deg = deg / deg.sum() * nnz
    # item popularity: Zipf(1.0) over a random permutation of item ids
    pop = 1.0 / np.arange(1, I + 1, dtype=np.float64) ** zipf
    pop = pop[rng_items.permutation(I)]
    cdf = np.cumsum(pop / pop.sum())
    keys = np.zeros(0, np.int64)
    over = 1.9
    while True:
        cnt = rng.poisson(deg * over).astype(np.int64)
        u = np.repeat(np.arange(U, dtype=np.int64), cnt)
        i = np.searchsorted(cdf, rng.random(u.shape[0], dtype=np.float32).astype(np.float64), side="right").astype(np.int64)
        i = np.minimum(i, I - 1)
        keys = np.sort(np.concatenate([keys, u * I + i]))
        keys = keys[np.concatenate([[True], keys[1:] != keys[:-1]])]      # unique of a sorted array
        if keys.shape[0] >= nnz:
            break
        over = 2.0 * (nnz - keys.shape[0]) / nnz + 0.05
    if keys.shape[0] > nnz:
        drop = rng.choice(keys.shape[0], keys.shape[0] - nnz, replace=False)
        mask = np.ones(keys.shape[0], bool)
        mask[drop] = False
        keys = keys[mask]
    u = (keys // I).astype(np.int64)
    col = (keys % I).astype(np.int32)
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(u, minlength=U))]).astype(np.int64)
    if binary:
        val = np.ones(nnz, np.float32)
    else:
        r = 16
        ps = rng.normal(0, 1.0, (U, r)).astype(np.float32)
        qs = rng_items.normal(0, 1.0, (I, r)).astype(np.float32)
        bu = rng.normal(0, 0.3, U).astype(np.float32)
        bi = rng_items.normal(0, 0.3, I).astype(np.float32)
        val = np.empty(nnz, np.float32)
        step = 1 << 22
        for a in range(0, nnz, step):
            uu, ii = u[a:a + step], col[a:a + step]
            x = 3.5 + bu[uu] + bi[ii] + 0.125 * np.einsum("ij,ij->i", ps[uu], qs[ii]) + rng.normal(0, 0.5, uu.shape[0]).astype(np.float32)
            val[a:a + step] = np.clip(np.round(x * 2.0) / 2.0, 0.5, 5.0)
    if cache:
        tmp = path + ".tmp.%d.npz" % os.getpid()
        np.savez(tmp, rowptr=rowptr, col=col, val=val)
        os.replace(tmp, path)
    return {"U": U, "I": I, "rowptr": rowptr, "col": col, "val": val.astype(np.float64)}


def init_factors(U, I, k, seed, biased):
    """N(0, 0.001^2) like MatrixFactorizationRecommender.setup (:86-93) -- numpy RNG, not java.util.Random"""
    rng = np.random.default_rng(seed)
    sd = float(np.float32(0.001))
    P = rng.normal(0.0, sd, (U, k))
    Q = rng.normal(0.0, sd, (I, k))
    bu = rng.normal(0.0, sd, U) if biased else None
    bi = rng.normal(0.0, sd, I) if biased else None
    return P, Q, bu, bi
