"""Multi-GPU DSGD parity check -- run under torchrun with one rank per GPU:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tests/dsgd_gpu_check.py
(1) conflict-free matrix: one DSGD epoch == the oracle's epoch up to fp32 rounding;
(2) config C1 (seeded ml-100k split, biasedmf-test.properties): RMSE / MAE within 1e-3 of the oracle;
(3) BPR across ranks (every rank keeps the full item matrix and samples like the reference over the whole catalogue; the change
    of the item matrix is all-reduced 8 times per epoch, csrc/dsgd.cuh dsgd_bpr_epoch): Precision@10 on the binarised C1 split at
    least 90 % of the single-GPU BPR of the same library (r01's stratified sampler reached 0.225 / 0.142 on 2 / 8 ranks vs 0.325).
(4) an invalid CSR shard on one rank fails on every rank; (5) BPR on a catalogue as small as the world size does not hang;
(6) every rank's staged stream and lrk_stage_stats equal the restatement of librec_b200/dsgd_plan.py (stream_order).
Prints "DSGD-CHECK OK" on rank 0.  `--fused` runs the same checks through the experimental fused epoch kernel.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


import dsgd_checks
from dsgd_checks import run_dsgd as _run_dsgd


def run_dsgd(capi, dist, torch, O, model, full, k, P, Q, bu, bi, mu, hyper, iters, rank, world, local):
    return _run_dsgd(capi, dist, O, model, full, k, P, Q, bu, bi, mu, hyper, iters, rank, world, local)[:5]


def main():
    if "--fused" in sys.argv:                      # opt-in: the experimental one-kernel epoch (csrc/dsgd_fused.cuh)
        os.environ["LRK_DSGD_FUSED"] = "1"
    import torch
    import torch.distributed as dist
    from librec_b200 import capi
    from oracle import oracle as O
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    capi.load()

    r1 = dsgd_checks.conflict_free(capi, dist, O, rank, world, local)
    ok1 = r1["ok"]
    r2 = dsgd_checks.c1(capi, dist, O, rank, world, local)
    ok2 = r2["ok"]
    z, tr, te, pins = dsgd_checks.load_c1(O)
    # (3) BPR: stratified DSGD vs one GPU, Precision@10 of the exact top-10 lists against the test split
    def precision_at_10(gP, gQ):
        users = np.flatnonzero(np.diff(te.rowptr) > 0).astype(np.int32)
        items, _, counts = O.recommend_rank(O.BPR, tr.U, tr.I, 32, gP, gQ, None, None, 0.0, tr, 10, users=users)
        hits = 0
        for r, u in enumerate(users):
            hits += np.intersect1d(items[r, :counts[r]], te.col[te.rowptr[u]:te.rowptr[u + 1]]).shape[0]
        return hits / (10.0 * users.shape[0])
    rng = np.random.default_rng(11)
    Pb, Qb = rng.normal(0, 0.01, (tr.U, 32)), rng.normal(0, 0.01, (tr.I, 32))
    ones = O.Csr(tr.U, tr.I, tr.rowptr, tr.col, np.ones_like(tr.val))
    gP, gQ, _, _, bl = run_dsgd(capi, dist, torch, O, capi.MODEL_BPR, ones, 32, Pb, Qb, None, None, 0.0,
                                (0.05, 0.01, 0.01, 0.0), 30, rank, world, local)
    prec_dsgd = prec_one = 0.0
    if rank == 0:
        with capi.Handle(capi.MODEL_BPR, 32, device=local, seed=1) as h1:
            h1.set_train_csr(ones.U, ones.I, ones.rowptr, ones.col, ones.val)
            h1.set_factors(Pb, Qb)
            l1 = [h1.sgd_epoch(0.05, 0.01, 0.01, 0.0, it + 1) for it in range(30)]
            sP, sQ, _, _ = h1.get_factors()
        prec_dsgd, prec_one = precision_at_10(gP, gQ), precision_at_10(sP, sQ)
        print("BPR DSGD world=%d: P@10 %.4f (one GPU %.4f)  loss_30 %.1f (one GPU %.1f)" % (world, prec_dsgd, prec_one, bl[-1], l1[-1]))
    ok3 = rank != 0 or (prec_dsgd > 0.1 and prec_dsgd >= 0.9 * prec_one)
    ok2 = ok2 and ok3
    # (4) ADVICE r01: an invalid CSR on ONE rank must fail on EVERY rank with LRK_ERR_INVALID (no rank left waiting in NCCL)
    sh = dsgd_checks.shard_rows(tr.U, world)
    mine = dsgd_checks.local_csr(O, tr, sh[rank], sh[rank + 1])
    bad_col = mine.col.copy()
    if rank == world - 1 and bad_col.shape[0]:
        bad_col[0] = tr.I + 7
    h4 = capi.Handle(capi.MODEL_BIASEDMF, 8, device=local, seed=1)
    uid = [capi.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h4.comm_init(rank, world, uid[0])
    try:
        h4.set_train_csr(mine.U, mine.I, mine.rowptr, bad_col, mine.val)
        ok4 = False
    except capi.LibrecException as e:
        ok4 = e.status == capi.ERR_INVALID and "column index out of range" in str(e)
    h4.close()
    # (5) ADVICE r01: a BPR stratum in which no local user has both a positive and a free negative must be skipped, not spin:
    #     I == world -> every item block has width 1
    n5 = 64
    rng5 = np.random.default_rng(5)
    dense = (rng5.random((n5, world)) < 0.6)
    dense[:, 0] |= ~dense.any(axis=1)
    r5, c5 = np.nonzero(dense)
    rp5 = np.zeros(n5 + 1, np.int64); np.add.at(rp5, r5 + 1, 1)
    tiny = O.Csr(n5, world, np.cumsum(rp5), c5.astype(np.int32), np.ones(r5.shape[0]))
    P5, Q5 = rng5.normal(0, 0.1, (n5, 8)), rng5.normal(0, 0.1, (world, 8))
    gP5, gQ5, _, _, l5 = run_dsgd(capi, dist, torch, O, capi.MODEL_BPR, tiny, 8, P5, Q5, None, None, 0.0, (0.05, 0.01, 0.01, 0.0), 2, rank, world, local)
    ok5 = bool(np.isfinite(l5).all())
    if rank == 0:
        print("invalid shard fails everywhere: %s   width-1 BPR blocks are skipped: %s (losses %s)" % (ok4, ok5, l5))
    # (6) the rank's C1 shard is staged in the order stream_order restates: item blocks from the GLOBAL item counts, the block in
    #     the top key bits, block-local item ids, the handle's seed + 977 * rank
    from librec_b200.dsgd_plan import item_bounds, stream_order
    h6 = capi.Handle(capi.MODEL_BIASEDMF, 8, device=local, seed=1)
    uid = [capi.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h6.comm_init(rank, world, uid[0])
    h6.set_train_csr(mine.U, mine.I, mine.rowptr, mine.col, mine.val)
    bounds = item_bounds(np.bincount(tr.col, minlength=tr.I), world)
    su, si, sr, run_tiles, max_deg = stream_order(mine.rowptr, mine.col, mine.val, tr.I, 1 + 977 * rank, bounds)
    gu, gi, gr, _ = h6.debug_stream(mine.col.shape[0])
    st6 = h6.stage_stats()
    h6.close()
    ok6 = (np.array_equal(gu, su) and np.array_equal(gi, si) and np.array_equal(gr.view(np.int32), sr.view(np.int32))
           and (st6["ratings"], st6["run_tile_ratings"], st6["max_item_degree"]) == (mine.col.shape[0], 32 * run_tiles, max_deg))
    all6 = [None] * world
    dist.all_gather_object(all6, bool(ok6))
    ok6 = all(all6)
    if rank == 0:
        print("staged stream of every rank = stream_order: %s (%s; rank 0: %d run-tile ratings)" % (ok6, all6, 32 * run_tiles))
    ok2 = ok2 and ok4 and ok5 and ok6
    if rank == 0:
        print("conflict-free:", r1)
        print("C1 DSGD world=%d:" % world, r2)
        print("DSGD-CHECK OK" if (ok1 and ok2) else "DSGD-CHECK FAILED")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if (ok1 and ok2) else 1)


if __name__ == "__main__":
    main()
