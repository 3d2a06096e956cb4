#!/usr/bin/env python
"""Secondary measurements on one B200 for the BASELINE.json configs that bench.py does not headline:
  C3: BPR k=128 SGD epoch (samples/s) on the synthetic ML-20M shape (implicit feedback, device-side sampling)
  BPR reference order (--only bprref): k=10 and k=128 on the binarised ML-20M shape, bit-identical to the StrictMath epoch of
  tests/bpr_strict_reference.cpp
  N3 (--only n3): RankSGD k=10 (ranksgd-test.properties) on the ML-20M shape, one update per train entry
  C4: PMF k=128 SGD epoch (updates/s) on the synthetic Netflix shape (480 189 x 17 770, 100 480 507 ratings); under torchrun
      (N ranks) the users are split into N contiguous blocks and the epoch runs as DSGD (strong scaling of the one data set)
One JSON line per config: device-resident epochs timed with CUDA events (lrk_last_epoch_ms), L2 flushed between
epochs, algorithmic-byte roofline per SURVEY.md 8(d)."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def run_dsgd(name, model_name, shape, k, lr, reg, steps, warmup):
    """strong scaling: the one data set, users split into WORLD_SIZE contiguous blocks"""
    import torch
    import torch.distributed as dist
    from librec_b200 import capi, synth
    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0}
    d = synth.make_ratings(shape)
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    lo, hi = rank * U // world, (rank + 1) * U // world
    a, b = int(d["rowptr"][lo]), int(d["rowptr"][hi])
    rowptr = np.ascontiguousarray(d["rowptr"][lo:hi + 1] - a)
    col, val = np.ascontiguousarray(d["col"][a:b]), np.ascontiguousarray(d["val"][a:b])
    P, Q, _, _ = synth.init_factors(U, I, k, 11, False)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    h = capi.Handle(capi.MODEL_PMF, k, device=local, seed=1)
    uid = [capi.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h.comm_init(rank, world, uid[0])
    h.set_train_csr(hi - lo, I, rowptr, col, val)
    h.set_factors(P[lo:hi], Q)
    ms, losses = [], []
    for s in range(warmup + steps):
        flush.zero_(); torch.cuda.synchronize(); dist.barrier()
        losses.append(h.sgd_epoch(lr, reg, reg, 0.0, s + 1))
        if s >= warmup:
            ms.append(h.last_epoch_ms())
    guard = h.sgd_safeguard()
    h.close()
    t = torch.tensor([float(np.mean(ms))], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    kms = float(t.item())
    if rank == 0:
        bytes_per = 12 + 4 * k * 4
        achieved = bytes_per * nnz / world / (kms * 1e-3) / 1e9
        print(json.dumps({"config": name, "metric": "MF SGD rating-updates/s", "value": nnz / (kms * 1e-3), "unit": "updates/s", "n_gpus": world,
                          "scaling": "strong", "steps": steps, "warmup": warmup, "ms_per_step": kms,
                          "workload": "%s k=%d, synthetic %s shape (%d x %d, %d ratings), DSGD over %d user blocks, lr %g reg %g" % (
                              model_name, k, shape, U, I, nnz, world, lr, reg),
                          "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s (per GPU)",
                                       "frac": achieved / peaks["hbm_gbs"], "algorithmic_bytes_per_unit": bytes_per},
                          "losses": losses, "safeguard": guard}), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def run(name, model_name, shape, k, lr, reg, steps, warmup):
    import torch
    from librec_b200 import capi, synth
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0}
    bpr = model_name == "bpr"
    ranksgd = model_name == "ranksgd"
    d = synth.make_ratings(shape, binary=bpr or model_name == "gbpr")
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    P, Q, _, _ = synth.init_factors(U, I, k, 11, False)
    gbpr = model_name == "gbpr"
    aobpr = model_name == "aobpr"
    bpr = bpr or aobpr
    model = capi.MODEL_AOBPR if aobpr else capi.MODEL_BPR if bpr else (capi.MODEL_RANKSGD if ranksgd else (capi.MODEL_GBPR if gbpr else capi.MODEL_PMF))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    with capi.Handle(model, k, seed=1) as h:
        if aobpr:
            h.set_param("aobpr.lambda", 0.05)
        h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
        h.set_factors(P, Q, None, np.zeros(I) if gbpr else None)
        ms, losses = [], []
        for s in range(warmup + steps):
            flush.zero_(); torch.cuda.synchronize()
            losses.append(h.sgd_epoch(lr, reg, reg, 0.01 if gbpr else 0.0, s + 1))
            if s >= warmup:
                ms.append(h.last_epoch_ms())
        guard = h.sgd_safeguard()
        # the L2 gather + RED rate for this row length and working set (lrk_probe_l2): what bounds these kernels (DESIGN.md 4.1)
        ld = 4
        while ld < k and ld < 128:
            ld *= 2
        l2 = h.probe_l2((U + I) * ld * 4, ld) if ld in (64, 128) else None
    kms = float(np.mean(ms))
    # GBPR: r/w of the group's user rows (2 users), q_i, q_j
    bytes_per = 8 * k * 4 if gbpr else 6 * k * 4 if bpr else (12 + 6 * k * 4 if ranksgd else 12 + 4 * k * 4)     # RankSGD: triple + r/w of p_u, q_i, q_j
    achieved = bytes_per * nnz / (kms * 1e-3) / 1e9
    print(json.dumps({"config": name, "metric": "GBPR samples/s" if gbpr else "AoBPR samples/s" if aobpr else "BPR samples/s" if bpr else ("RankSGD updates/s" if ranksgd else "MF SGD rating-updates/s"), "value": nnz / (kms * 1e-3),
                      "unit": "samples/s" if (bpr or gbpr) else "updates/s", "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": kms,
                      "workload": "%s k=%d, synthetic %s shape (%d x %d, %d ratings), lr %g reg %g" % (model_name, k, shape, U, I, nnz, lr, reg),
                      "roofline": ({"bound": "l2", "achieved": achieved, "peak": l2["mix"], "unit": "GB/s", "frac": achieved / l2["mix"],
                                    "peak_source": "lrk_probe_l2 in this run (row gathers + vector REDs 1:1, %d B rows; gathers alone %.0f, REDs alone %.0f GB/s)" % (ld * 4, l2["gather"], l2["red"]),
                                    "algorithmic_bytes_per_unit": bytes_per, "frac_of_hbm_peak": achieved / peaks["hbm_gbs"],
                                    "note": "BPR-type samples gather and RED-update three full rows (no run tiles): the algorithmic bytes ARE the L2 row traffic"}
                                   if (l2 and (bpr or gbpr)) else
                                   {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                                    "algorithmic_bytes_per_unit": bytes_per}),
                      "loss_first_last": [losses[0], losses[-1]], "losses": losses, "safeguard": guard}), flush=True)


def run_reference_order(name, model_name, shape, k, lr, reg, reg_b):
    """LRK_UPDATE_REFERENCE_ORDER (csrc/sgd_exact.cuh): the reference's sequential CSR-order walk as a dependency wavefront, fp64,
    learned factors bit-identical to the reference arithmetic -- the mode that meets the 1e-3 RMSE bar for PMF by construction.
    Bounded by the longest dependency chain (the most-rated item), not by bandwidth: this is its throughput beside the fast mode's."""
    import time
    from librec_b200 import capi, synth
    d = synth.make_ratings(shape)
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    biased = model_name == "biasedmf"
    P, Q, bu, bi = synth.init_factors(U, I, k, 11, biased)
    with capi.Handle(capi.MODEL_BIASEDMF if biased else capi.MODEL_PMF, k, seed=1, update_mode=capi.UPDATE_REFERENCE_ORDER) as h:
        t0 = time.perf_counter()
        h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
        t_stage = time.perf_counter() - t0
        h.set_factors(P, Q, bu, bi, float(d["val"].mean()) if biased else 0.0)
        ms, losses = [], []
        for s in range(3):
            losses.append(h.sgd_epoch(lr, reg, reg, reg_b, s + 1))
            ms.append(h.last_epoch_ms())
    kms = float(np.mean(ms[1:]))
    print(json.dumps({"config": name, "mode": "LRK_UPDATE_REFERENCE_ORDER (wavefront, fp64, bit-identical to the reference arithmetic)",
                      "metric": "MF SGD rating-updates/s", "value": nnz / (kms * 1e-3), "unit": "updates/s", "n_gpus": 1, "ms_per_step": kms,
                      "workload": "%s k=%d, synthetic %s shape (%d x %d, %d ratings), lr %g reg %g" % (model_name, k, shape, U, I, nnz, lr, reg),
                      "schedule_build_s": t_stage, "max_item_degree": int(np.bincount(d["col"], minlength=I).max()), "losses": losses}), flush=True)


def _chain_length(U, trip):
    """longest dependency chain of an epoch's samples: a sample follows the previous ones that touched its user or either item"""
    lv_u, lv_i = [0] * U, {}
    longest = 0
    for u, i, j in trip.tolist():
        lv = max(lv_u[u], lv_i.get(i, 0), lv_i.get(j, 0)) + 1
        lv_u[u] = lv_i[i] = lv_i[j] = lv
        longest = max(longest, lv)
    return longest


def run_bpr_reference_order(k):
    """BPR in reference order (csrc/sgd_bpr_exact.cuh) on the binarised ML-20M shape: one epoch timed after a warm-up epoch, both
    compared bit for bit with the StrictMath epoch of tests/bpr_strict_reference.cpp run from the same state on one CPU core"""
    import subprocess
    import time
    from librec_b200 import capi, synth
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bpr_strict
    L = bpr_strict.lib()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                          text=True).stdout.strip().splitlines()[0]
    d = synth.make_ratings("ml-20m", binary=True)
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    P, Q, _, _ = synth.init_factors(U, I, k, 11, False)
    lr, reg = 0.01, 0.01                                                   # bpr-test.properties
    with capi.Handle(capi.MODEL_BPR, k, seed=1, update_mode=capi.UPDATE_REFERENCE_ORDER) as h:
        h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
        h.set_factors(P, Q)
        s0 = int(h.get_matrix("jdk.random.state", (1,))[0])
        h.sgd_epoch(lr, reg, reg, 0.0, 1)                                 # warm-up
        warm_ms = h.last_epoch_ms()
        h.synchronize()
        t0 = time.perf_counter()
        trip = h.bpr_peek_samples(2, 0, nnz)                              # the draw stage alone, plus the copy of the triples
        draw_ms = (time.perf_counter() - t0) * 1e3
        h.sgd_epoch(lr, reg, reg, 0.0, 2)
        ms = h.last_epoch_ms()
        gP, gQ, _, _ = h.get_factors()
        gs = int(h.get_matrix("jdk.random.state", (1,))[0])
    L.lro_set_jrandom_state(s0)
    oP, oQ, oms = P.copy(), Q.copy(), []
    for _ in range(2):
        t0 = time.perf_counter()
        L.lro_bpr_epoch_strict(U, I, d["rowptr"], d["col"], k, oP, oQ, lr, reg, reg, nnz, None, None)
        oms.append((time.perf_counter() - t0) * 1e3)
    same = bool(np.array_equal(gP.view(np.int64), oP.view(np.int64)) and np.array_equal(gQ.view(np.int64), oQ.view(np.int64))
                and gs == L.lro_jrandom_state())
    print(json.dumps({"config": "BPR-reforder k=%d" % k, "mode": "LRK_UPDATE_REFERENCE_ORDER (BPR: java.util.Random stream, fp64, bit-identical)",
                      "metric": "BPR samples/s", "value": nnz / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "card": card,
                      "ms_per_epoch": ms, "warmup_epoch_ms": warm_ms, "draw_stage_and_copy_ms": draw_ms, "chain_length": _chain_length(U, trip),
                      "oracle_one_core_ms_per_epoch": oms, "speedup_vs_oracle": oms[1] / ms, "bit_identical_to_oracle": same,
                      "workload": "bpr k=%d, synthetic binarised ml-20m shape (%d x %d, %d samples per epoch), lr %g reg %g" % (k, U, I, nnz, lr, reg)}),
          flush=True)


def run_svdpp(steps, warmup, oracle_epochs=2):
    """N3: SVD++ (svdpp-test.properties: k=20, lr 0.002, reg 0.01) on the ML-20M shape; the oracle's sequential loop runs the first
    epochs beside it so that the loss curve at full concurrency is seen next to the reference's"""
    import time
    import torch
    from librec_b200 import capi, synth
    from oracle import oracle as O
    d = synth.make_ratings("ml-20m")
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    k, lr, reg = 20, 0.002, 0.01
    P, Q, bu, bi = synth.init_factors(U, I, k, 11, True)
    Y = np.random.default_rng(12).normal(0, 0.001, (I, k))
    mu = float(d["val"].mean())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    with capi.Handle(capi.MODEL_SVDPP, k, seed=1) as h:
        h.set_param("svdpp.reg_imp", reg)
        h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
        h.set_factors(P, Q, bu, bi, mu)
        h.set_matrix("svdpp.y", Y)
        ms, losses = [], []
        for s in range(warmup + steps):
            flush.zero_(); torch.cuda.synchronize()
            losses.append(h.sgd_epoch(lr, reg, reg, reg, s + 1))
            if s >= warmup:
                ms.append(h.last_epoch_ms())
    oP, oQ, oY, obu, obi = P.copy(), Q.copy(), Y.copy(), bu.copy(), bi.copy()
    t0 = time.perf_counter()
    ol = [O.lib().lro_svdpp_epoch(U, d["rowptr"], d["col"], d["val"], k, oP, oQ, oY, obu, obi, mu, lr, reg, reg, reg, reg) for _ in range(oracle_epochs)]
    t_or = (time.perf_counter() - t0) / max(1, oracle_epochs)
    kms = float(np.mean(ms))
    print(json.dumps({"config": "N3-SVD++", "metric": "MF SGD rating-updates/s", "value": nnz / (kms * 1e-3), "unit": "updates/s", "n_gpus": 1,
                      "steps": steps, "warmup": warmup, "ms_per_step": kms,
                      "workload": "svdpp k=%d, synthetic ml-20m shape (%d x %d, %d ratings), lr %g reg %g" % (k, U, I, nnz, lr, reg),
                      "losses": losses, "oracle_losses_first_epochs": ol, "oracle_updates_per_s_one_core": nnz / t_or,
                      "row_transfers_per_rating": "3 gathers (y_j, q_i, y_j) + 2 REDs (q_i, y_j); the user side is register-resident"}), flush=True)


def run_als(model_name, k, steps, warmup, shape="ml-20m", oracle_parity=True):
    """N3: WRMF (wrmf-test.properties: k=20, reg 0.01, coefficient 4) / eALS (eals-test.properties: k=200, reg 0.01, judge 1,
    coefficient 1) on the ML-20M shape.  The first iteration runs beside the oracle's and the factors are compared BITWISE; then
    `steps` timed iterations."""
    import time
    import torch
    from librec_b200 import capi, synth
    from oracle import oracle as O
    d = synth.make_ratings(shape)
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    reg = 0.01
    wrmf = model_name == "wrmf"
    lut = {float(v): (O.lib().lro_wrmf_weight(float(v), 4.0) if wrmf else O.lib().lro_eals_weight(float(v), 1.0, 1)) for v in np.unique(d["val"])}
    val = np.array([lut[float(v)] for v in d["val"]])
    P, Q, _, _ = synth.init_factors(U, I, k, 11, False)
    if not wrmf:
        P = np.zeros_like(P)                                   # EALSRecommender.java:125
    conf = np.ones(I)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = {"config": "N3-" + ("WRMF" if wrmf else "eALS"), "metric": "ALS train entries/s (one iteration = both sides)", "unit": "entries/s", "n_gpus": 1,
           "workload": "%s k=%d, synthetic %s shape (%d x %d, %d ratings), reg %g" % (model_name, k, shape, U, I, nnz, reg)}
    with capi.Handle(capi.MODEL_WRMF if wrmf else capi.MODEL_EALS, k, seed=1) as h:
        h.set_train_csr(U, I, d["rowptr"], d["col"], val)
        if not wrmf:
            h.set_matrix("eals.confidences", conf)
        h.set_factors(P, Q)
        h.sgd_epoch(0.0, reg, reg, 0.0, 1)
        first_ms = h.last_epoch_ms()
        if oracle_parity:
            gP, gQ, _, _ = h.get_factors()
            oP, oQ = P.copy(), Q.copy()
            t0 = time.perf_counter()
            if wrmf:
                O.lib().lro_wrmf_epoch(U, I, d["rowptr"], d["col"], val, k, oP, oQ, reg, reg)
            else:
                O.lib().lro_eals_epoch(U, I, d["rowptr"], d["col"], val, k, oP, oQ, conf, reg, reg)
            t_or = time.perf_counter() - t0
            out["parity"] = {"factors_bit_identical_after_1_iteration": bool(np.array_equal(gP, oP) and np.array_equal(gQ, oQ)),
                             "max_abs_diff": float(max(np.abs(gP - oP).max(), np.abs(gQ - oQ).max()))}
            out["oracle_entries_per_s_one_core"] = nnz / t_or
            out["oracle_s_per_iteration"] = t_or
        ms = []
        for s in range(warmup + steps):
            flush.zero_(); torch.cuda.synchronize()
            h.sgd_epoch(0.0, reg, reg, 0.0, s + 2)
            if s >= warmup:
                ms.append(h.last_epoch_ms())
        gP, gQ, _, _ = h.get_factors()
    kms = float(np.mean(ms))
    out.update({"value": nnz / (kms * 1e-3), "steps": steps, "warmup": warmup, "ms_per_step": kms, "first_iteration_ms": first_ms,
                "finite": bool(np.isfinite(gP).all() and np.isfinite(gQ).all())})
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    if dist_env()[1] > 1:
        run_dsgd("C4", "pmf", "netflix", 128, 0.01, 0.08, a.steps, a.warmup)    # pmf-test.properties, DSGD
        sys.exit(0)
    if a.only in ("", "c3"):
        run("C3", "bpr", "ml-20m", 128, 0.01, 0.01, a.steps, a.warmup)          # bpr-test.properties
    if a.only in ("", "c4"):
        run("C4", "pmf", "netflix", 128, 0.01, 0.08, a.steps, a.warmup)         # pmf-test.properties
    if a.only == "reforder":
        run_reference_order("C2-reforder", "biasedmf", "ml-20m", 64, 0.002, 0.01, 0.01)
        run_reference_order("C4p-reforder", "pmf", "netflix-10m", 128, 0.01, 0.08, 0.0)
        run_reference_order("C4-reforder", "pmf", "netflix", 128, 0.01, 0.08, 0.0)
    if a.only == "bprref":
        run_bpr_reference_order(10)
        run_bpr_reference_order(128)
    if a.only == "aobpr":
        run("N3-AoBPR", "aobpr", "ml-20m", 10, 0.01, 0.01, a.steps, a.warmup)       # aobpr-test-like: lambda 0.05 * numItems
    if a.only == "svdpp":
        run_svdpp(a.steps, a.warmup)
    if a.only in ("als", "wrmf"):
        run_als("wrmf", 20, a.steps, a.warmup)                              # wrmf-test.properties, bitwise parity at scale
        run_als("wrmf", 64, a.steps, a.warmup, oracle_parity=False)         # a larger k, timing only (the oracle needs minutes)
    if a.only in ("als", "eals"):
        run_als("eals", 32, a.steps, a.warmup)                              # bitwise parity at scale (the oracle needs 40 s at k=32, 4 min at k=200)
        run_als("eals", 200, a.steps, a.warmup, oracle_parity=False)        # eals-test.properties' k, timing only
    if a.only == "gbpr":
        # gbpr defaults: rho 1.5, group size 2.  GBPR adds the SUM of an epoch's factor updates at its end (GBPRRecommender.java:167-168),
        # so its effective step grows with the samples per row: lr 0.05 is fine on ml-100k (80 k samples), turns around after 4 epochs
        # on an ML-1M-shaped matrix in the ORACLE as well, and explodes at 20 M samples; the timing run scales lr with 1 / samples
        run("N3-GBPR", "gbpr", "ml-20m", 10, 0.0002, 0.01, a.steps, a.warmup)
    if a.only == "n3":
        run("N3", "ranksgd", "ml-20m", 10, 0.01, 0.0, a.steps, a.warmup)        # ranksgd-test.properties (SURVEY 8f N3)
