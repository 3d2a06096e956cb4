#!/usr/bin/env python
"""WRMF on 1, 2, 4 and 8 devices of one multi-device handle (lrk_create_multi), ML-20M shape, k = 20 and 64, in one process.

Per (k, device count): one warm-up iteration, then --steps timed iterations.  Each lrk_sgd_epoch returns after the devices have
synchronised, so the host clock around the call is the iteration's wall time; lrk_last_epoch_ms is printed beside it.  With two or
more devices LRK_ALS_TRACE=1 makes the library print the per-device phase split from CUDA events (Gram, solve, wait for the slowest
device, row exchange, per side); the script reads those lines from its own stderr.  After the timed iterations the factors are
compared bit for bit with the one-device run's.  No L2 flush between iterations: the train matrix alone (20 M entries as CSR and CSC
with fp64 values) is several times the 126 MB of L2.

Output: one JSON line per (k, device count) with the GPU name and power limit read in the same run; --out also writes them to a file.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from librec_b200 import capi, synth  # noqa: E402
from oracle import oracle as O  # noqa: E402

PHASES = ("gram_q", "solve_u", "wait_p", "xchg_p", "gram_p", "solve_i", "wait_q", "xchg_q")


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return [l.strip() for l in r.stdout.splitlines() if l.strip()]
    except (OSError, subprocess.SubprocessError) as e:
        return ["nvidia-smi failed: %s" % e]


class StderrCapture:
    """fd 2 into a temporary file (the library writes its trace lines with fprintf(stderr))"""

    def __enter__(self):
        sys.stderr.flush()
        self.f = tempfile.TemporaryFile(mode="w+")
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *a):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def parse_trace(text):
    """[als] device D gram_q x solve_u x ... total x ms -> {device: [{phase: ms}, ...]} in iteration order"""
    out = {}
    for line in text.splitlines():
        if not line.startswith("[als] device"):
            continue
        f = line.split()
        vals = dict(zip(f[3::2], (float(x) for x in f[4::2])))
        out.setdefault(int(f[2]), []).append({p: vals[p] for p in PHASES})
    return out


def run(d, val, k, ndev, steps, reg=0.01):
    U, I = d["U"], d["I"]
    P, Q, _, _ = synth.init_factors(U, I, k, 11, False)
    res = {"k": k, "n_devices": ndev}
    with capi.Handle(capi.MODEL_WRMF, k, seed=1, devices=list(range(ndev))) as h:
        t0 = time.perf_counter()
        h.set_train_csr(U, I, d["rowptr"], d["col"], val)
        h.set_factors(P, Q)
        res["setup_s"] = time.perf_counter() - t0
        h.sgd_epoch(0.0, reg, reg, 0.0, 1)                       # warm-up
        wall, lib = [], []
        with StderrCapture() as cap:
            for s in range(steps):
                t = time.perf_counter()
                h.sgd_epoch(0.0, reg, reg, 0.0, s + 2)
                wall.append((time.perf_counter() - t) * 1e3)
                lib.append(h.last_epoch_ms())
        gP, gQ, _, _ = h.get_factors()
    sys.stderr.write(cap.text.replace("[als]", "[als k=%d n=%d]" % (k, ndev)))
    res.update({"steps": steps, "warmup": 1, "wall_ms": wall, "wall_ms_mean": float(np.mean(wall)), "last_epoch_ms": lib})
    tr = parse_trace(cap.text)
    if tr:
        # mean over the timed iterations, per device; the slowest device's solves set the iteration's pace
        res["phase_ms"] = {str(dev): {p: float(np.mean([it[p] for it in its])) for p in PHASES} for dev, its in sorted(tr.items())}
    return res, gP, gQ


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--ks", default="20,64")
    ap.add_argument("--devices", default="1,2,4,8")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    os.environ["LRK_ALS_TRACE"] = "1"
    have = capi.device_count()
    if have < 1:
        raise SystemExit("no CUDA device: this benchmark measures the GPU path and has no CPU fallback")
    info = gpu_info()
    d = synth.make_ratings("ml-20m")
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    lut = {float(v): O.lib().lro_wrmf_weight(float(v), 4.0) for v in np.unique(d["val"])}    # wrmf-test.properties: coefficient 4
    val = np.array([lut[float(v)] for v in d["val"]])
    lines = []
    for k in (int(x) for x in a.ks.split(",")):
        ref = None
        for ndev in (int(x) for x in a.devices.split(",")):
            if ndev > have:
                lines.append({"k": k, "n_devices": ndev, "skipped": "only %d devices" % have})
                continue
            res, gP, gQ = run(d, val, k, ndev, a.steps)
            if ref is None and ndev == 1:
                ref = (gP, gQ)
            res["bit_identical_to_1_device"] = None if ref is None else bool(np.array_equal(gP, ref[0]) and np.array_equal(gQ, ref[1]))
            res.update({"workload": "WRMF k=%d, synthetic ml-20m shape (%d x %d, %d entries), reg 0.01, coefficient 4" % (k, U, I, nnz),
                        "entries_per_s": nnz / (res["wall_ms_mean"] * 1e-3), "gpus": info})
            lines.append(res)
            print(json.dumps(res), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
