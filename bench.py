#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native LibRec MF path.

Contract (one JSON line on stdout, rank 0):
    python bench.py --gpus N --steps K --warmup W [--impl reference]
N=1 workload = BASELINE.json configs[1]: BiasedMF k=64 on the synthetic ML-20M shape
(138 493 x 26 744, 20 000 263 ratings).  A "step" is one SGD epoch (one pass of trainModel()'s inner
loop over all ratings).  metric = MF SGD rating-updates/s.
  value    : device-resident epochs (inputs already in HBM), CUDA events, max over ranks
  e2e      : the same metric through the C ABI with HOST buffers -- one trainModel() call of the
             shim = stage CSR + factors H2D, E epochs, factors D2H -- all inside the timed region
  roofline : algorithmic bytes (1052 B / BiasedMF update, SURVEY.md 8d) / kernel time vs measured HBM peak
  cpu_baseline : the oracle's single-thread fp64 restatement of the reference loop on this box
--impl reference times that CPU restatement alone (the Java reference cannot run: no JVM).
N>1 (torchrun, one process per GPU): every rank owns one ML-20M-shaped user shard over the same item
catalogue (N x 20 000 263 ratings in total), trained with DSGD strata, item blocks rotated over NCCL;
value = ratings processed by all ranks / max-over-ranks time ("scaling": "weak").
The same line carries the second half of BASELINE.json's metric in "topn": top-10 users scored/s on
configs[4] (1 048 576 users x 1 048 576 items, k=128, sharded by user block over the N ranks, no
collective), measured through lrk_topn with pinned host result buffers (D2H inside the timed region),
with the tensor-pipe roofline of topn_tc_kernel from CUDA events on its stream.
--dump-outputs DIR (N=1) writes what the last timed step computed as DIR/<name>.npy, so that two builds can be compared output
for output on identical seeded inputs: the factors a trainModel() caller reads back after the last timed epoch (P, Q, bu, bi,
fp32 like the device state), that epoch's loss, and the top-10 lists of the last timed top-N call for a fixed seeded sample of
users (topn_users / topn_items / topn_scores / topn_counts).  The epochs update the factors with float atomics whose order varies,
so two runs of one build agree on the factors and the loss only to a tolerance (13 epochs on a B200: factors within 5e-5 of
each other, biases within 1.2e-2, loss within 1e-5 relative); the top-N lists are bit-identical.
"""
import argparse
import csv
import ctypes
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                # the benchmark writes nothing into the tree (it may be read-only)

METRIC = "MF SGD rating-updates/s"
UNIT = "updates/s"
K_FACTORS = 64
LR, REG, REG_B = 0.002, 0.01, 0.01           # biasedmf-test.properties (config C2)
BYTES_PER_UPDATE = 12 + 4 * K_FACTORS * 4 + 16   # SURVEY.md 8(d): 1052 B for k=64 fp32
E2E_EPOCHS = 10                               # epochs per trainModel() call in the e2e leg
# config C4 (BASELINE configs[3]): PMF k=128 on the Netflix shape, pmf-test.properties, DSGD at 2/4/8 GPUs (strong scaling)
C4_K, C4_LR, C4_REG = 128, 0.01, 0.08
C4_BYTES_PER_UPDATE = 12 + 4 * C4_K * 4      # SURVEY.md 8(d): 2060 B for k=128 fp32
DUMP_LIMIT = 64 << 20                         # bytes of --dump-outputs in all
DUMP_TOPN_USERS, DUMP_SEED = 1 << 15, 0x4C52D0  # the full top-N lists (1M users) exceed DUMP_LIMIT: a fixed sample of users


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """samples SM clock + throttle reasons while the timed region runs (pynvml, nvidia-smi fallback)"""

    def __init__(self, index=0, period=0.02):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._dev, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            log("pynvml unavailable:", e)
            self._nvml = None

    def _decode(self, mask):
        n = self._nvml
        names = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(n, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        return [k for k, bit in names.items() if mask & bit]

    def _run(self):
        n = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(n.nvmlDeviceGetClockInfo(self._dev, n.NVML_CLOCK_SM))
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(self._dev)
                except Exception:
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._dev)
                self.reasons.update(self._decode(mask))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self._nvml:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._stop.set()
            self._thr.join()
        if not self._nvml:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [int(x) for x in out.strip().split(",")]
                self.samples, self.max_mhz = [a], b
            except Exception:
                pass
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def workload_c2(U, I, nnz):
    return "BiasedMF k=%d SGD epoch, synthetic ML-20M shape (%d users x %d items, %d ratings), lr %g reg %g" % (
        K_FACTORS, U, I, nnz, LR, REG)


def workload_c4(U, I, nnz, world):
    return ("PMF k=%d SGD epoch, synthetic Netflix shape (%d users x %d items, %d ratings), lr %g reg %g, DSGD over %d GPUs "
            "(users in %d contiguous blocks, strong scaling)" % (C4_K, U, I, nnz, C4_LR, C4_REG, world, world))


# ------------------------------------------------------------------------------------------------
def cpu_reference_rate(d, sample_ratings, steps, warmup, model="biasedmf"):
    """time the oracle's faithful restatement (1 thread, CSR order, fp64) on a CSR prefix"""
    from oracle import oracle as O
    from librec_b200 import synth
    L = O.lib()
    U, I = d["U"], d["I"]
    nnz = int(d["rowptr"][-1])
    n = min(nnz, sample_ratings)
    u_end = int(np.searchsorted(d["rowptr"], n, side="left"))
    u_end = max(1, min(U, u_end))
    n = int(d["rowptr"][u_end])
    rowptr = np.ascontiguousarray(d["rowptr"][:u_end + 1])
    biased = model == "biasedmf"
    k = K_FACTORS if biased else C4_K
    P, Q, bu, bi = synth.init_factors(U, I, k, 7, biased)
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        if biased:
            L.lro_biasedmf_epoch(u_end, rowptr, d["col"], d["val"], k, P, Q, bu, bi, 3.5, LR, REG, REG, REG_B, None, None)
        else:
            L.lro_pmf_epoch(u_end, rowptr, d["col"], d["val"], k, P, Q, C4_LR, C4_REG, C4_REG, None, None)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    total = float(np.sum(times))
    return n * len(times) / total, n, total / len(times)


def run_reference(args):
    """the reference's CPU path on this box's host cores: the oracle port (the Java reference cannot run: no JVM), one thread
    because the reference's trainModel is single-threaded; same workload as our arm at this --gpus"""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    from librec_b200 import synth
    c4 = args.gpus > 1
    d = synth.make_ratings("netflix" if c4 else "ml-20m")
    nnz = int(d["rowptr"][-1])
    model = "pmf" if c4 else "biasedmf"
    # probe 1M ratings to size the per-step sample so K+W steps end within ~2.5 minutes
    rate, _, _ = cpu_reference_rate(d, 1_000_000, 1, 0, model)
    budget_s = 150.0 / max(1, args.steps + args.warmup)
    sample = int(min(nnz, max(1_000_000, rate * budget_s)))
    rate, n, sec = cpu_reference_rate(d, sample, args.steps, args.warmup, model)
    what = "PMFSimilarityRecommender.trainModel" if c4 else "BiasedMFRecommender.trainModel"
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong" if c4 else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_c4(d["U"], d["I"], nnz, args.gpus) if c4 else workload_c2(d["U"], d["I"], nnz)},
        "reference": "oracle port of %s (Java reference cannot run: no JVM)" % what,
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": "one epoch over the first %d ratings in CSR order per step (of %d); the reference's trainModel is single-threaded" % (n, nnz)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def pinned_array(capi, shape, dtype):
    """numpy view over a cudaMallocHost buffer from the C ABI (what the Java shim's direct buffers are)"""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = ctypes.c_void_p()
    rc = capi.load().lrk_host_alloc(ctypes.byref(p), max(nbytes, 1))
    if rc != 0:
        raise RuntimeError("lrk_host_alloc failed")
    buf = (ctypes.c_char * max(nbytes, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr, p


def ncu_dram_bytes(probe, kernel_regex, skip, count=1):
    """DRAM bytes (read + write) of ONE launch of `kernel_regex`, measured by running this script's --traffic-probe mode under
    ncu (two counters, --clock-control none) -- outside the timed region, in the same bench run.  None when ncu cannot profile here."""
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--print-units", "base",
           "-k", "regex:" + kernel_regex, "-s", str(skip), "-c", str(count), "--csv", sys.executable, os.path.abspath(__file__),
           "--traffic-probe", probe]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0"))
    except Exception as e:  # pragma: no cover
        return None, "ncu failed: %s" % e
    per_launch, header = {}, None
    for row in csv.reader(r.stdout.splitlines()):
        if header is None:
            if "Metric Name" in row and "Metric Value" in row:
                header = {name: i for i, name in enumerate(row)}
            continue
        try:
            if row[header["Metric Name"]].startswith("dram__bytes_"):
                per_launch.setdefault(row[header["ID"]], []).append(float(row[header["Metric Value"]].replace(",", "")))
        except (IndexError, ValueError, KeyError):
            pass
    full = [sum(v) for v in per_launch.values() if len(v) >= 2]
    if not full:
        return None, "ncu gave no dram counters (rc %d): %s" % (r.returncode, (r.stdout + r.stderr)[-300:].replace("\n", " "))
    return max(full), ("ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum -k regex:%s -s %d -c %d, largest launch (this run)"
                       % (kernel_regex, skip, count))


def traffic_probe(which):
    """child of ncu_dram_bytes: launches the kernel in question a few times on the benchmark shape and exits"""
    from librec_b200 import capi, synth
    if which == "sgd":
        d = synth.make_ratings("ml-20m")
        P0, Q0, bu0, bi0 = synth.init_factors(d["U"], d["I"], K_FACTORS, 100, True)
        with capi.Handle(capi.MODEL_BIASEDMF, K_FACTORS, seed=1) as h:
            h.set_train_csr(d["U"], d["I"], d["rowptr"], d["col"], d["val"])
            h.set_factors(P0, Q0, bu0, bi0, float(d["val"].mean()))
            for it in range(5):
                h.sgd_epoch(LR, REG, REG, REG_B, it + 1)
    elif which == "topn":
        nu, rowptr, col, val, P, Q = topn_inputs(0, 1)
        with capi.Handle(capi.MODEL_BPR, TOPN_K) as h:
            h.set_train_csr(nu, TOPN_ITEMS, rowptr, col, val)
            h.set_factors(P, Q)
            h.topn(TOPN_N, nq=4096)
            h.topn(TOPN_N)


def issued_l2_row_bytes(item_deg, k, biased):
    """bytes of factor rows (and biases) one epoch of the item-run-tile kernel REQUESTS from L2, counted from the staged layout
    (csrc/staging.cuh, csrc/sgd_rating_body.inc): a rating on the general path gathers and RED-updates both rows; a rating of an
    item-run tile (items with >= 128 ratings, 32 ratings per tile) gathers and RED-updates only the user row, the item row once per
    flush period (8 ratings; 16 from 512 ratings per item, 32 from 1024)."""
    deg = np.asarray(item_deg, np.int64)
    row, b = k * 4, (4 if biased else 0)
    run = np.where(deg >= 128, (deg // 32) * 32, 0)
    period = np.where(deg >= 1024, 32, np.where(deg >= 512, 16, 8))
    general = deg - run
    per_run_rating = 2 * (row + b) + 2.0 * (row + b) / period
    return float((general * (4 * row + 4 * b)).sum() + (run * per_run_rating).sum()), float(run.sum()) / float(max(1, deg.sum()))


def sgd_roofline(h, kernel, kms, nnz_launch, bytes_per_update, row_floats, working_set_bytes, peaks, which, traffic, traffic_how,
                 issued_bytes=None):
    """roofline object of an SGD epoch kernel.  The kernel gathers and RED-updates factor rows that live in L2, so its bound is
    the L2's gather+RED rate, measured HERE by lrk_probe_l2 with the same instructions and row length on a working set of the same
    size.  `achieved` = the row bytes the kernel requests from L2 per launch (issued_l2_row_bytes) / kernel time; SURVEY 8(d)'s
    algorithmic bytes (no cache or register credit) and the HBM figures ride along."""
    l2 = h.probe_l2(working_set_bytes, row_floats)
    algo = bytes_per_update * nnz_launch / (kms * 1e-3) / 1e9
    issued = None if issued_bytes is None else issued_bytes / (kms * 1e-3) / 1e9
    achieved = issued if issued is not None else algo
    out = {"bound": "l2", "achieved": achieved, "peak": l2["mix"], "unit": "GB/s", "frac": achieved / l2["mix"], "traffic": traffic,
           "achieved_is": "row bytes requested from L2 (gathers + REDs, counted from the staged layout)" if issued is not None
                          else "algorithmic bytes (SURVEY 8d)",
           "peak_source": "lrk_probe_l2 in this run: random %d B row gathers (ld.global.cg.v4) + red.global.add.v4.f32 1:1 on a %.0f MB "
                          "working set; gathers alone %.0f GB/s, REDs alone %.0f GB/s" % (row_floats * 4, working_set_bytes / 1e6, l2["gather"], l2["red"]),
           "kernel": kernel, "kernel_ms": kms,
           "algorithmic": {"bytes_per_launch": bytes_per_update * nnz_launch, "achieved": algo, "frac_of_l2_peak": algo / l2["mix"],
                           "frac_of_hbm_peak": algo / peaks["hbm_gbs"],
                           "note": "SURVEY 8(d): 12 + 4*k*4 (+16) B per update, no cache credit; exceeds 1 because item-run tiles keep a popular "
                                   "item's row in registers for 8-32 ratings -- bytes the model counts and the kernel never requests"},
           "traffic_source": traffic_how,
           "hbm": {"peak": peaks["hbm_gbs"], "peak_source": which,
                   "achieved_dram": None if traffic is None else traffic / (kms * 1e-3) / 1e9,
                   "frac_dram": None if traffic is None else traffic / (kms * 1e-3) / 1e9 / peaks["hbm_gbs"]},
           "note": "the factor set is L2-resident (DRAM moves the COO stream only, hbm.frac_dram), so the binding resource is the L2's rate for "
                   "row gathers + vector REDs; the REDs are the scarce half (peak_source)"}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from librec_b200 import _build, capi, synth

    rank, world, local = dist_env()
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if not os.path.exists(_build.LIB_PATH):
        _build.build()
    capi.load()
    outputs = {} if args.dump_outputs else None
    if world > 1:
        line = run_c4_dsgd(args, torch, dist, capi, synth, rank, world, local, dev)
    else:
        line = run_c2_single(args, torch, capi, synth, local, dev, outputs)
    if not args.no_topn:
        tn = topn_leg(args, capi, torch, dist, rank, world, local, dev, outputs)
        if rank == 0:
            line["topn"] = tn
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def timed_epochs(torch, dist, h, world, stream, flush, steps, warmup, hyper, first_epoch=1):
    """W untimed + K timed epochs; barrier + synchronize on both sides; CUDA events per step on `stream`; -> (total ms max over
    ranks, mean device ms of the epoch's kernels on this rank, losses)"""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    losses = []
    for w in range(warmup):
        losses.append(h.sgd_epoch(*hyper, first_epoch + w))
    barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kernel_ms = []
    for s in range(steps):
        flush.zero_()                                   # evict L2 between timed steps (not timed)
        evs[s][0].record(stream)
        losses.append(h.sgd_epoch(*hyper, first_epoch + warmup + s))
        evs[s][1].record(stream)
        kernel_ms.append(h.last_epoch_ms())
    barrier()
    total_ms = float(np.sum([a.elapsed_time(b) for a, b in evs]))
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    return total_ms, float(np.mean(kernel_ms)), losses


def write_outputs(out_dir, outputs):
    """--dump-outputs: one DIR/<name>.npy per array (float32 or float64)"""
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log("--dump-outputs: %d arrays, %d bytes in %s" % (len(outputs), total, out_dir))


def run_c2_single(args, torch, capi, synth, local, dev, outputs=None):
    d = synth.make_ratings("ml-20m")
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    P0, _, bu0, _ = synth.init_factors(U, I, K_FACTORS, 100, True)
    _, Q0, _, bi0 = synth.init_factors(U, I, K_FACTORS, 1, True)
    mu = float(d["val"].mean())
    h = capi.Handle(capi.MODEL_BIASEDMF, K_FACTORS, device=local, seed=1)
    stream = torch.cuda.current_stream()
    h.set_stream(stream.cuda_stream)
    h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
    h.set_factors(P0, Q0, bu0, bi0, mu)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    sampler = ClockSampler(index=local)
    for w in range(args.warmup):                                    # warm-up outside the sampler
        h.sgd_epoch(LR, REG, REG, REG_B, w + 1)
    launches0 = h.launch_count()
    sampler.start()
    total_ms, kms, losses = timed_epochs(torch, None, h, 1, stream, flush, args.steps, 0, (LR, REG, REG, REG_B), args.warmup + 1)
    clocks = sampler.stop()
    launches = h.launch_count() - launches0
    if outputs is not None:                     # the device state is fp32, so float32 holds the factors exactly
        gP, gQ, gbu, gbi = h.get_factors()
        outputs.update(P=gP.astype(np.float32), Q=gQ.astype(np.float32), bu=gbu.astype(np.float32), bi=gbi.astype(np.float32),
                       loss=np.array([losses[-1]], np.float64))
    value = nnz * args.steps / (total_ms * 1e-3)
    peaks, which = measured_peaks()
    traffic, traffic_how = (None, "skipped (--no-traffic)") if args.no_traffic else ncu_dram_bytes("sgd", "sgd_rating_epoch_kernel", 4)
    ws = (U + I) * (K_FACTORS + 1) * 4
    stage = h.stage_stats()
    issued, run_share = issued_l2_row_bytes(np.bincount(d["col"], minlength=I), K_FACTORS, True)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_c2(U, I, nnz)},
        "run": {"update_mode": "atomic (REDG.E.ADD.F32x4)",
                "l2": "L2 flushed between timed steps (256 MiB memset, untimed); COO stream 240 MB > L2",
                "parallelism": "single GPU", "final_loss": losses[-1],
                "item_popularity": "Zipf(1.0) over %d items (the survey's generator); share of ratings staged as item-run tiles: %.3f"
                                   % (I, stage["run_tile_share"]),
                "run_tile_share": stage["run_tile_share"]},
        "roofline": sgd_roofline(h, "sgd_rating_epoch_kernel<16,1,true,true>", kms, nnz, BYTES_PER_UPDATE, K_FACTORS, ws, peaks, which,
                                 traffic, traffic_how, issued_bytes=issued),
        "gpu_launches": int(launches), "clocks": clocks,
    }

    # ---- the same shape with a flatter item popularity (Zipf 0.5: the head of real MovieLens data is far flatter than the survey's
    #      Zipf 1.0 generator), so that the headline is not a property of the generator's head
    if not args.no_flat:
        df = synth.make_ratings("ml-20m", zipf=0.5)
        h.set_train_csr(U, I, df["rowptr"], df["col"], df["val"])
        h.set_factors(P0, Q0, bu0, bi0, float(df["val"].mean()))
        tf_ms, kf_ms, lf = timed_epochs(torch, None, h, 1, stream, flush, max(3, min(args.steps, 10)), 3, (LR, REG, REG, REG_B), 1)
        fdeg = np.bincount(df["col"], minlength=I)
        line["run"]["flat_popularity"] = {
            "workload": "same shape and hyper-parameters, item popularity Zipf(0.5)", "value": nnz / (kf_ms * 1e-3), "unit": UNIT,
            "kernel_ms": kf_ms, "run_tile_share": h.stage_stats()["run_tile_share"],
            "top_item_share": float(fdeg.max()) / nnz, "top_item_share_headline": float(np.bincount(d["col"], minlength=I).max()) / nnz,
            "final_loss": lf[-1]}
        h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
        h.set_factors(P0, Q0, bu0, bi0, mu)

    # ---- e2e: one trainModel() call of the shim per step, host buffers, copies inside the timed region
    if not args.no_e2e:
        rp, p1 = pinned_array(capi, (U + 1,), np.int64); rp[:] = d["rowptr"]
        cl, p2 = pinned_array(capi, (nnz,), np.int32); cl[:] = d["col"]
        vl, p3 = pinned_array(capi, (nnz,), np.float64); vl[:] = d["val"]
        hP, p4 = pinned_array(capi, (U, K_FACTORS), np.float64); hQ, p5 = pinned_array(capi, (I, K_FACTORS), np.float64)
        hbu, p6 = pinned_array(capi, (U,), np.float64); hbi, p7 = pinned_array(capi, (I,), np.float64)
        hloss, p8 = pinned_array(capi, (E2E_EPOCHS,), np.float64)
        bufs = [p1, p2, p3, p4, p5, p6, p7, p8]
        L = capi.load()
        vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        breakdown = {"set_train_csr": [], "set_factors": [], "epochs": [], "get_factors": []}

        def train_model_call(record=True):
            hP[:] = P0; hQ[:] = Q0; hbu[:] = bu0; hbi[:] = bi0
            t0 = time.perf_counter()
            rc = L.lrk_set_train_csr(h._h, U, I, vp(rp), vp(cl), vp(vl))
            t1 = time.perf_counter()
            rc |= L.lrk_set_factors(h._h, vp(hP), vp(hQ), vp(hbu), vp(hbi), mu)
            t2 = time.perf_counter()
            # rec.learnrate.bolddriver=false, decay=1, no early stop (biasedmf-test.properties): the shim batches the iterations
            rc |= L.lrk_sgd_epochs(h._h, E2E_EPOCHS, LR, 1.0, LR, REG, REG, REG_B, 1, vp(hloss))
            t3 = time.perf_counter()
            rc |= L.lrk_get_factors(h._h, vp(hP), vp(hQ), vp(hbu), vp(hbi))
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            if rc != 0:
                raise RuntimeError("e2e call failed: %s" % L.lrk_last_error(h._h))
            if record:
                for key, dt in zip(breakdown, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                    breakdown[key].append(dt * 1e3)
            return t4 - t0

        e2e_steps = max(2, min(args.steps, 5))
        train_model_call(record=False)                      # warm-up
        tt = [train_model_call() for _ in range(e2e_steps)]
        h2d = rp.nbytes + cl.nbytes + vl.nbytes + hP.nbytes + hQ.nbytes + hbu.nbytes + hbi.nbytes
        d2h = hP.nbytes + hQ.nbytes + hbu.nbytes + hbi.nbytes + 8 * E2E_EPOCHS
        line["e2e"] = {"value": nnz * E2E_EPOCHS * e2e_steps / float(np.sum(tt)), "unit": UNIT,
                       "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "step": "one trainModel() call through the C ABI from pinned host buffers: lrk_set_train_csr + "
                               "lrk_set_factors + lrk_sgd_epochs(%d) + lrk_get_factors" % E2E_EPOCHS,
                       "ms_per_call": float(np.mean(tt)) * 1e3, "calls": e2e_steps,
                       "breakdown_ms": {k_: float(np.mean(v)) for k_, v in breakdown.items()}}
        for p in bufs:
            L.lrk_host_free(p)
    else:
        line["e2e"] = None
    h.close()

    # ---- parity at scale, same run: the fast kernel at full concurrency vs the oracle's sequential loop, held-out RMSE / MAE
    if not args.no_parity:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import parity_scale
        from oracle import oracle as O
        r = parity_scale.rating_parity(capi, O, "c2", epochs=10, device=local)
        line["parity"] = {"what": "BiasedMF k=64, 10 epochs from identical factors on a seeded 80/20 split of the benchmark matrix: held-out "
                                  "RMSE / MAE of the fast kernel vs the oracle's sequential fp64 loop", **r}
        if not r["ok"]:
            log("PARITY FAILED:", r)
            print(json.dumps(line), flush=True)
            sys.exit(3)

    # ---- cpu baseline: oracle port on this box's host cores
    if not args.no_cpu_baseline:
        rate, n, sec = cpu_reference_rate(d, nnz, 1, 0)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": "one full epoch (%d ratings) of the oracle's restatement of BiasedMFRecommender.trainModel, "
                                          "CSR order, fp64, 1 thread (the reference loop is single-threaded); %.1f s" % (n, sec)}
        try:
            from oracle import oracle as O
            nt = O.lib().lro_max_threads()
            rows = np.repeat(np.arange(U, dtype=np.int32), np.diff(d["rowptr"]))
            perm = np.random.default_rng(0).permutation(nnz)
            us, is_, rs = rows[perm], d["col"][perm], d["val"][perm].astype(np.float32)
            P, Q, bu, bi = [a.astype(np.float32) for a in (P0, Q0, bu0, bi0)]
            t0 = time.perf_counter()
            O.lib().lro_sgd_epoch_hogwild_f32(0, us, is_, rs, nnz, K_FACTORS, P, Q, bu.ctypes.data, bi.ctypes.data,
                                              mu, LR, REG, REG, REG_B, nt)
            dt = time.perf_counter() - t0
            line["cpu_best_effort"] = {"value": nnz / dt, "unit": UNIT, "cores": nt,
                                       "what": "OpenMP Hogwild fp32 epoch over shuffled triples (NOT the reference's algorithm)"}
        except Exception as e:  # pragma: no cover
            log("best-effort cpu leg failed:", e)
    return line


def run_c4_dsgd(args, torch, dist, capi, synth, rank, world, local, dev):
    """N > 1: BASELINE configs[3] -- PMF k=128 on the Netflix shape, ONE data set split into N user blocks (strong scaling), DSGD
    strata with the item blocks rotating over NVLink.  Parity is checked inside the run, before the timed region."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import dsgd_checks
    from oracle import oracle as O
    stream = torch.cuda.current_stream()

    # ---- parity first: a run whose DSGD does not reproduce the oracle is not measured
    par_cf = dsgd_checks.conflict_free(capi, dist, O, rank, world, local)
    par_c1 = dsgd_checks.c1(capi, dist, O, rank, world, local)
    parity = {"conflict_free_epoch_vs_oracle": par_cf, "c1_biasedmf_100_epochs_vs_oracle": par_c1,
              "ok": bool(par_cf["ok"] and par_c1["ok"])}
    if not parity["ok"]:
        if rank == 0:
            log("DSGD PARITY FAILED:", parity)
            print(json.dumps({"metric": METRIC, "value": None, "n_gpus": world, "parity": parity}), flush=True)
        dist.barrier()
        sys.exit(3)

    d = synth.make_ratings("netflix")
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    lo, hi = rank * U // world, (rank + 1) * U // world
    a, b = int(d["rowptr"][lo]), int(d["rowptr"][hi])
    rowptr = np.ascontiguousarray(d["rowptr"][lo:hi + 1] - a)
    col, val = np.ascontiguousarray(d["col"][a:b]), np.ascontiguousarray(d["val"][a:b])
    P0, Q0, _, _ = synth.init_factors(U, I, C4_K, 11, False)
    hyper = (C4_LR, C4_REG, C4_REG, 0.0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    h = capi.Handle(capi.MODEL_PMF, C4_K, device=local, seed=1)
    h.set_stream(stream.cuda_stream)
    uid = [capi.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h.comm_init(rank, world, uid[0])
    h.set_train_csr(hi - lo, I, rowptr, col, val)
    h.set_factors(P0[lo:hi], Q0)
    sampler = ClockSampler(index=local)
    wl = []
    for w in range(args.warmup):
        wl.append(h.sgd_epoch(*hyper, w + 1))
    launches0 = h.launch_count()
    sampler.start()
    total_ms, kms, losses = timed_epochs(torch, dist, h, world, stream, flush, args.steps, 0, hyper, args.warmup + 1)
    clocks = sampler.stop()
    launches = h.launch_count() - launches0
    guard = h.sgd_safeguard()
    losses = wl + losses
    value = nnz * args.steps / (total_ms * 1e-3)

    # ---- e2e at N GPUs: every rank stages its shard from pinned host buffers, trains E epochs, reads its factors back
    e2e = None
    if not args.no_e2e:
        nl = int(rowptr[-1])
        rp, p1 = pinned_array(capi, rowptr.shape, np.int64); rp[:] = rowptr
        cl, p2 = pinned_array(capi, (nl,), np.int32); cl[:] = col
        vl, p3 = pinned_array(capi, (nl,), np.float64); vl[:] = val
        hP, p4 = pinned_array(capi, (hi - lo, C4_K), np.float64); hQ, p5 = pinned_array(capi, (I, C4_K), np.float64)
        hloss, p6 = pinned_array(capi, (E2E_EPOCHS,), np.float64)
        L = capi.load()
        vp = lambda x: x.ctypes.data_as(ctypes.c_void_p)

        phases = []

        def call():
            hP[:] = P0[lo:hi]; hQ[:] = Q0
            dist.barrier(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            rc = L.lrk_set_train_csr(h._h, hi - lo, I, vp(rp), vp(cl), vp(vl))
            t1 = time.perf_counter()
            rc |= L.lrk_set_factors(h._h, vp(hP), vp(hQ), None, None, 0.0)
            t2 = time.perf_counter()
            rc |= L.lrk_sgd_epochs(h._h, E2E_EPOCHS, C4_LR, 1.0, C4_LR, C4_REG, C4_REG, 0.0, 1, vp(hloss))
            t3 = time.perf_counter()
            rc |= L.lrk_get_factors(h._h, vp(hP), vp(hQ), None, None)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            phases.append([(t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3, (time.perf_counter() - t3) * 1e3])
            if rc != 0:
                raise RuntimeError("e2e call failed: %s" % L.lrk_last_error(h._h))
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        call()
        calls = 3
        tt = [call() for _ in range(calls)]
        byt = torch.tensor([rp.nbytes + cl.nbytes + vl.nbytes + hP.nbytes + hQ.nbytes, hP.nbytes + hQ.nbytes + 8 * E2E_EPOCHS],
                           dtype=torch.float64, device="cuda")
        dist.all_reduce(byt)
        e2e = {"value": nnz * E2E_EPOCHS * calls / float(np.sum(tt)), "unit": UNIT, "h2d_bytes_per_step": int(byt[0].item()),
               "d2h_bytes_per_step": int(byt[1].item()),
               "step": "one trainModel() per rank through the C ABI from pinned host buffers: lrk_set_train_csr(shard) + lrk_set_factors + "
                       "lrk_sgd_epochs(%d) + lrk_get_factors (ring gather of the item factors); wall clock between barriers, max over ranks; "
                       "bytes summed over ranks" % E2E_EPOCHS,
               "ms_per_call": float(np.mean(tt)) * 1e3, "calls": calls, "ms_calls": [x * 1e3 for x in tt],
               "rank0_phases_ms": {"names": ["set_train_csr", "set_factors", "sgd_epochs(%d)" % E2E_EPOCHS, "get_factors"], "calls": phases[1:]}}
        for p in (p1, p2, p3, p4, p5, p6):
            L.lrk_host_free(p)
    peaks, which = measured_peaks()
    roof = None
    if rank == 0:
        ws = ((hi - lo) + I) * C4_K * 4
        issued, _ = issued_l2_row_bytes(np.bincount(col, minlength=I), C4_K, False)
        roof = sgd_roofline(h, "sgd_rating_epoch_kernel<32,1,false,true,true> (one launch per DSGD stratum)", kms, int(rowptr[-1]),
                            C4_BYTES_PER_UPDATE, C4_K, ws, peaks, which, None, "not measured under DSGD (ncu runs one GPU)",
                            issued_bytes=issued)
        roof["kernel_ms"] = kms
        roof["note"] = "per GPU (rank 0): kernel_ms is the epoch on the stream = N stratum kernels + N ring exchanges + loss all-reduce; " + roof["note"]
    h.close()

    # ---- the same data set on ONE GPU of this box (rank 0, the others wait): the base of the strong-scaling claim and of the loss check
    base = None
    if not args.no_base:
        if rank == 0:
            h1 = capi.Handle(capi.MODEL_PMF, C4_K, device=local, seed=1)
            h1.set_stream(stream.cuda_stream)
            h1.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
            h1.set_factors(P0, Q0)
            t1_ms, k1_ms, l1 = timed_epochs(torch, None, h1, 1, stream, flush, args.steps, args.warmup, hyper, 1)
            g1 = h1.sgd_safeguard()
            h1.close()
            v1 = nnz * args.steps / (t1_ms * 1e-3)
            base = {"workload": workload_c4(U, I, nnz, 1), "n_gpus": 1, "value": v1, "unit": UNIT, "ms_per_step": t1_ms / args.steps,
                    "final_loss": l1[-1], "rollbacks": g1["rollbacks"],
                    "loss_ratio_dsgd_over_1gpu": losses[-1] / l1[-1], "speedup": value / v1}
        dist.barrier()

    # ---- r01's weak-scaling line (N ML-20M-shaped user shards), kept as an extra key
    weak = None
    if not args.no_weak:
        weak = weak_ml20m(args, torch, dist, capi, synth, rank, world, local, dev, stream, flush)

    if rank != 0:
        return None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_c4(U, I, nnz, world)},
        "run": {"update_mode": "atomic (REDG.E.ADD.F32x4)", "l2": "L2 flushed between timed steps (256 MiB memset, untimed)",
                "parallelism": "DSGD %d strata per epoch, item blocks rotate over NVLink (%s)" % (world, h_exchange_desc()),
                "losses": losses, "final_loss": losses[-1], "rollbacks": guard["rollbacks"], "conc_div": guard["conc_div"],
                "note": "N=1 of this bench is BASELINE configs[1] (BiasedMF k=64, ML-20M shape), N>1 is configs[3] (this line): the two "
                        "values are different workloads; the strong-scaling base of THIS workload is in strong_scaling_base"},
        "parity": parity,
        "strong_scaling_base": base,
        "roofline": roof, "e2e": e2e, "weak_ml20m": weak,
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if guard["rollbacks"]:
        log("WARNING: %d rollbacks" % guard["rollbacks"])
    return line


def h_exchange_desc():
    if os.environ.get("LRK_DSGD_FUSED", "") == "0":
        return "LRK_DSGD_FUSED=0: grouped ncclSend/ncclRecv after every stratum kernel"
    return "one cooperative kernel per epoch: peer stores into the ring neighbour's buffer + system-scope flags (csrc/dsgd_fused.cuh)"


def weak_ml20m(args, torch, dist, capi, synth, rank, world, local, dev, stream, flush):
    """every rank owns one ML-20M-shaped user shard over the same item catalogue (N x 20 000 263 ratings), BiasedMF k=64"""
    d = synth.make_ratings("ml-20m", shard=rank)
    U, I, nnz = d["U"], d["I"], int(d["rowptr"][-1])
    P0, _, bu0, _ = synth.init_factors(U, I, K_FACTORS, 100 + rank, True)
    _, Q0, _, bi0 = synth.init_factors(U, I, K_FACTORS, 1, True)          # item side identical on every rank
    m = torch.tensor([float(d["val"].mean())], dtype=torch.float64, device=dev)
    dist.all_reduce(m)
    mu = float(m.item()) / world
    h = capi.Handle(capi.MODEL_BIASEDMF, K_FACTORS, device=local, seed=1)
    h.set_stream(stream.cuda_stream)
    uid = [capi.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h.comm_init(rank, world, uid[0])
    h.set_train_csr(U, I, d["rowptr"], d["col"], d["val"])
    h.set_factors(P0, Q0, bu0, bi0, mu)
    total_ms, kms, losses = timed_epochs(torch, dist, h, world, stream, flush, args.steps, args.warmup, (LR, REG, REG, REG_B), 1)
    guard = h.sgd_safeguard()
    h.close()
    return {"metric": METRIC, "scaling": "weak", "value": nnz * world * args.steps / (total_ms * 1e-3), "unit": UNIT,
            "ms_per_step": total_ms / args.steps, "kernel_ms": kms, "final_loss": losses[-1], "rollbacks": guard["rollbacks"],
            "workload": "BiasedMF k=%d SGD epoch, %d ML-20M-shaped user shards (%d users x %d items, %d ratings in total), lr %g reg %g"
                        % (K_FACTORS, world, U * world, I, nnz * world, LR, REG)}


# ------------------------------------------------------------------------------------------------
TOPN_USERS, TOPN_ITEMS, TOPN_K, TOPN_N, TOPN_TRAIN = 1 << 20, 1 << 20, 128, 10, 32


def topn_inputs(rank, world):
    """this rank's user block of configs[4]: factors N(0, 0.1^2) rounded through fp32, a 32-item train mask per user"""
    U, I, k = TOPN_USERS, TOPN_ITEMS, TOPN_K
    lo, hi = rank * U // world, (rank + 1) * U // world
    nu = hi - lo
    rng_q = np.random.default_rng(0x4C520005)                       # item side identical on every rank
    Q = rng_q.normal(0, 0.1, (I, k)).astype(np.float32).astype(np.float64)
    rng = np.random.default_rng([0x4C520005, rank, world])
    P = rng.normal(0, 0.1, (nu, k)).astype(np.float32).astype(np.float64)
    # train mask: one random item out of each of 32 equal strata of the catalogue -> distinct, ascending
    edges = np.linspace(0, I, TOPN_TRAIN + 1).astype(np.int64)
    cols = (edges[:-1][None, :] + (rng.random((nu, TOPN_TRAIN)) * np.diff(edges)[None, :]).astype(np.int64)).astype(np.int32)
    rowptr = np.arange(nu + 1, dtype=np.int64) * TOPN_TRAIN
    col = np.ascontiguousarray(cols.reshape(-1))
    val = np.ones(col.shape[0], np.float64)
    return nu, rowptr, col, val, P, Q


def topn_leg(args, capi, torch, dist, rank, world, local, dev, outputs=None):
    """top-10 users scored/s on configs[4]; users are sharded by contiguous block over the ranks (strong scaling,
    no collective: every rank holds the full item matrix).  Returns the "topn" object (rank 0) or None."""
    U, I, k, N = TOPN_USERS, TOPN_ITEMS, TOPN_K, TOPN_N
    nu, rowptr, col, val, P, Q = topn_inputs(rank, world)
    h = capi.Handle(capi.MODEL_BPR, k, device=local)
    h.set_train_csr(nu, I, rowptr, col, val)
    h.set_factors(P, Q)
    items, p1 = pinned_array(capi, (nu, N), np.int32)
    scores, p2 = pinned_array(capi, (nu, N), np.float64)
    counts, p3 = pinned_array(capi, (nu,), np.int32)
    h.topn(N, nq=min(nu, 4096))                                     # builds the item operand (cached afterwards)
    h.topn(N, out=(items, scores, counts))                          # warm-up of the full call
    steps = max(2, min(args.steps, 3))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    wall, sweep, dev_ms, stats = [], [], [], None
    for s in range(steps):
        t0 = time.perf_counter()
        h.topn(N, out=(items, scores, counts))
        wall.append(time.perf_counter() - t0)
        stats = h.topn_stats()
        sweep.append(stats["phase_ms"]["sweep"]); dev_ms.append(stats["ms"])
    if outputs is not None:                     # user and item ids are < 2^24: exact in float32
        users = np.sort(np.random.default_rng(DUMP_SEED).choice(nu, min(nu, DUMP_TOPN_USERS), replace=False))
        outputs.update(topn_users=users.astype(np.float32), topn_items=items[users].astype(np.float32),
                       topn_scores=scores[users].astype(np.float64), topn_counts=counts[users].astype(np.float32))
    t = torch.tensor([float(np.sum(wall))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_s = float(t.item())
    out = None
    if rank == 0:
        peaks, which = measured_peaks()
        tn_traffic, tn_traffic_how = None, "skipped"
        if world == 1 and not args.no_traffic:
            tn_traffic, tn_traffic_how = ncu_dram_bytes("topn", "topn_tc_kernel", 0, 6)
        kms = float(np.mean(sweep))
        flop = 2.0 * nu * I * k                                     # this rank's launch
        tf = flop / (kms * 1e-3) / 1e12
        # parity spot check against the oracle (64 users, the checker only)
        from oracle import oracle as O
        tr = O.Csr(nu, I, rowptr, col, val)
        sample = np.linspace(0, nu - 1, 64).astype(np.int32)
        t0 = time.perf_counter()
        oi, os_, oc = O.recommend_rank(O.BPR, nu, I, k, P, Q, None, None, 0.0, tr, N, users=sample)
        cpu_dt = time.perf_counter() - t0
        ok = bool(np.array_equal(items[sample], oi) and np.array_equal(scores[sample].view(np.int64), os_.view(np.int64))
                  and np.array_equal(counts[sample], oc))
        out = {"metric": "top-%d users scored/s" % N, "value": U * steps / total_s, "unit": "users/s", "n_gpus": world, "steps": steps,
               "scaling": "strong", "dtype": "f16 sweep (f32 accumulate) + f64 exact re-score",
               "config": {"workload": "top-%d over %d users x %d items, k=%d, %d train items/user masked; users sharded by block over %d rank(s)"
                                      % (N, U, I, k, TOPN_TRAIN, world)},
               "e2e": {"value": U * steps / total_s, "unit": "users/s", "h2d_bytes_per_step": 0,
                       "d2h_bytes_per_step": int(items.nbytes + scores.nbytes + counts.nbytes),
                       "step": "one lrk_topn call per rank (factors resident, result lists copied into pinned host buffers inside the timed region)"},
               "ms_per_step": total_s / steps * 1e3, "device_ms": float(np.mean(dev_ms)), "phase_ms": stats["phase_ms"],
               "certificate": {"fallback_users": stats["fallback_users"], "resweep_users": stats["resweep_users"],
                               "sweep_error_over_bound": stats["sweep_error_over_bound"]},
               "roofline": {"bound": "tensor", "kernel": "topn_tc_kernel", "kernel_ms": kms, "achieved": tf, "peak": peaks["bf16_tflops"],
                            "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"],
                            "frac_of_sustained": tf / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]),
                            "peak_source": which, "flop_per_launch": flop, "traffic": tn_traffic, "traffic_source": tn_traffic_how},
               "parity": {"users_checked": 64, "bit_identical": ok},
               "cpu_baseline": {"value": 64 / cpu_dt, "unit": "users/s", "cores": int(O.lib().lro_max_threads()), "kind": "port",
                                "sample": "64 users against the full catalogue, oracle restatement of recommendRank, OpenMP over users"}}
    h.close()
    L = capi.load()
    for p in (p1, p2, p3):
        L.lrk_host_free(p)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-topn", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the at-scale parity leg (N=1)")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu DRAM-traffic probes (N=1)")
    ap.add_argument("--no-flat", action="store_true", help="skip the flatter-popularity extra line (N=1)")
    ap.add_argument("--no-base", action="store_true", help="skip the 1-GPU base of the strong-scaling workload (N>1)")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling ML-20M extra line (N>1)")
    ap.add_argument("--traffic-probe", default="", help="internal: child mode of the ncu traffic probe (sgd | topn)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (N=1; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1 or dist_env()[1] != 1):
        ap.error("--dump-outputs covers the one-GPU run of --impl ours")
    if args.traffic_probe:
        traffic_probe(args.traffic_probe)
        return
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
