#!/usr/bin/env python
# -*- coding: utf-8 -*-
"""bench.py -- PSMF/rPSMF filter steps/sec on B200 (BASELINE.json metric).

Workload L (default; BASELINE.json configs[3], the configuration the metric is quoted on): one series, d = 1,000,000
rows, r = 16, T = 10,000 time steps, rPSMF (Student-t scales) with 20 % missing entries, fp64, synthetic data
generated on the device by a counter-based, N-invariant generator (bench_data.py; SURVEY.md 8(d)).  One bench "step"
is ONE launch of the persistent filter kernel over `--window` (default 500) consecutive filter steps; the default
K = 20 steps cover the T = 10k sequence.  `value` = filter steps per second over all GPUs (N > 1: rows of C sharded,
strong scaling at fixed d, statistics exchanged per step through in-kernel NVLink mailboxes).

Workload B (`--workload B`; configs[4]): 4096 independent series of d = 512 rows, r = 8, T = 5,000, split over the
GPUs with no communication; `value` = series-steps per second.

Before anything is timed a PARITY PROLOGUE filters the first `--parity-steps` (default 8) steps of the very problem
being benchmarked and compares x_t, C and the replicated state with the CPU oracle (oracle/psmf_oracle_c.c, else the
numpy oracle) run by rank 0 on the global problem; the result goes into the JSON line (`parity`) and a relative error
above the tolerance (1e-9 fp64, 1e-4 fp32) ends the run with exit code 3 before any number is printed as valid.

--dump-outputs DIR writes, after the timed steps, what the last timed step computed (see dump_outputs); the inputs are
generated from a fixed seed, so two builds run with the same arguments can be compared output for output.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]  # CUDA arm
  python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # reference arm: CPU oracle port on the host cores
  python bench.py --impl nccl --gpus N ...                               # baseline: one launch per step + ncclAllReduce
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import bench_data as bd  # noqa: E402

init_state = bd.init_state
SM_COUNT = 148
SMEM_BYTES_PER_CLK_PER_SM = 128


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "nccl"])
    ap.add_argument("--workload", default="L", choices=["L", "B"])
    ap.add_argument("--d", "--rows", dest="d", type=int, default=0, help="rows of C (--rows: torchrun's parser trips over --d); default 1M (L) / 512 (B)")
    ap.add_argument("--r", type=int, default=0, help="latent rank; default 16 (L) / 8 (B)")
    ap.add_argument("--T", type=int, default=0, help="length of the resident synthetic sequence; default 10000 (L) / 5000 (B)")
    ap.add_argument("--series", type=int, default=4096, help="workload B: independent series over all GPUs")
    ap.add_argument("--window", type=int, default=500, help="filter steps per kernel launch (= per bench step)")
    ap.add_argument("--mask", default="iid", choices=["iid", "segments"],
                    help="missing pattern: iid Bernoulli (default) or runs of 20 steps per row (common.py:50-76)")
    ap.add_argument("--mask-encoding", default="nan", choices=["bytes", "nan"],
                    help="nan (default): missing entries are NaN in y -- the raw data form the reference ingests "
                         "(rPSMF.py:160-164) -- and there is no mask stream (SURVEY.md 8(d): 0 mask bytes); bytes: zero-filled y "
                         "+ one mask byte per entry (rPSMF.py:198-202)")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--ctas", type=int, default=0)
    ap.add_argument("--kernel", type=int, default=0)
    ap.add_argument("--parity-steps", type=int, default=8, help="filter steps of the parity prologue (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=0, help="filter steps of the CPU baseline sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (X, and the filter state) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA arm (--impl b200)")
    if a.workload == "L":
        a.d, a.r, a.T = a.d or 1_000_000, a.r or 16, a.T or 10_000
    else:
        a.d, a.r, a.T = a.d or 512, a.r or 8, a.T or 5_000
    return a


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self._halt = threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [s.strip() for s in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(self.samples))


# --------------------------------------------------------------------------------------------------
# configuration record shared by all arms (the driver compares it between the CUDA and the reference arm)
# --------------------------------------------------------------------------------------------------
def regime_of(c_bytes):
    """Where the C shard of one GPU lives during a launch (SURVEY.md 8(d)): decided by its size alone."""
    if c_bytes <= 147 * 112 * 1024:
        return "smem"            # resident in shared memory for the whole launch
    if c_bytes <= 70e6:
        return "l2"              # streams through the chunk ring but stays in the 126 MB L2 (ncu: 64 MB shard, 94.5 % L2 hits,
                                 # DRAM 28 MB per step against 132 MB algorithmic: profiles/traffic_r02.json)
    if c_bytes <= 126e6:
        return "hbm+l2"          # streams from HBM, a large part of it still hits in L2
    return "hbm"


def config_record(args, world):
    d, r, T, W = args.d, args.r, max(args.T // args.window, 1) * args.window, args.window
    esize = 8 if args.dtype == "f64" else 4
    mb = 0 if args.mask_encoding == "nan" else 1                # mask bytes per entry
    ym = "NaN-encoded Y" if mb == 0 else "Y/M"
    if args.workload == "B":
        S = args.series
        return dict(workload="B: %d independent rPSMF series of d=%d r=%d T=%d, 20%% missing, %s; one bench step = one kernel launch "
                             "over %d filter steps of every series" % (S, d, r, T, args.dtype, W),
                    series=S, d=d, r=r, T=T, window=W, missing=0.2, mask=args.mask, mask_encoding=args.mask_encoding, robust=True,
                    series_per_gpu=S // world,
                    l2_policy="C of every series (%.0f kB) is resident in shared memory for the whole launch; %s windows "
                              "(%.1f GB per GPU) are larger than L2 and stream from HBM" %
                              (d * r * esize / 1e3, ym, (S // world) * W * d * (esize + mb) / 1e9),
                    parallelism="series split over %d GPU(s), no communication" % world)
    from rpsmf_b200 import shard_rows
    d_loc = max(b - a for a, b in (shard_rows(d, world, k) for k in range(world)))
    regime = regime_of(d_loc * r * esize)
    pol = {"hbm": "inputs larger than L2: C (%.0f MB) and the YM windows (%.1f GB) stream from HBM every filter step",
           "hbm+l2": "C shard (%.0f MB) streams through the chunk ring and partly stays in the 126 MB L2 between filter steps (by "
                     "design: it is re-read every step); YM windows (%.1f GB) are larger than L2 and stream from HBM",
           "l2": "C shard (%.0f MB) streams through the chunk ring but fits the 126 MB L2 (by design: it is re-read every step); "
                 "YM windows (%.1f GB) are larger than L2 and stream from HBM",
           "smem": "C shard (%.0f MB) is resident in shared memory for the whole launch; YM windows (%.1f GB) are larger than "
                   "L2 and stream from HBM"}[regime].replace("YM", ym) % (d_loc * r * esize / 1e6, W * d_loc * (esize + mb) / 1e9)
    return dict(workload="L: rPSMF d=%d r=%d T=%d, 20%% missing, %s; one bench step = one kernel launch over %d filter steps"
                         % (d, r, T, args.dtype, W),
                d=d, r=r, T=T, window=W, missing=0.2, mask=args.mask, mask_encoding=args.mask_encoding, robust=True,
                rows_per_gpu=d_loc, regime=regime, l2_policy=pol, parallelism="rows of C sharded over %d GPU(s)" % world)


def metric_name(args):
    return "PSMF filter steps/sec at d=1M,r=16" if args.workload == "L" else "PSMF series-steps/sec, 4096 x (d=512, r=8)"


def unit_name(args):
    return "filter steps/s" if args.workload == "L" else "series-steps/s"


# --------------------------------------------------------------------------------------------------
# CPU oracle helpers (checker of the parity prologue, cpu_baseline leg, reference arm)
# --------------------------------------------------------------------------------------------------
def oracle_run(C0, x0, Y, M, r, want_X=True):
    """K steps of the CPU restatement: the C/OpenMP port with all host threads when built, else numpy.
    Returns (dict(C, x, P, V, X), threads, name)."""
    init = init_state(r)
    from oracle import psmf_oracle_c as pc
    if pc.available():
        threads = pc.use_all_cores()
        res = pc.run(C0, x0, init["P"], init["V"], init["Q"], init["rho"], init["lam"], Y, M, want_X=want_X)
        assert res["bad"] == -1, "CPU oracle reported a non-finite step"
        return res, threads, "oracle/psmf_oracle_c.c (C/OpenMP O(d r^2) restatement)"
    from oracle import psmf_oracle as po
    try:
        from threadpoolctl import threadpool_info
        threads = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        threads = os.cpu_count() or 1
    st = po.OracleState(np.array(C0, dtype=np.float64), np.array(x0, dtype=np.float64), init["P"], init["V"], init["Q"],
                        init["rho"], init["lam"])
    st, X, _, _ = po.run(st, po.OracleConfig(robust=True), np.asarray(Y, dtype=np.float64), np.asarray(M, dtype=np.float64))
    return dict(C=st.C, x=st.x, P=st.P, V=st.V, X=X), threads, "oracle/psmf_oracle.py (numpy/OpenBLAS O(d r^2) restatement)"


def host_prefix(torch, Y, M, n):
    """First n steps as (float64 zero-filled Y, uint8 M) host arrays, whatever the device encoding."""
    Yh = Y[..., :n, :].double()
    if M is None:
        Mh = ~torch.isnan(Yh)
        Yh = torch.nan_to_num(Yh, nan=0.0)
    else:
        Mh = M[..., :n, :] != 0
    return Yh.cpu().numpy(), Mh.to(torch.uint8).cpu().numpy()


def relerr(a, b):
    den = float(np.max(np.abs(b))) or 1.0
    return float(np.max(np.abs(np.asarray(a, dtype=np.float64) - b))) / den


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        run_reference(args, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = dict(args=args, world=world, rank=rank, local_rank=local_rank, dev=dev, torch=torch, dist=dist)
    if args.impl == "nccl":
        line, rc = run_nccl_baseline(ctx)
    elif args.workload == "B":
        line, rc = run_workload_B(ctx)
    else:
        line, rc = run_workload_L(ctx)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.exit(rc)


def bind_to_gpu_numa_node(torch, index):
    """Pin this process to the CPU cores of the NUMA node the GPU hangs off, so that the pinned staging buffers it allocates
    next are placed there (first touch): with several ranks per box, host buffers on a remote node halve the H2D rate.
    Returns a short description for the JSON line (None when the topology cannot be read)."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=10).stdout.strip().lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                          # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return "default placement (the kernel reports no NUMA node for %s)" % bus
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = set(os.sched_getaffinity(0)) & set(cpus)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return "NUMA node %d (%d cores)" % (node, len(allowed))
        return "default placement (no allowed core on NUMA node %d)" % node
    except Exception as ex:
        return "default placement (%s: %s)" % (type(ex).__name__, str(ex)[:80])


def _barrier(ctx):
    if ctx["world"] > 1:
        ctx["dist"].barrier()
    ctx["torch"].cuda.synchronize(ctx["dev"])


def _max_over_ranks(ctx, ms):
    if ctx["world"] > 1:
        t = ctx["torch"].tensor([ms], dtype=ctx["torch"].float64, device=ctx["dev"])
        ctx["dist"].all_reduce(t, op=ctx["dist"].ReduceOp.MAX)
        return float(t.item())
    return ms


def _peaks():
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    return json.load(open(pk_path)) if os.path.exists(pk_path) else {}


def measure_l2_copy_gbs(torch, dev, mbytes=16):
    """Copy bandwidth (read + write bytes) of a buffer pair that stays in L2: the denominator of an L2-resident shard."""
    n = mbytes * 1024 * 1024 // 8
    a = torch.zeros(n, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    for _ in range(5):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(5):
        e0.record()
        for _ in range(20):
            b.copy_(a)
        e1.record()
        torch.cuda.synchronize(dev)
        best = max(best, 20 * 2 * n * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def measure_hbm_copy_gbs(torch, dev, seconds=1.0, mbytes=1024):
    """Plain device copy (read + write bytes) of a buffer pair far larger than L2, back to back for ~`seconds`: the copy
    bandwidth THIS GPU sustains right after the timed region, under the same power / clock conditions.  Reported next to
    the roofline (informative); `roofline.peak` stays the driver-measured burst figure of MEASURED_PEAKS.json."""
    n = mbytes * 1024 * 1024 // 8
    a = torch.zeros(n, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        b.copy_(a)
    torch.cuda.synchronize(dev)
    reps = max(10, int(seconds * 6.0e12 / (2 * n * 8)))
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize(dev)
    return reps * 2 * n * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9


def traffic_for(d_loc, r, dtype, W):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu capture of the same
    shard size (profiles/traffic_r02.json; the N-GPU shard profiled on one GPU -- the kernel's traffic depends on its rows
    only), scaled by the row ratio when the shard differs by a tile or two; None when no capture within 1 % exists."""
    p = os.path.join(ROOT, "profiles", "traffic_r02.json")
    if not os.path.exists(p):
        return None
    try:
        best = None
        for key, rec in json.load(open(p)).get("shards", {}).items():
            rows, rr, dt = key.split(":")
            if int(rr) == r and dt == dtype and abs(int(rows) - d_loc) <= 0.01 * d_loc:
                if best is None or abs(int(rows) - d_loc) < abs(best[0] - d_loc):
                    best = (int(rows), rec["dram_bytes_per_filter_step"])
        return None if best is None else best[1] * (d_loc / best[0]) * W
    except Exception:
        return None


DUMP_FILE_BYTES = 8 << 20        # per .npy file of --dump-outputs; at most 8 files, so 64 MB in all
DUMP_SEED = 12345


def dump_outputs(ctx, arrays):
    """--dump-outputs: write `arrays` -- name -> (local, off, total) -- as DIR/<name>.npy from rank 0.  `local` holds rows
    [off, off + len(local)) of a (total, ...) array whose rows are split over the ranks; total = None marks an array that
    every rank holds whole.  An array larger than DUMP_FILE_BYTES is written as a fixed, seeded sample of its rows
    (sorted row indices), so two runs with the same arguments write the same rows.  Every rank must call this."""
    torch = ctx["torch"]
    for name, (local, off, total) in arrays.items():
        sharded = total is not None
        total = total if sharded else local.shape[0]
        row_bytes = local[:1].numel() * local.element_size()
        k = max(1, DUMP_FILE_BYTES // row_bytes)
        idx = torch.arange(total) if total <= k else torch.from_numpy(np.sort(np.random.default_rng(DUMP_SEED).choice(total, k, replace=False)))
        mine = (idx >= off) & (idx < off + local.shape[0])
        out = torch.zeros((len(idx),) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        out[mine.to(local.device)] = local[(idx[mine] - off).to(local.device)]
        if sharded and ctx["world"] > 1:
            ctx["dist"].all_reduce(out)          # every row has one owner and zeros elsewhere: the sum is exact
        if ctx["rank"] == 0:
            os.makedirs(ctx["args"].dump_outputs, exist_ok=True)
            np.save(os.path.join(ctx["args"].dump_outputs, name + ".npy"), out.cpu().numpy())


# --------------------------------------------------------------------------------------------------
# workload L
# --------------------------------------------------------------------------------------------------
def run_workload_L(ctx):
    args, world, rank, dev, torch, dist = (ctx[k] for k in ("args", "world", "rank", "dev", "torch", "dist"))
    from rpsmf_b200 import FilterEngine, shard_rows
    d, r, W = args.d, args.r, args.window
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    esize = 8 if args.dtype == "f64" else 4
    nan_enc = args.mask_encoding == "nan"
    row0, row1 = shard_rows(d, world, rank)
    d_loc = row1 - row0
    T = max(args.T // W, 1) * W
    nwin = T // W

    def allreduce(v):
        if world > 1:
            dist.all_reduce(v)
        return v

    Y, M, C0, x0 = bd.make_series(torch, dev, d_loc, row0, d, r, T, dtype, mask=args.mask, nan_encoded=nan_enc, allreduce=allreduce)
    torch.cuda.empty_cache()                 # the generator's temporaries go back to the driver (the data alone is 90 GB)
    init = init_state(r)
    eng = FilterEngine(d_loc, r, dtype=dtype, robust=True, device=ctx["local_rank"], d_global=d, world_size=world, rank=rank,
                       ctas=args.ctas, kernel=args.kernel, nan_mask=nan_enc)
    if world > 1:
        eng.connect(dist)

    def reset():
        eng.set_state(C_=C0.to(dtype), V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])

    # ---- parity prologue: the first K steps of THIS problem against the CPU oracle on the global rows ----
    parity, rc = None, 0
    K = min(args.parity_steps, T)
    if K > 0:
        reset()
        out = eng.run(Y[:K], None if M is None else M[:K], k0=1, want_X=True)
        bad = eng.status()
        Xg = out["X"].clone()
        st = eng.get_state()
        same = True
        if world > 1:
            allx = [torch.empty_like(Xg) for _ in range(world)]
            dist.all_gather(allx, Xg)
            small = torch.cat([st["x"].reshape(-1), st["P"].reshape(-1), st["V"].reshape(-1), st["rho"].reshape(-1), st["lam"].reshape(-1)])
            alls = [torch.empty_like(small) for _ in range(world)]
            dist.all_gather(alls, small)
            same = all(torch.equal(allx[0], g) for g in allx) and all(torch.equal(alls[0], g) for g in alls)
        Cref = torch.empty((d, r), dtype=torch.float64, device=dev) if world > 1 else None
        xerr = perr = verr = None
        tol = 1e-9 if args.dtype == "f64" else 1e-4
        if rank == 0:
            # rank 0 regenerates the GLOBAL problem for the first K steps (the generator is N-invariant)
            Yg, Mg, C0g, _ = (Y, M, C0, None) if world == 1 else bd.make_series(torch, dev, d, 0, d, r, K, dtype, mask=args.mask,
                                                                                nan_encoded=nan_enc)
            if world > 1 and args.mask == "segments":
                raise SystemExit("parity prologue with --mask segments needs the global mask: run it with --gpus 1")
            Yh, Mh = host_prefix(torch, Yg, Mg, K)
            ref, threads, what = oracle_run(C0g.to(dtype).double().cpu().numpy(), x0.numpy(), Yh, Mh, r)
            xerr = relerr(Xg.cpu().numpy(), ref["X"])
            perr = relerr(st["P"].cpu().numpy(), ref["P"])
            verr = relerr(st["V"].cpu().numpy(), ref["V"])
            if world > 1:
                Cref.copy_(torch.as_tensor(ref["C"]))
            else:
                Cref = torch.as_tensor(ref["C"]).to(dev)
            del Yg, Mg, C0g
        if world > 1:
            dist.broadcast(Cref, 0)
        mine = Cref[row0:row1]
        cerr_t = torch.stack([(st["C"].double() - mine).abs().max(), Cref.abs().max()])
        if world > 1:
            dist.all_reduce(cerr_t, op=dist.ReduceOp.MAX)
        cerr = float(cerr_t[0] / cerr_t[1])
        del Cref, mine
        if rank == 0:
            ok = bool(same and bad == -1 and max(xerr, cerr, perr, verr) < tol)
            parity = dict(steps=K, X_relerr=xerr, C_relerr=cerr, P_relerr=perr, V_relerr=verr, replicas_identical=bool(same),
                          tolerance=tol, checker=what, checker_threads=threads, ok=ok,
                          X_checksum=float(Xg.double().sum()))
            rc = 0 if ok else 3
        flag = torch.tensor([rc], device=dev)
        if world > 1:
            dist.broadcast(flag, 0)
        rc = int(flag.item())
        if rc != 0:
            line = dict(metric=metric_name(args), value=None, unit=unit_name(args), n_gpus=world, parity=parity,
                        error="parity prologue FAILED: the CUDA path does not match the CPU oracle; nothing was timed")
            eng.close()
            return line, rc

    reset()
    Xbuf = torch.empty((1, W, r), dtype=torch.float64, device=dev)

    def one_step(i):
        w = i % nwin
        eng.run(Y[w * W:(w + 1) * W], None if M is None else M[w * W:(w + 1) * W], k0=1 + i * W, want_X=False, X_out=Xbuf)

    torch.cuda.profiler.start()          # ncu --profile-from-start off: skip the data generation kernels
    for i in range(args.warmup):
        one_step(i)
    _barrier(ctx)
    sampler = ClockSampler(ctx["local_rank"])
    sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    _barrier(ctx)
    evs[0].record()
    for i in range(args.steps):
        one_step(args.warmup + i)
        evs[i + 1].record()
    _barrier(ctx)
    clocks = sampler.stop()
    torch.cuda.profiler.stop()
    bad = eng.status()
    total_ms = _max_over_ranks(ctx, evs[0].elapsed_time(evs[-1]))
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    filter_steps = args.steps * W
    value = filter_steps / (total_ms * 1e-3)
    info = eng.launch_info()
    if args.dump_outputs:
        # X of the last launch (W, r) and the state it leaves: C row-sharded, the rest replicated (leading dim: 1 series)
        st = eng.get_state()
        arrays = {"X": (Xbuf[0], 0, None), "C": (st["C"], row0, d)}
        arrays.update({k: (st[k].unsqueeze(0), 0, None) for k in ("x", "P", "V", "Q", "rho", "lam")})
        dump_outputs(ctx, arrays)

    # ---- roofline of the dominant (only) kernel, against the bound of ITS regime (SURVEY.md 8(d)) ----
    peaks = _peaks()
    mean_launch_s = float(np.mean(per_launch_ms)) * 1e-3
    mask_bytes = 0 if nan_enc else d_loc
    hbm_step = d_loc * esize + mask_bytes                      # y_t + mask byte: streamed in every regime
    c_step = 2 * d_loc * r * esize                             # one read + one write of the C shard
    regime = "smem" if info.get("resident") else regime_of(d_loc * r * esize)
    kname = "%s<%d,%s>" % ("psmf_stream_kernel" if info.get("kernel") == "tma" else "psmf_filter_kernel", r, "double" if esize == 8 else "float")
    if regime == "smem":
        clk = (clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0) * 1e6
        peak = SM_COUNT * SMEM_BYTES_PER_CLK_PER_SM * clk / 1e9
        alg = c_step
        roofline = dict(bound="smem", peak_source="148 SMs x 128 B/clk x the SM clock observed under load (%.0f MHz)" % (clk / 1e6),
                        hbm_bytes_per_filter_step=hbm_step, hbm_achieved_gbs=hbm_step * W / mean_launch_s / 1e9,
                        note="latency-bound regime: the step is the chain pass -> reduction -> r x r solve -> publish (two steps in "
                             "flight), see profiles/")
    elif regime == "l2":
        peak = measure_l2_copy_gbs(torch, dev)
        alg = c_step + hbm_step
        roofline = dict(bound="l2", peak_source="measured live: torch copy of an L2-resident 16 MB buffer pair (read + write bytes)",
                        hbm_bytes_per_filter_step=hbm_step, hbm_achieved_gbs=hbm_step * W / mean_launch_s / 1e9)
    else:
        peak = float(peaks.get("hbm_gbs", 6650.0))
        alg = c_step + hbm_step
        roofline = dict(bound="hbm", peak_source="MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s")
        if regime == "hbm+l2":
            roofline["note"] = "the C shard (%.0f MB) partly stays in the 126 MB L2 between steps: frac can exceed 1 against the HBM peak" % (
                d_loc * r * esize / 1e6)
    achieved = alg * W / mean_launch_s / 1e9
    if regime == "hbm" and world == 1:
        try:
            roofline["copy_sustained_gbs_now"] = measure_hbm_copy_gbs(torch, dev)
            roofline["copy_sustained_note"] = ("torch copy of a 1 GiB buffer pair for ~1 s on this GPU right after the timed region "
                                               "(informative: what a plain copy sustains under the same power cap)")
        except Exception:
            pass
    roofline.update(achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic_for(d_loc, r, args.dtype, W),
                    algorithmic_bytes_per_filter_step=alg, kernel=kname, mean_launch_ms=float(np.mean(per_launch_ms)), regime=regime)

    # ---- end to end through the public API with HOST buffers (pinned), H2D inside the timed region ----
    e2e = None
    if not args.no_e2e:
        nw = min(2, nwin)
        numa = bind_to_gpu_numa_node(torch, ctx["local_rank"])
        Yh = torch.empty((nw * W, d_loc), dtype=dtype).pin_memory()
        Yh.copy_(Y[: nw * W])
        Mh = None
        if M is not None:
            Mh = torch.empty((nw * W, d_loc), dtype=torch.uint8).pin_memory()
            Mh.copy_(M[: nw * W])
        reset()
        eng.run_host(Yh[:W], None if Mh is None else Mh[:W], window=min(W, 125), k0=1)      # warm-up (allocates the staging buffers)
        reset()
        _barrier(ctx)
        t0 = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        Xh = eng.run_host(Yh, Mh, window=min(W, 125), k0=1)
        e1.record()
        _barrier(ctx)
        ms = _max_over_ranks(ctx, e0.elapsed_time(e1))
        e2e = dict(value=nw * W / (ms * 1e-3), unit=unit_name(args),
                   h2d_bytes_per_step=int((d_loc * esize + mask_bytes) * W), d2h_bytes_per_step=int(W * r * 8),
                   wall_s=time.perf_counter() - t0, host_buffers=numa or "default placement",
                   note="per bench step of %d filter steps; pinned host Y%s, double-buffered H2D; the "
                   "run starts from the initial state, so `checksum` (sum of the filtered x_t) is the same for every N" % (W, "" if nan_enc else "/M"),
                   checksum=float(Xh.sum()))
        del Yh, Mh

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:                      # reported at N = 1 only
        ns = args.cpu_steps or max(8, min(400, int(300e6 / max(d, 1))))     # ~10-20 s of host work at d = 1M
        ns = min(ns, T)
        Yh, Mh = host_prefix(torch, Y, M, ns)
        C0h = C0.cpu().numpy()
        oracle_run(C0h[:1024], x0.numpy(), Yh[:2, :1024], Mh[:2, :1024], r)              # warm-up (threads, page faults)
        t0 = time.perf_counter()
        _, threads, what = oracle_run(C0h, x0.numpy(), Yh, Mh, r, want_X=False)
        dt = time.perf_counter() - t0
        cpu = dict(value=ns / dt, unit=unit_name(args), cores=threads, kind="port",
                   sample="%d filter steps of the same workload prefix (d=%d rows, r=%d) through %s; the reference's "
                          "d x d form cannot run at d=1M" % (ns, d_loc, r, what))

    line = None
    if rank == 0:
        line = dict(
            metric=metric_name(args), value=value, unit=unit_name(args), n_gpus=world,
            steps=args.steps, warmup=args.warmup, ms_per_step=total_ms / args.steps, higher_is_better=True,
            scaling="strong", vs_baseline=None, dtype=args.dtype, data="synthetic",
            config=config_record(args, world), parity=parity,
            e2e=e2e, gpu_launches=args.steps, roofline=roofline, cpu_baseline=cpu, clocks=clocks,
            launch=info, first_bad_step=bad)
    eng.close()
    return line, 0


# --------------------------------------------------------------------------------------------------
# workload B: independent series, no communication
# --------------------------------------------------------------------------------------------------
def run_workload_B(ctx):
    args, world, rank, dev, torch, dist = (ctx[k] for k in ("args", "world", "rank", "dev", "torch", "dist"))
    from rpsmf_b200 import FilterEngine, shard_series
    d, r, W, S = args.d, args.r, args.window, args.series
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    esize = 8 if args.dtype == "f64" else 4
    nan_enc = args.mask_encoding == "nan"
    s0, s1 = shard_series(S, world, rank)
    S_loc = s1 - s0
    T = max(args.T // W, 1) * W
    nwin = T // W
    Y, M, C0, x0 = bd.make_batch(torch, dev, s0, S_loc, S, d, r, T, dtype, nan_encoded=nan_enc)
    init = init_state(r)
    eng = FilterEngine(d, r, n_series=S_loc, dtype=dtype, robust=True, device=ctx["local_rank"], nan_mask=nan_enc, ctas=args.ctas,
                       kernel=args.kernel)

    def reset():
        eng.set_state(C_=C0.to(dtype), V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])

    # ---- parity prologue: a sample of this rank's series over the first K steps against the CPU oracle ----
    parity, rc = None, 0
    K = min(args.parity_steps * 4, T)
    if K > 0:
        reset()
        out = eng.run(Y[:, :K], None if M is None else M[:, :K], k0=1, want_X=True)
        bad = eng.status()
        st = eng.get_state()
        sample = sorted(set([0, S_loc // 3, (2 * S_loc) // 3, S_loc - 1]))
        tol = 1e-9 if args.dtype == "f64" else 1e-4
        errs = []
        what, threads = None, None
        for s in sample:
            Yh, Mh = host_prefix(torch, Y[s], None if M is None else M[s], K)
            ref, threads, what = oracle_run(C0[s].to(dtype).double().cpu().numpy(), x0[s].cpu().numpy(), Yh, Mh, r)
            Xs = out["X"][s] if S_loc > 1 else out["X"]
            Cs = st["C"][s] if S_loc > 1 else st["C"]
            errs.append(max(relerr(Xs.cpu().numpy(), ref["X"]), relerr(Cs.double().cpu().numpy(), ref["C"])))
        worst = torch.tensor([max(errs), float(bad != -1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        ok = bool(float(worst[0]) < tol and float(worst[1]) == 0.0)
        parity = dict(steps=K, series_checked_per_gpu=len(sample), max_relerr_X_C=float(worst[0]), tolerance=tol, checker=what,
                      checker_threads=threads, ok=ok, X_checksum_rank0=float(out["X"].double().sum()))
        rc = 0 if ok else 3
        if rc != 0:
            eng.close()
            return dict(metric=metric_name(args), value=None, unit=unit_name(args), n_gpus=world, parity=parity,
                        error="parity prologue FAILED: the CUDA path does not match the CPU oracle; nothing was timed"), rc

    reset()

    def one_step(i):
        w = i % nwin
        eng.run(Y[:, w * W:(w + 1) * W], None if M is None else M[:, w * W:(w + 1) * W], k0=1 + i * W, want_X=False)

    torch.cuda.profiler.start()
    for i in range(args.warmup):
        one_step(i)
    _barrier(ctx)
    sampler = ClockSampler(ctx["local_rank"])
    sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    _barrier(ctx)
    evs[0].record()
    for i in range(args.steps):
        one_step(args.warmup + i)
        evs[i + 1].record()
    _barrier(ctx)
    clocks = sampler.stop()
    torch.cuda.profiler.stop()
    bad = eng.status()
    total_ms = _max_over_ranks(ctx, evs[0].elapsed_time(evs[-1]))
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    value = args.steps * W * S / (total_ms * 1e-3)
    info = eng.launch_info()
    if args.dump_outputs:
        # the timed launches return no X: the state they leave, series-sharded (C as rows of (series, row) pairs)
        st = {k: (v.unsqueeze(0) if S_loc == 1 else v) for k, v in eng.get_state().items() if v is not None}
        arrays = {"C": (st["C"].reshape(S_loc * d, r), s0 * d, S * d)}
        arrays.update({k: (st[k], s0, S) for k in ("x", "P", "V", "Q", "rho", "lam")})
        dump_outputs(ctx, arrays)
    peaks = _peaks()
    mean_launch_s = float(np.mean(per_launch_ms)) * 1e-3
    clk = (clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0) * 1e6
    peak = SM_COUNT * SMEM_BYTES_PER_CLK_PER_SM * clk / 1e9
    alg = 2 * d * r * esize                                     # per series-step: one read + one write of the resident C
    hbm = d * esize + (0 if nan_enc else d)
    achieved = alg * W * S_loc / mean_launch_s / 1e9
    roofline = dict(bound="smem", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=None,
                    peak_source="148 SMs x 128 B/clk x the SM clock observed under load (%.0f MHz)" % (clk / 1e6),
                    algorithmic_bytes_per_series_step=alg, hbm_bytes_per_series_step=hbm,
                    hbm_achieved_gbs=hbm * W * S_loc / mean_launch_s / 1e9,
                    fp64_flops_per_series_step=d * (r * (r + 1) + 6 * r + 10),
                    fp64_achieved_tflops=d * (r * (r + 1) + 6 * r + 10) * W * S_loc / mean_launch_s / 1e12,
                    kernel="%s<%d,%s>" % ({"batch": "psmf_batch_kernel", "direct": "psmf_filter_kernel"}.get(info.get("kernel"), "?"), r,
                                          "double" if esize == 8 else "float"),
                    mean_launch_ms=float(np.mean(per_launch_ms)), regime="smem",
                    note="C of a series stays in shared memory for the launch; the step is bound by its per-series latency chain "
                         "(pass -> CTA reduction -> r x r solve) times the CTAs resident per SM")

    e2e = None
    if not args.no_e2e:
        ns = min(S_loc, 64)                                     # a bounded slice of the batch through host buffers
        Yh = torch.empty((ns, W, d), dtype=dtype).pin_memory()
        Yh.copy_(Y[:ns, :W])
        Mh = None
        if M is not None:
            Mh = torch.empty((ns, W, d), dtype=torch.uint8).pin_memory()
            Mh.copy_(M[:ns, :W])
        eng2 = FilterEngine(d, r, n_series=ns, dtype=dtype, robust=True, device=ctx["local_rank"], nan_mask=nan_enc)
        eng2.set_state(C_=C0[:ns].to(dtype), V=init["V"], P=init["P"], x=x0[:ns], Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        Xh = torch.empty((ns, W, r), dtype=torch.float64).pin_memory()

        def host_step():
            Yd = Yh.to(dev, non_blocking=True)
            Md = None if Mh is None else Mh.to(dev, non_blocking=True)
            o = eng2.run(Yd, Md, k0=1, want_X=True)
            Xh.copy_(o["X"].reshape(ns, W, r), non_blocking=True)
            torch.cuda.synchronize(dev)
        host_step()
        _barrier(ctx)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 3
        for _ in range(reps):
            host_step()
        e1.record()
        _barrier(ctx)
        ms = _max_over_ranks(ctx, e0.elapsed_time(e1))
        e2e = dict(value=reps * ns * W * world / (ms * 1e-3), unit=unit_name(args),
                   h2d_bytes_per_step=int(ns * W * (d * esize + (0 if nan_enc else d))), d2h_bytes_per_step=int(ns * W * r * 8),
                   note="%d series x %d steps per host call from pinned host Y/M, X read back; PCIe-bound" % (ns, W),
                   checksum=float(Xh.sum()))
        eng2.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ns = min(T, args.cpu_steps or 2000)
        Yh1, Mh1 = host_prefix(torch, Y[0], None if M is None else M[0], ns)
        t0 = time.perf_counter()
        _, threads, what = oracle_run(C0[0].cpu().numpy(), x0[0].cpu().numpy(), Yh1, Mh1, r, want_X=False)
        dt = time.perf_counter() - t0
        cpu = dict(value=ns / dt, unit=unit_name(args), cores=threads, kind="port",
                   sample="ONE series (d=%d, r=%d), %d filter steps through %s" % (d, r, ns, what))

    line = None
    if rank == 0:
        line = dict(metric=metric_name(args), value=value, unit=unit_name(args), n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=total_ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype=args.dtype,
                    data="synthetic", config=config_record(args, world), parity=parity, e2e=e2e, gpu_launches=args.steps,
                    roofline=roofline, cpu_baseline=cpu, clocks=clocks, launch=info, first_bad_step=bad)
    eng.close()
    return line, 0


# --------------------------------------------------------------------------------------------------
# NCCL baseline arm (north_star: "in-kernel NVLink P2P stores with NCCL as the baseline")
# --------------------------------------------------------------------------------------------------
def run_nccl_baseline(ctx):
    """Same workload, same kernels' arithmetic, but the per-step statistics exchange is ncclAllReduce: the filter runs ONE
    step per launch in split-phase mode (exchange = external): pass + grid reduction -> all-reduce of the statistics
    vector on the stream -> r x r update.  A bench step is `window` such filter steps."""
    args, world, rank, dev, torch, dist = (ctx[k] for k in ("args", "world", "rank", "dev", "torch", "dist"))
    from rpsmf_b200 import FilterEngine, shard_rows
    d, r = args.d, args.r
    W = min(args.window, 100)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    row0, row1 = shard_rows(d, world, rank)
    d_loc = row1 - row0
    T = W * 4
    nan_enc = args.mask_encoding == "nan"
    Y, M, C0, x0 = bd.make_series(torch, dev, d_loc, row0, d, r, T, dtype, mask=args.mask, nan_encoded=nan_enc)
    init = init_state(r)
    eng = FilterEngine(d_loc, r, dtype=dtype, robust=True, device=ctx["local_rank"], d_global=d, world_size=world, rank=rank,
                       exchange="external", nan_mask=nan_enc)
    eng.set_state(C_=C0.to(dtype), V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    stats = eng.stats_buffer()

    def allreduce(buf):
        if world > 1:
            dist.all_reduce(buf)

    # parity: K steps against the in-kernel mailbox path is covered by tests; here against the oracle at N = 1 shape
    X = torch.empty((T, r), dtype=torch.float64, device=dev)

    def one_filter_step(t, k):
        eng.run_split(Y[t:t + 1], None if M is None else M[t:t + 1], k0=k, allreduce=allreduce, X_out=X[t:t + 1])

    for t in range(min(W, 20)):
        one_filter_step(t, 1 + t)
    _barrier(ctx)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 0
    e0.record()
    for i in range(args.steps):
        for t in range(W):
            one_filter_step((i * W + t) % T, 21 + n)
            n += 1
    e1.record()
    _barrier(ctx)
    ms = _max_over_ranks(ctx, e0.elapsed_time(e1))
    bad = eng.status()
    line = dict(impl="nccl", metric=metric_name(args), value=n / (ms * 1e-3), unit=unit_name(args), n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms / args.steps, us_per_filter_step=ms * 1e3 / n, higher_is_better=True,
                scaling="strong", vs_baseline=None, dtype=args.dtype, data="synthetic", config=config_record(args, world),
                gpu_launches=2 * n, first_bad_step=bad, nstat=int(stats.numel()),
                note="baseline arm: one filter step = pass kernel -> ncclAllReduce(%d doubles) -> update kernel, host-driven; the "
                     "product path runs all steps in ONE persistent launch with the exchange inside the kernel" % int(stats.numel()))
    eng.close()
    return line, 0


# --------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU algorithm (oracle port) on the host cores
# --------------------------------------------------------------------------------------------------
def run_reference(args, world):
    """Reference arm: the reference's own CPU algorithm (oracle port; the d x d reference code cannot run at
    d = 1M) on the host cores, same config / metric / unit.  A bench step is a bounded sample of filter steps."""
    d, r = args.d, args.r
    est = 0.05 * d / 1e6 + 1e-4                      # seconds per filter step of the C/OpenMP port (8 threads)
    per_step = int(max(1, min(40, 40.0 / ((args.steps + args.warmup) * est))))
    if args.workload == "B":
        per_step = 500
    rng = np.random.RandomState(bd.SEED % (2 ** 31))
    Ct = rng.randn(d, r)
    x = rng.randn(r)
    Y = np.empty((per_step, d)); M = np.empty((per_step, d), dtype=np.uint8)
    for t in range(per_step):
        x = x + 0.1 * rng.randn(r)
        M[t] = rng.rand(d) >= 0.2
        Y[t] = (Ct @ x + np.sqrt(0.1) * rng.standard_t(3, d)) * M[t]
    C0 = rng.rand(d, r); x0 = rng.rand(r)
    init = init_state(r)
    from oracle import psmf_oracle_c as pc
    if pc.available():
        threads = pc.use_all_cores()
        what = "oracle/psmf_oracle_c.c (C/OpenMP port, %d threads)" % threads
        st = dict(C=C0, x=x0, P=init["P"], V=init["V"], Q=init["Q"], rho=init["rho"], lam=init["lam"])

        def advance(a, b):
            res = pc.run(st["C"], st["x"], st["P"], st["V"], st["Q"], st["rho"], st["lam"], Y[a:b], M[a:b], want_X=False)
            st.update({k: res[k] for k in ("C", "x", "P", "V", "Q", "rho", "lam")})
    else:
        from oracle import psmf_oracle as po
        try:
            from threadpoolctl import threadpool_info
            threads = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
        except Exception:
            threads = os.cpu_count() or 1
        what = "oracle/psmf_oracle.py (numpy/OpenBLAS port)"
        box = [po.OracleState(C0, x0, init["P"], init["V"], init["Q"], init["rho"], init["lam"])]
        cfg = po.OracleConfig(robust=True)

        def advance(a, b):
            for t in range(a, b):
                box[0], _ = po.step(box[0], cfg, Y[t], M[t].astype(np.float64))
    for _ in range(args.warmup):
        advance(0, per_step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        advance(0, per_step)
    dt = time.perf_counter() - t0
    v = args.steps * per_step / dt
    if args.workload == "B":
        sample = "ONE series at a time: %d filter steps per bench step, d=%d r=%d, %s" % (per_step, d, r, what)
    else:
        sample = "%d filter steps per bench step on a pool of %d synthetic steps of the same shape, d=%d r=%d, %s" % (
            per_step, per_step, d, r, what)
    line = dict(impl="reference", metric=metric_name(args), value=v, unit=unit_name(args),
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=dt / args.steps * 1e3,
                higher_is_better=True, scaling="strong", vs_baseline=None, dtype=args.dtype, data="synthetic",
                config=config_record(args, max(1, args.gpus)),
                cpu_baseline=dict(value=v, unit=unit_name(args), cores=threads, kind="port", sample=sample),
                e2e=dict(value=v, unit=unit_name(args), h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
