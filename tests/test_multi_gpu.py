"""N > 1 path.

* CPU (gloo, world_size 2): the exchange protocol of the row-sharded filter -- every rank reduces the
  sufficient statistics of its row shard, all ranks add the per-rank totals in rank order and run the same
  r x r update -- reproduces the unsharded oracle, and the replicated state is bit-identical on all ranks.
* GPU (needs >= 2 devices): tests/multi_gpu_check.py under torchrun.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import psmf_oracle as po
    from synth import impute_init, make_problem
    from rpsmf_b200 import shard_rows
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    d, r, T = 333, 6, 25
    Y, M, C0, x0 = make_problem(d, r, T, seed=42)
    init = impute_init(r)
    b, e = shard_rows(d, world, rank)
    cfg = po.OracleConfig(robust=True, d_global=d)
    st = po.OracleState(C0[b:e].copy(), x0.copy(), init["P"], init["V"], init["Q"], init["rho"], init["lam"])
    keys = ("s", "q1", "q0", "nobs")
    X = np.zeros((T, r))
    for t in range(T):
        xbar, F = po.dynamics(cfg.dynamics, None, st.x, t + 1)
        vx = st.V @ xbar; vxt = st.V.T @ xbar; a = float(xbar @ vx)
        yhat, err, S = po.local_stats(st.C, xbar, a, st.rho, Y[t, b:e], M[t, b:e].astype(float))
        vec = np.concatenate([S["G"].ravel(), S["b"], [S[k] for k in keys]])
        allv = [torch.zeros(vec.size, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(allv, torch.from_numpy(vec))
        tot = np.zeros(vec.size)
        for v in allv:                                  # rank order, the same on every rank
            tot = tot + v.numpy()
        Sg = dict(G=tot[: r * r].reshape(r, r), b=tot[r * r: r * r + r], **{k: float(tot[r * r + r + i]) for i, k in enumerate(keys)})
        x_new, P_new, V_new, Q_new, rho_new, lam_new, g, scal = po.small_update(st, cfg, xbar, F, vx, vxt, a, Sg, d)
        st = po.OracleState(st.C + np.outer(err, g), x_new, P_new, V_new, Q_new, rho_new, lam_new)
        X[t] = x_new
    ref = po.OracleState(C0.copy(), x0.copy(), init["P"], init["V"], init["Q"], init["rho"], init["lam"])
    ref, oX, _, _ = po.run(ref, po.OracleConfig(robust=True), Y, M.astype(float))
    xs = [torch.zeros(T * r, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(xs, torch.from_numpy(X.ravel().copy()))
    same = all(torch.equal(xs[0], x) for x in xs)
    err_x = float(np.max(np.abs(X - oX)) / np.max(np.abs(oX)))
    err_c = float(np.max(np.abs(st.C - ref.C[b:e])) / np.max(np.abs(ref.C)))
    out.put((rank, same, err_x, err_c, (b, e)))
    dist.destroy_process_group()


def test_sharded_statistics_exchange_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 400)
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(60)
    rows = sorted(r[4] for r in res)
    assert rows[0][0] == 0 and rows[0][1] == rows[1][0] and rows[1][1] == 333
    for rank, same, err_x, err_c, _ in res:
        assert same, "replicated x_t differs between ranks"
        assert err_x < 1e-9 and err_c < 1e-9


def test_shard_rows_partition():
    from rpsmf_b200 import shard_rows
    for d in (1, 31, 32, 33, 1000, 1_000_000):
        for world in (1, 2, 3, 4, 8):
            parts = [shard_rows(d, world, r) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == d
            for a, b in zip(parts[:-1], parts[1:]):
                assert a[1] == b[0] and a[1] % 32 == 0
    assert shard_rows(1_000_000, 8, 0) == (0, 124992)


@pytest.mark.gpu
def test_row_sharded_filter_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29511", os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def _torchrun(nproc, port, *extra, env=None, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "multi_gpu_check.py")] + list(extra)
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=e)


@pytest.mark.gpu
@pytest.mark.parametrize("nranks", [2, 5, 8])
def test_row_sharded_filter_ranks_share_one_gpu(nranks):
    """The N > 1 CUDA path where only ONE GPU is leased: the ranks share cuda:0, their persistent kernels time-slice
    on the device and exchange the statistics through each other's mailboxes (CUDA IPC).  Same checks as the
    multi-GPU run: bit-identical replicas, 1e-9 against the unsharded oracle, one collectively chosen kernel.
    (5 and 8 ranks: a miscompiled gather over more than one peer went unnoticed with 2.)"""
    r = _torchrun(nranks, 29513 + nranks, "--same-device", "--quick", env={"PSMF_SPIN_TIMEOUT_MS": "60000"})
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count(" OK") >= 3 * nranks and "FAIL" not in r.stdout


@pytest.mark.gpu
def test_gather_ranks_unit():
    """gather_ranks (the rank-ordered, concurrently polled sum of one statistics entry over the GPUs) in isolation: every
    world size 2..8, first / last rank, with and without a local tagged cell, peers arriving one after the other."""
    import shutil
    import tempfile
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "gather_test")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-I", os.path.join(ROOT, "rpsmf_b200", "csrc"),
                        os.path.join(ROOT, "tests", "cuda", "gather_test.cu"), "-o", exe], check=True, timeout=600)
        r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.count(": ok") == 28 and "FAIL" not in r.stdout, r.stdout[-2000:]


@pytest.mark.gpu
def test_deserting_rank_times_out_instead_of_hanging():
    """A rank that dies after connecting must not hang the others: the bounded waits expire, the launch drains and
    psmf_status returns PSMF_E_STATE."""
    r = _torchrun(2, 29514, "--same-device", "--desert", "1", env={"PSMF_SPIN_TIMEOUT_MS": "1500"}, timeout=180)
    assert "rank 0:" in r.stdout and "OK" in r.stdout and "FAIL" not in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
