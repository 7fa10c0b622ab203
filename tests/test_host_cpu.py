"""CPU-only tests: the C-ABI library loads and exports every symbol the header declares (no compute calls
without a GPU), and the host-side logic of the Python surface."""

import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "psmf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(psmf_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from rpsmf_b200 import _capi
    names = _header_functions()
    assert len(names) >= 12
    assert sorted(_capi.EXPORTS) == names, "rpsmf_b200/_capi.py EXPORTS is out of sync with include/psmf_b200.h"
    lib = ctypes.CDLL(_capi.LIB_PATH)
    for n in names:
        assert getattr(lib, n) is not None
    assert _capi.lib().psmf_version() >= 100


def test_struct_layouts_match_header():
    from rpsmf_b200 import _capi
    # psmf_config: 2 x int64, 10 x int32, 2 x double, 2 x int32; psmf_io: 20 pointer / int64 / double slots
    assert ctypes.sizeof(_capi.PsmfConfig) == 2 * 8 + 10 * 4 + 2 * 8 + 2 * 4
    assert ctypes.sizeof(_capi.PsmfIO) == 20 * 8
    hdr = open(os.path.join(ROOT, "include", "psmf_b200.h")).read()
    for flag, val in (("PSMF_ROBUST", _capi.ROBUST), ("PSMF_SIMPLIFIED", _capi.SIMPLIFIED), ("PSMF_CUPDATE_VT", _capi.CUPDATE_VT),
                      ("PSMF_FIXED_LAMBDA", _capi.FIXED_LAMBDA), ("PSMF_LL_STUDENT", _capi.LL_STUDENT), ("PSMF_NAN_MASK", _capi.NAN_MASK),
                      ("PSMF_DYN_LINEAR", _capi.DYN_LINEAR), ("PSMF_KERNEL_BATCH", _capi.KERNEL_BATCH), ("PSMF_XCHG_EXTERNAL", _capi.XCHG_EXTERNAL),
                      ("PSMF_NEVAL", _capi.NEVAL), ("PSMF_EVAL_INSIDE", _capi.EVAL_INSIDE), ("PSMF_EVAL_COUNT", _capi.EVAL_COUNT),
                      ("PSMF_MAILBOX_BLOB_BYTES", _capi.MAILBOX_BLOB_BYTES),
                      ("PSMF_DYN_COS", _capi.DYN_COS), ("PSMF_DYN_EXTERNAL", _capi.DYN_EXTERNAL), ("PSMF_NSCAL", _capi.NSCAL)):
        m = re.search(r"#define\s+%s\s+(\d+)" % flag, hdr)
        assert m and int(m.group(1)) == val, flag


def test_create_without_gpu_fails_loudly():
    """No CPU fallback: without a device psmf_create returns an error code and a message."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a machine without a GPU")
    from rpsmf_b200 import _capi, FilterEngine
    L = _capi.lib()
    h = ctypes.c_void_p()
    cfg = _capi.PsmfConfig(d=64, d_global=64, r=4, n_series=1, dtype=0, flags=1, dynamics=0, device=0, world_size=1, rank=0,
                           ctas=0, kernel=0, alpha=1.0, beta=1.0)
    rc = L.psmf_create(ctypes.byref(h), ctypes.byref(cfg))
    assert rc < 0 and not h.value
    assert L.psmf_last_error(None)
    with pytest.raises(RuntimeError):
        FilterEngine(64, 4)
    bad = _capi.PsmfConfig(d=64, d_global=64, r=17, n_series=1, dtype=0, flags=0, dynamics=0, device=0, world_size=1, rank=0,
                           ctas=0, kernel=0, alpha=1.0, beta=1.0)
    assert L.psmf_create(ctypes.byref(h), ctypes.byref(bad)) == -1
    assert b"rank" in L.psmf_last_error(None)


def test_classify_and_jacobian():
    from rpsmf_b200 import _capi
    from rpsmf_b200.nonlinearities import RandomWalk, classify, cos_phase, jacobian_x
    assert classify(RandomWalk(), 3) == _capi.DYN_IDENTITY
    assert classify(cos_phase, 3) == _capi.DYN_COS
    assert classify(lambda th, x, t: np.cos(2 * np.pi * th * t + x), 5) == _capi.DYN_COS     # untagged, probed
    assert classify(lambda th, x, t: x, 2) == _capi.DYN_IDENTITY
    assert classify(lambda th, x, t: np.tanh(x), 2) == _capi.DYN_EXTERNAL
    A = np.array([[1.0, 0.2], [-0.3, 0.9]])
    x = np.array([[0.3], [-0.7]])
    F = jacobian_x(lambda th, x, t: np.tanh(A @ x), None, x, 1)
    assert np.allclose(F, (1 - np.tanh(A @ x) ** 2) * A, atol=1e-14)
    Fd = jacobian_x(lambda th, x, t: np.abs(x) * x, None, x, 1)           # not analytic -> central differences
    assert np.allclose(Fd, np.diag(2 * np.abs(x).reshape(-1)), atol=1e-6)


def test_r_and_q_validation():
    from rpsmf_b200.impute import _uniform_diag
    from rpsmf_b200.psmf import _constant_over_k, _uniform_rho
    assert _uniform_rho(3.0 * np.eye(4), 4, "R") == 3.0
    assert _uniform_diag(10 * np.eye(5), 5, "R") == 10.0
    assert np.array_equal(_uniform_rho(np.diag([1.0, 2.0]), 2, "R"), [1.0, 2.0])        # non-uniform diagonal: the vector
    assert np.array_equal(_uniform_diag(np.diag([3.0, 2.0, 7.0]), 3, "R"), [3.0, 2.0, 7.0])
    with pytest.raises(NotImplementedError):
        _uniform_rho(np.array([[1.0, 0.1], [0.1, 1.0]]), 2, "R")                       # not diagonal
    with pytest.raises(NotImplementedError):
        _uniform_diag(np.array([[1.0, 0.1], [0.1, 1.0]]), 2, "R")
    Q = np.eye(2)
    assert _constant_over_k({0: Q, 1: Q, 2: Q.copy()}, "Q") is not None
    with pytest.raises(NotImplementedError):
        _constant_over_k({0: Q, 1: 2 * Q}, "Q")


def test_hook_override_rejected_without_gpu():
    from rpsmf_b200 import PSMFIter

    class Bad(PSMFIter):
        def _update_coefficient_mean(self, *a):
            pass

    with pytest.raises(NotImplementedError):
        Bad(np.zeros((2, 1)), np.zeros((4, 2)), np.eye(2), np.zeros((2, 1)), np.eye(2), {0: np.eye(2)}, {0: np.eye(4)},
            lambda th, x, t: x)


def test_adam_and_learning_rates():
    from rpsmf_b200 import PSMFIter
    from rpsmf_b200.learning_rate import ConstantLearningRate, ExponentialLearningRate
    assert ConstantLearningRate(0.1).get(5) == 0.1
    assert abs(ExponentialLearningRate(1.0, 0.01, 10).get(10) - 0.01) < 1e-15
    o = PSMFIter(np.array([[0.5], [0.2]]), np.zeros((4, 2)), np.eye(2), np.zeros((2, 1)), np.eye(2), {0: np.eye(2)},
                 {0: np.eye(4)}, lambda th, x, t: x)
    o.adam_init(gam=1e-2)
    o._gradsum = np.array([[1.0], [-2.0]])
    o.adam_update(1)
    # first Adam step moves every coordinate by lr * sign(g) (psmf.py:224-242)
    assert np.allclose(o._theta[1], np.array([[0.49], [0.21]]), atol=1e-9)
    o.optim = "sgd"; o.sgd_init(gam=0.1); o.sgd_update(2)
    assert np.allclose(o._theta[2], np.maximum(o._theta[1] - 0.1 * o._gradsum, 0))


def test_plain_c_caller_compiles_and_links():
    """include/psmf_b200.h is valid C99 and examples/psmf_demo.c links against the library with nothing but a C
    compiler and the CUDA runtime (no torch, no C++ types across the boundary)."""
    import os
    import shutil
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gcc = shutil.which("gcc")
    cuda = "/usr/local/cuda"
    if not gcc or not os.path.exists(os.path.join(cuda, "include", "cuda_runtime_api.h")):
        pytest.skip("needs gcc and the CUDA runtime headers")
    with tempfile.TemporaryDirectory() as tmp:
        probe = os.path.join(tmp, "probe.c")
        with open(probe, "w") as fp:
            fp.write('#include "psmf_b200.h"\nint main(void) { return sizeof(psmf_config) == 80 && sizeof(psmf_io) == 160 ? 0 : 1; }\n')
        subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"), probe,
                        "-o", os.path.join(tmp, "probe")], check=True)
        assert subprocess.run([os.path.join(tmp, "probe")]).returncode == 0
        subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(root, "include"), "-I", os.path.join(cuda, "include"),
                        os.path.join(root, "examples", "psmf_demo.c"), "-o", os.path.join(tmp, "demo"),
                        "-L", os.path.join(root, "rpsmf_b200"), "-lpsmf_b200", "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm"],
                       check=True)


def test_bench_generator_is_N_invariant_and_segment_mask():
    """bench_data.py: every value is a function of (seed, global time, global row), so a row shard generated by any
    rank of any world size equals the same rows of the single-GPU problem -- bench.py relies on it for the parity
    prologue and for the N-independent X checksum.  --mask segments: runs of 20 missing steps per row until the
    requested GLOBAL ratio (common.py:50-76)."""
    import os
    import sys
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench_data as bd
    cpu = torch.device("cpu")
    d, r, T = 96, 4, 130
    Y, M, C0, x0 = bd.make_series(torch, cpu, d, 0, d, r, T, torch.float64, chunk=50)
    assert M.dtype == torch.uint8 and (Y[M == 0] == 0).all()
    miss = 1.0 - M.float().mean().item()
    assert 0.15 < miss < 0.25
    parts = [bd.make_series(torch, cpu, b - a, a, d, r, T, torch.float64, chunk=64) for a, b in ((0, 32), (32, 96))]
    assert torch.equal(torch.cat([p[0] for p in parts], 1), Y) and torch.equal(torch.cat([p[1] for p in parts], 1), M)
    assert torch.equal(torch.cat([p[2] for p in parts], 0), C0) and torch.equal(parts[0][3], x0) and torch.equal(parts[1][3], x0)
    # a later window of the same problem (t0 > 0) continues the same sequence
    Yw, Mw, _, _ = bd.make_series(torch, cpu, d, 0, d, r, 30, torch.float64, t0=100)
    assert torch.equal(Yw, Y[100:]) and torch.equal(Mw, M[100:])
    # NaN encoding carries the same mask and values
    Yn, Mn, _, _ = bd.make_series(torch, cpu, d, 0, d, r, T, torch.float64, nan_encoded=True)
    assert Mn is None and torch.equal(torch.isnan(Yn), M == 0) and torch.equal(torch.nan_to_num(Yn, nan=0.0), Y)
    # noise is heavy-tailed but sane, dictionary ~ N(0, 1), init ~ U[0, 1)
    assert 0.0 <= float(C0.min()) and float(C0.max()) < 1.0 and abs(float(C0.mean()) - 0.5) < 0.1
    # segment mask: global ratio reached, runs of >= 20 steps, starts at t >= 1, and N-invariant through the all-reduce hook
    Ms = bd.segment_mask(torch, cpu, 600, 0, 40, 40, 0.2)
    ratio = 1.0 - Ms.float().mean().item()
    assert 0.2 <= ratio < 0.26 and Ms[0].all()
    for c in (0, 3, 39):
        mm = np.concatenate([[0], (Ms[:, c].numpy() == 0).astype(int), [0]])
        edges = np.flatnonzero(np.diff(mm))
        runs = edges[1::2] - edges[0::2]
        assert runs.size > 0 and runs.min() >= 20
    # two "ranks" in lock step: each sweep sees the global count
    import threading
    halves, box, bar = [None, None], [None, None], threading.Barrier(2)

    def rank(k):
        def allreduce(v):
            box[k] = v.clone()
            bar.wait()
            tot = box[0] + box[1]
            bar.wait()
            return tot
        halves[k] = bd.segment_mask(torch, cpu, 600, 20 * k, 20, 40, 0.2, allreduce=allreduce)
    th = [threading.Thread(target=rank, args=(k,)) for k in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert torch.equal(torch.cat(halves, 1), Ms)
    # batch generator: a series depends on its global index only
    Yb, Mb, Cb, xb = bd.make_batch(torch, cpu, 0, 6, 6, 32, 3, 20, torch.float64, series_chunk=4)
    Y2, M2, C2, x2 = bd.make_batch(torch, cpu, 2, 3, 6, 32, 3, 20, torch.float64)
    assert torch.equal(Y2, Yb[2:5]) and torch.equal(M2, Mb[2:5]) and torch.equal(C2, Cb[2:5]) and torch.equal(x2, xb[2:5])


def test_reference_arm_prints_the_config_record_of_the_cuda_arm():
    """bench.py --impl reference (the CPU arm the driver times next to the CUDA arm) must describe the same workload: same
    metric, unit, higher_is_better and an identical `config` record (the driver compares them), plus its own
    cpu_baseline / e2e objects.  Run here at a tiny size; the record is built from the arguments alone."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    argv = ["--rows", "4096", "--r", "4", "--steps", "1", "--warmup", "0"]
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference"] + argv, capture_output=True, text=True,
                         check=True, cwd=root).stdout
    line = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    old = sys.argv
    try:
        sys.argv = ["bench.py"] + argv
        args = bench.parse()
    finally:
        sys.argv = old
    assert line["impl"] == "reference"
    assert line["config"] == bench.config_record(args, 1)
    assert line["config"]["mask_encoding"] == "nan" and line["config"]["d"] == 4096
    assert line["metric"] == bench.metric_name(args) and line["unit"] == bench.unit_name(args) and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"] > 0


def test_bench_dump_outputs_is_bounded_and_reproducible(tmp_path):
    """bench.py --dump-outputs: an array up to 8 MB is written whole, a larger one as the same seeded sample of its rows on
    every run; the shard of a row-split array lands on its global rows; --steps must be >= 1."""
    import os
    import subprocess
    import sys
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench

    class Args:
        pass
    d, r = 300_000, 16                                                    # 38 MB of float64: sampled
    C = torch.arange(d * r, dtype=torch.float64).reshape(d, r)
    X = torch.randn(500, r, dtype=torch.float64)
    for run in ("a", "b"):
        a = Args()
        a.dump_outputs = str(tmp_path / run)
        ctx = dict(torch=torch, dist=None, world=1, rank=0, args=a)
        bench.dump_outputs(ctx, {"X": (X, 0, None), "C": (C[1000:], 1000, d)})      # this rank holds rows 1000 .. d - 1
    Xa, Ca, Cb = (np.load(str(tmp_path / p)) for p in ("a/X.npy", "a/C.npy", "b/C.npy"))
    assert np.array_equal(Xa, X.numpy()) and np.array_equal(Ca, Cb)
    assert Ca.nbytes <= bench.DUMP_FILE_BYTES and Ca.shape == (bench.DUMP_FILE_BYTES // (r * 8), r)
    idx = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(d, len(Ca), replace=False))
    assert np.array_equal(Ca, np.where((idx >= 1000)[:, None], C.numpy()[idx], 0.0))         # other ranks' rows: zero here
    bad = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=root)
    assert bad.returncode == 2 and "--steps" in bad.stderr
