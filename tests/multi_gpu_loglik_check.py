"""Row-sharded per-step log-likelihood record (PSMF_LOGLIK) vs the same series filtered on one GPU.  Launch:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29523 \
        tests/multi_gpu_loglik_check.py --same-device

Every rank filters its row shard with the statistics exchanged inside the kernel; the small state is replicated, so every
rank writes the same record.  Checks: the 10-wide records bit-identical on all ranks, and nll_k and log p_k within 1e-9 of
the one-GPU engine on all rows, for the direct-load and the TMA-staged kernel.

    --same-device   all ranks share cuda:0 (process group on gloo), as in tests/multi_gpu_check.py
"""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from synth import impute_init, make_problem  # noqa: E402
from rpsmf_b200 import FilterEngine, _capi, shard_rows  # noqa: E402


def rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def ll_run(eng, Y, M, x0, C0, init, dev, T):
    eng.set_state(C_=C0, V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
    Yd = torch.as_tensor(np.ascontiguousarray(Y)).cuda(dev)
    Md = torch.as_tensor(np.ascontiguousarray(M)).cuda(dev)
    sc = []
    for a, b in ((0, T // 2), (T // 2, T)):
        sc.append(eng.run(Yd[a:b], Md[a:b], k0=1 + a, want_X=False, want_loglik=True)["scal"].cpu().numpy())
    assert eng.status() == -1
    return np.concatenate(sc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--same-device", action="store_true")
    args = ap.parse_args()
    rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ["LOCAL_RANK"])
    if args.same_device:
        lr = 0
        torch.cuda.set_device(0)
        dist.init_process_group("gloo")
    else:
        torch.cuda.set_device(lr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    ok = True
    for (d, r, T, kernel) in [(1888, 9, 8, 1), (3840, 16, 8, 2)]:
        Y, M, C0, x0 = make_problem(d, r, T, seed=d + r)
        Y = Y * M
        init = impute_init(r)
        b, e = shard_rows(d, world, rank)
        kw = dict(robust=True, ll_student=True, kernel=kernel, loglik=True)
        eng = FilterEngine(e - b, r, device=lr, d_global=d, world_size=world, rank=rank, **kw)
        eng.connect(dist)
        sc = ll_run(eng, Y[:, b:e], M[:, b:e], x0, C0[b:e], init, lr, T)
        kname = eng.launch_info()["kernel"]
        eng.close()
        dist.barrier()
        vec = torch.from_numpy(sc.ravel().copy())
        gathered = [torch.empty_like(vec) for _ in range(world)]
        dist.all_gather(gathered, vec)
        same = all(torch.equal(gathered[0], g) for g in gathered)
        one = FilterEngine(d, r, device=lr, **kw)
        ref = ll_run(one, Y, M, x0, C0, init, lr, T)
        one.close()
        errs = dict(nll=rel(sc[:, _capi.SCAL_NLL], ref[:, _capi.SCAL_NLL]), logpred=rel(sc[:, _capi.SCAL_LOGPRED], ref[:, _capi.SCAL_LOGPRED]))
        good = same and kname == {1: "direct", 2: "tma"}[kernel] and max(errs.values()) < 1e-9
        ok = ok and good
        print("rank %d d=%d r=%d kernel=%s rows[%d:%d) ranks_identical=%s errs=%s %s"
              % (rank, d, r, kname, b, e, same, {k: "%.1e" % v for k, v in errs.items()}, "OK" if good else "FAIL"), flush=True)
        dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
