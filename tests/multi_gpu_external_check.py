"""Row sharding through the NVLink mailboxes vs the one-process emulation of the caller-driven exchange
(tests/test_gpu_sharded_exchange.py).  Launch:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 \
        tests/multi_gpu_external_check.py --same-device

Every rank filters its row shard with the direct-load kernel and the statistics exchanged inside the kernel.  Rank 0 then
builds one external-exchange engine per shard in its own process, sums their statistics buffers in rank order and finishes
each step on each engine.  Both sum the same per-rank totals in the same order, so the NVLink X, scalar record and
replicated state must equal the emulation's in value, and so must each shard's C.  This ties the single-process matrix of
test_gpu_sharded_exchange.py to the real transport.

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
from rpsmf_b200 import FilterEngine, shard_rows  # noqa: E402


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
    d, T = 1888, 8
    for r in (3, 16):
        Y, M, C0, x0 = make_problem(d, r, T, seed=d + r)
        Y = Y * M
        init = impute_init(r)
        b, e = shard_rows(d, world, rank)
        eng = FilterEngine(e - b, r, device=lr, robust=True, kernel=1, d_global=d, world_size=world, rank=rank)
        eng.connect(dist)
        eng.set_state(C_=C0[b:e], V=init["V"], P=init["P"], x=x0, Q=init["Q"], rho=[init["rho"]], lam=[init["lam"]])
        Yd = torch.as_tensor(np.ascontiguousarray(Y[:, b:e])).cuda(lr)
        Md = torch.as_tensor(np.ascontiguousarray(M[:, b:e])).cuda(lr)
        out = eng.run(Yd, Md, k0=1, want_X=True, want_scal=True)
        bad = eng.status()
        st = {k: (v.cpu().numpy() if v is not None else None) for k, v in eng.get_state().items()}
        mine = dict(X=out["X"].cpu().numpy(), scal=out["scal"].cpu().numpy(), state=st, kernel=eng.launch_info()["kernel"], bad=bad)
        eng.close()
        dist.barrier()
        got = [None] * world
        dist.all_gather_object(got, mine)
        verdict = [None]
        if rank == 0:
            from test_gpu_sharded_exchange import _close, _sharded_run
            emu = _sharded_run([shard_rows(d, world, i) for i in range(world)], r, Y, M, C0, x0, init)
            good = all(g["bad"] == -1 and g["kernel"] == "direct" for g in got) and (emu["status"] == -1).all()
            for i, g in enumerate(got):
                good = good and np.array_equal(g["X"], emu["X"][i]) and np.array_equal(g["scal"], emu["scal"][i])
                for k in ("C", "x", "P", "V", "Q", "rho", "lam"):
                    good = good and np.array_equal(g["state"][k], emu["state"][i][k])
            _close(emu)
            verdict = [bool(good)]
        dist.broadcast_object_list(verdict, src=0)
        ok = ok and verdict[0]
        print("rank %d d=%d r=%d rows[%d:%d) kernel=%s nvlink == emulation: %s %s"
              % (rank, d, r, b, e, mine["kernel"], verdict[0], "OK" if verdict[0] else "FAIL"), flush=True)
        dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
