"""The collectives of parallel.match_dsc_sharded on CPU: world size 2 over gloo (127.0.0.1), on synthetic per-rank counts
(the counting itself needs the GPU: tests/test_match_dsc_sharded.py).  Covers the padding of unequal shares, the
gather, the guard that turns ranks holding different problems into an error on every rank, and P == 0, which must
return at once without any collective."""
import datetime
import os
import socket
import sys

import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    sys.path[:0] = [REPO]
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=60))
    try:
        from mad_b200 import parallel as par
        from mad_b200._lib import MadError
        res = {}
        for n_pairs in (1, 2, 7, 1000):
            s, e = par.shard_bounds(n_pairs, world)[rank]
            local = (torch.arange(s, e, dtype=torch.int32) * 3 + 1)          # count of pair p: 3 p + 1
            got = par.gather_pair_counts(local, n_pairs, 50, 60)
            res["gather_%d" % n_pairs] = bool(got.dtype == torch.int32 and torch.equal(got, torch.arange(n_pairs, dtype=torch.int32) * 3 + 1))
        empty = torch.empty(0, dtype=torch.int32)
        res["p0"] = par.gather_pair_counts(empty, 0, 50, 60).numel() == 0
        if rank == 0:                                                   # alone: a collective here would time out
            res["p0_alone"] = par.gather_pair_counts(empty, 0, 50 + rank, 60).numel() == 0
        else:
            res["p0_alone"] = True
        for what, args in (("rows", (7, 50 + rank, 60)), ("pairs", (7 + rank, 50, 60))):
            s, e = par.shard_bounds(args[0], world)[rank]
            try:
                par.gather_pair_counts(torch.zeros(e - s, dtype=torch.int32), *args)
                res["mismatch_" + what] = False
            except MadError:
                res["mismatch_" + what] = True
        dist.barrier()                                                  # both ranks are still in step after the errors
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_world_size_2_gloo_pair_count_gather():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=180) for _ in range(world)), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [r[0] for r in res] == [0, 1]
    for rank, r in res:
        bad = [k for k, v in r.items() if not v]
        assert not bad, "rank %d: %s" % (rank, bad)
