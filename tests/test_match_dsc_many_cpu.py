"""The host side of parallel.match_dsc_many_sharded, without a GPU: the work-weighted shares of a batch's pairs
(shard_bounds_weighted), and the gather of the counts over explicit share bounds at world size 2 over gloo."""
import datetime
import os
import socket
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check_bounds(par, pair_off, H, world):
    b = par.shard_bounds_weighted(pair_off, H, world)
    n_pairs = int(pair_off[-1])
    assert len(b) == world and b[0][0] == 0 and b[-1][1] == n_pairs
    assert all(s <= e for s, e in b) and all(b[r][1] == b[r + 1][0] for r in range(world - 1))
    w = np.repeat(np.asarray(H, dtype=np.int64), np.diff(np.asarray(pair_off, dtype=np.int64)))
    assert len(w) == n_pairs
    total = int(w.sum())
    top = int(w.max()) if n_pairs else 0
    for s, e in b:                                           # every share within one pair's work of an equal split
        assert abs(int(w[s:e].sum()) * world - total) < max(top, 1) * world
    assert par.shard_bounds_weighted(pair_off, H, world) == b
    return b


def test_shard_bounds_weighted():
    from mad_b200 import parallel as par
    rng = np.random.default_rng(7)
    for _ in range(200):
        G = int(rng.integers(1, 9))
        n = rng.integers(0, 40, size=G) * (rng.random(G) < 0.7)
        H = np.where(n > 0, rng.integers(1, 5000, size=G), 0)
        pair_off = np.concatenate([[0], np.cumsum(n)])
        for world in (1, 2, 3, 8, int(pair_off[-1]) + 3):
            _check_bounds(par, pair_off, H, world)
    # equal H: the plain equal split up to rounding; a heavy structure gets a short share
    assert _check_bounds(par, [0, 10], [7], 2) == [(0, 5), (5, 10)]
    assert _check_bounds(par, [0, 2, 12], [1000, 10], 2) == [(0, 2), (2, 12)]
    assert _check_bounds(par, [0, 0, 3, 3], [0, 5, 0], 8)[-1] == (3, 3)              # zero-pair structures, world > P
    assert par.shard_bounds_weighted([0, 0], [0], 3) == [(0, 0)] * 3


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
        for pair_off, H in (([0, 1], [3]), ([0, 3, 3, 10], [5, 0, 2]), ([0, 2, 1000], [4000, 3]), ([0, 600, 1000], [1, 1])):
            n_pairs = pair_off[-1]
            bounds = par.shard_bounds_weighted(pair_off, H, world)
            s, e = bounds[rank]
            local = torch.arange(s, e, dtype=torch.int32) * 3 + 1                  # count of pair p: 3 p + 1
            got = par.gather_pair_counts(local, n_pairs, 50, 60, bounds=bounds, n_structures=len(H))
            res["gather_%d" % n_pairs] = bool(got.dtype == torch.int32 and
                                              torch.equal(got, torch.arange(n_pairs, dtype=torch.int32) * 3 + 1))
        bounds = par.shard_bounds_weighted([0, 3, 7], [2, 2], world)
        s, e = bounds[rank]
        try:
            par.gather_pair_counts(torch.zeros(e - s, dtype=torch.int32), 7, 50, 60, bounds=bounds, n_structures=2 + rank)
            res["mismatch_structures"] = False
        except MadError as err:
            res["mismatch_structures"] = "structures" in str(err)
        dist.barrier()
        q.put((rank, res))
    finally:
        dist.destroy_process_group()


def test_world_size_2_gloo_gather_with_explicit_bounds():
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
