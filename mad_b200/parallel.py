"""Multi-GPU plumbing of the two paths that shard (SURVEY.md 8e); one process per GPU,
``torch.distributed`` (NCCL on the GPUs; the same code runs over gloo on CPU tensors in the tests).

* batches of maps / conformational snapshots (``MaD.py:143-162,178-189`` loops): independent units,
  map i -> rank i mod G, no data-path collective; ``gather_varlen`` collects per-map result tables;
* all-pairs matching (``MaD.py:420-424``): the lo (reference) axis is cut into G contiguous shards,
  every rank holds all hi rows and computes its local top-k with GLOBAL lo indices; one
  ``all_gather`` of the [M, k] lists and a k-way merge with the (score desc, index asc) rule give
  a result bit-identical to one GPU.  Threshold mode (the parity contract, ``MaD.py:423-424``): every rank lists its
  pairs with GLOBAL lo indices; pair counts are all-gathered, the lists travel in one padded all-gather and are merged
  in (hi, lo) order -- the row-major order of ``np.where`` on the whole score matrix.
* ``MaD._match_dsc`` (``MaD.py:414-453``): the threshold matching and the anchor clouds are replicated (cheap next to the
  per-pair repeatability); the pairs are cut into G contiguous shares, every rank counts the hits of its share, one
  all_gather of the int32 counts and the row expansion on every rank give the 1-GPU table.
"""
import torch
import torch.distributed as dist


def shard_bounds(n, world):
    """Contiguous near-equal split of range(n): [(start, end)] * world (first n % world shards one longer)."""
    base, extra = divmod(int(n), int(world))
    out, s = [], 0
    for r in range(world):
        e = s + base + (1 if r < extra else 0)
        out.append((s, e))
        s = e
    return out


def assign_units(n_units, rank, world):
    """Round-robin ownership of independent units (maps, snapshots)."""
    return list(range(int(rank), int(n_units), int(world)))


def _world(group):
    return dist.get_world_size(group) if dist.is_initialized() else 1


def gather_topk(idx_local, score_local, group=None):
    """all_gather of per-shard top-k lists: ([M, k] int32, [M, k] float64) -> ([G, M, k], [G, M, k])."""
    g = _world(group)
    if g == 1:
        return idx_local[None], score_local[None]
    idx_g = torch.empty((g,) + tuple(idx_local.shape), dtype=idx_local.dtype, device=idx_local.device)
    sc_g = torch.empty((g,) + tuple(score_local.shape), dtype=score_local.dtype, device=score_local.device)
    try:                                                    # straight into the [G, M, k] buffers the merge kernel reads
        dist.all_gather_into_tensor(idx_g, idx_local.contiguous(), group=group)
        dist.all_gather_into_tensor(sc_g, score_local.contiguous(), group=group)
    except (RuntimeError, NotImplementedError):             # a backend without the tensor form
        dist.all_gather(list(idx_g.unbind(0)), idx_local.contiguous(), group=group)
        dist.all_gather(list(sc_g.unbind(0)), score_local.contiguous(), group=group)
    return idx_g, sc_g


def gather_varlen(t, group=None):
    """all_gather of tensors whose first dimension differs per rank (pair lists, descriptor tables):
    counts first, then one padded all_gather; returns the list of per-rank tensors.  Rows travel as raw bytes, so any
    dtype works (NCCL has no int16)."""
    g = _world(group)
    if g == 1:
        return [t]
    row_shape = tuple(t.shape[1:])
    row_bytes = t.element_size()
    for d in row_shape:
        row_bytes *= int(d)
    n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
    counts = [torch.zeros_like(n) for _ in range(g)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    cap = max(max(counts), 1)
    pad = torch.zeros((cap, row_bytes), dtype=torch.uint8, device=t.device)
    if t.shape[0]:
        pad[: t.shape[0]] = t.contiguous().view(-1).view(torch.uint8).view(t.shape[0], row_bytes)
    bufs = [torch.empty_like(pad) for _ in range(g)]
    dist.all_gather(bufs, pad, group=group)
    return [b[:c].contiguous().view(-1).view(t.dtype).view((c,) + row_shape) for b, c in zip(bufs, counts)]


def match_topk_sharded(hi_set, lo_shard_set, k, lo_index_base, group=None, impl=None):
    """Per hi row the k best rows of the WHOLE lo set, of which this rank holds the shard starting at
    global row ``lo_index_base``.  Every rank returns the same merged ([M, k] idx, [M, k] score)."""
    from . import pipeline as P
    idx, sc = P.match_topk(hi_set, lo_shard_set, k, lo_index_base=lo_index_base, impl=impl)
    idx_g, sc_g = gather_topk(idx, sc, group)
    if idx_g.shape[0] == 1:
        return idx, sc
    return P.topk_merge(idx_g, sc_g)


def merge_pair_lists(parts):
    """[(hi int32 [P_r], lo_global int32 [P_r], score float64 [P_r])] in rank order (= ascending lo shards), each already in
    (hi, lo) order -> one list in (hi, lo) order.  A stable sort by hi keeps, inside a hi row, the rank order and the
    per-rank lo order, which is ascending global lo."""
    hi = torch.cat([p[0] for p in parts])
    lo = torch.cat([p[1] for p in parts])
    sc = torch.cat([p[2] for p in parts])
    if len(parts) == 1 or hi.numel() == 0:
        return hi, lo, sc
    order = torch.sort(hi, stable=True).indices
    return hi[order], lo[order], sc[order]


def gather_pair_lists(pair_hi, pair_lo_global, score, group=None):
    """all-gather-v of per-rank pair lists (counts first, then ONE padded all_gather of the packed rows)."""
    packed = torch.stack([(pair_hi.to(torch.int64) << 32) | pair_lo_global.to(torch.int64), score.contiguous().view(torch.int64)], 1)
    parts = gather_varlen(packed, group)
    return [((q[:, 0] >> 32).to(torch.int32), (q[:, 0] & 0xFFFFFFFF).to(torch.int32), q[:, 1].contiguous().view(torch.float64))
            for q in parts]


def match_threshold_sharded(hi_set, lo_shard_set, cc, lo_index_base, group=None, impl=None, local=None):
    """All pairs (i, j) with cosine(hi_i, lo_j) > cc over the WHOLE lo set, of which this rank holds the shard starting at
    global row ``lo_index_base`` (shards ascending with the rank).  Every rank returns the same (hi, lo_global, score) in
    np.where's row-major order (mad/MaD.py:420-424).  ``local`` = precomputed (hi, lo_local, score) of this shard."""
    if local is None:
        from . import pipeline as P
        local = P.match_threshold(hi_set, lo_shard_set, cc, impl=impl)
    ph, pl, sc = local
    pl = pl + int(lo_index_base)
    if _world(group) == 1:
        return ph, pl, sc
    return merge_pair_lists(gather_pair_lists(ph, pl, sc, group))


def collect_units(local_tables, n_units, group=None, like=None):
    """Result collection of the batch path (map i -> rank i mod G, ``assign_units``): ``local_tables`` = this rank's
    per-unit tensors [rows_u, ...] in its unit order; returns the ``n_units`` tables in unit order on every rank
    (one all-gather of the row counts, one padded all-gather of the concatenated rows).  A rank that owns no unit
    passes ``like`` = any tensor with the tables' dtype, device and row shape."""
    g = _world(group)
    if g == 1:
        return list(local_tables)
    rank = dist.get_rank(group)
    if not local_tables and like is None:
        raise ValueError("collect_units: a rank without units needs `like` to fix dtype and row shape")
    like = local_tables[0] if local_tables else like
    dev = like.device
    per_rank = (int(n_units) + g - 1) // g
    counts = torch.zeros(per_rank, dtype=torch.int64, device=dev)
    for j, t in enumerate(local_tables):
        counts[j] = t.shape[0]
    all_counts = [torch.empty_like(counts) for _ in range(g)]
    dist.all_gather(all_counts, counts, group=group)
    rows = torch.cat(list(local_tables)) if local_tables else like[:0]
    parts = gather_varlen(rows, group)
    out = [None] * int(n_units)
    for r in range(g):
        offs = 0
        for j, u in enumerate(assign_units(n_units, r, g)):
            c = int(all_counts[r][j])
            out[u] = parts[r][offs:offs + c]
            offs += c
    assert all(o is not None for o in out) and len(local_tables) == len(assign_units(n_units, rank, g))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# 2-D rank grid for all-pairs top-k: hi row blocks x lo (reference-axis) shards
# ---------------------------------------------------------------------------------------------------------------------
def _topk_launch_units(pairs, tiles, sms=148, fixed=53):
    """One launch of the uint8 top-8 kernel in tile-equivalents: the library's segment chooser (match_u8.cu:u8_segments):
    min over lo segments s of waves(2 pairs s CTAs) x (tiles / s + fixed per-CTA cost)."""
    best = None
    for s_ in range(1, max(tiles, 1) + 1):
        per = -(-tiles // s_)
        if -(-tiles // per) != s_:
            continue
        c = -(-(2 * pairs * s_) // sms) * (per + fixed)
        best = c if best is None else min(best, c)
    return best


def topk_grid_cost(m, n, gh, gl, sms=148, unit_us=2.5):
    """Model of one rank's matching time on a (gh x gl) grid, mirroring mad_match_topk: CTA pairs own 256 hi rows and sweep
    the rank's lo shard in 256-column tiles; a CTA costs its tiles + 53 tile-equivalents of fixed work (hi-tile load,
    thread-local start-up tiles); the rows of a last wave that is at most half full get a second, segmented launch.
    Checked against measured launches on B200 (DESIGN.md section 6): within 10 %."""
    rows, cols = -(-m // gh), -(-n // gl)
    pairs, tiles, per_wave = -(-rows // 256), -(-cols // 256), sms // 2
    tail = pairs % per_wave
    if pairs > per_wave and 0 < tail <= per_wave // 2:
        units = _topk_launch_units(pairs - tail, tiles, sms) + _topk_launch_units(tail, tiles, sms)
    else:
        units = _topk_launch_units(pairs, tiles, sms)
    return units * unit_us


def pick_topk_grid(m, n, world, min_lo_shards=2):
    """(hi blocks, lo shards) with hi blocks * lo shards == world that minimises the modelled launch time.  The lo
    (reference) axis is what north_star shards; cutting it ALONE leaves every rank with all ceil(m / 256) CTA pairs, each
    paying its fixed start-up for an ever shorter sweep, so for larger worlds part of the factor goes to the hi axis."""
    best = None
    for gl in range(1, world + 1):
        if world % gl or (world > 1 and gl < min(min_lo_shards, world)):
            continue                                          # the reference axis is always cut (both operands shrink per rank)
        gh = world // gl
        c = topk_grid_cost(m, n, gh, gl) + (60.0 if gl > 1 else 0.0)     # (permute + merge launch when the lo axis is cut)
        if best is None or c < best[0] - 1e-9:
            best = (c, gh, gl)
    return best[1], best[2]


def grid_coords(rank, gh, gl):
    """rank -> (hi block, lo shard); ranks of one hi block are consecutive."""
    return rank // gl, rank % gl


def match_topk_grid(hi_block_set, lo_shard_set, k, m_total, grid, group=None, impl=None, local=None):
    """Per hi row of the WHOLE hi set the k best rows of the WHOLE lo set, on a (gh x gl) rank grid: rank r holds hi block
    r // gl (rows ``shard_bounds(m_total, gh)``) and lo shard r % gl.  Every rank computes its block x shard top-k with
    global lo indices; ONE all_gather over the world brings all G lists to every rank; the gl lists of each hi block are
    merged with the (score desc, index asc) rule and the blocks concatenated: ([m_total, k] idx, score), identical on every
    rank and bit-identical to one GPU.  ``local`` = precomputed (idx, score) of this rank's block x shard."""
    gh, gl = grid
    g = _world(group)
    assert gh * gl == g, "grid %r does not match the world size %d" % (grid, g)
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    bh, bl = grid_coords(rank, gh, gl)
    from . import pipeline as P
    if local is None:
        raise ValueError("match_topk_grid: pass local=(idx, score) of this rank's block x shard, or call match_topk_grid_sets")
    idx, sc = local
    rows_max = max(e - s for s, e in shard_bounds(m_total, gh))
    if idx.shape[0] < rows_max:                               # ragged blocks: pad to the longest (padding rows are dropped below)
        pad = rows_max - idx.shape[0]
        idx = torch.cat([idx, torch.full((pad, k), -1, dtype=idx.dtype, device=idx.device)])
        sc = torch.cat([sc, torch.full((pad, k), float("-inf"), dtype=sc.dtype, device=sc.device)])
    idx_g, sc_g = gather_topk(idx, sc, group)                 # [G, rows_max, k], rank-major = [gh][gl]
    if gl > 1:
        idx_g = idx_g.view(gh, gl, rows_max, k).permute(1, 0, 2, 3).contiguous().view(gl, gh * rows_max, k)
        sc_g = sc_g.view(gh, gl, rows_max, k).permute(1, 0, 2, 3).contiguous().view(gl, gh * rows_max, k)
        if idx_g.is_cuda:
            mi, ms = P.topk_merge(idx_g, sc_g)
        else:
            mi, ms = _merge_lists_host(idx_g, sc_g)
            if bool((mi == -2).any()):                        # the lists are on the host already: checking costs nothing
                from ._lib import MadError
                raise MadError("match_topk_grid: a shard's top-k list is incomplete (kernel hand-off time-out)")
    else:
        mi, ms = idx_g.view(gh * rows_max, k), sc_g.view(gh * rows_max, k)
    if m_total % gh:                                          # drop the padding rows of the shorter blocks
        keep = torch.cat([torch.arange(b * rows_max, b * rows_max + (e - s), device=mi.device) for b, (s, e) in enumerate(shard_bounds(m_total, gh))])
        mi, ms = mi[keep], ms[keep]
    return mi, ms


def _merge_lists_host(idx_g, sc_g):
    """(score desc, index asc) k-way merge of [G, M, k] lists on CPU tensors (gloo tests; the GPU path uses mad_topk_merge).
    Index -1 is padding; a row with a -2 (incomplete list) in any input comes out as all -2 / -inf, as mad_topk_merge does."""
    g, m, k = idx_g.shape
    idx = idx_g.permute(1, 0, 2).reshape(m, g * k)
    sc = sc_g.permute(1, 0, 2).reshape(m, g * k)
    big = torch.iinfo(torch.int64).max
    key_i = torch.where(idx < 0, torch.full_like(idx, big, dtype=torch.int64), idx.to(torch.int64))
    order = torch.argsort(key_i, dim=1, stable=True)          # index asc first, then a STABLE sort by score desc
    sc1, idx1 = torch.gather(sc, 1, order), torch.gather(idx, 1, order)
    order2 = torch.argsort(-sc1, dim=1, stable=True)[:, :k]
    mi, ms = torch.gather(idx1, 1, order2), torch.gather(sc1, 1, order2)
    bad = (idx == -2).any(dim=1, keepdim=True)
    return torch.where(bad, torch.full_like(mi, -2), mi), torch.where(bad, torch.full_like(ms, float("-inf")), ms)


def match_topk_grid_sets(hi_block_set, lo_shard_set, k, m_total, lo_index_base, grid, group=None, impl=None):
    """``match_topk_grid`` with the block x shard launch done here (GPU): ``hi_block_set`` / ``lo_shard_set`` are this rank's
    DescriptorSets, ``lo_index_base`` the global row of the lo shard's first row."""
    from . import pipeline as P
    idx, sc = P.match_topk(hi_block_set, lo_shard_set, k, lo_index_base=lo_index_base, impl=impl)
    return match_topk_grid(hi_block_set, lo_shard_set, k, m_total, grid, group=group, impl=impl, local=(idx, sc))


# ---------------------------------------------------------------------------------------------------------------------
# MaD._match_dsc with the per-pair repeatability shared out over the ranks
# ---------------------------------------------------------------------------------------------------------------------
def pad_counts(local, n_pairs, world, bounds=None):
    """This rank's counts padded to the longest share: of ``bounds`` if given, else of ``shard_bounds(n_pairs, world)``
    (the first)."""
    per = max(e - s for s, e in bounds) if bounds is not None else shard_bounds(n_pairs, world)[0][1]
    out = torch.zeros(per, dtype=torch.int32, device=local.device)
    out[:local.numel()] = local
    return out


def join_counts(gathered, n_pairs, bounds=None):
    """[G, per] padded shares in rank order -> the counts of all ``n_pairs`` pairs (shares ``bounds``, by default
    ``shard_bounds(n_pairs, G)``)."""
    g = gathered.shape[0]
    bounds = shard_bounds(n_pairs, g) if bounds is None else bounds
    return torch.cat([gathered[r, :e - s] for r, (s, e) in enumerate(bounds)])


def check_same_problem(rows_hi, rows_lo, n_pairs, device, group=None, n_structures=None):
    """One all_reduce (max of (x, -x)): raises MadError on every rank if the ranks do not hold the same sets and pair
    count -- and, for a batch, the same number of structures -- where a gather of differently sized shares would hang."""
    if n_structures is None:
        names, vals = "(hi rows, lo rows, pairs)", [rows_hi, rows_lo, n_pairs]
    else:
        names, vals = "(structures, lo rows, hi rows, pairs)", [n_structures, rows_lo, rows_hi, n_pairs]
    t = torch.tensor(vals, dtype=torch.int64, device=device)
    both = torch.cat([t, -t])
    dist.all_reduce(both, op=dist.ReduceOp.MAX, group=group)
    k = len(vals)
    hi_, lo_ = both[:k].tolist(), [-v for v in both[k:].tolist()]
    if hi_ != lo_:
        from ._lib import MadError
        what = "match_dsc_sharded" if n_structures is None else "match_dsc_many_sharded"
        raise MadError("%s: the ranks disagree on %s: from %r to %r" % (what, names, lo_, hi_))


def gather_pair_counts(local, n_pairs, rows_hi, rows_lo, group=None, bounds=None, n_structures=None):
    """The counts of all ``n_pairs`` pairs on every rank from each rank's share (``bounds[rank]``; by default
    ``shard_bounds(n_pairs, G)[rank]``): the consistency check, then ONE all_gather of the shares padded to equal size
    (``all_gather_into_tensor``, or the list form on a backend without it).  ``n_structures``: the batch size of a
    ``match_dsc_many_sharded`` call, also checked.  No collective at all for n_pairs == 0, so the check cannot catch one
    rank with no pairs while another has some: the ranks with pairs then wait in the check's all_reduce until the
    backend's time-out."""
    g = _world(group)
    if g == 1 or n_pairs == 0:
        return local
    check_same_problem(rows_hi, rows_lo, n_pairs, local.device, group, n_structures)
    bounds = shard_bounds(n_pairs, g) if bounds is None else bounds
    pad = pad_counts(local, n_pairs, g, bounds)
    out = torch.empty((g, pad.numel()), dtype=torch.int32, device=local.device)
    try:
        dist.all_gather_into_tensor(out, pad, group=group)
    except (RuntimeError, NotImplementedError):             # a backend without the tensor form
        dist.all_gather(list(out.unbind(0)), pad, group=group)
    return join_counts(out, n_pairs, bounds)


def match_dsc_local(m, rank, world):
    """This rank's step of ``match_dsc_sharded`` on a ``pipeline.DscMatch``: the counts of its share of the pairs."""
    s, e = shard_bounds(m.p, world)[rank]
    return m.counts(s, e)


def match_dsc_sharded(lo, hi, anchor_dist_thresh=4, cc_threshold=0.65, group=None, impl=None):
    """``pipeline.match_dsc`` with the per-pair repeatability shared out over the ranks of ``group``.  Every rank holds
    both FeatureTables and computes the same pair list and anchor clouds (threshold matching is replicated, not sharded:
    it is cheap next to the per-pair loop); rank r counts the hits of its contiguous share of the pairs
    (``shard_bounds(P, G)[r]``, equal work per pair), the counts are all-gathered and every rank expands all P rows.
    Every rank returns what ``pipeline.match_dsc`` returns on one GPU, bit for bit."""
    from . import pipeline as P
    m = P.DscMatch(lo, hi, anchor_dist_thresh, cc_threshold, impl)
    if m.p == 0:
        return m.result(m.empty())
    g = _world(group)
    rank = dist.get_rank(group) if g > 1 else 0
    counts = gather_pair_counts(match_dsc_local(m, rank, g), m.p, hi.set.rows, lo.set.rows, group)
    return m.result(m.rows(counts))


def match_dsc_lists_sharded(lo_dsc_list, hi_dsc_list, anchor_dist_thresh=4, cc_threshold=0.65, group=None):
    """Drop-in for ``MaD._match_dsc`` under torchrun (INTEGRATION.md): the arguments and return value of
    ``pipeline.match_dsc_lists``, computed by ``match_dsc_sharded``."""
    from . import pipeline as P
    res, lo_cloud, hi_cloud = match_dsc_sharded(P.FeatureTable.from_features(lo_dsc_list), P.FeatureTable.from_features(hi_dsc_list),
                                                anchor_dist_thresh, cc_threshold, group=group)
    return list(res.cpu().numpy()), lo_cloud, hi_cloud


# ---------------------------------------------------------------------------------------------------------------------
# one map against G structures in one batch, the per-pair repeatability shared out by work
# ---------------------------------------------------------------------------------------------------------------------
def shard_bounds_weighted(pair_off, H, world):
    """Contiguous shares [(start, end)] * world of the pairs of a batch, of about equal work: a pair of structure g (the
    pairs [pair_off[g], pair_off[g+1])) costs H[g], the size of that structure's hi cloud.  Rank r's share starts at the
    first pair p whose preceding work is >= r / world of the total, so every share is within one pair's work of an equal
    split.  Exact integer arithmetic on values every rank holds: every rank computes the same bounds."""
    pair_off = [int(v) for v in pair_off]
    H = [int(h) for h in H]
    world = int(world)
    n_pairs = pair_off[-1]
    before = [0]                                              # work of the pairs before structure g
    for g in range(len(H)):
        before.append(before[-1] + (pair_off[g + 1] - pair_off[g]) * H[g])
    total = before[-1]
    cuts = [0]
    for r in range(1, world):
        t, p = r * total, n_pairs                             # first p with world * work(pairs < p) >= t
        for g in range(len(H)):
            n_g = pair_off[g + 1] - pair_off[g]
            if n_g and before[g + 1] * world >= t:
                need = t - before[g] * world
                k = -(-need // (H[g] * world)) if H[g] > 0 and need > 0 else 0
                p = pair_off[g] + min(k, n_g)
                break
        cuts.append(max(p, cuts[-1]))
    cuts.append(n_pairs)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def match_dsc_many_local(m, rank, world):
    """This rank's step of ``match_dsc_many_sharded`` on a ``pipeline.DscMatchMany``: the counts of its weighted share."""
    s, e = shard_bounds_weighted(m.pair_off, m.hi_n, world)[rank]
    return m.counts(s, e)


def match_dsc_many_sharded(lo, his, anchor_dist_thresh=4, cc_threshold=0.65, group=None, impl=None):
    """``pipeline.match_dsc_many`` with the per-pair repeatability shared out over the ranks of ``group``.  Every rank holds
    the map and all structures and computes the same pairs, clouds and grids; rank r counts the hits of its contiguous
    share ``shard_bounds_weighted(pair_off, H, G)[r]`` (equal work, not equal pair count: a pair of structure g visits
    its H_g hi anchors), the counts are all-gathered and every rank expands all rows.  Every rank returns what
    ``pipeline.match_dsc_many`` returns on one GPU, bit for bit.  Ranks holding different batches raise MadError (the
    check compares structures, lo rows, hi rows and pairs), except that, as for ``match_dsc_sharded``, a batch without
    pairs returns at once without a collective: a rank with no pairs next to ranks with pairs leaves those waiting in
    the check until the backend's time-out."""
    from . import pipeline as P
    m = P.DscMatchMany(lo, his, anchor_dist_thresh, cc_threshold, impl)
    if m.p == 0:
        return m.results(m.empty())
    g = _world(group)
    rank = dist.get_rank(group) if g > 1 else 0
    bounds = shard_bounds_weighted(m.pair_off, m.hi_n, g)
    s, e = bounds[rank]
    counts = gather_pair_counts(m.counts(s, e), m.p, int(m.hi_row_off[-1]), lo.set.rows, group, bounds=bounds,
                                n_structures=m.G)
    return m.results(m.rows(counts))
