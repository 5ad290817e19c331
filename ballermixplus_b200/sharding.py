"""Multi-GPU scan -- SURVEY.md §8 row e.

Centres are independent (/root/reference/BalLeRMix+_v1.py:606 calls ``calcBaller`` once per
centre and nothing is shared between calls), so a scan shards by contiguous centre ranges:
one process per GPU, every rank holds the (read-only) site arrays and tables of the
sequences it touches, scans its range, and ONE collective gathers the per-centre rows on
rank 0.  Ranges are balanced by cost (sites within alpha-reach, summed over A), not by
count, because centres near sequence ends and in sparse regions are cheaper.
"""
import numpy as np


def centre_costs(genpos, t, lo, hi, A, seg_start=None):
    """Sites a centre touches, summed over the A grid (the kernel's work per centre / n_xa).

    ``seg_start``: first site of each segment of a segmented problem (blmx_load_segmented), inside which
    genpos is non-decreasing.  A window inside one segment is then cut at alpha reach within that segment, as
    the kernel cuts it; a window across a boundary is charged whole."""
    genpos = np.asarray(genpos)
    t = np.asarray(t, dtype=np.float64)
    if seg_start is not None and len(seg_start) > 1:
        return _segmented_costs(genpos, t, lo, hi, A, np.asarray(seg_start, dtype=np.int64))
    cost = np.zeros(len(t), dtype=np.float64)
    sorted_ok = len(genpos) < 2 or bool(np.all(np.diff(genpos) >= 0))
    for a in np.asarray(A, dtype=np.float64):
        if sorted_ok and a > 0:
            r = 18.420680743952367 / a
            l = np.maximum(np.searchsorted(genpos, t - r, 'left'), lo)
            h = np.minimum(np.searchsorted(genpos, t + r, 'right') - 1, hi)
        else:
            l, h = np.asarray(lo), np.asarray(hi)
        cost += np.maximum(h - l + 1, 0)
    return cost + 1.0          # never zero: every centre costs a launch slot


def _segmented_costs(genpos, t, lo, hi, A, seg_start):
    n = len(genpos)
    ends = np.append(seg_start[1:], n)
    # the library treats the whole problem as unsorted when any segment is (blmx_load_segmented)
    d = np.diff(genpos) >= 0
    d[seg_start[1:] - 1] = True
    sorted_ok = bool(np.all(d)) and not np.any(np.isnan(genpos[seg_start]))
    L = np.maximum(np.asarray(lo, dtype=np.int64), 0)
    H = np.minimum(np.asarray(hi, dtype=np.int64), n - 1)
    seg = np.clip(np.searchsorted(seg_start, L, 'right') - 1, 0, len(seg_start) - 1)
    inside = sorted_ok & (L <= H) & (H < ends[seg])
    idx = np.flatnonzero(inside)
    idx = idx[np.argsort(seg[idx], kind='stable')]          # the centres of each segment, together
    segs, first = np.unique(seg[idx], return_index=True)
    groups = [(s, idx[b:e]) for s, b, e in zip(segs, first, np.append(first[1:], len(idx)))]
    cost = np.zeros(len(t), dtype=np.float64)
    for a in np.asarray(A, dtype=np.float64):
        l, h = L.copy(), H.copy()
        if a > 0:
            r = 18.420680743952367 / a
            for s, m in groups:
                b, e = seg_start[s], ends[s]
                l[m] = np.maximum(np.searchsorted(genpos[b:e], t[m] - r, 'left') + b, L[m])
                h[m] = np.minimum(np.searchsorted(genpos[b:e], t[m] + r, 'right') - 1 + b, H[m])
        cost += np.maximum(h - l + 1, 0)
    return cost + 1.0


def partition(costs, world):
    """Split range(len(costs)) into `world` contiguous slices of near-equal total cost.

    Returns a list of (begin, end) pairs covering [0, n) in order.
    """
    n = len(costs)
    if world < 1:
        raise ValueError('world must be >= 1')
    cum = np.concatenate(([0.], np.cumsum(np.asarray(costs, dtype=np.float64))))
    total = cum[-1]
    cuts = [0]
    for r in range(1, world):
        k = int(np.searchsorted(cum, total * r / world, 'left'))
        cuts.append(min(max(k, cuts[-1]), n))
    cuts.append(n)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def pack_rows(T, iA, ix, ia, ns, torch):
    """Results of one rank as a single int32 [n, 6] tensor (the 8 bytes of T, then 4 ints)."""
    out = torch.empty((T.shape[0], 6), dtype=torch.int32, device=T.device)
    out[:, 0:2] = T.contiguous().view(torch.int32).view(-1, 2)
    out[:, 2] = iA
    out[:, 3] = ix
    out[:, 4] = ia
    out[:, 5] = ns
    return out


def unpack_rows(rows, torch):
    T = rows[:, 0:2].contiguous().view(torch.float64).view(-1)
    return T, rows[:, 2], rows[:, 3], rows[:, 4], rows[:, 5]


def pack_split_rows(rows, torch):
    """The 15 results of a ``--balPos`` scan (the rows, then the bal and the pos rows, five each) as one int32
    [n, 18] tensor: the rows' six columns of ``pack_rows`` first, then six per half."""
    return torch.cat([pack_rows(*rows[5 * k:5 * k + 5], torch) for k in range(3)], dim=1)


def unpack_split_rows(rows, torch):
    return tuple(v for k in range(3) for v in unpack_rows(rows[:, 6 * k:6 * k + 6], torch))


def gather_rows(rows, counts, rank, world, dist, torch, dst=0):
    """The path's only collective: gather every rank's rows on `dst`, in rank order.

    `counts[r]` is rank r's row count (known to all ranks from the partition), ranks pad
    to the maximum so that one fixed-size gather moves everything.
    """
    if world == 1:
        return rows
    width = int(max(counts))
    padded = torch.zeros((width, rows.shape[1]), dtype=rows.dtype, device=rows.device)
    padded[:rows.shape[0]] = rows
    if rank == dst:
        bufs = [torch.empty_like(padded) for _ in range(world)]
        dist.gather(padded, gather_list=bufs, dst=dst)
        return torch.cat([bufs[r][:counts[r]] for r in range(world)], dim=0)
    dist.gather(padded, gather_list=None, dst=dst)
    return None


def genome_costs(seqs):
    """``centre_costs`` of several sequences, concatenated in sequence order.  ``seqs``: one
    (genpos, A, t, lo, hi, seg_start) per sequence -> (costs, offs), offs[i] = first centre of sequence i
    in the concatenated centre list (offs[-1] = all centres)."""
    costs = [centre_costs(g, t, lo, hi, A, seg) for g, A, t, lo, hi, seg in seqs]
    offs = np.concatenate(([0], np.cumsum([len(c) for c in costs]))).astype(np.int64)
    return (np.concatenate(costs) if costs else np.zeros(0)), offs


def pieces(offs, b, e):
    """The sequences a range [b, e) of the concatenated centre list touches -> [(sequence, lb, le)] with
    [lb, le) a non-empty range of that sequence's own centres, in order.  An empty range touches none."""
    out = []
    for i in range(len(offs) - 1):
        lb, le = max(b, offs[i]), min(e, offs[i + 1])
        if lb < le:
            out.append((i, int(lb - offs[i]), int(le - offs[i])))
    return out


def scan_sharded_seqs(seqs, rank, world, scan_fn, dist, torch, device=None, split=False):
    """Scan the centres of several sequences (one per chromosome: a genome) on `world` ranks and gather the
    rows on rank 0.

    The genome is sharded, not each sequence: the centres of all sequences, laid end to end, are cut into
    `world` cost-balanced contiguous ranges, so a rank's range may hold the end of one sequence and the
    start of the next, and a small sequence may lie within one rank's range.  ``seqs`` holds one
    (genpos, A, t, lo, hi, seg_start) per sequence.  `scan_fn(i, t, lo, hi)` scans a contiguous slice of
    sequence i's centre list on this rank's device and returns torch tensors (T float64, iA, ix, ia,
    nsites int32) living on that device; it is called once per sequence the rank's range touches, in order,
    and never for the others, so a rank needs only those sequences on its device.  A rank whose range is
    empty sends an empty block made on ``device``.  Returns the five gathered tensors on rank 0 (the
    concatenated centre list, in order) and None elsewhere.  ``split`` (``--balPos``): `scan_fn` returns the 15
    tensors of a split scan, packed wider for the same one gather (``pack_split_rows``), and 15 come back.
    """
    costs, offs = genome_costs(seqs)
    parts = partition(costs, world)
    counts = [e - b for b, e in parts]
    blocks = []
    pack, unpack = (pack_split_rows, unpack_split_rows) if split else (lambda r, tc: pack_rows(*r, tc), unpack_rows)
    for i, lb, le in pieces(offs, *parts[rank]):
        t, lo, hi = (np.asarray(a)[lb:le] for a in seqs[i][2:5])
        blocks.append(pack(scan_fn(i, t, lo, hi), torch))
    if not blocks:
        rows = torch.zeros((0, 18 if split else 6), dtype=torch.int32, device=device)
    else:
        rows = blocks[0] if len(blocks) == 1 else torch.cat(blocks, dim=0)
    got = gather_rows(rows, counts, rank, world, dist, torch)
    return unpack(got, torch) if got is not None else None


def scan_sharded(genpos, A, t, lo, hi, rank, world, scan_fn, dist, torch, seg_start=None, device=None):
    """Scan one sequence's centres on `world` ranks and gather the rows on rank 0: ``scan_sharded_seqs``
    with one sequence.

    `scan_fn(t, lo, hi)` scans a contiguous slice of the centre list on this rank's device and
    returns torch tensors (T float64, iA, ix, ia, nsites int32) living on that device (the
    product passes ``DeviceScan.run_device``, i.e. ``blmx_scan_device`` on torch's current stream, so the
    rows never leave the GPU before the gather; CPU tests pass the oracle).
    Returns the five gathered tensors on rank 0 (in centre order) and None elsewhere.
    ``seg_start``: the segment starts of a segmented problem, for the costs.  ``device``: where a rank with
    no centres makes its empty block.
    """
    return scan_sharded_seqs([(genpos, A, t, lo, hi, seg_start)], rank, world,
                             lambda i, ts, los, his: scan_fn(ts, los, his), dist, torch, device=device)
