"""Candidate regions from the scan's rows (``--regions FILE``, ``--threshold C``).

Neighbouring centres share almost all of their window, so one selected locus gives a run of many rows above any
cut.  This module turns the rows of one input into one line per run (DESIGN.md §3.12):

  * a **region** is a maximal run of consecutive non-gap rows whose CLR is >= the cut (NaN never qualifies);
    regions never cross gap rows or the ends of an input;
  * its **peak** is the row with the largest CLR, the first one in row order on ties (the scan's strict '>');
  * the **position support interval** of a peak: each row's CLR is the maximum of T over (A, x, alpha) at that
    centre, so the CLR along the rows is the profile likelihood of the target's position.  From the peak the
    interval extends over consecutive non-gap rows while CLR >= CLR_peak - q, and stops at a gap row, a NaN or
    the end of the input; it may reach past the region when q > CLR_peak - cut.  As in support.py this is a
    support interval of a composite likelihood, not a calibrated confidence interval;
  * with ``--null``, the **region p-value** (1 + #{replicates whose maximum CLR >= CLR_peak}) / (1 + R): the
    probability that a neutral replicate holds a row this high.  It is a family-wise p-value only for a scanned
    sequence of the replicates' length; it is not scaled to the genome.

Pure numpy and O(rows): no Python loop over rows, only the region lines are formatted in Python.
"""
import math

import numpy as np

from . import null as null_mod

REGION_HEADER = ('input\tstart_physPos\tend_physPos\tnRows\tpeak_physPos\tpeak_genPos\tCLR\tx_hat\ts_hat\tA_hat\t'
                 'nSites\tpos_lo\tpos_hi\tp_region\n')

#: rows per block of the position-interval search (``_left_ends``)
_BLOCK = 64


def check_threshold(c):
    """The cut as a float; raises ValueError unless it is finite and > 0 (the CLR is never below 0, so a cut
    <= 0 would make every row a region)."""
    c = float(c)
    if not math.isfinite(c) or c <= 0:
        raise ValueError(f'the region threshold must be a finite number > 0, got {c!r}')
    return c


def row_clr(T, iA):
    """The CLR of every row as the main file prints it: T, and 0 for the all-zero row (``iA < 0``)."""
    return np.where(np.asarray(iA) < 0, 0.0, np.asarray(T, dtype=np.float64))


def call_regions(T, gap, cut):
    """(first, last) row indices of every maximal run of non-gap rows with T >= cut."""
    ok = np.concatenate(([False], (np.asarray(T, dtype=np.float64) >= cut) & ~np.asarray(gap, dtype=bool),
                         [False]))
    edge = np.flatnonzero(ok[1:] != ok[:-1])
    return edge[0::2], edge[1::2] - 1


def peaks(T, first, last):
    """Row index of the largest T of every region [first, last] (every T in a region is a number); the first
    such row on ties."""
    T = np.asarray(T, dtype=np.float64)
    if len(first) == 0:
        return np.zeros(0, np.int64)
    size = last - first + 1
    start = np.cumsum(size) - size                      # of each region in the concatenation of all regions
    rows = np.arange(size.sum()) + np.repeat(first - start, size)
    label = np.repeat(np.arange(len(first)), size)
    v = T[rows]
    hit = np.flatnonzero(v == np.maximum.reduceat(v, start)[label])
    return rows[hit[np.concatenate(([True], label[hit][1:] != label[hit][:-1]))]]


def _left_ends(Te, p, L):
    """For every query (p, L): the smallest i <= p with Te[i:p] >= L everywhere.  Te holds -inf where a row may
    not be crossed.  Rows are grouped in blocks of _BLOCK; a sparse table of block minima finds, in log steps,
    the nearest block to the left that holds a row below L, and only that block and p's own are read row by
    row, so the cost is O(rows + queries * (_BLOCK + log rows)) whatever the intervals' lengths."""
    n, B = len(Te), _BLOCK
    nb = -(-n // B)
    blocks = np.full(nb * B, -np.inf)
    blocks[:n] = Te
    blocks = blocks.reshape(nb, B)
    col = np.arange(B)

    def last_below(b, L, before):
        """Last column of block b below L among the columns < before (-1: none)."""
        below = (blocks[b] < L[:, None]) & (col < before[:, None])
        return np.where(below.any(axis=1), B - 1 - np.argmax(below[:, ::-1], axis=1), -1)

    bp = p // B
    own = last_below(bp, L, p - bp * B)
    table = [blocks.min(axis=1)]                        # table[l][i] = min of blocks [i, i + 2^l)
    while 2 ** len(table) <= nb:
        s, prev = 2 ** (len(table) - 1), table[-1]
        table.append(np.minimum(prev[:-s], prev[s:]))
    cur = bp.copy()                                     # blocks [cur, bp) hold no row below L
    for lvl in range(len(table) - 1, -1, -1):
        cand = cur - 2 ** lvl
        ok = cand >= 0
        ok[ok] = table[lvl][cand[ok]] >= L[ok]
        cur = np.where(ok, cand, cur)
    lo = np.zeros(len(p), np.int64)
    far = (own < 0) & (cur > 0)
    lo[far] = (cur[far] - 1) * B + last_below(cur[far] - 1, L[far], np.full(int(far.sum()), B)) + 1
    lo[own >= 0] = bp[own >= 0] * B + own[own >= 0] + 1
    return lo


def position_interval(T, gap, peak, q):
    """(lo, hi) row indices of the position support interval of every peak: the run of consecutive non-gap rows
    around the peak with T >= T[peak] - q, stopped by a gap row, a NaN or the end of the input."""
    T = np.asarray(T, dtype=np.float64)
    peak = np.asarray(peak, dtype=np.int64)
    if len(peak) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    Te = np.where(np.asarray(gap, dtype=bool) | np.isnan(T), -np.inf, T)
    L = T[peak] - q
    lo = _left_ends(Te, peak, L)
    hi = len(T) - 1 - _left_ends(Te[::-1], len(T) - 1 - peak, L)
    return lo, hi


def cut_of(threshold, maxima):
    """-> (cut, where it came from): ``threshold`` when given, else the quantile of the per-replicate maximum CLRs
    ``maxima`` (``null.replicate_maxima``) that ``null.summary`` prints first (0.95), unrounded."""
    if threshold is not None:
        return threshold, '--threshold'
    if len(maxima) == 0:
        raise ValueError('--regions: no replicate has a maximum CLR, so the null gives no cut')
    q = null_mod.QUANTILES[0]
    return float(np.quantile(maxima, q)), f'{q} quantile of {len(maxima)} replicate maxima'


def region_lines(name, plan, order, rows, gap, cut, q, maxima=None):
    """Lines of the regions file for one input: ``rows`` = (T, iA, ix, ia, nsites) of ``plan``'s rows, ``gap`` its
    gap rows; ``maxima``: the per-replicate maximum CLRs (None: p_region is NA).  Positions, CLR and grid values are
    the main file's text of those rows."""
    T, iA, ix, ia, ns = rows
    clr = row_clr(T, iA)
    first, last = call_regions(clr, gap, cut)
    peak = peaks(clr, first, last)
    lo, hi = position_interval(clr, gap, peak, q)
    # (1 + #{maxima >= CLR_peak}) / (1 + R)
    p = null_mod.pvalues(clr[peak], maxima) if maxima is not None else [None] * len(peak)
    lines = []
    for f, l, k, a, b, pk in zip(first, last, peak, lo, hi, p):
        pos, gen = plan.text(k)
        Tm, xh, ah, Ah, w = order.decode(T[k], iA[k], ix[k], ia[k], ns[k])
        lines.append(f'{name}\t{plan.text(f)[0]}\t{plan.text(l)[0]}\t{l - f + 1}\t{pos}\t{gen}\t{Tm}\t{xh}\t{ah}\t'
                     f'{Ah}\t{w}\t{plan.text(a)[0]}\t{plan.text(b)[0]}\t{"NA" if pk is None else float(pk)}\n')
    return lines


def write_regions(path, per_input, cut, source, q):
    """Write the regions file: a comment line with the cut, where it came from and the drop q, the header, then
    ``per_input``'s lines (one list per input, in input order).  Returns the console line."""
    with open(path, 'w') as fh:
        fh.write(f'# CLR cut {cut!r} ({source}); position support drop q = {q!r}\n')
        fh.write(REGION_HEADER)
        for lines in per_input:
            fh.writelines(lines)
    n = sum(len(lines) for lines in per_input)
    hit = sum(1 for lines in per_input if lines)
    return f'regions: {n} above CLR {cut!r} ({source}) in {hit} of {len(per_input)} inputs, written to {path}'
