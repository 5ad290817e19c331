"""Empirical null of the CLR from scans of neutral replicates (``--null LIST``, ``--pvalues FILE``).

The scan's likelihood is a composite likelihood (linked sites are multiplied as if independent), so chi-square
quantiles do not calibrate its CLR (DESIGN.md §3.7).  The usual remedy is an empirical null: scan sequences
simulated under a neutral demographic model with exactly the flags and spectrum of the real run, and compare
each real CLR with the pooled null CLRs.  This module does that bookkeeping (DESIGN.md §3.9):

  * every replicate is read with ``InputData`` under the run's flags and keeps the ``minCount`` it derives
    (it enters the selection tables' normalisation, v1:399-433);
  * classes are keyed (k, n, minCount), and (k, n, minCount, bin) in a binned run (bins.py: a replicate's sites
    are binned by the map lines that name its file name); G and P come from the run's spectrum, the selection rows from one
    ``NormalizedBetaBinom`` per distinct minCount, so every row has the bits a standalone run would build;
  * every replicate is planned with the run's window flags, gap rows are dropped and the windows are offset to
    the replicate's segment of one segmented problem (blmx_load_segmented), scanned in one call;
  * p = (1 + #{null >= T}) / (1 + N_null).

The null is the multiset of CLR values that standalone runs on the replicates would write (gap rows excluded),
within the scan's parity bar (class order and block alignment differ from a standalone run).  The p-values are
only as good as the neutral model the replicates were simulated under, and they are not corrected for multiple
testing.
"""
import contextlib
import io
import os
import sys

import numpy as np

from . import windows
from .inputs import InputData
from .bins import BinnedNeutral, binned_classes
from .native import ScanProblem
from .neutral import site_classes
from .problem import GridOrder
from .selection import NormalizedBetaBinom

PVALUE_HEADER = 'physPos\tgenPos\tCLR\tp_value\n'
QUANTILES = (0.95, 0.99, 0.999)


def read_list(path, flag='--null', item='replicate'):
    """Replicate input files named by the list `path`, one per line; relative paths are taken from the list's
    directory, blank lines and lines starting with '#' are skipped.  A missing or empty list, or a missing
    replicate, raises before anything is read.  `flag` and `item` name the option and what it lists in the
    messages (``--inputList`` reads its inputs with the same rules)."""
    if not os.path.isfile(path):
        raise FileNotFoundError(f'{flag}: {item} list {path} not found')
    base = os.path.dirname(os.path.abspath(path))
    out = []
    with open(path) as fh:
        for line in fh:
            name = line.strip()
            if not name or name.startswith('#'):
                continue
            full = name if os.path.isabs(name) else os.path.join(base, name)
            if not os.path.isfile(full):
                raise FileNotFoundError(f'{flag}: {item} {full} (listed in {path}) not found')
            out.append(full)
    if not out:
        raise ValueError(f'{flag}: {item} list {path} names no {item}')
    return out


def flags_of(data, sel):
    """(nofreq, MAF, nosub, minCount) of the run that built `data` and `sel`: the statistic of the selection
    tables, and the command line's --minCount (which InputData keeps as given only with --noFreq)."""
    stat = getattr(sel, 'stat', None)
    if stat is None:
        raise ValueError('--null needs the selection tables of this package (NormalizedBetaBinom.stat)')
    return stat == 'B1', stat in ('B2maf', 'B0maf'), stat in ('B0', 'B0maf'), data.minCount


def _held(fn, name, quiet=True):
    """fn(), with its console output held back (quiet); if it exits the way the reference does on bad input,
    the output is shown with the replicate's name."""
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf) if quiet else contextlib.nullcontext():
            return fn()
    except SystemExit:
        sys.stdout.write(buf.getvalue())
        print(f'(neutral replicate {name})')
        raise


def read_replicates(paths, nofreq, MAF, nosub, minCount, phys, Rrate):
    reps = []
    for p in paths:
        try:
            d = _held(lambda: InputData(p, nofreq, MAF, nosub, minCount, phys=phys, Rrate=Rrate), p)
        except ValueError as exc:
            raise ValueError(f'neutral replicate {p}: {exc}') from None
        if d.numSites == 0:
            raise ValueError(f'neutral replicate {p} has no sites')
        reps.append(d)
    return reps


def null_problem(reps, names, neutral, grids, nofreq, MAF, nosub):
    """One segmented problem of all replicates -> (ScanProblem with seg_start, GridOrder)."""
    order = GridOrder(grids)
    if isinstance(neutral, BinnedNeutral):          # a replicate's sites are binned by the map lines of its name
        per = [binned_classes(d.count, d.total, neutral.site_bins(os.path.basename(name), d.position))
               for d, name in zip(reps, names)]
    else:
        per = [site_classes(d.count, d.total) for d in reps]
        per = [(ck, cn, np.zeros(len(ck), np.int64), c) for ck, cn, c in per]
    for (ck, cn, cb, _), name in zip(per, names):
        _held(lambda: neutral.class_tables(ck, cn, cb) if cb.any() else neutral.class_tables(ck, cn), name,
              quiet=False)                                                  # the run's message + exit
    mins = [int(d.minCount) for d in reps]
    # classes keyed (minCount, bin, n, k)
    keys = np.concatenate([np.column_stack((np.full(len(ck), m, np.int64), cb, cn, ck))
                           for (ck, cn, cb, _), m in zip(per, mins)])
    uniq, inv = np.unique(keys, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    cm, cb_all, cn_all, ck_all = uniq[:, 0], uniq[:, 1], uniq[:, 2], uniq[:, 3]
    G, P = neutral.class_tables(ck_all, cn_all, cb_all) if cb_all.any() else neutral.class_tables(ck_all, cn_all)
    # selection rows: one table per distinct minCount, over that minCount's classes
    own = {m: d.minCount for d, m in zip(reps, mins)}              # a replicate's own minCount object
    rows = {(x, a): np.empty(len(uniq)) for x in order.x for a in order.a}
    for m in np.unique(cm):
        idx = np.flatnonzero(cm == m)
        sub = InputData.from_arrays(np.zeros(len(idx), np.int64), np.zeros(len(idx)), ck_all[idx], cn_all[idx],
                                    minCount=own[int(m)], Rrate=reps[0].Rrate)
        sel = NormalizedBetaBinom(sub, grids, nofreq, MAF, nosub)
        for key, row in rows.items():
            row[idx] = sel.get(*key)
    SP = np.empty((len(order.x) * len(order.a), len(uniq)), dtype=np.float64)
    r = 0
    for x in order.x:
        for a in order.a:
            SP[r] = rows[(x, a)] * P
            r += 1
    sizes = np.array([d.numSites for d in reps], dtype=np.int64)
    seg_start = np.concatenate(([0], np.cumsum(sizes)[:-1])).astype(np.int64)
    offs = np.concatenate(([0], np.cumsum([len(ck) for ck, _, _, _ in per])))
    cls = np.concatenate([inv[offs[i] + c] for i, (_, _, _, c) in enumerate(per)]).astype(np.int32)
    genpos = np.concatenate([d.genPos for d in reps])
    prob = ScanProblem(genpos, cls, G, SP, np.array([float(v) for v in order.A]), len(order.x), len(order.a),
                       seg_start=seg_start)
    return prob, order


def null_plan(reps, names, seg_start, fixSize=False, r=0, s=1, phys=False, noCenter=False):
    """Centres of every replicate under the run's window flags, gap rows dropped, windows offset to the
    replicate's segment -> (t, lo, hi, replicate index) of the null rows."""
    out = [[], [], [], []]
    for i, (d, name, b) in enumerate(zip(reps, names, seg_start)):
        plan = _held(lambda: windows.make_plan(d, fixSize=fixSize, r=r, s=s, phys=phys, noCenter=noCenter), name)
        t, lo, hi, gap = plan.arrays()
        keep = ~gap
        for col, v in zip(out, (t[keep], lo[keep] + b, hi[keep] + b, np.full(int(keep.sum()), i, np.int64))):
            col.append(v)
    return tuple(np.concatenate(c) if c else np.zeros(0) for c in out)


class NullSetup:
    """Everything the null scan needs, prepared before any scan: replicates, their segmented problem and the
    centres of the null rows."""

    def __init__(self, list_path, data, neutral, sel, grids, fixSize=False, r=0, s=1, phys=False, noCenter=False):
        self.paths = read_list(list_path)
        nofreq, MAF, nosub, minCount = flags_of(data, sel)
        reps = read_replicates(self.paths, nofreq, MAF, nosub, minCount, phys, data.Rrate)
        self.problem, self.order = null_problem(reps, self.paths, neutral, grids, nofreq, MAF, nosub)
        self.t, self.lo, self.hi, self.rep = null_plan(reps, self.paths, self.problem.seg_start, fixSize=fixSize,
                                                       r=r, s=s, phys=phys, noCenter=noCenter)
        if len(self.t) == 0:
            raise ValueError('--null: the replicates give no null rows (every row is a gap row)')

    @property
    def n_replicates(self):
        return len(self.paths)


def pvalues(T, null):
    """p = (1 + #{null >= T}) / (1 + N_null) per entry of T, from one sort and a binary search (ties count as
    >=).  NaN in T gives NaN (written NA); NaN null values cannot be compared and are left out of N_null."""
    null = np.asarray(null, dtype=np.float64)
    null = np.sort(null[~np.isnan(null)])
    if len(null) == 0:
        raise ValueError('the empirical null is empty: no replicate row has a CLR')
    T = np.asarray(T, dtype=np.float64)
    ge = len(null) - np.searchsorted(null, T, 'left')
    p = (1.0 + ge) / (1.0 + len(null))
    p[np.isnan(T)] = np.nan
    return p


def format_pvalues(plan, order, T, iA, ix, ia, ns, p):
    """Lines of the p-value file: the main file's physPos, genPos and CLR text, then p (NA for gap rows and
    NaN CLRs)."""
    lines = [PVALUE_HEADER]
    f0, f1 = plan.f0, plan.f1
    for j in range(len(plan)):
        if plan.gap[j]:
            a, b, c = f0[j].split('\t')[:3]
            lines.append(f'{a}\t{b}\t{c}\tNA\n')
            continue
        Tm = order.decode(T[j], iA[j], ix[j], ia[j], ns[j])[0]
        pj = float(p[j])
        lines.append(f'{f0[j]}\t{f1[j]}\t{Tm}\t{"NA" if pj != pj else pj}\n')
    return lines


def replicate_maxima(null, rep, n_replicates):
    """The maximum CLR of every replicate that has one: ``null`` the null CLRs, ``rep`` their replicates.  NaN
    values are left out; a replicate without a row (or with NaN rows only) has no maximum and is dropped."""
    null = np.asarray(null, dtype=np.float64)
    ok = ~np.isnan(null)
    mx = np.full(n_replicates, -np.inf)
    np.maximum.at(mx, np.asarray(rep)[ok], null[ok])
    return mx[mx > -np.inf]


def summary(null, rep, n_replicates):
    """Console lines: replicate and row counts, and the QUANTILES of the null CLR and of the per-replicate
    maximum CLR (``replicate_maxima``)."""
    null = np.asarray(null, dtype=np.float64)
    ok = ~np.isnan(null)
    mx = replicate_maxima(null, rep, n_replicates)

    def q(v):
        return ', '.join(f'{k}: {np.quantile(v, k):.6g}' for k in QUANTILES) if len(v) else 'none'
    return [f'Empirical null: {n_replicates} neutral replicates, {len(null)} null rows.',
            f'  quantiles of the null CLR:              {q(null[ok])}',
            f'  quantiles of the per-replicate max CLR: {q(mx)}']
