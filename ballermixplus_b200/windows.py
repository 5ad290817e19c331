"""Centres and inclusive windows of the four scan modes -- SURVEY.md §8 row a6.

Restates the window rules of ``Scan._fixSize_noCenter``, ``_fixSize_siteCenter``,
``_siteBased`` and ``_alpha`` (/root/reference/BalLeRMix+_v1.py:513-610) as array
planners: each returns a ``ScanPlan`` with, per output row, the test position
``t``, the inclusive index window ``[lo, hi]`` handed to ``calcBaller`` and the two
leading output fields already formatted the way the reference's f-strings
format them (SURVEY.md appendix A.5/A.6).  Rows of the --noCenter mode that fall
into a gap (start_i >= end_i, v1:534) carry ``gap = True`` and are never sent to
the GPU.
"""
import math

import numpy as np


class ScanPlan:
    """Rows of one scan.  Site-centred modes keep the two leading output columns as the numpy
    values the reference prints (``site_phys`` int64, ``site_gen`` float64) so that a whole
    genome is never formatted row by row in Python; ``f0``/``f1`` give them as text on demand."""

    def __init__(self):
        self.t = []          # float64 test positions
        self.lo = []
        self.hi = []
        self._f0 = []        # first output column (physPos) as text
        self._f1 = []        # second output column (genPos) as text
        self.gap = []        # --noCenter gap rows (already complete in f0)
        self._pos = []       # --noCenter: the numeric midpoint of every row (f0 and gap lines hold it as text)
        self.site_phys = None
        self.site_gen = None

    def add(self, t, lo, hi, f0, f1, pos=None):
        self.t.append(t); self.lo.append(lo); self.hi.append(hi)
        self._f0.append(f0); self._f1.append(f1); self.gap.append(False); self._pos.append(pos)

    def set_sites(self, data, idx):
        """All rows are centred on the sites `idx` (a numpy index array)."""
        self.site_phys = np.ascontiguousarray(data.position[idx], dtype=np.int64)
        self.site_gen = np.ascontiguousarray(data.genPos[idx], dtype=np.float64)

    @property
    def f0(self):
        if self.site_phys is not None:
            return [f'{v}' for v in self.site_phys]
        return self._f0

    @property
    def f1(self):
        if self.site_gen is not None:
            return [f'{v}' for v in self.site_gen]
        return self._f1

    def text(self, j):
        """(physPos, genPos) text of non-gap row j, as ``f0[j]``, ``f1[j]`` give it, without formatting every row."""
        if self.site_phys is not None:
            return f'{self.site_phys[j]}', f'{self.site_gen[j]}'
        return self._f0[j], self._f1[j]

    def add_gap(self, line, pos=None):
        self.t.append(0.); self.lo.append(0); self.hi.append(-1)
        self._f0.append(line); self._f1.append(''); self.gap.append(True); self._pos.append(pos)

    def phys(self):
        """float64 [rows]: the physPos of every row as a number (the site's position, or the --noCenter midpoint,
        gap rows included)."""
        if self.site_phys is not None:
            return self.site_phys.astype(np.float64)
        return np.array(self._pos, dtype=np.float64)

    def take(self, idx):
        """A plan of the rows ``idx`` (ascending indices) only, in that order."""
        sub = ScanPlan()
        sub.t, sub.lo, sub.hi, sub.gap = (np.asarray(a)[idx] for a in (self.t, self.lo, self.hi, self.gap))
        if self.site_phys is not None:
            sub.site_phys, sub.site_gen = self.site_phys[idx], self.site_gen[idx]
        else:
            sub._f0, sub._f1, sub._pos = ([v[i] for i in idx] for v in (self._f0, self._f1, self._pos))
        return sub

    def arrays(self):
        return (np.array(self.t, dtype=np.float64), np.array(self.lo, dtype=np.int64),
                np.array(self.hi, dtype=np.int64), np.array(self.gap, dtype=bool))

    def __len__(self):
        return len(self.t)


def plan_alpha(data, s):
    """Default mode (v1:598-610): every int(s)-th site, window = all sites."""
    step = int(s)
    if step < 1:
        raise ValueError('-s/--step must be at least 1 in this mode (the reference would loop forever)')
    N = data.numSites
    plan = ScanPlan()
    idx = np.arange(0, N, step)
    plan.t = data.genPos[idx]
    plan.lo = np.zeros(len(idx), np.int64)
    plan.hi = np.full(len(idx), N - 1, np.int64)
    plan.gap = np.zeros(len(idx), bool)
    plan.set_sites(data, idx)
    return plan


def _sorted(a):
    return len(a) < 2 or bool(np.all(a[1:] >= a[:-1]))


def plan_site_based(data, r, s):
    """-w r (v1:580-594): r sites to the left, r+1 to the right, centre index int(i)."""
    if not s > 0:
        raise ValueError('-s/--step must be positive')
    N = data.numSites
    plan = ScanPlan()
    if float(s).is_integer() and float(r).is_integer():
        # whole-number steps (the usual case; argparse hands -s over as a float): same ranges, as arrays
        c = np.arange(0, N, int(s), dtype=np.int64)
        plan.t = data.genPos[c]
        plan.lo = np.maximum(0, c - int(r))
        plan.hi = np.minimum(N - 1, c + int(r) + 1)
        plan.gap = np.zeros(len(c), bool)
        plan.set_sites(data, c)
        return plan
    i = 0
    centres = []
    while i < N:
        c = int(i)
        w = np.arange(max(0, i - r), min(N - 1, i + r + 1) + 1, dtype=int)   # as v1:588-589
        plan.add(data.genPos[c], int(w[0]), int(w[-1]), None, None)
        centres.append(c)
        i += s
    plan.set_sites(data, np.array(centres, dtype=np.int64))
    return plan


def plan_fixsize_site_center(data, w, s):
    """--fixWinSize -w W (v1:549-577): bp window around every int(s)-th site."""
    step = int(s)
    if step < 1:
        raise ValueError('-s/--step must be at least 1 in this mode (the reference would loop forever)')
    N = data.numSites
    pos = data.position
    plan = ScanPlan()
    if N and _sorted(pos):
        # sorted positions: the reference's two monotone pointers are two binary searches
        idx = np.arange(0, N, step, dtype=np.int64)
        ts = pos[idx]
        start = np.maximum(0, ts - w / 2)
        end = np.minimum(ts + w / 2, pos[-1])
        plan.t = data.genPos[idx]
        plan.lo = np.searchsorted(pos, start, 'left').astype(np.int64)
        plan.hi = np.minimum(np.searchsorted(pos, end, 'left'), N - 1).astype(np.int64)
        plan.gap = np.zeros(len(idx), bool)
        plan.set_sites(data, idx)
        return plan
    si = ei = 0
    last = pos[-1] if N else 0
    for i in range(0, N, step):
        ts = pos[i]
        start = max(0, ts - w / 2)
        end = min(ts + w / 2, last)
        while pos[si] < start:
            si += 1
        while ei < N and pos[ei] < end:
            ei += 1
        if ei < si:
            print(start, si, end, ei)
            raise SystemExit(1)                                          # v1:566-570
        ei = min(ei, N - 1)
        plan.add(data.genPos[i], si, ei, None, None)
    plan.set_sites(data, np.arange(0, N, step))
    return plan


def plan_fixsize_no_center(data, w, s):
    """--fixWinSize --noCenter -w W -s S (v1:513-545): windows of S bp on a W/2 grid origin."""
    if not s > 0:
        raise ValueError('-s/--step must be positive')
    N = data.numSites
    pos = data.position
    plan = ScanPlan()
    if N == 0:
        return plan
    start = int(math.floor(2 * float(pos[0]) / w) * (w / 2))
    end = start + s
    midpos = start + s / 2
    si = ei = 0
    while midpos <= pos[-1]:
        while pos[si] < start:
            si += 1
        while (ei + 1) < N and pos[ei] < end:
            ei += 1
        gen_site = midpos * data.Rrate
        if si >= ei:
            plan.add_gap('%d\t%g\t0\tNA\tNA\tNA\t0\n' % (midpos, gen_site), midpos)
        else:
            plan.add(gen_site, si, ei, f'{midpos}', f'{midpos * data.Rrate}', midpos)
        start += s; midpos += s; end += s
    return plan


def make_plan(data, fixSize=False, r=0, s=1, phys=False, noCenter=False):
    """Mode selection of ``Scan.__init__`` (v1:613-639), with its console messages."""
    if fixSize:
        print('You\'ve chosen to fix the size (in nt) of sliding window for scanning.')
        if r == 0:
            print('Please set a window width in nt with "-w" or "--window" command.')
            raise SystemExit(0)
        if not phys:
            print(f'Please make sure to use physical positions as coordinates if fixed-length '
                  f'windows are chosen (--fixSize). Scan will continue with physical positions '
                  f'with a rec rate of {data.Rrate} cM/nt.')
        w = float(r)
        if noCenter:
            print('Computing LR on %.3f kb windows on every %s nt. Using physical positions by '
                  'default.' % (w / 1e3, s))
            return plan_fixsize_no_center(data, w, s)
        print('Computing LR on %.3f kb windows on every %g informative sites. Using physical '
              'positions by default.' % (w / 1e3, s))
        return plan_fixsize_site_center(data, w, s)
    if r != 0:
        print('Computing LR on every %s site/s, with a radius of %g informative sites on either '
              'side.' % (s, r))
        return plan_site_based(data, r, s)
    print('Computing LR on every %s site/s, using informative sites with exp(-A*dist) >= 1e-8.' % (s))
    return plan_alpha(data, s)
