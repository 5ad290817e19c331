"""Selection-model tables -- host side of SURVEY.md §8 row a4.

Mirrors ``NormalizedBetaBinom`` of the reference
(/root/reference/BalLeRMix+_v1.py:310-433): constructor
``NormalizedBetaBinom(InputData, Grids, nofreq, MAF, nosub)`` and ``get(x, a)``
returning the per-site normalised probabilities.  The table is built per
(k, n) CLASS, not per site: ``classProbs[(x, a)]`` is float64[C].  The arithmetic
is the reference's, call for call, so the entries are bit-identical to the
reference's per-site values (tests/test_reference_objects.py checks that against the
reference itself when /root/reference is present; tests/test_host_pipeline.py checks the
per-class tables against the oracle's per-site restatement everywhere):

  b(x, a) = a/x - a                                                   (v1:316)
  BB_x(j) = scipy.stats.betabinom(n, a, b(x, a)).pmf(j)                (v1:366-371)
  raw(k)  : B2/B0     BB(k)
            B2maf/B0maf  BB(k)+BB(n-k), halved at k == n/2 for even n  (v1:388-394)
            B1        BB(n) for k == 0, 1-BB(n)-BB(n) for k == 1 (sic) (v1:382)
  folded  = 0.5*(raw_x + raw_{1-x})                                    (v1:337-351)
  normBase = 1 - sum_{j in E} 0.5*(BB_x(j)+BB_{1-x}(j))                (v1:399-433)
      E: B2,B1 0..m-1 | B2maf 0..m-1, n-m+1..n-1 | B0 0..m-1, n
         B0maf 0..m-1, n-m+1..n          (m = InputData.minCount)
  probs  = folded / normBase

scipy's betabinom is the third-party arithmetic the parity bar hangs on
(SURVEY.md §8c: requirements.txt pins scipy>=1.5.0; 1.18.1 installed); it is
called here exactly as the reference calls it.
"""
import numpy as np
from scipy.stats import betabinom

from .neutral import site_classes


def stat_name(nofreq, MAF, nosub):
    if nofreq:
        return 'B1'
    if MAF:
        return 'B0maf' if nosub else 'B2maf'
    return 'B0' if nosub else 'B2'


class NormalizedBetaBinom:
    """Built per (k, n) class with ONE broadcast scipy call per sample size and side of the fold
    (x and 1-x): ``betabinom.pmf(j, n, a, b)`` over j = 0..n and the whole (x, a) grid.  scipy evaluates
    the pmf elementwise, so every entry has the bits of the reference's per-(x, a) frozen-distribution
    calls (tests/test_reference_objects.py compares all tables with the reference's, bit for bit;
    ``_slow_row`` keeps the call-for-call form for tests/test_host_pipeline.py)."""

    @staticmethod
    def _get_b(x, a):
        return a / x - a

    def __init__(self, InputData, Grids, nofreq, MAF, nosub):
        self.stat = stat_name(nofreq, MAF, nosub)
        self.class_k, self.class_n, self.cls = site_classes(InputData.count, InputData.total)
        self.minCount = InputData.minCount
        self._dist = {}
        self.classProbs = {}
        sizes = sorted(set(self.class_n.tolist()))
        members = {n: np.flatnonzero(self.class_n == n) for n in sizes}
        if self.stat == 'B1':
            for n in sizes:
                assert set(self.class_k[members[n]].tolist()) == {0, 1}
        xs, alphas = list(Grids.x), list(Grids.abeta)
        rows = {(x, a): np.zeros(len(self.class_k)) for x in xs for a in alphas}
        avec = np.array([float(a) for a in alphas])
        for n in sizes:
            j = np.arange(n + 1)
            # pmf[side][ix][ia][j]; b = a/x - a in Python arithmetic exactly as v1:316 forms it
            pmf = []
            for side in (lambda x: x, lambda x: 1. - x):
                bmat = np.array([[self._get_b(side(x), a) for a in alphas] for x in xs], dtype=np.float64)
                pmf.append(betabinom.pmf(j[None, None, :], n, avec[None, :, None], bmat[:, :, None]))
            k = self.class_k[members[n]]
            excl = self._excluded(n)
            for ix, x in enumerate(xs):
                for ia, a in enumerate(alphas):
                    px, pc = pmf[0][ix, ia], pmf[1][ix, ia]
                    folded = 0.5 * (self._raw_from(px, k, n) + self._raw_from(pc, k, n))
                    base = 1. - np.sum(0.5 * (px[excl] + pc[excl]))
                    rows[(x, a)][members[n]] = folded / base
        self.classProbs = rows

    def get(self, x, a):
        """Per-site normalised selection probabilities (reference API, v1:362)."""
        return self.classProbs[(x, a)][self.cls]

    def rows_at(self, pairs):
        """float64 [len(pairs), C]: the class rows at an explicit list of (x, a) points, with the constructor's
        arithmetic (one broadcast pmf per sample size and side of the fold), so a point of the scan's grid gets
        the bits of ``classProbs[(x, a)]``.  The fine grid of refine.py uses it."""
        out = np.zeros((len(pairs), len(self.class_k)))
        if not len(pairs):
            return out
        avec = np.array([float(a) for _, a in pairs])
        for n in sorted(set(self.class_n.tolist())):
            members = np.flatnonzero(self.class_n == n)
            j = np.arange(n + 1)
            pmf = []
            for side in (lambda x: x, lambda x: 1. - x):
                bvec = np.array([self._get_b(side(x), a) for x, a in pairs], dtype=np.float64)
                pmf.append(betabinom.pmf(j[None, :], n, avec[:, None], bvec[:, None]))
            k = self.class_k[members]
            excl = self._excluded(n)
            for r in range(len(pairs)):
                px, pc = pmf[0][r], pmf[1][r]
                folded = 0.5 * (self._raw_from(px, k, n) + self._raw_from(pc, k, n))
                base = 1. - np.sum(0.5 * (px[excl] + pc[excl]))
                out[r, members] = folded / base
        return out

    # -- pieces -----------------------------------------------------------------
    def _raw_from(self, p, k, n):
        """Unfolded probabilities of the classes k from the pmf p[0..n] (v1:375-396)."""
        s = self.stat
        if s == 'B1':
            return np.where(k == 0, p[n], (1. - p[n] - p[n]))
        if s in ('B2', 'B0'):
            return p[k]
        probs = p[k] + p[n - k]
        if n % 2 == 0:
            probs = np.where(k == int(n / 2), probs / 2, probs)
        return probs

    def _slow_row(self, x, a):
        """The same row built call for call as the reference does (v1:337-355); tests only."""
        sizes = sorted(set(self.class_n.tolist()))
        row = np.zeros(len(self.class_k))
        for n in sizes:
            idx = np.flatnonzero(self.class_n == n)
            k = self.class_k[idx]
            folded = 0.5 * (self._raw(k, n, x, a) + self._raw(k, n, 1. - x, a))
            row[idx] = folded / self._norm_base(n, x, a)
        return row

    def _pmf(self, j, n, x, a):
        key = (n, x, a)
        d = self._dist.get(key)
        if d is None:
            d = self._dist[key] = betabinom(n, a, self._get_b(x, a))
        return d.pmf(j)

    def _raw(self, k, n, x, a):
        s = self.stat
        if s == 'B1':
            sub = self._pmf(n, n, x, a)
            return np.where(k == 0, sub, (1. - sub - sub))
        if s in ('B2', 'B0'):
            return self._pmf(k, n, x, a)
        probs = self._pmf(k, n, x, a) + self._pmf(n - k, n, x, a)
        if n % 2 == 0:
            probs = np.where(k == int(n / 2), probs / 2, probs)
        return probs

    def _excluded(self, n):
        m = self.minCount
        s = self.stat
        if s in ('B2', 'B1'):
            return np.arange(m)
        if s == 'B2maf':
            return np.concatenate((np.arange(m), np.arange(n - m + 1, n)))
        if s == 'B0':
            return np.concatenate((np.arange(m), np.array([n])))
        return np.concatenate((np.arange(m), np.arange(n - m + 1, n + 1)))

    def _norm_base(self, n, x, a):
        excl = self._excluded(n)
        excluded_probs = 0.5 * (self._pmf(excl, n, x, a) + self._pmf(excl, n, 1. - x, a))
        return 1. - np.sum(excluded_probs)
