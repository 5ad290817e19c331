"""Turn the host objects (InputData, NeutralSFS, NormalizedBetaBinom, Grids) into the
class-indexed tables the C ABI takes (include/blmx.h, blmx_problem).

Everything ``calcBaller`` reads per site (/root/reference/BalLeRMix+_v1.py:470-497) depends
on the site only through its (k, n) class, so the device gets one row per class:
  G[c]       = NeutralSFS.probs of the class                               (v1:476)
  SP[xa][c]  = NormalizedBetaBinom.get(x, a) * NeutralSFS.propSizes        (v1:479,492)
with x, a (and A) in the iteration order of the reference's ``set(...)`` loops
(v1:453,473,474), which is what decides exact ties.

A binned run (bins.py: ``data.siteBin`` and a ``BinnedNeutral``) keys the classes (k, n, bin): G and P come from the
bin's spectrum, the selection row of the class's (k, n), multiplied by the class's P.
"""
import numpy as np

from .native import ScanProblem
from .bins import binned_classes
from .neutral import site_classes


class GridOrder:
    """The three grids in visiting order, with the Python objects kept for output."""

    def __init__(self, grids):
        # list(set(...)) is what the reference's loops iterate (v1:453,473,474); works on the
        # reference's own Grids object as well as on ours
        self.A, self.x, self.a = list(set(grids.A)), list(set(grids.x)), list(set(grids.abeta))

    @property
    def n_points(self):
        return len(self.A) * len(self.x) * len(self.a)

    def decode(self, T, iA, ix, ia, ns):
        """One result -> the reference's [T, x, a, A, nSites] list (v1:451,502)."""
        if iA < 0:
            return [0., 0., 0., 0., 0.]
        return [np.float64(T), self.x[ix], self.a[ia], self.A[iA], int(ns)]


def build_problem(data, neutral, sel, grids):
    """-> (ScanProblem, GridOrder)."""
    order = GridOrder(grids)
    if getattr(data, 'siteBin', None) is not None:
        return build_binned(data, neutral, sel, order)
    class_k, class_n, cls = site_classes(data.count, data.total)
    pairs = list(zip(class_k.tolist(), class_n.tolist()))
    if hasattr(neutral, 'class_tables'):
        G, P = neutral.class_tables(class_k, class_n)
    else:                                   # the reference's NeutralSFS: same dictionaries (v1:271,275)
        G = np.array([neutral.spect[p] for p in pairs], dtype=np.float64)
        P = np.array([neutral.sampProps[p[1]] for p in pairs], dtype=np.float64)
    if hasattr(sel, 'classProbs'):
        if not (np.array_equal(class_k, sel.class_k) and np.array_equal(class_n, sel.class_n)):
            raise ValueError('selection tables were built for different data')
        rows = sel.classProbs
    else:                                   # the reference's NormalizedBetaBinom: per-site arrays (v1:359)
        first = np.zeros(len(pairs), dtype=np.int64)
        first[cls[::-1]] = np.arange(len(cls))[::-1]          # first site of every class
        rows = {key: np.asarray(v)[first] for key, v in sel.normProbs.items()}
    SP = np.empty((len(order.x) * len(order.a), len(G)), dtype=np.float64)
    r = 0
    for x in order.x:
        for a in order.a:
            SP[r] = rows[(x, a)] * P
            r += 1
    prob = ScanProblem(data.genPos, cls, G, SP, np.array([float(v) for v in order.A]),
                       len(order.x), len(order.a))
    return prob, order


def binned_layout(data, neutral, sel):
    """Classes keyed (k, n, bin) -> (cls int32[N], G[C], P[C], sel_class int64[C]): sel_class[c] is the index of
    class c's (k, n) among the selection tables' classes."""
    ck, cn, cb, cls = binned_classes(data.count, data.total, data.siteBin)
    G, P = neutral.class_tables(ck, cn, cb)
    kmax = int(max(ck.max(), sel.class_k.max())) + 1 if len(ck) else 1
    sel_key = sel.class_n * kmax + sel.class_k            # ascending: site_classes sorts by (n, k)
    sel_class = np.searchsorted(sel_key, cn * kmax + ck)
    if len(ck) and not np.array_equal(sel_key[np.minimum(sel_class, len(sel_key) - 1)], cn * kmax + ck):
        raise ValueError('selection tables were built for different data')
    return cls, G, P, sel_class


def build_binned(data, neutral, sel, order):
    """``build_problem`` of a binned run -> (ScanProblem, GridOrder); the problem keeps ``layout`` = (P,
    sel_class) for the fine rows of refine.py."""
    cls, G, P, sel_class = binned_layout(data, neutral, sel)
    SP = np.empty((len(order.x) * len(order.a), len(G)), dtype=np.float64)
    r = 0
    for x in order.x:
        for a in order.a:
            SP[r] = sel.classProbs[(x, a)][sel_class] * P
            r += 1
    prob = ScanProblem(data.genPos, cls, G, SP, np.array([float(v) for v in order.A]), len(order.x), len(order.a))
    prob.layout = (P, sel_class)
    return prob, order
