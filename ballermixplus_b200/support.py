"""Support intervals for A_hat, x_hat and s_hat from the profiles of the likelihood surface.

The scan's statistic is T = 2 log LR of a composite likelihood: every site of the window enters as if it
were independent of the others.  For one centre, the profile of a grid axis is the maximum of T over the
other two axes (``blmx_scan_profile``: TA, Tx, Ta).  The support set of an axis at drop q is the set of its
grid values v whose profile is within q of the row's maximum:

    profile(v) >= T_hat - q,     T_hat = the row's CLR.

The default q, 3.841458820694124, is the 0.95 quantile of chi-square with one degree of freedom, the drop
that would give a 95 % confidence interval for an ordinary likelihood.  Sites are not independent, so for
this composite likelihood the interval is a *support interval*, not a calibrated confidence interval.

Pure numpy: no device is needed here.
"""
import math

import numpy as np

#: default drop in T units (T = 2 log LR): the chi-square(1) 0.95 quantile
DEFAULT_DROP = 3.841458820694124

SUPPORT_HEADER = 'physPos\tgenPos\tCLR\tA_lo\tA_hi\tx_lo\tx_hi\ts_lo\ts_hi\n'


def check_drop(q):
    """The drop as a float; raises ValueError unless it is finite and >= 0."""
    q = float(q)
    if not math.isfinite(q) or q < 0:
        raise ValueError(f'the support drop must be a finite number >= 0, got {q!r}')
    return q


def _hull(profile, T_hat, values, q):
    """(lo, hi) grid indices of the numerically lowest and highest value whose profile is >= T_hat - q;
    -1 where no value qualifies."""
    values = np.asarray([float(v) for v in values])
    by_value = np.argsort(values, kind='stable')
    ok = (np.asarray(profile, dtype=np.float64) >= (T_hat - q)[:, None])[:, by_value]
    any_ok = ok.any(axis=1)
    first = np.argmax(ok, axis=1)
    last = ok.shape[1] - 1 - np.argmax(ok[:, ::-1], axis=1)
    lo = np.where(any_ok, by_value[first], -1)
    hi = np.where(any_ok, by_value[last], -1)
    return lo.astype(np.int32), hi.astype(np.int32)


def support_intervals(T, iA, TA, Tx, Ta, order, q=DEFAULT_DROP):
    """Support intervals of A, x and s (the beta-binomial alpha) for every row.

    T, iA     the rows of the scan (``T`` is the CLR, ``iA < 0`` marks the all-zero row)
    TA, Tx, Ta  the profiles, [n, n_A], [n, n_x], [n, n_a], grid axes in visiting order
    order     the ``GridOrder`` the scan ran with (the grid values of each axis)
    q         drop in T units

    Returns a dict of six int32 arrays, ``A_lo, A_hi, x_lo, x_hi, s_lo, s_hi``: visiting-order indices of
    the lowest and highest grid value (by numeric value, whatever the visiting order) whose profile is
    ``>= T - q``.  The interval is the hull of that set: grid values inside it may fall below the cut when
    the set is not contiguous.  Rows with no grid point at T > 0 (the all-zero row) get -1 everywhere.
    NaN and -inf profile entries never qualify.
    """
    q = check_drop(q)
    T = np.asarray(T, dtype=np.float64)
    none = np.asarray(iA) < 0
    out = {}
    for name, prof, values in (('A', TA, order.A), ('x', Tx, order.x), ('s', Ta, order.a)):
        lo, hi = _hull(prof, T, values, q)
        lo[none] = -1
        hi[none] = -1
        out[name + '_lo'], out[name + '_hi'] = lo, hi
    return out


def format_support(plan, order, T, iA, ix, ia, ns, iv):
    """Lines of the support file, one per row of the main output.  The first three fields carry the main
    file's text; each interval end is the grid value printed as the main file prints A_hat, x_hat and s_hat
    (f'{v}'); rows without an interval print NA.  --noCenter gap rows: the main row's two position fields, 0
    and six NA."""
    text = {'A': [f'{v}' for v in order.A], 'x': [f'{v}' for v in order.x], 's': [f'{v}' for v in order.a]}
    f0, f1 = plan.f0, plan.f1
    lines = []
    for j in range(len(plan)):
        if plan.gap[j]:
            p0, p1 = f0[j].split('\t')[:2]
            lines.append(f'{p0}\t{p1}\t0' + '\tNA' * 6 + '\n')
            continue
        Tm = order.decode(T[j], iA[j], ix[j], ia[j], ns[j])[0]
        ends = []
        for axis in ('A', 'x', 's'):
            lo, hi = iv[axis + '_lo'][j], iv[axis + '_hi'][j]
            ends += ['NA', 'NA'] if lo < 0 else [text[axis][lo], text[axis][hi]]
        lines.append(f'{f0[j]}\t{f1[j]}\t{Tm}\t' + '\t'.join(ends) + '\n')
    return lines
