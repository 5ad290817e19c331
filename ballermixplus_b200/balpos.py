"""Balancing-versus-sweep rows (``--balPos``): the row maximum over each half of the (A, x, alpha) grid.

The beta-binomial shapes with alpha >= 1 are the balancing footprint (``--findBal`` scans exactly those) and the
shapes with alpha < 1 the sweep-like one.  One scan (``blmx_scan_split``) gives, per centre, the main row and the
reference's rule restricted to each half: A in visiting order, then (x, a) in visiting order, strict '>' from
T = 0, an A without sites skipped (v1:451,458,501).  Each half keeps the run's A and x grids, so with the default x
grid the ``bal`` half is the ``--findBal`` grid; the ``pos`` half is not the ``--findPos`` statistic, which also
changes the x grid.  ``CLR_bal - CLR_pos`` is a difference of composite-likelihood maxima: it ranks how clearly a row
prefers one half, it is not a calibrated test.

Pure numpy: no device is needed here.
"""
import numpy as np

BALPOS_HEADER = ('physPos\tgenPos\tCLR_bal\tx_bal\ts_bal\tA_bal\tnSites_bal\tCLR_pos\tx_pos\ts_pos\tA_pos\t'
                 'nSites_pos\n')

#: half_of_a values: an alpha of the balancing half, of the sweep half
BAL, POS = 0, 1


def half_of_a(alphas):
    """The half of every alpha of ``alphas`` (the visiting order, ``GridOrder.a``) -> int8 array, 0 (bal) where
    alpha >= 1, 1 (pos) where alpha < 1."""
    return np.array([BAL if float(a) >= 1 else POS for a in alphas], dtype=np.int8)


def check_grid(alphas):
    """Refuse a grid with no alpha on one side of 1 (``--fixAlpha``, ``--findBal``, ``--findPos``): one of the two
    halves would be empty.  Raises ValueError."""
    half = half_of_a(alphas)
    for h, name, side in ((BAL, 'bal', '>= 1'), (POS, 'pos', '< 1')):
        if not np.any(half == h):
            raise ValueError(f'--balPos needs alpha values on both sides of 1: the grid ({len(half)} alpha) has none '
                             f'{side} for the {name} half (--fixAlpha, --findBal and --findPos leave one half empty)')


def format_balpos(plan, order, bal, pos):
    """Lines of the --balPos file, one per row of the main output: the main row's two position fields, then each
    half's CLR, x, s, A and nSites printed as the main file prints them (``GridOrder.decode``, f'{v}').  --noCenter
    gap rows: the gap row's two position fields and, for each half, the gap row's 0 NA NA NA 0.  ``bal`` and ``pos``
    are the half rows (T, iA, ix, ia, nsites) of ``plan``."""
    f0, f1 = plan.f0, plan.f1
    lines = []
    for j in range(len(plan)):
        if plan.gap[j]:
            p0, p1 = f0[j].split('\t')[:2]
            lines.append(f'{p0}\t{p1}' + '\t0\tNA\tNA\tNA\t0' * 2 + '\n')
            continue
        fields = []
        for rows in (bal, pos):
            Tm, xh, ah, Ah, w = order.decode(*(col[j] for col in rows))
            fields.append(f'{Tm}\t{xh}\t{ah}\t{Ah}\t{w}')
        lines.append(f'{f0[j]}\t{f1[j]}\t' + '\t'.join(fields) + '\n')
    return lines


def write_balpos(path, plan, order, bal, pos):
    with open(path, 'w') as fh:
        fh.write(BALPOS_HEADER)
        fh.writelines(format_balpos(plan, order, bal, pos))
