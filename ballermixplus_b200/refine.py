"""Local grid refinement of A_hat, x_hat and s_hat (``--refine``, DESIGN.md §3.10).

Each output row reports the grid point where T is largest, and the default grids are coarse.  Refinement takes,
for every row with T > 0, the best point of a finer grid inside a box around the row's grid maximum:

* Fine axis, for A, x and a separately: with v_0 < ... < v_{m-1} the distinct coarse values in numeric order and
  K the refinement factor, F[iK + j] = sub(v_i, v_{i+1}, j, K) for i < m - 1, j < K, and F[(m-1)K] = v_{m-1}.
  sub(lo, hi, 0, K) is the coarse Python object itself, so a fine point that is a coarse point prints as the
  main file prints it.  For j > 0 sub is geometric, lo * (hi / lo) ** (j / K), for A and a when lo > 0 and
  hi > 0, and arithmetic, lo + (hi - lo) * j / K, otherwise (always for x).  A one-value axis is not refined.
* Box: a coarse maximum at sorted index i takes the fine indices [max(0, (i-1)K), min((m-1)K, (i+1)K)] of its
  axis, which hold the coarse value.
* Class rows are built only at the fine (x, a) points some box needs, with NormalizedBetaBinom's arithmetic
  (``NormalizedBetaBinom.rows_at``); at coarse points they are bit-identical to the scan's rows.
* The device (``blmx_refine``) takes the box maximum with the scan's visiting rules.

A refined CLR is a maximum over more points than the coarse CLR, so it is biased upward relative to it and must
not be compared with CLRs of a coarse null (``--null``).  It is still a grid maximum, not a continuous MLE.

Pure numpy apart from the device object handed to ``refine_rows``.
"""
import numpy as np

MAX_STEPS = 8
DEFAULT_STEPS = 4


def check_steps(K):
    """The refinement factor as an int; raises ValueError unless it is an integer in 1..MAX_STEPS."""
    try:
        k = int(K.strip()) if isinstance(K, str) else int(K)
        ok = k == K or isinstance(K, str)
    except (TypeError, ValueError, AttributeError):
        ok = False
    if not ok or not 1 <= k <= MAX_STEPS:
        raise ValueError(f'the refinement factor must be an integer from 1 to {MAX_STEPS}, got {K!r}')
    return k


def _sub(lo, hi, j, K, geometric):
    if j == 0:
        return lo
    if geometric and lo > 0 and hi > 0:
        return lo * (hi / lo) ** (j / K)
    return lo + (hi - lo) * j / K


def fine_axis(values, K, geometric):
    """-> (F, rank): the fine axis of the coarse ``values`` (a list, numeric order) and, per coarse value in the
    order given, its index in numeric order (the fine index of a coarse value i is rank[i] * K)."""
    by_value = sorted(range(len(values)), key=lambda i: float(values[i]))
    v = [values[i] for i in by_value]
    rank = np.empty(len(values), np.int64)
    rank[by_value] = np.arange(len(values))
    F = []
    for i in range(len(v) - 1):
        F.extend(_sub(v[i], v[i + 1], j, K, geometric) for j in range(K))
    F.append(v[-1])
    return F, rank


def box_range(i, m, K):
    """Inclusive fine index range of the box around sorted coarse index i of an axis with m values."""
    return max(0, (i - 1) * K), min((m - 1) * K, (i + 1) * K)


class RefineGrid:
    """The fine axes of a GridOrder at factor K: ``A``, ``x``, ``a`` (lists of values, numeric order)."""

    def __init__(self, order, K):
        self.K = check_steps(K)
        self.m = (len(order.A), len(order.x), len(order.a))
        self.A, self.rank_A = fine_axis(order.A, self.K, True)
        self.x, self.rank_x = fine_axis(order.x, self.K, False)
        self.a, self.rank_a = fine_axis(order.a, self.K, True)

    def coarse(self, iA, ix, ia):
        """Fine indices of coarse (visiting-order) indices."""
        return (self.rank_A[iA] * self.K, self.rank_x[ix] * self.K, self.rank_a[ia] * self.K)

    def boxes(self, iA, ix, ia):
        """int32 [n, 6]: fA0, fA1, fx0, fx1, fa0, fa1 around the coarse maxima (visiting-order indices)."""
        out = np.empty((len(iA), 6), np.int32)
        for k, (r, m) in enumerate(((self.rank_A[iA], self.m[0]), (self.rank_x[ix], self.m[1]),
                                    (self.rank_a[ia], self.m[2]))):
            out[:, 2 * k] = np.maximum(0, (r - 1) * self.K)
            out[:, 2 * k + 1] = np.minimum((m - 1) * self.K, (r + 1) * self.K)
        return out


def fine_tables(grid, boxes, neutral, sel, layout=None):
    """Class rows at the fine (x, a) points the boxes need -> (row_of int32 [n_fx * n_fa], SP [n_rows, C]).
    row_of[fx * n_fa + fa] is the row of SP of that point, or -1; SP = rows * propSizes as build_problem forms it.
    ``layout`` (a binned problem's (P, sel_class), problem.build_binned): the classes are the problem's (k, n, bin)
    classes, each the selection row of its (k, n) times its bin's P."""
    n_fx, n_fa = len(grid.x), len(grid.a)
    need = np.zeros((n_fx, n_fa), bool)
    for b in np.unique(np.asarray(boxes)[:, 2:], axis=0):
        need[b[0]:b[1] + 1, b[2]:b[3] + 1] = True
    idx = np.flatnonzero(need.ravel())
    row_of = np.full(n_fx * n_fa, -1, np.int32)
    row_of[idx] = np.arange(len(idx), dtype=np.int32)
    rows = sel.rows_at([(grid.x[q // n_fa], grid.a[q % n_fa]) for q in idx])
    if layout is not None:
        P, sel_class = layout
        return row_of, rows[:, sel_class] * P[None, :]
    _, P = neutral.class_tables(sel.class_k, sel.class_n)
    return row_of, rows * P[None, :]


def refine_rows(dev, neutral, sel, K, t, lo, hi, iA, ix, ia):
    """Refine every row with a coarse maximum (iA >= 0) -> (grid, (T, fA, fx, fa, nsites)).

    ``dev`` is the DeviceScan of the coarse scan (``order``, ``load_refine``, ``refine``).  Rows without a
    coarse maximum get T = -inf and -1 indices.  One ``refine`` call; the library cuts it into launches."""
    grid = RefineGrid(dev.order, K)
    n = len(iA)
    T = np.full(n, -np.inf)
    fA, fx, fa = (np.full(n, -1, np.int32) for _ in range(3))
    ns = np.zeros(n, np.int32)
    live = np.flatnonzero(np.asarray(iA) >= 0)
    if len(live):
        boxes = grid.boxes(iA[live], ix[live], ia[live])
        row_of, SP = fine_tables(grid, boxes, neutral, sel, dev.problem.layout)
        dev.load_refine(np.array([float(v) for v in grid.A]), len(grid.x), len(grid.a), row_of, SP)
        got = dev.refine(t[live], lo[live], hi[live], boxes)
        for col, v in zip((T, fA, fx, fa, ns), got):
            col[live] = v
    return grid, (T, fA, fx, fa, ns)


def moved(grid, T, iA, ix, ia, refined):
    """bool [n]: rows whose box winner is not the coarse maximum's point and beats the row's CLR strictly."""
    rT, fA, fx, fa, _ = refined
    has = (np.asarray(iA) >= 0) & (fA >= 0)
    cA, cx, ca = (np.where(has, c, -1) for c in grid.coarse(np.where(has, iA, 0), np.where(has, ix, 0),
                                                             np.where(has, ia, 0)))
    return has & ((fA != cA) | (fx != cx) | (fa != ca)) & (rT > np.asarray(T))


def format_refined(plan, main_lines, grid, refined, move):
    """Lines of the refine file: the main file's line, except on moved rows, which print the refined point in
    the main file's row format (values f'{v}', as A_hat, x_hat and s_hat are printed)."""
    rT, fA, fx, fa, ns = refined
    lines = list(main_lines)
    rows = np.flatnonzero(move)
    if len(rows):
        f0, f1 = plan.f0, plan.f1
        for j in rows:
            lines[j] = (f'{f0[j]}\t{f1[j]}\t{np.float64(rT[j])}\t{grid.x[fx[j]]}\t{grid.a[fa[j]]}\t{grid.A[fA[j]]}'
                        f'\t{int(ns[j])}\n')
    return lines
