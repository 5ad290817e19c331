"""Seeded problems for the variant parity tests (test infrastructure, not product code).

Grids whose size n_x * n_a sits on both sides of every width edge of the scan kernel (per_lane = ceil(n_xa / 32)
picks J in {1, 2, 4, 8, 16}; more than 512 points take several passes), with n_a mostly not dividing 32 so that
alpha halves and x rows straddle lanes and passes.  Class tables with huge ratios, underflow, exact zeros, a class
with G = 0, a class with SP = G = 0, alpha -> 1 and duplicated rows; A grids with A = 0 and A < 0 next to positive
A; sorted, shuffled and segmented layouts; ragged, empty and out-of-range windows.  Refine boxes whose point counts
sit on both sides of every width edge of refine_kernel, mixed with smaller boxes in one call.
"""
import numpy as np

from test_support_gpu import _ragged

# (n_x, n_a): n_xa = 1, 32, 33, 64, 65, 128, 129, 256, 257, 512, 513, 700
GRIDS = [(1, 1), (1, 32), (11, 3), (1, 64), (13, 5), (2, 64), (43, 3), (4, 64), (1, 257), (8, 64), (19, 27),
         (28, 25)]
KINDS = ['plain', 'huge', 'underflow', 'sp0', 'g0', 'spg0', 'alpha1', 'dup']
LAYOUTS = ['sorted', 'shuffled', 'segmented']
N_PROBLEMS = 2 * len(GRIDS)
# refine box sides (x points, a points): 32/33, 64/65, 96/98, 128/130, 192/195, 256/272 and 289 points
REFINE_BOXES = [(2, 16), (3, 11), (4, 16), (5, 13), (6, 16), (7, 14), (8, 16), (10, 13), (12, 16), (13, 15),
                (16, 16), (16, 17), (17, 17)]
N_FX, N_FA = 18, 19                 # fine axes: every box fits, at more than one offset
ALPHAS = [0.001, 0.01, 0.05, 0.1, 0.2, 0.5, 0.8, 1, 2, 5, 10, 50, 100, 300, 1e3, 1e4, 1e6, 1e9]


def scan_width(n_xa):
    """The scan kernel's rule: (J, passes over the grid)."""
    per_lane = (n_xa + 31) // 32
    J = 1 if per_lane <= 1 else 2 if per_lane <= 2 else 4 if per_lane <= 4 else 8 if per_lane <= 8 else 16
    return J, -(-n_xa // (32 * J))


def refine_width(max_pts):
    """refine_kernel's rule: J from the largest box of the call."""
    per_lane = (max_pts + 31) // 32
    for J in (1, 2, 3, 4, 6, 8, 16):
        if per_lane <= J:
            return J
    raise ValueError(max_pts)


def _table(rng, G, n_rows, kind, special):
    """SP [n_rows, C] around G, with the problem's extreme entries."""
    C = len(G)
    SP = G[None, :] * 10.0 ** rng.normal(0, 0.7, (n_rows, C))
    r = rng.integers(0, n_rows, 3)
    if kind == 'huge':
        SP[r[0], :] = G * 10.0 ** rng.uniform(3, 9, C)
        SP[r[1], rng.integers(0, C)] *= 1e9
    elif kind == 'underflow':
        SP[r[0], :] *= 1e-300
    elif kind == 'sp0':
        SP[r, rng.integers(0, C, 3)] = 0.0
    elif kind == 'g0':
        SP[:, special] = 10.0 ** rng.uniform(-3, 0, n_rows)          # R = SP / 0 = +inf
    elif kind == 'spg0':
        SP[:, special] = np.where(rng.random(n_rows) < 0.5, 0.0, 10.0 ** rng.uniform(-3, 0, n_rows))  # NaN or +inf
    elif kind == 'alpha1':
        SP[:, special] = G[special] * 10.0 ** rng.uniform(-30, -20, n_rows)       # R -> 0 where alpha -> 1
    elif kind == 'dup' and n_rows > 1:
        for _ in range(max(1, n_rows // 4)):                           # exact ties between grid points
            a, b = np.sort(rng.choice(n_rows, 2, replace=False))
            SP[b] = SP[a]
    return SP


def problem_name(k):
    n_x, n_a = GRIDS[k // 2]
    nonpos = (k + k // len(KINDS)) % 2 == 1
    return f'{k}-{n_x}x{n_a}-{KINDS[k % len(KINDS)]}-{LAYOUTS[k % len(LAYOUTS)]}-{"Anonpos" if nonpos else "Apos"}'


def make_problem(k):
    """Problem k of the campaign -> dict(prob, t, lo, hi, alphas, kind, layout, nonpos, batch, name)."""
    from ballermixplus_b200.native import ScanProblem
    rng = np.random.default_rng(7000 + k)
    n_x, n_a = GRIDS[k // 2]
    kind = KINDS[k % len(KINDS)]
    layout = LAYOUTS[k % len(LAYOUTS)]
    nonpos = (k + k // len(KINDS)) % 2 == 1
    n_xa = n_x * n_a
    n_sites = int(rng.choice([70, 160, 300]))
    C = int(rng.choice([2, 5, 13, 40]))
    span = 10.0 ** rng.uniform(-4, -1)
    g = np.sort(rng.random(n_sites)) * span
    if rng.random() < 0.5:                                             # exact duplicate positions
        d = rng.integers(1, n_sites - 1, 6)
        g[d] = g[d - 1]
    w = rng.random(C) ** 3 + 1e-2
    cls = rng.choice(C, size=n_sites, p=w / w.sum()).astype(np.int32)
    G = rng.random(C) * 10.0 ** rng.uniform(-6, 0, C) + 1e-12
    special = int(np.argmin(np.bincount(cls, minlength=C) + (np.bincount(cls, minlength=C) == 0) * n_sites))
    mid = n_sites // 2
    g_mid = g[mid]
    if kind == 'alpha1':                                               # near-duplicates around one centre
        g[mid - 12:mid + 12] = g[mid] + span * 1e-13 * np.arange(-12, 12)
        cls[mid - 12:mid + 12:2] = special
    SP = _table(rng, G, n_xa, kind, special)
    if kind in ('g0', 'spg0'):
        G[special] = 0.0
    # A in visiting order: windows from a few sites to all of them; A = 0 and A < 0 (alpha > 1) next to them
    n_pos = int(rng.choice([1, 3, 5]))
    A = 10.0 ** rng.uniform(0, 6, n_pos)
    A *= 18.42 / (A.min() * span) * 10.0 ** rng.uniform(-2, 1)
    if nonpos:
        A = np.concatenate([A, [0.0], -rng.uniform(0.05, 0.6, 2) / span])
    A = rng.permutation(A)
    # layout
    seg = None
    if layout == 'shuffled':
        perm = rng.permutation(n_sites)
        g, cls = g[perm], cls[perm]
    elif layout == 'segmented':                                       # two sequences end to end
        n1 = n_sites // 3
        g = np.concatenate([g[:n1] + 0.3 * span, g[n1:]])
        seg = np.array([0, n1], np.int64)
    prob = ScanProblem(g, cls, G, SP, A, n_x, n_a, seg_start=seg)
    m = 28
    c, lo, hi = _ragged(n_sites, m, seed=k)
    if layout == 'segmented':                                         # windows across the boundary
        c[1:4] = seg[1] + np.array([-2, 0, 1])
        lo[1:4], hi[1:4] = c[1:4] - 30, c[1:4] + 30
    if kind == 'alpha1':                                              # at the cluster, on and next to a site
        c[0] = c[1] = int(np.argmin(np.abs(g - g_mid)))
    t = g[c].copy()
    t[1::3] += span * 10.0 ** rng.uniform(-14, -3, len(t[1::3]))     # centres between sites
    alphas = rng.permutation(ALPHAS)[:n_a] if n_a <= len(ALPHAS) else rng.permutation(
        np.concatenate([ALPHAS, 10.0 ** rng.uniform(-3, 9, n_a - len(ALPHAS))]))
    return dict(prob=prob, t=t, lo=lo.astype(np.int64), hi=hi.astype(np.int64), alphas=alphas, kind=kind,
                layout=layout, nonpos=nonpos, batch=int([3, 7, 4096][k % 3]), special=special,
                k=k, name=problem_name(k))


def half_patterns(alphas, rng):
    """half_of_a patterns: the alpha >= 1 cut, alternating halves, one alpha alone in its half, all in one half."""
    from ballermixplus_b200.balpos import half_of_a
    n_a = len(alphas)
    alone = np.zeros(n_a, np.int8)
    alone[rng.integers(0, n_a)] = 1
    return {'alpha>=1': half_of_a(alphas), 'alternate': (np.arange(n_a) % 2).astype(np.int8), 'alone': alone,
            'one half': np.full(n_a, int(rng.integers(0, 2)), np.int8)}


def refine_case(k, p):
    """Fine tables and one refine call for problem k (dict of make_problem): the box of its first centre has the
    point count REFINE_BOXES[k % 13], the others are smaller boxes -> dict(fA, n_fx, n_fa, row_of, SP, box)."""
    rng = np.random.default_rng(9000 + k)
    prob = p['prob']
    n_rows = int(rng.integers(8, 40))                                 # few rows: a box holds its best row twice,
    SP = _table(rng, np.where(prob.G > 0, prob.G, 1e-3), n_rows, p['kind'], p['special'])    # so exact ties occur
    row_of = rng.integers(0, n_rows, N_FX * N_FA).astype(np.int32)
    row_of[1::7] = row_of[0::7][:len(row_of[1::7])]                   # neighbouring points share a row
    Apos = np.sort(np.abs(prob.A[prob.A > 0])) if np.any(prob.A > 0) else np.array([1e3])
    fA = np.geomspace(Apos[0] * 0.5, Apos[-1] * 2.0, 6)
    if p['nonpos']:
        fA = np.concatenate([np.sort(prob.A[prob.A <= 0]), fA])
    n = len(p['t'])
    box = np.zeros((n, 6), np.int32)
    bx, ba = REFINE_BOXES[k % len(REFINE_BOXES)]
    for j in range(n):
        nx, na = (bx, ba) if j % 4 == 0 else (int(rng.integers(1, bx + 1)), int(rng.integers(1, ba + 1)))
        a0 = int(rng.integers(0, len(fA)))
        a1 = int(rng.integers(a0, len(fA)))
        x0 = int(rng.integers(0, N_FX - nx + 1))
        y0 = int(rng.integers(0, N_FA - na + 1))
        box[j] = [a0, a1, x0, x0 + nx - 1, y0, y0 + na - 1]
    return dict(fA=fA, n_fx=N_FX, n_fa=N_FA, row_of=row_of, SP=SP, box=box)


def box_points(box):
    return (box[:, 3] - box[:, 2] + 1) * (box[:, 5] - box[:, 4] + 1)
