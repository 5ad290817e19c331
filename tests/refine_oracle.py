"""Box maxima of the fine grid from the literal surface (surface_oracle.c), for the --refine tests (not product
code).  ``refine`` restates blmx_refine's contract; ``OracleDev`` stands in for a DeviceScan in refine.py."""
import numpy as np

import surface_oracle
import util


def box_surface(prob, fA, n_fa, row_of, SP, t, lo, hi, b):
    """Literal T over one box -> (S [n_A_box, n_x_box, n_a_box], nsA [n_A_box])."""
    pts = [row_of[ix * n_fa + ia] for ix in range(b[2], b[3] + 1) for ia in range(b[4], b[5] + 1)]
    S, ns = surface_oracle.surface(prob.genpos, prob.cls, prob.G, np.asarray(SP)[pts], fA[b[0]:b[1] + 1], [t], [lo],
                                   [hi], b[3] - b[2] + 1, b[5] - b[4] + 1)
    return S[0], ns[0]


def refine(prob, fA, n_fx, n_fa, row_of, SP, t, lo, hi, box):
    """blmx_refine's result from the literal surface: visiting order fine A, x, a; strict '>' from -inf; an A
    without sites skipped -> (T, fA, fx, fa, nsites)."""
    n = len(t)
    T = np.full(n, -np.inf)
    oA, ox, oa = (np.full(n, -1, np.int32) for _ in range(3))
    ons = np.zeros(n, np.int32)
    for j in range(n):
        b = box[j]
        S, ns = box_surface(prob, np.asarray(fA), n_fa, row_of, SP, t[j], lo[j], hi[j], b)
        nfa = b[5] - b[4] + 1
        for k in range(len(ns)):
            if ns[k] == 0:
                continue
            flat = S[k].ravel()
            for p, v in enumerate(flat):
                if v > T[j]:
                    T[j], oA[j], ox[j], oa[j], ons[j] = v, b[0] + k, b[2] + p // nfa, b[4] + p % nfa, ns[k]
    return T, oA, ox, oa, ons


class OracleDev:
    """What refine.refine_rows needs of a DeviceScan, computed by ``refine`` on the CPU."""

    def __init__(self, prob, order):
        self.problem, self.order = prob, order

    def load_refine(self, fA, n_fx, n_fa, row_of, SP):
        self.tables = (np.asarray(fA), n_fx, n_fa, np.asarray(row_of), np.asarray(SP))

    def refine(self, t, lo, hi, box):
        return refine(self.problem, *self.tables, t, lo, hi, box)


def coarse_case(argv):
    """Host objects, plan and the coarse rows of a CLI argv from the C oracle (no GPU) -> dict."""
    from ballermixplus_b200 import windows
    from ballermixplus_b200.problem import build_problem
    from oracle import oracle_c
    opt, data, neutral, grid, sel = util.host_objects(argv)
    prob, order = build_problem(data, neutral, sel, grid)
    with util.quiet():
        plan = windows.make_plan(data, fixSize=opt.size, r=opt.w, s=opt.step, phys=opt.phys, noCenter=opt.noCenter)
    t, lo, hi, gap = plan.arrays()
    n = len(plan)
    T = np.zeros(n)
    iA, ix, ia = (np.full(n, -1, np.int32) for _ in range(3))
    ns = np.zeros(n, np.int32)
    live = np.flatnonzero(~gap)
    if len(live):
        rT, rA, rxa, rn, _ = oracle_c.scan(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t[live], lo[live], hi[live])
        T[live], iA[live], ns[live] = rT, rA, rn
        ix[live] = np.where(rA >= 0, rxa // prob.n_a, -1)
        ia[live] = np.where(rA >= 0, rxa % prob.n_a, -1)
    return dict(opt=opt, data=data, neutral=neutral, grid=grid, sel=sel, prob=prob, order=order, plan=plan, t=t,
                lo=lo, hi=hi, gap=gap, rows=(T, iA, ix, ia, ns))


def check_refine_file(main_lines, ref_lines, move, T, iA):
    """The refine file's rules: a row is the main row verbatim unless it moved; a moved row keeps the two
    position fields, has CLR > the main CLR, and every row's CLR is >= the main CLR."""
    assert len(main_lines) == len(ref_lines)
    for j, (m, r) in enumerate(zip(main_lines, ref_lines)):
        if not move[j]:
            assert r == m, (j, m, r)
            continue
        a, b = m.rstrip('\n').split('\t'), r.rstrip('\n').split('\t')
        assert a[:2] == b[:2] and len(b) == 7 and iA[j] >= 0
        assert float(b[2]) > float(a[2]) and np.float64(b[2]) > T[j]
