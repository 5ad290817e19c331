"""CPU side of the variant parity tests: the seeded problems of variant_problems cover every kernel width, and the
references the GPU tests compare with (surface_oracle, oracle_c) keep the reference's literal arithmetic where the
kernels' product form would not: a negative factor (alpha > 1, A < 0), a class with G = 0, SP = G = 0."""
import numpy as np

import surface_oracle
import util
import variant_problems as vp
from ballermixplus_b200.native import ScanProblem
from oracle import oracle_c


def test_generator_hits_every_scan_width_and_edge():
    sizes = {n_x * n_a for n_x, n_a in vp.GRIDS}
    widths = {vp.scan_width(s) for s in sizes}
    assert {J for J, _ in widths} == {1, 2, 4, 8, 16}
    assert any(passes > 1 for _, passes in widths)                     # several passes over the grid
    for edge in (32, 64, 128, 256, 512):                               # both sides of every edge
        assert edge in sizes and edge + 1 in sizes
        assert vp.scan_width(edge)[0] * 2 == vp.scan_width(edge + 1)[0] or edge == 512
    assert vp.scan_width(513) == (16, 2)
    assert any(n_a > 1 and 32 % n_a for _, n_a in vp.GRIDS)
    kinds = {(vp.KINDS[k % len(vp.KINDS)], (k + k // len(vp.KINDS)) % 2) for k in range(vp.N_PROBLEMS)}
    assert kinds == {(kind, a) for kind in vp.KINDS for a in (0, 1)}  # every table with and without A <= 0
    assert {vp.LAYOUTS[k % 3] for k in range(vp.N_PROBLEMS)} == set(vp.LAYOUTS)


def test_generator_hits_every_refine_width_and_edge():
    pts = [x * a for x, a in vp.REFINE_BOXES]
    assert max(max(b) for b in vp.REFINE_BOXES) <= 17                  # kRefineMaxSide
    assert all(x <= vp.N_FX and a <= vp.N_FA for x, a in vp.REFINE_BOXES)
    assert {vp.refine_width(p) for p in pts} == {1, 2, 3, 4, 6, 8, 16}
    for edge in (32, 64, 96, 128, 192, 256):
        assert any(p <= edge and vp.refine_width(p) == vp.refine_width(edge) for p in pts)
        assert any(p > edge and vp.refine_width(p) > vp.refine_width(edge) for p in pts)
    assert 289 in pts
    used = {vp.REFINE_BOXES[k % len(vp.REFINE_BOXES)] for k in range(vp.N_PROBLEMS)}
    assert used == set(vp.REFINE_BOXES)


def test_generated_problems_are_what_they_claim():
    for k in range(vp.N_PROBLEMS):
        p = vp.make_problem(k)
        prob = p['prob']
        assert prob.n_x * prob.n_a == np.prod(vp.GRIDS[k // 2])
        assert (np.any(prob.A <= 0)) == p['nonpos'] and np.any(prob.A > 0)
        if p['nonpos']:
            assert np.any(prob.A == 0) and np.any(prob.A < 0)
        if p['kind'] in ('g0', 'spg0'):
            assert prob.G[p['special']] == 0 and np.any(prob.cls == p['special'])
        if p['kind'] == 'spg0':
            assert prob.n_x * prob.n_a == 1 or np.any(prob.SP[:, p['special']] == 0)
        assert np.any(p['lo'] > p['hi']) and np.any(p['lo'] < 0) and np.any(p['hi'] >= len(prob.genpos))
        r = vp.refine_case(k, p)
        pts = vp.box_points(r['box'])
        assert pts.max() == np.prod(vp.REFINE_BOXES[k % len(vp.REFINE_BOXES)]) and len(set(pts)) > 1
        assert np.all(r['box'][:, 3] < vp.N_FX) and np.all(r['box'][:, 5] < vp.N_FA)
        assert len(np.unique(r['row_of'])) < len(r['row_of'])           # shared rows: exact ties


def _two_site():
    """G = (0.2, 0.3), SP = (0.05, 0.1), A = -50, t = 0, g = (-0.03, 0.02): both factors negative."""
    G = np.array([0.2, 0.3])
    SP = np.array([[0.05, 0.1]])
    g = np.array([-0.03, 0.02])
    return ScanProblem(g, np.array([0, 1], np.int32), G, SP, np.array([-50.0]), 1, 1)


def test_surface_oracle_is_literal_for_negative_factors():
    prob = _two_site()
    t, lo, hi = np.array([0.0]), np.array([0]), np.array([1])
    al = np.exp(50 * np.abs(prob.genpos))
    mix = al * prob.SP[0] + (1 - al) * prob.G
    assert np.all(mix < 0)                                             # the literal T is NaN ...
    prod = np.prod((1 - al) + al * prob.SP[0] / prob.G)
    assert abs(2 * np.log(prod) - 1.302) < 1e-3                        # ... the product form's is finite
    S, ns = surface_oracle.problem_surface(prob, t, lo, hi)
    assert np.isnan(S[0, 0, 0, 0]) and ns[0, 0] == 2
    with np.errstate(invalid='ignore'):
        T, n = util.literal_T(prob, 0.0, 0, 1, 0, 0)
    assert np.isnan(T) and n == 2
    for report_all in (False, True):                                   # NaN never wins: the all-zero row
        rT, rA, rxa, rn, _ = oracle_c.scan(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t, lo, hi,
                                           report_all=report_all)
        assert rT[0] == 0 and rA[0] == -1 and rxa[0] == -1 and rn[0] == 0


def _zero_class_problem():
    """Class 1 has G = 0: SP > 0 at grid point 0 (T = +inf), SP = 0 at grid point 1 (T = NaN)."""
    G = np.array([0.3, 0.0])
    SP = np.array([[0.2, 0.1], [0.4, 0.0], [0.6, 0.2]])
    g = np.array([0.001, 0.002, 0.003, 0.004])
    return ScanProblem(g, np.array([0, 1, 0, 0], np.int32), G, SP, np.array([1e3, 1e9]), 1, 3)


def test_surface_oracle_and_oracle_c_keep_infinities():
    prob = _zero_class_problem()
    t = np.array([0.0025, 0.0035])
    lo, hi = np.array([0, 2]), np.array([3, 3])                        # the second window misses class 1
    S, ns = surface_oracle.problem_surface(prob, t, lo, hi)
    with np.errstate(divide='ignore', invalid='ignore'):
        for xa in range(3):
            T, n = util.literal_T(prob, t[0], lo[0], hi[0], 0, xa)
            assert np.array_equal(S[0, 0, 0, xa], T, equal_nan=True) and n == ns[0, 0] == 4
    assert S[0, 0, 0, 0] == np.inf and np.isnan(S[0, 0, 0, 1]) and S[0, 0, 0, 2] == np.inf
    assert np.all(np.isfinite(S[1, 0]))
    assert ns[0, 1] == 0 and np.all(S[0, 1] == -np.inf)                # A = 1e9: no site has alpha >= 1e-8
    rT, rA, rxa, rn, _ = oracle_c.scan(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t, lo, hi)
    assert rT[0] == np.inf and rA[0] == 0 and rxa[0] == 0 and rn[0] == 4        # the first +inf wins
    fin = S[1, 0, 0]
    want = int(np.argmax(fin)) if fin.max() > 0 else -1
    assert rxa[1] == want and (want < 0 or rT[1] == fin[want] or abs(rT[1] - fin[want]) <= 1e-12 * abs(fin[want]))
    # SP = G = 0 at every grid point: NaN everywhere, nothing wins
    nan_only = ScanProblem(prob.genpos, prob.cls, prob.G, np.where(np.arange(2) == 1, 0.0, prob.SP), prob.A, 1, 3)
    S2, _ = surface_oracle.problem_surface(nan_only, t[:1], lo[:1], hi[:1])
    assert np.all(np.isnan(S2[0, 0]))
    for report_all in (False, True):
        rT, rA, rxa, rn, _ = oracle_c.scan(nan_only.genpos, nan_only.cls, nan_only.G, nan_only.SP, nan_only.A,
                                           t[:1], lo[:1], hi[:1], report_all=report_all)
        assert rT[0] == 0 and rA[0] == -1 and rxa[0] == -1 and rn[0] == 0
