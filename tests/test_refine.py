"""Local grid refinement (refine.py, --refine / --refineSteps): fine axes, boxes, fine class rows, the flag checks
and the whole pipeline with the literal surface standing in for the device.  No GPU needed."""
import numpy as np
import pytest

import refine_oracle
import util
from ballermixplus_b200 import refine
from ballermixplus_b200.grids import Grids
from ballermixplus_b200.problem import GridOrder


def literal_axis(values, K, geometric):
    """The fine axis written out from its definition."""
    v = sorted(values, key=float)
    F = []
    for i in range(len(v) - 1):
        lo, hi = v[i], v[i + 1]
        F.append(lo)
        for j in range(1, K):
            if geometric and lo > 0 and hi > 0:
                F.append(lo * (hi / lo) ** (j / K))
            else:
                F.append(lo + (hi - lo) * j / K)
    F.append(v[-1])
    return F


def same_values(a, b):
    """Equal element by element in value, type and bits."""
    return len(a) == len(b) and all(type(p) is type(q) and repr(p) == repr(q) for p, q in zip(a, b))


@pytest.mark.parametrize('K', [1, 2, 4, 8])
def test_fine_axes_of_the_default_grid(K):
    order = GridOrder(Grids(None, None, False, False, None, None))
    g = refine.RefineGrid(order, K)
    for fine, coarse, geo in ((g.A, order.A, True), (g.x, order.x, False), (g.a, order.a, True)):
        assert same_values(fine, literal_axis(coarse, K, geo))
        assert len(fine) == (len(coarse) - 1) * K + 1
    # coarse points keep their Python objects: an int prints as the main file prints it
    assert g.A[0] == 100 and type(g.A[0]) is int and f'{g.A[0]}' == '100'
    assert g.A[-1] == 1e8 and g.a[0] == 0.001 and g.a[-1] == 1e9
    for vals, rank, fine in ((order.A, g.rank_A, g.A), (order.x, g.rank_x, g.x), (order.a, g.rank_a, g.a)):
        for i, v in enumerate(vals):
            assert fine[rank[i] * K] is v


def test_geometric_and_arithmetic_steps():
    F, _ = refine.fine_axis([100, 1e4], 2, True)
    assert F == [100, 100 * (1e4 / 100) ** (1 / 2), 1e4] and type(F[0]) is int
    F, _ = refine.fine_axis([0.25, 0.5], 4, False)
    assert F == [0.25, 0.25 + 0.25 * 1 / 4, 0.25 + 0.25 * 2 / 4, 0.25 + 0.25 * 3 / 4, 0.5]


def test_list_a_with_zero_and_negative_values_and_any_order():
    order = GridOrder(Grids(None, None, False, False, None, '500,-100,0,2000,100'))
    g = refine.RefineGrid(order, 4)
    assert same_values(g.A, literal_axis(order.A, 4, True))
    assert g.A[:9] == [-100.0, -75.0, -50.0, -25.0, 0.0, 25.0, 50.0, 75.0, 100.0]     # arithmetic through <= 0
    assert g.A[9] == 100.0 * (500.0 / 100.0) ** 0.25                                 # geometric above
    for i, v in enumerate(order.A):
        assert g.A[g.rank_A[i] * 4] == v


def test_single_value_axes_are_not_refined():
    order = GridOrder(Grids('0.3', 20, False, False, None, '1000'))
    g = refine.RefineGrid(order, 8)
    assert g.A == [1000.0] and g.x == [0.3] and g.a == [20.0]
    assert g.boxes(np.array([0]), np.array([0]), np.array([0])).tolist() == [[0, 0, 0, 0, 0, 0]]


def test_boxes_at_the_grid_edges_and_inside():
    order = GridOrder(Grids(None, None, False, False, None, '300,100,200,400'))
    g = refine.RefineGrid(order, 3)
    iA = np.array([order.A.index(100.0), order.A.index(200.0), order.A.index(400.0)])
    ix = np.array([order.x.index(min(order.x)), 3, order.x.index(max(order.x))])
    ia = np.zeros(3, np.int64)
    b = g.boxes(iA, ix, ia)
    assert b[:, :2].tolist() == [[0, 3], [0, 6], [6, 9]]
    assert b[0, 2:4].tolist() == [0, 3] and b[2, 2:4].tolist() == [24, 27]
    rx = g.rank_x[3]
    assert b[1, 2:4].tolist() == [(rx - 1) * 3, (rx + 1) * 3]
    for r in range(3):
        assert refine.box_range(g.rank_A[iA[r]], 4, 3) == tuple(b[r, :2])
        cA, cx, ca = g.coarse(iA[r], ix[r], ia[r])
        assert b[r, 0] <= cA <= b[r, 1] and b[r, 2] <= cx <= b[r, 3] and b[r, 4] <= ca <= b[r, 5]


@pytest.mark.parametrize('case,extra', [('ex2_B0_s5', []), ('Example2_B0maf_1kb-2site', []), ('Example1_B1', []),
                                        ('Example1_B2', []), ('Example1_B2maf', []), ('synth_mixed_n_B2_s20', []),
                                        ('Example1_B2', ['--minCount', '3']),
                                        ('Example2_B0maf_1kb-2site', ['--minCount', '2'])])
def test_fine_rows_at_coarse_points_are_the_scan_rows(case, extra):
    argv, _ = util.scan_cases()[case]
    opt, data, neutral, grid, sel = util.host_objects(argv + extra)
    order = GridOrder(grid)
    pairs = [(x, a) for x in order.x for a in order.a]
    rows = sel.rows_at(pairs)
    for r, p in enumerate(pairs):
        assert np.array_equal(rows[r].view(np.int64), sel.classProbs[p].view(np.int64)), p
    # and the SP rows of fine_tables at those points are build_problem's, bit for bit
    from ballermixplus_b200.problem import build_problem
    prob, _ = build_problem(data, neutral, sel, grid)
    g = refine.RefineGrid(order, 2)
    box = g.boxes(np.zeros(1, np.int64), np.zeros(1, np.int64), np.zeros(1, np.int64))
    row_of, SP = refine.fine_tables(g, box, neutral, sel)
    cA, cx, ca = g.coarse(0, 0, 0)
    assert np.array_equal(SP[row_of[cx * len(g.a) + ca]].view(np.int64), prob.SP[0].view(np.int64))


def test_fine_rows_between_coarse_points_follow_the_formula():
    """A fine row is the class row NormalizedBetaBinom would build with that (x, a) on its grid."""
    from ballermixplus_b200 import NormalizedBetaBinom
    argv, _ = util.scan_cases()['Example1_B2maf']
    opt, data, neutral, grid, sel = util.host_objects(argv)
    pairs = [(0.05 + 0.05 * 1 / 4, 5 * (10 / 5) ** (1 / 4)), (0.5, 1e9)]
    rows = sel.rows_at(pairs)

    class G1:
        x, abeta = [pairs[0][0]], [pairs[0][1]]
    one = NormalizedBetaBinom(data, G1, opt.nofreq, opt.MAF, opt.nosub)
    assert np.array_equal(rows[0], one.classProbs[pairs[0]])
    assert np.array_equal(rows[1], sel.classProbs[(0.5, 1e9)])


@pytest.mark.parametrize('bad', [0, 9, -1, 2.5, '2.5', 'x', None])
def test_check_steps_rejects(bad):
    with pytest.raises(ValueError):
        refine.check_steps(bad)


def test_check_steps_accepts():
    assert [refine.check_steps(k) for k in (1, '4', ' 8 ', 3.0)] == [1, 4, 8, 3]
    assert refine.DEFAULT_STEPS == 4 and refine.MAX_STEPS == 8


def _argv(tmp_path, *extra):
    argv, _ = util.scan_cases()['ex1_B2_fixgrid']
    return util.abs_paths(argv) + ['-o', str(tmp_path / 'out.txt')] + list(extra)


@pytest.mark.parametrize('bad', ['0', '9', '2.5', 'x'])
def test_cli_rejects_bad_refine_steps(bad, tmp_path, capsys):
    from ballermixplus_b200.cli import main
    with pytest.raises(SystemExit) as exc:
        main(_argv(tmp_path, '--refine', str(tmp_path / 'r.txt'), '--refineSteps', bad))
    assert exc.value.code == 2
    assert '--refineSteps' in capsys.readouterr().err


def test_cli_defaults():
    from ballermixplus_b200.cli import build_parser
    opt = build_parser().parse_args(['-i', 'a', '--spect', 'b'])
    assert opt.refine is None and opt.refineSteps == 4


def test_cli_refuses_refine_under_torchrun_before_any_work(tmp_path, monkeypatch, capsys):
    from ballermixplus_b200 import cli, native

    def no(*a, **k):
        raise AssertionError('reached the computation')

    monkeypatch.setenv('WORLD_SIZE', '2')
    monkeypatch.setattr(cli, 'InputData', no)
    monkeypatch.setattr(native, 'lib', no)
    with pytest.raises(SystemExit) as exc:
        cli.main(_argv(tmp_path, '--refine', str(tmp_path / 'r.txt')))
    assert exc.value.code == 2
    assert 'one GPU' in capsys.readouterr().err
    assert not (tmp_path / 'out.txt').exists() and not (tmp_path / 'r.txt').exists()


def test_scan_refuses_refine_under_torchrun_before_any_work(tmp_path, monkeypatch):
    from ballermixplus_b200 import native, scan
    monkeypatch.setenv('WORLD_SIZE', '2')
    monkeypatch.setattr(native, 'lib', lambda: (_ for _ in ()).throw(AssertionError('reached the device')))
    with pytest.raises(ValueError, match='one GPU'):
        scan.Scan(None, None, None, None, str(tmp_path / 'o.txt'), refine=str(tmp_path / 'r.txt'))
    monkeypatch.setenv('WORLD_SIZE', '1')
    with pytest.raises(ValueError):
        scan.Scan(None, None, None, None, str(tmp_path / 'o.txt'), refine=str(tmp_path / 'r.txt'), refine_steps=9)


#: one grid point on balancing data: rows with T > 0, nothing to refine
FIXED = ['-i', 'data/Example2_balancing_10MYA_DAF.txt', '--spect', 'data/HC_CEU_Neut_DAF_spect_for_B2.txt',
         '--fixX', '0.5', '--fixAlpha', '20', '--listA', '5000', '-s', '50']


def run_pipeline(case, K):
    """refine.py end to end with the literal surface as the device -> (case dict, grid, refined, moved, main
    lines, refine lines).  ``case``: a golden scan case, or an argv."""
    from ballermixplus_b200.scan import format_rows
    c = refine_oracle.coarse_case(util.scan_cases()[case][0] if isinstance(case, str) else case)
    T, iA, ix, ia, ns = c['rows']
    dev = refine_oracle.OracleDev(c['prob'], c['order'])
    grid, rows = refine.refine_rows(dev, c['neutral'], c['sel'], K, c['t'], c['lo'], c['hi'], iA, ix, ia)
    move = refine.moved(grid, T, iA, ix, ia, rows)
    main = format_rows(c['plan'], c['order'], T, iA, ix, ia, ns)
    return c, grid, rows, move, main, refine.format_refined(c['plan'], main, grid, rows, move)


@pytest.mark.parametrize('case,K', [('ex1_B2_w15_s7p5', 2), ('ex2_B0maf_noCenter_gaps', 4), ('ex2_B1_listA_s10', 3)])
def test_pipeline_with_the_literal_surface(case, K):
    c, grid, rows, move, main, lines = run_pipeline(case, K)
    T, iA, ix, ia, ns = c['rows']
    refine_oracle.check_refine_file(main, lines, move, T, iA)
    rT, fA, fx, fa, rns = rows
    live = iA >= 0
    assert np.all(rT[live] >= T[live] - 1e-9 * np.maximum(np.abs(T[live]), 1.))   # the coarse point is in the box
    assert np.all(fA[~live] == -1) and np.all(rT[~live] == -np.inf)
    if case != 'ex2_B0maf_noCenter_gaps':
        assert move.any()
    # a moved row prints the fine point, whose literal T is the printed CLR
    for j in np.flatnonzero(move)[:5]:
        f = lines[j].rstrip('\n').split('\t')
        assert f[3] == f'{grid.x[fx[j]]}' and f[4] == f'{grid.a[fa[j]]}' and f[5] == f'{grid.A[fA[j]]}'
        assert int(f[6]) == rns[j]


def test_pipeline_of_a_fixed_grid_copies_the_main_file():
    c, grid, rows, move, main, lines = run_pipeline(FIXED, 4)
    assert grid.A == [5000.0] and grid.x == [0.5] and grid.a == [20.0]
    assert (c['rows'][1] >= 0).sum() > 0 and not move.any() and lines == main
