"""Support intervals (support.py), the --support / --supportDrop flags and the surface oracle: no GPU needed."""
import math

import numpy as np
import pytest

import util
from ballermixplus_b200 import support
from ballermixplus_b200.windows import ScanPlan

NINF = -np.inf


class Order:
    """The three grid axes of a GridOrder, in visiting order."""

    def __init__(self, A, x, a):
        self.A, self.x, self.a = list(A), list(x), list(a)

    def decode(self, T, iA, ix, ia, ns):
        if iA < 0:
            return [0., 0., 0., 0., 0.]
        return [np.float64(T), self.x[ix], self.a[ia], self.A[iA], int(ns)]


def intervals(T, TA, Tx, Ta, order, q, iA=None):
    T = np.atleast_1d(np.asarray(T, np.float64))
    iA = np.zeros(len(T), np.int32) if iA is None else np.asarray(iA)
    return support.support_intervals(T, iA, np.atleast_2d(TA), np.atleast_2d(Tx), np.atleast_2d(Ta), order, q)


def test_lowest_and_highest_by_value_not_visiting_order():
    # --listA in any order: visiting order 500, 100, 2500, 50
    order = Order([500., 100., 2500., 50.], [0.5, 0.1], [1, 10, 100])
    iv = intervals(10., [10., 7., 7.5, 1.], [10., 9.], [NINF, 10., 8.], order, q=3.0)
    assert (iv['A_lo'][0], iv['A_hi'][0]) == (1, 2)        # 100 .. 2500 (50 falls out)
    assert (iv['x_lo'][0], iv['x_hi'][0]) == (1, 0)        # 0.1 .. 0.5
    assert (iv['s_lo'][0], iv['s_hi'][0]) == (1, 2)        # 10 .. 100


def test_ties_and_zero_drop():
    order = Order([100., 200., 300.], [0.5], [1., 2.])
    iv = intervals(5., [5., 2., 5.], [5.], [5., 5.], order, q=0.0)
    assert (iv['A_lo'][0], iv['A_hi'][0]) == (0, 2)        # two A tie at the maximum
    assert (iv['s_lo'][0], iv['s_hi'][0]) == (0, 1)
    iv = intervals(5., [5., 4.99, 1.], [5.], [5., 1.], order, q=0.0)
    assert (iv['A_lo'][0], iv['A_hi'][0]) == (0, 0)        # q = 0: the maximum alone
    assert (iv['s_lo'][0], iv['s_hi'][0]) == (0, 0)


def test_boundary_is_inclusive():
    order = Order([1., 2., 3.], [0.5], [1.])
    iv = intervals(10., [10., 10. - 2.5, 10. - 2.5000001], [10.], [10.], order, q=2.5)
    assert (iv['A_lo'][0], iv['A_hi'][0]) == (0, 1)


def test_nan_and_minus_inf_never_qualify():
    order = Order([1., 2., 3., 4.], [0.5], [1.])
    # A = 1 has no sites (-inf), A = 4 has a NaN profile
    iv = intervals(3., [NINF, 3., 2., np.nan], [3.], [3.], order, q=100.)
    assert (iv['A_lo'][0], iv['A_hi'][0]) == (1, 2)


def test_non_contiguous_support_set_gives_its_hull():
    order = Order([10., 20., 30., 40., 50.], [0.5], [1.])
    iv = intervals(8., [8., NINF, -50., 7., 1.], [8.], [8.], order, q=2.)
    # 10 and 40 qualify, 20 and 30 do not: the interval is the hull 10 .. 40
    assert (iv['A_lo'][0], iv['A_hi'][0]) == (0, 3)


def test_all_zero_rows_get_no_interval():
    order = Order([1., 2.], [0.5], [1.])
    iv = support.support_intervals(np.array([0., 4.]), np.array([-1, 1]), np.array([[-1., -2.], [1., 4.]]),
                                   np.array([[-1.], [4.]]), np.array([[-1.], [4.]]), order, 3.)
    for k in ('A_lo', 'A_hi', 'x_lo', 'x_hi', 's_lo', 's_hi'):
        assert iv[k][0] == -1 and iv[k][1] >= 0
    assert (iv['A_lo'][1], iv['A_hi'][1]) == (0, 1)


def test_several_rows_at_once():
    order = Order([3., 1., 2.], [0.5, 0.2], [1.])
    TA = np.array([[9., 8., 1.], [2., 2., 3.]])
    iv = intervals([9., 3.], TA, [[9., 0.], [3., 3.]], [[9.], [3.]], order, q=1.5)
    assert list(iv['A_lo']) == [1, 1] and list(iv['A_hi']) == [0, 0]
    assert list(iv['x_lo']) == [0, 1] and list(iv['x_hi']) == [0, 0]


@pytest.mark.parametrize('bad', [-1.0, -1e-12, math.nan, math.inf, -math.inf, 'abc'])
def test_check_drop_rejects(bad):
    with pytest.raises(ValueError):
        support.check_drop(bad)


def test_check_drop_accepts():
    assert support.check_drop('0') == 0.0 and support.check_drop(2) == 2.0
    assert support.DEFAULT_DROP == 3.841458820694124


def _plan(rows, gaps):
    plan = ScanPlan()
    for j, (t, f0, f1) in enumerate(rows):
        if j in gaps:
            plan.add_gap('%d\t%g\t0\tNA\tNA\tNA\t0\n' % (int(f0), float(f1)))
        else:
            plan.add(t, 0, 10, f0, f1)
    return plan


def test_format_support_text_of_grid_values_and_gap_rows():
    # ints stay ints, floats print as the main file prints them
    order = Order([100, 1000.0, 10000], [0.5, 0.25], [1, 2.5])
    plan = _plan([(1e-4, '100', '0.0001'), (0, '375', '0.000375'), (2e-4, '200', '0.0002')], gaps={1})
    T = np.array([12.5, 0., 0.])
    iA = np.array([1, -1, -1], np.int32)
    ix = np.array([0, -1, -1], np.int32)
    ia = np.array([1, -1, -1], np.int32)
    ns = np.array([7, 0, 0], np.int32)
    iv = {'A_lo': np.array([0, -1, -1]), 'A_hi': np.array([2, -1, -1]), 'x_lo': np.array([1, -1, -1]),
          'x_hi': np.array([0, -1, -1]), 's_lo': np.array([0, -1, -1]), 's_hi': np.array([1, -1, -1])}
    lines = support.format_support(plan, order, T, iA, ix, ia, ns, iv)
    assert lines == ['100\t0.0001\t12.5\t100\t10000\t0.25\t0.5\t1\t2.5\n',
                     '375\t0.000375\t0\tNA\tNA\tNA\tNA\tNA\tNA\n',
                     '200\t0.0002\t0.0\tNA\tNA\tNA\tNA\tNA\tNA\n']
    assert support.SUPPORT_HEADER.rstrip('\n').split('\t') == [
        'physPos', 'genPos', 'CLR', 'A_lo', 'A_hi', 'x_lo', 'x_hi', 's_lo', 's_hi']


def _argv(tmp_path, *extra):
    argv, _ = util.scan_cases()['ex1_B2_fixgrid']
    return util.abs_paths(argv) + ['-o', str(tmp_path / 'out.txt')] + list(extra)


@pytest.mark.parametrize('bad', ['-1', 'nan', 'inf', '-inf', 'x'])
def test_cli_rejects_bad_support_drop(bad, tmp_path, capsys):
    from ballermixplus_b200.cli import main
    with pytest.raises(SystemExit) as exc:
        main(_argv(tmp_path, '--support', str(tmp_path / 's.txt'), '--supportDrop', bad))
    assert exc.value.code == 2
    assert '--supportDrop' in capsys.readouterr().err


def test_cli_refuses_support_under_torchrun_before_any_work(tmp_path, monkeypatch, capsys):
    from ballermixplus_b200 import cli, native

    def no(*a, **k):
        raise AssertionError('reached the computation')

    monkeypatch.setenv('WORLD_SIZE', '2')
    monkeypatch.setattr(cli, 'InputData', no)
    monkeypatch.setattr(native, 'lib', no)
    with pytest.raises(SystemExit) as exc:
        cli.main(_argv(tmp_path, '--support', str(tmp_path / 's.txt')))
    assert exc.value.code == 2
    assert 'one GPU' in capsys.readouterr().err
    assert not (tmp_path / 'out.txt').exists() and not (tmp_path / 's.txt').exists()


def test_scan_refuses_support_under_torchrun_before_any_work(tmp_path, monkeypatch):
    from ballermixplus_b200 import native, scan
    monkeypatch.setenv('WORLD_SIZE', '2')
    monkeypatch.setattr(native, 'lib', lambda: (_ for _ in ()).throw(AssertionError('reached the device')))
    with pytest.raises(ValueError, match='one GPU'):
        scan.Scan(None, None, None, None, str(tmp_path / 'o.txt'), support=str(tmp_path / 's.txt'))
    with pytest.raises(ValueError):
        monkeypatch.setenv('WORLD_SIZE', '1')
        scan.Scan(None, None, None, None, str(tmp_path / 'o.txt'), support=str(tmp_path / 's.txt'), support_drop=-2)


def test_surface_oracle_is_the_literal_formula():
    """The C surface oracle against util.literal_T (math.fsum) at sampled grid points, and its -inf rows."""
    import surface_oracle
    from ballermixplus_b200.problem import build_problem
    argv, _ = util.scan_cases()['Example1_B2']
    opt, data, neutral, grid, sel = util.host_objects(argv)
    prob, order = build_problem(data, neutral, sel, grid)
    c = np.array([0, 300, 756])
    t = data.genPos[c]
    lo, hi = np.maximum(c - 40, 0), c + 40
    lo[2], hi[2] = 10, 5                                         # an empty window
    S, ns = surface_oracle.problem_surface(prob, t, lo, hi)
    assert S.shape == (3, len(prob.A), prob.n_x, prob.n_a)
    assert np.all(ns[2] == 0) and np.all(S[2] == -np.inf)
    rng = np.random.default_rng(0)
    for j in (0, 1):
        for _ in range(12):
            iA, ix, ia = rng.integers(len(prob.A)), rng.integers(prob.n_x), rng.integers(prob.n_a)
            T, n = util.literal_T(prob, t[j], lo[j], hi[j], iA, ix * prob.n_a + ia)
            assert n == ns[j, iA]
            if n == 0:
                assert S[j, iA, ix, ia] == -np.inf
            else:
                assert abs(S[j, iA, ix, ia] - T) <= 1e-12 * max(abs(T), 1.)
