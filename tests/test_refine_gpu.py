"""blmx_refine on the GPU: box maxima against the literal surface, the refine file against the reference's own
arithmetic at the refined point, K = 1 against the main file, the file invariants, argument errors and the
range-checked build."""
import os
import subprocess
import sys

import numpy as np
import pytest

import refine_oracle
import util
from ballermixplus_b200 import refine, windows
from ballermixplus_b200.native import BlmxError, Scanner
from ballermixplus_b200.scan import DeviceScan

pytestmark = pytest.mark.gpu

CASES = sorted(util.scan_cases())
SAMPLE = 24                                 # rows per case compared with the literal surface


def device_case(argv):
    """Host objects, plan, the device's coarse rows and the DeviceScan (caller closes it)."""
    opt, data, neutral, grid, sel = util.host_objects(argv)
    dev = DeviceScan(data, neutral, sel, grid)
    with util.quiet():
        plan = windows.make_plan(data, fixSize=opt.size, r=opt.w, s=opt.step, phys=opt.phys, noCenter=opt.noCenter)
    t, lo, hi, gap = plan.arrays()
    n = len(plan)
    T = np.zeros(n)
    iA, ix, ia = (np.full(n, -1, np.int32) for _ in range(3))
    ns = np.zeros(n, np.int32)
    live = np.flatnonzero(~gap)
    if len(live):
        T[live], iA[live], ix[live], ia[live], ns[live] = dev.run(t[live], lo[live], hi[live])
    return dict(opt=opt, neutral=neutral, sel=sel, dev=dev, plan=plan, t=t, lo=lo, hi=hi, rows=(T, iA, ix, ia, ns))


def compare_with_oracle(dev, g, neutral, sel, t, lo, hi, iA, ix, ia, got, rows):
    """Refined rows `rows` (indices into t) against the box maxima of the literal surface: T within 1e-9, equal
    nSites, equal argmax or a tie within 1e-12.  Returns the number of proven ties."""
    boxes = g.boxes(iA[rows], ix[rows], ia[rows])
    row_of, SP = refine.fine_tables(g, g.boxes(iA[iA >= 0], ix[iA >= 0], ia[iA >= 0]), neutral, sel)
    fA = np.array([float(v) for v in g.A])
    rT, rA, rx, ra, rn = refine_oracle.refine(dev.problem, fA, len(g.x), len(g.a), row_of, SP, t[rows], lo[rows],
                                              hi[rows], boxes)
    T, A, X, Aa, N = (v[rows] for v in got)
    assert np.all(np.abs(T - rT) <= 1e-9 * np.maximum(np.abs(rT), 1.)), np.max(np.abs(T - rT))
    assert np.array_equal(N, rn)
    ties = 0
    for k in np.flatnonzero((A != rA) | (X != rx) | (Aa != ra)):
        b = boxes[k]
        S, _ = refine_oracle.box_surface(dev.problem, fA, len(g.a), row_of, SP, t[rows][k], lo[rows][k], hi[rows][k], b)
        mine = S[A[k] - b[0], X[k] - b[2], Aa[k] - b[4]]
        theirs = S[rA[k] - b[0], rx[k] - b[2], ra[k] - b[4]]
        assert abs(mine - theirs) <= 1e-12 * max(abs(theirs), 1.), (k, mine, theirs)
        ties += 1
    return ties


@pytest.mark.parametrize('K', [2, 4])
@pytest.mark.parametrize('case', CASES)
def test_box_maxima_match_the_literal_surface(case, K):
    c = device_case(util.scan_cases()[case][0])
    try:
        T, iA, ix, ia, ns = c['rows']
        g, got = refine.refine_rows(c['dev'], c['neutral'], c['sel'], K, c['t'], c['lo'], c['hi'], iA, ix, ia)
        live = np.flatnonzero(iA >= 0)
        assert np.all(got[1][iA < 0] == -1)
        if not len(live):
            return
        rng = np.random.default_rng(K)
        rows = np.sort(rng.choice(live, min(SAMPLE, len(live)), replace=False))
        compare_with_oracle(c['dev'], g, c['neutral'], c['sel'], c['t'], c['lo'], c['hi'], iA, ix, ia, got, rows)
        # the coarse point is in every box
        assert np.all(got[0][live] >= T[live] - 1e-9 * np.maximum(T[live], 1.))
    finally:
        c['dev'].close()


def test_ragged_and_empty_windows():
    argv, _ = util.scan_cases()['Example1_B2']
    c = device_case(argv)
    try:
        rng = np.random.default_rng(3)
        n_sites = len(c['dev'].problem.genpos)
        idx = rng.choice(n_sites, 60, replace=False)
        t = c['dev'].problem.genpos[idx]
        lo = np.maximum(idx - rng.integers(0, 80, 60), 0)
        hi = idx + rng.integers(0, 80, 60)
        lo[:5], hi[:5] = idx[:5] + 3, idx[:5] - 3                  # empty windows
        hi[5:8] = idx[5:8]                                          # one-sided
        T, iA, ix, ia, ns = c['dev'].run(t, lo, hi)
        assert np.all(iA[:5] == -1)
        g, got = refine.refine_rows(c['dev'], c['neutral'], c['sel'], 4, t, lo, hi, iA, ix, ia)
        rows = np.flatnonzero(iA >= 0)
        assert len(rows) > 10
        compare_with_oracle(c['dev'], g, c['neutral'], c['sel'], t, lo, hi, iA, ix, ia, got, rows)
        # an empty window on a valid box: nothing qualifies
        box = g.boxes(iA[rows[:1]], ix[rows[:1]], ia[rows[:1]])
        r = c['dev'].refine(t[:1], lo[:1], hi[:1], box)
        assert r[0][0] == -np.inf and r[1][0] == -1 and r[4][0] == 0
    finally:
        c['dev'].close()


def test_unsorted_positions():
    """Shuffled input (no distance cut) gives the oracle's box maxima too."""
    from ballermixplus_b200.native import ScanProblem
    c = device_case(util.scan_cases()['ex1_B2_w20_s10'][0])
    try:
        p = c['dev'].problem
        perm = np.random.default_rng(5).permutation(len(p.genpos))
        sp = ScanProblem(p.genpos[perm], p.cls[perm], p.G, p.SP, p.A, p.n_x, p.n_a)
        c['dev'].scanner.load(sp)
        c['dev'].problem = sp
        t = sp.genpos[::25]
        lo = np.zeros(len(t), np.int64)
        hi = np.full(len(t), len(sp.genpos) - 1, np.int64)
        T, iA, ix, ia, ns = c['dev'].run(t, lo, hi)
        g, got = refine.refine_rows(c['dev'], c['neutral'], c['sel'], 2, t, lo, hi, iA, ix, ia)
        rows = np.flatnonzero(iA >= 0)
        assert len(rows)
        compare_with_oracle(c['dev'], g, c['neutral'], c['sel'], t, lo, hi, iA, ix, ia, got, rows[:20])
    finally:
        c['dev'].close()


def run_cli(tmp_path, argv, name, *extra):
    from ballermixplus_b200.cli import main
    out = tmp_path / f'{name}.txt'
    with util.quiet():
        main(util.abs_paths(argv) + ['-o', str(out)] + list(extra))
    return out


@pytest.mark.parametrize('case', ['Example2_B2', 'ex1_B2_w15_s7p5', 'ex2_B0maf_noCenter_gaps', 'ex2_B1_listA_s10'])
def test_refine_file_against_the_reference_arithmetic(case, tmp_path):
    """Every row obeys the file's rules, and sampled moved rows are what the numpy oracle computes when it is run
    at that single grid point with the same window flags."""
    from oracle import oracle_cli
    argv, _ = util.scan_cases()[case]
    main = run_cli(tmp_path, argv, 'main', '--refine', str(tmp_path / 'ref.txt'))
    main_lines = open(main).read().splitlines(keepends=True)
    ref_lines = open(tmp_path / 'ref.txt').read().splitlines(keepends=True)
    assert ref_lines[0] == main_lines[0]
    moved = [j for j, (a, b) in enumerate(zip(main_lines, ref_lines)) if a != b]
    for j in moved:
        a, b = main_lines[j].split('\t'), ref_lines[j].split('\t')
        assert a[:2] == b[:2] and float(b[2]) > float(a[2])
    if case != 'ex2_B0maf_noCenter_gaps':
        assert moved
    for j in moved[:: max(1, len(moved) // 3)][:3]:
        f = ref_lines[j].rstrip('\n').split('\t')
        kw = util.oracle_kwargs(argv)
        kw.update(x=repr(float(f[3])), abeta=float(f[4]), listA=repr(float(f[5])))
        lines = oracle_cli.scan_file(**kw)
        g = lines[j].rstrip('\n').split('\t')
        assert g[:2] == f[:2] and g[6] == f[6]
        assert abs(float(g[2]) - float(f[2])) <= 1e-9 * max(abs(float(f[2])), 1.), (g, f)


@pytest.mark.parametrize('case', ['Example1_B2', 'Example2_B2maf', 'ex2_B2_fixwin_s50'])
def test_k1_reproduces_the_main_file(case, tmp_path):
    """K = 1: the box holds coarse points only, so a row can move only to a grid point that ties with the coarse
    maximum within rounding."""
    argv, _ = util.scan_cases()[case]
    main = run_cli(tmp_path, argv, 'main', '--refine', str(tmp_path / 'ref.txt'), '--refineSteps', '1')
    main_lines = open(main).read().splitlines(keepends=True)
    ref_lines = open(tmp_path / 'ref.txt').read().splitlines(keepends=True)
    ties = [(j, r.rstrip('\n').split('\t'), m.rstrip('\n').split('\t'))
            for j, (m, r) in enumerate(zip(main_lines, ref_lines)) if m != r]
    if ties:
        util.assert_ties(argv, ties)


@pytest.mark.parametrize('case', ['Example2_B2', 'ex2_B0maf_noCenter_gaps'])
def test_main_and_support_files_do_not_change(case, tmp_path):
    argv, _ = util.scan_cases()[case]
    a = run_cli(tmp_path, argv, 'a', '--support', str(tmp_path / 'sa.txt'))
    b = run_cli(tmp_path, argv, 'b', '--support', str(tmp_path / 'sb.txt'), '--refine', str(tmp_path / 'r.txt'))
    assert open(a).read() == open(b).read()
    assert open(tmp_path / 'sa.txt').read() == open(tmp_path / 'sb.txt').read()


def test_pvalue_file_does_not_change(tmp_path):
    import null_data
    lst, _ = null_data.make_replicates(str(tmp_path), n_reps=2, n_sites=120)
    argv = ['-i', os.path.join(util.GOLD, 'data', 'synth_n200.txt'), '--spect', null_data.SPECT, '--usePhysPos',
            '--rec', '1e-8', '--listA', '1000,2000,5000', '-s', '20']
    from ballermixplus_b200.cli import main
    outs = []
    for k, extra in enumerate(([], ['--refine', str(tmp_path / 'r.txt')])):
        o, p = tmp_path / f'o{k}.txt', tmp_path / f'p{k}.txt'
        with util.quiet():
            main(argv + ['-o', str(o), '--null', lst, '--pvalues', str(p)] + extra)
        outs.append((open(o).read(), open(p).read()))
    assert outs[0] == outs[1]


def test_fully_fixed_grid_copies_the_main_file(tmp_path):
    argv = ['-i', 'data/Example2_balancing_10MYA_DAF.txt', '--spect', 'data/HC_CEU_Neut_DAF_spect_for_B2.txt',
            '--fixX', '0.5', '--fixAlpha', '20', '--listA', '5000', '-s', '50']
    main = run_cli(tmp_path, argv, 'main', '--refine', str(tmp_path / 'ref.txt'), '--refineSteps', '8')
    text = open(main).read()
    assert text == open(tmp_path / 'ref.txt').read()
    assert any(float(r.split('\t')[2]) > 0 for r in text.splitlines()[1:])


def test_argument_errors():
    argv, _ = util.scan_cases()['ex1_B2_w15_s7p5']
    opt, data, neutral, grid, sel = util.host_objects(argv)
    from ballermixplus_b200.problem import build_problem
    prob, order = build_problem(data, neutral, sel, grid)
    g = refine.RefineGrid(order, 8)
    fA = np.array([float(v) for v in g.A])
    t, lo, hi = prob.genpos[:2], np.zeros(2, np.int64), np.full(2, 100, np.int64)
    with Scanner() as sc:
        with pytest.raises(BlmxError, match='error -3'):          # no problem loaded
            sc.load_refine(fA, len(g.x), len(g.a), np.zeros(len(g.x) * len(g.a), np.int32), np.ones((1, len(prob.G))))
        sc.load(prob)
        with pytest.raises(BlmxError, match='error -3'):          # no fine tables
            sc.refine(t, lo, hi, np.zeros((2, 6), np.int32))
        box = g.boxes(np.array([0, 1]), np.array([3, 4]), np.array([10, 20]))
        row_of, SP = refine.fine_tables(g, box, neutral, sel)
        with pytest.raises(BlmxError, match='error -1'):          # row_of out of range
            sc.load_refine(fA, len(g.x), len(g.a), np.full_like(row_of, len(SP)), SP)
        sc.load_refine(fA, len(g.x), len(g.a), row_of, SP)
        sc.refine(t, lo, hi, box)
        for bad in ([3, 2], [0, len(fA)], [-1, 0]):                # empty or off the axis
            b = box.copy()
            b[1, :2] = bad
            with pytest.raises(BlmxError, match='error -1'):
                sc.refine(t, lo, hi, b)
        b = box.copy()
        b[0, 2:4] = [0, len(g.x) - 1]                              # a point without a row, and > 17 x values
        with pytest.raises(BlmxError, match='error -1'):
            sc.refine(t, lo, hi, b)
        # 18 x points all with rows: too wide
        wide = np.array([[0, 0, 0, 17, 0, 0]], np.int32)
        row_all = np.arange(len(g.x) * len(g.a), dtype=np.int32)
        sc.load_refine(fA, len(g.x), len(g.a), row_all, np.ones((len(row_all), len(prob.G))))
        with pytest.raises(BlmxError, match='error -1'):
            sc.refine(t[:1], lo[:1], hi[:1], wide)
        sc.refine(t[:1], lo[:1], hi[:1], np.array([[0, 0, 0, 16, 0, 16]], np.int32))
        sc.load(prob)                                              # a new load drops the fine tables
        with pytest.raises(BlmxError, match='error -3'):
            sc.refine(t[:1], lo[:1], hi[:1], wide)


def test_checked_build_sees_no_violation_in_refine():
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import util
from ballermixplus_b200 import refine
from ballermixplus_b200.native import ScanProblem
from test_refine_gpu import device_case
for case, K, shuffle in (('Example1_B2', 8, False), ('ex2_B0maf_noCenter_gaps', 4, False), ('ex1_B2_w20_s10', 3, True)):
    c = device_case(util.scan_cases()[case][0])
    dev, t, lo, hi = c['dev'], c['t'], c['lo'], c['hi']
    if shuffle:
        p = dev.problem
        perm = np.random.default_rng(1).permutation(len(p.genpos))
        dev.problem = ScanProblem(p.genpos[perm], p.cls[perm], p.G, p.SP, p.A, p.n_x, p.n_a)
        dev.scanner.load(dev.problem)
    T, iA, ix, ia, ns = dev.run(t, lo, hi)
    g, got = refine.refine_rows(dev, c['neutral'], c['sel'], K, t, lo, hi, iA, ix, ia)
    v = dev.scanner.counters_all()['range_violations']
    print(case, int((iA >= 0).sum()), 'VIOLATIONS', v)
    assert v == 0
    dev.close()
print('VIOLATIONS 0')
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0' in out.stdout, out.stdout[-500:]
