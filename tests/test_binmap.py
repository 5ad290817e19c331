"""Binned neutral spectra (--spectBins, --binMap) on the CPU: the parsers and their refusals (before any input is
read), the class-table path against a literal per-site restatement on the C oracle for all five statistics, a map
with every site in bin 0 against no map, bins equal to --spect, --getSpect with a map, and the null's classes."""
import os

import numpy as np
import pytest

import util
from ballermixplus_b200 import bins, cli, null, scan, windows
from ballermixplus_b200.grids import Grids
from ballermixplus_b200.helpers import getConfig, getSpect
from ballermixplus_b200.inputs import InputData
from ballermixplus_b200.problem import build_problem
from ballermixplus_b200.selection import NormalizedBetaBinom
from test_regions import OracleScan

D = os.path.join(util.GOLD, 'data')
# (input, --spect, flags) of the five statistics
VARIANTS = {
    'B1': ('Example1_fullSweep_200kya_DAF.txt', 'HC_CEU_Neut_config_for_B1.txt', dict(nofreq=True)),
    'B2': ('Example1_fullSweep_200kya_DAF.txt', 'HC_CEU_Neut_DAF_spect_for_B2.txt', dict()),
    'B2maf': ('Example1_fullSweep_200kya_MAF.txt', 'HC_CEU_Neut_MAF_spect_for_B2maf.txt', dict(MAF=True)),
    'B0': ('Example2_balancing_10MYA_DAF_nosub.txt', 'HC_CEU_Neut_DAF-nosub_spect_for_B0.txt', dict(nosub=True)),
    'B0maf': ('Example2_balancing_10MYA_MAF_nosub.txt', 'HC_CEU_Neut_MAF-noSub_spect_for_B0maf.txt',
              dict(MAF=True, nosub=True)),
}
FLAGS = {'nofreq': '--noFreq', 'MAF': '--MAF', 'nosub': '--noSub'}


def _write(path, text):
    with open(path, 'w') as fh:
        fh.write(text)
    return str(path)


def _bytes(path):
    with open(path, 'rb') as fh:
        return fh.read()


def _perturbed(src, dst, seed, nofreq):
    """A spectrum (configuration) file with the (k, n) of ``src`` and clearly different fractions, summing to 1."""
    if nofreq:
        n = open(src).read().split('\t')[0]
        s = [0.5, 0.25, 0.125][seed % 3]
        return _write(dst, f'{n}\t{s}\t{1.0 - s}\n')
    rows = [line.split('\t') for line in open(src).read().splitlines() if line.strip()]
    w = np.exp(np.random.default_rng(seed).normal(0, 1.0, len(rows))) * np.array([float(r[2]) for r in rows])
    w /= w.sum()
    return _write(dst, ''.join(f'{r[0]}\t{r[1]}\t{float(v)!r}\n' for r, v in zip(rows, w)))


def _setup(tmp_path, variant, n_bins=3, same=False):
    """Bin files, list and a map of ``n_bins`` bins over thirds of the input (a stretch in bin 0 between them)."""
    infile, spect, flags = VARIANTS[variant]
    infile, spect = os.path.join(D, infile), os.path.join(D, spect)
    pos = np.loadtxt(infile, skiprows=1)[:, 0]
    lines, maplines = [], ['input\tstart\tend\tlabel\n', '# a comment\n']
    cuts = np.quantile(pos, np.linspace(0, 1, n_bins + 2))
    for b in range(n_bins):
        label = f'bin{b + 1}'
        f = spect if same else _perturbed(spect, tmp_path / f'{label}.txt', b + 1, flags.get('nofreq', False))
        lines.append(f'{label}\t{os.path.relpath(f, tmp_path)}\n')
        lo, hi = cuts[b + 1], cuts[b + 2] - 1 if b < n_bins - 1 else cuts[-1]
        maplines.append(f'{os.path.basename(infile)}\t{lo:.0f}\t{hi:.0f}\t{label}\textra\n')
    return (infile, spect, flags, _write(tmp_path / 'bins.txt', ''.join(lines)),
            _write(tmp_path / 'map.txt', ''.join(maplines)))


def _neutral(infile, spect, flags, listf, mapf):
    b = bins.read_spect_bins(listf)
    m = bins.read_bin_map(mapf, [os.path.basename(infile)], [lab for lab, _ in b])
    return bins.BinnedNeutral.read(spect, b, m, flags.get('nofreq', False), flags.get('MAF', False),
                                   flags.get('nosub', False))


# ---- parsing and refusals -------------------------------------------------------------------------------------
def test_site_bins_follow_the_map(tmp_path):
    listf = _write(tmp_path / 'l.txt', f'# bins\nhi {os.path.join(D, VARIANTS["B2"][1])}\n\nlo x.txt\n'
                   .replace('x.txt', os.path.join(D, VARIANTS['B2'][1])))
    b = bins.read_spect_bins(listf)
    assert [lab for lab, _ in b] == ['hi', 'lo']
    mapf = _write(tmp_path / 'm.txt', 'chr 10 20 hi\nchr 15 30 hi\nchr 31 31 lo\nother 0 100 lo\n')
    m = bins.read_bin_map(mapf, ['chr', 'other'], ['hi', 'lo'])
    got = m.site_bins('chr', [9, 10, 20, 25, 30, 31, 32])
    assert got.tolist() == [0, 1, 1, 1, 1, 2, 0]
    assert m.site_bins('none', [1, 2]).tolist() == [0, 0]


@pytest.fixture
def no_input_reads(monkeypatch):
    def fake(*a, **k):
        raise AssertionError('an input was read')
    monkeypatch.setattr(cli, 'InputData', fake)


@pytest.mark.parametrize('case', ['no_map', 'no_list', 'missing_label', 'bad_line', 'bad_number', 'overlap',
                                  'unknown_input', 'list_line', 'list_missing_file', 'map_is_output',
                                  'list_is_output'])
def test_refusals_before_any_input_is_read(case, tmp_path, no_input_reads, capsys):
    infile, spect, flags, listf, mapf = _setup(tmp_path, 'B2')
    name = os.path.basename(infile)
    out = str(tmp_path / 'out.txt')
    argv = ['-i', infile, '--spect', spect, '-o', out, '--spectBins', listf, '--binMap', mapf]
    bad = {'missing_label': f'{name} 1 5 nolabel\n', 'bad_line': f'{name} 1 5\n', 'bad_number': f'{name} 1 x bin1\n',
           'overlap': f'{name} 1 50 bin1\n{name} 40 60 bin2\n', 'unknown_input': 'chrX 1 5 bin1\n'}
    if case == 'no_map':
        del argv[-2:]
    elif case == 'no_list':
        del argv[-4:-2]
    elif case in bad:
        argv[-1] = _write(tmp_path / 'bad_map.txt', bad[case])
    elif case == 'list_line':
        argv[-3] = _write(tmp_path / 'bad_list.txt', 'bin1\n')
    elif case == 'list_missing_file':
        argv[-3] = _write(tmp_path / 'bad_list.txt', 'bin1 nowhere.txt\n')
    elif case == 'map_is_output':
        argv[argv.index('-o') + 1] = mapf
    elif case == 'list_is_output':
        argv[argv.index('-o') + 1] = listf
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 2
    err = capsys.readouterr().err
    assert '--binMap' in err or '--spectBins' in err, err


# ---- the class tables against a literal per-site restatement --------------------------------------------------
def _oracle_rows(prob, t, lo, hi):
    from oracle import oracle_c
    T, iA, ixa, ns, _ = oracle_c.scan(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t, lo, hi)
    return T, iA, ixa, ns


@pytest.mark.parametrize('variant', sorted(VARIANTS))
def test_binned_classes_equal_the_per_site_restatement(variant, tmp_path):
    from ballermixplus_b200.native import ScanProblem
    infile, spect, flags, listf, mapf = _setup(tmp_path, variant)
    kw = {**dict(nofreq=False, MAF=False, nosub=False), **flags}
    with util.quiet():
        data = InputData(infile, kw['nofreq'], kw['MAF'], kw['nosub'], 1)
        neutral = _neutral(infile, spect, flags, listf, mapf)
        bins.attach(data, neutral, os.path.basename(infile))
        grid = Grids(None, None, False, False, None, None)
        sel = NormalizedBetaBinom(data, grid, kw['nofreq'], kw['MAF'], kw['nosub'])
        plan = windows.make_plan(data, r=25)
    assert len(set(data.siteBin.tolist())) == 4                      # bins 1..3 and the unbinned stretch
    prob, order = build_problem(data, neutral, sel, grid)
    assert len(prob.G) > len(sel.class_k)
    # literal: every site its own class, g and P looked up in its bin's file
    g = np.array([neutral.spects[b].spect[(int(k), int(n))] for k, n, b in zip(data.count, data.total, data.siteBin)])
    P = np.array([neutral.spects[b].sampProps[int(n)] for n, b in zip(data.total, data.siteBin)])
    SP = np.stack([sel.get(x, a) * P for x in order.x for a in order.a])
    lit = ScanProblem(data.genPos, np.arange(data.numSites, dtype=np.int32), g, SP, prob.A, prob.n_x, prob.n_a)
    t, lo, hi, gap = plan.arrays()
    t, lo, hi = t[~gap][::4], lo[~gap][::4], hi[~gap][::4]                # windows cross the bin edges
    T0, iA0, x0, n0 = _oracle_rows(lit, t, lo, hi)
    T1, iA1, x1, n1 = _oracle_rows(prob, t, lo, hi)
    assert np.all(np.abs(T1 - T0) <= 1e-9 * np.maximum(np.abs(T0), 1.0))
    assert np.array_equal(n0, n1)
    assert np.array_equal(iA0, iA1) and np.array_equal(x0, x1)
    assert np.any(T0 > 0)


# ---- the command line with the C oracle as the scan ----------------------------------------------------------
@pytest.fixture
def oracle_scan(monkeypatch):
    monkeypatch.setattr(scan, 'DeviceScan', OracleScan)
    OracleScan.NULLS = []
    return OracleScan.NULLS


def _run(argv):
    with util.quiet():
        cli.main(argv)


def _T(path):
    return np.loadtxt(path, skiprows=1, ndmin=2)


def test_a_map_with_every_site_in_bin_0_is_byte_identical(tmp_path, oracle_scan):
    infile, spect, flags, listf, _ = _setup(tmp_path, 'B2')
    mapf = _write(tmp_path / 'empty_map.txt', f'{os.path.basename(infile)}\t-10\t-1\tbin1\n')  # covers no site
    base = ['-i', infile, '--spect', spect, '-w', '20', '--listA', '1e6,1e7']
    _run(base + ['-o', str(tmp_path / 'a.txt')])
    _run(base + ['-o', str(tmp_path / 'b.txt'), '--spectBins', listf, '--binMap', mapf])
    assert _bytes(tmp_path / 'a.txt') == _bytes(tmp_path / 'b.txt')


def test_bins_equal_to_spect_agree_with_the_unbinned_run(tmp_path, oracle_scan):
    infile, spect, flags, listf, mapf = _setup(tmp_path, 'B2', same=True)
    base = ['-i', infile, '--spect', spect, '-w', '20', '--listA', '1e6,1e7']
    _run(base + ['-o', str(tmp_path / 'a.txt')])
    _run(base + ['-o', str(tmp_path / 'b.txt'), '--spectBins', listf, '--binMap', mapf])
    a, b = _T(tmp_path / 'a.txt'), _T(tmp_path / 'b.txt')
    assert np.all(np.abs(a[:, 2] - b[:, 2]) <= 1e-9 * np.maximum(np.abs(a[:, 2]), 1.0))
    assert np.array_equal(a[:, 6], b[:, 6])


@pytest.mark.parametrize('variant', sorted(VARIANTS))
def test_binned_cli_rows_equal_the_literal_restatement(variant, tmp_path, oracle_scan):
    """The main file of a binned command line (the oracle on the product's class tables) against the C oracle on
    the literal per-site tables of the same windows, and against the unbinned run (the bins change the CLR)."""
    from ballermixplus_b200.native import ScanProblem
    from ballermixplus_b200.problem import GridOrder
    infile, spect, flags, listf, mapf = _setup(tmp_path, variant)
    kw = {**dict(nofreq=False, MAF=False, nosub=False), **flags}
    base = ['-i', infile, '--spect', spect, '-w', '20', '--listA', '1e6,1e7'] + [FLAGS[f] for f in flags]
    _run(base + ['-o', str(tmp_path / 'a.txt')])
    _run(base + ['-o', str(tmp_path / 'b.txt'), '--spectBins', listf, '--binMap', mapf])
    a, b = _T(tmp_path / 'a.txt'), _T(tmp_path / 'b.txt')
    assert a.shape == b.shape and not np.array_equal(a[:, 2], b[:, 2])     # the bins change the statistic
    with util.quiet():
        data = InputData(infile, kw['nofreq'], kw['MAF'], kw['nosub'], 1)
        neutral = _neutral(infile, spect, flags, listf, mapf)
        bins.attach(data, neutral, os.path.basename(infile))
        grid = Grids(None, None, False, False, None, '1e6,1e7')
        sel = NormalizedBetaBinom(data, grid, kw['nofreq'], kw['MAF'], kw['nosub'])
        t, lo, hi, gap = windows.make_plan(data, r=20).arrays()
    order = GridOrder(grid)
    g = np.array([neutral.spects[s].spect[(int(k), int(n))] for k, n, s in zip(data.count, data.total, data.siteBin)])
    P = np.array([neutral.spects[s].sampProps[int(n)] for n, s in zip(data.total, data.siteBin)])
    SP = np.stack([sel.get(x, a) * P for x in order.x for a in order.a])
    lit = ScanProblem(data.genPos, np.arange(data.numSites, dtype=np.int32), g, SP,
                      np.array([float(v) for v in order.A]), len(order.x), len(order.a))
    assert not gap.any()
    T, iA, ixa, ns = _oracle_rows(lit, t, lo, hi)
    assert np.all(np.abs(b[:, 2] - T) <= 1e-9 * np.maximum(np.abs(T), 1.0))
    assert np.array_equal(b[:, 6], ns)
    A_hat = np.array([float(order.A[i]) if i >= 0 else 0.0 for i in iA])
    assert np.array_equal(b[:, 5], A_hat)


@pytest.mark.parametrize('config', [False, True])
def test_get_spect_with_a_map_is_get_spect_of_each_bin(config, tmp_path, no_input_reads):
    infile, spect, flags, listf, mapf = _setup(tmp_path, 'B2')
    out = str(tmp_path / 'made.txt')
    with util.quiet(), pytest.raises(SystemExit):
        cli.main(['-i', infile, '--spect', out, '--getConfig' if config else '--getSpect', '--binMap', mapf])
    rows = open(infile).read().splitlines()
    pos = np.array([float(r.split('\t')[0]) for r in rows[1:]])
    m = bins.read_bin_map(mapf, [os.path.basename(infile)], ['bin1', 'bin2', 'bin3'])
    b = m.site_bins(os.path.basename(infile), pos)
    for k, suffix in enumerate(['', '.bin1', '.bin2', '.bin3']):
        sub = _write(tmp_path / f'sub{k}.txt', '\n'.join([rows[0]] + [r for r, bb in zip(rows[1:], b) if bb == k])
                     + '\n')
        ref = str(tmp_path / f'ref{k}.txt')
        with util.quiet():
            getConfig(sub, ref) if config else getSpect(sub, ref, False, False)
        assert _bytes(out + suffix) == _bytes(ref), suffix


def test_null_classes_with_a_map_equal_standalone_replicates(tmp_path):
    import null_data
    rng = np.random.default_rng(3)
    reps = [null_data.write_input(str(tmp_path / f'rep{i}.txt'), 300, rng) or str(tmp_path / f'rep{i}.txt')
            for i in range(2)]
    spect = null_data.SPECT
    listf = _write(tmp_path / 'bins.txt', f'hi {_perturbed(spect, tmp_path / "hi.txt", 5, False)}\n'
                                          f'lo {_perturbed(spect, tmp_path / "lo.txt", 6, False)}\n')
    mapf = _write(tmp_path / 'map.txt', 'rep0.txt 1 1000000 hi\nrep0.txt 2000000 3000000 lo\nrep1.txt 500000 '
                                        '2500000 lo\n')
    b = bins.read_spect_bins(listf)
    m = bins.read_bin_map(mapf, ['rep0.txt', 'rep1.txt'], ['hi', 'lo'])
    neutral = bins.BinnedNeutral.read(spect, b, m, False, False, False)
    grid = Grids(None, None, False, False, None, '1e5,1e6')
    with util.quiet():
        ds = null.read_replicates(reps, False, False, False, 1, False, 1e-6)
        prob, order = null.null_problem(ds, reps, neutral, grid, False, False, False)
        t, lo, hi, rep = null.null_plan(ds, reps, prob.seg_start, r=15)
    T = _oracle_rows(prob, t, lo, hi)[0]
    for i, (d, path) in enumerate(zip(ds, reps)):
        with util.quiet():
            bins.attach(d, neutral, os.path.basename(path))
            sel = NormalizedBetaBinom(d, grid, False, False, False)
            p1, _ = build_problem(d, neutral, sel, grid)
            t1, lo1, hi1, gap = windows.make_plan(d, r=15).arrays()
        T1 = _oracle_rows(p1, t1[~gap], lo1[~gap], hi1[~gap])[0]
        assert len(np.unique(d.siteBin)) > 1
        got = T[rep == i]
        assert np.all(np.abs(np.sort(got) - np.sort(T1)) <= 1e-9 * np.maximum(np.abs(T1).max(), 1.0))
