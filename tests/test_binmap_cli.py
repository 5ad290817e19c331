"""Binned spectra through the whole command line on the CPU, with the C oracle as the scan: one input with
--support, --refine, --regions, --balPos and --null/--pvalues against a literal per-site restatement of the same run,
--targets as a line subset of the full binned run, --inputList against one-input runs, and the genome sharding of a
binned run over gloo against one process."""
import os

import numpy as np
import pytest
import torch.multiprocessing as mp

import null_data
import refine_oracle
import util
from ballermixplus_b200 import cli, scan
from ballermixplus_b200.native import ScanProblem
from ballermixplus_b200.problem import GridOrder
from test_balpos import SplitOracleScan
from test_binmap import _perturbed, _write
from test_targets import _free_port, _worker


class ClassOracle(SplitOracleScan):
    """The device scan of every option (plain, profile, split, refine) from the C oracle on the product's tables."""

    def load_refine(self, fA, n_fx, n_fa, row_of, SP):
        self.tables = (np.asarray(fA), n_fx, n_fa, np.asarray(row_of), np.asarray(SP))

    def refine(self, t, lo, hi, box):
        return refine_oracle.refine(self.problem, *self.tables, t, lo, hi, box)


class LiteralOracle(ClassOracle):
    """ClassOracle on the literal per-site tables: every site its own class, g_i and P_i looked up in the file of
    its bin, the selection row of its (k, n); the fine rows of --refine gathered the same way (``layout``)."""

    def __init__(self, data, neutral, sel, grids, device=0):
        order = GridOrder(grids)
        b = data.siteBin
        g = np.array([neutral.spects[s].spect[(int(k), int(n))] for k, n, s in zip(data.count, data.total, b)])
        P = np.array([neutral.spects[s].sampProps[int(n)] for n, s in zip(data.total, b)])
        SP = np.stack([sel.classProbs[(x, a)][sel.cls] * P for x in order.x for a in order.a])
        prob = ScanProblem(data.genPos, np.arange(data.numSites, dtype=np.int32), g, SP,
                           np.array([float(v) for v in order.A]), len(order.x), len(order.a))
        prob.layout = (P, sel.cls.astype(np.int64))
        self.problem, self.order = prob, order


def _lines(path):
    with open(path) as fh:
        return fh.readlines()


def _bytes(path):
    with open(path, 'rb') as fh:
        return fh.read()


def _same_numbers(a, b):
    """Two files with the same lines up to the last bits of their numbers (1e-9 relative, as the CLR contract)."""
    la, lb = _lines(a), _lines(b)
    assert len(la) == len(lb) and la[0] == lb[0]
    for x, y in zip(la, lb):
        for u, v in zip(x.split('\t'), y.split('\t'), strict=True):
            try:
                fu, fv = float(u), float(v)
            except ValueError:
                assert u == v
                continue
            assert fu == fv or abs(fu - fv) <= 1e-9 * max(abs(fv), 1.0), (x, y)


def _genome(d, names=('chrA.txt', 'chrB.txt'), n_sites=140):
    os.makedirs(os.path.join(d, 'in'), exist_ok=True)
    rng = np.random.default_rng(21)
    paths = [null_data.write_input(os.path.join(d, 'in', n), n_sites, rng, span=1_500_000) or
             os.path.join(d, 'in', n) for n in names]
    lst = _write(os.path.join(d, 'genome.txt'), '\n'.join(os.path.join('in', n) for n in names) + '\n')
    bins = _write(os.path.join(d, 'bins.txt'),
                  f'hi {_perturbed(null_data.SPECT, os.path.join(d, "hi.txt"), 4, False)}\n'
                  f'lo {_perturbed(null_data.SPECT, os.path.join(d, "lo.txt"), 9, False)}\n')
    return lst, paths, bins


def _map(d, tag, names):
    lines = {'chrA.txt': 'chrA.txt 1 400000 hi\nchrA.txt 900000 1500000 lo\n',
             'chrB.txt': 'chrB.txt 300000 1100000 lo\n',
             'rep0.txt': 'rep0.txt 1 700000 hi\n'}
    return _write(os.path.join(d, f'map_{tag}.txt'), 'input start end label\n' + ''.join(lines[n] for n in names))


def _run(argv):
    with util.quiet():
        cli.main(argv)


BASE = ['-w', '12', '--listA', '1e5,1e6,1e7', '--refineSteps', '2']


def test_one_input_every_option_equals_the_literal_restatement(tmp_path, monkeypatch):
    d = str(tmp_path)
    _, paths, bins = _genome(d)
    rng = np.random.default_rng(5)
    os.makedirs(os.path.join(d, 'reps'))
    reps = [null_data.write_input(os.path.join(d, 'reps', f'rep{i}.txt'), 80, rng, span=1_500_000) or
            f'reps/rep{i}.txt' for i in range(2)]
    null = _write(os.path.join(d, 'null.txt'), '\n'.join(reps) + '\n')
    mapf = _map(d, 'one', ['chrA.txt', 'rep0.txt'])

    def argv(tag):
        return (['-i', paths[0], '--spect', null_data.SPECT, '--spectBins', bins, '--binMap', mapf] + BASE +
                ['-o', os.path.join(d, f'{tag}_out.txt')] +
                [a for k in ('support', 'refine', 'balPos', 'pvalues', 'regions')
                 for a in (f'--{k}', os.path.join(d, f'{tag}_{k}.txt'))] + ['--null', null, '--threshold', '0.5'])
    monkeypatch.setattr(scan, 'DeviceScan', ClassOracle)
    _run(argv('class'))
    monkeypatch.setattr(scan, 'DeviceScan', LiteralOracle)
    _run(argv('literal'))
    for k in ('out', 'support', 'refine', 'balPos', 'pvalues', 'regions'):
        _same_numbers(os.path.join(d, f'class_{k}.txt'), os.path.join(d, f'literal_{k}.txt'))
    main = np.loadtxt(os.path.join(d, 'class_out.txt'), skiprows=1, ndmin=2)
    assert np.any(main[:, 2] > 0.5)                                        # rows above the cut: regions exist
    assert len(_lines(os.path.join(d, 'class_regions.txt'))) > 1
    assert _lines(os.path.join(d, 'class_refine.txt')) != _lines(os.path.join(d, 'class_out.txt'))   # rows moved


def test_targets_keep_the_lines_of_the_full_binned_run(tmp_path, monkeypatch):
    d = str(tmp_path)
    _, paths, bins = _genome(d)
    mapf = _map(d, 'one', ['chrA.txt'])
    pos = np.loadtxt(paths[0], skiprows=1)[:, 0]
    tfile = _write(os.path.join(d, 't.txt'), f'chrA.txt {pos[20]} {pos[60]}\n')     # across a bin edge
    monkeypatch.setattr(scan, 'DeviceScan', ClassOracle)

    def argv(tag, *extra):
        return (['-i', paths[0], '--spect', null_data.SPECT, '--spectBins', bins, '--binMap', mapf] + BASE +
                ['-o', os.path.join(d, f'{tag}_out.txt')] +
                [a for k in ('support', 'refine', 'balPos') for a in (f'--{k}', os.path.join(d, f'{tag}_{k}.txt'))] +
                list(extra))
    _run(argv('full'))
    _run(argv('part', '--targets', tfile))
    kept = (pos >= pos[20]) & (pos <= pos[60])
    for k in ('out', 'support', 'refine', 'balPos'):
        full, part = _lines(os.path.join(d, f'full_{k}.txt')), _lines(os.path.join(d, f'part_{k}.txt'))
        assert part == [full[0]] + [line for line, keep in zip(full[1:], kept) if keep], k


def test_input_list_equals_one_input_runs(tmp_path, monkeypatch):
    d = str(tmp_path)
    lst, paths, bins = _genome(d)
    monkeypatch.setattr(scan, 'DeviceScan', ClassOracle)
    kinds = ('out', 'support', 'refine', 'balPos')
    for tag in ('one', 'list'):
        for k in kinds:
            os.makedirs(os.path.join(d, tag, k))
    for p in paths:
        name = os.path.basename(p)
        _run(['-i', p, '--spect', null_data.SPECT, '--spectBins', bins, '--binMap', _map(d, name, [name])] + BASE +
             ['-o', os.path.join(d, 'one', 'out', name)] +
             [a for k in kinds[1:] for a in (f'--{k}', os.path.join(d, 'one', k, name))])
    _run(['--inputList', '-i', lst, '--spect', null_data.SPECT, '--spectBins', bins, '--binMap',
          _map(d, 'all', ['chrA.txt', 'chrB.txt'])] + BASE + ['-o', os.path.join(d, 'list', 'out')] +
         [a for k in kinds[1:] for a in (f'--{k}', os.path.join(d, 'list', k))])
    for k in kinds:
        for p in paths:
            name = os.path.basename(p)
            assert _bytes(os.path.join(d, 'list', k, name)) == _bytes(os.path.join(d, 'one', k, name)), (k, name)


def test_sharded_binned_run_equals_one_process(tmp_path, monkeypatch):
    from test_targets import ProfileOracleScan
    d = str(tmp_path)
    lst, paths, bins = _genome(d)
    mapf = _map(d, 'all', ['chrA.txt', 'chrB.txt'])
    monkeypatch.setattr(scan, 'DeviceScan', ProfileOracleScan)

    def argv(tag):
        os.makedirs(os.path.join(d, tag))
        return (['--inputList', '-i', lst, '--spect', null_data.SPECT, '--spectBins', bins, '--binMap', mapf] + BASE +
                ['-o', os.path.join(d, tag), '--regions', os.path.join(d, f'{tag}_r.txt'), '--threshold', '0.5'])
    _run(argv('one'))
    mp.spawn(_worker, args=(2, _free_port(), argv('many'), d), nprocs=2, join=True)
    for p in paths:
        name = os.path.basename(p)
        assert _bytes(os.path.join(d, 'many', name)) == _bytes(os.path.join(d, 'one', name))
    assert _bytes(os.path.join(d, 'many_r.txt')) == _bytes(os.path.join(d, 'one_r.txt'))


@pytest.mark.parametrize('flag', ['--getSpect', '--getConfig'])
def test_get_spect_refuses_a_listed_spectrum_it_would_write(flag, tmp_path, capsys):
    d = str(tmp_path)
    _, paths, _ = _genome(d)
    out = os.path.join(d, 'made.txt')
    _write(out + '.hi', '1\t200\t1.0\n')
    lst = _write(os.path.join(d, 'own.txt'), 'hi made.txt.hi\n')
    with pytest.raises(SystemExit) as e:
        cli.main(['-i', paths[0], '--spect', out, flag, '--spectBins', lst, '--binMap', _map(d, 'one', ['chrA.txt'])])
    assert e.value.code == 2
    assert 'is a file this run writes' in capsys.readouterr().err
    assert open(out + '.hi').read() == '1\t200\t1.0\n'


def test_get_spect_writes_no_empty_spectrum(tmp_path):
    d = str(tmp_path)
    _, paths, _ = _genome(d)
    out = os.path.join(d, 'made.txt')
    mapf = _write(os.path.join(d, 'all.txt'), 'chrA.txt 0 2000000 hi\n')          # covers every site
    with util.quiet(), pytest.raises(SystemExit):
        cli.main(['-i', paths[0], '--spect', out, '--getSpect', '--binMap', mapf])
    assert not os.path.exists(out) and os.path.getsize(out + '.hi') > 0


def test_fine_rows_of_a_binned_problem_are_the_per_site_rows(tmp_path):
    """refine.fine_tables on a binned problem: column c at fine point (x, a) is the selection row of c's (k, n) at
    (x, a) times the P of c's bin, checked per site against sel.rows_at and each bin's file; at a coarse point the
    fine row is the problem's SP row bit for bit."""
    from ballermixplus_b200 import bins as bins_mod, refine
    from ballermixplus_b200.grids import Grids
    from ballermixplus_b200.inputs import InputData
    from ballermixplus_b200.problem import build_problem
    from ballermixplus_b200.selection import NormalizedBetaBinom
    d = str(tmp_path)
    _, paths, bins = _genome(d)
    b = bins_mod.read_spect_bins(bins)
    m = bins_mod.read_bin_map(_map(d, 'one', ['chrA.txt']), ['chrA.txt'], ['hi', 'lo'])
    with util.quiet():
        neutral = bins_mod.BinnedNeutral.read(null_data.SPECT, b, m, False, False, False)
        data = bins_mod.attach(InputData(paths[0]), neutral, 'chrA.txt')
        grid = Grids(None, None, False, False, None, '1e5,1e6,1e7')
        sel = NormalizedBetaBinom(data, grid, False, False, False)
    prob, order = build_problem(data, neutral, sel, grid)
    assert prob.layout is not None and len(np.unique(data.siteBin)) == 3
    g = refine.RefineGrid(order, 3)
    box = g.boxes(np.array([1, 2]), np.array([0, 4]), np.array([3, 10]))
    row_of, SP = refine.fine_tables(g, box, neutral, sel, prob.layout)
    P = np.array([neutral.spects[s].sampProps[int(n)] for n, s in zip(data.total, data.siteBin)])
    live = np.flatnonzero(row_of >= 0)
    assert len(live) > 4
    for q in live:
        x, a = g.x[q // len(g.a)], g.a[q % len(g.a)]
        want = sel.rows_at([(x, a)])[0][sel.cls] * P
        assert np.array_equal(SP[row_of[q]][prob.cls], want), (x, a)
    cA, cx, ca = g.coarse(1, 0, 3)
    assert np.array_equal(SP[row_of[cx * len(g.a) + ca]], prob.SP[3])
