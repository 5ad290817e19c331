"""--targets on the GPU (run with -m gpu on a B200): a targeted run with --support, --refine, --null/--pvalues and
--regions against the full run, file by file (DESIGN.md §3.13), on one input and on a mixed-sample-size --inputList,
and two torchrun ranks writing the one-GPU targeted run's bytes."""
import os

import numpy as np
import pytest

import genome_data
import util
from test_genome_list_gpu import _torchrun
from test_regions_gpu import _null_maxima
from test_targets import _check_subset, _expected_regions, _kept, _lines

pytestmark = pytest.mark.gpu

FLAGS = ['-w', '40', '--supportDrop', '2.5', '--refineSteps', '2']
KINDS = {'out': '-o', 'support': '--support', 'pvalues': '--pvalues', 'refine': '--refine'}
DETAIL = ['support', 'pvalues', 'refine']


def _cli(argv):
    from ballermixplus_b200.cli import main
    with util.quiet():
        main(argv)


def _bytes(path):
    with open(path, 'rb') as fh:
        return fh.read()


def _cut(main_paths):
    """A cut that leaves several regions: the 0.7 quantile of the positive CLRs."""
    T = np.concatenate([[float(line.split('\t')[2]) for line in _lines(p)[1:]] for p in main_paths])
    return float(np.quantile(T[T > 0], 0.7))


def _check_refine(full, part, keep):
    """The refine file: the header and the full run's lines at the kept rows, byte for byte (DESIGN.md §3.13: why
    the fine tables of fewer rows give the same bits).  A CLR-only difference is reported with its size, after the
    weaker check that it stays within 1e-9 * max(|T|, 1) at the same fine point."""
    a, b = _lines(full), _lines(part)
    ref = a[:1] + [line for line, k in zip(a[1:], keep) if k]
    assert len(b) == len(ref)
    rel, other = [], 0
    for x, y in zip(ref, b):
        fx, fy = x.split('\t'), y.split('\t')
        other += fx[:2] + fx[3:] != fy[:2] + fy[3:]
        if x != y and fx[2] != 'CLR':
            rel.append(abs(float(fx[2]) - float(fy[2])) / max(abs(float(fx[2])), 1.0))
    assert other == 0 and max(rel, default=0.0) <= 1e-9
    assert not rel, f'{len(rel)} of {len(b) - 1} refine lines differ in CLR only, max rel {max(rel):.3e}'


def _run_pair(d, argv_of, names, reps, flags):
    """A plain run (for the cut), the full run with every option, and a run with --targets = its regions file ->
    (cut, the targets of every input)."""
    _cli(argv_of('plain', []) + flags)
    cut = _cut([os.path.join(d, 'plain', 'out', n) for n in names])
    extra = ['--null', reps, '--regions', os.path.join(d, 'full_r.txt'), '--threshold', repr(cut)]
    _cli(argv_of('full', DETAIL) + flags + extra)
    targets = os.path.join(d, 'full_r.txt')
    assert len(_lines(targets)) > 3
    _cli(argv_of('part', DETAIL) + flags + ['--null', reps, '--regions', os.path.join(d, 'part_r.txt'),
                                            '--threshold', repr(cut), '--targets', targets])
    ivs = {n: [] for n in names}
    for line in _lines(targets)[2:]:
        f = line.split('\t')
        ivs[f[0]].append((float(f[1]), float(f[2])))
    return cut, ivs


def _compare(d, names, ivs, maxima):
    """Every file of the targeted run against the full run's under the contract of DESIGN.md §3.13."""
    ref = []
    for n in names:
        main = _lines(os.path.join(d, 'full', 'out', n))[1:]
        keep = _kept(main, ivs[n])
        for kind in ('out', 'support', 'pvalues'):
            _check_subset(os.path.join(d, 'full', kind, n), os.path.join(d, 'part', kind, n), keep)
        _check_refine(os.path.join(d, 'full', 'refine', n), os.path.join(d, 'part', 'refine', n), keep)
        got = _lines(os.path.join(d, 'part_r.txt'))
        ref += _expected_regions(main, keep, n, float(got[0].split()[3]), float(got[0].split()[-1]), maxima)
    got = _lines(os.path.join(d, 'part_r.txt'))
    assert got[:2] == _lines(os.path.join(d, 'full_r.txt'))[:2]
    assert got[2:] == ref and len(ref) > 1


@pytest.mark.parametrize('case', ['one_input', 'inputList'])
def test_targeted_run_is_the_full_run_at_the_kept_rows(case, tmp_path):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    reps = genome_data.make_replicates(d, n_reps=4, n_sites=80)
    one = case == 'one_input'
    names = [os.path.basename(p) for p in (paths[:1] if one else paths)]

    def argv_of(tag, kinds):
        out = {}
        for k in ['out'] + kinds:
            out[k] = os.path.join(d, tag, k)
            os.makedirs(out[k])
        argv = ['-i', paths[0] if one else lst, '--spect', genome_data.SPECT] + ([] if one else ['--inputList'])
        for k, v in out.items():
            argv += [KINDS[k], os.path.join(v, names[0]) if one else v]
        return argv
    _, ivs = _run_pair(d, argv_of, names, reps, FLAGS)
    maxima = _null_maxima(paths[0], reps, ['-w', '40'])
    _compare(d, names, ivs, maxima)


@pytest.mark.parametrize('case', ['one_input', 'inputList'])
def test_torchrun_targeted_run_equals_one_gpu(case, tmp_path):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    reps = genome_data.make_replicates(d, n_reps=4, n_sites=80)
    one = case == 'one_input'
    name = os.path.basename(paths[0])
    with util.quiet():
        from ballermixplus_b200 import InputData
        p0 = InputData(paths[0]).position
    tfile = os.path.join(d, 'targets.txt')
    with open(tfile, 'w') as fh:
        fh.write(f'{name} {p0[50]} {p0[300]}\n{name} {p0[250]} {p0[420]}\n{name} {p0[600]} {p0[600]}\n')
        if not one:
            fh.write('chr3.txt 0 2e6\nchrX.txt 2e6 2.1e6\n')
    argv = {}
    for k in ('one', 'two'):
        for sub in ('out', 'p'):
            os.makedirs(os.path.join(d, k, sub))
        io = (['-i', paths[0], '-o', os.path.join(d, k, 'out', name), '--pvalues', os.path.join(d, k, 'p', name)]
              if one else ['--inputList', '-i', lst, '-o', os.path.join(d, k, 'out'), '--pvalues',
                           os.path.join(d, k, 'p')])
        argv[k] = io + ['--spect', genome_data.SPECT, '-w', '40', '--null', reps, '--regions',
                        os.path.join(d, f'{k}_r.txt'), '--threshold', '2.0', '--targets', tfile]
    _cli(argv['one'])
    out = _torchrun(argv['two'], 29575 if one else 29577)
    for n in ([name] if one else [os.path.basename(p) for p in paths]):
        for sub in ('out', 'p'):
            ref = _bytes(os.path.join(d, 'one', sub, n))
            assert _bytes(os.path.join(d, 'two', sub, n)) == ref
    assert len(_lines(os.path.join(d, 'one', 'out', name))) > 100
    assert _bytes(os.path.join(d, 'two_r.txt')) == _bytes(os.path.join(d, 'one_r.txt'))
    assert out.count('Empirical null:') == 1 and out.count(f'--targets: {name}: ') == 1
