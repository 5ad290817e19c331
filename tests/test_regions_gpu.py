"""--regions on the GPU (run with -m gpu on a B200): the regions file equals the regions an independent parser takes
from the main file's text, the main file does not change with --regions, the --inputList file is the one-input
runs' files laid end to end with the null's cut and region p-values, and torchrun writes the one-GPU run's bytes."""
import os

import numpy as np
import pytest

import genome_data
import util
from test_genome_list_gpu import _torchrun
from test_regions import brute_maxima, parse_regions, read_regions

pytestmark = pytest.mark.gpu

D = os.path.join(util.GOLD, 'data')
EX2 = ['-i', os.path.join(D, 'Example2_balancing_10MYA_DAF.txt'), '--spect',
       os.path.join(D, 'HC_CEU_Neut_DAF_spect_for_B2.txt')]
MODES = {'default': [], 'noCenter': ['--usePhysPos', '--fixWinSize', '-w', '300', '--noCenter', '-s', '150']}


def _cli(argv):
    from ballermixplus_b200.cli import main
    with util.quiet():
        main(argv)


def _bytes(path):
    with open(path, 'rb') as fh:
        return fh.read()


def _median_positive_clr(main_path):
    with open(main_path) as fh:
        T = np.array([float(line.split('\t')[2]) for line in fh.readlines()[1:]])
    return float(np.median(T[T > 0]))


@pytest.mark.parametrize('mode', sorted(MODES))
def test_one_input_regions_equal_the_main_file_parsed(mode, tmp_path):
    plain, out, reg = (str(tmp_path / k) for k in ('plain.txt', 'o.txt', 'r.txt'))
    _cli(EX2 + MODES[mode] + ['-o', plain])
    cut = _median_positive_clr(plain)
    _cli(EX2 + MODES[mode] + ['-o', out, '--regions', reg, '--threshold', repr(cut)])
    assert _bytes(out) == _bytes(plain)
    got_cut, source, q, lines = read_regions(reg)
    assert (got_cut, source) == (cut, '--threshold')
    assert lines == parse_regions(out, 'Example2_balancing_10MYA_DAF.txt', cut, q)
    assert len(lines) > 1
    if mode == 'noCenter':
        with open(out) as fh:
            assert any('\tNA\t' in line for line in fh)


def _genome(d):
    lst, paths = genome_data.make_genome(d)
    reps = genome_data.make_replicates(d, n_reps=8, n_sites=60)
    return lst, paths, reps


def _null_maxima(path, reps, flags):
    """Per-replicate maxima of ``Scan(...).null`` for one input; the replicate of every null row from its NullSetup."""
    from ballermixplus_b200 import null
    from ballermixplus_b200.scan import Scan
    opt, data, neutral, grid, sel = util.host_objects(['-i', path, '--spect', genome_data.SPECT] + flags)
    kw = dict(r=opt.w, s=opt.step, phys=opt.phys, fixSize=opt.size, noCenter=opt.noCenter)
    d = os.path.dirname(reps)
    with util.quiet():
        setup = null.NullSetup(reps, data, neutral, sel, grid, **kw)
        run = Scan(data, neutral, sel, grid, os.path.join(d, 'm.txt'), null=reps, pvalues=os.path.join(d, 'p.txt'),
                   **kw)
    return brute_maxima(run.null, setup.rep, setup.n_replicates)


def test_input_list_regions_with_null(tmp_path, capsys):
    d = str(tmp_path)
    lst, paths, reps = _genome(d)
    flags = ['-w', '40']
    for k in ('out', 'p', 'single', 'single_p'):
        os.makedirs(os.path.join(d, k))
    reg = os.path.join(d, 'genome_regions.txt')
    from ballermixplus_b200.cli import main
    main(['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', os.path.join(d, 'out'), '--pvalues',
          os.path.join(d, 'p'), '--null', reps, '--regions', reg] + flags)
    console = capsys.readouterr().out
    maxima = _null_maxima(paths[0], reps, flags)
    cut, source, q, lines = read_regions(reg)
    assert cut == float(np.quantile(maxima, 0.95)) and source == f'0.95 quantile of {len(maxima)} replicate maxima'
    assert f'per-replicate max CLR: 0.95: {cut:.6g},' in console
    ref = []
    for p in paths:
        name = os.path.basename(p)
        ref += parse_regions(os.path.join(d, 'out', name), name, cut, q, maxima)
    assert lines == ref and len(ref) > 1
    cat = []
    for p in paths:
        name = os.path.basename(p)
        one = os.path.join(d, 'single_' + name)
        _cli(['-i', p, '--spect', genome_data.SPECT, '-o', os.path.join(d, 'single', name), '--pvalues',
              os.path.join(d, 'single_p', name), '--null', reps, '--regions', one] + flags)
        with open(one) as fh:
            got = fh.readlines()
        cat += got if not cat else got[2:]
    assert _bytes(reg) == ''.join(cat).encode()


@pytest.mark.parametrize('case', ['one_input', 'inputList'])
def test_torchrun_regions_equal_one_gpu(case, tmp_path):
    d = str(tmp_path)
    if case == 'one_input':
        base = EX2 + ['--threshold', '8.0']
        argv = {k: base + ['-o', os.path.join(d, f'{k}.txt'), '--regions', os.path.join(d, f'{k}_regions.txt')]
                for k in ('one', 'two')}
    else:
        lst, _, reps = _genome(d)
        argv = {}
        for k in ('one', 'two'):
            for sub in ('out', 'p'):
                os.makedirs(os.path.join(d, k, sub))
            argv[k] = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-w', '40', '-o',
                       os.path.join(d, k, 'out'), '--null', reps, '--pvalues', os.path.join(d, k, 'p'), '--regions',
                       os.path.join(d, f'{k}_regions.txt')]
    _cli(argv['one'])
    out = _torchrun(argv['two'], 29567 if case == 'one_input' else 29569)
    ref = _bytes(os.path.join(d, 'one_regions.txt'))
    assert _bytes(os.path.join(d, 'two_regions.txt')) == ref and ref.count(b'\n') > 3
    assert out.count('regions: ') == 1
