"""--inputList on the GPU (run with -m gpu on a B200): every file a list run writes is byte-identical to the file a
one-input run with the same flags writes, plain and with --support, --refine and --null/--pvalues, on one GPU and
under torchrun (two ranks sharing the test box's GPU, so the gather runs over gloo)."""
import os
import subprocess
import sys

import pytest

import genome_data
import util

pytestmark = pytest.mark.gpu

NO_CENTER = ['--usePhysPos', '--fixWinSize', '--noCenter', '-w', '200000', '-s', '50000']


def _cli(argv):
    from ballermixplus_b200.cli import main
    with util.quiet():
        main(argv)


def _dirs(root, names):
    out = {}
    for n in names:
        out[n] = os.path.join(root, n)
        os.makedirs(out[n])
    return out


def _same_files(list_dirs, single_dirs, paths):
    """Every file of the list run equals the one-input run's file, byte for byte."""
    for kind, d in list_dirs.items():
        for p in paths:
            name = os.path.basename(p)
            with open(os.path.join(d, name), 'rb') as a, open(os.path.join(single_dirs[kind], name), 'rb') as b:
                got, ref = a.read(), b.read()
            assert got == ref, f'{kind}/{name} differs from the one-input run'
            assert got.count(b'\n') > 1


def _single_runs(paths, flags, dirs):
    for p in paths:
        name = os.path.basename(p)
        argv = ['-i', p, '--spect', genome_data.SPECT, '-o', os.path.join(dirs['out'], name)] + flags
        for kind in ('support', 'refine', 'pvalues'):
            if kind in dirs:
                argv += [f'--{kind}', os.path.join(dirs[kind], name)]
        _cli(argv)


def _list_argv(lst, dirs, flags):
    argv = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', dirs['out']] + flags
    for kind in ('support', 'refine', 'pvalues'):
        if kind in dirs:
            argv += [f'--{kind}', dirs[kind]]
    return argv


def _min_counts(paths):
    from ballermixplus_b200 import InputData
    with util.quiet():
        return {int(InputData(p).minCount) for p in paths}


@pytest.mark.parametrize('mode', ['default', 'noCenter'])
@pytest.mark.parametrize('extras', ['plain', 'support_refine_null'])
def test_list_run_equals_single_input_runs(mode, extras, tmp_path):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    assert len(_min_counts(paths)) >= 2                     # one input derives a different minCount
    flags = NO_CENTER if mode == 'noCenter' else ['-w', '40']
    kinds = ['out']
    if extras != 'plain':
        flags = flags + ['--null', genome_data.make_replicates(d), '--supportDrop', '2.5', '--refineSteps', '2']
        kinds += ['support', 'refine', 'pvalues']
    one, many = _dirs(os.path.join(d, 'single'), kinds), _dirs(os.path.join(d, 'list'), kinds)
    _single_runs(paths, flags, one)
    _cli(_list_argv(lst, many, flags))
    _same_files(many, one, paths)
    if mode == 'noCenter':                                  # the gap rows are there
        with open(os.path.join(many['out'], 'chr1.txt')) as fh:
            assert any('\tNA\t' in line for line in fh)


def _torchrun(argv, port):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(port), '-m', 'ballermixplus_b200'] + argv
    res = subprocess.run(cmd, cwd=util.ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    return res.stdout


@pytest.mark.parametrize('mode', ['default', 'noCenter'])
def test_list_run_under_torchrun(mode, tmp_path):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    flags = (NO_CENTER if mode == 'noCenter' else ['-w', '40']) + ['--null', genome_data.make_replicates(d)]
    one, many = (_dirs(os.path.join(d, k), ['out', 'pvalues']) for k in ('single', 'list'))
    _single_runs(paths, flags, one)
    out = _torchrun(_list_argv(lst, many, flags), 29561 if mode == 'default' else 29563)
    _same_files(many, one, paths)
    assert out.count('Empirical null:') == 1                # the replicates are scanned once, for every input
    assert 'on 2 ranks' in out
    for p in paths:
        assert f'{os.path.basename(p)}: ' in out


def test_torchrun_refuses_support_with_a_list(tmp_path):
    d = str(tmp_path)
    lst, _ = genome_data.make_genome(d, chroms=genome_data.CHROMS[:1])
    dirs = _dirs(d, ['out', 'support'])
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29565', '-m', 'ballermixplus_b200'] + _list_argv(lst, dirs, [])
    res = subprocess.run(cmd, cwd=util.ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode != 0
    assert '--support runs on one GPU; launch without torchrun' in res.stderr
    assert os.listdir(dirs['out']) == []
