"""--balPos on the CPU: grid validation and early refusals, the half of every alpha in set order, the line format
(all-zero halves, --noCenter gap rows, --targets subsets), the --inputList directory rules, the wider packing of
the sharded rows, and the host pipeline on one process and sharded over gloo with the C oracle as the scan."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import genome_data
import null_data
import surface_oracle
import util
from ballermixplus_b200 import balpos, cli, native, scan, sharding
from ballermixplus_b200.grids import Grids
from ballermixplus_b200.problem import GridOrder
from test_regions import OracleScan


# ---- grid, refusals --------------------------------------------------------------------------------------------
def test_half_of_a_follows_the_set_order():
    order = GridOrder(Grids(None, None, False, False, None, None))
    half = balpos.half_of_a(order.a)
    assert half.dtype == np.int8 and len(half) == len(order.a)
    assert half.tolist() == [0 if float(a) >= 1 else 1 for a in order.a]
    assert order.a != sorted(order.a)                        # set order, not numeric order
    assert sorted(float(a) for a, h in zip(order.a, half) if h == 1) == [0.001, 0.01, 0.05, 0.1, 0.2, 0.5, 0.8]
    balpos.check_grid(order.a)


@pytest.mark.parametrize('flags', [['--fixAlpha', '2'], ['--fixAlpha', '0.5'], ['--findBal'], ['--findPos']])
def test_grid_with_an_empty_half_is_refused(flags):
    g = Grids(None, dict(zip(flags[::2], flags[1::2])).get('--fixAlpha'), '--findBal' in flags, '--findPos' in flags,
              None, None)
    with pytest.raises(ValueError, match='both sides of 1'):
        balpos.check_grid(g.abeta)


class _Read(Exception):
    pass


@pytest.fixture
def no_input_reads(monkeypatch):
    def fake(path, *a, **k):
        raise _Read(path)
    monkeypatch.setattr(cli, 'InputData', fake)


def _refused(argv, capsys):
    with pytest.raises(SystemExit) as exc:
        cli.main(argv)
    assert exc.value.code == 2
    return capsys.readouterr().err


def test_refusals_come_before_any_input_is_read(tmp_path, capsys, no_input_reads):
    inp = str(tmp_path / 'in.txt')
    base = ['-i', inp, '--spect', null_data.SPECT, '-o', str(tmp_path / 'o.txt')]
    bp = ['--balPos', str(tmp_path / 'bp.txt')]
    for extra in (['--fixAlpha', '3'], ['--findBal'], ['--findPos']):
        assert 'both sides of 1' in _refused(base + bp + extra, capsys)
    assert '--getSpect' in _refused(base + bp + ['--getSpect'], capsys)
    assert '--getSpect' in _refused(base + bp + ['--getConfig'], capsys)
    for clash in (inp, str(tmp_path / 'o.txt'), null_data.SPECT):
        assert 'reads or writes' in _refused(base + ['--balPos', clash], capsys)
    assert 'reads or writes' in _refused(base + bp + ['--support', str(tmp_path / 'bp.txt')], capsys)
    with pytest.raises(_Read):                               # a good --balPos gets as far as reading the input
        cli.main(base + bp)


def test_input_list_directory_rules(tmp_path, capsys, no_input_reads):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    os.makedirs(os.path.join(d, 'out'))
    os.makedirs(os.path.join(d, 'bp'))
    base = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', os.path.join(d, 'out')]
    assert 'not an existing directory' in _refused(base + ['--balPos', os.path.join(d, 'nope')], capsys)
    assert 'same directory' in _refused(base + ['--balPos', os.path.join(d, 'out')], capsys)
    assert 'overwrite an input' in _refused(base + ['--balPos', os.path.dirname(paths[0])], capsys)
    files = scan.list_outputs(paths, out=os.path.join(d, 'out'), balpos=os.path.join(d, 'bp'))
    assert files['balpos'] == [os.path.join(d, 'bp', os.path.basename(p)) for p in paths]


# ---- line format -----------------------------------------------------------------------------------------------
class _Plan:
    def __init__(self, f0, f1, gap):
        self.f0, self.f1, self.gap = f0, f1, np.asarray(gap)

    def __len__(self):
        return len(self.f0)


def _rows(T, iA, ix, ia, ns):
    return (np.asarray(T, np.float64), *(np.asarray(v, np.int32) for v in (iA, ix, ia, ns)))


def test_lines_print_as_the_main_file_prints():
    order = GridOrder(Grids(None, None, False, False, '100,300,100', None))
    plan = _Plan(['10', '20\t2e-05\t0\tNA\tNA\tNA\t0\n', '30'], ['1e-05', '', '3e-05'], [False, True, False])
    bal = _rows([4.5, 0, 0.0], [1, -1, -1], [2, -1, -1], [order.a.index(5), -1, -1], [17, 0, 0])
    pos = _rows([0.0, 0, 2.25], [-1, -1, 0], [-1, -1, 0], [-1, -1, order.a.index(0.1)], [0, 0, 9])
    lines = balpos.format_balpos(plan, order, bal, pos)
    x = order.x
    assert lines[0] == f'10\t1e-05\t4.5\t{x[2]}\t5\t{order.A[1]}\t17' + '\t0.0' * 5 + '\n'      # the all-zero row
    assert lines[1] == '20\t2e-05\t0\tNA\tNA\tNA\t0\t0\tNA\tNA\tNA\t0\n'
    assert lines[2] == f'30\t3e-05' + '\t0.0' * 5 + f'\t2.25\t{x[0]}\t0.1\t{order.A[0]}\t9\n'
    assert balpos.BALPOS_HEADER.rstrip('\n').split('\t')[2:7] == ['CLR_bal', 'x_bal', 's_bal', 'A_bal', 'nSites_bal']


def test_kept_halves_takes_the_targets_rows():
    h = (_rows([1, 2, 3], [0, 1, 2], [0, 0, 0], [1, 1, 1], [5, 6, 7]),) * 2
    keep = np.array([True, False, True])
    got = scan.kept_halves(keep, h)
    assert [c.tolist() for c in got[0]] == [[1, 3], [0, 2], [0, 0], [1, 1], [5, 7]]
    assert scan.kept_halves(None, h) is h and scan.kept_halves(keep, None) is None


# ---- packing of the sharded rows -------------------------------------------------------------------------------
def test_split_pack_unpack_roundtrip():
    rng = np.random.default_rng(1)
    for n in (0, 5):
        rows = []
        for _ in range(3):
            rows.append(torch.tensor((rng.normal(size=n) * 1e3).tolist(), dtype=torch.float64))
            rows += [torch.tensor(rng.integers(-1, 900, n).tolist(), dtype=torch.int32) for _ in range(4)]
        packed = sharding.pack_split_rows(rows, torch)
        assert packed.shape == (n, 18) and packed.dtype == torch.int32
        assert torch.equal(packed[:, :6], sharding.pack_rows(*rows[:5], torch))      # the plain row first
        back = sharding.unpack_split_rows(packed, torch)
        assert len(back) == 15 and all(torch.equal(a, b) for a, b in zip(back, rows))


# ---- host pipeline with the C oracle as the scan ---------------------------------------------------------------
class SplitOracleScan(OracleScan):
    """OracleScan with ``run_split``: the halves by the reference's rule on the oracle surface."""
    class scanner:                              # the one-input torchrun path reads the handle's device
        device = 0

    def run_split(self, t, lo, hi):
        from test_support_gpu import _rows_from_surface
        rows = self.run(t, lo, hi)
        S, nsA = surface_oracle.problem_surface(self.problem, t, lo, hi)
        half = balpos.half_of_a(self.order.a)[None, None, None, :]
        halves = tuple(_rows_from_surface(np.where(half == h, S, -np.inf), nsA) for h in (0, 1))
        return (rows, *halves)

    def run_profile(self, t, lo, hi):
        T, iA, ix, ia, ns = self.run(t, lo, hi)
        S, nsA = surface_oracle.problem_surface(self.problem, t, lo, hi)
        return T, iA, ix, ia, ns, S.max(axis=(2, 3)), S.max(axis=(1, 3)), S.max(axis=(1, 2)), nsA


def _lines(p):
    with open(p) as fh:
        return fh.readlines()


def _check_file(bp, main):
    b, m = _lines(bp), _lines(main)
    assert len(b) == len(m) and b[0] == balpos.BALPOS_HEADER
    for lb, lm in zip(b[1:], m[1:]):
        fb, fm = lb.rstrip('\n').split('\t'), lm.rstrip('\n').split('\t')
        assert fb[:2] == fm[:2]
        if fm[3] == 'NA':
            assert fb[2:] == ['0', 'NA', 'NA', 'NA', '0'] * 2
        else:
            assert float(fm[2]) == max(float(fb[2]), float(fb[7]))
    return b


@pytest.mark.parametrize('mode', ['default', 'noCenter'])
def test_one_input_pipeline(mode, tmp_path, monkeypatch):
    monkeypatch.setattr(scan, 'DeviceScan', SplitOracleScan)
    d = str(tmp_path)
    flags = {'default': ['-w', '15'],
             'noCenter': ['--fixWinSize', '--noCenter', '-w', '60000', '-s', '8000', '--usePhysPos']}[mode]
    inp = null_data.write_input(os.path.join(d, 'main.txt'), 120, np.random.default_rng(8), span=1_500_000)
    base = ['-i', inp, '--spect', null_data.SPECT] + flags
    with util.quiet():
        cli.main(base + ['-o', os.path.join(d, 'plain.txt')])
        cli.main(base + ['-o', os.path.join(d, 'main.txt.out'), '--balPos', os.path.join(d, 'bp.txt')])
        cli.main(base + ['-o', os.path.join(d, 'sup.out'), '--support', os.path.join(d, 'sup.txt'), '--balPos',
                         os.path.join(d, 'bp_sup.txt')])
    assert _lines(os.path.join(d, 'plain.txt')) == _lines(os.path.join(d, 'main.txt.out'))
    b = _check_file(os.path.join(d, 'bp.txt'), os.path.join(d, 'plain.txt'))
    assert _lines(os.path.join(d, 'bp_sup.txt')) == b
    pos = [float(line.split('\t')[0]) for line in b[1:]]
    tfile = os.path.join(d, 't.txt')
    with open(tfile, 'w') as fh:
        fh.write(f'main.txt {pos[10]} {pos[40]}\n')
    with util.quiet():
        cli.main(base + ['-o', os.path.join(d, 'part.out'), '--balPos', os.path.join(d, 'part.txt'), '--targets', tfile])
    assert _lines(os.path.join(d, 'part.txt')) == b[:1] + b[11:42]
    if mode == 'noCenter':
        assert any('\tNA\t' in line for line in b)
    else:
        assert any(float(line.split('\t')[2]) > 0 for line in b[1:])


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, argvs):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), LOCAL_WORLD_SIZE=str(world),
                      MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    native.device_count = lambda: 0             # no CUDA device: every rank scans with the oracle, gathers on gloo
    scan.DeviceScan = SplitOracleScan
    with util.quiet():
        for argv in argvs:
            cli.main(argv)


@pytest.mark.parametrize('world', [2, 3])
def test_sharded_runs_equal_one_process(world, tmp_path, monkeypatch):
    monkeypatch.setattr(scan, 'DeviceScan', SplitOracleScan)
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    with util.quiet():
        n_pos = len(cli.InputData(paths[2]).position)
    tfile = os.path.join(d, 't.txt')
    with util.quiet():
        pos = cli.InputData(paths[2]).position
    with open(tfile, 'w') as fh:                 # one kept centre: every rank but one has no centre
        fh.write(f'chr3.txt {pos[n_pos // 2] - 0.5} {pos[n_pos // 2]}\nchr1.txt 0 0\n')

    def argvs(tag):
        for k in ('out', 'bp', 'tout', 'tbp'):
            os.makedirs(os.path.join(d, tag, k))
        flags = ['--spect', genome_data.SPECT, '-w', '30']
        return [['--inputList', '-i', lst, '-o', os.path.join(d, tag, 'out'), '--balPos', os.path.join(d, tag, 'bp')]
                + flags,
                ['--inputList', '-i', lst, '-o', os.path.join(d, tag, 'tout'), '--balPos', os.path.join(d, tag, 'tbp'),
                 '--targets', tfile] + flags,
                ['-i', paths[0], '-o', os.path.join(d, tag, 'one.txt'), '--balPos', os.path.join(d, tag, 'one_bp.txt')]
                + flags]
    with util.quiet():
        for argv in argvs('one'):
            cli.main(argv)
    mp.spawn(_worker, args=(world, _free_port(), argvs('many')), nprocs=world, join=True)
    for p in paths:
        n = os.path.basename(p)
        for sub in ('out', 'bp', 'tout', 'tbp'):
            assert _lines(os.path.join(d, 'many', sub, n)) == _lines(os.path.join(d, 'one', sub, n))
        _check_file(os.path.join(d, 'one', 'bp', n), os.path.join(d, 'one', 'out', n))
    assert len(_lines(os.path.join(d, 'one', 'tbp', 'chr3.txt'))) == 2
    for f in ('one.txt', 'one_bp.txt'):
        assert _lines(os.path.join(d, 'many', f)) == _lines(os.path.join(d, 'one', f))
