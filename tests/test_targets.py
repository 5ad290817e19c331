"""--targets on the CPU: the targets file and its refusals (before any input is read), the row selection of the four
planners against a brute-force loop, the whole host pipeline (one input and --inputList, with --support, --null,
--pvalues and --regions) with the C oracle standing in for the device scan, and the genome sharding of a targeted
run over gloo (world sizes 2 and 3)."""
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

import genome_data
import null_data
import surface_oracle
import util
from ballermixplus_b200 import cli, native, regions, scan, targets, windows
from ballermixplus_b200.inputs import InputData
from test_regions import OracleScan, brute_interval, brute_maxima, brute_p, brute_peak, brute_regions


def _write(path, text):
    with open(path, 'w') as fh:
        fh.write(text)
    return str(path)


def _bytes(path):
    with open(path, 'rb') as fh:
        return fh.read()


def _lines(path):
    with open(path) as fh:
        return fh.readlines()


class _Plan:
    """A plan stand-in with given numeric physPos values."""

    def __init__(self, pos):
        self.pos = np.asarray(pos, dtype=np.float64)

    def phys(self):
        return self.pos


# ---- the targets file ---------------------------------------------------------------------------------------
def test_a_regions_file_is_a_targets_file(tmp_path):
    line = '{}\t{}\t{}\t3\t{}\t1e-05\t7.5\t0.5\t100\t1000\t12\t{}\t{}\tNA\n'
    per_input = [[line.format('chr1.txt', 100, 300, 200, 90, 310), line.format('chr1.txt', 900, 950, 920, 880, 990)],
                 [line.format('chr2.txt', 5, 5, 5, 5, 5)]]
    path = str(tmp_path / 'r.txt')
    regions.write_regions(path, per_input, 4.5, '--threshold', 3.84)
    got = targets.read_targets(path, ['chr1.txt', 'chr2.txt', 'chr3.txt'])
    pos = [4, 5, 6, 99, 100, 300, 301, 899, 900, 950, 951]
    assert got.keep('chr1.txt', _Plan(pos)).tolist() == [p in (100, 300, 900, 950) for p in pos]
    assert got.keep('chr2.txt', _Plan(pos)).tolist() == [p == 5 for p in pos]
    assert not got.keep('chr3.txt', _Plan(pos)).any()


def test_comments_header_overlapping_and_unsorted_targets(tmp_path):
    path = _write(tmp_path / 't.txt', '# targets\n\ninput start end\n  a 50 60\n# a 0 1000\na 10 20.5\n'
                                      'a 15 30\na 55 55\nb -5 -1\n\na 40 40.25\n')
    got = targets.read_targets(path, ['a', 'b'])
    pos = np.array([9.99, 10, 12, 20.5, 25, 30, 30.01, 40, 40.25, 40.5, 49, 50, 55, 60, 61, -3])
    ref = [any(s <= p <= e for s, e in [(50, 60), (10, 20.5), (15, 30), (55, 55), (40, 40.25)]) for p in pos]
    assert got.keep('a', _Plan(pos)).tolist() == ref
    assert got.keep('b', _Plan(pos)).tolist() == [p == -3 for p in pos]
    # only the first non-comment line can be a header
    with pytest.raises(ValueError, match='line 2: .*not an input'):
        targets.read_targets(_write(tmp_path / 'h.txt', 'a 1 2\ninput 3 4\n'), ['a'])


class _Read(Exception):
    pass


@pytest.fixture
def no_input_reads(monkeypatch):
    """InputData that fails the test's way if it is ever constructed."""
    seen = []

    def fake(path, *a, **k):
        seen.append(path)
        raise _Read(path)
    monkeypatch.setattr(cli, 'InputData', fake)
    return seen


def _refused(argv, capsys):
    with pytest.raises(SystemExit) as exc:
        cli.main(argv)
    assert exc.value.code == 2
    return capsys.readouterr().err


BAD_FILES = [
    ('absent', None, 'cannot read'),
    ('dir', None, 'cannot read'),
    ('two fields', 'in.txt 5 9\nin.txt 5\n', 'line 2: expected "name start end"'),
    ('not a number', '# c\nin.txt 5 9\nin.txt 5 ten\n', "line 3: start and end must be finite numbers"),
    ('nan', 'in.txt nan 9\n', 'line 1: start and end must be finite'),
    ('inf', 'in.txt 1 inf\n', 'line 1: start and end must be finite'),
    ('start after end', 'input s e\nin.txt 9 5\n', 'line 2: start 9 is after end 5'),
    ('unknown name', 'in.txt 1 2\nin.tx 1 2\n', "line 2: 'in.tx' is not an input of this run (inputs: in.txt)"),
    ('empty', '# nothing\n\n', 'holds no target'),
    ('header only', 'input start_physPos end_physPos\n', 'holds no target'),
]


@pytest.mark.parametrize('case, text, message', BAD_FILES, ids=[c[0] for c in BAD_FILES])
def test_bad_targets_are_refused_before_any_input_is_read(case, text, message, tmp_path, no_input_reads, capsys):
    t = str(tmp_path / 't')
    if case == 'dir':
        os.makedirs(t)
    elif text is not None:
        _write(t, text)
    out = tmp_path / 'out'
    out.mkdir()
    argv = ['-i', str(tmp_path / 'in.txt'), '--spect', null_data.SPECT, '-o', str(out / 'o.txt'), '--targets', t]
    err = _refused(argv, capsys)
    assert message in err and (case in ('absent', 'dir') or f'--targets {t}' in err)
    assert no_input_reads == [] and os.listdir(out) == []


def test_targets_the_run_writes_and_helper_runs_are_refused(tmp_path, no_input_reads, capsys):
    t = _write(tmp_path / 't.txt', 'in.txt 1 2\n')
    base = ['-i', str(tmp_path / 'in.txt'), '--spect', null_data.SPECT, '--targets', t]
    for extra in (['-o', t], ['-o', str(tmp_path / 'o.txt'), '--support', t],
                  ['-o', str(tmp_path / 'o.txt'), '--regions', t, '--threshold', '3']):
        assert 'is a file this run writes' in _refused(base + extra, capsys)
    for helper in ('--getSpect', '--getConfig'):
        assert '--getSpect and --getConfig do not scan' in _refused(base + [helper], capsys)
    assert _lines(t) == ['in.txt 1 2\n'] and sorted(os.listdir(tmp_path)) == ['t.txt']
    # --inputList: names are the listed inputs' file names; an output of the list run is refused
    lst, paths = genome_data.make_genome(str(tmp_path / 'g'), chroms=genome_data.CHROMS[:2])
    out = tmp_path / 'g' / 'out'
    out.mkdir()
    base = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', str(out), '--targets']
    assert "'in.txt' is not an input of this run (inputs: chr1.txt, chr2.txt)" in _refused(base + [t], capsys)
    assert 'is a file this run writes' in _refused(base + [str(out / 'chr2.txt')], capsys)
    reg = str(tmp_path / 'g' / 'r.txt')
    assert 'is a file this run writes' in _refused(base + [reg, '--regions', reg, '--threshold', '3'], capsys)
    assert no_input_reads == [] and os.listdir(out) == []


# ---- row selection --------------------------------------------------------------------------------------------
def _noncentre_midpoints(data, w, s):
    """The --noCenter midpoints, restated from the reference's loop (v1:513-545)."""
    pos = data.position
    mid = int(np.floor(2 * float(pos[0]) / w) * (w / 2)) + s / 2
    out = []
    while mid <= pos[-1]:
        out.append(mid)
        mid += s
    return out


SELECTION_MODES = {
    'default': (dict(), None),
    'w': (dict(r=20), None),
    'fixWinSize': (dict(fixSize=True, r=200000, phys=True), None),
    'noCenter': (dict(fixSize=True, r=200000, s=20001, phys=True, noCenter=True), (200000, 20001)),
}


@pytest.mark.parametrize('mode', sorted(SELECTION_MODES))
def test_kept_rows_equal_brute_force(mode, tmp_path):
    kw, nc = SELECTION_MODES[mode]
    rng = np.random.default_rng(3)
    inp = null_data.write_input(str(tmp_path / 'in.txt'), 90, rng, span=3_000_000)
    with util.quiet():
        data = InputData(inp, phys=kw.get('phys', False))
        plan = windows.make_plan(data, **kw)
    if nc is None:
        pos = [float(v) for v in data.position]               # every site is a centre at -s 1
    else:
        pos = _noncentre_midpoints(data, *nc)
        assert any(p != int(p) for p in pos)                 # fractional midpoints
        assert np.any(plan.arrays()[3]) and not np.all(plan.arrays()[3])   # gap rows and scanned rows
    assert len(pos) == len(plan)
    for trial in range(20):
        ivs = []
        for _ in range(int(rng.integers(1, 6))):
            a, b = sorted(rng.choice(pos, 2))                # targets starting and ending exactly on a row
            if rng.random() < 0.5:
                a, b = a - rng.random() * 5e4, b + rng.random() * 5e4
            ivs.append((float(a), float(b)))
        text = ''.join(f'in.txt {a!r} {b!r}\n' for a, b in ivs) + 'other.txt 0 1e9\n'
        got = targets.read_targets(_write(tmp_path / 't.txt', text), ['in.txt', 'other.txt']).keep('in.txt', plan)
        ref = [any(a <= p <= b for a, b in ivs) for p in pos]
        assert got.tolist() == ref
    assert plan.phys().tolist() == pos


def test_take_keeps_the_text_of_every_row(tmp_path):
    inp = null_data.write_input(str(tmp_path / 'in.txt'), 60, np.random.default_rng(4))
    for kw in (dict(r=5), dict(fixSize=True, r=200000, s=20001, phys=True, noCenter=True)):
        with util.quiet():
            plan = windows.make_plan(InputData(inp, phys=kw.get('phys', False)), **kw)
        idx = np.flatnonzero(np.arange(len(plan)) % 3 != 1)
        sub = plan.take(idx)
        assert len(sub) == len(idx)
        assert sub.f0 == [plan.f0[j] for j in idx] and sub.f1 == [plan.f1[j] for j in idx]
        assert all(np.array_equal(a, b[idx]) for a, b in zip(sub.arrays(), plan.arrays()))
        assert np.array_equal(sub.phys(), plan.phys()[idx])


# ---- the host pipeline, the C oracle standing in for the device scan ------------------------------------------
class ProfileOracleScan(OracleScan):
    """OracleScan with the profiles of ``--support`` (from the literal surface); every input it loads is recorded
    in ``LOADS`` by its number of sites."""
    LOADS = []

    def __init__(self, data, neutral, sel, grids, device=0):
        ProfileOracleScan.LOADS.append(int(data.numSites))
        super().__init__(data, neutral, sel, grids, device)

    def run_profile(self, t, lo, hi):
        T, iA, ix, ia, ns = self.run(t, lo, hi)
        S, nsA = surface_oracle.problem_surface(self.problem, t, lo, hi)
        return T, iA, ix, ia, ns, S.max(axis=(2, 3)), S.max(axis=(1, 3)), S.max(axis=(1, 2)), nsA


@pytest.fixture
def oracle_scan(monkeypatch):
    monkeypatch.setattr(scan, 'DeviceScan', ProfileOracleScan)
    OracleScan.NULLS = []
    ProfileOracleScan.LOADS = []
    return OracleScan.NULLS


def _run(argv):
    with util.quiet():
        cli.main(argv)


def _kept(main_lines, ivs):
    """Brute force: rows of a full run's main file (header dropped) whose physPos text lies in a target."""
    return [any(a <= float(line.split('\t')[0]) <= b for a, b in ivs) for line in main_lines]


def _expected_regions(main_lines, keep, name, cut, q, maxima):
    """Region lines from the full run's main file with every row that is not kept taken as a gap row."""
    rows = [line.rstrip('\n').split('\t') for line in main_lines]
    T = [float(f[2]) for f in rows]
    gap = [f[3] == 'NA' or not k for f, k in zip(rows, keep)]
    out = []
    for f, l in brute_regions(T, gap, cut):
        p = brute_peak(T, f, l)
        lo, hi = brute_interval(T, gap, p, q)
        pv = 'NA' if maxima is None else f'{brute_p(T[p], maxima)}'
        out.append('\t'.join([name, rows[f][0], rows[l][0], str(l - f + 1)] + rows[p][:7] + [rows[lo][0], rows[hi][0],
                                                                                           pv]) + '\n')
    return out


def _check_subset(full, part, keep, header_lines=1):
    """``part`` = the header of ``full`` and its lines at the kept rows."""
    a, b = _lines(full), _lines(part)
    assert b == a[:header_lines] + [line for line, k in zip(a[header_lines:], keep) if k]


def _clear_of_edges(line, main_lines, keep):
    """True when a region line's rows and position interval keep off the first and last kept row of its target."""
    pos = [line_.split('\t')[0] for line_ in main_lines]
    f = line.split('\t')
    lo, hi = min(pos.index(f[1]), pos.index(f[11])), max(pos.index(f[2]), pos.index(f[12]))
    return lo > 0 and keep[lo - 1] and hi + 1 < len(keep) and keep[hi + 1]


def _check_regions(full_reg, part_reg, main_lines, keep, name, maxima, must_cut=True):
    full_lines = _lines(full_reg)
    got = _lines(part_reg)
    assert got[:2] == full_lines[:2]
    cut, q = float(got[0].split()[3]), float(got[0].split()[-1])
    ref = _expected_regions(main_lines, keep, name, cut, q, maxima)
    assert got[2:] == ref and len(ref) > 0
    clear = [line for line in ref if _clear_of_edges(line, main_lines, keep)]
    assert all(line in full_lines for line in clear)
    if must_cut:
        assert any(line not in full_lines for line in ref)     # some region or interval was cut at an edge
    return clear


@pytest.mark.parametrize('mode', ['default', 'noCenter'])
def test_one_input_pipeline_with_oracle_scan(mode, tmp_path, oracle_scan, capsys):
    d = str(tmp_path)
    flags = {'default': ['-w', '15'],
             'noCenter': ['--fixWinSize', '--noCenter', '-w', '60000', '-s', '8000', '--usePhysPos']}[mode]
    inp = null_data.write_input(os.path.join(d, 'main.txt'), 160, np.random.default_rng(8), span=1_500_000)
    lst, _ = null_data.make_replicates(d, n_reps=3, n_sites=40, seed=7)
    base = ['-i', inp, '--spect', null_data.SPECT, '--null', lst] + flags

    def argv(tag, *extra):
        return base + ['-o', os.path.join(d, f'{tag}.txt'), '--support', os.path.join(d, f'{tag}_sup.txt'),
                       '--pvalues', os.path.join(d, f'{tag}_p.txt'), '--regions', os.path.join(d, f'{tag}_r.txt'),
                       '--supportDrop', '2.0'] + list(extra)
    _run(argv('full0', '--threshold', '1e9'))
    main_lines = _lines(os.path.join(d, 'full0.txt'))[1:]
    T = np.array([float(line.split('\t')[2]) for line in main_lines])
    cut = float(np.quantile(T[T > 0], 0.6))
    _run(argv('full', '--threshold', repr(cut)))
    full_reg = os.path.join(d, 'full_r.txt')
    (null_T, rep, n_rep) = oracle_scan[0]
    maxima = brute_maxima(null_T, rep, n_rep)
    pos = [float(line.split('\t')[0]) for line in main_lines]
    wide = (pos[len(pos) // 5], pos[4 * len(pos) // 5])
    cases = {
        # the full run's regions file itself, and a few wide overlapping, unsorted targets
        'regions': (full_reg, [tuple(float(v) for v in line.split('\t')[1:3]) for line in _lines(full_reg)[2:]]),
        'wide': (_write(os.path.join(d, 'wide_targets.txt'), f'main.txt {wide[1] - 1e5} {wide[1]}\nmain.txt {wide[0]} '
                        f'{wide[1] - 2e5}\nmain.txt {pos[2]} {pos[5]}\n'),
                 [(wide[1] - 1e5, wide[1]), (wide[0], wide[1] - 2e5), (pos[2], pos[5])]),
    }
    clear = 0
    for tag, (tfile, ivs) in cases.items():
        keep = _kept(main_lines, ivs)
        assert 0 < sum(keep) < len(keep)
        ProfileOracleScan.LOADS = []
        capsys.readouterr()
        cli.main(argv(tag, '--threshold', repr(cut), '--targets', tfile))
        assert f'--targets: main.txt: {sum(keep)} of {len(keep)} planned rows kept' in capsys.readouterr().out
        for suffix in ('.txt', '_sup.txt', '_p.txt'):
            _check_subset(os.path.join(d, 'full' + suffix), os.path.join(d, tag + suffix), keep)
        clear += len(_check_regions(full_reg, os.path.join(d, f'{tag}_r.txt'), main_lines, keep, 'main.txt', maxima,
                                    must_cut=tag == 'regions'))
        assert len(oracle_scan) == 2 + list(cases).index(tag) + 1         # the null is scanned in full every run
        assert np.array_equal(oracle_scan[-1][0], null_T)
    assert clear > 0
    if mode == 'noCenter':
        assert any('\tNA\t' in line for line in _lines(os.path.join(d, 'wide.txt')))


def test_input_list_pipeline_with_oracle_scan(tmp_path, oracle_scan, capsys):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    reps = genome_data.make_replicates(d, n_reps=3, n_sites=60)
    names = [os.path.basename(p) for p in paths]
    sizes = {n: c[1] for n, c in zip(names, genome_data.CHROMS)}
    for tag in ('full', 'part'):
        for k in ('out', 'sup', 'p'):
            os.makedirs(os.path.join(d, tag, k))

    def argv(tag, *extra):
        return ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-w', '30', '--null', reps] + \
            [a for k, o in (('-o', 'out'), ('--support', 'sup'), ('--pvalues', 'p'))
             for a in (k, os.path.join(d, tag, o))] + ['--regions', os.path.join(d, f'{tag}_r.txt')] + list(extra)
    _run(argv('full', '--threshold', '1e9'))
    main = {n: _lines(os.path.join(d, 'full', 'out', n))[1:] for n in names}
    T = np.concatenate([[float(line.split('\t')[2]) for line in v] for v in main.values()])
    cut = float(np.quantile(T[T > 0], 0.6))
    _run(argv('full', '--threshold', repr(cut)))
    (null_T, rep, n_rep) = oracle_scan[0]
    maxima = brute_maxima(null_T, rep, n_rep)
    # chr1: two overlapping targets and one exactly on rows; chr3: one; chr2: none; chrX: one that holds no row
    p1 = [float(line.split('\t')[0]) for line in main['chr1.txt']]
    p3 = [float(line.split('\t')[0]) for line in main['chr3.txt']]
    ivs = {'chr1.txt': [(p1[400], p1[650]), (p1[30] - 0.5, p1[300] + 0.5), (p1[250], p1[420])],
           'chr3.txt': [(p3[60], p3[200])], 'chr2.txt': [], 'chrX.txt': [(2.0e6, 2.1e6)]}
    text = '# targets\n' + ''.join(f'{n}\t{a!r}\t{b!r}\n' for n in ('chr3.txt', 'chrX.txt', 'chr1.txt')
                                   for a, b in ivs[n][::-1])
    tfile = _write(os.path.join(d, 'targets.txt'), text)
    ProfileOracleScan.LOADS = []
    capsys.readouterr()
    cli.main(argv('part', '--threshold', repr(cut), '--targets', tfile))
    console = capsys.readouterr().out
    assert sorted(ProfileOracleScan.LOADS) == sorted([sizes['chr1.txt'], sizes['chr3.txt']])
    keeps = {n: _kept(main[n], ivs[n]) for n in names}
    assert sum(keeps['chrX.txt']) == 0 and sum(keeps['chr2.txt']) == 0
    for n in names:
        assert f'--targets: {n}: {sum(keeps[n])} of {len(keeps[n])} planned rows kept' in console
        for k in ('out', 'sup', 'p'):
            _check_subset(os.path.join(d, 'full', k, n), os.path.join(d, 'part', k, n), keeps[n])
    total = sum(sum(k) for k in keeps.values())
    assert f'--targets: {total} of {sum(len(k) for k in keeps.values())} planned rows kept in 2 of 4 inputs' in console
    # the genome regions file: per input, the full rows with every row not kept taken as a gap row
    got = _lines(os.path.join(d, 'part_r.txt'))
    full_lines = _lines(os.path.join(d, 'full_r.txt'))
    assert got[:2] == full_lines[:2]
    ref = []
    for n in names:
        ref += _expected_regions(main[n], keeps[n], n, cut, float(got[0].split()[-1]), maxima)
    assert got[2:] == ref and len(ref) > 1
    assert any(line in full_lines for line in ref) and any(line not in full_lines for line in ref)


# ---- genome sharding of a targeted run over gloo ---------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, argv, out_dir):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), LOCAL_WORLD_SIZE=str(world),
                      MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    native.device_count = lambda: 0             # no CUDA device: every rank scans with the oracle, gathers on gloo
    scan.DeviceScan = ProfileOracleScan
    ProfileOracleScan.LOADS = []
    with util.quiet():
        cli.main(argv)
    with open(os.path.join(out_dir, f'loads{rank}.txt'), 'w') as fh:
        fh.write(' '.join(str(v) for v in ProfileOracleScan.LOADS))


@pytest.mark.parametrize('world', [2, 3])
def test_sharded_targeted_run_equals_one_process(world, tmp_path, oracle_scan):
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    with util.quiet():
        pos = InputData(paths[2]).position                       # chr3.txt
    # one kept centre, in chr3 (the chr1 target holds no row): every rank but one has no centre
    tfile = _write(os.path.join(d, 't.txt'), f'chr3.txt {pos[100] - 0.5} {pos[100]}\nchr1.txt 0 0\n')

    def argv(tag):
        for k in ('out', 'p'):
            os.makedirs(os.path.join(d, tag, k))
        return ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-w', '30', '-o', os.path.join(d, tag, 'out'),
                '--regions', os.path.join(d, f'{tag}_r.txt'), '--threshold', '0.5', '--targets', tfile]
    _run(argv('one'))
    mp.spawn(_worker, args=(world, _free_port(), argv('many'), d), nprocs=world, join=True)
    for p in paths:
        name = os.path.basename(p)
        assert _bytes(os.path.join(d, 'many', 'out', name)) == _bytes(os.path.join(d, 'one', 'out', name))
    assert len(_lines(os.path.join(d, 'one', 'out', 'chr3.txt'))) == 2
    assert _bytes(os.path.join(d, 'many_r.txt')) == _bytes(os.path.join(d, 'one_r.txt'))
    loads = [_lines(os.path.join(d, f'loads{r}.txt')) for r in range(world)]
    assert sorted(v for r in loads for v in (r[0].split() if r else [])) == ['260']    # chr3 only, on one rank
