"""--regions / --threshold on the CPU: regions, peaks, position intervals and region p-values against brute-force
loops, the null-derived cut against the printed quantile, early refusals of the command line, and the whole host
pipeline (one input and --inputList, with and without --null) with the C oracle standing in for the device scan."""
import os
import re

import numpy as np
import pytest

import genome_data
import null_data
import util
from ballermixplus_b200 import cli, null, regions, scan
from ballermixplus_b200.problem import build_problem
from ballermixplus_b200.support import DEFAULT_DROP


# ---- brute-force restatements --------------------------------------------------------------------------------
def brute_regions(T, gap, cut):
    out, j, n = [], 0, len(T)
    while j < n:
        if not gap[j] and T[j] >= cut:
            k = j
            while k + 1 < n and not gap[k + 1] and T[k + 1] >= cut:
                k += 1
            out.append((j, k))
            j = k + 1
        else:
            j += 1
    return out


def brute_peak(T, f, l):
    best = f
    for j in range(f + 1, l + 1):
        if T[j] > T[best]:
            best = j
    return best


def brute_interval(T, gap, p, q):
    level = T[p] - q
    lo = hi = p
    while lo > 0 and not gap[lo - 1] and T[lo - 1] >= level:
        lo -= 1
    while hi < len(T) - 1 and not gap[hi + 1] and T[hi + 1] >= level:
        hi += 1
    return lo, hi


def brute_maxima(null_T, rep, n_replicates):
    best = {}
    for v, r in zip(null_T, rep):
        if v == v:
            best[int(r)] = max(best.get(int(r), -np.inf), float(v))
    return [best[r] for r in range(n_replicates) if r in best]


def brute_p(T_peak, maxima):
    return (1 + sum(1 for m in maxima if m >= T_peak)) / (1 + len(maxima))


def _rows(rng, n):
    """Rows with ties and plateaus (a few discrete levels), NaN, gap rows and continuous values."""
    levels = np.array([0.0, 0.5, 1.0, 2.0, 3.0, 5.0, 8.0, np.nan])
    T = np.where(rng.random(n) < 0.6, rng.choice(levels, n), rng.exponential(3.0, n))
    gap = rng.random(n) < 0.05
    if n > 2 and rng.random() < 0.5:                 # runs touching both ends
        T[:2], T[-2:], gap[:2], gap[-2:] = 9.0, 9.0, False, False
    return T, gap


# ---- regions, peaks and intervals -----------------------------------------------------------------------------
@pytest.mark.parametrize('block', [64, 5, 1])
def test_regions_peaks_and_intervals_equal_brute_force(block, monkeypatch):
    monkeypatch.setattr(regions, '_BLOCK', block)
    rng = np.random.default_rng(17)
    n_regions = 0
    for n in [1, 2, 3, 63, 64, 65, 129, 500, 3000] * 4:
        T, gap = _rows(rng, n)
        finite = T[np.isfinite(T) & ~gap]
        cuts = [2.0, 0.7] + ([float(rng.choice(finite))] if len(finite) and finite.max() > 0 else [])
        for cut in cuts:                               # 2.0 and the drawn one: a cut equal to rows' CLRs
            if not cut > 0:
                continue
            first, last = regions.call_regions(T, gap, cut)
            ref = brute_regions(T, gap, cut)
            assert list(zip(first.tolist(), last.tolist())) == ref
            peak = regions.peaks(T, first, last)
            assert peak.tolist() == [brute_peak(T, f, l) for f, l in ref]
            for q in (0.0, 1.5, DEFAULT_DROP, 1e9):
                lo, hi = regions.position_interval(T, gap, peak, q)
                assert list(zip(lo.tolist(), hi.tolist())) == [brute_interval(T, gap, p, q) for p in peak.tolist()]
            n_regions += len(ref)
    assert n_regions > 500


def test_interval_crosses_the_region_and_stops_at_a_gap_row():
    T = np.array([0.0, 1.0, 2.0, 5.0, 2.0, 1.0, 0.0])
    gap = np.zeros(7, bool)
    first, last = regions.call_regions(T, gap, 4.0)
    assert (first.tolist(), last.tolist()) == ([3], [3])
    peak = regions.peaks(T, first, last)
    assert [v.tolist() for v in regions.position_interval(T, gap, peak, 3.5)] == [[2], [4]]   # past the region
    assert [v.tolist() for v in regions.position_interval(T, gap, peak, 10.0)] == [[0], [6]]
    gap[1] = True
    assert [v.tolist() for v in regions.position_interval(T, gap, peak, 10.0)] == [[2], [6]]
    T[5] = np.nan
    assert [v.tolist() for v in regions.position_interval(T, gap, peak, 10.0)] == [[2], [4]]
    assert [v.tolist() for v in regions.position_interval(T, gap, peak, 0.0)] == [[3], [3]]


def test_all_zero_rows_print_zero_and_empty_input():
    assert regions.row_clr([5.0, 7.0, np.nan], [0, -1, 2]).tolist()[:2] == [5.0, 0.0]
    first, last = regions.call_regions(np.zeros(0), np.zeros(0, bool), 1.0)
    assert len(first) == len(last) == len(regions.peaks(np.zeros(0), first, last)) == 0


@pytest.mark.parametrize('bad', ['0', '-1', 'nan', 'inf', '-inf'])
def test_threshold_must_be_finite_and_positive(bad):
    with pytest.raises(ValueError):
        regions.check_threshold(bad)
    assert regions.check_threshold('2.5') == 2.5


# ---- region p-values and the null's cut -------------------------------------------------------------------------
def test_region_pvalues_and_cut_equal_brute_force():
    rng = np.random.default_rng(5)
    n_rep = 9
    rep = rng.integers(0, n_rep, 400)
    rep = rep[(rep != 3) & (rep != 7)]                   # replicate 3 has no row
    null_T = rng.exponential(2.0, len(rep))
    null_T[rng.random(len(rep)) < 0.1] = np.nan
    null_T = np.concatenate((null_T, [np.nan, np.nan]))  # replicate 7 has NaN rows only
    rep = np.concatenate((rep, [7, 7]))
    mx = null.replicate_maxima(null_T, rep, n_rep)
    ref = brute_maxima(null_T, rep, n_rep)
    assert mx.tolist() == ref and len(ref) == n_rep - 2
    peaks = np.concatenate((rng.choice(ref, 4), rng.exponential(3.0, 30), [0.0, 1e9]))
    assert null.pvalues(peaks, mx).tolist() == [brute_p(t, ref) for t in peaks]        # the region p-value
    cut, source = regions.cut_of(None, mx)
    assert cut == float(np.quantile(ref, 0.95)) and source == f'0.95 quantile of {len(ref)} replicate maxima'
    printed = re.search(r'per-replicate max CLR: 0\.95: (\S+),', null.summary(null_T, rep, n_rep)[2]).group(1)
    assert printed == f'{cut:.6g}'
    assert regions.cut_of(2.5, mx) == (2.5, '--threshold')


# ---- the command line refuses before any input is read -------------------------------------------------------
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


@pytest.mark.parametrize('extra, message', [
    (['--regions', 'R'], '--regions needs a cut'),
    (['--threshold', '3'], '--threshold needs --regions'),
    (['--regions', 'R', '--threshold', '0'], 'finite number > 0'),
    (['--regions', 'R', '--threshold', '-2'], 'finite number > 0'),
    (['--regions', 'R', '--threshold', 'nan'], 'finite number > 0'),
    (['--regions', 'R', '--threshold', 'inf'], 'finite number > 0'),
])
def test_one_input_refusals(extra, message, tmp_path, no_input_reads, capsys):
    argv = ['-i', str(tmp_path / 'in.txt'), '--spect', null_data.SPECT, '-o', str(tmp_path / 'o.txt')]
    argv += [str(tmp_path / a) if a == 'R' else a for a in extra]
    assert message in _refused(argv, capsys)
    assert no_input_reads == [] and os.listdir(tmp_path) == []


def test_list_mode_refusals(tmp_path, no_input_reads, capsys):
    lst, paths = genome_data.make_genome(str(tmp_path), chroms=genome_data.CHROMS[:2])
    reps = genome_data.make_replicates(str(tmp_path), n_reps=1)
    out = str(tmp_path / 'out')
    os.makedirs(out)
    base = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '-o', out, '--threshold', '3', '--regions']
    cases = [(out, 'is a directory'), (str(tmp_path / 'absent' / 'r.txt'), 'does not exist'),
             (paths[1], 'reads or writes'), (os.path.join(out, 'chr1.txt'), 'reads or writes'),
             (lst, 'reads or writes'), (genome_data.SPECT, 'reads or writes')]
    for path, message in cases:
        assert message in _refused(base + [path], capsys), path
    null_argv = ['--null', reps, '--pvalues', str(tmp_path / 'p')]
    os.makedirs(tmp_path / 'p')
    assert 'reads or writes' in _refused(base + [os.path.join(str(tmp_path), 'reps', 'rep0.txt')] + null_argv, capsys)
    assert 'reads or writes' in _refused(base + [os.path.join(str(tmp_path), 'p', 'chr2.txt')] + null_argv, capsys)
    assert '--regions needs a cut' in _refused(base[:-3] + ['--regions', str(tmp_path / 'r.txt')], capsys)
    assert no_input_reads == [] and os.listdir(out) == []
    assert not os.path.exists(tmp_path / 'r.txt')


def test_regions_are_allowed_under_torchrun(tmp_path, monkeypatch, no_input_reads):
    monkeypatch.setenv('WORLD_SIZE', '2')
    with pytest.raises(_Read):
        cli.main(['-i', str(tmp_path / 'in.txt'), '--spect', null_data.SPECT, '-o', str(tmp_path / 'o.txt'),
                  '--regions', str(tmp_path / 'r.txt'), '--threshold', '3'])


# ---- the host pipeline, the C oracle standing in for the device scan ------------------------------------------
class OracleScan:
    """scan.DeviceScan with the C oracle as the scan; every null scan it runs is recorded in ``NULLS``."""
    NULLS = []

    def __init__(self, data, neutral, sel, grids, device=0):
        self.problem, self.order = build_problem(data, neutral, sel, grids)

    @classmethod
    def from_problem(cls, problem, order, device=0):
        self = cls.__new__(cls)
        self.problem, self.order = problem, order
        return self

    def run(self, t, lo, hi):
        from oracle import oracle_c
        p = self.problem
        T, iA, ixa, ns, _ = oracle_c.scan(p.genpos, p.cls, p.G, p.SP, p.A, t, lo, hi)
        ix = np.where(ixa >= 0, ixa // p.n_a, -1).astype(np.int32)
        ia = np.where(ixa >= 0, ixa % p.n_a, -1).astype(np.int32)
        if getattr(p, 'seg_start', None) is not None:
            OracleScan.NULLS.append((T.copy(), np.searchsorted(p.seg_start, lo, 'right') - 1, len(p.seg_start)))
        return T, iA, ix, ia, ns

    def close(self):
        pass


@pytest.fixture
def oracle_scan(monkeypatch):
    monkeypatch.setattr(scan, 'DeviceScan', OracleScan)
    OracleScan.NULLS = []
    return OracleScan.NULLS


def parse_regions(main_path, name, cut, q, maxima=None):
    """Region lines computed from the text of a main output file, row by row."""
    with open(main_path) as fh:
        rows = [line.rstrip('\n').split('\t') for line in fh][1:]
    T = [float(f[2]) for f in rows]
    gap = [f[3] == 'NA' for f in rows]
    out = []
    for f, l in brute_regions(T, gap, cut):
        p = brute_peak(T, f, l)
        lo, hi = brute_interval(T, gap, p, q)
        pv = 'NA' if maxima is None else f'{brute_p(T[p], maxima)}'
        out.append('\t'.join([name, rows[f][0], rows[l][0], str(l - f + 1)] + rows[p][:7] + [rows[lo][0], rows[hi][0],
                                                                                           pv]) + '\n')
    return out


def read_regions(path):
    with open(path) as fh:
        lines = fh.readlines()
    m = re.match(r'# CLR cut (\S+) \((.*)\); position support drop q = (\S+)\n$', lines[0])
    assert m and lines[1] == regions.REGION_HEADER
    return float(m.group(1)), m.group(2), float(m.group(3)), lines[2:]


def _run(argv):
    with util.quiet():
        cli.main(argv)


def _cut_between_peaks(main_path):
    """A cut that leaves more than one region: the median of the positive CLRs."""
    with open(main_path) as fh:
        T = np.array([float(line.split('\t')[2]) for line in fh.readlines()[1:]])
    return float(np.median(T[T > 0]))


def _bytes(path):
    with open(path, 'rb') as fh:
        return fh.read()


@pytest.mark.parametrize('mode', ['default', 'w', 'noCenter'])
def test_one_input_pipeline_with_oracle_scan(mode, tmp_path, oracle_scan):
    flags = null_data.MODES[mode][1]
    inp = null_data.write_input(str(tmp_path / 'main.txt'), 120, np.random.default_rng(8))
    base = ['-i', inp, '--spect', null_data.SPECT] + flags
    plain = str(tmp_path / 'plain.txt')
    _run(base + ['-o', plain])
    cut = _cut_between_peaks(plain)
    out, reg = str(tmp_path / 'o.txt'), str(tmp_path / 'r.txt')
    _run(base + ['-o', out, '--regions', reg, '--threshold', repr(cut), '--supportDrop', '1.5'])
    assert _bytes(out) == _bytes(plain)
    got_cut, source, q, lines = read_regions(reg)
    assert (got_cut, source, q) == (cut, '--threshold', 1.5)
    ref = parse_regions(out, 'main.txt', cut, 1.5)
    assert lines == ref and len(ref) > 1
    if mode == 'noCenter':
        assert any('\tNA\t' in line for line in open(out))


def test_one_input_with_null_takes_the_printed_cut(tmp_path, oracle_scan, capsys):
    # replicates much shorter than the input: the input's rows reach above their maxima
    lst, _ = null_data.make_replicates(str(tmp_path), n_reps=6, n_sites=30, seed=7)
    inp = null_data.write_input(str(tmp_path / 'main.txt'), 400, np.random.default_rng(8))
    out, reg, pv = (str(tmp_path / k) for k in ('o.txt', 'r.txt', 'p.txt'))
    cli.main(['-i', inp, '--spect', null_data.SPECT, '-o', out, '--null', lst, '--pvalues', pv, '--regions', reg])
    console = capsys.readouterr().out
    (null_T, rep, n_rep), = oracle_scan
    maxima = brute_maxima(null_T, rep, n_rep)
    cut, source, q, lines = read_regions(reg)
    assert cut == float(np.quantile(maxima, 0.95)) and source == f'0.95 quantile of {n_rep} replicate maxima'
    printed = re.search(r'per-replicate max CLR: 0\.95: (\S+),', console).group(1)
    assert printed == f'{cut:.6g}'
    assert q == DEFAULT_DROP
    assert lines == parse_regions(out, 'main.txt', cut, q, maxima) and len(lines) > 0
    assert any(line.split('\t')[-1] != '1.0\n' for line in lines)
    assert f'regions: {len(lines)} above CLR {cut!r}' in console


def test_input_list_pipeline_with_oracle_scan(tmp_path, oracle_scan, capsys):
    d = str(tmp_path)
    chroms = genome_data.CHROMS[1:]
    lst, paths = genome_data.make_genome(d, chroms=chroms)
    reps = genome_data.make_replicates(d)
    flags = ['--spect', genome_data.SPECT, '-w', '40', '--null', reps]
    for k in ('out', 'p', 'single', 'single_p'):
        os.makedirs(os.path.join(d, k))
    reg = os.path.join(d, 'genome_regions.txt')
    cli.main(['--inputList', '-i', lst, '-o', os.path.join(d, 'out'), '--pvalues', os.path.join(d, 'p'),
              '--regions', reg] + flags)
    console = capsys.readouterr().out
    (null_T, rep, n_rep), = oracle_scan
    maxima = brute_maxima(null_T, rep, n_rep)
    cut, source, q, lines = read_regions(reg)
    assert cut == float(np.quantile(maxima, 0.95))
    ref = []
    for p in paths:
        name = os.path.basename(p)
        ref += parse_regions(os.path.join(d, 'out', name), name, cut, q, maxima)
    assert lines == ref and len(ref) > 1
    hit = len({line.split('\t')[0] for line in ref})
    assert f'regions: {len(ref)} above CLR {cut!r} ({source}) in {hit} of {len(paths)} inputs' in console
    # the genome file is the one-input runs' files laid end to end, comment line and header once
    cat = []
    for p in paths:
        name = os.path.basename(p)
        one = os.path.join(d, 'single_' + name)
        _run(['-i', p, '-o', os.path.join(d, 'single', name), '--pvalues', os.path.join(d, 'single_p', name),
              '--regions', one] + flags)
        with open(one) as fh:
            got = fh.readlines()
        cat += got if not cat else got[2:]
        assert _bytes(os.path.join(d, 'single', name)) == _bytes(os.path.join(d, 'out', name))
    assert _bytes(reg) == ''.join(cat).encode()
