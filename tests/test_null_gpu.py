"""Segmented problems (blmx_load_segmented) and --null / --pvalues on the GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest

import null_data
import util


def _replicates(sizes=(3000, 800, 5000, 1200), seed=50):
    """Replicates with one shared class table (bench's synthetic chromosomes) -> (alone problems, segmented
    concatenation, the same concatenation without segments, segment starts)."""
    import bench
    from ballermixplus_b200.native import ScanProblem
    probs = bench.make_problem([bench.make_chromosome(n, seed + i) for i, n in enumerate(sizes)])
    seg = np.concatenate(([0], np.cumsum(sizes)[:-1])).astype(np.int64)
    p0 = probs[0]
    g = np.concatenate([p.genpos for p in probs])
    c = np.concatenate([p.cls for p in probs])
    cat = ScanProblem(g, c, p0.G, p0.SP, p0.A, p0.n_x, p0.n_a, seg_start=seg)
    plain = ScanProblem(g, c, p0.G, p0.SP, p0.A, p0.n_x, p0.n_a)
    return probs, cat, plain, seg


def _centres(probs, seg, stride=7):
    """Whole-replicate windows (the default mode) on every stride-th site, per replicate and offset."""
    out = []
    for p, b in zip(probs, seg):
        n = len(p.genpos)
        c = np.arange(0, n, stride)
        out.append((p.genpos[c], np.zeros(len(c), np.int64), np.full(len(c), n - 1, np.int64), b))
    return out


def _scan(prob, t, lo, hi, farfield=None, **opts):
    from ballermixplus_b200.native import Scanner
    with Scanner(device=0, farfield=farfield).load(prob) as sc:
        for k, v in opts.items():
            sc.set_option(k, v)
        return sc.scan(t, lo, hi), sc.counters_all()


def _assert_parity(prob_alone, t, lo, hi, a, b):
    """Rows a (segmented) and b (standalone) of the same centres: T within 1e-9, nSites identical, argmax
    identical or a literal tie."""
    Ta, Tb = a[0], b[0]
    assert np.all(np.abs(Ta - Tb) <= 1e-9 * np.maximum(np.abs(Tb), 1.0)), np.max(np.abs(Ta - Tb))
    assert np.array_equal(a[4], b[4])
    n_xa = prob_alone.n_a
    for j in np.flatnonzero((a[1] != b[1]) | (a[2] != b[2]) | (a[3] != b[3])):
        assert a[1][j] >= 0 and b[1][j] >= 0, j
        va, _ = util.literal_T(prob_alone, t[j], lo[j], hi[j], a[1][j], a[2][j] * n_xa + a[3][j])
        vb, _ = util.literal_T(prob_alone, t[j], lo[j], hi[j], b[1][j], b[2][j] * n_xa + b[3][j])
        assert abs(va - vb) <= 1e-12 * max(abs(vb), 1.0), (j, va, vb)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['default', 'group1', 'farfield0', 'report_all'])
def test_segmented_load_equals_standalone_loads(mode):
    probs, cat, plain, seg = _replicates()
    opts = {'group1': dict(group=1), 'report_all': dict(report_all=1)}.get(mode, {})
    ff = 0 if mode == 'farfield0' else None
    cs = _centres(probs, seg)
    t = np.concatenate([c[0] for c in cs])
    lo = np.concatenate([c[1] + c[3] for c in cs])
    hi = np.concatenate([c[2] + c[3] for c in cs])
    rows, k = _scan(cat, t, lo, hi, farfield=ff, **opts)
    off = 0
    for p, (tt, ll, hh, _) in zip(probs, cs):
        alone, _ = _scan(p, tt, ll, hh, farfield=ff, **opts)
        sl = slice(off, off + len(tt))
        _assert_parity(p, tt, ll, hh, [r[sl] for r in rows], alone)
        off += len(tt)
    if mode == 'default':
        assert k['far_sites'] > 0 and k['pruned_items'] > 0, k       # the fast paths run on the segmented load
        _, kp = _scan(plain, t, lo, hi)
        assert kp['pruned_items'] == 0 and kp['far_blocks'] == 0, kp   # not without the segments
    if mode == 'report_all':
        assert k['far_sites'] > 0


def _crossing(cat, seg, rng):
    n = len(cat.genpos)
    b = np.repeat(seg[1:], 40)
    c = np.clip(b + rng.integers(-50, 50, size=len(b)), 0, n - 1)
    lo = c - rng.integers(0, 400, size=len(b))
    hi = c + rng.integers(0, 400, size=len(b))
    inside = rng.integers(0, n, size=100)                 # and windows inside one segment
    c = np.concatenate((c, inside))
    lo = np.concatenate((lo, inside - 30))
    hi = np.concatenate((hi, inside + 30))
    return cat.genpos[c].copy(), lo, hi


@pytest.mark.gpu
def test_crossing_windows_are_exact():
    probs, cat, plain, seg = _replicates()
    t, lo, hi = _crossing(cat, seg, np.random.default_rng(3))
    a, ka = _scan(cat, t, lo, hi)
    b, _ = _scan(plain, t, lo, hi)
    _assert_parity(plain, t, lo, hi, a, b)
    assert ka['pruned_items'] > 0                         # the inside windows still take the fast paths


@pytest.mark.gpu
def test_one_segment_is_blmx_load():
    from ballermixplus_b200.native import ScanProblem
    probs, _, _, _ = _replicates(sizes=(6000,))
    p = probs[0]
    one = ScanProblem(p.genpos, p.cls, p.G, p.SP, p.A, p.n_x, p.n_a, seg_start=[0])
    (t, lo, hi, _), = _centres(probs, [0], stride=5)
    for opts in ({}, {'report_all': 1}):
        a, ka = _scan(one, t, lo, hi, **opts)
        b, kb = _scan(p, t, lo, hi, **opts)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
        ka.pop('launches'); kb.pop('launches')
        assert ka == kb


@pytest.mark.gpu
@pytest.mark.parametrize('starts', [[1, 5], [0, 5, 5], [0, 7, 3], [0, 10**6], [0, -1], []])
def test_bad_segment_starts(starts):
    from ballermixplus_b200.native import BlmxError, ScanProblem, Scanner
    probs, _, _, _ = _replicates(sizes=(300,))
    p = probs[0]
    bad = ScanProblem(p.genpos, p.cls, p.G, p.SP, p.A, p.n_x, p.n_a, seg_start=starts)
    with Scanner(device=0) as sc, pytest.raises(BlmxError, match='error -1'):
        sc.load(bad)


@pytest.mark.gpu
def test_range_checked_build_sees_no_violation_with_segments():
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import test_null_gpu as T
probs, cat, plain, seg = T._replicates()
t, lo, hi = T._crossing(cat, seg, np.random.default_rng(9))
cs = T._centres(probs, seg, stride=11)
t = np.concatenate([t] + [c[0] for c in cs])
lo = np.concatenate([lo] + [c[1] + c[3] for c in cs])
hi = np.concatenate([hi] + [c[2] + c[3] for c in cs])
bad = pruned = far = 0
for opts in ({}, {'report_all': 1}, {'group': 1}):
    rows, k = T._scan(cat, t, lo, hi, batch=53, **opts)
    bad += k['range_violations']; pruned += k['pruned_items']; far += k['far_sites']
print('VIOLATIONS', bad, 'PRUNED', pruned, 'FAR', far)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [x for x in out.stdout.split('\n') if x.startswith('VIOLATIONS')][-1]
    f = line.split()
    assert f[1] == '0' and int(f[3]) > 0 and int(f[5]) > 0, line


def _cli(argv):
    from ballermixplus_b200.cli import main
    with util.quiet():
        main(argv)


def _clr_of(path):
    """CLR of every row of a main output file that is not a --noCenter gap row."""
    out = []
    with open(path) as fh:
        next(fh)
        for line in fh:
            f = line.rstrip('\n').split('\t')
            if f[3] != 'NA':
                out.append(float(f[2]))
    return np.array(out)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['default', 'w', 'noCenter'])
def test_cli_pvalues_end_to_end(mode, tmp_path):
    from ballermixplus_b200 import null
    _, flags = null_data.MODES[mode]
    d = str(tmp_path)
    lst, paths = null_data.make_replicates(d, n_reps=4, n_sites=400, seed=21)
    main_in = null_data.write_input(os.path.join(d, 'main.txt'), 400, np.random.default_rng(22))
    base = ['--spect', null_data.SPECT] + flags
    plain, with_null, pv = (os.path.join(d, n) for n in ('plain.txt', 'with_null.txt', 'p.txt'))
    _cli(['-i', main_in, '-o', plain] + base)
    _cli(['-i', main_in, '-o', with_null, '--null', lst, '--pvalues', pv] + base)
    with open(plain, 'rb') as a, open(with_null, 'rb') as b:
        assert a.read() == b.read()                        # the main output does not change
    # the null from the CLI's own outputs, one standalone run per replicate
    nulls = []
    for i, p in enumerate(paths):
        out = os.path.join(d, f'rep{i}.out')
        _cli(['-i', p, '-o', out] + base)
        nulls.append(_clr_of(out))
    nl = np.concatenate(nulls)
    real = _clr_of(plain)
    assert np.any(real > 0) and np.any(nl > 0)
    pos = nl[nl > 0]
    for T in real[real > 0]:                               # no null value within the parity bar of a real CLR
        assert np.all(np.abs(pos - T) > 1e-9 * max(T, 1.0))
    with open(plain) as fh:
        main_rows = fh.read().splitlines()[1:]
    with open(pv) as fh:
        got = fh.read().splitlines()
    assert got[0] + '\n' == null.PVALUE_HEADER and len(got) == len(main_rows) + 1
    for m, g in zip(main_rows, got[1:]):
        mf, gf = m.split('\t'), g.split('\t')
        assert gf[:3] == mf[:3]
        if mf[3] == 'NA':
            assert gf[3] == 'NA'
        else:
            assert gf[3] == f'{float(null.pvalues([float(mf[2])], nl)[0])}', (m, g)
