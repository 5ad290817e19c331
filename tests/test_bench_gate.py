"""bench.py's host logic (no GPU): the parity gate must fail on a wrong row, the centre sample must contain the
rows that carry a real maximum, the output dump must hold the rows, and the flop accounting must add up."""
import os

import numpy as np

import bench


class _P:
    n_a = 51


def _fake(n=40, seed=0):
    rng = np.random.default_rng(seed)
    T = np.where(rng.random(n) < 0.5, rng.random(n) * 30, 0.0)
    iA = np.where(T > 0, rng.integers(0, 100, n), -1).astype(np.int32)
    ix = np.where(T > 0, rng.integers(0, 10, n), -1).astype(np.int32)
    ia = np.where(T > 0, rng.integers(0, 51, n), -1).astype(np.int32)
    ns = np.where(T > 0, rng.integers(1, 5000, n), 0).astype(np.int32)
    return T, iA, ix, ia, ns


def _oracle_view(rows, idx):
    T, iA, ix, ia, ns = (a[idx] for a in rows)
    return T.copy(), iA.copy(), np.where(iA >= 0, ix * 51 + ia, -1), ns.copy(), 0


def test_parity_gate_passes_on_equal_rows_and_fails_on_any_difference():
    rows = _fake()
    plans = [(np.zeros(25), None, None), (np.zeros(15), None, None)]
    sample, bounds = bench.parity_sample(plans, rows[0], n_positive=8, n_any=6)
    picked = np.concatenate([bounds[c] + idx for c, idx in sample])
    assert np.count_nonzero(rows[0][picked] > 0) >= min(8, np.count_nonzero(rows[0] > 0))
    kept = ([(c, idx, _oracle_view(rows, bounds[c] + idx)) for c, idx in sample], [])
    ok = bench.parity_check([_P(), _P()], kept, bounds, rows, None)
    assert ok['ok'] and ok['centres'] == len(picked) and ok['rows_T_gt_0'] == np.count_nonzero(rows[0][picked] > 0)
    j = int(picked[np.flatnonzero(rows[0][picked] > 0)[0]])
    for field, delta in ((0, 1e-6), (1, 1), (3, 1), (4, 1)):            # T, A, a, nSites
        bad = [a.copy() for a in rows]
        bad[field][j] += delta
        res = bench.parity_check([_P(), _P()], kept, bounds, tuple(bad), None)
        assert not res['ok'], field
    # the report_all leg is checked the same way
    kept_all = (kept[0], kept[0])
    rows_all = tuple(np.concatenate([a[bounds[c] + idx] for c, idx in sample]) for a in rows)
    assert bench.parity_check([_P(), _P()], kept_all, bounds, rows, rows_all)['ok']
    wrong = [a.copy() for a in rows_all]
    wrong[0][0] += 1.0
    assert not bench.parity_check([_P(), _P()], kept_all, bounds, rows, tuple(wrong))['ok']


def test_dump_outputs_writes_every_row_or_a_fixed_sample(tmp_path):
    rows = _fake(n=1000)
    bench.dump_outputs(str(tmp_path / 'all'), rows)
    got = {f: np.load(tmp_path / 'all' / f'{f}.npy') for f in ('centre', 'T', 'iA', 'ix', 'ia', 'nsites')}
    assert all(a.dtype == np.float64 and a.shape == (1000,) for a in got.values())
    assert np.array_equal(got['centre'], np.arange(1000))
    for f, a in zip(('T', 'iA', 'ix', 'ia', 'nsites'), rows):
        assert np.array_equal(got[f], a)
    limit = 48 * 300                                          # room for 300 rows of the six fields
    for run in ('s1', 's2'):
        bench.dump_outputs(str(tmp_path / run), rows, limit=limit)
    c1, c2 = (np.load(tmp_path / run / 'centre.npy') for run in ('s1', 's2'))
    assert len(c1) == 300 and np.array_equal(c1, c2) and np.all(np.diff(c1) > 0)
    assert np.array_equal(np.load(tmp_path / 's1' / 'T.npy'), rows[0][c1.astype(np.int64)])
    assert sum(os.path.getsize(p) for p in (tmp_path / 's1').iterdir()) <= limit + 6 * 128


def test_flop_accounting():
    cnt = {'pairs': 1000, 'single': 0, 'far_sites': 700, 'edge_sites': 50, 'far_blocks': 10, 'far_terms': 40}
    f = bench.algorithmic_flops(cnt, 510, 2)
    direct = 300
    want = (510 * 2.25 * direct + bench.FLOP_QUAD_COEF * direct + 34 * (direct + 50) + 9 * 50 + bench.FLOP_BLOCK * 10
            + 2 * 510 * 40 + 50 * 510 * 2)
    assert abs(f - want) < 1e-6
    assert bench.FLOP_BLOCK == 34 + 32 * 12


def test_genome_and_centres():
    sizes = bench.genome_sizes(10_000_000)
    assert sum(sizes) == 10_000_000 and len(sizes) == 22 and sizes[0] > 800_000
    c = bench.make_chromosome(5000, seed=3)
    assert len(c['pos']) == 5000 and np.all(np.diff(c['pos']) > 0) and c['k'].max() == 200
    assert abs(np.mean(c['k'] == 200) - 0.7) < 0.03
