"""Binned neutral spectra on the GPU: the pruner past 256 classes (bound_kernel's slab path) keeps the rows of
prune = 0 and proves items, the range-checked build sees no violation on it, and the command line with a 3-bin map
writes the rows of the C oracle on the binned class tables."""
import os
import subprocess
import sys

import numpy as np
import pytest

import util

sys.path.insert(0, os.path.join(util.ROOT, 'tools'))


def _problem(n_sites=20000, n_bins=3, seed=12345):
    import bench
    import binmap_cost
    return binmap_cost.binned_problem(bench.make_chromosome(n_sites, seed=seed), n_bins, same=False)


def _scan(prob, t, lo, hi, prune, **opts):
    from ballermixplus_b200.native import Scanner
    with Scanner(device=0, **opts).load(prob) as sc:
        sc.set_option('prune', prune)
        return sc.scan(t, lo, hi), sc.counters_all()


@pytest.mark.gpu
@pytest.mark.parametrize('n_bins', [2, 3])
def test_prune_past_256_classes_keeps_the_rows(n_bins):
    prob = _problem(n_bins=n_bins)
    assert len(prob.G) > 256
    n = len(prob.genpos)
    rng = np.random.default_rng(n_bins)
    c = np.concatenate([np.arange(0, n, 50), rng.integers(0, n, 200)])
    t = prob.genpos[c].copy()
    lo = np.where(np.arange(len(c)) % 3 == 0, 0, c - rng.integers(0, 4000, len(c)))
    hi = np.where(np.arange(len(c)) % 3 == 0, n - 1, c + rng.integers(0, 4000, len(c)))
    r0, k0 = _scan(prob, t, lo, hi, 0)
    r1, k1 = _scan(prob, t, lo, hi, 1, batch=97)
    for a, b in zip(r0, r1):
        assert np.array_equal(a, b)
    assert k0['pruned_items'] == 0
    assert k1['pruned_items'] > 0.3 * len(c) * len(prob.A)
    assert k0['pairs'] == k1['pairs']


@pytest.mark.gpu
def test_range_checked_build_sees_no_violation_past_256_classes():
    lib = os.path.join(util.ROOT, 'ballermixplus_b200', 'libblmx_checked.so')
    assert os.path.exists(lib), 'run __graft_entry__.build() first'
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)
import bench, binmap_cost
from ballermixplus_b200.native import Scanner
prob = binmap_cost.binned_problem(bench.make_chromosome(20000, seed=7), 3, same=False)
assert len(prob.G) > 256
n = len(prob.genpos)
rng = np.random.default_rng(17)
c = rng.integers(0, n, size=150)
t = prob.genpos[c] + np.where(rng.random(150) < 0.2, 1e-7, 0.0)
lo = c - rng.integers(-20, 9000, size=150)
hi = c + rng.integers(-20, 9000, size=150)
lo[::5] = 0; hi[::5] = n - 1
bad = pruned = 0
res = []
for pr in (0, 1):
    with Scanner(device=0, batch=37).load(prob) as sc:
        sc.set_option('prune', pr)
        res.append(sc.scan(t, lo, hi))
        k = sc.counters_all()
        bad += k['range_violations']
        pruned += k['pruned_items']
for a, b in zip(*res):
    assert np.array_equal(a, b)
print('VIOLATIONS', bad, 'PRUNED', pruned)
''' % (util.ROOT, os.path.join(util.ROOT, 'tests'), os.path.join(util.ROOT, 'tools'))
    env = dict(os.environ, BLMX_LIB=lib)
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert 'VIOLATIONS 0 ' in out.stdout, out.stdout[-500:]
    assert 'PRUNED 0' not in out.stdout.split('\n')[-2], out.stdout[-500:]


@pytest.mark.gpu
@pytest.mark.parametrize('variant', ['B1', 'B2', 'B2maf', 'B0', 'B0maf'])
def test_cli_with_a_three_bin_map_equals_the_oracle(variant, tmp_path):
    from test_binmap import FLAGS, _setup
    from test_regions import OracleScan
    from ballermixplus_b200 import cli, scan
    infile, spect, flags, listf, mapf = _setup(tmp_path, variant)
    argv = ['-i', infile, '--spect', spect, '-w', '30', '--spectBins', listf, '--binMap', mapf]
    argv += [FLAGS[f] for f in flags]
    with util.quiet():
        cli.main(argv + ['-o', str(tmp_path / 'gpu.txt')])
    keep = scan.DeviceScan
    scan.DeviceScan = OracleScan
    try:
        with util.quiet():
            cli.main(argv + ['-o', str(tmp_path / 'oracle.txt')])
    finally:
        scan.DeviceScan = keep
    g = np.loadtxt(tmp_path / 'gpu.txt', skiprows=1, ndmin=2)
    o = np.loadtxt(tmp_path / 'oracle.txt', skiprows=1, ndmin=2)
    assert g.shape == o.shape
    assert np.all(np.abs(g[:, 2] - o[:, 2]) <= 1e-9 * np.maximum(np.abs(o[:, 2]), 1.0))
    assert np.array_equal(g[:, 6], o[:, 6])


@pytest.mark.gpu
def test_prune_past_256_classes_with_more_than_512_grid_points():
    """The slab path gathers every slab again per 512 grid points: 663 points (two groups, the second ragged)."""
    from ballermixplus_b200.native import ScanProblem
    prob = _problem(n_bins=3)
    SP = np.vstack([prob.SP, prob.SP[:153] * 0.999])
    wide = ScanProblem(prob.genpos, prob.cls, prob.G, SP, prob.A, 13, prob.n_a)
    assert len(wide.G) > 256 and wide.n_x * wide.n_a == 663
    n = len(wide.genpos)
    c = np.arange(0, n, 80)
    t, lo, hi = wide.genpos[c], np.maximum(c - 3000, 0), np.minimum(c + 3000, n - 1)
    r0, k0 = _scan(wide, t, lo, hi, 0)
    r1, k1 = _scan(wide, t, lo, hi, 1)
    for a, b in zip(r0, r1):
        assert np.array_equal(a, b)
    assert k1['pruned_items'] > 0.3 * len(c) * len(wide.A)


@pytest.mark.gpu
def test_prune_with_many_slabs():
    """Every binned class split into 10 classes by position (same tables): about 5 700 classes, so a
    whole-chromosome window takes some 25 slabs, each summed on its own; the rows equal prune = 0's and items are
    proved.  (One class per site would switch the pruner off: no class run is long enough for far-field blocks.)"""
    from ballermixplus_b200.native import ScanProblem
    prob = _problem(n_bins=3)
    n = len(prob.genpos)
    cls = prob.cls.astype(np.int64) * 10 + np.arange(n) * 10 // n
    many = ScanProblem(prob.genpos, cls.astype(np.int32), np.repeat(prob.G, 10), np.repeat(prob.SP, 10, axis=1),
                       prob.A, prob.n_x, prob.n_a)
    assert len(many.G) > 20 * 256
    c = np.arange(0, n, 250)
    whole = np.arange(len(c)) % 2 == 0
    t = many.genpos[c]
    lo = np.where(whole, 0, np.maximum(c - 2000, 0))
    hi = np.where(whole, n - 1, np.minimum(c + 2000, n - 1))
    r0, _ = _scan(many, t, lo, hi, 0)
    r1, k1 = _scan(many, t, lo, hi, 1)
    for x, y in zip(r0, r1):
        assert np.array_equal(x, y)
    assert k1['pruned_items'] > 0.3 * len(c) * len(many.A)


@pytest.mark.gpu
def test_binned_input_list_under_torchrun_equals_one_gpu(tmp_path):
    """--inputList with a bin map under torchrun (two ranks on one card, gather over gloo) writes the bytes of the
    one-GPU run."""
    import genome_data
    from test_binmap import _perturbed, _write
    from test_genome_list_gpu import _torchrun
    from ballermixplus_b200 import cli
    d = str(tmp_path)
    lst, paths = genome_data.make_genome(d)
    bins = _write(os.path.join(d, 'bins.txt'), f'hi {_perturbed(genome_data.SPECT, os.path.join(d, "hi.txt"), 2, False)}'
                                               f'\nlo {_perturbed(genome_data.SPECT, os.path.join(d, "lo.txt"), 3, False)}\n')
    names = [os.path.basename(p) for p in paths]
    mapf = _write(os.path.join(d, 'map.txt'), f'{names[0]} 1 900000 hi\n{names[0]} 2600000 4000000 lo\n'
                                              f'{names[-1]} 0 3000000 lo\n')
    for k in ('one', 'many'):
        os.makedirs(os.path.join(d, k))
    argv = ['--inputList', '-i', lst, '--spect', genome_data.SPECT, '--spectBins', bins, '--binMap', mapf, '-w', '40']
    with util.quiet():
        cli.main(argv + ['-o', os.path.join(d, 'one')])
    out = _torchrun(argv + ['-o', os.path.join(d, 'many')], 29571)
    assert 'on 2 ranks' in out
    for name in names:
        with open(os.path.join(d, 'one', name), 'rb') as a, open(os.path.join(d, 'many', name), 'rb') as b:
            got, ref = b.read(), a.read()
        assert got == ref and got.count(b'\n') > 1, name
