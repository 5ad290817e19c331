"""--null / --pvalues on the CPU: p-value arithmetic, the replicate list, flag pairing, null plans, the per-minCount
selection rows, the whole null pipeline with the C oracle as the scan, and segment-aware sharding costs."""
import os
import socket

import numpy as np
import pytest

import null_data
import util
from ballermixplus_b200 import Grids, InputData, NeutralSFS, NormalizedBetaBinom, null, sharding, windows
from ballermixplus_b200.cli import main
from ballermixplus_b200.problem import build_problem


# ---- p-values ------------------------------------------------------------------------------------------------
def test_pvalue_arithmetic():
    nl = [0.0, 1.0, 2.0, 2.0, 5.0, np.inf, np.nan]          # NaN is left out: N_null = 6
    p = null.pvalues([2.0, 0.0, np.inf, np.nan, 100.0, 5.0, -1.0], nl)
    assert p[0] == 5 / 7                                     # ties count as >=: 2, 2, 5, inf
    assert p[1] == 1.0                                       # CLR 0: exactly 1
    assert p[2] == 2 / 7                                     # only inf >= inf
    assert np.isnan(p[3])
    assert p[4] == 2 / 7
    assert p[5] == 3 / 7
    assert p[6] == 1.0
    with pytest.raises(ValueError):
        null.pvalues([1.0], [])
    with pytest.raises(ValueError):
        null.pvalues([1.0], [np.nan])


def test_pvalue_file_format():
    class Plan:
        f0, f1, gap = ['10', '100\t1e-06\t0\tNA\tNA\tNA\t0\n', '30'], ['1e-07', '', '3e-07'], [False, True, False]

        def __len__(self):
            return 3

    from ballermixplus_b200.problem import GridOrder
    order = GridOrder(Grids(None, None, False, False, None, None))
    T = np.array([3.5, 0.0, np.nan])
    lines = null.format_pvalues(Plan(), order, T, [0, -1, 0], [0, -1, 0], [0, -1, 0], [5, 0, 5],
                                null.pvalues(T, [1.0, 4.0, 3.5]))
    assert lines == [null.PVALUE_HEADER, f'10\t1e-07\t3.5\t{3 / 4}\n', '100\t1e-06\t0\tNA\n', '30\t3e-07\tnan\tNA\n']


# ---- the replicate list --------------------------------------------------------------------------------------
def test_list_parsing(tmp_path):
    lst, paths = null_data.make_replicates(str(tmp_path), n_reps=2, n_sites=20)
    with open(lst, 'a') as fh:
        fh.write(f'   \n# {paths[0]}\n{paths[0]}\n')                 # an absolute path, a comment, blanks
    got = null.read_list(lst)
    assert got == [paths[0], paths[1], paths[0]]
    with pytest.raises(FileNotFoundError):
        null.read_list(str(tmp_path / 'absent.txt'))
    empty = tmp_path / 'empty.txt'
    empty.write_text('# nothing\n\n')
    with pytest.raises(ValueError):
        null.read_list(str(empty))
    bad = tmp_path / 'bad.txt'
    bad.write_text('reps/rep0.txt\nreps/missing.txt\n')
    with pytest.raises(FileNotFoundError, match='missing.txt'):
        null.read_list(str(bad))


def test_missing_replicate_fails_before_any_scan(tmp_path, capsys):
    bad = tmp_path / 'bad.txt'
    bad.write_text('nowhere.txt\n')
    # the input file does not exist either: the list is checked before anything is read
    argv = ['-i', str(tmp_path / 'no_input.txt'), '--spect', null_data.SPECT, '-o', str(tmp_path / 'o.txt'),
            '--null', str(bad), '--pvalues', str(tmp_path / 'p.txt')]
    with pytest.raises(SystemExit) as e:
        main(argv)
    assert e.value.code == 2 and 'nowhere.txt' in capsys.readouterr().err
    # the Python API: the error comes before a GPU problem is built (there is none on a CPU machine)
    inp = null_data.write_input(str(tmp_path / 'in.txt'), 50, np.random.default_rng(1))
    data, neutral, grid, sel = _objects(inp)
    from ballermixplus_b200.scan import Scan
    with util.quiet(), pytest.raises(FileNotFoundError):
        Scan(data, neutral, sel, grid, str(tmp_path / 'o.txt'), null=str(bad), pvalues=str(tmp_path / 'p.txt'))


@pytest.mark.parametrize('flags', [['--null', 'x.txt'], ['--pvalues', 'p.txt']])
def test_flag_pairing(flags, tmp_path, capsys):
    argv = ['-i', 'in.txt', '--spect', 's.txt', '-o', str(tmp_path / 'o.txt')] + flags
    with pytest.raises(SystemExit) as e:
        main(argv)
    assert e.value.code == 2 and 'together' in capsys.readouterr().err
    from ballermixplus_b200.scan import Scan
    with pytest.raises(ValueError, match='together'):
        Scan(None, None, None, None, str(tmp_path / 'o.txt'), **({'null': 'x'} if '--null' in flags else {'pvalues': 'p'}))


# ---- null plans, tables and the whole pipeline ----------------------------------------------------------------
def _objects(infile, **mode):
    with util.quiet():
        data = InputData(infile, False, False, False, 1, phys=mode.get('phys', False), Rrate=1e-6)
        neutral = NeutralSFS(null_data.SPECT, False, False, False)
        neutral.get_neut_probs(data)
        grid = Grids(None, None, False, False, None, None)
        sel = NormalizedBetaBinom(data, grid, False, False, False)
    return data, neutral, grid, sel


@pytest.mark.parametrize('mode', list(null_data.MODES))
def test_plan_offsets_and_gap_rows(mode, tmp_path):
    kw, _ = null_data.MODES[mode]
    lst, paths = null_data.make_replicates(str(tmp_path), n_reps=3, n_sites=120, seed=3)
    reps = [_objects(p, **kw)[0] for p in paths]
    seg = np.concatenate(([0], np.cumsum([d.numSites for d in reps])[:-1]))
    t, lo, hi, rep = null.null_plan(reps, paths, seg, **kw)
    n_gap = 0
    for i, d in enumerate(reps):
        with util.quiet():
            plan = windows.make_plan(d, **kw)
        pt, plo, phi, gap = plan.arrays()
        n_gap += int(gap.sum())
        m = rep == i
        np.testing.assert_array_equal(t[m], pt[~gap])
        np.testing.assert_array_equal(lo[m], plo[~gap] + seg[i])
        np.testing.assert_array_equal(hi[m], phi[~gap] + seg[i])
        assert np.all(lo[m] >= seg[i]) and np.all(hi[m] < seg[i] + d.numSites)
    assert (n_gap > 0) == (mode == 'noCenter')


def test_class_rows_per_mincount_are_bit_identical(tmp_path):
    lst, paths = null_data.make_replicates(str(tmp_path), n_reps=3, n_sites=150, seed=5)
    objs = [_objects(p) for p in paths]
    mins = [int(o[0].minCount) for o in objs]
    assert len(set(mins)) == 2                                  # replicate 1 has its own minCount
    data, neutral, grid, sel = objs[0]
    setup = null.NullSetup(lst, data, neutral, sel, grid)
    prob = setup.problem
    for i, (d, nt, g, s) in enumerate(objs):
        alone, _ = build_problem(d, nt, s, g)
        b = prob.seg_start[i]
        cls = prob.cls[b:b + d.numSites]
        # same site -> same G and the same SP column, bit for bit
        assert np.array_equal(prob.G[cls], alone.G[alone.cls])
        assert np.array_equal(prob.SP[:, cls], alone.SP[:, alone.cls])
        assert np.array_equal(prob.genpos[b:b + d.numSites], alone.genpos)


def _oracle_T(prob, t, lo, hi):
    from oracle import oracle_c
    return oracle_c.scan(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t, lo, hi)[0]


def _standalone_null(paths, mode):
    """CLR values the oracle CLI writes for each replicate on its own, gap rows left out."""
    from oracle import oracle_cli
    out = []
    for p in paths:
        argv = ['-i', p, '--spect', null_data.SPECT] + null_data.MODES[mode][1]
        kw = util.oracle_kwargs(argv)
        kw['infile'], kw['spectfile'] = p, null_data.SPECT
        for line in oracle_cli.scan_file(**kw)[1:]:
            f = line.rstrip('\n').split('\t')
            if f[3] == 'NA':
                continue
            out.append(float(f[2]))
    return np.array(out)


@pytest.mark.parametrize('mode', ['default', 'w', 'noCenter'])
def test_null_pipeline_with_oracle_scan(mode, tmp_path):
    kw, _ = null_data.MODES[mode]
    lst, paths = null_data.make_replicates(str(tmp_path), n_reps=3, n_sites=120, seed=7)
    main_in = null_data.write_input(str(tmp_path / 'main.txt'), 120, np.random.default_rng(8))
    data, neutral, grid, sel = _objects(main_in, **kw)
    with util.quiet():
        setup = null.NullSetup(lst, data, neutral, sel, grid, **kw)
    got = np.sort(_oracle_T(setup.problem, setup.t, setup.lo, setup.hi))
    ref = np.sort(_standalone_null(paths, mode))
    assert len(got) == len(ref) > 0
    assert np.all(np.abs(got - ref) <= 1e-9 * np.maximum(np.abs(ref), 1.0))
    assert np.any(ref > 0)
    lines = null.summary(got, setup.rep, setup.n_replicates)
    assert f'{setup.n_replicates} neutral replicates, {len(got)} null rows' in lines[0]


# ---- segment-aware sharding costs -----------------------------------------------------------------------------
def _segmented_case():
    rng = np.random.default_rng(11)
    sizes = [300, 50, 700, 1]
    g = np.concatenate([np.sort(rng.uniform(0, 0.01, n)) for n in sizes])
    seg = np.concatenate(([0], np.cumsum(sizes)[:-1]))
    return g, seg, sizes


def test_centre_costs_with_segments():
    g, seg, sizes = _segmented_case()
    A = [1e3, 1e4, 1e5, 0.0]
    parts_t, parts_lo, parts_hi, ref = [], [], [], []
    for b, n in zip(seg, sizes):
        c = np.arange(0, n, 3)
        lo, hi = np.maximum(0, c - 40), np.minimum(n - 1, c + 60)
        ref.append(sharding.centre_costs(g[b:b + n], g[b + c], lo, hi, A))       # each segment on its own
        parts_t.append(g[b + c]); parts_lo.append(lo + b); parts_hi.append(hi + b)
    t, lo, hi = np.concatenate(parts_t), np.concatenate(parts_lo), np.concatenate(parts_hi)
    np.testing.assert_array_equal(sharding.centre_costs(g, t, lo, hi, A, seg), np.concatenate(ref))
    # without the segments the array is not monotone: whole windows
    np.testing.assert_array_equal(sharding.centre_costs(g, t, lo, hi, A), len(A) * (hi - lo + 1) + 1.0)
    # a window across a boundary is charged whole
    x = sharding.centre_costs(g, [g[299]], [250], [320], A, seg)
    assert x[0] == len(A) * 71 + 1.0
    # one segment is the plain call
    s0 = sharding.centre_costs(g[:300], t[:100], lo[:100], hi[:100], A, [0])
    np.testing.assert_array_equal(s0, sharding.centre_costs(g[:300], t[:100], lo[:100], hi[:100], A))


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _seg_problem(tmp):
    lst, paths = null_data.make_replicates(tmp, n_reps=3, n_sites=100, seed=13)
    data, neutral, grid, sel = _objects(paths[0], **null_data.MODES['w'][0])
    with util.quiet():
        setup = null.NullSetup(lst, data, neutral, sel, grid, **null_data.MODES['w'][0])
    return setup


def _oracle_rows(prob):
    import torch
    from oracle import oracle_c

    def fn(t, lo, hi):
        T, iA, ixa, ns, _ = oracle_c.scan(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t, lo, hi, n_threads=1)
        ix = np.where(ixa >= 0, ixa // prob.n_a, -1).astype(np.int32)
        ia = np.where(ixa >= 0, ixa % prob.n_a, -1).astype(np.int32)
        return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in (T, iA, ix, ia, ns))
    return fn


def _worker(rank, world, port, tmp, out_path):
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        s = _seg_problem(tmp)
        p = s.problem
        got = sharding.scan_sharded(p.genpos, p.A, s.t, s.lo, s.hi, rank, world, _oracle_rows(p), dist, torch,
                                    seg_start=p.seg_start)
        if rank == 0:
            torch.save([g.clone() for g in got], out_path)
        else:
            assert got is None
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world', [2, 3])
def test_segmented_sharded_scan_equals_single_process(world, tmp_path):
    import torch
    import torch.multiprocessing as mp
    tmp = str(tmp_path)
    s = _seg_problem(tmp)
    costs = sharding.centre_costs(s.problem.genpos, s.t, s.lo, s.hi, s.problem.A, s.problem.seg_start)
    whole = len(s.problem.A) * (s.hi - s.lo + 1) + 1.0
    assert np.all(costs <= whole) and np.any(costs < whole)      # cut at alpha reach inside each segment
    out = str(tmp_path / 'rows.pt')
    mp.spawn(_worker, args=(world, _free_port(), tmp, out), nprocs=world, join=True)
    got = torch.load(out)
    ref = _oracle_rows(s.problem)(s.t, s.lo, s.hi)
    for a, b in zip(got, ref):
        assert torch.equal(a, b)
