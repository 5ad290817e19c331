"""The product against the reference: its host objects against the reference's OWN objects where the unmodified
reference script is at hand (oracle/_ref/, copied there by oracle/make_ref.sh), and everywhere the calcBaller
seam (INTEGRATION.md section 2) fed objects shaped like the reference's, and the reference's own printed rows."""
import importlib.util
import os
from types import SimpleNamespace

import numpy as np
import pytest

import util

REF = os.path.join(util.ROOT, 'oracle', '_ref', 'BalLeRMix+_v1.py')


@pytest.fixture(scope='module')
def ref():
    if not os.path.exists(REF):
        pytest.skip('the reference script is not in oracle/_ref (oracle/make_ref.sh copies it there)')
    spec = importlib.util.spec_from_file_location('ballermix_ref', REF)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _ref_objects(ref, argv):
    from ballermixplus_b200.cli import build_parser
    opt = build_parser().parse_args(util.abs_paths(argv))
    with util.quiet():
        data = ref.InputData(opt.infile, opt.nofreq, opt.MAF, opt.nosub, opt.minCount, phys=opt.phys, Rrate=opt.Rrate)
        neutral = ref.NeutralSFS(opt.spectfile, opt.nofreq, opt.MAF, opt.nosub)
        neutral.get_neut_probs(data)
        grid = ref.Grids(opt.x, opt.abeta, opt.bal, opt.pos, opt.seqA, opt.listA)
        sel = ref.NormalizedBetaBinom(data, grid, opt.nofreq, opt.MAF, opt.nosub)
    return data, neutral, grid, sel


@pytest.mark.parametrize('name', ['Example1_B2', 'Example2_B2maf', 'Example1_B1', 'ex2_B0_s5',
                                  'Example2_B0maf_1kb-2site', 'synth_mixed_n_B2_s20'])
def test_host_objects_equal_reference_objects(ref, name):
    argv, _ = util.scan_cases()[name]
    rdata, rneutral, rgrid, rsel = _ref_objects(ref, argv)
    opt, data, neutral, grid, sel = util.host_objects(argv)
    assert np.array_equal(data.position, rdata.position) and np.array_equal(data.genPos, rdata.genPos)
    assert np.array_equal(data.count, rdata.count) and np.array_equal(data.total, rdata.total)
    assert data.minCount == rdata.minCount and data.sampSizes == rdata.sampSizes
    assert np.array_equal(neutral.probs, rneutral.probs) and np.array_equal(neutral.propSizes, rneutral.propSizes)
    assert grid.x == rgrid.x and grid.A == rgrid.A and grid.abeta == rgrid.abeta
    assert [type(v) for v in grid.abeta] == [type(v) for v in rgrid.abeta]
    for key, per_site in rsel.normProbs.items():
        assert np.array_equal(sel.get(*key), per_site), key        # bit-identical, all 510 tables


def _reference_shaped(data, neutral, grid, sel):
    """The host objects reduced to what the reference's own objects offer build_problem and calcBaller: per-site
    arrays, NeutralSFS's spect / sampProps dictionaries (v1:271,275), per-site normProbs (v1:359), plain grids."""
    rdata = SimpleNamespace(position=data.position, genPos=data.genPos, count=data.count, total=data.total,
                            numSites=data.numSites)
    rneutral = SimpleNamespace(probs=neutral.probs, logProbs=neutral.logProbs, propSizes=neutral.propSizes,
                               spect=dict(neutral.spect), sampProps=dict(neutral.sampProps))
    rsel = SimpleNamespace(normProbs={k: sel.get(*k) for k in sel.classProbs})
    rgrid = SimpleNamespace(x=list(grid.x), A=list(grid.A), abeta=list(grid.abeta))
    return rdata, rneutral, rsel, rgrid


def test_problem_from_reference_objects_is_identical():
    """build_problem accepts the reference's objects (what the calcBaller drop-in relies on): from objects with
    only the reference's attributes it builds the same problem as from the product's own."""
    from ballermixplus_b200.problem import build_problem
    argv, _ = util.scan_cases()['Example1_B2maf']
    opt, data, neutral, grid, sel = util.host_objects(argv)
    rdata, rneutral, rsel, rgrid = _reference_shaped(data, neutral, grid, sel)
    assert not hasattr(rneutral, 'class_tables') and not hasattr(rsel, 'classProbs')
    a, oa = build_problem(rdata, rneutral, rsel, rgrid)
    b, ob = build_problem(data, neutral, sel, grid)
    for f in ('genpos', 'cls', 'G', 'SP', 'A'):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert (oa.A, oa.x, oa.a) == (ob.A, ob.x, ob.a)


def test_reference_calcballer_vs_oracle_on_strided_centres():
    """The reference's own calcBaller rows (its output for `-w 15 -s 7.5`, tests/golden/gen/ex1_B2_w15_s7p5.txt,
    which evaluates centre i on sites [i-15, i+16]) against the numpy oracle fed objects shaped like the
    reference's, on four centres across the chromosome: both ends (windows clipped at 0 and at the last site) and
    two interior centres.  Only centres on that output's 7.5-site stride have a reference row, so centres off the
    stride are not covered here."""
    from oracle import oracle_np
    argv, gold = util.scan_cases()['ex1_B2_w15_s7p5']
    rdata, rneutral, rsel, rgrid = _reference_shaped(*util.host_objects(argv)[1:])
    with open(gold) as fh:
        rows = {int(f[0]): f for f in (line.rstrip('\n').split('\t') for line in fh.readlines()[1:])}
    A, x, a = list(set(rgrid.A)), list(set(rgrid.x)), list(set(rgrid.abeta))
    for i in (0, 105, 375, 750):
        want = rows[int(rdata.position[i])]
        assert float(want[1]) == rdata.genPos[i]
        lo, hi = max(0, i - 15), min(rdata.numSites - 1, i + 16)
        got = oracle_np.calc_baller(lo, hi, rdata.genPos[i], rdata.genPos, rneutral.probs, rneutral.logProbs,
                                    rneutral.propSizes, rsel.normProbs, A, x, a)
        assert [float(v) for v in want[3:6]] + [int(want[6])] == got[1:]
        assert abs(float(want[2]) - got[0]) <= 1e-12 * max(1., abs(float(want[2])))
