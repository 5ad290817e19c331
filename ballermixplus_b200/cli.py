"""Command line -- SURVEY.md §8 rows a8/b: the flag surface of BalLeRMix+_v1.py.

Same flags, defaults, precedence and console messages as the reference's ``main``
(/root/reference/BalLeRMix+_v1.py:715-802); one extra flag, ``--device``, picks the
GPU, ``--support`` / ``--supportDrop`` write support intervals of A_hat, x_hat and s_hat (support.py), and
``--null`` / ``--pvalues`` write empirical p-values from scans of neutral replicates (null.py), and ``--refine``
/ ``--refineSteps`` write the rows again at the best point of a finer grid around each maximum (refine.py).
Differences, all on paths where the reference raises (SURVEY.md appendix A.2,
DESIGN.md "flags without a reference behaviour"): ``--rangeA``, ``--findPos`` and
``--minCount`` with ``--noFreq`` work here.
"""
import argparse
import os
import sys
from datetime import datetime

from .grids import Grids
from .helpers import getConfig, getSpect
from .inputs import InputData
from .neutral import NeutralSFS
from .null import read_list
from .refine import DEFAULT_STEPS, MAX_STEPS, check_steps
from .scan import Scan
from .selection import NormalizedBetaBinom
from .support import DEFAULT_DROP, check_drop


def build_parser():
    p = argparse.ArgumentParser()
    p.add_argument('-i', '--input', dest='infile', required=True, help='Path and name of your input file.\n')
    p.add_argument('-o', '--output', dest='outfile', help='Path and name of your output file.\n')
    p.add_argument('--spect', dest='spectfile', required=True,
                   help='Path and name of the allele frequency spectrum file or configuration file.\n')
    p.add_argument('--minCount', dest='minCount', default=1,
                   help='If rare variants are removed from the input, please provide the smallest '
                        'allele count included in the input. Default value is 1.')
    p.add_argument('--getSpect', dest='getSpec', action='store_true', default=False,
                   help='Generate the frequency spectrum file from the concatenated input (-i) into --spect.')
    p.add_argument('--getConfig', dest='getConfig', action='store_true', default=False,
                   help='Generate the substitution/polymorphism configuration file from the '
                        'concatenated input (-i) into --spect.')
    p.add_argument('--findBal', dest='bal', action='store_true', default=False,
                   help='Only look for footprints of balancing selection.')
    p.add_argument('--findPos', dest='pos', action='store_true', default=False,
                   help='Only look for footprints of positive selection.')
    p.add_argument('--noFreq', dest='nofreq', action='store_true', default=False,
                   help='Compute B_1 (ignore allele frequencies).')
    p.add_argument('--noSub', dest='nosub', action='store_true', default=False,
                   help='Do not include substitutions: B_0 or B_0maf.')
    p.add_argument('--MAF', dest='MAF', action='store_true', default=False,
                   help='Use minor allele frequencies: B_2maf or B_0maf.')
    p.add_argument('--usePhysPos', action='store_true', dest='phys', default=False,
                   help='Use physical positions (times --rec) instead of genetic positions.')
    p.add_argument('--rec', dest='Rrate', default=1e-6, type=float,
                   help='Uniform recombination rate in cM/nt (default 1e-6).')
    p.add_argument('--fixWinSize', action='store_true', dest='size', default=False,
                   help='Fix the size (nt) of the sliding windows; give the width with -w.')
    p.add_argument('-w', '--window', dest='w', type=int, default=0,
                   help='Sites flanking the test locus on either side, or the window width in bp with --fixWinSize.')
    p.add_argument('--noCenter', action='store_true', dest='noCenter', default=False,
                   help='Windows not centred on informative sites (needs --fixWinSize -w and --usePhysPos).')
    p.add_argument('-s', '--step', dest='step', type=float, default=1,
                   help='Step size in bp (--noCenter) or in informative sites. Default 1.')
    p.add_argument('--fixX', dest='x', help='Fix the presumed equilibrium frequency.')
    p.add_argument('--fixAlpha', dest='abeta', type=float, default=None,
                   help='Fix the alpha parameter of the beta-binomial distribution.')
    p.add_argument('--rangeA', dest='seqA', help='<Amin>,<Amax>,<Astep> grid for the linkage parameter A.')
    p.add_argument('--listA', dest='listA', help='Comma-separated list of A values.')
    p.add_argument('--device', dest='device', type=int, default=0, help='CUDA device to run the scan on.')
    p.add_argument('--support', dest='support', default=None,
                   help='Also write FILE: per output row, the lowest and highest A, x and s whose profile '
                        'likelihood is within --supportDrop of the row\'s CLR. These are support intervals of a '
                        'composite likelihood: sites are not independent, so they are not calibrated confidence '
                        'intervals. One GPU only (not under torchrun).')
    p.add_argument('--supportDrop', dest='supportDrop', type=_drop, default=DEFAULT_DROP,
                   help='Drop in T = 2 log LR units that defines the --support intervals. Default '
                        f'{DEFAULT_DROP} (the chi-square(1) 0.95 quantile).')
    p.add_argument('--null', dest='null', default=None,
                   help='Text file listing neutral replicate inputs, one path per line (relative to the list; '
                        'blank and # lines skipped). Every replicate is scanned with exactly the flags and '
                        '--spect of this run, and --pvalues gets each row\'s empirical p-value against the '
                        'pooled replicate CLRs, p = (1 + #{null >= CLR}) / (1 + N_null). The p-values are only as '
                        'good as the neutral model the replicates were simulated under, and they are not '
                        'corrected for multiple testing (the printed quantiles of the per-replicate maximum CLR '
                        'give a region-level threshold). Needs --pvalues.')
    p.add_argument('--pvalues', dest='pvalues', default=None,
                   help='With --null: write FILE with physPos, genPos, CLR and p_value per output row.')
    p.add_argument('--refine', dest='refine', default=None,
                   help='Also write FILE, in the output\'s format: every row with CLR > 0 whose best point on a grid '
                        '--refineSteps times finer (geometric steps for A and alpha, arithmetic for x), inside a box '
                        'of one coarse step either side of the row\'s maximum, beats its CLR takes that point; every '
                        'other row is copied. A refined CLR is a maximum over more points, so it is biased upward '
                        'relative to the coarse CLR and must not be compared with --null CLRs; it is still a grid '
                        'maximum, not a continuous MLE. One GPU only (not under torchrun).')
    p.add_argument('--refineSteps', dest='refineSteps', type=_steps, default=DEFAULT_STEPS,
                   help=f'Fine points per coarse step of --refine, 1 to {MAX_STEPS}. Default {DEFAULT_STEPS}.')
    return p


def _steps(text):
    try:
        return check_steps(text)
    except ValueError as exc:
        raise argparse.ArgumentTypeError(str(exc)) from None


def _drop(text):
    try:
        return check_drop(text)
    except ValueError as exc:
        raise argparse.ArgumentTypeError(str(exc)) from None


def main(argv=None):
    argv = sys.argv[1:] if argv is None else list(argv)
    if int(os.environ.get('RANK', '0')) != 0:          # torchrun: only rank 0 talks and writes
        sys.stdout = open(os.devnull, 'w')
    parser = build_parser()
    if len(argv) == 0:
        parser.print_help()
        sys.exit()
    opt = parser.parse_args(argv)
    if opt.support is not None and int(os.environ.get('WORLD_SIZE', '1')) > 1:
        parser.error('--support runs on one GPU; launch without torchrun (WORLD_SIZE > 1)')
    if opt.refine is not None and int(os.environ.get('WORLD_SIZE', '1')) > 1:
        parser.error('--refine runs on one GPU; launch without torchrun (WORLD_SIZE > 1)')
    if (opt.null is None) != (opt.pvalues is None):
        parser.error('--null and --pvalues must be given together')
    if opt.null is not None:
        try:
            read_list(opt.null)             # a bad list fails before any input is read
        except (OSError, ValueError) as exc:
            parser.error(str(exc))

    if opt.getSpec:
        print('You\'ve chosen to generate site frequency spectrum...')
        print('Concatenated input: %s \nSpectrum file: %s' % (opt.infile, opt.spectfile))
        getSpect(opt.infile, opt.spectfile, opt.MAF, opt.nosub)
        sys.exit()
    elif opt.getConfig:
        print('You\'ve chosen to generate the substitution-polymorphism configuration...')
        print('Concatenated input: %s \nConfiguration file: %s' % (opt.infile, opt.spectfile))
        getConfig(opt.infile, opt.spectfile)
        sys.exit()

    print(f'\n{datetime.now()}. Reading input from {opt.infile}')
    data = InputData(opt.infile, opt.nofreq, opt.MAF, opt.nosub, opt.minCount, phys=opt.phys,
                     Rrate=opt.Rrate)
    Neutral = NeutralSFS(opt.spectfile, opt.nofreq, opt.MAF, opt.nosub)

    print(f'\n{datetime.now()}. Initializing...')
    print('Retrieving per-site neutral probabilities...')
    Neutral.get_neut_probs(data)

    grid = Grids(opt.x, opt.abeta, opt.bal, opt.pos, opt.seqA, opt.listA)
    print('\nOptimizing over x= ' + ', '.join(['%g' % (x) for x in grid.x]))
    print('\n \t alpha= ' + ', '.join([str(a) for a in grid.abeta]))
    print('\n \t A= ' + ', '.join([str(A) for A in grid.A]))

    Sel_Probs = NormalizedBetaBinom(data, grid, opt.nofreq, opt.MAF, opt.nosub)

    print('\n%s. Start computing likelihood raito...' % (datetime.now()))
    Scan(data, Neutral, Sel_Probs, grid, opt.outfile, fixSize=opt.size, r=opt.w, s=opt.step,
         phys=opt.phys, noCenter=opt.noCenter, device=opt.device, support=opt.support,
         support_drop=opt.supportDrop, null=opt.null, pvalues=opt.pvalues, refine=opt.refine,
         refine_steps=opt.refineSteps)
    print(f'\n{datetime.now()}. Pipeline finished.')


if __name__ == '__main__':
    main()
