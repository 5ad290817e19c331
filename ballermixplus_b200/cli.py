"""Command line -- SURVEY.md §8 rows a8/b: the flag surface of BalLeRMix+_v1.py.

Same flags, defaults, precedence and console messages as the reference's ``main``
(/root/reference/BalLeRMix+_v1.py:715-802); one extra flag, ``--device``, picks the
GPU, ``--support`` / ``--supportDrop`` write support intervals of A_hat, x_hat and s_hat (support.py), and
``--null`` / ``--pvalues`` write empirical p-values from scans of neutral replicates (null.py), ``--refine``
/ ``--refineSteps`` write the rows again at the best point of a finer grid around each maximum (refine.py),
``--inputList`` scans one input per chromosome in one run (scan.GenomeScan), and ``--regions`` / ``--threshold``
write one line per run of rows above a CLR cut, with its peak, a support interval for the target's position and,
with ``--null``, a region p-value (regions.py), ``--targets`` scans only the rows whose centre lies in listed
intervals, every output a line-for-line subset of the full scan's (targets.py), and ``--balPos`` writes each row's
maximum over the alpha >= 1 and the alpha < 1 half of the grid from the same scan (balpos.py), and ``--spectBins`` /
``--binMap`` give each site the neutral spectrum of its bin (bins.py).
Differences, all on paths where the reference raises (SURVEY.md appendix A.2,
DESIGN.md "flags without a reference behaviour"): ``--rangeA``, ``--findPos`` and
``--minCount`` with ``--noFreq`` work here.
"""
import argparse
import os
import sys
from datetime import datetime

from .balpos import check_grid
from .bins import BinnedNeutral, attach, read_bin_map, read_spect_bins
from .grids import Grids
from .helpers import getConfig, getSpect, getSpectBinned
from .inputs import InputData
from .neutral import NeutralSFS
from .null import read_list
from .refine import DEFAULT_STEPS, MAX_STEPS, check_steps
from .regions import check_threshold
from .scan import REGIONS_NEED_A_CUT, GenomeScan, Scan, check_regions_file, input_list, list_outputs, names_one_of
from .selection import NormalizedBetaBinom
from .support import DEFAULT_DROP, check_drop
from .targets import read_targets


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
                   help='Drop in T = 2 log LR units that defines the --support intervals and the position '
                        f'interval of --regions. Default {DEFAULT_DROP} (the chi-square(1) 0.95 quantile).')
    p.add_argument('--null', dest='null', default=None,
                   help='Text file listing neutral replicate inputs, one path per line (relative to the list; '
                        'blank and # lines skipped). Every replicate is scanned with exactly the flags and '
                        '--spect of this run, and --pvalues gets each row\'s empirical p-value against the '
                        'pooled replicate CLRs, p = (1 + #{null >= CLR}) / (1 + N_null). The p-values are only as '
                        'good as the neutral model the replicates were simulated under, and they are not '
                        'corrected for multiple testing (the printed quantiles of the per-replicate maximum CLR '
                        'give a region-level threshold, which --regions applies). Needs --pvalues.')
    p.add_argument('--pvalues', dest='pvalues', default=None,
                   help='With --null: write FILE with physPos, genPos, CLR and p_value per output row.')
    p.add_argument('--refine', dest='refine', default=None,
                   help='Also write FILE, in the output\'s format: every row with CLR > 0 whose best point on a grid '
                        '--refineSteps times finer (geometric steps for A and alpha, arithmetic for x), inside a box '
                        'of one coarse step either side of the row\'s maximum, beats its CLR takes that point; every '
                        'other row is copied. A refined CLR is a maximum over more points, so it is biased upward '
                        'relative to the coarse CLR and must not be compared with --null CLRs; it is still a grid '
                        'maximum, not a continuous MLE. One GPU only (not under torchrun).')
    p.add_argument('--inputList', dest='inputList', action='store_true', default=False,
                   help='Scan a genome in one run: -i names a text file listing one input per line (one per '
                        'chromosome; relative to the list, blank and # lines skipped), and -o, --support, '
                        '--pvalues and --refine name existing directories. Input chr7.txt writes DIR/chr7.txt, '
                        'the file a run on chr7.txt alone with the same flags writes. The --null replicates are '
                        'scanned once for all inputs. Under torchrun the whole genome is sharded over the GPUs. '
                        'With --getSpect or --getConfig: the helper file of all listed inputs together.')
    p.add_argument('--refineSteps', dest='refineSteps', type=_steps, default=DEFAULT_STEPS,
                   help=f'Fine points per coarse step of --refine, 1 to {MAX_STEPS}. Default {DEFAULT_STEPS}.')
    p.add_argument('--regions', dest='regions', default=None,
                   help='Also write FILE: one line per region, a maximal run of consecutive rows (no gap row) with '
                        'CLR >= the cut, giving its first and last physPos, its row count, its peak row (largest CLR, '
                        'first on ties) with the peak\'s physPos, genPos, CLR, x_hat, s_hat, A_hat and nSites as the '
                        'output prints them, and pos_lo / pos_hi: the rows around the peak whose CLR is within '
                        '--supportDrop of the peak\'s. Each CLR is the maximum over A, x and alpha at its centre, so '
                        'this is a support interval for the target\'s position, of a composite likelihood: not a '
                        'calibrated confidence interval. With --null, p_region = (1 + #{replicates whose maximum CLR '
                        '>= the peak CLR}) / (1 + R): the chance that a neutral replicate holds a row this high, a '
                        'family-wise p-value only for a sequence of the replicates\' length, not scaled to the '
                        'genome; NA without --null. The cut is --threshold, or with --null the 0.95 quantile of the '
                        'per-replicate maximum CLR. With --inputList: one FILE for the whole genome. Works under '
                        'torchrun; no other output changes. With --targets, a row that is not kept ends a region and '
                        'stops a position interval, as a gap row does, so regions are cut at the target edges.')
    p.add_argument('--threshold', dest='threshold', type=_threshold, default=None,
                   help='With --regions: the CLR cut, a finite number > 0. Default with --null: the 0.95 quantile '
                        'of the per-replicate maximum CLR.')
    p.add_argument('--targets', dest='targets', default=None,
                   help='Scan only the rows whose physPos lies in a target of FILE: one target per line, "name start '
                        'end", name the input\'s file name (with --inputList, of a listed input), start and end '
                        'inclusive physPos values compared as numbers; blank and # lines, a header line starting with '
                        '"input" and fields after the third are skipped, so a --regions file is a targets file as '
                        'written. Targets may overlap. Every output file holds the header and, in order, exactly the '
                        'lines the same run without --targets writes at the kept rows (DESIGN.md §3.13). --regions '
                        'is the exception: a row that is not kept ends a region and stops a '
                        'position interval, as a gap row does, so a region or interval that reaches the first or last '
                        'kept row of a target is cut there. The --null replicates are still scanned in full.')
    p.add_argument('--balPos', dest='balPos', default=None,
                   help='Also write FILE: per output row, the row\'s maximum over the balancing half of the grid (alpha '
                        '>= 1: CLR_bal, x_bal, s_bal, A_bal, nSites_bal) and over the sweep half (alpha < 1: CLR_pos '
                        '...), each by the reference\'s rule restricted to its points and printed as the output prints '
                        'its row; max(CLR_bal, CLR_pos) is the row\'s CLR. Both come from the same scan as the output. '
                        'Each half keeps this run\'s A and x grids: with the default x grid the bal half is the '
                        '--findBal grid, but the pos half is not the --findPos statistic, which also changes the x grid '
                        '(0.1..0.9). CLR_bal - CLR_pos is a difference of composite-likelihood maxima that ranks how '
                        'clearly a row prefers one half; it is not a calibrated test. Needs alpha values on both sides '
                        'of 1 (not --fixAlpha, --findBal or --findPos). With --inputList: an existing directory, input '
                        'chr7.txt writes DIR/chr7.txt. With --support the halves take a second scan. Works under '
                        'torchrun; no other output changes.')
    p.add_argument('--spectBins', dest='spectBins', default=None,
                   help='With --binMap: text file with one bin per line, "label path", path (relative to the list) a '
                        'spectrum or configuration file read as --spect is; blank and # lines skipped.')
    p.add_argument('--binMap', dest='binMap', default=None,
                   help='With --spectBins: one interval per line, "name start end label", name the input\'s file name '
                        '(with --inputList, of a listed input; or of a --null replicate), start and end inclusive physPos '
                        'values; blank and # lines, a header line starting with "input" and fields after the fourth are '
                        'skipped.  A site covered by an interval takes the neutral spectrum of its label (g and the '
                        'sample-size proportion of its k and n in that file), every other site --spect; two overlapping '
                        'intervals of one input with different labels are refused.  With --getSpect or --getConfig '
                        '(no --spectBins needed): write --spect from the sites no interval covers and --spect.LABEL from '
                        'the sites of each label, each only when it has sites (no --spect file when the map covers '
                        'every site).')
    return p


def _steps(text):
    try:
        return check_steps(text)
    except ValueError as exc:
        raise argparse.ArgumentTypeError(str(exc)) from None


def _threshold(text):
    try:
        return check_threshold(text)
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
    if opt.threshold is not None and opt.regions is None:
        parser.error('--threshold needs --regions')
    if opt.regions is not None and opt.threshold is None and opt.null is None:
        parser.error(REGIONS_NEED_A_CUT)

    if opt.balPos is not None:
        _check_balpos(parser, opt)

    inputs = opt.infile
    if opt.inputList:
        inputs = _check_list_mode(parser, opt)
    targets = _check_targets(parser, opt, inputs)
    binned = _check_bins(parser, opt, inputs)

    if (opt.getSpec or opt.getConfig) and binned is not None:
        print('You\'ve chosen to generate binned helper files...')
        getSpectBinned(inputs, opt.spectfile, opt.MAF, opt.nosub, binned, config=opt.getConfig)
        sys.exit()
    if opt.getSpec:
        print('You\'ve chosen to generate site frequency spectrum...')
        print('Concatenated input: %s \nSpectrum file: %s' % (opt.infile, opt.spectfile))
        getSpect(inputs, opt.spectfile, opt.MAF, opt.nosub)
        sys.exit()
    elif opt.getConfig:
        print('You\'ve chosen to generate the substitution-polymorphism configuration...')
        print('Concatenated input: %s \nConfiguration file: %s' % (opt.infile, opt.spectfile))
        getConfig(inputs, opt.spectfile)
        sys.exit()
    if opt.inputList:
        _main_list(opt, inputs, targets, binned)
        return

    print(f'\n{datetime.now()}. Reading input from {opt.infile}')
    data = InputData(opt.infile, opt.nofreq, opt.MAF, opt.nosub, opt.minCount, phys=opt.phys,
                     Rrate=opt.Rrate)
    Neutral = _neutral(opt, binned)
    attach(data, Neutral, os.path.basename(opt.infile))

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
         refine_steps=opt.refineSteps, regions=opt.regions, threshold=opt.threshold,
         input_name=os.path.basename(opt.infile), targets=targets, balpos=opt.balPos)
    print(f'\n{datetime.now()}. Pipeline finished.')


def _check_list_mode(parser, opt):
    """``--inputList``: the inputs the list names; a bad list or output directory fails before any input is
    read."""
    try:
        inputs = input_list(opt.infile)
    except (OSError, ValueError) as exc:
        parser.error(str(exc))
    if opt.getSpec or opt.getConfig:
        return inputs
    if opt.outfile is None:
        parser.error('--inputList needs -o DIR')
    for flag, d in (('-o', opt.outfile), ('--support', opt.support), ('--pvalues', opt.pvalues),
                    ('--refine', opt.refine), ('--balPos', opt.balPos)):
        if d is not None and not os.path.isdir(d):
            parser.error(f'--inputList: {flag} {d} is not an existing directory')
    try:
        files = list_outputs(inputs, out=opt.outfile, support=opt.support, pvalues=opt.pvalues, refine=opt.refine,
                             balpos=opt.balPos)
        if opt.regions is not None:
            reads = [opt.infile, opt.spectfile] + ([opt.null] + read_list(opt.null) if opt.null else [])
            check_regions_file(opt.regions, inputs, files, reads)
    except ValueError as exc:
        parser.error(str(exc))
    return inputs


def _check_balpos(parser, opt):
    """``--balPos``: refused before any input is read with --getSpect or --getConfig, for a grid with no alpha on
    one side of 1, and (one input) for a file the run reads or writes; --inputList checks its directory with the
    other output directories (``_check_list_mode``)."""
    if opt.getSpec or opt.getConfig:
        parser.error('--balPos writes rows of a scan; --getSpect and --getConfig do not scan')
    try:
        check_grid(Grids(opt.x, opt.abeta, opt.bal, opt.pos, opt.seqA, opt.listA).abeta)
    except ValueError as exc:
        parser.error(str(exc))
    if opt.inputList:
        return
    others = [opt.infile, opt.spectfile, opt.outfile, opt.support, opt.pvalues, opt.refine, opt.regions, opt.targets,
              opt.null] + (read_list(opt.null) if opt.null else [])
    if names_one_of(opt.balPos, others):
        parser.error(f'--balPos {opt.balPos} is a file this run reads or writes')


def _check_targets(parser, opt, inputs):
    """``--targets``: the parsed targets file (None without the option).  Refused before any input is read with
    --getSpect or --getConfig, when the run writes the file, and when the file is bad (targets.read_targets)."""
    if opt.targets is None:
        return None
    if opt.getSpec or opt.getConfig:
        parser.error('--targets selects the rows of a scan; --getSpect and --getConfig do not scan')
    if opt.inputList:
        names = [os.path.basename(p) for p in inputs]
        files = list_outputs(inputs, out=opt.outfile, support=opt.support, pvalues=opt.pvalues, refine=opt.refine,
                             balpos=opt.balPos)
        written = [f for fs in files.values() for f in fs] + [opt.regions]
    else:
        names = [os.path.basename(opt.infile)]
        written = [opt.outfile, opt.support, opt.pvalues, opt.refine, opt.regions, opt.balPos]
    if names_one_of(opt.targets, written):
        parser.error(f'--targets {opt.targets} is a file this run writes')
    try:
        return read_targets(opt.targets, names)
    except ValueError as exc:
        parser.error(str(exc))


def _check_bins(parser, opt, inputs):
    """``--spectBins`` / ``--binMap``: the parsed map (None without them), refused before any input is read when
    one comes without the other (with --getSpect/--getConfig only the map is needed), when the run writes either
    file and when either is bad (bins.read_spect_bins, bins.read_bin_map).  Keeps the list's bins in opt._bins."""
    helper = opt.getSpec or opt.getConfig
    if opt.binMap is None:
        if opt.spectBins is not None:
            parser.error('--spectBins needs --binMap')
        return None
    if opt.spectBins is None and not helper:
        parser.error('--binMap needs --spectBins')
    if opt.inputList:
        names = [os.path.basename(p) for p in inputs]
        written = [] if helper else [f for fs in list_outputs(inputs, out=opt.outfile, support=opt.support,
                                                               pvalues=opt.pvalues, refine=opt.refine,
                                                               balpos=opt.balPos).values() for f in fs]
        written.append(opt.regions)
    else:
        names = [os.path.basename(opt.infile)]
        written = [opt.outfile, opt.support, opt.pvalues, opt.refine, opt.regions, opt.balPos]
    if opt.null is not None:
        names += [os.path.basename(p) for p in read_list(opt.null)]
    try:
        bins = read_spect_bins(opt.spectBins) if opt.spectBins is not None else []
        labels = _map_labels(opt.binMap) if helper and opt.spectBins is None else [label for label, _ in bins]
        if helper:
            written += [opt.spectfile] + [f'{opt.spectfile}.{label}' for label in labels]
        for flag, path in (('--spectBins', opt.spectBins), ('--binMap', opt.binMap)):
            if path is not None and names_one_of(path, written):
                raise ValueError(f'{flag} {path} is a file this run writes')
        for label, path in bins:                # --getSpect/--getConfig would overwrite a listed spectrum
            if names_one_of(path, written):
                raise ValueError(f'--spectBins {opt.spectBins}: the spectrum {path} of bin {label} is a file this '
                                 f'run writes')
        binmap = read_bin_map(opt.binMap, names, labels)
    except ValueError as exc:
        parser.error(str(exc))
    opt._bins = bins
    return binmap


def _map_labels(path):
    """The labels a --binMap file names, in order of first use (--getSpect/--getConfig without --spectBins)."""
    labels = []
    try:
        with open(path) as fh:
            for line in fh:
                f = line.split()
                if len(f) >= 4 and not f[0].startswith('#') and f[0] != 'input' and f[3] not in labels:
                    labels.append(f[3])
    except (OSError, UnicodeDecodeError):
        pass                                    # read_bin_map reports it
    return labels


def _neutral(opt, binned):
    """The run's neutral model: NeutralSFS of --spect, or with a bin map the BinnedNeutral of --spect and the
    --spectBins files."""
    if binned is None:
        return NeutralSFS(opt.spectfile, opt.nofreq, opt.MAF, opt.nosub)
    return BinnedNeutral.read(opt.spectfile, opt._bins, binned, opt.nofreq, opt.MAF, opt.nosub)


def _main_list(opt, inputs, targets=None, binned=None):
    """One run over every listed input (scan.GenomeScan), each read and tabulated as the one-input run reads it."""
    print(f'\n{datetime.now()}. {len(inputs)} inputs listed in {opt.infile}')
    Neutral = _neutral(opt, binned)
    grid = Grids(opt.x, opt.abeta, opt.bal, opt.pos, opt.seqA, opt.listA)
    print('\nOptimizing over x= ' + ', '.join(['%g' % (x) for x in grid.x]))
    print('\n \t alpha= ' + ', '.join([str(a) for a in grid.abeta]))
    print('\n \t A= ' + ', '.join([str(A) for A in grid.A]))

    def read(path):
        print(f'\n{datetime.now()}. Reading input from {path}')
        data = InputData(path, opt.nofreq, opt.MAF, opt.nosub, opt.minCount, phys=opt.phys, Rrate=opt.Rrate)
        attach(data, Neutral, os.path.basename(path))
        Neutral.get_neut_probs(data)
        return data, NormalizedBetaBinom(data, grid, opt.nofreq, opt.MAF, opt.nosub)

    print('\n%s. Start computing likelihood raito...' % (datetime.now()))
    GenomeScan(inputs, read, Neutral, grid, opt.outfile, fixSize=opt.size, r=opt.w, s=opt.step, phys=opt.phys,
               noCenter=opt.noCenter, device=opt.device, support=opt.support, support_drop=opt.supportDrop,
               null=opt.null, pvalues=opt.pvalues, refine=opt.refine, refine_steps=opt.refineSteps,
               regions=opt.regions, threshold=opt.threshold, targets=targets, balpos=opt.balPos)
    print(f'\n{datetime.now()}. Pipeline finished.')


if __name__ == '__main__':
    main()
