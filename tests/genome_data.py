"""Seeded multi-input ("genome") test data for the --inputList tests (not product code): chromosomes whose sites are
resampled from tests/golden/data/synth_mixed_n.txt (sample sizes 48 and 50), so that every (k, n) class is in
gen/synth_mixed_n_spect.txt."""
import os

import numpy as np

import util

SRC = os.path.join(util.GOLD, 'data', 'synth_mixed_n.txt')
SPECT = os.path.join(util.GOLD, 'gen', 'synth_mixed_n_spect.txt')

#: (file name, sites, sample sizes drawn from, smallest k, seed): very different sizes, sample sizes 48, 50 and
#: both, and one input without k < 3 so that its derived minCount differs from the others'
CHROMS = [('chr1.txt', 700, (48, 50), 1, 1), ('chr2.txt', 40, (50,), 1, 2), ('chr3.txt', 260, (48,), 3, 3),
          ('chrX.txt', 9, (48, 50), 1, 4)]


def write_chrom(path, n_sites, sizes, min_k, seed, span=4_000_000, hole=None):
    """One input file; ``hole`` = (start, end) of a stretch of physical positions without sites (gap rows of a
    --noCenter scan)."""
    rng = np.random.default_rng(seed)
    rows = np.loadtxt(SRC, skiprows=1)
    rows = rows[(rows[:, 2] >= min_k) & np.isin(rows[:, 3], sizes)]
    pick = rows[rng.integers(0, len(rows), n_sites)]
    cand = np.arange(1, span)
    if hole is not None:
        cand = cand[(cand < hole[0]) | (cand >= hole[1])]
    pos = np.sort(rng.choice(cand, n_sites, replace=False))
    with open(path, 'w') as fh:
        fh.write('physPos\tgenPos\tx\tn\n')
        for p, k, n in zip(pos, pick[:, 2].astype(int), pick[:, 3].astype(int)):
            fh.write(f'{p}\t{float(p) * 1e-8!r}\t{k}\t{n}\n')
    return path


def make_genome(d, chroms=CHROMS, hole=(1_000_000, 2_500_000)):
    """The CHROMS under d/in/, listed (relative paths, a comment and a blank line) in d/genome.txt -> (list,
    paths).  Every chromosome has the same stretch without sites."""
    os.makedirs(os.path.join(d, 'in'), exist_ok=True)
    paths = [write_chrom(os.path.join(d, 'in', name), n, sizes, k, seed, hole=hole)
             for name, n, sizes, k, seed in chroms]
    lst = os.path.join(d, 'genome.txt')
    with open(lst, 'w') as fh:
        fh.write('# chromosomes\n\n' + '\n'.join(os.path.join('in', name) for name, *_ in chroms) + '\n')
    return lst, paths


def make_replicates(d, n_reps=3, n_sites=200, seed=50):
    """Neutral replicates under d/reps/, listed in d/null.txt -> list path."""
    os.makedirs(os.path.join(d, 'reps'), exist_ok=True)
    names = []
    for r in range(n_reps):
        name = os.path.join('reps', f'rep{r}.txt')
        write_chrom(os.path.join(d, name), n_sites, (48, 50), 3 if r == 1 else 1, seed + r)
        names.append(name)
    lst = os.path.join(d, 'null.txt')
    with open(lst, 'w') as fh:
        fh.write('\n'.join(names) + '\n')
    return lst
