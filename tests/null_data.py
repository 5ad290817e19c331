"""Seeded neutral-replicate inputs for the --null tests (not product code): sites whose (k, n) classes are
resampled from tests/golden/data/synth_n200.txt, so that every class is in gen/synth_n200_spect.txt."""
import os

import numpy as np

import util

SRC = os.path.join(util.GOLD, 'data', 'synth_n200.txt')
SPECT = os.path.join(util.GOLD, 'gen', 'synth_n200_spect.txt')

#: flags of the four window modes: product keyword arguments (Scan / make_plan) and CLI argv
MODES = {
    'default': (dict(), []),
    'w': (dict(r=20), ['-w', '20']),
    'fixWinSize': (dict(fixSize=True, r=200000, phys=True), ['--fixWinSize', '-w', '200000', '--usePhysPos']),
    'noCenter': (dict(fixSize=True, r=200000, s=20000, phys=True, noCenter=True),
                 ['--fixWinSize', '--noCenter', '-w', '200000', '-s', '20000', '--usePhysPos']),
}


def write_input(path, n_sites, rng, min_k=1, span=3_000_000):
    rows = np.loadtxt(SRC, skiprows=1)
    rows = rows[rows[:, 2] >= min_k]
    pick = rows[rng.integers(0, len(rows), n_sites)]
    pos = np.sort(rng.choice(np.arange(1, span), n_sites, replace=False))
    with open(path, 'w') as fh:
        fh.write('physPos\tgenPos\tx\tn\n')
        for p, k, n in zip(pos, pick[:, 2].astype(int), pick[:, 3].astype(int)):
            fh.write(f'{p}\t{float(p) * 1e-8!r}\t{k}\t{n}\n')
    return path


def make_replicates(d, n_reps=3, n_sites=150, seed=0, subdir='reps'):
    """n_reps replicate files under d/subdir, listed (relative paths, a comment and a blank line) in
    d/null.txt; replicate 1 has no site with k < 3, so its minCount differs from the others'."""
    rng = np.random.default_rng(seed)
    os.makedirs(os.path.join(d, subdir), exist_ok=True)
    names = []
    for r in range(n_reps):
        name = os.path.join(subdir, f'rep{r}.txt')
        write_input(os.path.join(d, name), n_sites, rng, min_k=3 if r == 1 else 1)
        names.append(name)
    lst = os.path.join(d, 'null.txt')
    with open(lst, 'w') as fh:
        fh.write('# neutral replicates\n\n' + '\n'.join(names) + '\n')
    return lst, [os.path.join(d, n) for n in names]
