"""Helper-file generators -- SURVEY.md §8 row a7.

``getSpect(infile, spectfile, MAF, nosub)`` and ``getConfig(infile, configfile)``
with the reference's signatures (/root/reference/BalLeRMix+_v1.py:645-710).
Integer class counting, then one ``count / float(numSites)`` division per class
at write time, formatted with ``%s`` -- so the files are byte-identical to the
reference's (tests compare against reference-generated fixtures).

Rules kept:
  getSpect (v1:667-710): header skipped; (x, n) = last two columns as ints;
    --MAF folds x > n/2 to n-x (message once); DAF input with x == 0 prints the
    reference's message and exits(0); --noSub skips x == n*(1-MAF) (message
    once; note for --MAF this is x == 0); rows sorted by (x, n).
  getConfig (v1:645-664): x == 0 rows are reported and skipped; per n the pair
    [#substitutions (x == n), #polymorphisms]; rows sorted by n.

``infile`` may also be a list of paths (``--inputList``): the helper file is then the one the concatenation of
the inputs (in list order, first header kept) gives, so a genome-wide spectrum needs no hand-made file.
"""
import os
import sys

import numpy as np

from . import fastio
from .inputs import read_site_table


def _read_xn(infile):
    """(x, n) of every site of `infile`, or, for a list of paths, of the inputs laid end to end in list order:
    the sites of their concatenation with only the first file's header kept (``--inputList``)."""
    if not isinstance(infile, (str, bytes, os.PathLike)):
        parts = [_read_xn(p) for p in infile]
        return (np.concatenate([x for x, _ in parts]).astype(np.int64),
                np.concatenate([n for _, n in parts]).astype(np.int64))
    fast = fastio.read_sites(infile, True, 1.0, strict_columns=True)     # C++ reader; None -> the loop below
    if fast is not None:
        return fast[2], fast[3]
    xs, ns = [], []
    with open(infile, 'r') as fh:
        next(fh, None)
        for line in fh:
            x, n = [int(v) for v in line.strip().split('\t')[2:]]
            xs.append(x)
            ns.append(n)
    return np.array(xs, dtype=np.int64), np.array(ns, dtype=np.int64)


def getConfig(infile, configfile):
    x, n = _read_xn(infile)
    _write_config(x, n, configfile)


def _write_config(x, n, configfile):
    zero = x == 0
    for _ in range(int(zero.sum())):
        print('Please make sure the input has derived allele frequency. Sites with 0 observed '
              'allele count (k=0) will be ignored.\n')
    x, n = x[~zero], n[~zero]
    numSites = int(len(x))
    sizes, inv = np.unique(n, return_inverse=True)
    subs = np.bincount(inv, weights=(x == n), minlength=len(sizes)).astype(np.int64)
    tot = np.bincount(inv, minlength=len(sizes)).astype(np.int64)
    with open(configfile, 'w') as fh:
        for N, s, t in zip(sizes.tolist(), subs.tolist(), tot.tolist()):
            fh.write('%s\t%s\t%s\n' % (N, s / float(numSites), (t - s) / float(numSites)))
    print('Done')


def getSpect(infile, spectfile, MAF, nosub):
    x, n = _read_xn(infile)
    _write_spect(x, n, spectfile, MAF, nosub)


def _bin_sites(infile, binmap):
    """(x, n, bin) of every site of `infile` (or of a list of paths), each site's bin from ``binmap``
    (bins.BinMap) at its physPos: the first column read as the input reader reads it."""
    paths = [infile] if isinstance(infile, (str, bytes, os.PathLike)) else list(infile)
    xs, ns, bs = [], [], []
    for p in paths:
        x, n = _read_xn(p)
        pos = read_site_table(p, True, 1.0)[0]
        xs.append(x); ns.append(n); bs.append(binmap.site_bins(os.path.basename(p), pos))
    return np.concatenate(xs), np.concatenate(ns), np.concatenate(bs)


def getSpectBinned(infile, spectfile, MAF, nosub, binmap, config=False):
    """--getSpect / --getConfig with --binMap: ``spectfile`` from the sites no interval covers and
    ``spectfile.label`` for every label, each only when it has sites and each the file getSpect (getConfig) writes
    for those sites alone -> the files written.  A bin without sites gets no file (it would be empty, which
    NeutralSFS refuses), so ``spectfile`` is not written when the map covers every site."""
    x, n, b = _bin_sites(infile, binmap)
    out = []
    for k in [k for k in range(len(binmap.labels) + 1) if np.any(b == k)]:
        path = spectfile if k == 0 else f'{spectfile}.{binmap.labels[k - 1]}'
        print(f'Bin {binmap.labels[k - 1] if k else "(no interval)"}: {int(np.sum(b == k))} sites -> {path}')
        if config:
            _write_config(x[b == k], n[b == k], path)
        else:
            _write_spect(x[b == k], n[b == k], path, MAF, nosub)
        out.append(path)
    return out


def _write_spect(x, n, spectfile, MAF, nosub):
    if MAF:
        over = x > n / 2
        if np.any(over):
            print('Input data includes non-MAF site/s (frequency >= 0.5) despite choosing to use '
                  'B_maf (with --MAF). These frequencies will be folded for following analyses.')
            x = np.where(over, n - x, x)
        x = np.minimum(x, n - x)
    elif np.any(x == 0):
        print('Please make sure the input has derived allele frequency. Sites with 0 observed '
              'allele count (k=0) should not be included.\n')
        sys.exit()
    if nosub:
        skip = x == (n * (1 - int(bool(MAF))))
        if np.any(skip):
            print('Input includes substitutions despite choosing to use B_0 or B_0maf (with '
                  '--noSub). These sites will not be accounted for.')
            x, n = x[~skip], n[~skip]
    numSites = int(len(x))
    if numSites:
        base = int(x.max()) + 1 if int(x.max()) >= 0 else 1
        xmin = int(x.min())
        key = (x - xmin) * (int(n.max()) + 1) + n          # sorts by (x, n)
        uniq, counts = np.unique(key, return_counts=True)
        stride = int(n.max()) + 1
        rows = [(int(u // stride) + xmin, int(u % stride), int(c)) for u, c in zip(uniq, counts)]
    else:
        rows = []
    with open(spectfile, 'w') as fh:
        for xx, nn, c in rows:
            fh.write('%s\t%s\t%s\n' % (xx, nn, float(c) / float(numSites)))
    print('Done.')
