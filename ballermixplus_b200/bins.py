"""Binned neutral spectra (``--spectBins LIST``, ``--binMap MAP``): each site's neutral probabilities from the
spectrum of its bin (DESIGN.md §3.15).

  * LIST has one bin per line, ``label path``: ``path`` (relative to LIST) is a spectrum or configuration file, read
    by ``NeutralSFS`` with the run's --noFreq/--MAF/--noSub and its checks.  Blank and '#' lines are skipped.
  * MAP has one interval per line, ``name start end label``, with the parsing rules of ``--targets`` (targets.py):
    ``name`` is an input's file name, ``start`` and ``end`` are inclusive physPos values compared as numbers, blank
    and '#' lines, a first line starting with ``input`` and fields after the fourth are skipped.
  * A site's bin is the label of the interval of its input covering its physPos; a site no interval covers uses
    --spect (bin 0).  Two intervals of one input that overlap with different labels are refused.

Per site, g_i = spect_bin(i)(k_i, n_i) and P_i = sampProps_bin(i)(n_i); the selection rows S(k, n; x, a) do not
change.  The scan only sees classes, so binning only means more classes: they are keyed (k, n, bin), and ordered
by (bin, n, k), so a map that puts every site in bin 0 builds the unbinned problem bit for bit.

Pure numpy.
"""
import math
import os

import numpy as np

from .neutral import NeutralSFS


def read_spect_bins(path):
    """Parse a --spectBins list -> [(label, spectrum path)], paths relative to the list.  Raises ValueError when the
    list cannot be read or holds no bin, and, naming the line, at a line without two fields, a label given twice or
    a spectrum file that does not exist."""
    try:
        with open(path) as fh:
            lines = fh.readlines()
    except (OSError, UnicodeDecodeError) as exc:
        raise ValueError(f'--spectBins: cannot read {path}: {exc}') from None
    base = os.path.dirname(os.path.abspath(path))
    out, seen = [], set()
    for n, line in enumerate(lines, 1):
        f = line.split()
        if not f or f[0].startswith('#'):
            continue
        where = f'--spectBins {path}, line {n}'
        if len(f) != 2:
            raise ValueError(f'{where}: expected "label path", got {line.strip()!r}')
        label, spect = f[0], os.path.join(base, f[1])
        if label in seen:
            raise ValueError(f'{where}: label {label!r} is given twice')
        if not os.path.isfile(spect):
            raise ValueError(f'{where}: {spect} is not a file')
        seen.add(label)
        out.append((label, spect))
    if not out:
        raise ValueError(f'--spectBins {path} holds no bin')
    return out


class BinMap:
    """The intervals of a --binMap file by input name: ``site_bins(name, position)`` gives each site's bin, 0 for a
    site no interval covers and ``labels.index(label) + 1`` otherwise."""

    def __init__(self, path, labels, intervals):
        self.path, self.labels = path, list(labels)
        self._by_name = {}
        for name, iv in intervals.items():
            iv = sorted(iv, key=lambda v: (v[0], v[1]))
            merged = []                              # disjoint after merging same-label overlaps
            for start, end, b, line in iv:
                if merged and start <= merged[-1][1]:
                    if merged[-1][2] != b:
                        raise ValueError(f'--binMap {path}, line {line}: {name} {start:g}..{end:g} overlaps an '
                                         f'interval with label {self.labels[merged[-1][2] - 1]!r}')
                    merged[-1][1] = max(merged[-1][1], end)
                else:
                    merged.append([start, end, b])
            m = np.array(merged, dtype=np.float64).reshape(-1, 3)
            self._by_name[name] = (m[:, 0], m[:, 1], m[:, 2].astype(np.int32))

    def site_bins(self, name, position):
        """int32 [N]: the bin of every site of the input named ``name`` at physPos ``position``."""
        pos = np.asarray(position, dtype=np.float64)
        if name not in self._by_name:
            return np.zeros(len(pos), np.int32)
        start, end, b = self._by_name[name]
        k = np.searchsorted(start, pos, 'right') - 1
        kk = np.maximum(k, 0)
        return np.where((k >= 0) & (end[kk] >= pos), b[kk], 0).astype(np.int32)

    def used_labels(self):
        return sorted({int(b) for _, _, bs in self._by_name.values() for b in bs})


def read_bin_map(path, names, labels):
    """Parse a --binMap file for a run whose inputs are named ``names`` and whose bins are ``labels`` -> BinMap.
    Raises ValueError when the file cannot be read or holds no interval, and, naming the line, at a line with
    fewer than four fields, a start or end that is not a finite number, start > end, a name that is no input of
    the run, a label missing from --spectBins, and two overlapping intervals of one input with different labels."""
    names, index = set(names), {lab: i + 1 for i, lab in enumerate(labels)}
    intervals = {}
    header_done = False
    try:
        with open(path) as fh:
            lines = fh.readlines()
    except (OSError, UnicodeDecodeError) as exc:
        raise ValueError(f'--binMap: cannot read {path}: {exc}') from None
    for n, line in enumerate(lines, 1):
        f = line.split()
        if not f or f[0].startswith('#'):
            continue
        if not header_done:
            header_done = True
            if f[0] == 'input':
                continue
        where = f'--binMap {path}, line {n}'
        if len(f) < 4:
            raise ValueError(f'{where}: expected "name start end label", got {line.strip()!r}')
        try:
            start, end = float(f[1]), float(f[2])
        except ValueError:
            start = end = math.nan
        if not (math.isfinite(start) and math.isfinite(end)):
            raise ValueError(f'{where}: start and end must be finite numbers, got {f[1]!r} and {f[2]!r}')
        if start > end:
            raise ValueError(f'{where}: start {f[1]} is after end {f[2]}')
        if f[0] not in names:
            raise ValueError(f'{where}: {f[0]!r} is not an input of this run (inputs: {", ".join(sorted(names))})')
        if f[3] not in index:
            raise ValueError(f'{where}: label {f[3]!r} is not in --spectBins (labels: {", ".join(labels)})')
        intervals.setdefault(f[0], []).append((start, end, index[f[3]], n))
    if not intervals:
        raise ValueError(f'--binMap {path} holds no interval')
    return BinMap(path, labels, intervals)


def binned_classes(count, total, site_bin):
    """Unique (k, n, bin) classes -> (class_k, class_n, class_bin int64[C], cls int32[N]), sorted by (bin, n, k).
    With every site in bin 0 these are ``neutral.site_classes``'s classes in its order."""
    count = np.asarray(count, dtype=np.int64)
    total = np.asarray(total, dtype=np.int64)
    site_bin = np.asarray(site_bin, dtype=np.int64)
    if count.size == 0:
        z = np.zeros(0, np.int64)
        return z, z, z, np.zeros(0, np.int32)
    if count.min() < 0 or total.min() < 0:
        raise ValueError('negative allele count or sample size in input')
    kmax, nmax = int(count.max()) + 1, int(total.max()) + 1
    key = (site_bin * nmax + total) * kmax + count
    uniq, inv = np.unique(key, return_inverse=True)
    return uniq % kmax, (uniq // kmax) % nmax, uniq // (kmax * nmax), inv.reshape(-1).astype(np.int32)


class BinnedNeutral:
    """The neutral model of a binned run: bin 0 is --spect, bin b >= 1 the b-th --spectBins file, and ``map`` says
    which bin each site is in.  ``class_tables(k, n, bin)`` gives G and P of classes keyed (k, n, bin)."""

    def __init__(self, spect0, bins, binmap):
        self.spects = [spect0] + [sfs for _, sfs in bins]
        self.labels = [label for label, _ in bins]
        self.map = binmap

    @classmethod
    def read(cls, spectfile, bins, binmap, nofreq, MAF, nosub):
        spect0 = NeutralSFS(spectfile, nofreq, MAF, nosub)
        return cls(spect0, [(label, NeutralSFS(p, nofreq, MAF, nosub)) for label, p in bins], binmap)

    def site_bins(self, name, position):
        return self.map.site_bins(name, position)

    def class_tables(self, class_k, class_n, class_bin=None):
        """(G[C], P[C]) from each class's bin (bin 0 without ``class_bin``); a (k, n) missing from its bin's
        spectrum gets NeutralSFS's message and exit."""
        class_bin = np.zeros(len(class_k), np.int64) if class_bin is None else np.asarray(class_bin)
        G, P = np.empty(len(class_k)), np.empty(len(class_k))
        for b in np.unique(class_bin):
            m = class_bin == b
            G[m], P[m] = self.spects[int(b)].class_tables(np.asarray(class_k)[m], np.asarray(class_n)[m])
        return G, P

    def get_neut_probs(self, data):
        """Check every class of ``data`` (its ``siteBin``) against its bin's spectrum, as NeutralSFS does."""
        ck, cn, cb, _ = binned_classes(data.count, data.total, data.siteBin)
        self.class_tables(ck, cn, cb)


def attach(data, neutral, name):
    """Give ``data`` the bins of its sites (``data.siteBin``) when ``neutral`` is binned; returns ``data``."""
    if isinstance(neutral, BinnedNeutral):
        data.siteBin = neutral.site_bins(name, data.position)
    return data
