"""Targeted scans (``--targets FILE``): scan only the rows whose centre lies in listed intervals (DESIGN.md §3.13).

The file holds one target per line, ``name start end`` separated by whitespace:

  * ``name`` is an input's file name (``os.path.basename`` of ``-i``, or of a listed input with ``--inputList``);
  * ``start`` and ``end`` are inclusive, in the units of the main file's physPos column, and compared as numbers
    (``--noCenter`` prints fractional midpoints);
  * blank lines, lines starting with '#' and a first non-comment line whose first field is ``input`` (a header) are
    skipped, and fields after the third are ignored, so a ``--regions`` file (columns ``input start_physPos
    end_physPos ...``) is a targets file as written;
  * targets may overlap and come in any order: a row is kept once if any target of its input covers it.

A row of the full plan is kept when its physPos (``ScanPlan.phys``: the site's position, or the ``--noCenter``
midpoint, gap rows included) lies in a target of its input.  The scan treats a row that is not kept as it treats a
gap row, and the writers then drop it (scan.py).

Pure numpy.
"""
import math

import numpy as np


class Targets:
    """The targets of one file, by input name: ``keep(name, plan)`` selects the rows of a plan."""

    def __init__(self, path, intervals):
        self.path = path
        self._by_name = {}
        for name, iv in intervals.items():
            iv = np.array(sorted(iv), dtype=np.float64).reshape(-1, 2)
            # sorted by start; reach[k] = the largest end among the first k + 1 targets
            self._by_name[name] = (iv[:, 0], np.maximum.accumulate(iv[:, 1]))

    def keep(self, name, plan):
        """bool [rows]: the rows of ``plan`` (an input named ``name``) whose physPos lies in one of its targets."""
        pos = plan.phys()
        if name not in self._by_name:
            return np.zeros(len(pos), bool)
        start, reach = self._by_name[name]
        k = np.searchsorted(start, pos, 'right') - 1            # last target starting at or before pos
        return (k >= 0) & (reach[np.maximum(k, 0)] >= pos)


def read_targets(path, names):
    """Parse a targets file for a run whose inputs are named ``names`` -> Targets.  Raises ValueError when the file
    cannot be read, when it holds no target, and, naming the line, at the first line with fewer than three fields, a
    start or end that is not a finite number, start > end, or a name that is no input of the run."""
    names = set(names)
    intervals = {}
    header_done = False
    try:
        with open(path) as fh:
            lines = fh.readlines()
    except (OSError, UnicodeDecodeError) as exc:
        raise ValueError(f'--targets: cannot read {path}: {exc}') from None
    for n, line in enumerate(lines, 1):
        f = line.split()
        if not f or f[0].startswith('#'):
            continue
        if not header_done:
            header_done = True
            if f[0] == 'input':
                continue
        where = f'--targets {path}, line {n}'
        if len(f) < 3:
            raise ValueError(f'{where}: expected "name start end", got {line.strip()!r}')
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
        intervals.setdefault(f[0], []).append((start, end))
    if not intervals:
        raise ValueError(f'--targets {path} holds no target')
    return Targets(path, intervals)


def kept_line(name, keep):
    """Console line: how many of an input's planned rows the targets keep."""
    return f'--targets: {name}: {int(np.count_nonzero(keep))} of {len(keep)} planned rows kept'
