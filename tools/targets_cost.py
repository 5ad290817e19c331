#!/usr/bin/env python3
"""What ``--targets`` saves on a detailed rescan: the genome of tools/genome_cli_cost.py (22 chromosomes of
bench.make_genome, the genome spectrum from ``--getSpect --inputList``, every site a centre, ``--usePhysPos --rec 1e-8
--rangeA 1000,10900,100``), wall clock of whole processes:

  1. a plain ``--inputList`` run, whose CLRs give the cut C, the ``--quantile`` quantile of all of them (as
     tools/regions_cost.py takes it);
  2. the full detailed run: ``--support DIR --regions REGIONS --threshold C``;
  3. the targeted run: the same flags and ``--targets REGIONS``.

The record compares the outputs of 2 and 3 under the contract of DESIGN.md §3.13: every main and support file of 3 is
the header and the lines of 2 at the kept rows, byte for byte, and every region line of 3 whose rows and position
interval keep off its target's first and last kept row is a line of 2.  The card's name, power limit and max SM clock
are recorded beside the times.

    python tools/targets_cost.py --sites 1000000 --out profiles/r11_targets_cost.json
"""
import argparse
import json
import os
import shutil
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import genome_cli_cost as g                                      # noqa: E402


def lines(path):
    with open(path) as fh:
        return fh.readlines()


def kept(main, ivs):
    """Rows of a main file (header dropped) whose physPos lies in a target."""
    pos = np.array([float(line.split('\t', 1)[0]) for line in main])
    keep = np.zeros(len(pos), bool)
    for a, b in ivs:
        keep |= (pos >= a) & (pos <= b)
    return keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=1_000_000, help='informative sites of the genome')
    ap.add_argument('--quantile', type=float, default=0.999, help='quantile of all CLRs used as the cut')
    ap.add_argument('--out', default='targets_cost.json', help='where the JSON record goes')
    opt = ap.parse_args()
    from ballermixplus_b200 import native
    if native.device_count() < 1:
        sys.exit('targets_cost: no CUDA device')
    work = tempfile.mkdtemp(prefix='blmx_targets_')
    lst, paths, _ = g.write_genome(work, opt.sites, 0)
    names = [os.path.basename(p) for p in paths]
    spect = os.path.join(work, 'genome_spect.txt')
    g.run([sys.executable, '-m', 'ballermixplus_b200', '--inputList', '--getSpect', '-i', lst, '--spect', spect],
          '--getSpect --inputList')
    flags = ['--usePhysPos', '--rec', str(g.bench.REC_RATE), '--rangeA', g.bench.RANGE_A]
    cmd = g.launcher(1, 0) + ['--inputList', '-i', lst, '--spect', spect] + flags
    dirs = {k: os.path.join(work, k) for k in ('plain', 'full', 'full_sup', 'part', 'part_sup')}
    for d in dirs.values():
        os.makedirs(d)
    wall_plain, _ = g.run(cmd + ['-o', dirs['plain']], 'plain run')
    T = np.concatenate([[float(line.split('\t')[2]) for line in lines(os.path.join(dirs['plain'], n))[1:]]
                        for n in names])
    cut = float(np.quantile(T, opt.quantile))
    reg, part_reg = os.path.join(work, 'regions.txt'), os.path.join(work, 'part_regions.txt')
    wall_full, _ = g.run(cmd + ['-o', dirs['full'], '--support', dirs['full_sup'], '--regions', reg, '--threshold',
                                repr(cut)], 'full --support run')
    wall_part, out = g.run(cmd + ['-o', dirs['part'], '--support', dirs['part_sup'], '--regions', part_reg,
                                  '--threshold', repr(cut), '--targets', reg], 'targeted --support run')
    ivs = {n: [] for n in names}
    for line in lines(reg)[2:]:
        f = line.split('\t')
        ivs[f[0]].append((float(f[1]), float(f[2])))
    bad, n_kept, by_name = [], 0, {}
    for n in names:
        main_lines = lines(os.path.join(dirs['full'], n))
        keep = kept(main_lines[1:], ivs[n])
        n_kept += int(keep.sum())
        for a, b in (('full', 'part'), ('full_sup', 'part_sup')):
            ref = lines(os.path.join(dirs[a], n))
            if lines(os.path.join(dirs[b], n)) != ref[:1] + [x for x, k in zip(ref[1:], keep) if k]:
                bad.append(f'{b}/{n}')
        pos = {line.split('\t', 1)[0]: j for j, line in enumerate(main_lines[1:])}
        by_name[n] = (keep, pos)
    full_regions = set(lines(reg)[2:])
    clear = clear_same = 0
    for line in lines(part_reg)[2:]:
        f = line.split('\t')
        keep, pos = by_name[f[0]]
        lo, hi = min(pos[f[1]], pos[f[11]]), max(pos[f[2]], pos[f[12]])
        if lo > 0 and keep[lo - 1] and hi + 1 < len(keep) and keep[hi + 1]:
            clear += 1
            clear_same += line in full_regions
    res = {'what': 'a full --support --regions --inputList run against the same run with --targets = its regions '
                   'file, wall clock of whole processes',
           'genome': f'{opt.sites} sites, {len(paths)} chromosomes (bench.make_genome), n = {g.bench.N_SAMPLE}',
           'flags': ' '.join(flags), 'gpu': g.gpu_info(), 'rows': int(len(T)), 'cut': cut,
           'cut_quantile': opt.quantile, 'targets': len(lines(reg)) - 2, 'rows_kept': n_kept,
           'wall_s_plain_run': wall_plain, 'wall_s_full_support_run': wall_full,
           'wall_s_targeted_support_run': wall_part, 'ratio_full_over_targeted': wall_full / wall_part,
           'main_and_support_mismatches': bad,
           'regions_targeted_run': len(lines(part_reg)) - 2,
           'regions_identical_to_a_full_run_line': sum(line in full_regions for line in lines(part_reg)[2:]),
           'regions_clear_of_target_edges': clear,
           'regions_clear_of_target_edges_identical': clear_same,
           'console': [line.replace(work, '<work>') for line in out.splitlines() if line.startswith('--targets: ')]}
    shutil.rmtree(work, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
    with open(opt.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != 'console'}))
    if bad or clear_same != clear or res['targets'] == 0:
        sys.exit('targets_cost: CHECK FAILED')


if __name__ == '__main__':
    main()
