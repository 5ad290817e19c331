#!/usr/bin/env python3
"""What ``--regions`` adds to a genome run: one ``--inputList`` run without it and one with ``--regions FILE
--threshold C``, on the genome of tools/genome_cli_cost.py (22 chromosomes of bench.make_genome, the genome
spectrum from ``--getSpect --inputList``, the same flags, every site a centre), wall clock of whole processes.

C is the ``--quantile`` quantile of every CLR of the run without ``--regions`` (taken from its main files).  The
record says whether the main files of the two runs are byte-identical and whether every peak line of the regions
file (peak_physPos through nSites) is a line of its input's main file.  The card's name, power limit and max SM
clock are recorded beside the times.

    python tools/regions_cost.py --sites 1000000 --out profiles/r10_regions_cost.json
"""
import argparse
import filecmp
import json
import os
import shutil
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import genome_cli_cost as g                                      # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=1_000_000, help='informative sites of the genome')
    ap.add_argument('--quantile', type=float, default=0.999, help='quantile of all CLRs used as the cut')
    ap.add_argument('--out', default='regions_cost.json', help='where the JSON record goes')
    opt = ap.parse_args()
    from ballermixplus_b200 import native
    if native.device_count() < 1:
        sys.exit('regions_cost: no CUDA device')
    work = tempfile.mkdtemp(prefix='blmx_regions_')
    lst, paths, _ = g.write_genome(work, opt.sites, 0)
    spect = os.path.join(work, 'genome_spect.txt')
    g.run([sys.executable, '-m', 'ballermixplus_b200', '--inputList', '--getSpect', '-i', lst, '--spect', spect],
          '--getSpect --inputList')
    flags = ['--usePhysPos', '--rec', str(g.bench.REC_RATE), '--rangeA', g.bench.RANGE_A]
    cmd = g.launcher(1, 0) + ['--inputList', '-i', lst, '--spect', spect] + flags
    plain, withr = os.path.join(work, 'plain'), os.path.join(work, 'with_regions')
    os.makedirs(plain)
    os.makedirs(withr)
    wall_plain, _ = g.run(cmd + ['-o', plain], 'run without --regions')
    main_lines = {}
    for p in paths:
        name = os.path.basename(p)
        with open(os.path.join(plain, name)) as fh:
            main_lines[name] = fh.read().splitlines()[1:]
    T = np.concatenate([[float(line.split('\t')[2]) for line in v] for v in main_lines.values()])
    cut = float(np.quantile(T, opt.quantile))
    reg = os.path.join(work, 'regions.txt')
    wall_regions, out = g.run(cmd + ['-o', withr, '--regions', reg, '--threshold', repr(cut)], 'run with --regions')
    with open(reg) as fh:
        lines = fh.read().splitlines()
    rows_of = {name: set(v) for name, v in main_lines.items()}
    found = 0
    for line in lines[2:]:
        f = line.split('\t')
        found += '\t'.join(f[4:11]) in rows_of[f[0]]
    res = {'what': 'one --inputList run without and one with --regions, wall clock of whole processes',
           'genome': f'{opt.sites} sites, {len(paths)} chromosomes (bench.make_genome), n = {g.bench.N_SAMPLE}',
           'flags': ' '.join(flags), 'rows': int(len(T)), 'cut': cut, 'cut_quantile': opt.quantile,
           'gpu': g.gpu_info(), 'wall_s_without_regions': wall_plain, 'wall_s_with_regions': wall_regions,
           'added_s': wall_regions - wall_plain, 'regions': len(lines) - 2,
           'inputs_with_regions': len({line.split('\t')[0] for line in lines[2:]}),
           'peaks_found_in_main_files': found,
           'main_files_identical': all(filecmp.cmp(os.path.join(plain, os.path.basename(p)),
                                                   os.path.join(withr, os.path.basename(p)), shallow=False)
                                       for p in paths),
           'console': [line.replace(work, '<work>') for line in out.splitlines() if line.startswith('regions: ')]}
    shutil.rmtree(work, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
    with open(opt.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not res['main_files_identical'] or found != res['regions'] or res['regions'] == 0:
        sys.exit('regions_cost: CHECK FAILED')


if __name__ == '__main__':
    main()
