#!/usr/bin/env python3
"""What a whole genome costs through the command line: one ``--inputList`` run against one run per chromosome.

Writes the cfg5-style synthetic genome (22 chromosomes of bench.make_chromosome, sizes in proportion to the human
autosomes, files written by bench.write_reference_inputs, as tools/full_scan.py builds it) at ``--sites`` sites,
makes the genome-wide spectrum with ``--getSpect --inputList``, and then times, as wall clock around whole
processes (imports, CUDA start-up and process-group set-up included):

  1 GPU         one ``--inputList`` run   vs  22 single-input runs, one after another
  torchrun N    the same two, each launched with ``torchrun --nproc-per-node N`` (when N GPUs are present)

Flags of every run: --usePhysPos --rec 1e-8 --rangeA 1000,10900,100 (51 000 grid points), every site a centre.
``--null K`` adds K neutral replicates (more synthetic chromosomes) and --pvalues to every run.  Every output file
of every arm is compared byte for byte with the 1-GPU single-input runs.  The card's name, power limit and max SM
clock are recorded beside the times.

    python tools/genome_cli_cost.py --sites 1000000 --out profiles/r9_genome_cli_cost.json
"""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                     # noqa: E402


def gpu_info():
    q = 'name,power.limit,clocks.max.sm'
    try:
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
    except OSError:
        out = []
    return {'query': q, 'gpus': out}


def write_genome(work, sites, n_null):
    """Inputs, their list, and (n_null > 0) replicates and their list -> (list, paths, null list or None)."""
    paths = []
    os.makedirs(os.path.join(work, 'in'))
    os.makedirs(os.path.join(work, 'reps'))
    for c, chrom in enumerate(bench.make_genome(sites)):
        prefix = os.path.join(work, 'in', f'chr{c + 1}')
        bench.write_reference_inputs(prefix, chrom)
        paths.append(prefix + '.txt')
    lst = os.path.join(work, 'genome.txt')
    with open(lst, 'w') as fh:
        fh.write('\n'.join(os.path.relpath(p, work) for p in paths) + '\n')
    null = None
    if n_null:
        reps = []
        for r in range(n_null):
            prefix = os.path.join(work, 'reps', f'rep{r}')
            bench.write_reference_inputs(prefix, bench.make_chromosome(max(1000, sites // 22), seed=900 + r))
            reps.append(prefix + '.txt')
        null = os.path.join(work, 'null.txt')
        with open(null, 'w') as fh:
            fh.write('\n'.join(reps) + '\n')
    return lst, paths, null


def run(cmd, what):
    t0 = time.perf_counter()
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
    wall = time.perf_counter() - t0
    if res.returncode != 0:
        sys.exit(f'{what} failed:\n' + res.stdout[-3000:] + res.stderr[-3000:])
    return wall, res.stdout


def launcher(nproc, port):
    if nproc == 1:
        return [sys.executable, '-m', 'ballermixplus_b200']
    return [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(nproc),
            '--master-addr', '127.0.0.1', '--master-port', str(port), '-m', 'ballermixplus_b200']


def arm(nproc, lst, paths, spect, flags, work, null, port):
    """One list run and one run per input, launched with nproc processes -> (record, list dir, single dir)."""
    tag = f'np{nproc}'
    d_list, d_one = os.path.join(work, f'{tag}_list'), os.path.join(work, f'{tag}_single')
    pv_list, pv_one = d_list + '_p', d_one + '_p'
    for d in (d_list, d_one, pv_list, pv_one):
        os.makedirs(d)
    extra = ['--null', null, '--pvalues'] if null else []
    wall_list, out = run(launcher(nproc, port) + ['--inputList', '-i', lst, '--spect', spect, '-o', d_list] + flags
                         + (extra + [pv_list] if null else []), f'{tag} --inputList run')
    walls = []
    for p in paths:
        name = os.path.basename(p)
        w, _ = run(launcher(nproc, port) + ['-i', p, '--spect', spect, '-o', os.path.join(d_one, name)] + flags
                   + (extra + [os.path.join(pv_one, name)] if null else []), f'{tag} run on {name}')
        walls.append(w)
    rec = {'processes': nproc, 'wall_s_inputList_run': wall_list, 'wall_s_single_runs_total': sum(walls),
           'wall_s_single_runs': walls, 'ratio_single_over_list': sum(walls) / wall_list,
           'list_run_console_tail': out.replace(work, '<work>').splitlines()[-30:]}
    return rec, (d_list, pv_list), (d_one, pv_one)


def compare(dirs_a, dirs_b, paths):
    bad = []
    for a, b in zip(dirs_a, dirs_b):
        for p in paths:
            name = os.path.basename(p)
            fa, fb = os.path.join(a, name), os.path.join(b, name)
            if os.path.exists(fa) or os.path.exists(fb):
                if not filecmp.cmp(fa, fb, shallow=False):
                    bad.append(f'{fa} != {fb}')
    return bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=10_000_000, help='informative sites of the genome')
    ap.add_argument('--nproc', type=int, default=8, help='torchrun arm: processes (run when that many GPUs exist)')
    ap.add_argument('--null', type=int, default=0, help='neutral replicates for --null / --pvalues (0: none)')
    ap.add_argument('--out', default='genome_cli_cost.json', help='where the JSON record goes')
    opt = ap.parse_args()
    from ballermixplus_b200 import native
    n_gpu = native.device_count()
    if n_gpu < 1:
        sys.exit('genome_cli_cost: no CUDA device')
    work = tempfile.mkdtemp(prefix='blmx_genome_')
    t0 = time.perf_counter()
    lst, paths, null = write_genome(work, opt.sites, opt.null)
    t_write = time.perf_counter() - t0
    spect = os.path.join(work, 'genome_spect.txt')
    t_spect, _ = run([sys.executable, '-m', 'ballermixplus_b200', '--inputList', '--getSpect', '-i', lst, '--spect',
                      spect], '--getSpect --inputList')
    flags = ['--usePhysPos', '--rec', str(bench.REC_RATE), '--rangeA', bench.RANGE_A]
    res = {'what': 'one --inputList run vs one run per chromosome, wall clock of whole processes',
           'genome': f'{opt.sites} sites, {len(paths)} chromosomes (bench.make_genome), n = {bench.N_SAMPLE}',
           'flags': ' '.join(flags), 'null_replicates': opt.null, 'gpu': gpu_info(), 'input_write_s': t_write,
           'getSpect_inputList_s': t_spect, 'arms': []}
    rec, ref_list, ref_one = arm(1, lst, paths, spect, flags, work, null, 0)
    rec['mismatches_list_vs_single'] = compare(ref_list, ref_one, paths)
    res['arms'].append(rec)
    if n_gpu >= opt.nproc > 1:
        rec, d_list, d_one = arm(opt.nproc, lst, paths, spect, flags, work, null, 29571)
        rec['mismatches_list_vs_1gpu_single'] = compare(d_list, ref_one, paths)
        rec['mismatches_single_vs_1gpu_single'] = compare(d_one, ref_one, paths)
        res['arms'].append(rec)
    else:
        res['torchrun_arm'] = f'not run: {n_gpu} GPU(s) present, {opt.nproc} wanted'
    shutil.rmtree(work, ignore_errors=True)
    res['identical'] = not any(v for a in res['arms'] for k, v in a.items() if k.startswith('mismatches'))
    os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
    with open(opt.out, 'w') as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != 'arms'}))
    for a in res['arms']:
        print(json.dumps({k: v for k, v in a.items() if k not in ('wall_s_single_runs', 'list_run_console_tail')}))
    if not res['identical']:
        sys.exit('genome_cli_cost: OUTPUTS DIFFER')


if __name__ == '__main__':
    main()
