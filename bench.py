#!/usr/bin/env python3
"""Benchmark of the CLR scan: centres x grid-points / s on synthetic whole-genome data.

Workload (BASELINE.json configs[4], SURVEY.md §8d): 10 M informative sites over 22
chromosomes (sizes proportional to the human autosomes, mean spacing 70 nt), n = 200 at
every site, P(substitution) = 0.7 else P(k) ~ 1/k, genPos = pos * 1e-8 (--usePhysPos --rec
1e-8), B2 statistic, default x (10) and alpha (51) grids, A = --rangeA 1000,10900,100
(100 values) -> 51 000 grid points per centre, default window mode (alpha >= 1e-8).
Scanning every site of that genome takes minutes even at roofline, so a "step" scans the
whole genome with the CLI's own --step flag: every S-th informative site is a centre
(S = 1024/N for N GPUs: per-GPU work is fixed, "weak" scaling).  Every centre still sees
the full 10 M-site data, exactly like `-s S` in the reference (v1:603-608).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo, CUDA
    python bench.py --dump-outputs DIR [...]                      # also write the rows of the last timed step
                                                                  # (CUDA arm only: the reference arm has no timed rows)
    python bench.py --impl reference [...]                        # CPU arm: the reference's own path on host cores
                                                                  # (C port on every step + the unmodified script once)

Every CUDA run carries a parity gate: rows of the timed scan are compared with the CPU oracle
(`parity` in the JSON line) and the run fails on a mismatch.  The synthetic genome and the centre list are
seeded, so two builds run with the same arguments scan the same inputs and their dumps compare row for row.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HUMAN_AUTOSOME_MB = [249.25, 243.20, 198.02, 191.15, 180.92, 171.12, 159.14, 146.36, 141.21, 135.53,
                     135.01, 133.85, 115.17, 107.35, 102.53, 90.35, 81.20, 78.08, 59.13, 63.03, 48.13, 51.30]
N_SAMPLE = 200
SPACING = 70
REC_RATE = 1e-8
RANGE_A = '1000,10900,100'
BASE_STRIDE = 1024
FP64_NOMINAL_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12        # 37.2: 148 SM x 64 DFMA/clk x 1.965 GHz
# algorithmic FP64 flops (SURVEY.md §8d: FMA = 2, MUL/ADD = 1; libdevice exp = 31, log = 47)
FLOP_SINGLE = 3.0          # (1-alpha) + alpha*R (FMA) and the running product (MUL), per site and grid point
FLOP_GROUPED = 2.25        # four sites: 4 FMA (quartic in R) + 1 MUL
FLOP_EXP = 34.0            # alpha = exp(-A*|g - t|): once per (centre, A, site) evaluated site by site
FLOP_QUAD_COEF = 23.0 / 4  # f0..f4 of a quartic from its four alphas (one lane), per grouped site
FLOP_LOG = 47.0 + 3.0      # one log + exponent fold-in per (centre, A, grid point)
FLOP_BLOCK = FLOP_EXP + 32 * (10.0 + 2.0)   # far field, per unit visit: one exp, then on each of the 32 moment lanes
                                            # ten multiplications (power by squaring) and one FMA
FLOP_EDGE = 9.0            # far field: five moments of a block-remainder site (besides its exp)
FLOP_POLY = 2.0            # far field: one Horner FMA per polynomial term and grid point
DUMP_BYTES = 60_000_000    # --dump-outputs: array data per run, so that the files with their headers stay within 64 MB


def algorithmic_flops(cnt, n_xa, n_items):
    """FP64 flops the formulation needs for the work the kernel's own counters report (DESIGN.md §3.3):
    sites evaluated per grid point (singly or four at a time), one exp per site that is looked at
    individually, the far-field block visits / remainder sites / polynomial terms, one log per grid point."""
    direct = cnt['pairs'] - cnt['far_sites']
    grouped = direct - cnt['single']
    return (n_xa * (FLOP_SINGLE * cnt['single'] + FLOP_GROUPED * grouped) + FLOP_QUAD_COEF * grouped
            + FLOP_EXP * (direct + cnt['edge_sites']) + FLOP_EDGE * cnt['edge_sites']
            + FLOP_BLOCK * cnt['far_blocks'] + FLOP_POLY * n_xa * cnt['far_terms'] + FLOP_LOG * n_xa * n_items)


# ------------------------------------------------------------------------ synthetic data
def make_chromosome(n_sites, seed, n=N_SAMPLE, spacing=SPACING):
    """SURVEY.md §8(d): positions = sorted sample without replacement from [1, L)."""
    rng = np.random.default_rng(seed)
    length = max(n_sites * spacing, n_sites + 2)
    pos = np.sort(rng.choice(length - 1, size=n_sites, replace=False)).astype(np.int64) + 1
    is_sub = rng.random(n_sites) < 0.7
    w = 1. / np.arange(1, n)
    k = np.where(is_sub, n, rng.choice(np.arange(1, n), size=n_sites, p=w / w.sum())).astype(np.int64)
    return {'pos': pos, 'k': k, 'n': n}


def genome_sizes(total_sites):
    w = np.array(HUMAN_AUTOSOME_MB) / sum(HUMAN_AUTOSOME_MB)
    sizes = np.floor(w * total_sites).astype(np.int64)
    sizes[0] += total_sites - sizes.sum()
    return sizes.tolist()


def make_genome(total_sites, seed=12345):
    return [make_chromosome(int(s), seed + c) for c, s in enumerate(genome_sizes(total_sites))]


def make_problem(chroms, range_a=RANGE_A):
    """Host precompute with the product's own classes (what the CLI does, without files):
    spectrum = empirical class frequencies of the concatenation (what --getSpect writes)."""
    from ballermixplus_b200 import Grids, InputData, NeutralSFS, NormalizedBetaBinom
    from ballermixplus_b200.native import ScanProblem
    from ballermixplus_b200.problem import GridOrder
    n = chroms[0]['n']
    counts = np.zeros(n + 1, np.int64)
    for c in chroms:
        counts += np.bincount(c['k'], minlength=n + 1)
    total = counts.sum()
    ks = np.flatnonzero(counts)
    spect = {(int(k), n): float(counts[k]) / float(total) for k in ks}
    classes = InputData.from_arrays(np.arange(len(ks)), np.arange(len(ks)) * 1e-6, ks, np.full(len(ks), n))
    neutral = NeutralSFS.from_spect(spect)
    grid = Grids(None, None, False, False, range_a, None)
    sel = NormalizedBetaBinom(classes, grid, False, False, False)
    G, P = neutral.class_tables(sel.class_k, sel.class_n)
    order = GridOrder(grid)
    SP = np.stack([sel.classProbs[(x, a)] * P for x in order.x for a in order.a])
    A = np.array([float(v) for v in order.A])
    class_of_k = np.full(n + 1, -1, np.int64)
    class_of_k[sel.class_k] = np.arange(len(sel.class_k))
    out = []
    for c in chroms:
        out.append(ScanProblem(c['pos'] * REC_RATE, class_of_k[c['k']].astype(np.int32), G, SP, A,
                               len(order.x), len(order.a)))
    return out


def plan_centres(problems, stride):
    """Default mode, `-s stride`: (chromosome, t, lo, hi) for every stride-th site (v1:598-610)."""
    plans = []
    for p in problems:
        n = len(p.genpos)
        idx = np.arange(0, n, stride)
        plans.append((p.genpos[idx].copy(), np.zeros(len(idx), np.int64), np.full(len(idx), n - 1, np.int64)))
    return plans


# ------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.device)],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        with open(self.path) as fh:
            for line in fh:
                f = [v.strip() for v in line.split(',')]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(names, f[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'power_w_max': float(max(pw)),
                'samples': len(sm), 'reasons': sorted(reasons)}


def host_threads():
    """Host cores this process may use (torchrun exports OMP_NUM_THREADS=1: not a limit on what the box has)."""
    return len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)


def cpu_sample_size(problems, plans, threads, target_s=15.0):
    """Centres for about `target_s` seconds of CPU work on this host: time two centres first
    (an interior centre of the 10 M-site workload is 6.6e8 log evaluations, parallelised over
    (centre, A) tasks), then scale."""
    secs, centres, _ = run_cpu_oracle(problems, plans, cpu_sample(problems, plans, 2, threads), threads)
    per_centre = max(secs / max(centres, 1), 1e-3)
    return int(min(4096, max(2, round(target_s / per_centre))))


def cpu_sample(problems, plans, n_centres, threads):
    """A bounded sample for the CPU arm: centres spread evenly over the whole genome."""
    sizes = np.array([len(p[0]) for p in plans])
    picks = np.linspace(0, sizes.sum() - 1, n_centres).astype(np.int64)
    bounds = np.concatenate(([0], np.cumsum(sizes)))
    sample = []
    for c in range(len(plans)):
        mine = picks[(picks >= bounds[c]) & (picks < bounds[c + 1])] - bounds[c]
        if len(mine):
            sample.append((c, mine))
    return sample


def run_cpu_oracle(problems, plans, sample, threads, report_all=False, keep=None):
    """Literal calcBaller (oracle/oracle_c.c, OpenMP) on the sample -> (seconds, centres, site pairs).
    `keep`: a list that receives (chromosome, centre indices, oracle result) per chromosome."""
    from oracle import oracle_c
    t0 = time.perf_counter()
    centres = pairs = 0
    for c, idx in sample:
        p = problems[c]
        t, lo, hi = plans[c]
        res = oracle_c.scan(p.genpos, p.cls, p.G, p.SP, p.A, t[idx], lo[idx], hi[idx], n_threads=threads,
                            report_all=report_all)
        centres += len(idx)
        pairs += res[4]
        if keep is not None:
            keep.append((c, idx, res))
    return time.perf_counter() - t0, centres, pairs


def dump_outputs(out_dir, rows, limit=DUMP_BYTES):
    """Write the rows one step returns, (T, iA, ix, ia, nsites) per centre in global centre order, as
    <out_dir>/<field>.npy in float64 (exact for the int32 fields), with centre.npy: the index of each row.
    Rows beyond `limit` bytes are replaced by a fixed, seeded sample of the centres."""
    fields = [np.asarray(a, dtype=np.float64) for a in rows]
    n = len(fields[0])
    per_row = 8 * (len(fields) + 1)
    keep = np.arange(n)
    if n * per_row > limit:
        keep = np.sort(np.random.default_rng(0).choice(n, limit // per_row, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in zip(('centre', 'T', 'iA', 'ix', 'ia', 'nsites'), [keep.astype(np.float64)] + fields):
        np.save(os.path.join(out_dir, name + '.npy'), a if name == 'centre' else a[keep])


def parity_sample(plans, T_rows, n_positive=64, n_any=32):
    """Centres for the parity gate, chosen from the rows of the timed scan: `n_positive` centres whose
    row carries a real maximum (T > 0; neutral synthetic data gives the all-zero row for most centres)
    and `n_any` centres spread evenly whatever their row."""
    sizes = np.array([len(p[0]) for p in plans])
    bounds = np.concatenate(([0], np.cumsum(sizes)))
    pos = np.flatnonzero(T_rows > 0)
    picks = set(np.linspace(0, bounds[-1] - 1, n_any).astype(np.int64).tolist())
    if len(pos):
        picks |= set(pos[np.linspace(0, len(pos) - 1, min(n_positive, len(pos))).astype(np.int64)].tolist())
    picks = np.array(sorted(picks), dtype=np.int64)
    sample = []
    for c in range(len(plans)):
        mine = picks[(picks >= bounds[c]) & (picks < bounds[c + 1])] - bounds[c]
        if len(mine):
            sample.append((c, mine))
    return sample, bounds


def parity_check(problems, kept, bounds, rows, rows_all):
    """Compare GPU rows (global centre order) with the oracle results `kept` -> the `parity` object.
    rows = (T, iA, ix, ia, ns) of the timed scan (the reference's rule, T > 0 only); rows_all = the same
    centres scanned with option report_all (oracle run the same way), so every compared centre carries a
    real T and argmax."""
    out = {'centres': 0, 'rows_T_gt_0': 0, 'max_rel_dT': 0.0, 'argmax_mismatch': 0, 'nsites_mismatch': 0,
           'tolerance': '|dT| <= 1e-9*max(|T|,1); identical (A, x, a) and nSites'}
    for which, (res_list, got) in (('', (kept[0], rows)), ('_report_all', (kept[1], rows_all))):
        if got is None:
            continue
        n = pos = bad_arg = bad_ns = 0
        worst = 0.0
        k = 0
        for c, idx, (rT, rA, rxa, rn, _) in res_list:
            n_a = problems[c].n_a
            if which:
                sel = slice(k, k + len(idx))
                k += len(idx)
            else:
                sel = bounds[c] + idx
            T, iA, ix, ia, ns = (np.asarray(a)[sel] for a in got)
            xa = np.where(iA >= 0, ix * n_a + ia, -1)
            rel = np.abs(T - rT) / np.maximum(np.abs(rT), 1.)
            worst = max(worst, float(rel.max()))
            bad_arg += int(np.sum((iA != rA) | (xa != rxa)))
            bad_ns += int(np.sum(ns != rn))
            n += len(idx)
            pos += int(np.sum(rA >= 0))
        if which:
            out['report_all'] = {'centres': n, 'rows_with_T': pos, 'max_rel_dT': worst,
                                 'argmax_mismatch': bad_arg, 'nsites_mismatch': bad_ns}
        else:
            out.update({'centres': n, 'rows_T_gt_0': pos, 'max_rel_dT': worst, 'argmax_mismatch': bad_arg,
                        'nsites_mismatch': bad_ns})
    ra = out.get('report_all', {})
    out['ok'] = bool(out['max_rel_dT'] <= 1e-9 and out['argmax_mismatch'] == 0 and out['nsites_mismatch'] == 0
                     and ra.get('max_rel_dT', 0.0) <= 1e-9 and ra.get('argmax_mismatch', 0) == 0
                     and ra.get('nsites_mismatch', 0) == 0)
    return out


def run_numpy_oracle_one_centre(problems, plans):
    """The vectorised numpy restatement (oracle/oracle_np.py, what the reference's numpy/scipy path
    costs once its Python-list indexing overhead is removed), ONE interior centre, one thread."""
    from oracle import oracle_np
    c = int(np.argmax([len(p.genpos) for p in problems]))
    p = problems[c]
    t = plans[c][0]
    tj = float(t[len(t) // 2])
    reach = 18.420680743952367 / float(p.A.min()) * 1.001
    lo = int(np.searchsorted(p.genpos, tj - reach, 'left'))
    hi = int(np.searchsorted(p.genpos, tj + reach, 'right'))
    g = p.genpos[lo:hi]
    cls = p.cls[lo:hi]
    probs = p.G[cls]
    selmat = np.ascontiguousarray(p.SP[:, cls])
    t0 = time.perf_counter()
    oracle_np.calc_baller_fast(0, len(g) - 1, tj, g, probs, np.log(probs), np.ones_like(probs), selmat, p.A)
    secs = time.perf_counter() - t0
    n_grid = p.n_x * p.n_a * len(p.A)
    return {'value': n_grid / secs, 'unit': 'centre*gridpoint/s', 'cores': 1, 'kind': 'port',
            'sample': f'1 interior centre, {n_grid} grid points, numpy restatement (oracle/oracle_np.py), {secs:.1f} s'}


# ------------------------------------------------------ the unmodified reference script
REF_SCRIPT = os.path.join(ROOT, 'oracle', '_ref', 'BalLeRMix+_v1.py')     # copied there by oracle/make_ref.sh


def write_reference_inputs(prefix, chrom):
    """One synthetic chromosome as the reference's own input + --spect helper files."""
    n = chrom['n']
    with open(prefix + '.txt', 'w') as fh:
        fh.write('physPos\tgenPos\tx\tn\n')
        for pos, k in zip(chrom['pos'].tolist(), chrom['k'].tolist()):
            fh.write(f'{pos}\t{pos * REC_RATE}\t{k}\t{n}\n')
    cnt = np.bincount(chrom['k'], minlength=n + 1)
    with open(prefix + '_spect.txt', 'w') as fh:
        for k in np.flatnonzero(cnt):
            fh.write('%s\t%s\t%s\n' % (k, n, cnt[k] / float(len(chrom['k']))))


def run_reference_script(cores, n_sites=3000, centres_per_proc=2):
    """BASELINE.md §3.3: the reference as shipped (BalLeRMix+_v1.py, numpy/scipy, single-threaded, no shard
    flag), one unmodified process per host core, each on its own synthetic chromosome of the bench shape
    (n = 200, same generator, same 100 x 10 x 51 grid passed as --listA because the reference's --rangeA
    raises TypeError, v1:169-171) with `-s` chosen for `centres_per_proc` centres.  Returns the
    cpu_baseline_reference object, or why it could not run."""
    if not os.path.exists(REF_SCRIPT):
        return {'kind': 'reference', 'unavailable': 'oracle/_ref/BalLeRMix+_v1.py missing (run oracle/make_ref.sh '
                                                    'where /root/reference exists)'}
    lo_a, hi_a, step_a = (float(v) for v in RANGE_A.split(','))
    list_a = ','.join(str(lo_a + step_a * i) for i in range(int((hi_a - lo_a) / step_a) + 1))
    n_A = list_a.count(',') + 1
    stride = n_sites // centres_per_proc
    work = tempfile.mkdtemp(prefix='blmx_ref_')
    procs = []
    site_evals = 0
    t0 = time.perf_counter()
    for p in range(cores):
        chrom = make_chromosome(n_sites, seed=777 + p)
        prefix = os.path.join(work, f'c{p}')
        write_reference_inputs(prefix, chrom)
        g = chrom['pos'] * REC_RATE
        for c in range(0, n_sites, stride):
            for a in list_a.split(','):
                al = np.exp(-float(a) * np.abs(g - g[c]))
                site_evals += int(np.sum((al >= 1e-8) & (g != g[c]))) * 510
        cmd = [sys.executable, REF_SCRIPT, '-i', prefix + '.txt', '--spect', prefix + '_spect.txt', '-o',
               prefix + '_out.txt', '--usePhysPos', '--rec', str(REC_RATE), '--listA', list_a, '-s', str(stride)]
        env = dict(os.environ, OMP_NUM_THREADS='1', OPENBLAS_NUM_THREADS='1', MKL_NUM_THREADS='1')
        procs.append(subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env, cwd=work))
    t_launch = time.perf_counter()
    rcs = [q.wait() for q in procs]
    secs = time.perf_counter() - t_launch
    rows = 0
    for p in range(cores):
        try:
            with open(os.path.join(work, f'c{p}_out.txt')) as fh:
                rows += max(0, len(fh.read().splitlines()) - 1)
        except OSError:
            pass
    if any(rcs) or rows == 0:
        return {'kind': 'reference', 'unavailable': f'reference script exited with {rcs[:4]}..., {rows} rows'}
    n_grid = n_A * 510
    return {
        'kind': 'reference', 'cores': cores, 'processes': cores, 'centres': rows, 'seconds': secs,
        's_per_centre': secs * cores / rows, 'value': rows * n_grid / secs, 'unit': 'centre*gridpoint/s',
        'site_evals_per_s': site_evals / secs, 'site_evals_per_s_per_core': site_evals / secs / cores,
        'sample': f'unmodified BalLeRMix+_v1.py (copied to oracle/_ref by oracle/make_ref.sh), {cores} concurrent '
                  f'single-threaded processes, each a {n_sites}-site synthetic chromosome (n = 200, bench generator), '
                  f'-s {stride} ({centres_per_proc} centres), --listA = the bench A grid, {n_grid} grid points per '
                  f'centre; wall {secs:.0f} s incl. the script\'s own table precompute; windows here hold <= {n_sites} '
                  f'sites against 12 710 on average in the benchmark, so compare site_evals_per_s, not value',
        'setup_s': t_launch - t0,
    }


# ---------------------------------------------------------------------------------- arms
def reference_arm(opt, rank):
    """CPU arm = the reference's own implementation of the path on the box's host cores: every step times the
    C port of calcBaller (oracle/oracle_c.c, OpenMP on all cores) on a bounded sample of the workload; once
    per run the unmodified script itself is timed beside it (cpu_baseline_reference)."""
    if rank != 0:
        return
    threads = host_threads()
    chroms = make_genome(opt.sites)
    problems = make_problem(chroms)
    stride = max(1, BASE_STRIDE // opt.gpus)
    plans = plan_centres(problems, stride)
    n_grid = problems[0].n_x * problems[0].n_a * len(problems[0].A)
    # a bounded sample per step: about 12 s of CPU work, less when many steps are asked for, so that the whole
    # arm (steps + one run of the unmodified script) ends within a few minutes
    per_step = opt.cpu_centres or cpu_sample_size(problems, plans, threads,
                                                  target_s=max(3.0, min(12.0, 100.0 / max(1, opt.steps))))
    sample = cpu_sample(problems, plans, per_step, threads)
    for _ in range(min(opt.warmup, 2)):
        run_cpu_oracle(problems, plans, cpu_sample(problems, plans, 1, threads), threads)
    secs = centres = pairs = 0
    for _ in range(opt.steps):
        s, c, p = run_cpu_oracle(problems, plans, sample, threads)
        secs += s; centres += c; pairs += p
    value = centres * n_grid / secs
    line = {
        'impl': 'reference', 'metric': 'centres x grid-points / s (B2 scan)', 'value': value,
        'unit': 'centre*gridpoint/s', 'n_gpus': opt.gpus, 'steps': opt.steps, 'warmup': opt.warmup,
        'ms_per_step': secs / opt.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(opt, stride, problems, plans),
        'cpu_baseline': {'value': value, 'unit': 'centre*gridpoint/s', 'cores': threads, 'kind': 'port',
                         'sample': f'{per_step} centres per step spread evenly over the genome, all '
                                   f'{n_grid} grid points each, literal calcBaller in C (oracle/oracle_c.c), '
                                   f'OpenMP on {threads} threads',
                         'site_evals_per_s': pairs * problems[0].n_x * problems[0].n_a / secs},
        'e2e': {'value': value, 'unit': 'centre*gridpoint/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    if not opt.no_ref_script:
        ref = run_reference_script(threads)
        if 'site_evals_per_s' in ref:
            # the script's rate on the benchmark's own windows: its cost is per site-evaluation (BASELINE.md §2)
            mean_w = pairs / max(1, centres * len(problems[0].A))
            ref['value_at_bench_windows'] = ref['site_evals_per_s'] / mean_w
            ref['note'] = ('value_at_bench_windows = site_evals_per_s / (mean sites per (centre, A) of the benchmark, '
                           f'{mean_w:.0f}): the extrapolation to the 10 M-site windows, reported separately')
        line['cpu_baseline_reference'] = ref
    print(json.dumps(line), flush=True)


def workload_config(opt, stride, problems, plans):
    n_sites = int(sum(len(p.genpos) for p in problems))
    return {
        'workload': f'cfg5 synthetic whole-genome B2 scan: {n_sites} sites / {len(problems)} chromosomes, n=200, '
                    f'--usePhysPos --rec 1e-8, --rangeA {RANGE_A} x default x/alpha grids, default window '
                    f'mode, centres = every {stride}-th site (-s {stride})',
        'sites': n_sites, 'chromosomes': len(problems), 'centres_per_step': int(sum(len(p[0]) for p in plans)),
        'grid_points_per_centre': problems[0].n_x * problems[0].n_a * len(problems[0].A),
        'centre_stride': stride, 'parallelism': f'centre-range shards x{opt.gpus}',
        'l2': 'site arrays (200 MB at 10 M sites) exceed the 126 MB L2; an extra 256 MB write flushes L2 between steps',
    }


class Shard:
    """This rank's cost-balanced contiguous slice of the centre list for one centre stride, with the
    device buffers of a step."""

    def __init__(self, problems, stride, rank, world, torch, dev, sharding):
        self.plans = plan_centres(problems, stride)
        costs = np.concatenate([sharding.centre_costs(p.genpos, pl[0], pl[1], pl[2], p.A)
                                for p, pl in zip(problems, self.plans)])
        parts = sharding.partition(costs, world)
        self.counts = [e - b for b, e in parts]
        begin, end = parts[rank]
        self.offs = np.concatenate(([0], np.cumsum([len(pl[0]) for pl in self.plans])))
        self.mine = []           # (chromosome, slice into its plan)
        for c in range(len(self.plans)):
            b, e = max(begin, self.offs[c]), min(end, self.offs[c + 1])
            if e > b:
                self.mine.append((c, slice(int(b - self.offs[c]), int(e - self.offs[c]))))
        self.begin, self.n_mine, self.total = int(begin), int(end - begin), int(self.offs[-1])
        host_in = {c: tuple(np.ascontiguousarray(a[sl]) for a in self.plans[c]) for c, sl in self.mine}
        self.pinned = {c: tuple(torch.from_numpy(a).pin_memory() for a in host_in[c]) for c in host_in}
        self.d_in = {c: tuple(x.to(dev) for x in self.pinned[c]) for c in self.pinned}
        self.d_T = torch.zeros(self.n_mine, dtype=torch.float64, device=dev)
        self.d_idx = [torch.zeros(self.n_mine, dtype=torch.int32, device=dev) for _ in range(4)]


def cuda_arm(opt, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from ballermixplus_b200 import native, sharding

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    chroms = make_genome(opt.sites)
    problems = make_problem(chroms)
    del chroms
    # the host copies of the inputs live in pinned memory: blmx_load's H2D copies are then true async DMA
    pinned_inputs = []
    for p in problems:
        for name in ('genpos', 'cls'):
            buf = torch.from_numpy(getattr(p, name)).pin_memory()
            pinned_inputs.append(buf)
            setattr(p, name, buf.numpy())
    stride = max(1, BASE_STRIDE // world)
    n_xa = problems[0].n_x * problems[0].n_a
    n_A = len(problems[0].A)
    n_grid = n_xa * n_A
    shard = Shard(problems, stride, rank, world, torch, dev, sharding)
    plans, mine, counts, total_centres, n_mine = shard.plans, shard.mine, shard.counts, shard.total, shard.n_mine

    # resident problems: one handle per chromosome this rank touches
    scanners = {}
    for c, _ in mine:
        scanners[c] = native.Scanner(device=local_rank, group=opt.group, farfield=opt.farfield).load(problems[c])
        scanners[c].set_option('timing', 1)
    info = [scanners[c].problem_info() for c, _ in mine]
    main_stream = torch.cuda.current_stream()
    # chromosomes are independent launches: issued round-robin on a few streams so that the tail of one
    # launch (its last, cheapest work items) overlaps the head of the next
    side = [torch.cuda.Stream(device=dev) for _ in range(max(1, opt.streams))]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def scan_into(sh, reload_problem=False, n_streams=None):
        """One step on this rank: every chromosome of the shard, then pack + gather (the only collective)."""
        fork = torch.cuda.Event()
        fork.record(main_stream)
        o = 0
        use = side[:n_streams] if n_streams else side
        for k, (c, _) in enumerate(sh.mine):
            st = use[k % len(use)]
            st.wait_event(fork)
            with torch.cuda.stream(st):
                if reload_problem:
                    scanners[c].load(problems[c])               # H2D of sites + tables, class sort, block moments
                    t, lo, hi = (x.to(dev, non_blocking=True) for x in sh.pinned[c])   # H2D of the centres
                else:
                    t, lo, hi = sh.d_in[c]
                n = t.shape[0]
                scanners[c].scan_device(n, t.data_ptr(), lo.data_ptr(), hi.data_ptr(), sh.d_T[o:].data_ptr(),
                                        *[x[o:].data_ptr() for x in sh.d_idx], stream=st.cuda_stream)
                if reload_problem:
                    for x in (t, lo, hi):
                        x.record_stream(st)
            o += n
        for st in side:
            join = torch.cuda.Event()
            join.record(st)
            main_stream.wait_event(join)
        rows = sharding.pack_rows(sh.d_T, *sh.d_idx, torch)
        return sharding.gather_rows(rows, sh.counts, rank, world, dist, torch)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def collect(sh):
        """Per-launch kernel events and work counters of the LAST step, summed over this rank's scanners."""
        tot = {'pairs': 0, 'single': 0, 'far_blocks': 0, 'far_terms': 0, 'far_sites': 0, 'edge_sites': 0,
               'quads': 0, 'launches': 0}
        k_ms, k_n = 0.0, 0
        for c, _ in sh.mine:
            kms, kn = scanners[c].kernel_ms()
            k_ms += kms; k_n += kn
            for key, v in scanners[c].counters_all().items():
                tot[key] = tot.get(key, 0) + v
        return tot, k_ms, k_n

    def timed(fn, steps, flush_l2=True):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
            if flush_l2:
                flush.zero_()
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ms = float(tmax.item())
        return ms, out

    def reduce_sum(values):
        if world == 1:
            return [float(v) for v in values]
        agg = torch.tensor([float(v) for v in values], dtype=torch.float64, device=dev)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
        return agg.tolist()

    # ---- device-resident timing -------------------------------------------------------
    for _ in range(opt.warmup):
        scan_into(shard)
        flush.zero_()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, gathered = timed(lambda: scan_into(shard), opt.steps)
    clocks = sampler.stop() if rank == 0 else None
    # roofline pass: the same step once more on ONE stream, so that the CUDA events the library records around
    # every scan_kernel launch time that kernel alone (on several streams the launches overlap at their tails
    # and the per-launch durations would count the shared time twice)
    timed(lambda: scan_into(shard, n_streams=1), 1)
    cnt, kernel_ms, kernel_launches = collect(shard)
    pairs_all, launches_all = (int(v) for v in reduce_sum([cnt['pairs'], cnt['launches']]))
    value = total_centres * n_grid * opt.steps / (ms * 1e-3)
    resident_rows = sharding.unpack_rows(gathered.cpu(), torch) if rank == 0 else None
    if rank == 0 and opt.dump_outputs:
        dump_outputs(opt.dump_outputs, [a.numpy() for a in resident_rows])

    # the same workload with every site evaluated directly (option farfield = 0): the FP64-bound kernel
    direct = None
    if opt.farfield and world == 1 and not opt.profile:
        for c, _ in mine:
            scanners[c].set_option('farfield', 0)
        scan_into(shard, n_streams=1)
        d_ms, _ = timed(lambda: scan_into(shard, n_streams=1), 1, flush_l2=False)     # one stream: exact per-launch events
        d_cnt, d_kms, d_kn = collect(shard)
        direct = (d_ms, d_cnt, d_kms, d_kn)
        for c, _ in mine:
            scanners[c].set_option('farfield', 1)

    # ---- end to end through the C ABI with host buffers ---------------------------------
    e2e = None
    if not opt.profile:
        def scan_e2e():
            g = scan_into(shard, reload_problem=True)
            return g.cpu() if g is not None else None                 # D2H of every row on rank 0
        scan_e2e()
        sync_all()
        t0 = time.perf_counter()
        e2e_ms, host_rows = timed(scan_e2e, opt.steps, flush_l2=False)
        wall_ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            tmax = torch.tensor([wall_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            wall_ms = float(tmax.item())
        e2e_ms = max(e2e_ms, wall_ms)
        h2d = sum(problems[c].h2d_bytes + 24 * (sl.stop - sl.start) for c, sl in mine)
        d2h = 24 * total_centres if rank == 0 else 0
        h2d, d2h = (int(v) for v in reduce_sum([h2d, d2h]))
        e2e = {'value': total_centres * n_grid * opt.steps / (e2e_ms * 1e-3), 'unit': 'centre*gridpoint/s',
               'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms / opt.steps,
               'includes': 'blmx_load of every chromosome (H2D of sites and tables, device class sort, far-field '
                           'block moments), H2D of the centres, scan, gather, D2H of every row'}
        if rank == 0:
            er = sharding.unpack_rows(host_rows, torch)
            same = all(bool((a == b).all()) for a, b in zip(er, resident_rows))
            e2e['rows_equal_resident_run'] = same

    # ---- strong scaling: the SAME centre list (stride 128) whatever the number of GPUs ----------
    strong = None
    if opt.strong_stride > 0 and not opt.profile:
        sh2 = Shard(problems, opt.strong_stride, rank, world, torch, dev, sharding)
        scan_into(sh2)
        s_ms, _ = timed(lambda: scan_into(sh2), opt.strong_steps)
        strong = {'centre_stride': opt.strong_stride, 'centres_per_step': sh2.total, 'steps': opt.strong_steps,
                  'ms_per_step': s_ms / opt.strong_steps, 'value': sh2.total * n_grid * opt.strong_steps / (s_ms * 1e-3),
                  'unit': 'centre*gridpoint/s', 'scaling': 'strong',
                  'note': 'total work fixed for every N (the weak-scaling headline divides the stride by N)'}
        del sh2

    # ---- parity gate (rank 0): rows of the timed run against the CPU oracle ----------------
    if rank == 0:
        line = {
            'metric': 'centres x grid-points / s (B2 scan)', 'value': value, 'unit': 'centre*gridpoint/s',
            'n_gpus': world, 'steps': opt.steps, 'warmup': opt.warmup, 'ms_per_step': ms / opt.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(opt, stride, problems, plans),
            'site_evals_per_s': pairs_all * n_xa / (ms / opt.steps * 1e-3),
            'mean_sites_per_centre_A': pairs_all / max(1, total_centres * n_A),
            'gpu_launches': int(launches_all * opt.steps),
            'clocks': clocks,
        }
        if e2e is not None:
            line['e2e'] = e2e
        if strong is not None:
            line['strong'] = strong

        threads = host_threads()
        cpu = None
        if not opt.no_cpu:
            T_rows = resident_rows[0].numpy()
            sample, bounds = parity_sample(plans, T_rows, opt.parity_positive, opt.parity_any)
            kept = ([], [])
            secs, centres, cpairs = run_cpu_oracle(problems, plans, sample, threads, keep=kept[0])
            run_cpu_oracle(problems, plans, sample, threads, report_all=True, keep=kept[1])
            # the same centres with option report_all on the GPU (this rank's device, outside the timed region)
            got_all = [[] for _ in range(5)]
            for c, idx in sample:
                t, lo, hi = plans[c]
                with native.Scanner(device=local_rank, group=opt.group, farfield=opt.farfield) as sc:
                    sc.set_option('report_all', 1)
                    sc.load(problems[c])
                    for k, a in enumerate(sc.scan(t[idx], lo[idx], hi[idx])):
                        got_all[k].append(a)
            rows_all = tuple(np.concatenate(a) for a in got_all)
            rows_np = tuple(a.numpy() for a in resident_rows)
            line['parity'] = parity_check(problems, kept, bounds, rows_np, rows_all)
            line['parity']['checker'] = 'oracle/oracle_c.c (literal calcBaller, compensated sums)'
            cpu = {'value': centres * n_grid / secs, 'unit': 'centre*gridpoint/s', 'cores': threads, 'kind': 'port',
                   'sample': f'{centres} centres of the timed scan ({line["parity"]["rows_T_gt_0"]} with T > 0, the '
                             f'rest spread evenly), all {n_grid} grid points each, literal calcBaller in C '
                             f'(oracle/oracle_c.c), OpenMP on {threads} threads, {secs:.1f} s',
                   'site_evals_per_s': cpairs * n_xa / secs}

        peak_tf, peak_mhz = native.measure_fp64_peak(local_rank, 0.5)
        n_items = n_mine * n_A
        flops = algorithmic_flops(cnt, n_xa, n_items)
        k_s = kernel_ms * 1e-3
        achieved = flops / k_s / 1e12 if k_s > 0 else None
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tpath):
            with open(tpath) as fh:
                traffic = json.load(fh)
        hbm_peak = None
        mp = os.path.join(ROOT, 'MEASURED_PEAKS.json')
        if os.path.exists(mp):
            with open(mp) as fh:
                hbm_peak = json.load(fh).get('hbm_gbs')
        n_sites_mine = sum(len(problems[c].genpos) for c, _ in mine)
        moment_bytes = sum(i['moment_bytes'] for i in info)
        # HBM bytes one launch must move at least once: the chromosome's site arrays (g, gs: 8 B, is: 4 B per
        # site), the R table, its far-field block moments, and the (centre, A) candidates written and re-read
        hbm_algo = (20.0 * n_sites_mine + 8.0 * 512 * len(problems[0].G) * len(mine) + moment_bytes
                    + 2 * 16.0 * n_items) / max(1, kernel_launches)
        line['roofline'] = {
            'bound': 'fp64', 'kernel': 'scan_kernel<16,%d,%s>' % (opt.group, 'far' if opt.farfield else 'direct'),
            'achieved': achieved,
            'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': (achieved / peak_tf) if achieved and peak_tf else None,
            'peak_source': 'measured live: register-resident DFMA loop (blmx_measure_fp64_peak); '
                           'MEASURED_PEAKS.json has no FP64 entry',
            'peak_nominal': FP64_NOMINAL_TFLOPS,
            'frac_of_nominal': (achieved / FP64_NOMINAL_TFLOPS) if achieved else None,
            'kernel_ms_per_launch': kernel_ms / max(1, kernel_launches), 'launches_timed': kernel_launches,
            'kernel_share_of_step': kernel_ms / (ms / opt.steps) if ms > 0 else None,
            'timing': 'CUDA events recorded by the library around every scan_kernel launch, on the launching stream, '
                      f'in one extra step run on a single stream right after the timed region (the timed steps rotate '
                      f'the launches over {len(side)} streams, where per-launch events would overlap)',
            'algorithmic_flops_per_launch': flops / max(1, kernel_launches),
            'work': {k: cnt[k] for k in ('pairs', 'single', 'quads', 'far_sites', 'far_blocks', 'edge_sites', 'far_terms')},
            'sites_far_frac': cnt['far_sites'] / max(1, cnt['pairs']),
            'traffic': traffic.get('dram_bytes_per_launch') if traffic else None,
            'traffic_source': traffic.get('source') if traffic else None,
            'traffic_algorithmic_bytes_same_launch': traffic.get('algorithmic_bytes_of_that_launch') if traffic else None,
            'hbm': {'algorithmic_bytes_per_launch': hbm_algo,
                    'achieved_gbs': hbm_algo / (k_s / max(1, kernel_launches)) / 1e9 if k_s > 0 else None,
                    'peak_gbs': hbm_peak, 'moment_bytes_resident': moment_bytes,
                    'note': 'bytes a launch must fetch from HBM at least once (site arrays, table, block moments, '
                            'candidates); everything else is L2/L1 traffic. The path is FP64-bound.'},
        }
        line['mode'] = ('farfield: far sites through per-block precomputed power sums of alpha (DESIGN.md §3.4)'
                        if opt.farfield else 'direct: every site evaluated per grid point')
        if direct is not None:
            d_ms, d_cnt, d_kms, d_kn = direct
            d_flops = algorithmic_flops(d_cnt, n_xa, n_items)
            d_ach = d_flops / (d_kms * 1e-3) / 1e12
            line['direct'] = {
                'value': total_centres * n_grid / (d_ms * 1e-3), 'unit': 'centre*gridpoint/s', 'ms_per_step': d_ms,
                'roofline': {'bound': 'fp64', 'kernel': 'scan_kernel<16,%d,direct>' % opt.group, 'achieved': d_ach,
                             'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': d_ach / peak_tf,
                             'kernel_ms_per_launch': d_kms / max(1, d_kn), 'launches_timed': d_kn,
                             'algorithmic_flops_per_launch': d_flops / max(1, d_kn)},
                'note': 'same step with option farfield = 0 (one warm-up + one timed step)'}
        if cpu is not None:
            line['cpu_baseline'] = cpu
            if world == 1:
                line['cpu_baseline_numpy'] = run_numpy_oracle_one_centre(problems, plans)
        print(json.dumps(line), flush=True)
        parity_failed = 'parity' in line and not line['parity']['ok']
    else:
        parity_failed = False
    for s in scanners.values():
        s.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity_failed:
        sys.exit('bench: PARITY GATE FAILED (see "parity" in the JSON line)')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
    ap.add_argument('--sites', type=int, default=10_000_000, help='informative sites in the synthetic genome')
    ap.add_argument('--group', type=int, default=4, choices=[1, 4])
    ap.add_argument('--farfield', type=int, default=1, choices=[0, 1],
                    help='1 (default): far sites enter through power sums; 0: every site evaluated directly')
    ap.add_argument('--streams', type=int, default=3, help='CUDA streams the per-chromosome launches rotate over')
    ap.add_argument('--strong-stride', type=int, default=128,
                    help='centre stride of the fixed-work (strong scaling) leg; 0 = skip it')
    ap.add_argument('--strong-steps', type=int, default=1)
    ap.add_argument('--parity-positive', type=int, default=64, help='parity gate: centres whose row has T > 0')
    ap.add_argument('--parity-any', type=int, default=32, help='parity gate: centres spread evenly')
    ap.add_argument('--cpu-centres', type=int, default=0, help='reference arm: centres per step (default: ~12 s)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the parity gate and the cpu_baseline leg')
    ap.add_argument('--no-ref-script', action='store_true',
                    help='reference arm: skip the run of the unmodified script (oracle/_ref)')
    ap.add_argument('--profile', action='store_true',
                    help='only the device-resident timed steps (for ncu): no direct / e2e / strong legs')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the rows of the last timed step to DIR/<field>.npy; CUDA arm only, '
                         'refused with --impl reference')
    opt = ap.parse_args()
    if opt.steps < 1 or opt.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if opt.dump_outputs and opt.impl != 'cuda':
        ap.error('--dump-outputs writes the rows of the CUDA arm')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if opt.impl == 'reference':
        reference_arm(opt, rank)
        return
    if world != opt.gpus and world > 1:
        opt.gpus = world
    if opt.profile:
        opt.no_cpu = True
    cuda_arm(opt, rank, world, local_rank)


if __name__ == '__main__':
    main()
