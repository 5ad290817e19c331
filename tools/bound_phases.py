"""Split of bound_kernel's time between its phases on the benchmark's workload (bench.py --gpus 1:
bench.make_genome / make_problem at --sites, centres on every --stride-th site, every chromosome resident).

Uses the -DBLMX_BOUND_PHASES build (libblmx_phases.so, built by __graft_entry__.build_cuda(phases=True) when
missing; --lib takes another build of the same kind).  Each warp of bound_kernel adds the clock64() cycles of its
set-up (item window), its per-class gather (counts and alpha sums) and its grid-point phase (the bound at every
grid point); the tool sums them over --steps steps after one warm-up step and reports each phase's share of the
summed warp cycles, with the pruned-item count and the card it ran on.  Writes JSON to --out and prints it.

    python tools/bound_phases.py --out profiles/r8_bound_phases.json
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

PHASES = ('setup', 'gather', 'grid_points')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sites', type=int, default=10_000_000)
    ap.add_argument('--stride', type=int, default=None)
    ap.add_argument('--steps', type=int, default=2)
    ap.add_argument('--lib', default=None, help='a -DBLMX_BOUND_PHASES build (default: libblmx_phases.so)')
    ap.add_argument('--out', default=None)
    opt = ap.parse_args()
    if opt.lib is None:
        import __graft_entry__
        opt.lib = __graft_entry__.build_cuda(phases=True)
    os.environ['BLMX_LIB'] = os.path.abspath(opt.lib)             # read when ballermixplus_b200.native loads

    import bench
    from ballermixplus_b200 import native
    from ballermixplus_b200.native import Scanner
    from bound_cost import gpu_info

    L = native.lib()
    if not hasattr(L, 'blmx_last_bound_cycles'):
        sys.exit(f'{opt.lib} was not built with -DBLMX_BOUND_PHASES')
    L.blmx_last_bound_cycles.argtypes = [C.c_void_p, C.POINTER(C.c_uint64 * 3)]
    L.blmx_last_bound_cycles.restype = C.c_int

    stride = bench.BASE_STRIDE if opt.stride is None else opt.stride
    problems = bench.make_problem(bench.make_genome(opt.sites))
    plans = bench.plan_centres(problems, stride)
    scanners = [Scanner(device=0).load(p) for p in problems]

    def step():
        cyc = [0, 0, 0]
        pruned = items = 0
        for sc, (t, lo, hi), p in zip(scanners, plans, problems):
            sc.scan(t, lo, hi)
            v = (C.c_uint64 * 3)()
            if L.blmx_last_bound_cycles(sc._h, C.byref(v)) != 0:
                sys.exit('blmx_last_bound_cycles failed')
            cyc = [a + b for a, b in zip(cyc, v)]
            pruned += sc.counters_all()['pruned_items']
            items += len(t) * len(p.A)
        return cyc, pruned, items

    step()                                                       # module load, scratch allocations
    total = [0, 0, 0]
    for _ in range(opt.steps):
        cyc, pruned, items = step()
        total = [a + b for a, b in zip(total, cyc)]
    s = sum(total)
    out = {'gpu': gpu_info(), 'lib': os.path.basename(opt.lib), 'sites': opt.sites, 'chromosomes': len(problems),
           'centre_stride': stride, 'items_per_step': int(items), 'pruned_items_per_step': int(pruned),
           'steps': opt.steps,
           'warp_cycles_per_step': {k: v / opt.steps for k, v in zip(PHASES, total)},
           'share': {k: v / s if s else 0.0 for k, v in zip(PHASES, total)},
           'timing': 'clock64() deltas per warp of bound_kernel, summed over warps (lane 0 of each); a share of '
                     'warp-resident cycles, not of kernel time'}
    for sc in scanners:
        sc.close()
    line = json.dumps(out, indent=1)
    print(line)
    if opt.out:
        os.makedirs(os.path.dirname(os.path.abspath(opt.out)), exist_ok=True)
        with open(opt.out, 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
