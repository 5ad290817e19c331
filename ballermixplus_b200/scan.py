"""Scan driver and the ``calcBaller`` seam -- SURVEY.md §8 rows a5/a6.

``calcBaller`` and ``Scan`` keep the reference's names, arguments and return values
(/root/reference/BalLeRMix+_v1.py:436-507 and :510-640); the work is done by the
CUDA library behind include/blmx.h.  ``Scan`` plans all centres of the run first
(windows.py), sends them to the GPU in one ``blmx_scan`` call and then writes the
rows with the reference's f-string formatting.  ``GenomeScan`` runs ``Scan``'s work over one input per
chromosome (``--inputList``).
"""
import os
import time
from datetime import datetime

import numpy as np

from . import balpos as balpos_mod, fastio, null as null_mod, refine as refine_mod, regions as regions_mod
from . import support as support_mod, targets as targets_mod, windows
from .native import Scanner
from .problem import GridOrder, build_problem

HEADER = 'physPos\tgenPos\tCLR\tx_hat\ts_hat\tA_hat\tnSites\n'


class DeviceScan:
    """A problem resident on one GPU plus the grid objects needed to decode results."""

    def __init__(self, InputData, NeutralSFS, NormalizedBetaBinom, Grids, device=0, group=None,
                 farfield=None):
        self._start(*build_problem(InputData, NeutralSFS, NormalizedBetaBinom, Grids), device, group, farfield)

    @classmethod
    def from_problem(cls, problem, order, device=0, group=None, farfield=None):
        """A ScanProblem built elsewhere (a segmented one: null.py) and its GridOrder."""
        self = cls.__new__(cls)
        self._start(problem, order, device, group, farfield)
        return self

    def _start(self, problem, order, device, group, farfield):
        self.problem, self.order = problem, order
        if farfield is None and os.environ.get('BLMX_FARFIELD'):
            farfield = int(os.environ['BLMX_FARFIELD'])
        self.scanner = Scanner(device=device, group=group, farfield=farfield).load(self.problem)

    def run(self, t, lo, hi):
        """-> (T float64[n], iA, ix, ia, nsites int32[n]); indices into the visiting order."""
        return self.scanner.scan(t, lo, hi)

    def run_profile(self, t, lo, hi):
        """``run`` plus the profiles of the likelihood surface -> (T, iA, ix, ia, nsites, TA, Tx, Ta, nsA)."""
        return self.scanner.scan_profile(t, lo, hi)

    def surface(self, t, lo, hi):
        """The whole likelihood surface of a few centres -> (S [n, n_A, n_x, n_a], nsA [n, n_A])."""
        return self.scanner.scan_surface(t, lo, hi)

    def load_refine(self, fA, n_fx, n_fa, row_of, SP):
        """Fine tables for ``refine`` (refine.py builds them)."""
        self.scanner.load_refine(fA, n_fx, n_fa, row_of, SP)

    def refine(self, t, lo, hi, box):
        """Box maxima of the fine grid -> (T, fA, fx, fa, nsites), fine indices (refine.py)."""
        return self.scanner.refine(t, lo, hi, box)

    def run_device(self, t, lo, hi, torch, device):
        """Same scan with the centres uploaded once and the results LEFT ON THE DEVICE as torch tensors
        (T float64, iA, ix, ia, nsites int32), asynchronous on torch's current stream: the multi-GPU path
        hands them to the NCCL gather without a host round trip."""
        n = len(t)
        d_t = torch.from_numpy(np.ascontiguousarray(t, dtype=np.float64)).to(device)
        d_lo = torch.from_numpy(np.ascontiguousarray(lo, dtype=np.int64)).to(device)
        d_hi = torch.from_numpy(np.ascontiguousarray(hi, dtype=np.int64)).to(device)
        T = torch.zeros(n, dtype=torch.float64, device=device)
        idx = [torch.full((n,), -1, dtype=torch.int32, device=device) for _ in range(4)]
        idx[3].zero_()
        self.scanner.scan_device(n, d_t.data_ptr(), d_lo.data_ptr(), d_hi.data_ptr(), T.data_ptr(),
                                 *[x.data_ptr() for x in idx], stream=torch.cuda.current_stream(device).cuda_stream)
        self._keep = (d_t, d_lo, d_hi)              # inputs stay alive until the stream has consumed them
        return (T, *idx)

    def run_split(self, t, lo, hi):
        """``run`` plus the rows of the balancing (alpha >= 1) and the sweep (alpha < 1) half of the grid, from one
        scan (blmx_scan_split, balpos.py) -> (rows, bal rows, pos rows), each (T, iA, ix, ia, nsites)."""
        return self.scanner.scan_split(t, lo, hi, balpos_mod.half_of_a(self.order.a))

    def run_split_device(self, t, lo, hi, torch, device):
        """``run_split`` with the results left on the device, as ``run_device`` -> 15 tensors: the rows, then the
        bal rows, then the pos rows, each (T float64, iA, ix, ia, nsites int32)."""
        n = len(t)
        d_t = torch.from_numpy(np.ascontiguousarray(t, dtype=np.float64)).to(device)
        d_lo = torch.from_numpy(np.ascontiguousarray(lo, dtype=np.int64)).to(device)
        d_hi = torch.from_numpy(np.ascontiguousarray(hi, dtype=np.int64)).to(device)
        out = []
        for _ in range(3):
            idx = [torch.full((n,), -1, dtype=torch.int32, device=device) for _ in range(4)]
            idx[3].zero_()
            out.append((torch.zeros(n, dtype=torch.float64, device=device), *idx))
        ptrs = [tuple(x.data_ptr() for x in rows) for rows in out]
        self.scanner.scan_split_device(n, d_t.data_ptr(), d_lo.data_ptr(), d_hi.data_ptr(),
                                       balpos_mod.half_of_a(self.order.a), ptrs[0], ptrs[1:],
                                       stream=torch.cuda.current_stream(device).cuda_stream)
        self._keep = (d_t, d_lo, d_hi)
        return tuple(x for rows in out for x in rows)

    def decode(self, T, iA, ix, ia, ns):
        return self.order.decode(T, iA, ix, ia, ns)

    def close(self):
        self.scanner.close()


class Unloaded:
    """Stands in for the DeviceScan of an input none of whose rows is scanned (``--targets`` keeps no row of it that
    is not a gap row): the writers need only its grid order, so nothing is loaded on a GPU."""

    def __init__(self, grids):
        self.order = GridOrder(grids)

    def close(self):
        pass


_cache = {}       # 'objs': the four host objects of the resident problem (strong references), 'dev': its DeviceScan


def clear_cache():
    """Release the GPU-resident problem that ``calcBaller`` keeps between calls."""
    dev = _cache.pop('dev', None)
    _cache.clear()
    if dev is not None:
        dev.close()


def calcBaller(window_indice, testSite, InputData, NeutralSFS, NormalizedBetaBinom, Grids):
    """Drop-in for the reference function (v1:436): one centre, same 5-element result.

    ``window_indice`` must be a contiguous ascending index range, which is all the
    reference's callers ever pass (v1:538,572,589,606).  The problem built from the four
    objects stays on the GPU for the next call with the SAME objects (compared by identity,
    and held here so that their ids cannot be recycled); mutating them in place between
    calls is not detected -- call ``clear_cache()`` after doing so, and to free the device memory.
    """
    objs = (InputData, NeutralSFS, NormalizedBetaBinom, Grids)
    held = _cache.get('objs')
    if held is None or any(a is not b for a, b in zip(held, objs)):
        clear_cache()
        _cache['dev'] = DeviceScan(*objs)
        _cache['objs'] = objs
    dev = _cache['dev']
    w = np.asarray(window_indice)
    if len(w) == 0:
        return [0., 0., 0., 0., 0.]
    if len(w) > 1 and not np.all(np.diff(w) == 1):
        raise ValueError('window_indice must be a contiguous ascending range')
    T, iA, ix, ia, ns = dev.run([float(testSite)], [int(w[0])], [int(w[-1])])
    return dev.decode(T[0], iA[0], ix[0], ia[0], ns[0])


def format_rows(plan, order, T, iA, ix, ia, ns):
    """Output lines for a plan and its results (v1:535,540,574,591,607), formatted by Python
    exactly as the reference's f-strings do."""
    lines = []
    f0, f1 = plan.f0, plan.f1
    for j in range(len(plan)):
        if plan.gap[j]:
            lines.append(f0[j])
            continue
        Tm, xh, ah, Ah, w = order.decode(T[j], iA[j], ix[j], ia[j], ns[j])
        lines.append(f'{f0[j]}\t{f1[j]}\t{Tm}\t{xh}\t{ah}\t{Ah}\t{w}\n')
    return lines


def write_scan(outfile, plan, order, T, iA, ix, ia, ns):
    """Write the output file: the C++ writer for site-centred scans without gap rows (same bytes,
    tests/test_fastio.py), the Python formatter otherwise."""
    if plan.site_phys is not None and not np.any(plan.gap):
        texts = [[f'{v}' for v in grid] for grid in (order.A, order.x, order.a)]
        if fastio.write_rows(outfile, HEADER, plan.site_phys, plan.site_gen, T, iA, ix, ia, ns, *texts):
            return
    with open(outfile, 'w') as scores:
        scores.write(HEADER)
        scores.writelines(format_rows(plan, order, T, iA, ix, ia, ns))


def _world():
    """(rank, world, local_rank) of a torchrun launch, (0, 1, 0) otherwise."""
    return (int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1')),
            int(os.environ.get('LOCAL_RANK', '0')))


def _local_world():
    """Ranks of this launch that run on THIS node (torchrun exports LOCAL_WORLD_SIZE)."""
    return int(os.environ.get('LOCAL_WORLD_SIZE', os.environ.get('WORLD_SIZE', '1')))


def ranks_own_a_gpu():
    """True when every rank on this node can have its own CUDA device."""
    from .native import device_count
    return device_count() >= _local_world()


def scan_rows_multi_gpu(dev, t, lo, hi, rank, world, local_rank, keep_group=False, split=False):
    """One process per GPU (torchrun): every rank scans a cost-balanced contiguous slice of the centres,
    one gather brings the rows to rank 0 (sharding.py).  When every rank of the node has its own GPU the rows
    stay on the device from the scan kernel to the NCCL gather (``DeviceScan.run_device``); when several ranks
    share one device (tests on a one-GPU box) the gather runs over gloo on host tensors.  Returns the five
    result arrays on rank 0 and None elsewhere.  ``keep_group``: leave the process group this call starts
    running for a later scan (``end_group`` ends it).  ``split`` (``--balPos``): the scan is ``run_split`` and 15
    arrays come back, the rows and then the bal and the pos rows."""
    seq = (dev.problem.genpos, dev.problem.A, t, lo, hi, getattr(dev.problem, 'seg_start', None))
    return scan_seqs_multi_gpu([seq], lambda i: dev, dev.scanner.device, rank, world, keep_group=keep_group,
                               split=split)


def scan_seqs_multi_gpu(seqs, open_dev, device, rank, world, keep_group=False, release=False, split=False):
    """``scan_rows_multi_gpu`` over several sequences (sharding.scan_sharded_seqs): the centres of all of them are
    cut into cost-balanced ranges, and a rank scans only the sequences its range touches, on the DeviceScan
    ``open_dev(i)`` gives for sequence i.  ``seqs``: one (genpos, A, t, lo, hi, seg_start) per sequence.
    ``release``: close each DeviceScan once its rows are computed, so that one sequence at a time is resident.
    Returns the five result arrays of the concatenated centre list on rank 0 and None elsewhere (with ``split``:
    the 15 of ``run_split``, gathered in one wider block, sharding.pack_split_rows)."""
    import torch
    import torch.distributed as dist
    from . import sharding
    own_gpu = ranks_own_a_gpu()
    started = not dist.is_initialized()
    if started:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29500')
        if own_gpu:
            torch.cuda.set_device(device)
            dist.init_process_group('nccl', rank=rank, world_size=world,
                                    device_id=torch.device('cuda', device))
        else:
            dist.init_process_group('gloo', rank=rank, world_size=world)

    where = torch.device('cuda', device) if own_gpu else torch.device('cpu')

    def scan_fn(i, ts, los, his):
        dev = open_dev(i)
        try:
            if own_gpu:
                got = (dev.run_split_device if split else dev.run_device)(ts, los, his, torch, where)
                if release:             # the rows stay on the device; the handle may go once they are written
                    torch.cuda.current_stream(where).synchronize()
                return got
            if split:
                return tuple(torch.from_numpy(np.ascontiguousarray(a)) for r in dev.run_split(ts, los, his) for a in r)
            return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in dev.run(ts, los, his))
        finally:
            if release:
                dev.close()

    ok = False
    try:
        got = sharding.scan_sharded_seqs(seqs, rank, world, scan_fn, dist, torch, device=where, split=split)
        ok = True
        return None if got is None else tuple(a.cpu().numpy() for a in got)
    finally:
        if started and not (ok and keep_group):
            if ok:                      # a rank that failed must not wait for the others (they would hang with it)
                dist.barrier()
            dist.destroy_process_group()


def end_group():
    """End the process group a ``scan_rows_multi_gpu(..., keep_group=True)`` left running."""
    import torch.distributed as dist
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()


#: centres per blmx_scan_profile call of ``Scan(..., support=...)``: bounds the host memory of the profiles
SUPPORT_CHUNK = 65536


def scan_with_support(dev, t, lo, hi, q):
    """The rows of ``dev.run`` plus their support intervals (support.py), scanned in chunks of centres so that
    only the intervals of a genome-sized run stay in host memory -> (rows, intervals)."""
    n = len(t)
    rows = [np.zeros(n), *(np.full(n, -1, np.int32) for _ in range(3)), np.zeros(n, np.int32)]
    iv = {k: np.full(n, -1, np.int32) for k in ('A_lo', 'A_hi', 'x_lo', 'x_hi', 's_lo', 's_hi')}
    for b in range(0, n, SUPPORT_CHUNK):
        e = min(n, b + SUPPORT_CHUNK)
        T, iA, ix, ia, ns, TA, Tx, Ta, _ = dev.run_profile(t[b:e], lo[b:e], hi[b:e])
        for col, v in zip(rows, (T, iA, ix, ia, ns)):
            col[b:e] = v
        for k, v in support_mod.support_intervals(T, iA, TA, Tx, Ta, dev.order, q).items():
            iv[k][b:e] = v
    return tuple(rows), iv


INTERVAL_KEYS = ('A_lo', 'A_hi', 'x_lo', 'x_hi', 's_lo', 's_hi')


def empty_rows(n):
    """Result arrays (T, iA, ix, ia, nsites) of n rows that have not been scanned (gap rows stay so)."""
    return (np.zeros(n), *(np.full(n, -1, np.int32) for _ in range(3)), np.zeros(n, np.int32))


def check_options(world, support, support_drop, refine, refine_steps, null, pvalues, regions=None, threshold=None,
                  balpos=None, grids=None):
    """Refuse option combinations before any work -> (support_drop, refine_steps, threshold), checked.  ``balpos``
    needs alpha values of ``grids`` on both sides of 1."""
    if balpos is not None:
        balpos_mod.check_grid(grids.abeta)
    if support is not None or regions is not None:
        support_drop = support_mod.check_drop(support_drop)
    if support is not None and world > 1:
        raise ValueError('--support runs on one GPU: launch without torchrun (WORLD_SIZE > 1)')
    if refine is not None:
        refine_steps = refine_mod.check_steps(refine_steps)
        if world > 1:
            raise ValueError('--refine runs on one GPU: launch without torchrun (WORLD_SIZE > 1)')
    if (null is None) != (pvalues is None):
        raise ValueError('--null and --pvalues go together')
    if threshold is not None:
        if regions is None:
            raise ValueError('--threshold needs --regions')
        threshold = regions_mod.check_threshold(threshold)
    if regions is not None and threshold is None and null is None:
        raise ValueError(REGIONS_NEED_A_CUT)
    return support_drop, refine_steps, threshold


REGIONS_NEED_A_CUT = ('--regions needs a cut: --threshold C, or --null (the 0.95 quantile of the per-replicate '
                      'maximum CLR)')


def open_outputs(*paths):
    """Open (truncate) every output file given (None: not asked for).  The reference opens its output before
    it computes anything (v1:516,551,582,600): a bad path must fail now, not after the scan."""
    for p in paths:
        if p is not None:
            with open(p, 'w'):
                pass


def scan_plan(dev, t, lo, hi, gap, support_drop=None, balpos=False):
    """The rows of a plan's arrays on one GPU (gap rows, and rows ``--targets`` skips, passed in ``gap``, left
    unscanned), with ``support_drop`` their support intervals, and with ``balpos`` the rows of the two halves of
    the grid (``--balPos``) -> (rows, intervals or None, (bal rows, pos rows) or None).  ``--balPos`` alone takes
    the rows and the halves from one ``run_split``; with ``--support`` the profile scan keeps the rows and a second
    scan, ``run_split``, gives the halves (DESIGN.md §3.14)."""
    rows = empty_rows(len(t))
    iv = {k: np.full(len(t), -1, np.int32) for k in INTERVAL_KEYS} if support_drop is not None else None
    halves = (empty_rows(len(t)), empty_rows(len(t))) if balpos else None
    live = np.flatnonzero(~gap)
    if len(live):
        got_halves = ()
        if support_drop is not None:
            got, got_iv = scan_with_support(dev, t[live], lo[live], hi[live], support_drop)
            for k, v in got_iv.items():
                iv[k][live] = v
            if balpos:
                got_halves = dev.run_split(t[live], lo[live], hi[live])[1:]
        elif balpos:
            got, *got_halves = dev.run_split(t[live], lo[live], hi[live])
        else:
            got = dev.run(t[live], lo[live], hi[live])
        for dst, src in zip((rows,) + (halves or ()), (got,) + tuple(got_halves)):
            for col, v in zip(dst, src):
                col[live] = v
    return rows, iv, halves


def select_rows(keep, plan, arrays, rows, iv):
    """What a run writes -> (plan, arrays, rows, intervals): everything when ``keep`` is None, else only the rows
    ``keep`` selects (``--targets``), in order.  ``arrays`` = (t, lo, hi, gap) of ``plan``, ``iv`` the support
    intervals or None."""
    if keep is None:
        return plan, arrays, rows, iv
    idx = np.flatnonzero(keep)
    return (plan.take(idx), tuple(a[idx] for a in arrays), tuple(c[idx] for c in rows),
            None if iv is None else {k: v[idx] for k, v in iv.items()})


def kept_halves(keep, halves):
    """The half rows of ``--balPos`` at the rows ``keep`` selects (as ``select_rows``; None passes through)."""
    if keep is None or halves is None:
        return halves
    idx = np.flatnonzero(keep)
    return tuple(tuple(c[idx] for c in h) for h in halves)


def skipped(gap, keep):
    """Rows not scanned: the gap rows, and with ``--targets`` (``keep``) every row it does not keep."""
    return gap if keep is None else gap | ~keep


def write_support(path, plan, order, rows, iv):
    with open(path, 'w') as fh:
        fh.write(support_mod.SUPPORT_HEADER)
        fh.writelines(support_mod.format_support(plan, order, *rows, iv))


def write_refine(dev, neutral, sel, K, path, plan, t, lo, hi, rows):
    """Refine ``rows`` on ``dev`` (refine.py) and write the refine file -> (fine grid, refined rows, moved)."""
    T, iA, ix, ia, ns = rows
    grid, refined = refine_mod.refine_rows(dev, neutral, sel, K, t, lo, hi, iA, ix, ia)
    move = refine_mod.moved(grid, T, iA, ix, ia, refined)
    with open(path, 'w') as fh:
        fh.write(HEADER)
        fh.writelines(refine_mod.format_refined(plan, format_rows(plan, dev.order, *rows), grid, refined, move))
    print(f'refine (K = {grid.K}): {int(move.sum())} of {int((iA >= 0).sum())} rows with T > 0 moved to a '
          f'finer grid point')
    return grid, refined, move


def write_pvalues(path, plan, order, rows, gap, null_T):
    """p-values of ``rows`` against the null CLRs (gap rows NA), written to ``path`` -> p."""
    p = null_mod.pvalues(np.where(gap, np.nan, rows[0]), null_T)
    with open(path, 'w') as fh:
        fh.writelines(null_mod.format_pvalues(plan, order, *rows, p))
    return p


class Scan:
    """Same constructor as the reference class (v1:613); runs the scan and writes ``outfile``.

    Launched under ``torchrun --nproc-per-node N`` the centres are sharded over N GPUs and rank 0
    writes the file (the other ranks write nothing).

    ``support`` (a path): also write, per row of ``outfile``, the support intervals of A_hat, x_hat and
    s_hat at a drop of ``support_drop`` in T units (support.py: intervals of a composite likelihood, not
    calibrated confidence intervals).  One GPU only.

    ``null`` (a replicate list) and ``pvalues`` (a path), given together: also scan the neutral replicates the
    list names with the same flags and tables, as one segmented problem, and write, per row of ``outfile``,
    its empirical p-value against the pooled null CLRs (null.py).  ``outfile`` is the same either way.

    ``refine`` (a path): also write ``outfile`` again with every row with T > 0 replaced by the best point of a
    grid ``refine_steps`` times finer inside a box around its maximum, where that point beats the row's CLR
    (refine.py).  One GPU only.  ``outfile``, the support and the p-value files stay on the coarse grid.

    ``regions`` (a path): also write one line per run of rows with CLR >= the cut, with its peak, the position
    support interval at drop ``support_drop`` and, with ``null``, a region p-value (regions.py).  The cut is
    ``threshold``, or without it the 0.95 quantile of the per-replicate maximum CLR of ``null``.  ``input_name``
    fills the file's first column (default: the file name of ``outfile``).  Works under torchrun; no other file
    changes.

    ``targets`` (a ``targets.Targets``): scan only the rows whose physPos lies in a target of the input named
    ``input_name``; every file then holds the header and, in order, exactly the lines of the full run at those rows
    (``results`` too holds those rows only).  A row not kept ends a region and stops a position interval, as a gap
    row does.

    ``balpos`` (a path): also write, per row of ``outfile``, the row maximum over the balancing (alpha >= 1) and
    over the sweep (alpha < 1) half of the grid (balpos.py), from the same scan.  Works under torchrun; no other
    file changes."""

    def __init__(self, InputData, NeutralSFS, NormalizedBetaBinom, Grids, outfile, fixSize=False,
                 r=0, s=1, phys=False, noCenter=False, device=0, support=None,
                 support_drop=support_mod.DEFAULT_DROP, null=None, pvalues=None, refine=None,
                 refine_steps=refine_mod.DEFAULT_STEPS, regions=None, threshold=None, input_name=None,
                 targets=None, balpos=None):
        rank, world, local_rank = _world()
        support_drop, refine_steps, threshold = check_options(world, support, support_drop, refine, refine_steps,
                                                              null, pvalues, regions, threshold, balpos, Grids)
        plan = windows.make_plan(InputData, fixSize=fixSize, r=r, s=s, phys=phys, noCenter=noCenter)
        name = os.path.basename(outfile) if input_name is None else input_name
        keep = None if targets is None else targets.keep(name, plan)
        if rank == 0:
            print('writing output to %s' % (outfile))
            open_outputs(outfile, support, pvalues, refine, regions, balpos)
            if keep is not None:
                print(targets_mod.kept_line(name, keep))
        setup = None
        if null is not None:
            setup = null_mod.NullSetup(null, InputData, NeutralSFS, NormalizedBetaBinom, Grids, fixSize=fixSize,
                                       r=r, s=s, phys=phys, noCenter=noCenter)
        if world > 1:
            from .native import device_count
            device = local_rank % max(1, device_count())
        t, lo, hi, gap = plan.arrays()
        skip = skipped(gap, keep)
        if keep is not None and skip.all():
            dev = Unloaded(Grids)
        else:
            dev = DeviceScan(InputData, NeutralSFS, NormalizedBetaBinom, Grids, device=device)
        try:
            if world > 1:
                live = np.flatnonzero(~skip)
                rows, iv = empty_rows(len(plan)), None
                halves = (empty_rows(len(plan)), empty_rows(len(plan))) if balpos is not None else None
                if len(live):
                    got = scan_rows_multi_gpu(dev, t[live], lo[live], hi[live], rank, world, local_rank,
                                              keep_group=setup is not None, split=balpos is not None)
                    if got is not None:
                        for col, v in zip(rows + sum(halves or (), ()), got):
                            col[live] = v
            else:
                rows, iv, halves = scan_plan(dev, t, lo, hi, skip, support_drop if support is not None else None,
                                             balpos=balpos is not None)
            wplan, (wt, wlo, whi, wgap), wrows, wiv = select_rows(keep, plan, (t, lo, hi, gap), rows, iv)
            self.results = wrows if rank == 0 else None
            if rank == 0:
                write_scan(outfile, wplan, dev.order, *wrows)
                if balpos is not None:
                    self.halves = kept_halves(keep, halves)
                    balpos_mod.write_balpos(balpos, wplan, dev.order, *self.halves)
                if support is not None:
                    self.support = wiv
                    write_support(support, wplan, dev.order, wrows, wiv)
                if refine is not None:
                    self._refine(dev, NeutralSFS, NormalizedBetaBinom, refine_steps, refine, wplan, wt, wlo, whi)
        finally:
            dev.close()
        maxima = None
        if setup is not None:
            null_T = self._scan_null(setup, device, rank, world, local_rank)
            if rank == 0:
                self.null = null_T
                for line in null_mod.summary(null_T, setup.rep, setup.n_replicates):
                    print(line)
                self.pvalues = write_pvalues(pvalues, wplan, dev.order, wrows, wgap, null_T)
                maxima = null_mod.replicate_maxima(null_T, setup.rep, setup.n_replicates)
        if regions is not None and rank == 0:
            cut, source = regions_mod.cut_of(threshold, maxima)
            self.regions = regions_mod.region_lines(name, plan, dev.order, rows, skip, cut, support_drop, maxima)
            print(regions_mod.write_regions(regions, [self.regions], cut, source, support_drop))
        if rank == 0:
            print(f'{datetime.now()}. Scan finished.')

    def _refine(self, dev, neutral, sel, K, path, plan, t, lo, hi):
        """Refine the rows of ``self.results`` on ``dev`` and write the refine file."""
        self.refine_grid, self.refined, self.moved = write_refine(dev, neutral, sel, K, path, plan, t, lo, hi,
                                                                  self.results)

    @staticmethod
    def _scan_null(setup, device, rank, world, local_rank):
        """CLR of every null row (rank 0; None elsewhere): one segmented load, one scan or one sharded scan."""
        ndev = DeviceScan.from_problem(setup.problem, setup.order, device=device)
        try:
            if world > 1:
                got = scan_rows_multi_gpu(ndev, setup.t, setup.lo, setup.hi, rank, world, local_rank)
                end_group()
                return None if got is None else got[0]
            return ndev.run(setup.t, setup.lo, setup.hi)[0]
        finally:
            ndev.close()


def input_list(path):
    """Inputs of ``--inputList``: the files the list ``path`` names, by the rules of ``null.read_list`` (paths
    relative to the list's directory, blank and '#' lines skipped).  Every input writes a file named as it is,
    so two inputs with the same file name are refused.  Raises before any input is read."""
    paths = null_mod.read_list(path, flag='--inputList', item='input')
    seen = {}
    for p in paths:
        name = os.path.basename(p)
        if name in seen:
            raise ValueError(f'--inputList: inputs {seen[name]} and {p} have the same file name {name}; '
                             f'their outputs would overwrite each other')
        seen[name] = p
    return paths


def list_outputs(inputs, **dirs):
    """The files of ``--inputList``: for every directory given (None: option not used), one file per input named
    as the input -> {option: [paths]}.  Two options naming the same directory, or an output that is one of the
    inputs, is refused."""
    files = {k: [os.path.join(d, os.path.basename(p)) for p in inputs] for k, d in dirs.items() if d is not None}
    out = [os.path.realpath(p) for paths in files.values() for p in paths]
    if len(set(out)) != len(out):
        raise ValueError('--inputList: two output options name the same directory')
    clash = set(out) & {os.path.realpath(p) for p in inputs}
    if clash:
        raise ValueError(f'--inputList: output {sorted(clash)[0]} would overwrite an input')
    return files


def check_regions_file(path, inputs, files, reads=()):
    """``--regions`` of ``--inputList`` names one file for the whole genome: refused when it is a directory, when
    its directory does not exist, or when it is a file the run reads (an input, ``reads``) or writes (``files``,
    from ``list_outputs``)."""
    if os.path.isdir(path):
        raise ValueError(f'--inputList: --regions {path} is a directory; it names one file for the whole genome')
    parent = os.path.dirname(os.path.abspath(path))
    if not os.path.isdir(parent):
        raise ValueError(f'--inputList: --regions {path}: directory {parent} does not exist')
    if names_one_of(path, list(inputs) + list(reads) + [f for fs in files.values() for f in fs]):
        raise ValueError(f'--inputList: --regions {path} is a file this run reads or writes')


def names_one_of(path, paths):
    """True when ``path`` names the same file as one of ``paths`` (None entries ignored), links and relative parts
    resolved."""
    return os.path.realpath(path) in {os.path.realpath(p) for p in paths if p is not None}


class GenomeScan:
    """Scan one input per chromosome (``--inputList``) as one run: one process, one CUDA context, one null.

    ``inputs``: the input paths (``input_list``); ``read(path)`` -> (InputData, NormalizedBetaBinom) of one input,
    after ``NeutralSFS.get_neut_probs`` of it, as the one-input command line builds them, so that each input keeps
    the minCount it derives and its own tables.  Every input is loaded as its own problem on its own handle (not
    one segmented problem: class order and block alignment would differ), and every file it writes is the file a
    one-input ``Scan`` with the same options writes for it.  ``outdir`` (and ``support``, ``pvalues``, ``refine``
    when given) are directories; input ``chr7.txt`` writes ``outdir/chr7.txt`` and so on.  Every output file is
    opened before any input is read.

    One GPU: the inputs are read, scanned and written one after another, with one problem resident at a time.
    Under torchrun the genome is sharded, not each input: the centres of all inputs are cut into cost-balanced
    ranges (``scan_seqs_multi_gpu``), each rank loads only the inputs its range touches, one gather brings every
    row to rank 0, which writes the files.  ``support`` and ``refine`` are one-GPU options, as in ``Scan``.

    ``null``/``pvalues``: the replicates are set up and scanned once (the null depends on the run's flags and
    spectrum, not on the input: ``null.flags_of``), and every input's p-values come from that pooled null.

    ``regions`` (a path, not a directory) and ``threshold``: one regions file for the whole genome (``Scan``), the
    lines of every input in input order, collected as its rows become available and written at the end.

    ``targets`` (a ``targets.Targets``, inputs named by file name): each input keeps only the rows in its targets, as
    in ``Scan``; the centres of the kept rows alone are scanned (and sharded under torchrun), and an input with no
    kept row to scan is read and planned but never loaded on a GPU.

    ``balpos`` (a directory, like ``outdir``): the ``--balPos`` file of every input, as ``Scan`` writes it; on one GPU
    and under torchrun, where the half rows travel in the same gather as the rows."""

    def __init__(self, inputs, read, NeutralSFS, Grids, outdir, fixSize=False, r=0, s=1, phys=False,
                 noCenter=False, device=0, support=None, support_drop=support_mod.DEFAULT_DROP, null=None,
                 pvalues=None, refine=None, refine_steps=refine_mod.DEFAULT_STEPS, regions=None, threshold=None,
                 targets=None, balpos=None):
        rank, world, local_rank = _world()
        support_drop, refine_steps, threshold = check_options(world, support, support_drop, refine, refine_steps,
                                                              null, pvalues, regions, threshold, balpos, Grids)
        self.inputs = list(inputs)
        self.files = list_outputs(self.inputs, out=outdir, support=support, pvalues=pvalues, refine=refine,
                                  balpos=balpos)
        if regions is not None:
            check_regions_file(regions, self.inputs, self.files)
        if rank == 0:
            print(f'writing {len(self.inputs)} outputs to {outdir}')
            for paths in self.files.values():
                open_outputs(*paths)
            open_outputs(regions)
        self.kw = dict(fixSize=fixSize, r=r, s=s, phys=phys, noCenter=noCenter)
        self.read, self.neutral, self.grids, self.null = read, NeutralSFS, Grids, null
        self.region_file, self.threshold, self.drop = regions, threshold, support_drop
        self.maxima, self.cut, self.regions = None, None, []
        self.targets, self.kept = targets, []
        if world > 1:
            from .native import device_count
            self._sharded(local_rank % max(1, device_count()), rank, world, local_rank)
        else:
            self._one_gpu(device, support_drop, refine_steps)
        if rank == 0:
            if regions is not None:
                print(regions_mod.write_regions(regions, self.regions, *self.cut, support_drop))
            if targets is not None:
                print(f'--targets: {sum(k for k, _ in self.kept)} of {sum(n for _, n in self.kept)} planned rows '
                      f'kept in {sum(1 for k, _ in self.kept if k)} of {len(self.kept)} inputs')
            print(f'{datetime.now()}. Scan finished.')

    def _null(self, data, sel, device, rank, world, local_rank):
        """Set up and scan the replicates once -> (NullSetup, null CLRs on rank 0)."""
        setup = null_mod.NullSetup(self.null, data, self.neutral, sel, self.grids, **self.kw)
        null_T = Scan._scan_null(setup, device, rank, world, local_rank)
        if rank == 0:
            self._null_summary(setup, null_T)
        return setup, null_T

    def _null_summary(self, setup, null_T):
        """Print the null's quantiles and keep its per-replicate maxima (the regions' cut and p-values)."""
        for line in null_mod.summary(null_T, setup.rep, setup.n_replicates):
            print(line)
        self.maxima = null_mod.replicate_maxima(null_T, setup.rep, setup.n_replicates)

    def _add_regions(self, path, plan, order, rows, gap):
        """Collect the regions of one input (``--regions``); the null, if any, has been scanned."""
        if self.region_file is None:
            return
        if self.cut is None:
            self.cut = regions_mod.cut_of(self.threshold, self.maxima)
        self.regions.append(regions_mod.region_lines(os.path.basename(path), plan, order, rows, gap, self.cut[0],
                                                     self.drop, self.maxima))

    def _plan(self, path, data):
        """-> (plan, t, lo, hi, gap, keep, skip) of one input (``keep`` None without ``--targets``)."""
        plan = windows.make_plan(data, **self.kw)
        t, lo, hi, gap = plan.arrays()
        keep = None
        if self.targets is not None:
            keep = self.targets.keep(os.path.basename(path), plan)
            self.kept.append((int(np.count_nonzero(keep)), len(plan)))
            print(targets_mod.kept_line(os.path.basename(path), keep))
        return plan, t, lo, hi, gap, keep, skipped(gap, keep)

    def _one_gpu(self, device, support_drop, refine_steps):
        null_T = None
        for i, path in enumerate(self.inputs):
            data, sel = self.read(path)
            if self.null is not None and null_T is None:
                _, null_T = self._null(data, sel, device, 0, 1, 0)
            plan, t, lo, hi, gap, keep, skip = self._plan(path, data)
            t0 = time.perf_counter()
            if keep is not None and skip.all():
                dev = Unloaded(self.grids)
            else:
                dev = DeviceScan(data, self.neutral, sel, self.grids, device=device)
            try:
                rows, iv, halves = scan_plan(dev, t, lo, hi, skip, support_drop if 'support' in self.files else None,
                                             balpos='balpos' in self.files)
                dt = time.perf_counter() - t0
                wplan, (wt, wlo, whi, wgap), wrows, wiv = select_rows(keep, plan, (t, lo, hi, gap), rows, iv)
                write_scan(self.files['out'][i], wplan, dev.order, *wrows)
                if halves is not None:
                    balpos_mod.write_balpos(self.files['balpos'][i], wplan, dev.order, *kept_halves(keep, halves))
                if wiv is not None:
                    write_support(self.files['support'][i], wplan, dev.order, wrows, wiv)
                if 'refine' in self.files:
                    write_refine(dev, self.neutral, sel, refine_steps, self.files['refine'][i], wplan, wt, wlo, whi,
                                 wrows)
            finally:
                dev.close()
            if null_T is not None:
                write_pvalues(self.files['pvalues'][i], wplan, dev.order, wrows, wgap, null_T)
            self._add_regions(path, plan, dev.order, rows, skip)
            print(f'{os.path.basename(path)}: {len(plan)} rows, scanned in {dt:.3f} s, written to '
                  f'{self.files["out"][i]}')

    def _sharded(self, device, rank, world, local_rank):
        items = []
        for path in self.inputs:
            data, sel = self.read(path)
            plan, t, lo, hi, gap, keep, skip = self._plan(path, data)
            items.append((data, sel, plan, t, lo, hi, gap, keep, skip, np.flatnonzero(~skip)))
        setup = None
        if self.null is not None:           # prepared now, scanned after the genome (the process group is kept)
            setup = null_mod.NullSetup(self.null, items[0][0], self.neutral, items[0][1], self.grids, **self.kw)
        A = np.array([float(v) for v in GridOrder(self.grids).A])
        # an input with no centre here is in no rank's range, so it is never loaded (sharding.pieces)
        seqs = [(d.genPos, A, t[live], lo[live], hi[live], None) for d, _, _, t, lo, hi, _, _, _, live in items]

        def open_dev(i):
            return DeviceScan(items[i][0], self.neutral, items[i][1], self.grids, device=device)

        t0 = time.perf_counter()
        got = None
        if sum(len(s[2]) for s in seqs):
            got = scan_seqs_multi_gpu(seqs, open_dev, device, rank, world, keep_group=setup is not None,
                                      release=True, split='balpos' in self.files)
        dt = time.perf_counter() - t0
        null_T = None
        if setup is not None:
            null_T = Scan._scan_null(setup, device, rank, world, local_rank)
        if rank != 0:
            return
        if null_T is not None:
            self._null_summary(setup, null_T)
        print(f'genome: {sum(len(s[2]) for s in seqs)} centres of {len(items)} inputs scanned on {world} ranks '
              f'in {dt:.3f} s')
        order = GridOrder(self.grids)
        o = 0
        for i, (data, sel, plan, t, lo, hi, gap, keep, skip, live) in enumerate(items):
            rows = empty_rows(len(plan))
            halves = (empty_rows(len(plan)), empty_rows(len(plan))) if 'balpos' in self.files else None
            if got is not None:
                for col, v in zip(rows + sum(halves or (), ()), got):
                    col[live] = v[o:o + len(live)]
            o += len(live)
            wplan, (_, _, _, wgap), wrows, _ = select_rows(keep, plan, (t, lo, hi, gap), rows, None)
            write_scan(self.files['out'][i], wplan, order, *wrows)
            if halves is not None:
                balpos_mod.write_balpos(self.files['balpos'][i], wplan, order, *kept_halves(keep, halves))
            if null_T is not None:
                write_pvalues(self.files['pvalues'][i], wplan, order, wrows, wgap, null_T)
            self._add_regions(self.inputs[i], plan, order, rows, skip)
            print(f'{os.path.basename(self.inputs[i])}: {len(plan)} rows, written to {self.files["out"][i]}')
