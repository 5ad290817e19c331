"""Scan driver and the ``calcBaller`` seam -- SURVEY.md §8 rows a5/a6.

``calcBaller`` and ``Scan`` keep the reference's names, arguments and return values
(/root/reference/BalLeRMix+_v1.py:436-507 and :510-640); the work is done by the
CUDA library behind include/blmx.h.  ``Scan`` plans all centres of the run first
(windows.py), sends them to the GPU in one ``blmx_scan`` call and then writes the
rows with the reference's f-string formatting.
"""
import os
from datetime import datetime

import numpy as np

from . import fastio, null as null_mod, refine as refine_mod, support as support_mod, windows
from .native import Scanner
from .problem import build_problem

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

    def decode(self, T, iA, ix, ia, ns):
        return self.order.decode(T, iA, ix, ia, ns)

    def close(self):
        self.scanner.close()


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


def scan_rows_multi_gpu(dev, t, lo, hi, rank, world, local_rank, keep_group=False):
    """One process per GPU (torchrun): every rank scans a cost-balanced contiguous slice of the centres,
    one gather brings the rows to rank 0 (sharding.py).  When every rank of the node has its own GPU the rows
    stay on the device from the scan kernel to the NCCL gather (``DeviceScan.run_device``); when several ranks
    share one device (tests on a one-GPU box) the gather runs over gloo on host tensors.  Returns the five
    result arrays on rank 0 and None elsewhere.  ``keep_group``: leave the process group this call starts
    running for a later scan (``end_group`` ends it)."""
    import torch
    import torch.distributed as dist
    from . import sharding
    own_gpu = ranks_own_a_gpu()
    started = not dist.is_initialized()
    if started:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29500')
        if own_gpu:
            torch.cuda.set_device(dev.scanner.device)
            dist.init_process_group('nccl', rank=rank, world_size=world,
                                    device_id=torch.device('cuda', dev.scanner.device))
        else:
            dist.init_process_group('gloo', rank=rank, world_size=world)

    if own_gpu:
        where = torch.device('cuda', dev.scanner.device)

        def scan_fn(ts, los, his):
            return dev.run_device(ts, los, his, torch, where)
    else:
        def scan_fn(ts, los, his):
            return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in dev.run(ts, los, his))

    ok = False
    try:
        got = sharding.scan_sharded(dev.problem.genpos, dev.problem.A, t, lo, hi, rank, world, scan_fn, dist, torch,
                                    seg_start=getattr(dev.problem, 'seg_start', None))
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
    (refine.py).  One GPU only.  ``outfile``, the support and the p-value files stay on the coarse grid."""

    def __init__(self, InputData, NeutralSFS, NormalizedBetaBinom, Grids, outfile, fixSize=False,
                 r=0, s=1, phys=False, noCenter=False, device=0, support=None,
                 support_drop=support_mod.DEFAULT_DROP, null=None, pvalues=None, refine=None,
                 refine_steps=refine_mod.DEFAULT_STEPS):
        rank, world, local_rank = _world()
        if support is not None:
            support_drop = support_mod.check_drop(support_drop)
            if world > 1:
                raise ValueError('--support runs on one GPU: launch without torchrun (WORLD_SIZE > 1)')
        if refine is not None:
            refine_steps = refine_mod.check_steps(refine_steps)
            if world > 1:
                raise ValueError('--refine runs on one GPU: launch without torchrun (WORLD_SIZE > 1)')
        if (null is None) != (pvalues is None):
            raise ValueError('--null and --pvalues go together')
        plan = windows.make_plan(InputData, fixSize=fixSize, r=r, s=s, phys=phys, noCenter=noCenter)
        if rank == 0:
            print('writing output to %s' % (outfile))
            # the reference opens the output before it computes anything (v1:516,551,582,600): a bad path
            # must fail now, not after the scan
            with open(outfile, 'w'):
                pass
            if support is not None:
                with open(support, 'w'):
                    pass
            if pvalues is not None:
                with open(pvalues, 'w'):
                    pass
            if refine is not None:
                with open(refine, 'w'):
                    pass
        setup = None
        if null is not None:
            setup = null_mod.NullSetup(null, InputData, NeutralSFS, NormalizedBetaBinom, Grids, fixSize=fixSize,
                                       r=r, s=s, phys=phys, noCenter=noCenter)
        if world > 1:
            from .native import device_count
            device = local_rank % max(1, device_count())
        dev = DeviceScan(InputData, NeutralSFS, NormalizedBetaBinom, Grids, device=device)
        try:
            t, lo, hi, gap = plan.arrays()
            live = np.flatnonzero(~gap)
            T = np.zeros(len(plan)); iA = np.full(len(plan), -1, np.int32)
            ix = iA.copy(); ia = iA.copy(); ns = np.zeros(len(plan), np.int32)
            iv = {k: np.full(len(plan), -1, np.int32) for k in ('A_lo', 'A_hi', 'x_lo', 'x_hi', 's_lo', 's_hi')}
            if len(live):
                if world > 1:
                    got = scan_rows_multi_gpu(dev, t[live], lo[live], hi[live], rank, world, local_rank,
                                              keep_group=setup is not None)
                elif support is not None:
                    got, got_iv = scan_with_support(dev, t[live], lo[live], hi[live], support_drop)
                    for k, v in got_iv.items():
                        iv[k][live] = v
                else:
                    got = dev.run(t[live], lo[live], hi[live])
                if got is not None:
                    T[live], iA[live], ix[live], ia[live], ns[live] = got
            self.results = (T, iA, ix, ia, ns) if rank == 0 else None
            if rank == 0:
                write_scan(outfile, plan, dev.order, T, iA, ix, ia, ns)
                if support is not None:
                    self.support = iv
                    with open(support, 'w') as fh:
                        fh.write(support_mod.SUPPORT_HEADER)
                        fh.writelines(support_mod.format_support(plan, dev.order, T, iA, ix, ia, ns, iv))
                if refine is not None:
                    self._refine(dev, NeutralSFS, NormalizedBetaBinom, refine_steps, refine, plan, t, lo, hi)
        finally:
            dev.close()
        if setup is not None:
            null_T = self._scan_null(setup, device, rank, world, local_rank)
            if rank == 0:
                p = null_mod.pvalues(np.where(gap, np.nan, T), null_T)
                self.null, self.pvalues = null_T, p
                for line in null_mod.summary(null_T, setup.rep, setup.n_replicates):
                    print(line)
                with open(pvalues, 'w') as fh:
                    fh.writelines(null_mod.format_pvalues(plan, dev.order, T, iA, ix, ia, ns, p))
        if rank == 0:
            print(f'{datetime.now()}. Scan finished.')

    def _refine(self, dev, neutral, sel, K, path, plan, t, lo, hi):
        """Refine the rows of ``self.results`` on ``dev`` and write the refine file."""
        T, iA, ix, ia, ns = self.results
        grid, rows = refine_mod.refine_rows(dev, neutral, sel, K, t, lo, hi, iA, ix, ia)
        move = refine_mod.moved(grid, T, iA, ix, ia, rows)
        self.refined, self.refine_grid, self.moved = rows, grid, move
        with open(path, 'w') as fh:
            fh.write(HEADER)
            fh.writelines(refine_mod.format_refined(plan, format_rows(plan, dev.order, T, iA, ix, ia, ns), grid,
                                                    rows, move))
        print(f'refine (K = {grid.K}): {int(move.sum())} of {int((iA >= 0).sum())} rows with T > 0 moved to a '
              f'finer grid point')

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
