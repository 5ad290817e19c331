"""ctypes binding of include/blmx.h (the C ABI of the CUDA scan library).

There is no CPU fallback: if ``libblmx.so`` is missing, or the library reports a
CUDA error, the call raises ``BlmxError``.  The library is built in-tree by
``__graft_entry__.build()`` (nvcc, sm_100a) next to this file.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BLMX_LIB') or os.path.join(_HERE, 'libblmx.so')   # BLMX_LIB: tuning builds

#: every symbol include/blmx.h declares (tests check that the library exports them)
ABI_SYMBOLS = (
    'blmx_abi_version', 'blmx_last_error', 'blmx_device_count', 'blmx_create', 'blmx_destroy',
    'blmx_load', 'blmx_scan', 'blmx_scan_device', 'blmx_scan_oneshot', 'blmx_set_option',
    'blmx_last_counters', 'blmx_last_counters6', 'blmx_last_counters8', 'blmx_last_counters9', 'blmx_problem_info',
    'blmx_last_kernel_ms', 'blmx_measure_fp64_peak', 'blmx_scan_profile', 'blmx_scan_surface',
    'blmx_load_segmented', 'blmx_load_refine', 'blmx_refine',
)


class BlmxError(RuntimeError):
    pass


class Problem(C.Structure):
    _fields_ = [('n_sites', C.c_int64), ('genpos', C.c_void_p), ('cls', C.c_void_p),
                ('n_classes', C.c_int32), ('G', C.c_void_p), ('SP', C.c_void_p),
                ('n_x', C.c_int32), ('n_a', C.c_int32), ('n_A', C.c_int32), ('A', C.c_void_p)]


class Result(C.Structure):
    _fields_ = [('T', C.c_void_p), ('iA', C.c_void_p), ('ix', C.c_void_p), ('ia', C.c_void_p),
                ('nsites', C.c_void_p)]


class Profile(C.Structure):
    _fields_ = [('TA', C.c_void_p), ('Tx', C.c_void_p), ('Ta', C.c_void_p), ('nsA', C.c_void_p)]


_lib = None


def lib():
    """Load libblmx.so once; raise loudly if it is not there."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BlmxError(f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ '
                            f'as g; g.build()"` (nvcc, sm_100a). There is no CPU fallback.')
        L = C.CDLL(LIB_PATH)
        L.blmx_last_error.restype = C.c_char_p
        L.blmx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.blmx_destroy.argtypes = [C.c_void_p]
        L.blmx_load.argtypes = [C.c_void_p, C.POINTER(Problem)]
        L.blmx_load_segmented.argtypes = [C.c_void_p, C.POINTER(Problem), C.c_int64, C.c_void_p]
        L.blmx_scan.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.POINTER(Result)]
        L.blmx_scan_profile.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(Result), C.POINTER(Profile)]
        L.blmx_scan_surface.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
        L.blmx_scan_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.POINTER(Result), C.c_void_p]
        L.blmx_scan_oneshot.argtypes = [C.c_int, C.POINTER(Problem), C.c_int64, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.POINTER(Result)]
        L.blmx_load_refine.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                       C.c_void_p, C.c_void_p]
        L.blmx_refine.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.POINTER(Result)]
        L.blmx_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
        L.blmx_last_counters.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_uint64)]
        L.blmx_last_counters6.argtypes = [C.c_void_p, C.POINTER(C.c_uint64 * 6), C.POINTER(C.c_uint64)]
        L.blmx_last_counters8.argtypes = [C.c_void_p, C.POINTER(C.c_uint64 * 8), C.POINTER(C.c_uint64)]
        L.blmx_last_counters9.argtypes = [C.c_void_p, C.POINTER(C.c_uint64 * 9), C.POINTER(C.c_uint64)]
        L.blmx_problem_info.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                        C.POINTER(C.c_int64)]
        L.blmx_last_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]
        L.blmx_measure_fp64_peak.argtypes = [C.c_int, C.c_double, C.POINTER(C.c_double),
                                             C.POINTER(C.c_double)]
        L.blmx_device_count.argtypes = [C.POINTER(C.c_int)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise BlmxError(f'libblmx error {rc}: {lib().blmx_last_error().decode()}')


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def device_count():
    n = C.c_int(0)
    _check(lib().blmx_device_count(C.byref(n)))
    return n.value


def measure_fp64_peak(device=0, seconds=0.5):
    tf, mhz = C.c_double(0), C.c_double(0)
    _check(lib().blmx_measure_fp64_peak(device, seconds, C.byref(tf), C.byref(mhz)))
    return tf.value, mhz.value


class ScanProblem:
    """Host arrays of one blmx_problem (see include/blmx.h for the meaning of each).

    ``seg_start`` (optional): first site of each segment of a problem made of several sequences laid end to
    end (blmx_load_segmented); ``Scanner.load`` then loads it segmented."""

    def __init__(self, genpos, cls, G, SP, A, n_x, n_a, seg_start=None):
        self.seg_start = None if seg_start is None else np.ascontiguousarray(seg_start, dtype=np.int64)
        self.genpos = np.ascontiguousarray(genpos, dtype=np.float64)
        self.cls = np.ascontiguousarray(cls, dtype=np.int32)
        self.G = np.ascontiguousarray(G, dtype=np.float64)
        self.SP = np.ascontiguousarray(SP, dtype=np.float64)
        self.A = np.ascontiguousarray(A, dtype=np.float64)
        self.n_x, self.n_a = int(n_x), int(n_a)
        if self.SP.shape != (self.n_x * self.n_a, len(self.G)):
            raise ValueError(f'SP must be [n_x*n_a, n_classes], got {self.SP.shape}')
        if len(self.genpos) != len(self.cls):
            raise ValueError('genpos and cls differ in length')

    def as_struct(self):
        return Problem(len(self.genpos), _ptr(self.genpos), _ptr(self.cls), len(self.G), _ptr(self.G),
                       _ptr(self.SP), self.n_x, self.n_a, len(self.A), _ptr(self.A))

    @property
    def h2d_bytes(self):
        return (self.genpos.nbytes + self.cls.nbytes + self.G.nbytes + self.SP.nbytes + self.A.nbytes)


class Scanner:
    """One handle on one device with one problem resident in HBM."""

    def __init__(self, device=0, group=None, batch=None, farfield=None):
        self._h = C.c_void_p()
        _check(lib().blmx_create(int(device), C.byref(self._h)))
        self.device = int(device)
        if group is not None:
            self.set_option('group', group)
        if batch is not None:
            self.set_option('batch', batch)
        if farfield is not None:
            self.set_option('farfield', farfield)

    def set_option(self, name, value):
        _check(lib().blmx_set_option(self._h, name.encode(), int(value)))

    def load(self, problem):
        self._problem = problem          # keep the host arrays alive during the call
        st = problem.as_struct()
        seg = getattr(problem, 'seg_start', None)
        if seg is None:
            _check(lib().blmx_load(self._h, C.byref(st)))
        else:
            _check(lib().blmx_load_segmented(self._h, C.byref(st), len(seg), _ptr(seg)))
        return self

    @staticmethod
    def _centres(t, lo, hi):
        t = np.ascontiguousarray(t, dtype=np.float64)
        lo = np.ascontiguousarray(lo, dtype=np.int64)
        hi = np.ascontiguousarray(hi, dtype=np.int64)
        if len(lo) != len(t) or len(hi) != len(t):
            raise ValueError('t, lo, hi differ in length')
        return t, lo, hi

    def _grid(self):
        p = getattr(self, '_problem', None)
        if p is None:
            raise BlmxError('no problem loaded')
        return len(p.A), p.n_x, p.n_a

    def scan(self, t, lo, hi):
        """HOST arrays in, HOST arrays out (H2D + kernels + D2H, synchronous)."""
        t, lo, hi = self._centres(t, lo, hi)
        n = len(t)
        T = np.zeros(n, np.float64)
        iA, ix, ia, ns = (np.full(n, -1, np.int32) for _ in range(4))
        res = Result(_ptr(T), _ptr(iA), _ptr(ix), _ptr(ia), _ptr(ns))
        _check(lib().blmx_scan(self._h, n, _ptr(t), _ptr(lo), _ptr(hi), C.byref(res)))
        return T, iA, ix, ia, ns

    def scan_profile(self, t, lo, hi):
        """``scan`` plus the profiles of the likelihood surface (blmx_scan_profile):
        -> (T, iA, ix, ia, nsites, TA [n, n_A], Tx [n, n_x], Ta [n, n_a], nsA [n, n_A])."""
        t, lo, hi = self._centres(t, lo, hi)
        n = len(t)
        n_A, n_x, n_a = self._grid()
        T = np.zeros(n, np.float64)
        iA, ix, ia, ns = (np.full(n, -1, np.int32) for _ in range(4))
        TA, Tx, Ta = np.empty((n, n_A)), np.empty((n, n_x)), np.empty((n, n_a))
        nsA = np.zeros((n, n_A), np.int32)
        res = Result(_ptr(T), _ptr(iA), _ptr(ix), _ptr(ia), _ptr(ns))
        prof = Profile(_ptr(TA), _ptr(Tx), _ptr(Ta), _ptr(nsA))
        _check(lib().blmx_scan_profile(self._h, n, _ptr(t), _ptr(lo), _ptr(hi), C.byref(res), C.byref(prof)))
        return T, iA, ix, ia, ns, TA, Tx, Ta, nsA

    def scan_surface(self, t, lo, hi):
        """The whole likelihood surface (blmx_scan_surface) -> (S [n, n_A, n_x, n_a], nsA [n, n_A]).
        S is T at every grid point; -inf everywhere for an A without sites.  n * n_A * n_x * n_a doubles come
        back to the host: meant for a few centres."""
        t, lo, hi = self._centres(t, lo, hi)
        n = len(t)
        n_A, n_x, n_a = self._grid()
        S = np.empty((n, n_A, n_x, n_a))
        nsA = np.zeros((n, n_A), np.int32)
        _check(lib().blmx_scan_surface(self._h, n, _ptr(t), _ptr(lo), _ptr(hi), _ptr(S), _ptr(nsA)))
        return S, nsA

    def load_refine(self, fA, n_fx, n_fa, row_of, SP):
        """Fine tables of blmx_load_refine: fine A values, the fine (x, a) axis lengths, row_of [n_fx * n_fa]
        (row of SP or -1) and SP [n_rows, n_classes]."""
        fA = np.ascontiguousarray(fA, dtype=np.float64)
        row_of = np.ascontiguousarray(row_of, dtype=np.int32)
        SP = np.ascontiguousarray(SP, dtype=np.float64)
        if row_of.shape != (int(n_fx) * int(n_fa),):
            raise ValueError('row_of must have n_fx * n_fa entries')
        n_rows = SP.shape[0] if SP.ndim == 2 else 0
        _check(lib().blmx_load_refine(self._h, len(fA), _ptr(fA), int(n_fx), int(n_fa), n_rows, _ptr(row_of),
                                      _ptr(SP)))
        self._refine_tables = (fA, row_of, SP)

    def refine(self, t, lo, hi, box):
        """Box maxima of the fine grid (blmx_refine); box is int [n, 6] -> (T, fA, fx, fa, nsites), fine
        indices."""
        t, lo, hi = self._centres(t, lo, hi)
        box = np.ascontiguousarray(box, dtype=np.int32)
        n = len(t)
        if box.shape != (n, 6):
            raise ValueError('box must be [n, 6]')
        T = np.full(n, -np.inf)
        fA, fx, fa, ns = (np.full(n, -1, np.int32) for _ in range(4))
        res = Result(_ptr(T), _ptr(fA), _ptr(fx), _ptr(fa), _ptr(ns))
        _check(lib().blmx_refine(self._h, n, _ptr(t), _ptr(lo), _ptr(hi), _ptr(box), C.byref(res)))
        return T, fA, fx, fa, ns

    def scan_device(self, n, d_t, d_lo, d_hi, d_T, d_iA, d_ix, d_ia, d_ns, stream=0):
        """Raw DEVICE pointers (ints) in and out, asynchronous on `stream`."""
        res = Result(d_T, d_iA, d_ix, d_ia, d_ns)
        _check(lib().blmx_scan_device(self._h, int(n), d_t, d_lo, d_hi, C.byref(res),
                                      C.c_void_p(stream)))

    def counters(self):
        """(site pairs, launches) of the most recent scan."""
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _check(lib().blmx_last_counters(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, c.value

    def counters_all(self):
        """dict of the work counters of the most recent scan (see blmx_last_counters9)."""
        v, c = (C.c_uint64 * 9)(), C.c_uint64(0)
        _check(lib().blmx_last_counters9(self._h, C.byref(v), C.byref(c)))
        return {'pairs': v[0], 'single': v[1], 'far_blocks': v[2], 'far_terms': v[3], 'far_sites': v[4],
                'range_violations': v[5], 'edge_sites': v[6], 'quads': v[7], 'pruned_items': v[8],
                'launches': c.value}

    def problem_info(self):
        """Far-field layout of the loaded problem: whole blocks, sites per block, bytes of moments in HBM."""
        a, b, c = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _check(lib().blmx_problem_info(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return {'far_blocks': a.value, 'far_block_sites': b.value, 'moment_bytes': c.value}

    def kernel_ms(self):
        """(summed scan-kernel ms, launches) of the most recent scan; needs option timing=1."""
        ms, n = C.c_double(0), C.c_int64(0)
        _check(lib().blmx_last_kernel_ms(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def close(self):
        if self._h:
            lib().blmx_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
