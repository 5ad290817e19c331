"""bound_kernel's evaluation (DESIGN.md §3.8): the per-point decision it makes in fp32, whole blocks of a class
run summed from the block moments, and its prune count against the CPU Jensen model."""
import sys

import numpy as np
import pytest

import util

sys.path.insert(0, util.ROOT)

LG2_ERR = 2.0 ** -22


def _lhs_f32(terms, D, lg2_err=0.0):
    """The kernel's decision value at one grid point, B + 1.005e-4 A + 1.001e-6 N + 1e-5 with B = sum n l,
    A = sum n |l|, l = lg2(y_up) over the (n, abar) terms, in float32; `lg2_err` is subtracted from every log2
    (relative to max(1, |l|)) to stand in for the worst error lg2.approx may make.  Proved when < 0."""
    f = np.float32
    B = A = f(0.0)
    N = 0
    for n, a in terms:
        a, d = f(a), f(D)
        y = max(f(np.fabs(d) * (a * f(3e-7)) + (d * a + f(1.0))), f(1.17549435e-38))
        l2 = f(np.log2(y))
        l2 = f(l2 - f(lg2_err) * max(f(1.0), np.fabs(l2)))
        B = f(B + f(n) * l2)
        A = f(A + f(n) * np.fabs(l2))
        N += n
    return float(f(f(A * f(1.005e-4) + B) + f(f(N) * f(1.001e-6) + f(1e-5))))


def _terms(alpha, split=0.5):
    out = []
    for m in (alpha < split, alpha >= split):
        if m.any():
            out.append((int(m.sum()), float(alpha[m].sum() / m.sum())))
    return out


def test_decision_is_never_below_the_literal_log_sum():
    """Whenever the kernel's fp32 decision value is < 0 the literal sum of log(1 + alpha D) is < 0 too, and the
    value is above the literal sum wherever both are finite; also when a class's sites are split among more
    groups than the two alpha bins (whole blocks of the tail enter as groups of their own)."""
    rng = np.random.default_rng(23)
    Ds = [-1.0, -1.0 + 1e-12, -0.999, -0.5, -1e-9, 0.0, 1e-9, 0.3, 5.0, 785.0, 1e6, 1e30]
    for trial in range(400):
        n = int(rng.integers(1, 300))
        kind = trial % 4
        if kind == 0:
            alpha = rng.random(n)
        elif kind == 1:
            alpha = np.exp(-rng.random(n) * 18.42)
        elif kind == 2:
            alpha = 1.0 - rng.random(n) * 1e-6
        else:
            alpha = np.clip(rng.choice([1e-8, 0.4999999, 0.5, 0.9999999999], n), 1e-8, 1.0)
        groups = _terms(alpha)
        if trial % 2:                   # tail split into blocks of 32 and the rest, as the units do
            tail = np.sort(alpha[alpha < 0.5])
            groups = _terms(alpha[alpha >= 0.5])
            for k in range(0, len(tail), 32):
                groups += _terms(tail[k:k + 32])
        for D in Ds + [float(rng.uniform(-1, 3))]:
            with np.errstate(divide='ignore'):
                exact = float(np.sum(np.log1p(alpha * D))) / np.log(2.0)
            lhs = _lhs_f32(groups, D, lg2_err=LG2_ERR)
            if np.isfinite(exact):
                assert lhs >= exact, (n, D, lhs, exact)
            else:
                assert exact == -np.inf


def test_decision_is_at_least_the_margin_of_the_per_term_rounding():
    """The decision value covers what the per-term allowance l + 1e-6 + 2^-21 |l| with margin 1e-4 A + 1e-5
    gives in exact arithmetic: folding the allowance into the sums loses nothing."""
    rng = np.random.default_rng(5)
    for _ in range(300):
        k = int(rng.integers(1, 60))
        n = rng.integers(1, 500, size=k)
        l = rng.normal(0.0, 3.0, size=k) * 10.0 ** rng.uniform(-6, 1, size=k)
        lu = l + 1e-6 + 2.0 ** -21 * np.abs(l)
        old = np.sum(n * lu) + 1e-4 * np.sum(n * np.abs(lu)) + 1e-5
        new = np.sum(n * l) + 1.005e-4 * np.sum(n * np.abs(l)) + 1.001e-6 * n.sum() + 1e-5
        assert new >= old - 1e-12 * max(1.0, abs(old))


# ----------------------------------------------------------------------------------------------- GPU
def _synthetic(n_sites=20000, seed=12345):
    import bench
    return bench.make_problem([bench.make_chromosome(n_sites, seed=seed)])[0]


def _scan(prob, t, lo, hi, prune, **opts):
    from ballermixplus_b200.native import Scanner
    with Scanner(device=0).load(prob) as sc:
        sc.set_option('prune', prune)
        for k, v in opts.items():
            sc.set_option(k, v)
        rows = sc.scan(t, lo, hi)
        return rows, sc.counters_all()


def _same_rows(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_pruned_count_matches_the_cpu_jensen_model():
    """A wrong n or abar (a block counted twice or dropped, a wrong moment row) shifts the count even where the
    rows cannot show it.  Items whose decision value is within the fp32 evaluation's reach of 0 may go either
    way; every other item must be decided as the double-precision model decides it."""
    prob = _synthetic()
    n = len(prob.genpos)
    C = prob.G.shape[0]
    D = prob.SP / prob.G[None, :] - 1.0                                   # [n_xa, C]
    centres = np.linspace(200, n - 200, 24).astype(np.int64)
    t = prob.genpos[centres]
    lo, hi = np.zeros(len(t), np.int64), np.full(len(t), n - 1, np.int64)
    sure = unsure = 0
    for tc in t:
        for A in prob.A:
            alpha = np.exp(-A * np.abs(prob.genpos - tc))
            keep = (alpha >= 1e-8) & (prob.genpos != tc)
            al, cl = alpha[keep], prob.cls[keep]
            Bl = np.zeros(D.shape[0])
            Al = np.zeros(D.shape[0])
            for m in (al < 0.5, al >= 0.5):
                cnt = np.bincount(cl[m], minlength=C).astype(np.float64)
                s1 = np.bincount(cl[m], weights=al[m], minlength=C)
                k = cnt > 0
                with np.errstate(divide='ignore', invalid='ignore'):
                    lg = cnt[k] * np.log2(1.0 + D[:, k] * (s1[k] / cnt[k]))
                Bl += lg.sum(-1)
                Al += np.abs(lg).sum(-1)
            v = Bl + 1.005e-4 * Al + 1.001e-6 * len(al) + 1e-5
            # fp32 sums, D and abar in float with the 3e-7 push, lg2.approx: well inside this
            slack = 5e-5 * Al + 2e-6 * len(al) + 1e-4 * np.maximum(1.0, np.abs(Bl))
            if np.all(v < -slack):
                sure += 1
            elif not np.all(v < slack):
                pass                                                      # certainly not proved
            else:
                unsure += 1
    _, k1 = _scan(prob, t, lo, hi, 1)
    assert sure > 0.3 * len(t) * len(prob.A)
    assert sure <= k1['pruned_items'] <= sure + unsure, (sure, unsure, k1['pruned_items'])


@pytest.mark.gpu
def test_prune_keeps_rows_with_whole_blocks_everywhere():
    """Centres on sites of the long class (g == t inside its run, duplicated positions too), between sites,
    and windows cut short of the alpha reach in the middle of a block, over every A: whole blocks on both sides
    of the centre, blocks across alpha = 1/2 and across the reach."""
    prob = _synthetic()
    g = prob.genpos.copy()
    g[1::97] = g[0:-1:97]                                                 # duplicated positions
    from ballermixplus_b200.native import ScanProblem
    prob = ScanProblem(g, prob.cls, prob.G, prob.SP, prob.A, prob.n_x, prob.n_a)
    n = len(g)
    long_cls = np.bincount(prob.cls).argmax()
    c = np.flatnonzero(prob.cls == long_cls)[100:-100:60]
    rng = np.random.default_rng(31)
    t = g[c].copy()
    t[1::3] += np.diff(g)[c[1::3]] * 0.5                                  # between two sites
    lo, hi = np.zeros(len(t), np.int64), np.full(len(t), n - 1, np.int64)
    cut = np.arange(len(t)) % 4 == 2                                       # windows shorter than the reach
    lo[cut] = c[cut] - rng.integers(40, 700, size=cut.sum())
    hi[cut] = c[cut] + rng.integers(40, 700, size=cut.sum())
    r0, k0 = _scan(prob, t, lo, hi, 0)
    r1, k1 = _scan(prob, t, lo, hi, 1)
    _same_rows(r0, r1)
    assert k1['pruned_items'] > 0.3 * len(t) * len(prob.A)
    assert k0['pairs'] == k1['pairs']


@pytest.mark.gpu
def test_prune_keeps_rows_on_a_segmented_problem():
    """Two replicates end to end (blmx_load_segmented): windows inside one segment use whole blocks, windows
    across the boundary are evaluated exactly."""
    import bench
    from ballermixplus_b200.native import ScanProblem
    probs = bench.make_problem([bench.make_chromosome(6000, seed=s) for s in (3, 4)])
    seg = np.array([0, 6000], np.int64)
    p0 = probs[0]
    g = np.concatenate([p.genpos for p in probs])
    cls = np.concatenate([p.cls for p in probs])
    cat = ScanProblem(g, cls, p0.G, p0.SP, p0.A, p0.n_x, p0.n_a, seg_start=seg)
    c = np.arange(50, 12000, 97)
    t = g[c]
    lo = np.where(c < 6000, 0, 6000).astype(np.int64)
    hi = np.where(c < 6000, 5999, 11999).astype(np.int64)
    cross = np.abs(c - 6000) < 1500                                       # these windows cross the boundary
    lo[cross] = c[cross] - 1500
    hi[cross] = c[cross] + 1500
    r0, _ = _scan(cat, t, lo, hi, 0)
    r1, k1 = _scan(cat, t, lo, hi, 1)
    _same_rows(r0, r1)
    assert k1['pruned_items'] > 0
