"""The read-only tables of the window kernel against high-precision references written from the math (mpmath, scipy),
not from either C++ builder: the k-mer frequency limits (Binomial quantiles, README convention C3) and the
position-likelihood tables DPn / DPsq / VSq with their supports.  The product's builder (daccord_b200/csrc/host_tables.hpp,
through the emulation library) and the oracle's (oracle/tables.hpp) are both checked, so an arithmetic error the two share
cannot hide behind their bit parity.  Also: dcu_create's check of est_cor, and deep windows (1300-2000 slices) where exact
and underflowing limits differ, emulation and CUDA against the oracle."""
import ctypes as C
import functools
import math
import numpy as np
import pytest
import mpmath
from mpmath import mp
from scipy.special import betainc
from common import default_params, synth_batch, run_oracle, run_emu, run_emu_lanes, compare_results, get_tables, oracle_lib, emu_lib

PREC = 200                 # bits of every mpmath reference
KLIMN = 2048               # the product's limit table: n = 0..2047 slices
EST_CORS = (0.5, 0.7, 0.85, 0.9, 0.95, 0.99, 0.999)
KS = tuple(range(3, 15))
BUILDERS = (("emu", "emu_get_tables"), ("oracle", "oracle_get_tables"))


def _lib(name):
    return emu_lib() if name == "emu" else oracle_lib()


# ---------------------------------------------------------------- k-mer limits: smallest m with Binomial(n, p) CDF(m) >= 0.99
def _cdf_screen(m, n, p):
    """Binomial(n, p) CDF at m (arrays), double precision: I_{1-p}(n-m, m+1); 0 below 0, 1 from n on"""
    m, n = np.asarray(m, np.int64), np.asarray(n, np.int64)
    inside = (m >= 0) & (m < n)
    a, b = np.where(inside, n - m, 1), np.where(inside, m + 1, 1)
    return np.where(inside, betainc(a, b, 1.0 - p), np.where(m >= n, 1.0, 0.0))


def _cdf_exact(m, n, p):
    if m < 0:
        return mp.mpf(0)
    if m >= n:
        return mp.mpf(1)
    with mp.workprec(PREC):
        return mpmath.betainc(n - m, m + 1, 0, 1 - mp.mpf(p), regularized=True)      # 1 - p exactly, not the rounded double


def _check_limit_row(lim, p):
    """lim[n] for n = 0..len-1 against the exact 0.99 quantile of Binomial(n, p).  Returns (wrong (n, m) pairs, knife-edge count):
    where the exact CDF(m) or CDF(m-1) lies within 1e-12 of 0.99, either neighbour is accepted."""
    n = np.arange(len(lim))
    m = np.asarray(lim, np.int64)
    c1, c0 = _cdf_screen(m, n, p), _cdf_screen(m - 1, n, p)
    ok = (c1 >= 0.99) & (c0 < 0.99)
    near = (np.abs(c1 - 0.99) < 1e-9) | (np.abs(c0 - 0.99) < 1e-9)
    wrong, knife = [], 0
    for i in np.nonzero(~ok | near)[0]:
        e1, e0 = _cdf_exact(int(m[i]), int(i), p), _cdf_exact(int(m[i]) - 1, int(i), p)
        if e1 >= 0.99 and e0 < 0.99:
            knife += bool(abs(e1 - 0.99) < 1e-12 or abs(e0 - 0.99) < 1e-12)
        elif (e1 < 0.99 and 0.99 - e1 < 1e-12) or (e0 >= 0.99 and e0 - 0.99 < 1e-12):
            knife += 1
        else:
            wrong.append((int(i), int(m[i])))
    return wrong, knife


def _limits(lib_name, est_cor, k_lo=KS[0], k_hi=KS[-1]):
    p = default_params(est_cor=est_cor, k_lo=k_lo, k_hi=k_hi)
    fn = dict(BUILDERS)[lib_name]
    return get_tables(_lib(lib_name), fn, p, 4, klimn=KLIMN).reshape(k_hi - k_lo + 1, KLIMN).astype(np.int64)


def _old_limit(p, n, lim=0.99):
    """the recurrence both builders used before: start from q^n (0 or a denormal once n ln q < -708) and add terms up"""
    q = 1.0 - p
    if q == 0.0:
        return n
    term = 1.0
    for _ in range(n):
        term *= q
    ratio, s = p / q, 0.0
    for m in range(n + 1):
        s += term
        if s >= lim:
            return m
        term = term * float(n - m) / float(m + 1) * ratio
    return n


@pytest.mark.parametrize("builder", [b[0] for b in BUILDERS])
def test_kmer_limits_are_exact_binomial_quantiles(builder):
    """every n < 2048, k = 3..14, est_cor from 0.5 to 0.999; p_k = est_cor ** k as the double std::pow gives"""
    wrong, knife = {}, 0
    for est_cor in EST_CORS:
        L = _limits(builder, est_cor)
        for ki, k in enumerate(KS):
            bad, kn = _check_limit_row(L[ki], math.pow(est_cor, k))
            knife += kn
            if bad:
                wrong[(est_cor, k)] = (len(bad), bad[:3])
    print("%s: %d knife-edge limits accepted" % (builder, knife))
    assert not wrong, wrong
    assert knife <= 5


def test_kmer_limits_of_the_known_underflow_rows():
    """values that the underflowing recurrence got wrong (too low once q^n was stuck at the smallest denormal, too high once it was 0)"""
    for builder, _ in BUILDERS:
        for est_cor, k, n, want in ((0.85, 5, 2047, 961), (0.9, 8, 1312, 607), (0.9, 8, 2047, 933), (0.95, 8, 677, 477), (0.99, 8, 290, 277), (0.85, 6, 1556, 631)):
            got = int(_limits(builder, est_cor, k, k)[0, n])
            assert got == want, (builder, est_cor, k, n, got)
            assert _cdf_exact(want, n, math.pow(est_cor, k)) >= 0.99 > _cdf_exact(want - 1, n, math.pow(est_cor, k))


def test_default_configuration_limits_unchanged():
    """est_cor 0.85, k = 8 (the default and the benchmark's): the old recurrence never underflowed below 2048 slices, so the row is the same"""
    old = [_old_limit(math.pow(0.85, 8), n) for n in range(KLIMN)]
    for builder, _ in BUILDERS:
        assert _limits(builder, 0.85, 8, 8)[0].tolist() == old, builder


def test_kmer_limits_of_degenerate_est_cor():
    """est_cor 1: every k-mer is correct, limit n; est_cor 0: limits 0 and the kernel's limit check is off (the oracle's graph skips it
    for p_k = 0, src/DebruijnGraph.hpp:1832-1837), which an emulation run against the oracle shows -- and which all-zero limits with the
    check on (est_cor 1e-3: p_k ~ 1e-24, CDF(0) ~ 1) would not reproduce"""
    for builder, _ in BUILDERS:
        assert (_limits(builder, 1.0) == np.arange(KLIMN)[None, :]).all(), builder
        assert (_limits(builder, 0.0) == 0).all(), builder
        assert (_limits(builder, 1e-3) == 0).all(), builder
    packed, win, sl, _ = synth_batch(30, 25, seed=61, repeat_frac=0.6, depth_jitter=3)
    p0, p1 = default_params(est_cor=0.0), default_params(est_cor=1e-3)
    r0 = run_emu(p0, packed, win, sl, 1)
    assert not compare_results(run_oracle(p0, packed, win, sl, 4), r0)
    assert compare_results(r0, run_emu(p1, packed, win, sl, 1)), "the batch does not tell a limit check that is off from all-zero limits"


# ---------------------------------------------------------------- position-likelihood tables
def _conv(a, b):
    out = []
    for s in range(len(a) + len(b) - 1):
        lo, hi = max(0, s - len(b) + 1), min(s, len(a) - 1)
        out.append(mp.fdot(a[lo:hi + 1], b[s - hi:s - lo + 1][::-1]))
    return out


@functools.lru_cache(maxsize=None)
def _position_reference(w, p_i, p_d):
    """P(read offset o | true offset l), l = 0..w: the (l+1)-fold geometric insertion law (P(c) = (1-p_i) p_i^c, c below the
    truncation of the reference's double loop f >= 1e-7, src/ComputeOffsetLikely.hpp:44-48) convolved with l - Binomial(l, p_d)
    kept bases; entries >= 1e-5 kept.  Returns the exact tables as numpy arrays plus the count of entries too close to 1e-5 to decide."""
    ngeo, f = 0, 1.0 - p_i
    while f >= 1e-7:
        ngeo += 1
        f *= p_i
    with mp.workprec(PREC):
        pi, pd = mp.mpf(p_i), mp.mpf(p_d)
        geo = [(1 - pi) * pi ** c for c in range(ngeo)]
        thr = mp.mpf(1e-5)
        ins = [mp.mpf(1)]
        rows, first, knife = [], [], 0
        for l in range(w + 1):
            ins = _conv(ins, geo)
            kept = [mp.binomial(l, i) * (1 - pd) ** i * pd ** (l - i) for i in range(l + 1)]     # i = l - d bases kept
            F = _conv(kept, ins)                                                                   # F[o], o = kept + inserted
            knife += sum(1 for v in F if abs(v - thr) < 1e-9 * thr)
            idx = [o for o, v in enumerate(F) if v >= thr]
            first.append(idx[0])
            rows.append([F[o] if F[o] >= thr else mp.mpf(0) for o in range(idx[0], idx[-1] + 1)])
        NP, MS = w + 1, max(f0 + len(r) for f0, r in zip(first, rows))
        colsum = [mp.fsum(r[pos - f0] for f0, r in zip(first, rows) if 0 <= pos - f0 < len(r)) for pos in range(MS)]
        DPn, DPsq = np.zeros((NP, MS)), np.zeros((NP, MS))
        VSq, Vnear = np.zeros((NP, MS), np.int64), np.zeros((NP, MS), bool)
        for l, (f0, r) in enumerate(zip(first, rows)):
            cn = 1 / mp.sqrt(mp.fsum(v * v for v in r))
            for o, v in enumerate(r):
                if v == 0:
                    continue
                DPn[l, f0 + o] = float(v / colsum[f0 + o])
                DPsq[l, f0 + o] = float(v * cn)
                x = v * cn * 2 ** 32
                VSq[l, f0 + o] = int(mp.floor(x))
                Vnear[l, f0 + o] = min(x - mp.floor(x), mp.ceil(x) - x) < 1e-3
        # supports: rows are ordered by first and by end (first + length); suplo[pos] = rows ending at or before pos, suphi[pos] = rows starting
        # at or before pos (src/OffsetLikely.hpp:81-93)
        end = [f0 + len(r) for f0, r in zip(first, rows)]
        sup = np.zeros((MS, 2), np.int64)
        j = k = 0
        for pos in range(MS):
            while j < NP and pos >= end[j]:
                j += 1
            while k < NP and first[k] <= pos:
                k += 1
            sup[pos] = (j, k)
    return dict(NP=NP, MS=MS, DPn=DPn, DPsq=DPsq, VSq=VSq, Vnear=Vnear, sup=sup, knife=knife)


def _check_position_tables(ref, got):
    """got: {which: array} of tables 0..3 and (NP, MS, ...) at 5.  Returns the number of VSq entries excused as near an integer."""
    NP, MS = ref["NP"], ref["MS"]
    assert got[5][:2].tolist() == [NP, MS]
    dpn, dpsq = got[0].reshape(NP, MS), got[1].reshape(NP, MS)
    for name, a, b in (("DPn", dpn, ref["DPn"]), ("DPsq", dpsq, ref["DPsq"])):
        assert ((a == 0) == (b == 0)).all(), name
        nz = b != 0
        rel = np.abs(a[nz] - b[nz]) / b[nz]
        assert rel.max() <= 1e-13, (name, rel.max())
    vsq = got[2].reshape(NP, MS).astype(np.int64)
    off = vsq != ref["VSq"]
    assert not (off & ~ref["Vnear"]).any(), np.argwhere(off & ~ref["Vnear"])[:5]
    assert (got[3].reshape(MS, 2).astype(np.int64) == ref["sup"]).all()
    return int(off.sum())


# (w, p_i, p_d): the whole grid {8, 24, 40, 56, 59} x {0, .01, .09, .2, .35} x {0, .045, .2, .6} (about a minute: mp.fdot keeps the
# largest set near 1.5 s)
POS_GRID = [(w, a, b) for w in (8, 24, 40, 56, 59) for a in (0.0, 0.01, 0.09, 0.2, 0.35) for b in (0.0, 0.045, 0.2, 0.6)]


@pytest.mark.parametrize("w,p_i,p_d", POS_GRID)
def test_position_tables_match_high_precision(w, p_i, p_d):
    ref = _position_reference(w, p_i, p_d)
    if ref["knife"]:
        pytest.skip("an entry within 1e-9 of the 1e-5 support threshold: the support is not decidable in double")
    p = default_params(w=w, p_i=p_i, p_d=p_d)
    for builder, fn in BUILDERS:
        got = {which: get_tables(_lib(builder), fn, p, which) for which in (0, 1, 2, 3, 5)}
        near = _check_position_tables(ref, got)
        assert near <= 2, (builder, near)


def test_position_grid_has_no_undecidable_support():
    """the skip above is for safety only: none of the committed parameter sets sits on the support threshold"""
    assert sum(_position_reference(*g)["knife"] for g in POS_GRID) == 0


# ---------------------------------------------------------------- dcu_create rejects est_cor outside [0, 1]
DCU_ERR_PARAM = 1           # include/daccord_b200.h


def test_create_rejects_est_cor_outside_unit_interval():
    import daccord_b200
    import os
    if not os.path.exists(daccord_b200.LIB_PATH):
        from daccord_b200 import build
        build.build()
    lib = C.CDLL(daccord_b200.LIB_PATH)       # the parameters are checked before the first CUDA call: no GPU needed
    for est_cor in (1.2, -0.5, float("nan"), float("inf"), 1.0 + 2 ** -52):
        p = daccord_b200.Params.default(est_cor=est_cor)
        ctx = C.c_void_p()
        rc = lib.dcu_create(C.byref(p), C.c_int(0), C.byref(ctx))
        if ctx.value:
            lib.dcu_destroy(ctx)
        assert rc == DCU_ERR_PARAM and not ctx.value, (est_cor, rc)


# ---------------------------------------------------------------- deep windows where the exact and the underflowing limit differ
# w = 24 keeps a 2000-slice pile below the 65000 bases the large workspace addresses (at w = 40 it passes that near 1550 slices)
DEEP = [("cor90_k8", dict(est_cor=0.9, k_lo=8, k_hi=8, w=24), 23),
        ("cor85_k5", dict(est_cor=0.85, k_lo=5, k_hi=5, w=24), 24)]


def _deep_batch(kw, seed, n):
    return synth_batch(n, 1650, seed=seed, w=kw["w"], repeat_frac=0.3, depth_jitter=340)      # 1310 .. 1990 slices


def _assert_batch_in_changed_region(kw, win):
    p = default_params(**kw)
    new = get_tables(emu_lib(), "emu_get_tables", p, 4, klimn=KLIMN)
    pk = math.pow(kw["est_cor"], kw["k_lo"])
    cnt = [min(int(c), KLIMN - 1) for c in win["slice_cnt"]]          # the kernel reads klim[slice_cnt]
    changed = sum(int(new[c]) != _old_limit(pk, c) for c in cnt)
    assert changed >= 0.8 * len(cnt), (changed, len(cnt))


@pytest.mark.parametrize("name,kw,seed", DEEP, ids=[d[0] for d in DEEP])
def test_deep_windows_emulation_matches_oracle(name, kw, seed):
    p = default_params(**kw)
    packed, win, sl, _ = _deep_batch(kw, seed, 8)
    assert 1300 <= win["slice_cnt"].min() and win["slice_cnt"].max() < KLIMN
    _assert_batch_in_changed_region(kw, win)
    ro = run_oracle(p, packed, win, sl, 4)
    assert (ro[0]["status"] == 1).sum() >= 6
    r1 = run_emu(p, packed, win, sl, 1)
    assert r1[3] == 0 and not compare_results(ro, r1), (name, compare_results(ro, r1))
    r0 = run_emu(p, packed, win, sl, 0)
    assert not [i for i in compare_results(ro, r0) if r0[0][i]["status"] != 250], name    # 250: beyond tier 0, re-run in the large workspace
    rl = run_emu_lanes(p, packed, win, sl, 1, 2, seed)
    assert rl[3] == 0 and not compare_results(ro, rl), name


# ---------------------------------------------------------------- the tables the kernel reads, and deep windows, on the GPU
def _engine(p):
    import daccord_b200 as d
    return d.Engine(d.Params.default(w=p.w, k_lo=p.k_lo, k_hi=p.k_hi, min_cov=p.min_cov, min_ff=p.min_ff, max_ff=p.max_ff, max_err=p.max_err,
                                     p_i=p.p_i, p_d=p.p_d, est_cor=p.est_cor), 0)


DEVICE_SETS = [dict(w=40, p_i=0.09, p_d=0.045, est_cor=0.85, k_lo=3, k_hi=14),
               dict(w=24, p_i=0.2, p_d=0.6, est_cor=0.99, k_lo=5, k_hi=9),
               dict(w=59, p_i=0.2, p_d=0.045, est_cor=0.9, k_lo=8, k_hi=11),
               dict(w=8, p_i=0.35, p_d=0.0, est_cor=0.999, k_lo=3, k_hi=4)]


@pytest.mark.gpu
@pytest.mark.parametrize("kw", DEVICE_SETS, ids=["w%d_cor%g" % (s["w"], s["est_cor"]) for s in DEVICE_SETS])
def test_device_tables_match_precision_references(kw):
    p = default_params(**kw)
    e = _engine(p)
    try:
        got = {which: e.tables(which) for which in range(6)}
    finally:
        e.close()
    assert got[5].tolist()[2] == KLIMN
    _check_position_tables(_position_reference(kw["w"], kw["p_i"], kw["p_d"]), got)
    L = got[4].reshape(kw["k_hi"] - kw["k_lo"] + 1, KLIMN)
    for ki, k in enumerate(range(kw["k_lo"], kw["k_hi"] + 1)):
        bad, knife = _check_limit_row(L[ki], math.pow(kw["est_cor"], k))
        assert not bad and knife <= 1, (k, bad[:3])


@pytest.mark.gpu
@pytest.mark.parametrize("name,kw,seed", DEEP, ids=[d[0] for d in DEEP])
def test_deep_windows_cuda_matches_oracle(name, kw, seed):
    p = default_params(**kw)
    packed, win, sl, _ = _deep_batch(kw, seed + 100, 40)
    assert 1300 <= win["slice_cnt"].min() and win["slice_cnt"].max() < KLIMN
    _assert_batch_in_changed_region(kw, win)
    ro = run_oracle(p, packed, win, sl, 8)
    e = _engine(p)
    try:
        e.set_reads(packed)
        rg = e.run(win, sl)
        st = e.stats()
    finally:
        e.close()
    bad = compare_results(ro, rg)
    assert not bad, (name, len(bad), [(ro[0][i], rg[0][i]) for i in bad[:3]])
    assert st["lost_windows"] == 0 and (rg[0]["status"] == 1).sum() >= 30
