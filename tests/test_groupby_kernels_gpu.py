"""K6 group-by kernels (``fugue_b200/csrc/fb_groupby.cu``) against an exact numpy reference, kernel by kernel.

``kernels.groupby_u64`` runs one of four device paths, chosen by ``partition=`` and the number of aggregates:

* ``partition=False``: ``fb_groupby_kernel`` over one table (what every input below 4 M rows gets);
* ``partition=True`` with 1..4 aggregates: ``fb_groupby_lean_kernel<N>``, one region of the table per hash partition;
* ``partition=True`` with more than 4 aggregates: ``fb_groupby_kernel`` in region mode;
* ``partition=True`` with ``GROUPBY_BATCHED``: ``fb_groupby_kernel`` batch by batch of regions.

Every aggregate is compared as a bit pattern.  The reference groups with ``np.unique`` (a NULL key is one group of
its own, whatever its bits) and reduces in sorted order: integer SUM wraps mod 2^64, float MIN / MAX follow the IEEE
total order of the order-preserving integer code (the device sort's order), float SUM is exact for dyadic values and
bounded for normal ones.  A group without any non-NULL value of a column has no defined accumulator (the engine
turns it into NULL through a hidden COUNT), so only its COUNT is compared."""
import math

import numpy as np
import pytest

from oracle import hash_partition as hp

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from fugue_b200 import _lib  # noqa: E402
from fugue_b200 import kernels as K  # noqa: E402

I64_MIN, I64_MAX = -(2**63), 2**63 - 1
POS_NAN, NEG_NAN = 0x7FF8000000000000, 0xFFF8000000000000
_SIGN = np.uint64(0x7FFFFFFFFFFFFFFF)


def _dev():
    return torch.device("cuda", 0)


def _d(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(_dev())


def _f64_bits(x) -> np.ndarray:
    return np.asarray(x, dtype=np.float64).view(np.uint64)


def _ordered(bits: np.ndarray) -> np.ndarray:
    """float64 bits -> int64 code whose signed order is the IEEE total order (-NaN < -inf < ... < +inf < +NaN)."""
    b = bits.view(np.int64)
    return np.where(b >= 0, b, (bits ^ _SIGN).view(np.int64))


def _unordered(code: np.ndarray) -> np.ndarray:
    u = code.view(np.uint64)
    return np.where(code >= 0, u, u ^ _SIGN)


# ---- exact reference ---------------------------------------------------------------------------------------------
class _Ref:
    """Groups of ``keys`` (int64) / ``kvalid`` (uint8 or None): valid keys ascending, then the NULL group."""

    def __init__(self, keys: np.ndarray, kvalid):
        n = len(keys)
        ok = np.ones(n, bool) if kvalid is None else kvalid.astype(bool)
        uk, inv = np.unique(keys[ok], return_inverse=True)
        g = np.empty(n, np.int64)
        g[ok] = inv
        g[~ok] = len(uk)
        has_null = bool((~ok).any())
        self.ng = len(uk) + int(has_null)
        self.keys = np.concatenate([uk, np.zeros(int(has_null), np.int64)])
        self.kvalid = np.concatenate([np.ones(len(uk), np.uint8), np.zeros(int(has_null), np.uint8)])
        self.order = np.argsort(g, kind="stable")
        self.g_sorted = g[self.order]

    def agg(self, op: int, bits, valid):
        """(accumulator bits uint64 [ng], number of non-NULL values [ng], sum of |v| [ng] for float sums)."""
        sel = np.ones(len(self.order), bool) if valid is None else valid.astype(bool)[self.order]
        gs = self.g_sorted[sel]
        cnt = np.bincount(gs, minlength=self.ng).astype(np.int64)
        out = np.zeros(self.ng, np.uint64)
        if op == K.AGG_COUNT:
            return cnt.astype(np.uint64), np.full(self.ng, 1, np.int64), None
        vs = np.asarray(bits).view(np.uint64)[self.order][sel]
        ne = cnt > 0
        starts = (np.cumsum(cnt) - cnt)[ne]
        abs_sum = None
        if len(vs) == 0:
            return out, cnt, np.zeros(self.ng)
        if op == K.AGG_SUM_I64:
            out[ne] = np.add.reduceat(vs, starts)                                     # wraps mod 2^64
        elif op in (K.AGG_MIN_I64, K.AGG_MAX_I64):
            f = np.minimum if op == K.AGG_MIN_I64 else np.maximum
            out[ne] = f.reduceat(vs.view(np.int64), starts).view(np.uint64)
        elif op in (K.AGG_MIN_F64, K.AGG_MAX_F64):
            f = np.minimum if op == K.AGG_MIN_F64 else np.maximum
            out[ne] = _unordered(f.reduceat(_ordered(vs), starts))
        elif op == K.AGG_SUM_F64:
            x = vs.view(np.float64)
            with np.errstate(all="ignore"):
                s = np.add.reduceat(x.astype(np.longdouble), starts).astype(np.float64)
            out[ne] = s.view(np.uint64)
            abs_sum = np.zeros(self.ng)
            abs_sum[ne] = np.add.reduceat(np.abs(x), starts)
        else:  # pragma: no cover
            raise AssertionError(op)
        return out, cnt, abs_sum


def _run(keys, kvalid, aggs, partition):
    """``aggs``: list of (op, value bits or None, validity or None).  Returns the kernel's groups in reference order
    (key columns, aggregate columns as uint64)."""
    dk = _d(keys)
    dv = _d(kvalid)
    vals = [_d(None if b is None else np.asarray(b).view(np.int64)) for _, b, _ in aggs]
    vvalid = [_d(m) for _, _, m in aggs]
    gk, gv, ga, ng = K.groupby_u64(dk, dv, vals, vvalid, [op for op, _, _ in aggs], partition=partition)
    gk = gk.cpu().numpy()
    gv = np.ones(ng, np.uint8) if gv is None else gv.cpu().numpy()
    order = np.lexsort((gk, gv == 0))
    return ng, gk[order], gv[order], [a.cpu().numpy().view(np.uint64)[order] for a in ga]


def _check(keys, kvalid, aggs, partition, normal_sums=()):
    """Kernel == reference, bit for bit; the float SUMs listed in ``normal_sums`` (aggregate positions) are held to
    |got - ref| <= count * 2^-52 * sum|v| instead."""
    ref = _Ref(keys, kvalid)
    ng, gk, gv, got = _run(keys, kvalid, aggs, partition)
    assert ng == ref.ng
    assert np.array_equal(gv, ref.kvalid)
    assert np.array_equal(gk[gv == 1], ref.keys[ref.kvalid == 1])
    ref.has = []
    for a, ((op, bits, valid), g) in enumerate(zip(aggs, got)):
        exp, cnt, abs_sum = ref.agg(op, bits, valid)
        has = cnt > 0
        ref.has.append(has)
        if a in normal_sums:
            gf, ef = g[has].view(np.float64), exp[has].view(np.float64)
            bound = cnt[has] * 2.0**-52 * abs_sum[has]
            bad = np.flatnonzero(np.abs(gf - ef) > bound)
            assert bad.size == 0, (a, gf[bad[:5]], ef[bad[:5]], bound[bad[:5]])
        else:
            bad = np.flatnonzero(g[has] != exp[has])
            assert bad.size == 0, (a, op, ref.keys[has][bad[:5]], g[has][bad[:5]], exp[has][bad[:5]])
    return ref, (ng, gk, gv, got)


# ---- the matrix ----------------------------------------------------------------------------------------------------
N = 300_000            # >= 200 K rows: enough slots per region when partition=True forces 256 regions
HOT = 0x1234_5678_9ABC


def _premerge_twins(rng):
    """Two distinct keys that share every hash bit the warp pre-merge compares - bits 20-25 of fmix64(key)
    (fb_groupby_kernel) and bits 40-45 of the partitioner's hash (fb_groupby_lean_kernel) - and the partition id
    (hash % 256), so that they stay neighbours after the hash partition."""
    cand = rng.integers(I64_MIN, I64_MAX, 1 << 14, dtype=np.int64, endpoint=True)
    fm = hp.fmix64(cand.view(np.uint64))
    rh = hp.row_hash([cand])
    sig = ((fm >> np.uint64(20)) & np.uint64(63)) | (((rh >> np.uint64(40)) & np.uint64(63)) << np.uint64(6)) | \
          ((rh & np.uint64(255)) << np.uint64(12))
    order = np.argsort(sig, kind="stable")
    i = int(np.flatnonzero(sig[order][1:] == sig[order][:-1])[0])
    a, b = int(cand[order[i]]), int(cand[order[i + 1]])
    assert a != b and -1 not in (a, b)
    return a, b


@pytest.fixture(scope="module")
def data():
    rng = np.random.default_rng(2024)
    n = N
    pool = rng.integers(I64_MIN, I64_MAX, 40_000, dtype=np.int64, endpoint=True)
    pool[:5] = [0, -1, I64_MIN, I64_MAX, 5]
    keys = pool[rng.integers(0, len(pool), n)]
    # one hot key on ~40 % of the rows: whole 32-row blocks (= whole warps of the unpartitioned kernel) and single rows
    blocks = np.repeat(rng.random(n // 32 + 1) < 0.2, 32)[:n]
    keys[blocks | (rng.random(n) < 0.25)] = HOT
    # the edge keys on a few rows each, some of them inside one warp
    keys[64:96] = np.resize(np.array([0, -1, I64_MIN, I64_MAX, 5], np.int64), 32)
    # pre-merge twins, alternating inside warps (and inside the warps of their partition)
    a, b = _premerge_twins(rng)
    for r0 in (1024, 77_760, 200_000):
        keys[r0:r0 + 96] = np.resize(np.array([a, b], np.int64), 96)
    # NULL keys (~1 %) whose bits are 5, -1 or any pool key: one group, apart from the valid keys 5 and -1
    kvalid = (rng.random(n) > 0.01).astype(np.uint8)
    kvalid[96:128] = 0
    keys[96:112], keys[112:128] = 5, -1
    # values: each column its own ~30 % NULL mask; the pool keys j::7 have no valid value of column j at all
    nul_of = {}
    cols = {}
    for j, name in enumerate(["fd", "fn", "i", "f"]):
        m = (rng.random(n) > 0.3).astype(np.uint8)
        m[np.isin(keys, pool[5 + j::7])] = 0
        nul_of[name] = m
    cols["fd"] = _f64_bits(rng.integers(-(2**30), 2**30, n) * 2.0**-10)            # dyadic: every order is exact
    cols["fn"] = _f64_bits(rng.standard_normal(n))
    i = rng.integers(I64_MIN, I64_MAX, n, dtype=np.int64, endpoint=True)
    i[rng.random(n) < 0.001] = I64_MIN
    i[rng.random(n) < 0.001] = I64_MAX
    cols["i"] = i.view(np.uint64)
    cols["i2"] = rng.integers(-1000, 1000, n).astype(np.int64).view(np.uint64)   # no validity mask
    specials = _f64_bits([0.0, -0.0, np.inf, -np.inf, 5e-324, -5e-324, 1e308, -1e308]).tolist() + [POS_NAN, NEG_NAN]
    f = _f64_bits(rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n))
    sp = rng.random(n) < 0.05
    f[sp] = np.array(specials, np.uint64)[rng.integers(0, len(specials), int(sp.sum()))]
    cols["f"] = f
    nul_of["i2"] = None
    return keys, kvalid, cols, nul_of


def _aggs(data, spec):
    _, _, cols, nul = data
    out = []
    for op, name in spec:
        if op == K.AGG_COUNT:
            out.append((op, None, None if name is None else nul[name]))
        else:
            out.append((op, cols[name], nul[name]))
    return out


S, SI, C, MNI, MXI, MNF, MXF = (K.AGG_SUM_F64, K.AGG_SUM_I64, K.AGG_COUNT, K.AGG_MIN_I64, K.AGG_MAX_I64,
                                K.AGG_MIN_F64, K.AGG_MAX_F64)
AGG_LISTS = {
    1: [(S, "fd")],
    2: [(C, None), (MNF, "f")],
    3: [(SI, "i"), (MXF, "f"), (C, "i")],
    4: [(MNI, "i"), (MXI, "i2"), (S, "fn"), (C, "fd")],
    5: [(S, "fd"), (SI, "i"), (C, None), (MNF, "f"), (MXI, "i")],
    16: [(S, "fd"), (S, "fn"), (SI, "i"), (SI, "i2"), (C, None), (C, "fd"), (C, "f"), (MNI, "i"), (MXI, "i"),
         (MNI, "i2"), (MXI, "i2"), (MNF, "f"), (MXF, "f"), (MNF, "fn"), (MXF, "fd"), (MNF, "fd")],
}
assert {op for spec in AGG_LISTS.values() for op, _ in spec} == set(range(7))


@pytest.mark.parametrize("path,naggs", [("generic", 4), ("generic", 16), ("lean", 1), ("lean", 2), ("lean", 3),
                                        ("lean", 4), ("region", 5), ("region", 16), ("batched", 4),
                                        ("batched", 16)])
def test_kernel_matrix_vs_exact_reference(data, path, naggs, monkeypatch):
    """generic: fb_groupby_kernel, one table; lean: fb_groupby_lean_kernel<naggs>; region: fb_groupby_kernel in
    region mode (> 4 aggregates); batched: fb_groupby_kernel batch by batch of regions."""
    if path == "batched":
        monkeypatch.setattr(K, "GROUPBY_BATCHED", True)
    keys, kvalid, _, _ = data
    spec = AGG_LISTS[naggs]
    aggs = _aggs(data, spec)
    ref, _ = _check(keys, kvalid, aggs, partition=path != "generic",
                    normal_sums=[a for a, (op, name) in enumerate(spec) if op == S and name == "fn"])
    # the shapes the matrix is about are present in the data: the edge keys, the NULL group, the hot key, and
    # groups without any valid value of a masked column
    assert ref.kvalid[-1] == 0 and {0, -1, 5, I64_MIN, I64_MAX, HOT} <= set(ref.keys.tolist())
    for (op, _, valid), has in zip(aggs, ref.has):
        assert has.any() and (op == K.AGG_COUNT or valid is None or not has.all())


def test_float_sum_of_normals_within_the_bound_not_a_relative_tolerance(data):
    """Standard normals into few groups (long atomic chains): |got - ref| <= count * 2^-52 * sum|v| per group, on
    the lean, region and unpartitioned kernels."""
    rng = np.random.default_rng(7)
    n = 400_000
    keys = rng.integers(0, 64, n).astype(np.int64)
    v = _f64_bits(rng.standard_normal(n))
    m = (rng.random(n) > 0.3).astype(np.uint8)
    for partition, extra in ((False, []), (True, []), (True, [(C, None, None)] * 4)):
        _check(keys, None, [(S, v, m)] + extra, partition, normal_sums=[0])


# ---- NaN, signed zeros and infinities in float MIN / MAX ------------------------------------------------------------
NAN_GROUPS = {  # key -> values; expected MIN / MAX = first / last in IEEE total order
    1: [POS_NAN],
    2: [NEG_NAN],
    3: [POS_NAN, _f64_bits(3.0).item()],
    4: [NEG_NAN, _f64_bits(3.0).item()],
    5: [_f64_bits(-0.0).item(), _f64_bits(0.0).item()],
    6: [_f64_bits(np.inf).item()],
    7: [_f64_bits(-np.inf).item(), POS_NAN],
}
NAN_EXPECTED = {1: (POS_NAN, POS_NAN), 2: (NEG_NAN, NEG_NAN), 3: (_f64_bits(3.0).item(), POS_NAN),
                4: (NEG_NAN, _f64_bits(3.0).item()), 5: (_f64_bits(-0.0).item(), _f64_bits(0.0).item()),
                6: (_f64_bits(np.inf).item(),) * 2, 7: (_f64_bits(-np.inf).item(), POS_NAN)}


@pytest.mark.parametrize("partition,naggs", [(False, 2), (True, 2), (True, 5)], ids=["generic", "lean", "region"])
def test_float_min_max_follow_the_total_order_with_nan(partition, naggs):
    """MIN{+NaN} is +NaN (not the +inf identity), MAX{-NaN} is -NaN, MIN{-0.0, +0.0} is -0.0: a device-built table
    or an arithmetic NaN (0/0) reaches the group-by with such values."""
    rng = np.random.default_rng(11)
    n = 250_000
    keys = rng.integers(100, 50_000, n).astype(np.int64)
    v = _f64_bits(rng.standard_normal(n))
    rows = rng.permutation(n)[:700]
    for j, r in enumerate(rows):
        k = 1 + j % 7
        keys[r] = k
        vals = NAN_GROUPS[k]
        v[r] = vals[(j // 7) % len(vals)]
    aggs = [(MNF, v, None), (MXF, v, None)] + [(C, None, None)] * (naggs - 2)
    _, (_, gk, _, (mn, mx, *_)) = _check(keys, None, aggs, partition)
    for k, (emin, emax) in NAN_EXPECTED.items():
        i = int(np.flatnonzero(gk == k)[0])
        assert (hex(mn[i]), hex(mx[i])) == (hex(emin), hex(emax)), k


# ---- the capacity estimate and the overflow retry -------------------------------------------------------------------
def test_estimate_from_partition_zero_then_overflow_retries(monkeypatch):
    """n >= 2^22 partitioned rows size the table from the distinct keys of hash partition 0.  Here partition 0 holds
    one key on 2048 rows and every other row is a distinct key: the estimate (~1.4 K groups) is far too small, the
    kernel overflows and the host retries with 4x the capacity until ~4.2 M groups fit."""
    rng = np.random.default_rng(5)
    n = (1 << 22) + 4096
    cand = rng.integers(I64_MIN, I64_MAX, n + n // 64 + 8192, dtype=np.int64, endpoint=True)
    pid = hp.partition_ids([cand], K.GROUPBY_PARTITIONS)
    k0 = int(cand[pid == 0][0])
    others = np.unique(cand[(pid != 0) & (cand != -1)])
    others = others[rng.permutation(len(others))][:n - 2048]
    keys = others.copy()
    assert len(keys) == n - 2048
    keys = np.insert(keys, np.sort(rng.integers(0, len(keys), 2048)), k0)
    v = rng.integers(I64_MIN, I64_MAX, n, dtype=np.int64, endpoint=True)
    lib = _lib.load()
    real = lib.fb_groupby_u64
    calls = []

    def counting(*args):
        calls.append(int(args[2]))  # nrows
        return real(*args)

    monkeypatch.setattr(lib, "fb_groupby_u64", counting)
    _check(keys, None, [(SI, v, None), (C, None, None)], partition=True)
    assert calls.count(2048) == 1            # the exact distinct count of partition 0
    assert calls.count(n) >= 2, calls        # at least one overflowing attempt, then a larger table


# ---- the engine at size ----------------------------------------------------------------------------------------------
NE = 4_500_000


@pytest.fixture(scope="module")
def engine_table():
    import pandas as pd

    from fugue_b200.table import B200Table

    rng = np.random.default_rng(99)
    n = NE
    pool = rng.integers(I64_MIN, I64_MAX, 200_000, dtype=np.int64, endpoint=True)
    pool[:4] = [0, -1, I64_MIN, I64_MAX]
    k = pool[rng.integers(0, len(pool), n)]
    kv = rng.random(n) > 0.01
    v = rng.integers(-(2**30), 2**30, n) * 2.0**-10
    vv = rng.random(n) > 0.3
    vv[np.isin(k, pool[4::11])] = False               # groups whose v is all NULL
    i = rng.integers(-50, 51, n).astype(np.int32)
    iv = rng.random(n) > 0.3
    iv[np.isin(k, pool[5::13])] = False
    b = rng.integers(0, 4, n).astype(np.int64)
    t = B200Table("k:long,v:double,i:int,b:long", [_d(k), _d(v), _d(i), _d(b)],
                  [_d(kv.astype(np.uint8)), _d(vv.astype(np.uint8)), _d(iv.astype(np.uint8)), None])
    pdf = pd.DataFrame({"k": pd.array(k, dtype="Int64"), "v": np.where(vv, v, np.nan),
                        "i": pd.array(i, dtype="Int32"), "b": b})
    pdf.loc[~kv, "k"] = pd.NA
    pdf.loc[~iv, "i"] = pd.NA
    return t, pdf


def _host(s, dtype):
    """(null mask, values with NULL -> 0) of a pandas column."""
    na = s.isna().to_numpy()
    return na, s.to_numpy(dtype=dtype, na_value=0)


def _engine_cols(tbl, name, dtype):
    j = tbl.schema.index_of_key(name)
    vals = tbl.columns[j].cpu().numpy().astype(dtype)
    na = np.zeros(len(vals), bool) if tbl.valid[j] is None else tbl.valid[j].cpu().numpy() == 0
    return na, np.where(na, 0, vals).astype(dtype)


def _canon(keycols):
    """Row order: key columns ascending, NULL last in each (same as pandas groupby(sort=True, dropna=False))."""
    return np.lexsort(tuple(x for na, vals in reversed(keycols) for x in (vals, na)))


def _engine_vs_oracle(engine_table, keys, aggs, expect_naccs):
    """aggs: name -> (column, func, result dtype).  The aggregate is run through the engine on the device table and
    compared, NULLs included, with oracle.native_engine.aggregate (FIRST / LAST with pandas' first / last)."""
    from fugue_b200 import api as fa
    from fugue_b200.column import all_cols, col, functions as ff
    from fugue_b200.dataframe import B200DataFrame
    from fugue_b200.partition import PartitionSpec
    from oracle import native_engine as ora

    t, pdf = engine_table
    fn = {"sum": ff.sum, "count": ff.count, "min": ff.min, "max": ff.max, "avg": ff.avg, "first": ff.first,
          "last": ff.last}
    cols = [fn[f](all_cols() if c == "*" else col(c)).alias(name) for name, (c, f, _) in aggs.items()]
    e = fa.make_execution_engine("b200")
    seen = []
    real = K.groupby_u64

    def spy(keys_, kv_, vals, vv, ops, **kw):
        seen.append(len(ops))
        return real(keys_, kv_, vals, vv, ops, **kw)

    K.groupby_u64 = spy
    try:
        got = e.aggregate(e.to_df(B200DataFrame(t)), PartitionSpec(by=keys), cols).native
    finally:
        K.groupby_u64 = real
    # accumulators of the call, hidden COUNT / key MIN / MAX included (then the 0-aggregate distinct count of
    # partition 0 that sizes the table)
    assert seen == [expect_naccs, 0], seen
    plain = {n: a for n, a in aggs.items() if a[1] not in ("first", "last")}
    exp = ora.aggregate(pdf, keys, {n: (c, f) for n, (c, f, _) in plain.items()})
    g = pdf.groupby(keys, dropna=False, sort=True)
    for n, (c, f, _) in aggs.items():
        if f in ("first", "last"):
            exp[n] = getattr(g[c], f)().reset_index(drop=True)
    kt = {k: (np.float64 if k == "v" else np.int64) for k in keys}
    ek = [_host(exp[k], kt[k]) for k in keys]
    gk = [_engine_cols(got, k, kt[k]) for k in keys]
    eo, go = _canon(ek), _canon(gk)
    assert got.num_rows == len(exp)
    for (ena, ev), (gna, gv) in zip(ek, gk):
        assert np.array_equal(ena[eo], gna[go]) and np.array_equal(ev[eo], gv[go])
    for n, (c, f, dt) in aggs.items():
        ena, ev = _host(exp[n], dt)
        gna, gv = _engine_cols(got, n, dt)
        ena, ev, gna, gv = ena[eo], ev[eo], gna[go], gv[go]
        if f == "sum":  # pandas sums a group without values to 0; SQL (and the engine) say NULL
            nonnull = pdf.groupby(keys, dropna=False, sort=True)[c].count().to_numpy()[eo]
            ena = ena | (nonnull == 0)
        assert np.array_equal(ena, gna), n
        bad = np.flatnonzero((ev != gv) & ~ena)
        assert bad.size == 0, (n, ev[bad[:5]], gv[bad[:5]])
        assert (f == "count" or ena.any()) and not ena.all(), n


def test_engine_aggregate_at_size_lean_kernel(engine_table):
    """4 accumulators in all (SUM + its hidden COUNT, MIN + its hidden COUNT): fb_groupby_lean_kernel<4>."""
    _engine_vs_oracle(engine_table, ["k"], {"s": ("v", "sum", np.float64), "m": ("i", "min", np.int64)}, 4)


def test_engine_aggregate_at_size_region_kernel(engine_table):
    """SUM / COUNT(*) / COUNT(v) / MIN / MAX / AVG / FIRST / LAST: 14 accumulators, fb_groupby_kernel in region mode."""
    _engine_vs_oracle(engine_table, ["k"], {
        "s": ("v", "sum", np.float64), "c": ("*", "count", np.int64), "cv": ("v", "count", np.int64),
        "mn": ("v", "min", np.float64), "mx": ("i", "max", np.int64), "av": ("i", "avg", np.float64),
        "f": ("v", "first", np.float64), "l": ("i", "last", np.int64)}, 14)


def test_engine_aggregate_at_size_three_keys(engine_table):
    """Three key columns: the group key is the row hash of the tuple, with hidden MIN / MAX / COUNT per key column
    as the collision check (3 + 3 + 2 + 1 row count + 3 = 12 accumulators)."""
    _engine_vs_oracle(engine_table, ["k", "i", "b"],
                      {"s": ("v", "sum", np.float64), "c": ("*", "count", np.int64)}, 12)


def test_reference_self_check():
    """The reference itself on a hand-made case: NULL key apart from key 5, wrapping sum, total order."""
    keys = np.array([5, 5, 5, -1, 7], np.int64)
    kvalid = np.array([1, 0, 1, 1, 1], np.uint8)
    ref = _Ref(keys, kvalid)
    assert ref.keys.tolist() == [-1, 5, 7, 0] and ref.kvalid.tolist() == [1, 1, 1, 0]
    wide = _Ref(np.array([I64_MAX, I64_MIN + 1, I64_MAX], np.int64), None)   # no NULL group: keys stay int64
    assert ref.keys.dtype == wide.keys.dtype == np.int64 and wide.keys.tolist() == [I64_MIN + 1, I64_MAX]
    big = np.array([I64_MAX, 0, 1, 3, 4], np.int64).view(np.uint64)
    s, cnt, _ = ref.agg(SI, big, None)
    assert s.view(np.int64).tolist() == [3, I64_MIN, 4, 0] and cnt.tolist() == [1, 2, 1, 1]
    f = np.array([POS_NAN, 0, _f64_bits(-0.0).item(), NEG_NAN, POS_NAN], np.uint64)
    mn, _, _ = ref.agg(MNF, f, np.array([1, 1, 1, 0, 1], np.uint8))
    mx, cnt, _ = ref.agg(MXF, f, np.array([1, 1, 1, 0, 1], np.uint8))
    assert [hex(x) for x in mn[:3]] == [hex(0), hex(_f64_bits(-0.0).item()), hex(POS_NAN)]
    assert [hex(x) for x in mx[1:3]] == [hex(POS_NAN), hex(POS_NAN)] and cnt[0] == 0
    assert math.isnan(mx[1:2].view(np.float64)[0])
