"""Parity of the sm_100a hash-partition kernels (through the C ABI) with the oracle."""
import os

import numpy as np
import pandas as pd
import pytest

from oracle import hash_partition as hp

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
HERE = os.path.dirname(os.path.abspath(__file__))


def _dev():
    return torch.device("cuda", 0)


def _to_dev(a: np.ndarray):
    if a.dtype == bool:
        return torch.from_numpy(a.view("u1").copy()).to(_dev())
    if a.dtype.kind == "u" and a.dtype.itemsize > 1:
        a = a.view(f"i{a.dtype.itemsize}")
    return torch.from_numpy(np.ascontiguousarray(a)).to(_dev())


def _bytes(t) -> np.ndarray:
    return t.cpu().numpy().view("u1")


def test_library_loaded_and_device_is_blackwell():
    import ctypes as C

    from fugue_b200 import _lib

    lib = _lib.load()
    sm, mem, maj, mnr = C.c_int(), C.c_size_t(), C.c_int(), C.c_int()
    _lib.check(lib.fb_device_info(0, C.byref(sm), C.byref(mem), C.byref(maj), C.byref(mnr)))
    assert maj.value == 10 and sm.value >= 100


def test_partition_ids_golden_vectors():
    from fugue_b200 import kernels as K

    gold = np.load(os.path.join(HERE, "golden", "hash_vectors.npz"), allow_pickle=False)
    for i, combo in enumerate(gold["combos"]):
        names = str(combo).split(",")
        keys = [_to_dev(gold[n]) for n in names]
        for num in (1, 2, 3, 107, 256, 1000, 65536, 2**31 - 1):
            got = K.partition_ids(keys, num).cpu().numpy().astype("int64")
            exp = (gold[f"hash_{i}"] % np.uint64(num)).astype("int64")
            assert np.array_equal(got, exp), (combo, num)


def test_partition_ids_reference_known_answer():
    # tests/fugue_dask/test_utils.py:106-108
    from fugue_b200 import kernels as K

    aa = np.array([0, 1, 1, 2, 3, 4], dtype="int64")
    pids = K.partition_ids([_to_dev(aa)], 3).cpu().numpy()
    buckets = sorted(sorted(aa[pids == p].tolist()) for p in np.unique(pids))
    assert buckets == [[0, 2], [1, 1, 3, 4]]
    keys = np.array([0, 1, 2, 3, 4, -5, 2**62, -(2**63)], dtype="int64")
    assert K.partition_ids([_to_dev(keys)], 256).cpu().tolist() == [99, 18, 81, 147, 63, 29, 114, 81]


def test_partition_ids_null_keys():
    from fugue_b200 import kernels as K

    rng = np.random.default_rng(0)
    n = 10000
    a = rng.integers(0, 50, n).astype("int64")
    b = rng.standard_normal(n)
    va = (rng.random(n) > 0.2).astype("uint8")
    got = K.partition_ids([_to_dev(a), _to_dev(b)], 256, [_to_dev(va), None]).cpu().numpy()
    exp = hp.partition_ids([a, b], 256, [va, None])
    assert np.array_equal(got, exp)


def _check_partition(cols, key_idx, num, valid=None):
    from fugue_b200 import kernels as K

    dcols = [_to_dev(c) for c in cols]
    dvalid = None if valid is None else [None if v is None else _to_dev(v) for v in valid]
    out, off = K.partition_columns(dcols, key_idx, num, dvalid)
    torch.cuda.synchronize()
    exp_cols, exp_off = hp.partition_table(list(cols), key_idx, num, None if valid is None else
                                           [valid[key_idx.index(i)] if i in key_idx else None
                                            for i in range(len(cols))])
    assert np.array_equal(off.cpu().numpy(), exp_off)
    for c, (a, b) in enumerate(zip(out, exp_cols)):
        assert np.array_equal(_bytes(a), np.ascontiguousarray(b).view("u1")), f"column {c} differs"


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 4095, 4096, 4097, 100003, 1 << 20, 3_000_017])
@pytest.mark.parametrize("num", [1, 2, 3, 256])
def test_partition_benchmark_schema_sizes(n, num):
    rng = np.random.default_rng(n * 31 + num)
    cols = [rng.integers(0, 1 << 16, n).astype("int64")] + \
           [rng.integers(-(2**62), 2**62, n).astype("int64") for _ in range(3)] + \
           [rng.standard_normal(n) for _ in range(4)]
    _check_partition(cols, [0], num)


@pytest.mark.parametrize("num", [7, 255, 257, 1000, 1024])
def test_partition_other_partition_counts(num):
    rng = np.random.default_rng(num)
    n = 200_001
    cols = [rng.integers(-1000, 1000, n).astype("int64"), rng.standard_normal(n)]
    _check_partition(cols, [0], num)


def test_partition_mixed_widths_multi_key_nulls():
    rng = np.random.default_rng(11)
    n = 150_000
    cols = [rng.integers(0, 300, n).astype("int32"), rng.integers(0, 5, n).astype("int16"),
            rng.standard_normal(n), rng.integers(0, 255, n).astype("uint8"),
            rng.standard_normal(n).astype("float32"), rng.integers(0, 2, n).astype(bool),
            np.arange(n, dtype="int64")]
    v0 = (rng.random(n) > 0.1).astype("uint8")
    _check_partition(cols, [0, 1], 64, [v0, None])
    _check_partition(cols, [2], 33)
    _check_partition(cols, [0, 1, 3, 5], 256)


def test_partition_skew_and_single_key():
    rng = np.random.default_rng(13)
    n = 500_000
    zipf = np.minimum(rng.zipf(1.2, n), 1 << 20).astype("int64")
    _check_partition([zipf, np.arange(n, dtype="int64")], [0], 256)
    same = np.full(n, 42, dtype="int64")
    _check_partition([same, np.arange(n, dtype="int64")], [0], 256)


def test_partition_matches_live_pandas_hash():
    # the reference expression itself (fugue_dask/_utils.py:155-161), evaluated live
    from fugue_b200 import kernels as K

    rng = np.random.default_rng(17)
    n = 300_000
    df = pd.DataFrame({"key": rng.integers(0, 1 << 16, n), "v": rng.standard_normal(n)})
    ref_pid = pd.util.hash_pandas_object(df[["key"]], index=False).mod(256).astype(int).to_numpy()
    out, off = K.partition_columns([_to_dev(df.key.to_numpy()), _to_dev(df.v.to_numpy())], [0], 256)
    off = off.cpu().numpy()
    assert np.array_equal(np.diff(off), np.bincount(ref_pid, minlength=256))
    k2 = out[0].cpu().numpy()
    v2 = out[1].cpu().numpy()
    order = np.argsort(ref_pid, kind="stable")
    assert np.array_equal(k2, df.key.to_numpy()[order]) and np.array_equal(v2, df.v.to_numpy()[order])


def test_plan_then_apply_column_by_column():
    from fugue_b200 import kernels as K

    rng = np.random.default_rng(19)
    n = 123_457
    cols = [rng.integers(0, 999, n).astype("int64"), rng.standard_normal(n), rng.standard_normal(n)]
    d = [_to_dev(c) for c in cols]
    plan = K.partition_plan([d[0]], 256)
    outs = [K.partition_apply(plan, [c])[0] for c in d]
    exp, exp_off = hp.partition_table(cols, [0], 256)
    assert np.array_equal(plan.offsets.cpu().numpy(), exp_off)
    for a, b in zip(outs, exp):
        assert np.array_equal(_bytes(a), b.view("u1"))


def test_full_size_properties_100m_rows():
    """BASELINE config 2 size (100 M rows x 8 cols): size-independent properties."""
    from fugue_b200 import kernels as K

    n, num = 100_000_000, 256
    g = torch.Generator(device=_dev()).manual_seed(0)
    key = torch.randint(0, 1 << 16, (n,), dtype=torch.int64, device=_dev(), generator=g)
    rowid = torch.arange(n, dtype=torch.int64, device=_dev())
    pay = [torch.randint(-(2**62), 2**62, (n,), dtype=torch.int64, device=_dev(), generator=g)
           for _ in range(2)]
    fcols = [torch.randn(n, dtype=torch.float64, device=_dev(), generator=g) for _ in range(4)]
    cols = [key, rowid] + pay + fcols
    out, off = K.partition_columns(cols, [0], num)
    # offsets are a histogram of the partition ids
    pid_in = K.partition_ids([key], num)
    hist = torch.bincount(pid_in.long(), minlength=num)
    assert torch.equal(off[1:] - off[:-1], hist) and int(off[0]) == 0 and int(off[-1]) == n
    # every output row sits in the partition its key hashes to
    pid_out = K.partition_ids([out[0]], num).long()
    seg = torch.repeat_interleave(torch.arange(num, device=_dev()), hist)
    assert torch.equal(pid_out, seg)
    del pid_out, seg, pid_in
    # stable: row ids increase inside each partition; boundaries are the only descents
    rid = out[1]
    desc = (rid[1:] < rid[:-1]).nonzero().flatten() + 1
    bounds = set(off[1:-1].cpu().tolist())
    assert set(desc.cpu().tolist()) <= bounds
    # rows are moved intact: gather the inputs by output row id and compare bit patterns
    for c in range(len(cols)):
        assert torch.equal(cols[c][rid].view(torch.int64), out[c].view(torch.int64)), c
    # permutation: every row id appears exactly once (checksum of checksums)
    assert int(rid.sum()) == n * (n - 1) // 2
    assert int((rid ^ (rid >> 7)).sum()) == int((rowid ^ (rowid >> 7)).sum())


def _sms() -> int:
    import ctypes as C

    from fugue_b200 import _lib

    sm, mem, maj, mnr = C.c_int(), C.c_size_t(), C.c_int(), C.c_int()
    _lib.check(_lib.load().fb_device_info(0, C.byref(sm), C.byref(mem), C.byref(maj), C.byref(mnr)))
    return sm.value


def _check_apply(dcols, key_idx, num, exp, out=None, **kw):
    """partition_plan + partition_apply(**kw) of the device columns ``dcols`` == ``exp``, the oracle's partition."""
    from fugue_b200 import kernels as K

    plan = K.partition_plan([dcols[i] for i in key_idx], num)
    got = K.partition_apply(plan, dcols, out=out, **kw)
    torch.cuda.synchronize()
    exp_cols, exp_off = exp
    assert np.array_equal(plan.offsets.cpu().numpy(), exp_off)
    for c, (a, b) in enumerate(zip(got, exp_cols)):
        assert np.array_equal(_bytes(a), np.ascontiguousarray(b).view("u1")), f"column {c} differs ({kw})"


@pytest.fixture(scope="module")
def ten_columns():
    rng = np.random.default_rng(23)
    n = 1_234_567
    cols = [rng.integers(0, 1 << 16, n).astype("int64")] + \
           [rng.integers(-(2**62), 2**62, n).astype("int64") for _ in range(4)] + \
           [rng.standard_normal(n) for _ in range(5)]          # 10 columns: more than one launch
    exp = {(0,): hp.partition_table(cols, [0], 256), (0, 5): hp.partition_table(cols, [0, 5], 200)}
    return [_to_dev(c) for c in cols], exp


@pytest.mark.parametrize("cols_per_launch", [0, 1, 2, 3, 5, 8])
@pytest.mark.parametrize("ctas", [None, 7, 1], ids=["all-sms", "7-ctas", "1-cta"])
def test_all_scatter_kernel_paths_agree(ten_columns, cols_per_launch, ctas):
    """The warp-specialised scatter kernel under every launch shape: ``cols_per_launch`` columns per launch (0 = the
    default grouping) on a grid cut to ``ctas`` CTAs by ``sm_reserve = sms - ctas``.  With one CTA, that CTA runs
    every chunk through one mbarrier pipeline (chunk-to-chunk hand-over: flush barrier, look-ahead of the next rank
    record, carry reset).  One key column at num 256 and two key columns at num 200: same bits as the oracle."""
    d, exp = ten_columns
    r = 0 if ctas is None else _sms() - ctas
    _check_apply(d, [0], 256, exp[(0,)], sm_reserve=r, cols_per_launch=cols_per_launch)
    _check_apply(d, [0, 5], 200, exp[(0, 5)], sm_reserve=r, cols_per_launch=cols_per_launch)


@pytest.mark.parametrize("num", [16, 17])
@pytest.mark.parametrize("shape", ["chunks+tail", "whole-tiles", "whole-tiles+1"])
def test_scatter_chunk_geometry(shape, num):
    """Row counts cut from the SM count at run time (4096-row tiles, at most 2 chunks per SM): 3 * (2 * sms) + 1 whole
    tiles plus a partial tile (4 tiles per chunk, a last chunk of one tile, a tail); exactly k whole tiles (no tail);
    k tiles and one row.  num 16 / 17 is the 4-bit / 8-bit boundary of the rank and scatter kernel templates."""
    sms = _sms()
    k = 2 * sms + 5
    n = {"chunks+tail": (3 * (2 * sms) + 1) * 4096 + 2049, "whole-tiles": 4096 * k, "whole-tiles+1": 4096 * k + 1}[shape]
    rng = np.random.default_rng(n + num)
    cols = [rng.integers(-(2**62), 2**62, n).astype("int64"), rng.standard_normal(n),
            rng.integers(-1000, 1000, n).astype("int32"), np.arange(n, dtype="int64"),
            rng.integers(0, 255, n).astype("uint8")]
    d = [_to_dev(c) for c in cols]
    for key_idx in ([0], [0, 2]):
        exp = hp.partition_table(cols, key_idx, num)
        for r in (0, sms - 1):
            _check_apply(d, key_idx, num, exp, sm_reserve=r)


def _misaligned(n: int, dtype):
    """A 1-d tensor of n elements that is 8-byte but not 16-byte aligned."""
    buf = torch.empty(n + 1, dtype=dtype, device=_dev())
    t = buf[1:]
    assert t.is_contiguous() and t.data_ptr() % 16 == 8
    return t


def test_scatter_mixes_aligned_and_misaligned_columns_in_one_call():
    """8-byte columns at 16-byte aligned addresses go to the warp-specialised kernel, those 8 bytes off to the generic
    one (and so do narrow columns) - in one call, with some outputs misaligned too."""
    rng = np.random.default_rng(29)
    n = 1_000_003
    cols = [rng.integers(0, 1 << 20, n).astype("int64"), rng.integers(-(2**62), 2**62, n).astype("int64"),
            rng.standard_normal(n), rng.integers(-(2**62), 2**62, n).astype("int64"), rng.standard_normal(n),
            rng.integers(-(2**30), 2**30, n).astype("int32")]
    d = []
    for i, c in enumerate(cols):
        t = _to_dev(c)
        if i in (1, 4):  # misaligned sources
            m = _misaligned(n, t.dtype)
            m.copy_(t)
            t = m
        d.append(t)
    assert [t.data_ptr() % 16 for t in d] == [0, 8, 0, 0, 8, 0]
    out = [torch.empty_like(t) if i in (0, 1, 5) else _misaligned(n, t.dtype) for i, t in enumerate(d)]
    exp = hp.partition_table(cols, [0], 256)
    for r in (0, _sms() - 1):
        _check_apply(d, [0], 256, exp, out=[o.fill_(0) for o in out], sm_reserve=r)


def test_fused_map_on_one_cta_with_a_tail_tile():
    """K4 (partition_apply_map) with 9 units - copies, one- and two-operand affine maps in float64 and wrapping int64 -
    on a single CTA (sm_reserve = sms - 1), n with a partial tail tile: the numpy epilogue model over the oracle's
    partition order, bit for bit."""
    import struct

    from fugue_b200 import kernels as K
    from test_colmap_plan import _epilogue

    sms = _sms()
    n = 4096 * (2 * sms + 5) + 1234
    rng = np.random.default_rng(31)
    key = rng.integers(0, 1 << 16, n).astype("int64")
    xs = [rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n) for _ in range(3)]
    js = [rng.integers(-(2**62), 2**62, n).astype("int64"), rng.integers(-1000, 1000, n).astype("int64")]
    fb = lambda v: struct.unpack("<Q", struct.pack("<d", v))[0]  # noqa: E731
    host = {f"x{i}": torch.from_numpy(a) for i, a in enumerate(xs)}
    host.update({f"j{i}": torch.from_numpy(a) for i, a in enumerate(js)})
    F, I, CP = K.MAP_AFFINE_F64, K.MAP_AFFINE_I64, K.MAP_COPY
    units = [("x0", None, CP, 0, 0, 0), ("j0", None, CP, 0, 0, 0),
             ("x0", None, F, fb(2.5), 0, fb(-0.0)), ("x1", "x2", F, fb(-1.25), fb(3.0), fb(0.5)),
             ("x2", "x0", F, fb(1e-3), fb(-7.0), fb(-2.0)),
             ("j0", None, I, 3, 0, -7), ("j0", "j1", I, 0x9E3779B97F4A7C15, -5, 11),
             ("j1", "j0", I, -1, 1, 0), ("x1", None, F, fb(-1.0), 0, fb(0.0))]
    assert len(units) == 9 and {u[2] for u in units} == {CP, F, I}
    dev = {k: v.to(_dev()) for k, v in host.items()}
    dkey = _to_dev(key)
    plan = K.partition_plan([dkey], 256)
    got = K.partition_apply_map(plan, [(dev[x], None if y is None else dev[y], m, a, b, c) for x, y, m, a, b, c in units],
                                sm_reserve=sms - 1)
    torch.cuda.synchronize()
    order, off = hp.stable_partition(hp.partition_ids([key], 256), 256)
    assert np.array_equal(plan.offsets.cpu().numpy(), off)
    for i, (x, y, m, a, b, c) in enumerate(units):
        mask = (1 << 64) - 1
        want = _epilogue((host[x], None if y is None else host[y], m, a & mask, b & mask, c & mask, None), n)[order]
        assert np.array_equal(got[i].cpu().numpy().view(np.uint64), want), f"unit {i}"
