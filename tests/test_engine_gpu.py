"""The B200 engine behind the reference's interface: cases follow
fugue_test/execution_suite.py (test_map :208-256, test_map_with_special_values :258-314) and
fugue_test/builtin_suite.py (test_transform_by :516-545), README.md:31-67 (config 1)."""
from typing import Any, Dict, List

import numpy as np
import pandas as pd
import pyarrow as pa
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from fugue_b200 import api as fa
from fugue_b200.dataframe import ArrayDataFrame, B200DataFrame, PandasDataFrame, df_eq
from fugue_b200.execution_engine import B200ExecutionEngine
from fugue_b200.partition import PartitionSpec
from fugue_b200.table import B200Table
from oracle import native_engine as ora


@pytest.fixture(scope="module")
def engine():
    return fa.make_execution_engine("b200")


def select_top(cursor, data):
    return ArrayDataFrame([cursor.row], cursor.row_schema)


def test_to_df_roundtrip(engine):
    o = ArrayDataFrame([[1.1, 2, "x", True], [None, None, None, None], [3.3, 4, "y", False]],
                       "a:double,b:int,c:str,d:bool")
    a = fa.as_fugue_engine_df(engine, o)
    assert isinstance(a, B200DataFrame) and not a.is_local and a.count() == 3
    assert engine.to_df(a) is a
    df_eq(a, o, throw=True)
    assert a.peek_array() == [1.1, 2, "x", True]
    df_eq(a[["c", "a"]], [["x", 1.1], [None, None], ["y", 3.3]], "c:str,a:double", throw=True)
    df_eq(a.rename({"a": "aa"}), o.as_array(), "aa:double,b:int,c:str,d:bool", throw=True)
    e = fa.as_fugue_engine_df(engine, [], "a:int,b:str")
    assert e.empty and e.count() == 0
    df_eq(e, [], "a:int,b:str", throw=True)
    p = engine.to_df(pd.DataFrame({"x": np.arange(5), "y": np.arange(5) * 0.5}))
    assert p.schema == "x:long,y:double" and p.as_array()[4] == [4, 2.0]


def test_map(engine):
    def noop(cursor, data):
        return data

    def on_init(partition_no, data):
        assert partition_no >= 0
        data.peek_array()

    e = engine
    o = ArrayDataFrame([[1, 2], [None, 2], [None, 1], [3, 4], [None, 4]], "a:double,b:int")
    a = fa.as_fugue_engine_df(e, o)
    c = e.map_engine.map_dataframe(a, noop, a.schema, PartitionSpec())
    df_eq(c, o, throw=True)
    c = e.map_engine.map_dataframe(a, noop, a.schema, PartitionSpec(by=["a"], presort="b"))
    df_eq(c, o, throw=True)
    c = e.map_engine.map_dataframe(a, select_top, a.schema, PartitionSpec(by=["a"], presort="b"))
    df_eq(c, [[None, 1], [1, 2], [3, 4]], "a:double,b:int", throw=True)
    c = e.map_engine.map_dataframe(a, select_top, a.schema,
                                   PartitionSpec(partition_by=["a"], presort="b DESC"))
    df_eq(c, [[None, 4], [1, 2], [3, 4]], "a:double,b:int", throw=True)
    c = e.map_engine.map_dataframe(a, select_top, a.schema,
                                   PartitionSpec(partition_by=["a"], presort="b DESC", num_partitions=3),
                                   on_init=on_init)
    df_eq(c, [[None, 4], [1, 2], [3, 4]], "a:double,b:int", throw=True)


def test_map_with_special_values(engine):
    e = engine
    o = ArrayDataFrame([[1, None, 1], [1, None, 0], [None, None, 2]], "a:double,b:double,c:int")
    c = e.map_engine.map_dataframe(o, select_top, o.schema, PartitionSpec(by=["a", "b"], presort="c"))
    df_eq(c, [[1, None, 0], [None, None, 2]], "a:double,b:double,c:int", throw=True)
    from datetime import datetime

    dt = datetime(2024, 5, 6, 7, 8, 9)
    o = ArrayDataFrame([[dt, 2, 1], [None, 2, None], [None, 1, None], [dt, 5, 1], [None, 4, None]],
                       "a:datetime,b:int,c:double")
    c = e.map_engine.map_dataframe(o, select_top, o.schema,
                                   PartitionSpec(by=["a", "c"], presort="b DESC"))
    df_eq(c, [[None, 4, None], [dt, 5, 1]], "a:datetime,b:int,c:double", throw=True)


def test_map_schema_mismatch_raises(engine):
    def bad(t: B200Table) -> B200Table:
        return t.select(["a"])

    with pytest.raises(AssertionError):
        fa.transform(ArrayDataFrame([[1, 2]], "a:long,b:long"), bad, schema="*", engine=engine)


def test_transform_readme_example(engine):
    # BASELINE config 1 / README.md:31-67: plumbing check on the engine
    input_df = pd.DataFrame({"id": [0, 1, 2], "value": ["A", "B", "C"]})
    map_dict = {"A": "Apple", "B": "Banana", "C": "Carrot"}

    def map_letter_to_food(df: pd.DataFrame, mapping: Dict[str, str]) -> pd.DataFrame:
        df["value"] = df["value"].map(mapping)
        return df

    res = fa.transform(input_df, map_letter_to_food, schema="*", params=dict(mapping=map_dict),
                       engine=engine, as_local=True)
    assert isinstance(res, pd.DataFrame)
    assert res.sort_values("id").values.tolist() == [[0, "Apple"], [1, "Banana"], [2, "Carrot"]]


def test_transform_by_keys_host_callbacks(engine):
    # builtin_suite.py:516-545: per logical partition callbacks, counts per key
    def count_rows(df: List[List[Any]]) -> List[List[Any]]:
        return [[df[0][0], len(df)]]

    rng = np.random.default_rng(0)
    keys = rng.integers(0, 37, 1000)
    pdf = pd.DataFrame({"k": keys, "v": rng.standard_normal(1000)})
    res = fa.transform(pdf, count_rows, schema="k:long,ct:long", partition=dict(by=["k"], num=16),
                       engine=engine, as_local=True)
    exp = pdf.groupby("k").size().reset_index(name="ct")
    assert sorted(res.values.tolist()) == sorted(exp.values.tolist())

    # same thing typed on pandas with presort: first row per key after sorting by v descending
    def top(df: pd.DataFrame) -> pd.DataFrame:
        return df.head(1)

    res = fa.transform(pdf, top, schema="*", partition=dict(by=["k"], presort="v desc"), engine=engine,
                       as_local=True)
    exp = ora.map_dataframe(pdf, lambda c, d: d.head(1), ["k", "v"], ["k"], {"v": False})
    assert df_eq(PandasDataFrame(res, "k:long,v:double"), exp.values.tolist(), "k:long,v:double", throw=True)


def test_transform_identity_device_function_matches_native_oracle(engine):
    """The hot path: hash PartitionSpec + identity map typed on the device table."""
    def identity(t: B200Table) -> B200Table:
        return t

    rng = np.random.default_rng(1)
    n = 200_000
    pdf = pd.DataFrame({"key": rng.integers(0, 1 << 16, n), "i1": rng.integers(-2**62, 2**62, n),
                        "v0": rng.standard_normal(n), "v1": rng.standard_normal(n)})
    spec = PartitionSpec(by="key", algo="hash", num=256)
    dev = fa.transform(pdf, identity, schema="*", partition=spec, engine=engine)
    assert isinstance(dev, B200Table) and dev.num_partitions == 256 and dev.partition_keys == ["key"]
    got = dev.to_pandas()
    # reference semantics (NativeExecutionEngine restated): same multiset of rows
    exp = ora.map_dataframe(pdf.iloc[:20000], lambda c, d: d, list(pdf.columns), ["key"])
    assert len(exp) == 20000
    s_got = got.sort_values(list(got.columns)).reset_index(drop=True)
    s_all = pdf.sort_values(list(pdf.columns)).reset_index(drop=True)
    pd.testing.assert_frame_equal(s_got, s_all, check_exact=True)
    # physical layout: rows of partition p are exactly the rows whose key hashes to p, input order kept
    pid = pd.util.hash_pandas_object(pdf[["key"]], index=False).mod(256).to_numpy()
    order = np.argsort(pid, kind="stable")
    pd.testing.assert_frame_equal(got, pdf.iloc[order].reset_index(drop=True), check_exact=True)
    off = dev.offsets.cpu().numpy()
    assert np.array_equal(np.diff(off), np.bincount(pid, minlength=256))


def test_transform_device_function_elementwise(engine):
    def scale(t: B200Table, factor: float) -> B200Table:
        cols = list(t.columns)
        cols[t.schema.index_of_key("v")] = t.column("v") * factor
        return t.with_columns(t.schema, cols, t.valid)

    pdf = pd.DataFrame({"k": [1, 2, 1, 3], "v": [1.0, 2.0, 3.0, 4.0]})
    res = fa.transform(pdf, scale, schema="*", params=dict(factor=2.0), partition=dict(by="k", num=4),
                       engine=engine, as_local=True)
    assert sorted(res.values.tolist()) == [[1, 2.0], [1, 6.0], [2, 4.0], [3, 8.0]]


def test_repartition_is_idempotent_and_keeps_nulls(engine):
    o = ArrayDataFrame([[1, "a"], [None, "b"], [2, None], [None, "d"], [1, "e"]], "k:long,s:str")
    spec = PartitionSpec(by=["k"], num=8)
    r1 = engine.repartition(o, spec)
    r2 = engine.repartition(r1, spec)
    assert r2 is r1
    df_eq(r1, o, throw=True)
    t = r1.native
    off = t.offsets.cpu().tolist()
    keys = t.to_pandas()["k"]
    # all NULL keys are in one physical partition
    parts = [set(np.where(keys.isna().to_numpy())[0])]
    nullpos = sorted(parts[0])
    assert len({next(p for p in range(8) if off[p] <= i < off[p + 1]) for i in nullpos}) == 1


def test_engine_context_and_missing_gpu_path():
    with fa.engine_context("b200") as e:
        assert fa.get_context_engine() is e
        assert isinstance(e, B200ExecutionEngine) and e.get_current_parallelism() == 1
    with pytest.raises(ValueError):
        fa.make_execution_engine("spark")


def test_multi_gpu_repartition_if_two_gpus_visible():
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533",
                        os.path.join(root, "tests", "dist_gpu_check.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "dist_gpu_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_streaming_transform_matches_plain_path(engine):
    """Host in / host out with a device function takes the pipelined path; same result as the
    step-by-step path (to_df -> map_dataframe -> as_local)."""
    def identity(t: B200Table) -> B200Table:
        return t

    def add_col(t: B200Table) -> B200Table:
        from fugue_b200.schema import Schema

        return B200Table(Schema(t.schema, "w:double"), list(t.columns) + [t.column("v0") * 2.0])

    rng = np.random.default_rng(4)
    n = 300_001
    pdf = pd.DataFrame({"key": rng.integers(0, 1 << 16, n), "i1": rng.integers(-2**62, 2**62, n),
                        "v0": rng.standard_normal(n), "f": rng.standard_normal(n).astype("float32")})
    spec = PartitionSpec(by="key", algo="hash", num=256)
    tbl = pa.Table.from_pandas(pdf, preserve_index=False)
    tbl = pa.concat_tables([tbl.slice(0, 100_000), tbl.slice(100_000)])      # two chunks
    got = fa.transform(tbl, identity, schema="*", partition=spec, engine=engine, as_local=True)
    pid = pd.util.hash_pandas_object(pdf[["key"]], index=False).mod(256).to_numpy()
    exp = pdf.iloc[np.argsort(pid, kind="stable")].reset_index(drop=True)
    pd.testing.assert_frame_equal(got, exp, check_exact=True)
    got2 = fa.transform(tbl, add_col, schema="*,w:double", partition=spec, engine=engine, as_local=True)
    exp2 = exp.assign(w=exp.v0 * 2.0)
    pd.testing.assert_frame_equal(got2, exp2, check_exact=True)
    # a table with NULLs is not eligible and silently takes the plain path
    pdf3 = pdf.copy()
    pdf3.loc[5, "v0"] = np.nan
    t3 = pa.Table.from_pandas(pdf3, preserve_index=False)
    t3 = t3.set_column(2, "v0", pa.array(pdf3.v0.where(pdf3.v0.notna(), None).tolist(), type=pa.float64()))
    got3 = fa.transform(t3, identity, schema="*", partition=spec, engine=engine, as_local=True)
    assert len(got3) == n and int(got3.v0.isna().sum()) == 1


def test_even_and_rand_partition_algos():
    """algo="even"/"rand" (fugue_dask/_utils.py:62-121): equal row ranges without keys; with keys the
    distinct key tuples are spread evenly over the partitions (num <= 0: one partition per group)."""
    e = fa.make_execution_engine("b200")
    rng = np.random.default_rng(4)
    n = 100_003
    pdf = pd.DataFrame({"k": rng.integers(0, 37, n), "j": rng.integers(0, 3, n).astype("int32"),
                        "v": np.arange(n, dtype="int64")})
    edf = e.to_df(pdf)

    def parts(df):
        t = df.native
        off = t.offsets.cpu().numpy()
        host = df.as_pandas()
        return [host.iloc[off[i]:off[i + 1]] for i in range(len(off) - 1)], host

    # no keys, even: contiguous equal ranges in input order
    ps, host = parts(e.repartition(edf, PartitionSpec(algo="even", num=7)))
    assert len(ps) == 7 and max(len(p) for p in ps) - min(len(p) for p in ps) <= 1
    assert np.array_equal(host["v"].to_numpy(), pdf["v"].to_numpy())
    # no keys, rand: same multiset, shuffled, equal sizes, reproducible
    r1 = e.repartition(edf, PartitionSpec(algo="rand", num=7))
    ps, host = parts(r1)
    assert max(len(p) for p in ps) - min(len(p) for p in ps) <= 1
    assert not np.array_equal(host["v"].to_numpy(), pdf["v"].to_numpy())
    assert np.array_equal(np.sort(host["v"].to_numpy()), pdf["v"].to_numpy())
    assert np.array_equal(parts(e.repartition(edf, PartitionSpec(algo="rand", num=7)))[1]["v"].to_numpy(),
                          host["v"].to_numpy())
    # keys, even: groups in key order, spread evenly; every key in exactly one partition
    for algo in ("even", "rand"):
        ps, host = parts(e.repartition(edf, PartitionSpec(algo=algo, by=["k", "j"], num=10)))
        assert len(ps) == 10 and sum(len(p) for p in ps) == n
        groups = [set(map(tuple, p[["k", "j"]].drop_duplicates().to_numpy())) for p in ps]
        assert sum(len(g) for g in groups) == len(set().union(*groups)) == 37 * 3     # co-located, none lost
        assert max(len(g) for g in groups) - min(len(g) for g in groups) <= 1        # evenly by group count
        assert np.array_equal(np.sort(host["v"].to_numpy()), pdf["v"].to_numpy())
        if algo == "even":
            firsts = [min(g) for g in groups]
            assert firsts == sorted(firsts)                                           # key order kept
    # num <= 0 with keys: one partition per group
    ps, _ = parts(e.repartition(edf, PartitionSpec(algo="even", by=["k"])))
    assert len(ps) == 37 and all(p["k"].nunique() == 1 for p in ps)
    # a keyed transform under algo="even" sees every logical partition once
    def count(df: pd.DataFrame) -> pd.DataFrame:
        return pd.DataFrame({"k": [df["k"].iloc[0]], "c": [len(df)]})

    out = fa.transform(pdf, count, schema="k:long,c:long", partition=PartitionSpec(algo="even", by=["k"], num=5),
                       engine=e, as_local=True)
    exp = pdf.groupby("k").size().reset_index(name="c")
    assert np.array_equal(out.sort_values("k")["c"].to_numpy(), exp["c"].to_numpy())


@pytest.mark.parametrize("spec_kw,nparts", [({"by": "key", "algo": "hash", "num": 65536}, 65536),
                                           ({"by": ["key", "b"], "num": 5000}, 5000)])
def test_repartition_beyond_one_radix_pass(engine, spec_kw, nparts):
    """num_partitions > 1024 (SURVEY.md 7.1: num=65536): byte-wise stable radix passes on the partition id;
    bit-exact with the oracle's stable partition (same rows, same order, same offsets)."""
    from oracle import hash_partition as hp

    rng = np.random.default_rng(11)
    n = 200_003
    cols = [rng.integers(-(2**40), 2**40, n).astype("int64"), rng.integers(0, 7, n).astype("int32"),
            rng.standard_normal(n), np.arange(n, dtype="int64")]
    t = B200Table("key:long,b:int,v:double,rid:long", [torch.from_numpy(c).cuda() for c in cols])
    res = engine.repartition(B200DataFrame(t), PartitionSpec(**spec_kw)).native
    assert res.num_partitions == nparts
    kidx = [0] if spec_kw["by"] == "key" else [0, 1]
    exp_cols, exp_off = hp.partition_table(cols, kidx, nparts)
    assert np.array_equal(res.offsets.cpu().numpy(), exp_off)
    for g, e in zip(res.columns, exp_cols):
        assert np.array_equal(g.cpu().numpy().view("u1"), e.view("u1"))


def test_repartition_per_row(engine):
    """``PartitionSpec("per_row")`` = algo even, num = ROWCOUNT (fugue/collections/partition.py:95,115,186-207):
    every row its own physical partition; and a hash spec whose num is the ROWCOUNT expression."""
    from oracle import hash_partition as hp

    rng = np.random.default_rng(12)
    n = 3000
    cols = [rng.integers(0, 10**9, n).astype("int64"), rng.standard_normal(n)]
    t = B200Table("key:long,v:double", [torch.from_numpy(c).cuda() for c in cols])
    spec = PartitionSpec("per_row")
    assert spec.num_partitions == "ROWCOUNT" and spec.algo == "even"
    res = engine.repartition(B200DataFrame(t), spec).native
    assert res.num_partitions == n and np.array_equal(res.offsets.cpu().numpy(), np.arange(n + 1))
    assert np.array_equal(res.columns[0].cpu().numpy(), cols[0])
    hspec = PartitionSpec(by="key", algo="hash", num="ROWCOUNT")
    res = engine.repartition(B200DataFrame(t), hspec).native
    exp_cols, exp_off = hp.partition_table(cols, [0], n)
    assert res.num_partitions == n and np.array_equal(res.offsets.cpu().numpy(), exp_off)
    assert np.array_equal(res.columns[0].cpu().numpy(), exp_cols[0])
    out = engine.map_engine.map_dataframe(B200DataFrame(t), lambda c, d: d, t.schema, hspec,
                                          map_func_format_hint="b200")
    assert out.count() == n


def test_transform_save_path_and_checkpoint(engine, tmp_path):
    """fugue/workflow/api.py:100-120: save_path -> the path is returned; + checkpoint -> the dataframe
    loaded back from it; checkpoint alone -> a file under fugue.workflow.checkpoint.path; a parquet
    path as input."""
    pdf = pd.DataFrame({"key": [3, 1, 2, 1, 3, 3], "v": [1.0, 2.0, 3.0, 4.0, 5.0, 6.0]})

    def ident(t: B200Table) -> B200Table:
        return t

    spec = PartitionSpec(by="key", algo="hash", num=4)
    p1 = str(tmp_path / "out.parquet")
    assert fa.transform(pdf, ident, schema="*", partition=spec, engine=engine, save_path=p1) == p1
    back = pd.read_parquet(p1).sort_values(["key", "v"]).reset_index(drop=True)
    pd.testing.assert_frame_equal(back, pdf.sort_values(["key", "v"]).reset_index(drop=True))
    p2 = str(tmp_path / "out2.parquet")
    res = fa.transform(pdf, ident, schema="*", partition=spec, engine=engine, save_path=p2, checkpoint=True,
                       as_local=True, as_fugue=True)
    assert res.count() == 6 and len(pd.read_parquet(p2)) == 6
    with pytest.raises(ValueError):
        fa.transform(pdf, ident, schema="*", engine=engine, checkpoint=True)        # no checkpoint path configured
    with pytest.raises(ValueError):
        fa.transform(pdf, ident, schema="*", engine=engine, save_path=str(tmp_path / "x.csv"))
    eng2 = fa.make_execution_engine("b200", {"fugue.workflow.checkpoint.path": str(tmp_path / "ckpt")})
    res = fa.transform(p1, ident, schema="*", partition=spec, engine=eng2, checkpoint=True, as_fugue=True)
    assert res.count() == 6
    import os

    assert len(os.listdir(tmp_path / "ckpt")) == 1


@pytest.mark.parametrize("n", [100_003, 4096 * 300, 1000])
def test_fused_column_map_matches_the_evaluator_bit_for_bit(engine, n):
    """K4: a ColumnMap of affine expressions is evaluated inside the scatter kernel of the hash partition
    (fb_partition_apply_map).  Same bits as partition -> expression evaluator (K8), and as numpy."""
    from fugue_b200.colmap import ColumnMap
    from fugue_b200.column import col

    rng = np.random.default_rng(21)
    key = rng.integers(0, 1 << 16, n).astype("int64")
    i1 = rng.integers(-(2**62), 2**62, n).astype("int64")
    v0, v1 = rng.standard_normal(n), rng.standard_normal(n)
    v0[:5] = [0.0, -0.0, np.inf, np.nan, 1e308]
    t = B200Table("key:long,i1:long,v0:double,v1:double", [torch.from_numpy(c).cuda() for c in (key, i1, v0, v1)])
    cmap = ColumnMap("key", col("v0").alias("z"), (col("v0") * 2 + col("v1")).alias("w"), (col("key") * 3 - 7).alias("k3"),
                     (col("v1") - col("v0") * 0.5 + 1.25).alias("u"), (-col("i1") + col("key")).alias("m"),
                     (col("v0") * -1.5).alias("s"))
    schema = "key:long,z:double,w:double,k3:long,u:double,m:long,s:double"
    spec = PartitionSpec(by="key", algo="hash", num=256)
    assert cmap.fusion_units(t) is not None
    fused = fa.transform(B200DataFrame(t), cmap, schema=schema, partition=spec, engine=engine, as_fugue=True).native
    assert fused.offsets is not None and fused.num_partitions == 256
    part = engine.repartition(B200DataFrame(t), spec).native
    plain = cmap(part)                                      # unfused: evaluator over the partitioned table
    for name in fused.schema.names:
        a, b = fused.column(name), plain.column(name)
        assert a.dtype == b.dtype and torch.equal(a.view(torch.int64), b.view(torch.int64)), name
    assert torch.equal(fused.offsets, part.offsets)
    k, a0, a1 = part.column("key").cpu().numpy(), part.column("v0").cpu().numpy(), part.column("v1").cpu().numpy()
    with np.errstate(all="ignore"):
        assert np.array_equal(fused.column("w").cpu().numpy().view("i8"), (a0 * 2 + a1).view("i8"))
        assert np.array_equal(fused.column("u").cpu().numpy().view("i8"), ((a1 - a0 * 0.5) + 1.25).view("i8"))
    assert np.array_equal(fused.column("k3").cpu().numpy(), k * 3 - 7)


def test_column_map_that_cannot_be_fused_still_runs_on_the_device(engine):
    from fugue_b200.colmap import ColumnMap
    from fugue_b200.column import col

    pdf = pd.DataFrame({"key": [1, 2, 1, 3], "a": [1.0, 2.0, 3.0, 4.0], "b": [2.0, 4.0, 8.0, 16.0]})
    cmap = ColumnMap("key", (col("a") / col("b")).alias("q"), ((col("a") + 1) * col("b")).alias("p"))
    assert cmap.fusion_units(engine.to_df(pdf).native) is None
    res = fa.transform(pdf, cmap, schema="key:long,q:double,p:double", partition=PartitionSpec(by="key", num=4),
                       engine=engine, as_local=True)
    exp = pdf.assign(q=pdf.a / pdf.b, p=(pdf.a + 1) * pdf.b)[["key", "q", "p"]]
    pd.testing.assert_frame_equal(res.sort_values(["key", "q"]).reset_index(drop=True),
                                  exp.sort_values(["key", "q"]).reset_index(drop=True))
