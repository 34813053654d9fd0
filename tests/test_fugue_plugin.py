"""``fugue_b200/fugue_plugin.py`` executed against the stand-in of the reference's plugin surface
(tests/fugue_standin.py): what it registers, and that the reference's expression trees (recorded from its
own ``fugue/column`` code in tests/golden/column_dsl_trees.json) survive the translation into the engine's
IR (replay of tests/golden/column_dsl_vectors.json through ``translate_expr``).
The device half (the adapter's engine running select / aggregate / join / SQL) is in the GPU test below."""
import json
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import fugue_standin  # noqa: E402


@pytest.fixture(scope="module")
def plugin():
    reg = fugue_standin.install()
    from fugue_b200 import fugue_plugin

    return reg, fugue_plugin


def test_module_registers_engine_sql_engine_candidates_and_test_backend(plugin):
    reg, mod = plugin
    assert "b200" in reg.engines and "b200" in reg.sql_engines          # fugue_duckdb/registry.py:41-75 pattern
    for name in ("infer_execution_engine", "as_fugue_dataset", "is_df", "count", "is_local", "is_bounded",
                 "is_empty", "get_num_partitions", "get_schema", "get_column_names"):
        assert len(reg.candidates[name]) == 1, name                     # fugue/dataframe/arrow_dataframe.py:263-331
    from fugue_b200.table import B200Table

    assert B200Table in reg.annotated and reg.annotated[B200Table]().format_hint() == "b200"
    assert reg.test_backends["b200"] is mod.B200TestBackend               # fugue/test/plugins.py:99-136
    # the engine's SQL facet is the device SQL engine (FugueSQL SELECT -> SQLEngine.select reaches the GPU)
    assert mod.FugueB200ExecutionEngine.create_default_sql_engine is not \
        sys.modules["fugue"].NativeExecutionEngine.__dict__.get("create_default_sql_engine")
    src = open(mod.__file__).read()
    assert "super().join(" not in src and "super().select(" not in src and "super().aggregate(" not in src  # no host fallback


def _rebuild(node):
    """A tree of tests/golden/column_dsl_trees.json, rebuilt with the expression classes under ``fugue.column``;
    each node takes the first class of its recorded class hierarchy that those modules define."""
    import pyarrow as pa

    if "py" in node:
        return node["py"]
    mods = (sys.modules["fugue.column.expressions"], sys.modules["fugue.column.functions"])
    cls = next(getattr(m, c) for c in node["mro"] for m in mods if hasattr(m, c))
    if "name" in node:
        e = cls(node["name"])
    elif "value" in node:
        e = cls(node["value"])
    elif "func" in node:
        e = cls(node["func"], *[_rebuild(a) for a in node["args"]], arg_distinct=node["is_distinct"],
                **{k: _rebuild(v) for k, v in node["kwargs"].items()})
    else:
        e = cls()
    e.as_name = node["as_name"]
    e.as_type = None if node["as_type"] is None else pa.type_for_alias(node["as_type"])
    return e


def test_reference_trees_translate_into_the_ir(plugin):
    _, mod = plugin
    from fugue_b200 import column as ir
    from fugue_b200.schema import Schema

    want = json.load(open(os.path.join(HERE, "golden", "column_dsl_vectors.json")))["expressions"]
    trees = json.load(open(os.path.join(HERE, "golden", "column_dsl_trees.json")))
    assert set(trees) == set(want)
    schema = Schema("a:int,b:long,c:bool,d:double,s:str")
    bad = []
    for name, node in trees.items():
        mine = mod.translate_expr(_rebuild(node))
        got = {"str": str(mine), "is_agg": ir.is_agg(mine), "sql": ir.to_sql(mine)}
        try:
            got["inferred_alias"] = mine.infer_alias().output_name
        except NotImplementedError:
            got["inferred_alias"] = "!NotImplementedError"
        tp = mine.infer_type(schema)
        got["inferred_type"] = None if tp is None else str(tp)
        for k, v in got.items():
            if want[name][k] != v:
                bad.append((name, k, v, want[name][k]))
    assert not bad, bad


@pytest.mark.gpu
def test_adapter_engine_runs_select_aggregate_join_and_sql_on_the_device(plugin):
    import numpy as np
    import pandas as pd

    reg, mod = plugin
    fe, ff = sys.modules["fugue.column.expressions"], sys.modules["fugue.column.functions"]
    from fugue_b200.partition import PartitionSpec
    from fugue_b200.sql import StructuredRawSQL

    eng = reg.engines["b200"]({})
    rng = np.random.default_rng(3)
    fact = pd.DataFrame({"key": rng.integers(0, 50, 5000), "v": rng.standard_normal(5000)})
    dim = pd.DataFrame({"key": np.arange(40), "w": rng.integers(0, 9, 40)})
    # aggregate through the reference-style expression classes
    agg = eng.aggregate(eng.to_df(fact), PartitionSpec(by=["key"]),
                        [ff.sum(fe.col("v")).alias("s"), ff.count(fe.all_cols()).alias("n")]).as_pandas()
    exp = fact.groupby("key").agg(s=("v", "sum"), n=("v", "size")).reset_index()
    got = agg.sort_values("key").reset_index(drop=True)
    assert np.array_equal(got["key"], exp["key"]) and np.array_equal(got["n"], exp["n"])
    assert np.allclose(got["s"], exp["s"], rtol=1e-9)
    # join (all on the device; a host fallback does not exist any more)
    j = eng.join(eng.to_df(fact), eng.to_df(dim), "inner", ["key"]).as_pandas()
    ej = fact.merge(dim, on="key")
    cols = ["key", "v", "w"]
    pd.testing.assert_frame_equal(j[cols].sort_values(cols).reset_index(drop=True),
                                  ej[cols].sort_values(cols).reset_index(drop=True), check_dtype=False)
    # the SQL facet: SQLEngine.select(dfs, StructuredRawSQL) with encoded table names
    sql = eng.sql_engine
    assert isinstance(sql, mod.FugueB200SQLEngine)
    st = StructuredRawSQL([(False, "SELECT key, SUM(v) AS s, COUNT(*) AS n FROM"), (True, "t"), (False, "GROUP BY key")])
    res = sql.select({"t": eng.to_df(fact)}, st).as_pandas().sort_values("key").reset_index(drop=True)
    assert np.array_equal(res["n"], exp["n"]) and np.allclose(res["s"], exp["s"], rtol=1e-9)
    # map_dataframe through the adapter's MapEngine (device function, hash partition)
    from fugue_b200.table import B200Table

    def ident(cursor, df):
        return df

    out = eng.map_engine.map_dataframe(eng.to_df(fact), ident, "key:long,v:double",
                                       PartitionSpec(by=["key"], algo="hash", num=8), map_func_format_hint="b200")
    assert isinstance(out.native, B200Table) and out.count() == len(fact) and out.native.num_partitions == 8
