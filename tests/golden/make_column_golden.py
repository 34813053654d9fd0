"""Generates tests/golden/column_dsl_vectors.json by running the REFERENCE's own column-expression
code (``/root/reference/fugue/column/{expressions,functions,sql}.py``) in this container.

The reference package cannot be imported as a whole (``triad`` / ``adagio`` are absent), but its column DSL
only needs a handful of triad helpers.  This script loads the three reference modules by file path under
their real names, with a minimal stand-in for those helpers (Schema / type names / quote_name / uuid /
assert_or_throw - nothing of the DSL logic), builds a catalogue of expressions with the reference classes
and records what the reference says about each: ``str(expr)``, the SQL its ``SQLExpressionGenerator`` emits,
the inferred alias and the inferred type.  ``tests/test_column_golden.py`` builds the same catalogue with
``fugue_b200.column`` and compares.  The reference's trees themselves go to ``column_dsl_trees.json``, which
``tests/test_fugue_plugin.py`` rebuilds and runs through the plugin's ``translate_expr``.  Run it where the
reference's sources are at ``REF``:

    python tests/golden/make_column_golden.py
"""
import importlib.util
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
REF = "/root/reference/fugue"


def _load_reference_column():
    from fugue_b200 import column as mine
    from fugue_b200 import schema as msch

    triad = types.ModuleType("triad")
    triad.Schema = msch.Schema
    def _to_uuid(*args):  # stand-in for triad.to_uuid: any deterministic id of nested values will do
        import hashlib

        def feed(v):
            if hasattr(v, "__uuid__"):
                return "u" + v.__uuid__()
            if isinstance(v, (list, tuple)):
                return "[" + ",".join(feed(x) for x in v) + "]"
            if isinstance(v, dict):
                return "{" + ",".join(feed(k) + ":" + feed(x) for k, x in v.items()) + "}"
            return type(v).__name__ + ":" + repr(v)

        return hashlib.md5(feed(args).encode()).hexdigest()

    triad.to_uuid = _to_uuid

    def assert_or_throw(cond, exc=None):
        if not cond:
            e = exc() if callable(exc) and not isinstance(exc, BaseException) else exc
            raise e if isinstance(e, BaseException) else AssertionError(e)

    triad.assert_or_throw = assert_or_throw
    tu = types.ModuleType("triad.utils")
    tpa = types.ModuleType("triad.utils.pyarrow")
    tpa._type_to_expression = msch.type_to_expr
    tpa.to_pa_datatype = mine.to_pa_datatype
    tsc = types.ModuleType("triad.utils.schema")
    tsc.quote_name = mine._quote
    fugue = types.ModuleType("fugue")
    fugue.__path__ = []
    fcol = types.ModuleType("fugue.column")
    fcol.__path__ = []
    fexc = types.ModuleType("fugue.exceptions")

    class FugueBug(Exception):
        pass

    fexc.FugueBug = FugueBug
    sys.modules.update({"triad": triad, "triad.utils": tu, "triad.utils.pyarrow": tpa, "triad.utils.schema": tsc,
                        "fugue": fugue, "fugue.column": fcol, "fugue.exceptions": fexc})
    mods = {}
    for name in ("expressions", "functions", "sql"):
        spec = importlib.util.spec_from_file_location(f"fugue.column.{name}", os.path.join(REF, "column", f"{name}.py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[f"fugue.column.{name}"] = m
        spec.loader.exec_module(m)
        mods[name] = m
    ns = types.SimpleNamespace(col=mods["expressions"].col, lit=mods["expressions"].lit, null=mods["expressions"].null,
                               all_cols=mods["expressions"].all_cols, function=mods["expressions"].function,
                               f=mods["functions"], SelectColumns=mods["sql"].SelectColumns,
                               SQLExpressionGenerator=mods["sql"].SQLExpressionGenerator, Schema=msch.Schema)
    return ns


def _tree(e):
    """A reference expression node as JSON: its class and base classes (``translate_expr`` dispatches on the
    bases) and the attributes ``translate_expr`` reads.  Plain Python values are stored as ``{"py": value}``."""
    fe = sys.modules["fugue.column.expressions"]
    if not isinstance(e, fe.ColumnExpr):
        return {"py": e}
    node = {"mro": [c.__name__ for c in type(e).__mro__ if c is not object], "as_name": e.as_name,
            "as_type": None if e.as_type is None else str(e.as_type)}
    if isinstance(e, fe._NamedColumnExpr):
        node["name"] = e.name
    elif isinstance(e, fe._LiteralColumnExpr):
        node["value"] = e.value
    elif isinstance(e, fe._FuncExpr):
        node.update(func=e.func, args=[_tree(a) for a in e.args], is_distinct=e.is_distinct,
                    kwargs={k: _tree(v) for k, v in e.kwargs.items()})
    return node


def main() -> None:
    from column_catalogue import _expressions, describe_all

    ns = _load_reference_column()
    out = describe_all(ns)
    path = os.path.join(HERE, "column_dsl_vectors.json")
    with open(path, "w") as fp:
        json.dump(out, fp, indent=1, sort_keys=True)
    print(f"wrote {path}: {len(out['expressions'])} expressions, {len(out['selects'])} selects")
    trees = {k: _tree(e) for k, e in _expressions(ns).items()}
    path = os.path.join(HERE, "column_dsl_trees.json")
    with open(path, "w") as fp:
        json.dump(trees, fp, indent=1, sort_keys=True)
    print(f"wrote {path}: {len(trees)} expression trees")


if __name__ == "__main__":
    main()
