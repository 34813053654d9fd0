"""A minimal stand-in for the parts of ``fugue`` / ``triad`` that ``fugue_b200/fugue_plugin.py`` binds to.

The reference package cannot be imported in the build image or on the GPU boxes (``triad`` / ``adagio``
are not installed, SURVEY.md F3), so without this the adapter would never execute.  The stand-in
re-creates only the *shape* of the reference's plugin surface - constructor signatures, the facet
plumbing (``EngineFacet``, fugue/execution/execution_engine.py:143-180), ``SQLEngine.encode`` (:202-207),
the ``conditional_dispatcher`` ``.candidate`` decorators, the registration functions - on top of this repo's
own host mirror (``fugue_b200.dataframe`` / ``partition`` / ``schema``).  It records every registration so
the tests can assert what the module registered.  Expression classes: small look-alikes of the reference's
``fugue/column`` classes with the same class names and attributes.
"""
import sys
import types
from typing import Any, Dict, List


class Registry:
    def __init__(self) -> None:
        self.engines: Dict[Any, Any] = {}
        self.sql_engines: Dict[str, Any] = {}
        self.candidates: Dict[str, List[Any]] = {}
        self.annotated: Dict[Any, Any] = {}
        self.test_backends: Dict[str, Any] = {}


class _Dispatcher:
    """``triad.conditional_dispatcher`` look-alike: ``@plugin.candidate(matcher)`` registers an
    implementation; calling the plugin runs the first implementation whose matcher accepts."""

    def __init__(self, name: str, reg: Registry):
        self._name, self._reg = name, reg
        reg.candidates[name] = []

    def candidate(self, matcher: Any, priority: float = 1.0) -> Any:
        def deco(fn: Any) -> Any:
            self._reg.candidates[self._name].append((matcher, fn))
            return fn

        return deco

    def __call__(self, *args: Any, **kwargs: Any) -> Any:
        for matcher, fn in self._reg.candidates[self._name]:
            if matcher(*args, **kwargs):
                return fn(*args, **kwargs)
        raise NotImplementedError(f"{self._name}: no candidate for {args!r}")


def _lookalike_column_modules() -> Dict[str, types.ModuleType]:
    """Expression classes with the reference's names and attributes; structure follows
    fugue/column/expressions.py:8-856 at the level of class names and public properties, nothing more."""
    fe = types.ModuleType("fugue.column.expressions")
    ff = types.ModuleType("fugue.column.functions")

    class ColumnExpr:
        def __init__(self) -> None:
            self.as_name, self.as_type = "", None

        def alias(self, n: str) -> Any:
            self.as_name = n
            return self

    class _NamedColumnExpr(ColumnExpr):
        def __init__(self, name: str):
            super().__init__()
            self.name = name

    class _WildcardExpr(ColumnExpr):
        pass

    class _LiteralColumnExpr(ColumnExpr):
        def __init__(self, value: Any):
            super().__init__()
            self.value = value

    class _FuncExpr(ColumnExpr):
        def __init__(self, func: str, *args: Any, arg_distinct: bool = False, **kwargs: Any):
            super().__init__()
            self.func, self.args, self.kwargs, self.is_distinct = func, list(args), kwargs, arg_distinct

    class _UnaryOpExpr(_FuncExpr):
        @property
        def op(self) -> str:
            return self.func

        @property
        def col(self) -> Any:
            return self.args[0]

    class _BinaryOpExpr(_FuncExpr):
        @property
        def op(self) -> str:
            return self.func

        @property
        def left(self) -> Any:
            return self.args[0]

        @property
        def right(self) -> Any:
            return self.args[1]

    class _UnaryAggFuncExpr(_FuncExpr):
        pass

    for c in (ColumnExpr, _NamedColumnExpr, _WildcardExpr, _LiteralColumnExpr, _FuncExpr, _UnaryOpExpr, _BinaryOpExpr):
        setattr(fe, c.__name__, c)
    fe.col = lambda n: _NamedColumnExpr(n)
    fe.lit = lambda v: _LiteralColumnExpr(v)
    fe.all_cols = lambda: _WildcardExpr()
    ff._UnaryAggFuncExpr = _UnaryAggFuncExpr
    for fn in ("sum", "count", "min", "max", "avg"):
        setattr(ff, fn, (lambda F: lambda c: _UnaryAggFuncExpr(F.upper(), c))(fn))
    return {"fugue.column.expressions": fe, "fugue.column.functions": ff}


def install() -> Registry:
    """Put the stand-in modules into ``sys.modules`` (idempotent per process) and return the registry."""
    if "fugue" in sys.modules and hasattr(sys.modules["fugue"], "_standin_registry"):
        return sys.modules["fugue"]._standin_registry
    from fugue_b200 import dataframe as MD
    from fugue_b200 import partition as MP
    from fugue_b200 import schema as MS

    reg = Registry()
    fugue = types.ModuleType("fugue")
    fugue.__path__ = []  # a package
    fugue._standin_registry = reg

    class EngineFacet:
        def __init__(self, execution_engine: Any):
            c = self.execution_engine_constraint
            if not isinstance(execution_engine, c):
                raise TypeError(f"{self} expects {c}")
            self._execution_engine = execution_engine

        @property
        def execution_engine(self) -> Any:
            return self._execution_engine

        @property
        def execution_engine_constraint(self) -> Any:
            return NativeExecutionEngine

        @property
        def conf(self) -> Any:
            return self._execution_engine.conf

        @property
        def log(self) -> Any:
            import logging

            return logging.getLogger("fugue")

    class MapEngine(EngineFacet):
        pass

    class SQLEngine(EngineFacet):
        def __init__(self, execution_engine: Any):
            super().__init__(execution_engine)
            self._uid = "_" + hex(id(self))[2:6] + "_"

        @property
        def dialect(self) -> Any:
            return None

        def encode_name(self, name: str) -> str:
            return self._uid + name

        def encode(self, dfs: Any, statement: Any) -> Any:
            return ({self.encode_name(k): v for k, v in dfs.items()}, statement.construct(self.encode_name))

    class NativeExecutionEngine:
        def __init__(self, conf: Any = None):
            self._conf = dict(conf or {})
            self._map_engine: Any = None
            self._sql_engine: Any = None

        @property
        def conf(self) -> Dict[str, Any]:
            return self._conf

        @property
        def map_engine(self) -> Any:
            if self._map_engine is None:
                self._map_engine = self.create_default_map_engine()
            return self._map_engine

        @property
        def sql_engine(self) -> Any:
            if self._sql_engine is None:
                self._sql_engine = self.create_default_sql_engine()
            return self._sql_engine

        def to_df(self, df: Any, schema: Any = None) -> Any:
            return df if isinstance(df, MD.DataFrame) else MD.as_fugue_df(df, schema)

    class LocalDataFrameParam:
        pass

    def fugue_annotated_param(annotation: Any, *args: Any, **kwargs: Any) -> Any:
        def deco(cls: Any) -> Any:
            reg.annotated[annotation] = cls
            return cls

        return deco

    fugue.ArrowDataFrame, fugue.DataFrame, fugue.LocalDataFrame = MD.ArrowDataFrame, MD.DataFrame, MD.LocalDataFrame
    fugue.MapEngine, fugue.SQLEngine, fugue.NativeExecutionEngine = MapEngine, SQLEngine, NativeExecutionEngine
    fugue.PartitionCursor, fugue.PartitionSpec = MP.PartitionCursor, MP.PartitionSpec
    f_df = types.ModuleType("fugue.dataframe")
    f_df.__path__ = []
    f_dfdf = types.ModuleType("fugue.dataframe.dataframe")
    f_dfdf.LocalBoundedDataFrame = MD.LocalBoundedDataFrame if hasattr(MD, "LocalBoundedDataFrame") else MD.LocalDataFrame
    f_dev = types.ModuleType("fugue.dev")
    f_dev.LocalDataFrameParam, f_dev.fugue_annotated_param = LocalDataFrameParam, fugue_annotated_param
    f_ex = types.ModuleType("fugue.execution")
    f_ex.__path__ = []
    f_fac = types.ModuleType("fugue.execution.factory")
    f_fac.register_execution_engine = lambda name, func, on_dup="overwrite": reg.engines.__setitem__(name, func)
    f_fac.register_sql_engine = lambda name, func, on_dup="overwrite": reg.sql_engines.__setitem__(name, func)
    f_pl = types.ModuleType("fugue.plugins")
    for name in ("as_fugue_dataset", "count", "get_column_names", "get_num_partitions", "get_schema",
                 "infer_execution_engine", "is_bounded", "is_df", "is_empty", "is_local"):
        setattr(f_pl, name, _Dispatcher(name, reg))
    f_test = types.ModuleType("fugue.test")

    class FugueTestBackend:
        name = ""

    def fugue_test_backend(cls: Any) -> Any:
        assert issubclass(cls, FugueTestBackend) and cls.name.strip() not in ("", "fugue")
        reg.test_backends[cls.name] = cls
        return cls

    f_test.FugueTestBackend, f_test.fugue_test_backend = FugueTestBackend, fugue_test_backend
    fugue.test = f_test
    triad = types.ModuleType("triad")
    triad.Schema = MS.Schema
    mods = {"fugue": fugue, "fugue.dataframe": f_df, "fugue.dataframe.dataframe": f_dfdf, "fugue.dev": f_dev,
            "fugue.execution": f_ex, "fugue.execution.factory": f_fac, "fugue.plugins": f_pl, "fugue.test": f_test,
            "triad": triad}
    sys.modules.update(mods)
    fcol = types.ModuleType("fugue.column")
    fcol.__path__ = []
    look = _lookalike_column_modules()
    sys.modules.update(look)
    sys.modules["fugue.column"] = fcol
    fcol.expressions, fcol.functions = look["fugue.column.expressions"], look["fugue.column.functions"]
    fugue.column = fcol
    return reg
