#!/usr/bin/env python
"""Benchmark of the hot path: ``fa.transform()`` with a hash PartitionSpec (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo (B200 engine)
    python bench.py --impl reference --steps K --warmup W    # reference's CPU path (restated)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last step's output (.npy)

One step = one pass of the hot path over one batch of synthetic input:
``transform(table, identity, schema="*", partition=PartitionSpec(by="key", algo="hash", num=256))``
on ``key:long,i1:long,i2:long,i3:long,v0:double,v1:double,v2:double,v3:double`` (64 B/row),
keys uniform over 2**16 values.  Prints ONE JSON line (see the task contract).
"""
import argparse
import json
import os

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # see fugue_b200/dist.py
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS_PER_GPU = 100_000_000     # BASELINE config 2 (1xB200)
ROWS_PER_GPU_DIST = 125_000_000  # BASELINE config 3: 1 B rows on 8xB200 = 125 M per GPU (used for every N > 1)
NUM_PARTITIONS = 256
KEY_CARDINALITY = 1 << 16
SCHEMA = "key:long,i1:long,i2:long,i3:long,v0:double,v1:double,v2:double,v3:double"
ALG_BYTES_PER_ROW = 128  # read every column once + write every column once (SURVEY.md 8d)
# CPU sample: the logical partitions of 1/100 of the keys, at the workload's rows-per-key ratio
# (100M rows / 65536 keys = 1526 rows per logical partition): 1M rows over 655 keys.
REF_SAMPLE_ROWS = int(os.environ.get("FB_BENCH_REF_ROWS", "1000000"))
REF_SAMPLE_KEYS = KEY_CARDINALITY * REF_SAMPLE_ROWS // ROWS_PER_GPU
METRIC = "transform() rows/sec, hash-partitioned (num=256) identity map, 8-col table"
# --dump-outputs: output rows sampled per column; 13 float64 arrays of 4 MiB (row_index, 4 float64 columns,
# 4 int64 columns written as two arrays each) plus the partition offsets stay under 64 MB
DUMP_ROWS = 1 << 19


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _profile_traffic():
    """DRAM bytes of the scatter kernel from the committed ncu capture (NOT measured in this run)."""
    for name in ("r2_summary.json", "r1_summary.json"):
        try:
            v = json.load(open(os.path.join(ROOT, "profiles", name))).get("scatter_dram_bytes_per_launch")
            if v is not None:
                return v, f"profiles/{name} (ncu --set full capture of the same kernel and size; not measured in this run)"
        except Exception:
            pass
    return None, None


def rows_for(world: int) -> int:
    return ROWS_PER_GPU if world == 1 else ROWS_PER_GPU_DIST


def dump_outputs(out, path: str) -> None:
    """Write the table a ``transform`` call returned as float64 ``.npy`` files under ``path``, so that two
    builds can be compared output for output: the partition offsets (``offsets``), the positions of a fixed,
    seeded sample of ``DUMP_ROWS`` output rows (``row_index``; every row when there are fewer) and those rows
    of every column.  An int64 column becomes two arrays that hold it exactly, ``<name>_hi32`` (signed high
    32 bits) and ``<name>_lo32`` (low 32 bits)."""
    import numpy as np
    import torch

    table = out.native
    n = table.num_rows
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(table.device)
    offsets = table.offsets if table.offsets is not None else table.segment_offsets  # multi-GPU: per source rank
    arrays = {"offsets": offsets.cpu().numpy().ravel().astype(np.float64), "row_index": rows.astype(np.float64)}
    for name, c in zip(table.schema.names, table.columns):
        v = c.index_select(0, idx).cpu().numpy()
        if v.dtype == np.int64:
            arrays[name + "_hi32"] = (v >> 32).astype(np.float64)
            arrays[name + "_lo32"] = (v & 0xFFFFFFFF).astype(np.float64)
        else:
            assert v.dtype == np.float64, f"{name}: {v.dtype}"
            arrays[name] = v
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ready = threading.Event()  # NVML is initialised and the first sample is in

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                self.ready.set()
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.004)  # the default timed region is ~40 ms: take several samples inside it
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")
            self.ready.set()

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (restated oracle)
# ------------------------------------------------------------------------------------------
def _workload(rows_per_gpu: int, world: int = 1) -> str:
    """The workload name both arms report (BASELINE.json configs 2 / 3)."""
    which = ("config 2 (1xB200, 100M rows)" if world == 1 and rows_per_gpu == ROWS_PER_GPU else
             f"config 3 share ({world}xB200, {rows_per_gpu * world} rows = {rows_per_gpu} per GPU"
             + ("; exactly config 3: 1B rows on 8 GPUs)" if rows_per_gpu * world == 1_000_000_000 else ")"))
    return (f"{which}: fa.transform identity map, PartitionSpec(by='key', algo='hash', num={NUM_PARTITIONS}) "
            f"on an int64x4+float64x4 table" + (", shuffle across GPUs over NVLink" if world > 1 else ""))


def _config(rows_per_gpu: int, world: int) -> dict:
    """Identical for both arms (the driver compares them)."""
    return {"workload": _workload(rows_per_gpu, world), "rows_per_gpu": rows_per_gpu,
            "rows_total": rows_per_gpu * world, "n_gpus": world, "num_partitions": NUM_PARTITIONS,
            "key_cardinality": KEY_CARDINALITY, "schema": SCHEMA,
            "l2": "inputs (>= 6.4 GB/GPU) are larger than L2 (126 MB); no flush needed"}


def _host_sample(rows: int, seed: int = 0):
    import numpy as np
    import pandas as pd

    rng = np.random.default_rng(seed)
    d = {"key": rng.integers(0, max(1, KEY_CARDINALITY * rows // ROWS_PER_GPU), rows)}
    for c in ("i1", "i2", "i3"):
        d[c] = rng.integers(-(2**62), 2**62, rows)
    for c in ("v0", "v1", "v2", "v3"):
        d[c] = rng.standard_normal(rows)
    return pd.DataFrame(d)


def _time_reference(rows: int, steps: int, warmup: int):
    """pandas restatement of PandasMapEngine.map_dataframe (native_execution_engine.py:81-169):
    one Python call of the map function per logical partition (distinct key), then concat."""
    from oracle import native_engine as ora

    pdf = _host_sample(rows)
    cols = list(pdf.columns)

    def step():
        out = ora.map_dataframe(pdf, lambda cursor, df: df, cols, ["key"])
        assert len(out) == rows

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return rows / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    n = args.rows or rows_for(world)
    steps, warmup = args.steps, max(3, args.warmup)
    rps, dt = _time_reference(REF_SAMPLE_ROWS, steps, warmup)
    sample = (f"each step = {REF_SAMPLE_ROWS} rows = the logical partitions of {REF_SAMPLE_KEYS} of the "
              f"{KEY_CARDINALITY} keys (same 1526 rows per key as the full workload), restated "
              "NativeExecutionEngine.map_dataframe (reference not importable: triad/adagio absent); 1 core: the "
              "reference's native engine is single-threaded (get_current_parallelism() == 1)")
    line = {
        "impl": "reference", "metric": METRIC, "value": rps, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64 (byte moves; u64 hash arithmetic)",
        "data": "synthetic", "config": _config(n, world),
        "cpu_baseline": {"value": rps, "unit": "rows/s", "cores": 1, "kind": "port", "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": rps, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from fugue_b200 import api as fa
    from fugue_b200 import kernels as K
    from fugue_b200.dataframe import B200DataFrame
    from fugue_b200.partition import PartitionSpec
    from fugue_b200.schema import Schema
    from fugue_b200.table import B200Table

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.rows or rows_for(world)
    steps, warmup = args.steps, max(3, args.warmup)

    # synthetic table of the BASELINE shape, generated on the device, seed = rank
    g = torch.Generator(device=dev).manual_seed(rank)
    cols = [torch.randint(0, KEY_CARDINALITY, (n,), dtype=torch.int64, device=dev, generator=g)]
    cols += [torch.randint(-(2**62), 2**62, (n,), dtype=torch.int64, device=dev, generator=g) for _ in range(3)]
    cols += [torch.randn(n, dtype=torch.float64, device=dev, generator=g) for _ in range(4)]
    table = B200Table(Schema(SCHEMA), cols)
    spec = PartitionSpec(by="key", algo="hash", num=NUM_PARTITIONS)

    def identity(t: B200Table) -> B200Table:
        return t

    if world > 1:
        from fugue_b200.dist import DistributedB200Engine

        engine = DistributedB200Engine({"fugue.b200.device": local_rank})
    else:
        engine = fa.make_execution_engine("b200", {"fugue.b200.device": local_rank})
    df_in = B200DataFrame(table)

    def step():
        return fa.transform(df_in, identity, schema="*", partition=spec, engine=engine)

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(warmup):
        out = step()
    sync()
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.ready.wait(timeout=10)  # importing / initialising NVML takes longer than the timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / steps
    total_rows = n * world
    value = total_rows / (ms_per_step * 1e-3)
    nrows_out = out.count() if hasattr(out, "count") else len(out)
    if args.dump_outputs:
        dump_outputs(out, os.path.join(args.dump_outputs, f"rank{rank}") if world > 1 else args.dump_outputs)
    del out

    # ---- roofline of the dominant kernel (scatter), timed live with CUDA events on its stream
    roofline = None
    if rank == 0:
        peak, peak_src = _peaks()
        plan = K.partition_plan([cols[0]], NUM_PARTITIONS)
        outs = [torch.empty_like(c) for c in cols]
        for _ in range(2):
            K.partition_apply(plan, cols, outs)
        torch.cuda.synchronize(dev)
        reps = 5
        e0.record()
        for _ in range(reps):
            K.partition_apply(plan, cols, outs)
        e1.record()
        torch.cuda.synchronize(dev)
        kms = e0.elapsed_time(e1) / reps
        e0.record()
        for _ in range(reps):
            K.partition_plan([cols[0]], NUM_PARTITIONS, scratch=plan.scratch, offsets=plan.offsets)
        e1.record()
        torch.cuda.synchronize(dev)
        pms = e0.elapsed_time(e1) / reps
        achieved = ALG_BYTES_PER_ROW * n / (kms * 1e-3) / 1e9
        traffic, traffic_src = _profile_traffic()
        roofline = {"bound": "hbm", "kernel": "fb_scatter_ws_kernel (pass 2: TMA ring + placement from rank records + write-combined scatter; "
                                              "2 launches x 4 columns, timed together)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": ALG_BYTES_PER_ROW * n,
                    "kernel_ms": kms, "pass1_rank_scan_ms": pms,
                    "step_frac": ALG_BYTES_PER_ROW * n / (ms_per_step * 1e-3) / 1e9 / peak}
        del outs, plan

    # ---- e2e: host Arrow table in pinned memory -> transform -> host Arrow table, every step
    e2e = None
    h2d = d2h = 0
    if not args.no_e2e:
        try:
            import pyarrow as pa

            host_cols = []
            for c in cols:
                h = torch.empty(c.shape, dtype=c.dtype, pin_memory=True)
                h.copy_(c)
                host_cols.append(h)
            torch.cuda.synchronize(dev)
            names = Schema(SCHEMA).names
            pa_types = Schema(SCHEMA).types
            arrays = [pa.Array.from_buffers(tp, n, [None, pa.py_buffer(h.numpy())])
                      for h, tp in zip(host_cols, pa_types)]
            host_table = pa.Table.from_arrays(arrays, names=names)
            h2d = sum(h.numel() * h.element_size() for h in host_cols)
            d2h = h2d
            from fugue_b200.dataframe import ArrowDataFrame

            host_df = ArrowDataFrame(host_table)
            del df_in, table
            e2e_steps = max(1, min(steps, 3))

            def e2e_step():
                res = fa.transform(host_df, identity, schema="*", partition=spec, engine=engine, as_local=True)
                return res.count()

            for _ in range(2):
                e2e_step()
            sync()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                cnt = e2e_step()
            sync()
            dt = (time.perf_counter() - t0) / e2e_steps
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            e2e = {"value": total_rows / dt, "unit": "rows/s", "h2d_bytes_per_step": h2d * world,
                   "d2h_bytes_per_step": d2h * world, "ms_per_step": dt * 1e3, "steps": e2e_steps,
                   "api": "fugue_b200.api.transform(host pyarrow table in pinned memory, as_local=True)"}
        except Exception as ex:  # the device-resident numbers above stay valid; say why e2e is missing
            e2e = {"error": repr(ex)[:300]}
            if world > 1:
                try:
                    dist.barrier()
                except Exception:
                    pass

    # ---- multi-GPU parity, outside the timed region: a small shard through the same engine object,
    #      checked on rank 0 against the oracle / pandas (tests/dist_gpu_check.py; collective)
    parity = None
    if world > 1 and not args.no_parity:
        import contextlib

        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import dist_gpu_check

        with contextlib.redirect_stdout(sys.stderr):
            ok, msg = dist_gpu_check.run_checks(engine, rank, world, dev)
        parity = {"ok": bool(ok), "detail": msg}

    # ---- secondary metrics: BASELINE configs 4 (GROUP BY) and 5 (JOIN) at their per-GPU share,
    #      through engine.aggregate / engine.join (distributed at N > 1; every rank takes part)
    extras = None
    if not args.no_extras:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import relational_bench

            torch.cuda.empty_cache()
            if world == 1:
                extras = relational_bench.measure(local_rank)
            else:
                extras = relational_bench.measure_dist(engine, rank, world, dev)
        except Exception as ex:  # pragma: no cover
            extras = {"error": repr(ex)[:300]}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            rps, dt = _time_reference(REF_SAMPLE_ROWS, 2, 0)
            cpu = {"value": rps, "unit": "rows/s", "cores": 1, "kind": "port",
                   "host_cores_available": os.cpu_count(),
                   "sample": f"{REF_SAMPLE_ROWS} rows = the logical partitions of {REF_SAMPLE_KEYS} of the "
                             f"{KEY_CARDINALITY} keys (1526 rows per key as in the full workload), 2 timed passes of the restated "
                             "NativeExecutionEngine.map_dataframe (pandas groupby-iterate + concat); "
                             "the reference is single-threaded (get_current_parallelism() == 1)"}
            if extras is not None and "error" not in extras and not args.no_extras:
                try:
                    extras["cpu_baseline"] = relational_bench.cpu_baselines()
                except Exception as ex:  # pragma: no cover
                    extras["cpu_baseline"] = {"error": repr(ex)[:200]}
        # per step: pass 1 (rank kernel), 2 scans, the scatter launches (+ histogram and scatter of the
        # tail tile); multi-GPU: scatter per column group + barrier kernels, copies are DMA (no kernel)
        if world == 1:
            launches_per_step = 5 + (2 if n % 4096 else 0)
        else:
            ngroups, left, gi = 0, 8, 0
            while left > 0:
                left -= engine._group_cols[min(gi, len(engine._group_cols) - 1)]
                ngroups, gi = ngroups + 1, gi + 1
            launches_per_step = 3 + ngroups + (1 + ngroups if n % 4096 else 0)
        cfg = _config(n, world)
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64+f64 (byte moves; u64 hash arithmetic)", "data": "synthetic",
            "config": cfg, "rows_out_rank0": nrows_out,
            "parallelism": f"dp{world}: rows range-sharded, one exchange over NVLink (copy engines), "
                           f"columns per scatter/exchange group: {engine._group_cols}" if world > 1 else "single GPU",
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * steps,
            "roofline": roofline, "cpu_baseline": cpu, "extras": extras,
        }
        if world > 1:
            line[f"parity_world_{world}"] = None if parity is None else parity["ok"]
            line["parity_detail"] = None if parity is None else parity["detail"]
            # NVLink-bound view of the same step (SURVEY.md 8d): 64 B/row x (G-1)/G leave every GPU
            out_bytes = 64.0 * n * (world - 1) / world
            line["nvlink"] = {"bytes_out_per_gpu": out_bytes, "achieved_GBps_per_gpu": out_bytes / (ms_per_step * 1e-3) / 1e9,
                              "peak_GBps_per_direction": 900.0,
                              "frac": out_bytes / (ms_per_step * 1e-3) / 1e9 / 900.0}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default: 100M at N=1 = config 2, "
                    "125M at N>1 = config 3's share)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's output as .npy files under DIR "
                         "(DIR/rank<r> with several GPUs); see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the output of the b200 arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
