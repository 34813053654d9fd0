"""Times pass 1 of the hash partition alone: ``partition_plan`` on the benchmark's key column.

The call runs ``fb_rank_kernel`` over the whole 4096-row tiles (partition ids, stable ranks and counts
of every tile, per-chunk histogram) plus the tail-tile histogram and the two small scans.  CUDA events
around ``--iters`` back-to-back calls after ``--warmup`` calls; prints one JSON line with the mean and
the bytes-over-peak floor of the kernel, computed from shapes:
  read   8 B per row (the int64 key)
  write  12800 B per whole tile (u8 id + u16 rank per row, u16 count per partition) + the histogram.
Usage: python tools/rank_bench.py [--rows 100000000] [--num 256] [--peak-tbs 6.57]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--num", type=int, default=256)
    ap.add_argument("--keys", type=int, default=65536, help="key cardinality (bench.py: 2**16)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3, help="timed windows; all are reported")
    ap.add_argument("--peak-tbs", type=float, default=6.57, help="copy bandwidth for the floor, TB/s")
    a = ap.parse_args()

    import torch

    from fugue_b200 import kernels as K

    if not torch.cuda.is_available():
        sys.exit("rank_bench needs a GPU")
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    key = torch.randint(0, a.keys, (a.rows,), dtype=torch.int64, device=dev, generator=g)
    scratch = torch.empty(K.partition_scratch_bytes(dev, a.rows, a.num), dtype=torch.uint8, device=dev)
    offsets = torch.empty(a.num + 1, dtype=torch.int64, device=dev)
    for _ in range(a.warmup):
        K.partition_plan([key], a.num, scratch=scratch, offsets=offsets)
    torch.cuda.synchronize()
    means = []
    for _ in range(a.repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.iters):
            K.partition_plan([key], a.num, scratch=scratch, offsets=offsets)
        e1.record()
        torch.cuda.synchronize()
        means.append(e0.elapsed_time(e1) / a.iters)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    tiles = a.rows // 4096
    nchunks = min(tiles, 2 * sms) + 1
    nbytes = 8 * a.rows + 12800 * tiles + 4 * nchunks * a.num
    floor_ms = nbytes / (a.peak_tbs * 1e12) * 1e3
    name = torch.cuda.get_device_name(dev)
    print(json.dumps({"what": "partition_plan (pass 1 + scans)", "device": name, "rows": a.rows, "num": a.num,
                      "ms_mean": round(sum(means) / len(means), 4), "ms_windows": [round(m, 4) for m in means],
                      "iters_per_window": a.iters, "bytes": nbytes, "peak_tbs": a.peak_tbs,
                      "floor_ms": round(floor_ms, 4)}))


if __name__ == "__main__":
    main()
