"""Pass 1 of the hash partition, byte for byte: the scratch that ``partition_plan`` leaves behind.

For ``num <= 256`` the scratch holds the per-chunk histogram (after the scan: the exclusive prefix of
every partition over the chunks) and one 12800-byte rank record per full 4096-row tile:
u8 partition id of every row, u16 rank of the row among the rows of its partition in the tile, and
u16 rows per partition in the tile (256 entries).  The reference below builds the same bytes with a
stable argsort per tile from the oracle's partition ids.
"""
import numpy as np
import pytest

from oracle import hash_partition as hp

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

TILE = 4096
REC_BYTES = 3 * TILE + 512


def _geometry(n: int):
    """Chunk geometry of the partition kernels: whole tiles cut into at most 2 x #SM chunks, plus a
    tail chunk for the partial last tile."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ntiles = n // TILE
    tpc = -(-ntiles // (2 * sms)) if ntiles > 0 else 1
    nchunks_full = -(-ntiles // tpc)
    nchunks = nchunks_full + (1 if ntiles * TILE < n else 0)
    return ntiles, tpc, nchunks_full, nchunks


def _reference(pids: np.ndarray, num: int):
    n = len(pids)
    ntiles, tpc, nchunks_full, nchunks = _geometry(n)
    full = ntiles * TILE
    p = pids[:full].astype(np.int64)
    key = (np.arange(full, dtype=np.int64) >> 12) * 256 + p  # (tile, partition)
    order = np.argsort(key, kind="stable")
    sk = key[order]
    starts = np.r_[0, np.flatnonzero(np.diff(sk)) + 1]
    first = np.repeat(starts, np.diff(np.r_[starts, full]))
    rank = np.empty(full, dtype=np.int64)
    rank[order] = np.arange(full) - first
    counts = np.bincount(key, minlength=ntiles * 256).reshape(ntiles, 256)
    rec = np.empty((ntiles, REC_BYTES), dtype=np.uint8)
    rec[:, :TILE] = p.reshape(ntiles, TILE)
    rec[:, TILE:3 * TILE] = rank.astype("<u2").reshape(ntiles, TILE).view(np.uint8)
    rec[:, 3 * TILE:] = counts.astype("<u2").view(np.uint8)
    row = np.arange(n, dtype=np.int64)
    chunk = np.where(row < full, (row >> 12) // tpc, nchunks_full)
    h = np.bincount(chunk * num + pids, minlength=nchunks * num).reshape(nchunks, num)
    hist = (np.cumsum(h, axis=0) - h).astype("<u4")
    return hist, rec


def _check(cols, num, valid=None):
    from fugue_b200 import kernels as K

    dev = torch.device("cuda", 0)
    keys = [torch.from_numpy(np.ascontiguousarray(c)).to(dev) for c in cols]
    vt = None if valid is None else [None if v is None else torch.from_numpy(v.astype(np.uint8)).to(dev) for v in valid]
    n = len(cols[0])
    need = K.partition_scratch_bytes(dev, n, num)
    scratch = torch.full((need,), 0xAB, dtype=torch.uint8, device=dev)
    plan = K.partition_plan(keys, num, vt, scratch=scratch)
    torch.cuda.synchronize()
    got = scratch.cpu().numpy()
    pids = hp.partition_ids(cols, num, valid)
    hist, rec = _reference(pids, num)
    ntiles, _, _, nchunks = _geometry(n)
    hist_bytes = (nchunks * num * 4 + 255) // 256 * 256
    rec0 = hist_bytes + 256
    assert np.array_equal(got[:hist.nbytes], hist.view(np.uint8).ravel()), "chunk histogram differs"
    got_rec = got[rec0:rec0 + ntiles * REC_BYTES].reshape(ntiles, REC_BYTES)
    bad = np.flatnonzero((got_rec != rec).any(axis=1))
    assert bad.size == 0, f"{bad.size} of {ntiles} rank records differ, first tile {bad[:1]}"
    offsets = plan.offsets.cpu().numpy()
    assert np.array_equal(offsets, np.r_[0, np.cumsum(np.bincount(pids, minlength=num))])


RNG = np.random.default_rng(20261017)
N_TAIL = 1025 * TILE + 77  # several tiles per chunk and a partial tail tile


@pytest.mark.parametrize("num", [2, 16, 17, 255, 256])
def test_uniform_keys(num):
    _check([RNG.integers(-(2**63), 2**63 - 1, N_TAIL, dtype=np.int64)], num)


@pytest.mark.parametrize("num", [17, 256])
def test_hot_key_on_40_percent_of_rows(num):
    k = RNG.integers(0, 1 << 16, N_TAIL, dtype=np.int64)
    k[RNG.random(N_TAIL) < 0.4] = 12345
    _check([k], num)


def test_single_key():
    _check([np.full(N_TAIL, 777, dtype=np.int64)], 256)


def test_whole_tiles_one_per_chunk():
    _check([RNG.integers(0, 1000, 3 * TILE, dtype=np.int64)], 256)


@pytest.mark.parametrize("num", [16, 256])
def test_multi_key_columns(num):
    a = RNG.integers(0, 300, N_TAIL, dtype=np.int64)
    b = RNG.integers(-5, 5, N_TAIL, dtype=np.int32)
    _check([a, b], num)


@pytest.mark.parametrize("num", [16, 255])
def test_nullable_key(num):
    k = RNG.integers(0, 1 << 20, N_TAIL, dtype=np.int64)
    v = RNG.random(N_TAIL) > 0.3
    _check([k], num, [v])


def test_many_tiles_per_warp():
    """More tiles per chunk than warps per CTA: every warp ranks several tiles of its chunk."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * sms * 35 * TILE + 1234
    _check([RNG.integers(0, 1 << 16, n, dtype=np.int64)], 256)
