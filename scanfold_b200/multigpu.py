"""Window-range sharding of one record over the ranks of a torch.distributed job (one process per GPU).

The scan itself needs no communication: windows are independent, the record is replicated, and the device
shuffles are keyed by absolute window index, so any sharding folds the same sequences.  The ScanFold-Fold
accumulators (ScanFold.py:1051-1139) overlap only at shard boundaries: the last W - step nucleotides a shard
touches are also covered by the first windows of the following shard(s).  Every rank OWNS the nucleotide rows from
its first nucleotide up to the first nucleotide of the next shard; rows it touches beyond that are sent to the
owner(s) -- more than one when shards are shorter than the overlap -- as integer counts / exact split sums, so the
merge is bit exact whatever the number of ranks.  Rank 0 then gathers the compact per-nucleotide partner lists and
the per-window columns as flat byte tensors (NCCL send/recv on device buffers, gloo on CPU tensors in the tests)
for the cheap argmin / competition / writers.
"""
import numpy as np

from . import foldstep


def shard_windows(total_windows, world, rank):
    """contiguous window range [w0, w1) of `rank`"""
    return total_windows * rank // world, total_windows * (rank + 1) // world


def shard_rows(total_windows, world, W, step):
    """Per rank (touch0, touch1, own0, own1): the nucleotide rows (0-based, half open) the rank's windows touch and the
    rows it owns.  Ranks without windows touch and own nothing."""
    touch = []
    for r in range(world):
        w0, w1 = shard_windows(total_windows, world, r)
        touch.append((w0 * step, (w1 - 1) * step + W) if w1 > w0 else (0, 0))
    out = []
    for r in range(world):
        t0, t1 = touch[r]
        if t1 == t0:
            out.append((0, 0, 0, 0))
            continue
        nxt = [touch[q][0] for q in range(r + 1, world) if touch[q][1] > touch[q][0]]
        out.append((t0, t1, t0, min(t1, nxt[0]) if nxt else t1))
    return out


def _sync_device(tensors):
    """NCCL work is ordered against torch's current stream only: make the host wait before the library's own launches"""
    if tensors and tensors[0].is_cuda:
        import torch
        torch.cuda.current_stream().synchronize()


def exchange_halo(acc, W, step, rank, world, dist, total_windows):
    """Send the rows this shard touches but later shards own, merge the rows earlier shards send us.
    `acc` (None on a rank without windows) has export_tensors(row0, n_rows) -> (count, first_seen, sums) and
    merge_tensors(row0, n_rows, ...), on whatever device the process group moves (CUDA for NCCL, CPU for gloo).
    Returns the number of owned rows (they start at row 0 of the accumulator)."""
    rows = shard_rows(total_windows, world, W, step)
    t0, t1, own0, own1 = rows[rank]
    if acc is not None and (acc.nt0 != t0 or acc.n_nt != t1 - t0):
        raise ValueError("accumulator geometry does not match the shard of rank %d" % rank)
    if world == 1:
        return own1 - own0
    ops, keep, recv = [], [], []
    for q in range(rank + 1, world):                       # rows of ours that rank q owns
        a, b = max(rows[q][2], t0), min(rows[q][3], t1)
        if acc is not None and b > a:
            send = acc.export_tensors(a - t0, b - a)
            keep.append(send)
            ops += [dist.P2POp(dist.isend, t, q) for t in send]
    for p in range(rank):                                  # rows of rank p's shard that we own
        a, b = max(own0, rows[p][0]), min(own1, rows[p][1])
        if acc is not None and b > a:
            buf = acc.empty_tensors(b - a)
            recv.append((a - t0, b - a, buf))
            ops += [dist.P2POp(dist.irecv, t, p) for t in buf]
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
        _sync_device([op.tensor for op in ops])
    for row0, n_rows, buf in recv:
        acc.merge_tensors(row0, n_rows, *buf)
    return own1 - own0


# ---------------------------------------------------------------------------------------------------------------
def _pack(arrays):
    """list of numpy arrays -> (uint8 payload, header of (dtype string, shape) per array)"""
    arrays = [np.ascontiguousarray(a) for a in arrays]
    payload = np.concatenate([a.reshape(-1).view(np.uint8) for a in arrays]) if arrays else np.zeros(0, np.uint8)
    return payload, [(a.dtype.str, a.shape) for a in arrays]


def _unpack(payload, header):
    out, off = [], 0
    for dt, shape in header:
        n = int(np.prod(shape)) * np.dtype(dt).itemsize
        out.append(payload[off:off + n].view(dt).reshape(shape).copy())
        off += n
    return out


def gather_arrays(arrays, rank, world, dist):
    """Every rank contributes a list of numpy arrays with the same dtypes and trailing dimensions (axis 0 may differ);
    rank 0 gets a list (per rank) of lists of arrays, the others None.  One flat byte tensor per rank moves through the
    process group (device buffers under NCCL); only the [n_arrays] vector of axis-0 lengths is exchanged first."""
    import torch
    if world == 1:
        return [list(arrays)]
    backend = dist.get_backend()
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    arrays = [np.ascontiguousarray(a) for a in arrays]
    lens = torch.tensor([a.shape[0] for a in arrays], dtype=torch.int64, device=dev)
    all_lens = [torch.empty_like(lens) for _ in range(world)]
    dist.all_gather(all_lens, lens)
    all_lens = [t.cpu().numpy() for t in all_lens]
    payload, _ = _pack(arrays)
    row_bytes = [int(np.prod(a.shape[1:], dtype=np.int64)) * a.dtype.itemsize for a in arrays]
    if rank != 0:
        if len(payload):
            t = torch.from_numpy(payload).to(dev)
            for req in dist.batch_isend_irecv([dist.P2POp(dist.isend, t, 0)]):
                req.wait()
            _sync_device([t])
        return None
    bufs, ops = [], []
    for p in range(1, world):
        nbytes = int(sum(int(n) * rb for n, rb in zip(all_lens[p], row_bytes)))
        bufs.append(torch.empty(nbytes, dtype=torch.uint8, device=dev))
        if nbytes:
            ops.append(dist.P2POp(dist.irecv, bufs[-1], p))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
        _sync_device(bufs)
    out = [list(arrays)]
    for p in range(1, world):
        header = [(a.dtype.str, (int(n),) + a.shape[1:]) for a, n in zip(arrays, all_lens[p])]
        out.append(_unpack(bufs[p - 1].cpu().numpy(), header))
    return out


def gather_tables(table, rank, world, dist):
    """per-rank PartnerTable over consecutive nucleotide ranges -> the whole table on rank 0 (None elsewhere)"""
    if world == 1:
        return table
    parts = gather_arrays([np.diff(table.nt_ptr), table.coord, table.partner, table.count, table.first_seen,
                           np.ascontiguousarray(table.sums.T)], rank, world, dist)
    if rank != 0:
        return None
    tabs = []
    for nparts, coord, partner, count, first, sums_t in parts:
        ptr = np.concatenate([[0], np.cumsum(nparts)])
        tabs.append(foldstep.PartnerTable(ptr, partner, count, first, sums_t.T, coord))
    return foldstep.concat_tables(tabs)


def empty_table():
    z = np.zeros(0, dtype=np.int64)
    return foldstep.PartnerTable(np.zeros(1, dtype=np.int64), z, z, z, np.zeros((6, 0), dtype=np.int64), z)


def pairprob_distributed(table, W, step, rank, world, dist, total_windows, cutoff):
    """Window-averaged pair probabilities of the whole record on rank 0: halo exchange of the PairProbTable rows (exact
    integer sums, so any sharding gives the same result), every rank reduces the rows it owns, rank 0 gathers them.
    `table` is None on a rank without windows.  -> (paired [nucleotides up to the end of the last window], i, j, p) on
    rank 0, None elsewhere.  Nucleotides no window holds (step > W) belong to no rank and stay 0."""
    own = exchange_halo(table, W, step, rank, world, dist, total_windows)
    if table is not None and own > 0:
        part = list(table.reduce(0, own, cutoff))
    else:
        part = [np.zeros(0), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0)]
    parts = gather_arrays(part, rank, world, dist)
    if rank != 0:
        return None
    rows = shard_rows(total_windows, world, W, step)
    paired = np.zeros(max(r[1] for r in rows))
    for r, p in zip(rows, parts):
        paired[r[2]:r[2] + len(p[0])] = p[0]
    return (paired,) + tuple(np.concatenate([p[k] for p in parts]) for k in range(1, 4))


def own_partner_table(acc, W, step, rank, world, dist, total_windows):
    """halo exchange + compaction: the complete partner lists of the nucleotides this rank owns"""
    own = exchange_halo(acc, W, step, rank, world, dist, total_windows)
    return foldstep.table_from_compact(*acc.compact(0, own), nt0=acc.nt0) if acc is not None and own > 0 else empty_table()


def partner_table_distributed(acc, W, step, rank, world, dist, total_windows):
    """halo exchange + compaction of the owned nucleotides + gather of the whole table on rank 0"""
    return gather_tables(own_partner_table(acc, W, step, rank, world, dist, total_windows), rank, world, dist)


_RESULT_FIELDS = ("coord", "part", "cov_z", "mean_z", "mean_mfe", "mean_ed", "total_windows", "num_bp")


def aggregate_distributed(table, seq, rank, world, dist, by_ed=False, with_logs=False):
    """ScanFold.py:1051-1260 sharded: every rank aggregates the nucleotides it owns (their partner lists are complete after
    the halo exchange) and rank 0 gathers the per-nucleotide results -- 64 bytes per nucleotide instead of the 80-byte
    entries of the whole partner table -- plus, for the CLI, the log text each rank produced for its rows.
    -> (NtResult, log text, pair-count text) on rank 0, (None, None, None) elsewhere."""
    import io
    log_total, sirna = (io.StringIO(), io.StringIO()) if with_logs else (None, None)
    res = foldstep.aggregate(table, seq, log_total, sirna, by_ed=by_ed)
    if world == 1:
        return res, (log_total.getvalue() if with_logs else None), (sirna.getvalue() if with_logs else None)
    arrays = [np.asarray(getattr(res, k)) for k in _RESULT_FIELDS]
    if with_logs:
        arrays += [np.frombuffer(log_total.getvalue().encode(), dtype=np.uint8),
                   np.frombuffer(sirna.getvalue().encode(), dtype=np.uint8)]
    parts = gather_arrays(arrays, rank, world, dist)
    if rank != 0:
        return None, None, None
    out = foldstep.NtResult()
    for n, k in enumerate(_RESULT_FIELDS):
        setattr(out, k, np.concatenate([p[n] for p in parts]))
    out.n_nt = len(out.coord)
    if not with_logs:
        return out, None, None
    return (out, "".join(p[-2].tobytes().decode() for p in parts), "".join(p[-1].tobytes().decode() for p in parts))


def table_checksum(table, rank, world, dist):
    """Order-independent 64-bit digest of a partner table spread over the ranks (sum of per-entry hashes mod 2^64, all-
    reduced): equal for any sharding iff the merged tables are equal entry by entry.  bench.py prints it in result_sha."""
    own = np.repeat(table.coord, np.diff(table.nt_ptr)).astype(np.uint64)
    with np.errstate(over="ignore"):
        h = own * np.uint64(0x9E3779B97F4A7C15)
        for k, a in enumerate([table.partner, table.count, table.first_seen] + list(table.sums)):
            h = (h ^ (h >> np.uint64(29))) * np.uint64(0xBF58476D1CE4E5B9) + np.asarray(a).astype(np.int64).view(np.uint64) * np.uint64(2 * k + 3)
        h = (h ^ (h >> np.uint64(32))) * np.uint64(0x94D049BB133111EB)
        total = int(h.sum(dtype=np.uint64)) if len(h) else 0
    if world > 1:
        import torch
        dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
        # two 32-bit halves: int64 all-reduce sums cannot wrap, the wrap is applied afterwards
        t = torch.tensor([total & 0xFFFFFFFF, total >> 32], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        lo, hi = (int(x) for x in t.tolist())
        total = (lo + (hi << 32)) & 0xFFFFFFFFFFFFFFFF
    return total


_WINDOW_COLUMNS = ("start1", "end1", "mfe_dcal", "mfe", "z", "p", "ed", "pair_tbl", "centroid_tbl",
                   "native_unconstrained_dcal")


def gather_window_tables(table, rank, world, dist, with_shuffle_energies=False):
    """per-rank scan.WindowTable shards -> one table on rank 0 (None elsewhere).  The shuffle energies stay on their
    rank unless asked for (--print_random): rank 0 only needs the per-window columns the writers print."""
    from .scan import WindowTable
    if world == 1:
        return table
    cols = _WINDOW_COLUMNS + (("shuffle_dcal",) if with_shuffle_energies else ())
    fin = table.final
    extra = np.array([[1.0, fin["mfe"], fin["z"], fin["p"], fin["ed"]]] if fin is not None else np.zeros((0, 5)))
    alln = np.asarray(table.alln, dtype=np.uint8) if getattr(table, "alln", None) is not None \
        else np.zeros(len(table.start1), dtype=np.uint8)
    parts = gather_arrays([np.asarray(getattr(table, k)) for k in cols] + [alln, extra], rank, world, dist)
    if rank != 0:
        return None
    res = WindowTable()
    res.W, res.step, res.r, res.first_window = table.W, table.step, table.r, table.first_window
    for n, k in enumerate(cols):
        setattr(res, k, np.concatenate([p[n] for p in parts]))
    if not with_shuffle_energies:
        res.shuffle_dcal = None
    alln_all = np.concatenate([p[-2] for p in parts]).astype(bool)
    res.alln = alln_all if alln_all.any() else None
    fins = [p[-1] for p in parts if len(p[-1])]
    res.final = dict(zip(("mfe", "z", "p", "ed"), (float(x) for x in fins[-1][0][1:]))) if fins else None
    return res
