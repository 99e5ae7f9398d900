"""Multi-GPU plumbing (one process per GPU, torch.distributed): reads shard across ranks with no data-path
collective.  The only exchanges are, once per byte range,
(1) one all-gather of an int64 per rank -- the contig of the rank's first kept line: the window a rank leaves open at the
    end of its slice is closed by the first kept line of the next rank that has one (reference semantics of
    extract_contexts.py:179 across the byte-range split of mCaller.py:63-68); the result stays on the device and is
    consumed there by mc_carry_close,
(2) the all-reduce of the per-site histograms: one SUM over the packed depth|meth counts, one MIN over the first-seen
    row indices (NCCL over NVLink on the GPU box, gloo when several ranks share a GPU), and
(3) only when a per-read summary is asked for (make_bed --vo / -p: `--bed_vo`, `--bed_positions`), the gather of every
    rank's row log to rank 0: one all-gather of the entry counts, one gather of the entries."""
import torch
import torch.distributed as dist


def shard_range(n_items, rank, world):
    """Contiguous slice [lo, hi) of n_items owned by `rank`."""
    lo = (n_items * rank) // world
    hi = (n_items * (rank + 1)) // world
    return lo, hi


def gather_first_kept(first_kept_contig, group=None):
    """first_kept_contig: int64 tensor [1] (-1 = the rank's slice holds no kept line).  Returns the int64 tensor [world] of
    every rank's value, on the same device; rank r's open window is closed by the first entry >= 0 after position r."""
    world = dist.get_world_size(group)
    out = torch.empty(world, dtype=torch.int64, device=first_kept_contig.device)
    dist.all_gather_into_tensor(out, first_kept_contig.contiguous(), group=group)
    return out


def closing_contig(all_first_kept, rank):
    """Host-side restatement of what mc_carry_close does with the gathered tensor (tests, CPU plumbing)."""
    for c in all_first_kept[rank + 1:].tolist():
        if c >= 0:
            return int(c)
    return -1


def allreduce_histogram(counts, first, group=None):
    """In-place combine of the per-site tables across ranks: counts = depth|meth packed in one int32 tensor."""
    dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(first, op=dist.ReduceOp.MIN, group=group)


def rank_row_base(rank):
    """Row-index offset that keeps first-seen order global: rows of rank r sort after those of rank r-1."""
    return int(rank) << 40


def close_and_reduce(engine, rank, group=None, fetch=True):
    """End of a rank's byte range in a multi-GPU run: close the window still open with the next rank's first kept line,
    then combine the histograms.  Returns the completed row (host array of one mc_call, kind MC_NONE when there was nothing
    to close) when `fetch`.  Under gloo (several ranks sharing one GPU) both exchanges are staged through host memory."""
    host = dist.get_backend(group) == "gloo"
    first_kept = engine.first_kept_contig_dev()
    allk = gather_first_kept(first_kept.cpu() if host else first_kept, group).to(engine.device)
    row = engine.close_carry(next_contigs=allk, start=rank + 1, fetch=fetch)
    if host:
        counts, first = engine.d_counts.cpu(), engine.d_first.cpu()
        allreduce_histogram(counts, first, group)
        engine.d_counts.copy_(counts)
        engine.d_first.copy_(first)
    else:
        allreduce_histogram(engine.d_counts, engine.d_first, group)
    return row


def gather_row_log(engine, rank, group=None, dst=0):
    """Every rank's row log (Engine.enable_row_log) -> rank `dst`: one all-gather of the counts, one gather of the entries.
    A gather moves equal sizes, so each rank sends max-count entries and `dst` receives them into one buffer of world x
    max-count entries, which the padding is then squeezed out of: with ranks of very different log sizes that buffer is
    up to world times the entries kept.  Returns (uint8 device tensor of the entries in rank order, their count) on `dst`,
    (None, 0) elsewhere.  Under gloo both steps are staged through host memory."""
    host = dist.get_backend(group) == "gloo"
    world = dist.get_world_size(group)
    d_log, n = engine.row_log()
    stride = engine.log_stride
    cnt = torch.tensor([n], dtype=torch.int64, device="cpu" if host else engine.device)
    counts = torch.empty(world, dtype=torch.int64, device=cnt.device)
    dist.all_gather_into_tensor(counts, cnt, group=group)
    counts = counts.tolist()
    width = max(max(counts), 1) * stride
    dev = "cpu" if host else engine.device
    send = torch.zeros(width, dtype=torch.uint8, device=dev)
    send[:n * stride].copy_(d_log)
    recv = torch.empty(world, width, dtype=torch.uint8, device=dev) if rank == dst else None
    dist.gather(send, list(recv.unbind(0)) if recv is not None else None, dst=dst, group=group)
    if rank != dst:
        return None, 0
    total = int(sum(counts))
    out = torch.empty(total * stride, dtype=torch.uint8, device=engine.device)
    o = 0
    for r, c in enumerate(counts):
        out[o:o + c * stride].copy_(recv[r, :c * stride])
        o += c * stride
    return out, total
