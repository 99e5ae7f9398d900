"""Multi-GPU run of the hot path on one eventalign file (SURVEY.md 8e): one process per GPU, rank r owns the reads whose
first line lies in byte range r of N (the reference's `-t N` split, mCaller.py:63-68, snapped to read boundaries), writes
its rows to `<prefix>.diffs.<k>.tmp<start>`, and the ranks exchange over NCCL the contig of each rank's first kept line
(closes the previous rank's last window, extract_contexts.py:179) and the per-site histograms (make_bed.py:86-96), from
which rank 0 writes the BED / GFF without ever parsing the `.diffs` text.  make_bed's per-read modes (`--bed_vo` = --vo,
`--bed_positions FILE` = -p) also need each locus's rows: every rank then logs the rows its histogram counts on the device
(probability, global row index, site slot and, with `--bed_positions`, the k features of the rows in that positions set),
the logs are gathered to rank 0 (the third exchange, dist.gather_row_log), grouped by locus there on the device and
handed to make_bed's BED writer.

    python -m mcaller_b200.cli mCaller -m GATC -r ref.fa -e x.eventalign.tsv -f x.fastq -d model.pkl --gpus 8 --bed

Results are identical to a single-worker run: the concatenation of the ranks' files in rank order is the `-t 1`
`.diffs.<k>` file, and the BED equals make_bed.py's on that file (rows in first-seen order).
"""
import math
import os
import socket
import sys


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def byte_ranges(size, world):
    """The reference's split (mCaller.py:63-68): chunk = ceil(size / N), worker i gets [chunk*i, chunk*(i+1))."""
    chunk = int(math.ceil(size / float(world))) if size else 0
    return [(chunk * i, min(size, chunk * (i + 1))) for i in range(world)]


def run_rank(rank, world, port, a, backend=None):
    """Body of one rank (spawned by `run`, or called under torchrun with port=None)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from . import dist as mdist, extract_contexts as ec, make_bed as mb, read_qual
    n_dev = torch.cuda.device_count()
    dev_index = rank % max(n_dev, 1)
    torch.cuda.set_device(dev_index)
    os.environ["MCALLER_B200_DEVICE"] = str(dev_index)
    shared_device = world > n_dev                     # several ranks per GPU (tests on a single-GPU box): NCCL cannot do that
    backend = backend or os.environ.get("MCALLER_B200_DIST_BACKEND") or ("gloo" if shared_device else "nccl")
    own_group = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if port is not None:
            os.environ["MASTER_PORT"] = str(port)
        if backend == "nccl":
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev_index))
        else:
            dist.init_process_group(backend, rank=rank, world_size=world)
        own_group = True
    try:
        size = os.path.getsize(a["tsv"])
        start, end = byte_ranges(size, world)[rank]
        read2qual = read_qual.extract_read_quality_device(a["fastq"], device="cuda:%d" % dev_index)
        if os.path.exists(ec_tmp_name(a["tsv"], a["k"], start)):
            os.remove(ec_tmp_name(a["tsv"], a["k"], start))                  # the reference appends to stale files (quirk Q7)
        run = ec.RangeRun(a["tsv"], a["reference"], read2qual, a["k"], a["skip"], a["qual"], a["modelfile"], start, endline=end,
                          base=a["base"], motif=a["motif"], positions_list=a["positions"], histogram=True,
                          row_base=mdist.rank_row_base(rank))
        bed_positions = a.get("bed_positions") if a.get("bed") else None
        per_read = bool(a.get("bed") and (a.get("bed_vo") or bed_positions))
        if per_read:                                  # make_bed --vo / -p: keep the rows of every locus (or of the listed ones)
            flags = mb.site_flags(run.ref, mb.make_pos_set(bed_positions)) if bed_positions else None
            run.eng.enable_row_log(a["k"] if bed_positions else 0, flags)
        import time
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run.stream()
        torch.cuda.synchronize()
        t_streamed = time.perf_counter()
        dt = t_streamed - t0
        print("rank %d: %.2f GB of eventalign text -> %d rows in %.2f s (%.1f GB/s, %.0f calls/s) on cuda:%d"
              % (rank, run.bytes_done / 1e9, run.sink.n_obs, dt, run.bytes_done / 1e9 / max(dt, 1e-9), run.sink.n_obs / max(dt, 1e-9), dev_index))
        eng = run.eng
        # the window still open at the end of my range <- the first kept line of the next rank that has one; the histograms
        run.consume_closed(mdist.close_and_reduce(eng, rank))
        odd = [None] * world
        dist.all_gather_object(odd, eng.odd_rows())
        d_log, n_log = mdist.gather_row_log(eng, rank) if per_read else (None, 0)
        run.print_counters()
        if rank == 0 and a.get("bed"):
            odd_rows = np.concatenate(odd) if any(len(o) for o in odd) else None
            out = mb.output_name(ec.diffs_name(a["tsv"], a["k"]), bed_positions, a["bed_control"], a["bed_gff"])
            depth, meth, first = eng.histogram_host()
            if per_read:
                mb.aggregate_from_rows(run.ref, depth, meth, first, d_log, n_log, eng.log_nfeat, out, a["bed_depth"], a["bed_thresh"],
                                       pos_list=bed_positions, control=a["bed_control"], verbose_results=a.get("bed_vo", False),
                                       gff=a["bed_gff"], ref=a["bed_ref"], odd_rows=odd_rows)
            else:
                mb.aggregate_from_histogram(run.ref, depth, meth, first, out, a["bed_depth"], a["bed_thresh"], control=a["bed_control"],
                                            gff=a["bed_gff"], ref=a["bed_ref"], odd_rows=odd_rows)
            if per_read:
                print("rank 0: %s written %.3f s after the end of streaming" % (out, time.perf_counter() - t_streamed))
        dist.barrier()
    finally:
        if own_group and dist.is_initialized():
            dist.destroy_process_group()
    return 0


def ec_tmp_name(tsv, k, start):
    """The file the rank (or `-t N` worker) whose byte range starts at `start` writes its rows to."""
    from .extract_contexts import diffs_name
    return diffs_name(tsv, k, start)


def merge_outputs(tsv, k, world, train=False):
    """Ranges do not overlap: concatenation in offset order == the -t 1 `.diffs.<k>` (no sort | uniq as in mCaller.py:103-107);
    with `train`, the `.diffs.<k>.train` of a training run."""
    from .extract_contexts import diffs_name
    size = os.path.getsize(tsv)
    out = diffs_name(tsv, k, train=train)
    with open(out, "wb") as dst:
        for start, _ in byte_ranges(size, world):
            tmp = diffs_name(tsv, k, start, train)
            if os.path.exists(tmp):
                with open(tmp, "rb") as src:
                    while True:
                        blk = src.read(1 << 24)
                        if not blk:
                            break
                        dst.write(blk)
                os.remove(tmp)
    return out


def run(a, world):
    """Spawn `world` ranks on this node (one per GPU) and merge their outputs.  The parent never imports torch (that alone is
    several seconds of a short run): plain `multiprocessing` with the spawn start method; a rank that fails takes the others
    down with it."""
    import multiprocessing
    import time
    ctx = multiprocessing.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=run_rank, args=(r, world, port, a)) for r in range(world)]
    for p in procs:
        p.start()
    failed = None
    while failed is None and any(p.is_alive() for p in procs):
        for r, p in enumerate(procs):
            p.join(0.05)
            if p.exitcode not in (None, 0):
                failed = (r, p.exitcode)
                break
    if failed is None:
        for r, p in enumerate(procs):
            p.join()
            if p.exitcode != 0:
                failed = (r, p.exitcode)
                break
    if failed is not None:
        for p in procs:
            if p.is_alive():
                p.terminate()
        deadline = time.time() + 10
        for p in procs:
            p.join(max(0.0, deadline - time.time()))
        raise RuntimeError("rank %d of %d exited with code %s" % (failed[0], world, failed[1]))
    return merge_outputs(a["tsv"], a["k"], world)


if __name__ == "__main__":
    sys.exit("use: python -m mcaller_b200.cli mCaller ... --gpus N")
