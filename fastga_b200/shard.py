"""Multi-GPU plumbing of the path: k-mer-space sharding (two all-to-alls of 16-byte records) and the
gather of the per-rank alignment record streams on rank 0."""
import numpy as np


def pack_alignments(alns, contig_map=None):
    """Alignments -> one uint8 buffer (fields | toff | pool); contig_map renumbers the shard's
    local A-contig numbers to global ones."""
    fields = alns.fields.copy()
    if contig_map is not None and len(fields):
        fields[:, 1] = np.asarray(contig_map, dtype=np.int32)[fields[:, 1]]
    n = np.array([len(alns), alns.pool.size if len(alns) else 0, alns.nraw], dtype=np.int64)
    pool = alns.pool if len(alns) else np.zeros(0, np.uint8)
    return np.concatenate([n.view(np.uint8), fields.reshape(-1).view(np.uint8),
                           alns.toff.view(np.uint8), pool.view(np.uint8)])


def unpack_alignments(buf):
    from .lib import Alignments
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    n, pb, nraw = (int(x) for x in buf[:24].view(np.int64))
    o = 24
    fields = buf[o:o + n * 36].view(np.int32).reshape(n, 9).copy()
    o += n * 36
    toff = buf[o:o + n * 8].view(np.int64).copy()
    o += n * 8
    pool = buf[o:o + pb].copy()
    return Alignments(fields, toff, pool if pb else np.zeros(1, np.uint8), nraw)


def gather_alignments(alns, contig_map, dist, device):
    """Variable-length gather of every rank's records on rank 0 (NCCL on GPUs, gloo in tests).
    Returns the merged Alignments in (aread, abpos, bread, comp) order on rank 0, None elsewhere."""
    import torch
    rank, world = dist.get_rank(), dist.get_world_size()
    payload = torch.from_numpy(pack_alignments(alns, contig_map)).to(device)
    size = torch.tensor([payload.numel()], dtype=torch.int64, device=device)
    sizes = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(sizes, size)
    mx = max(int(s.item()) for s in sizes)
    pad = torch.zeros(mx, dtype=torch.uint8, device=device)
    pad[:payload.numel()] = payload
    bufs = [torch.zeros(mx, dtype=torch.uint8, device=device) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, bufs, dst=0)
    if rank != 0:
        return None
    parts = [unpack_alignments(b[:int(s.item())].cpu().numpy()) for b, s in zip(bufs, sizes)]
    return merge_alignments(parts)


def merge_alignments(parts):
    """Concatenates per-shard results and restores the global SORT_MAP order (FastGA.c:3800-3836)."""
    from .lib import Alignments
    fields = np.concatenate([p.fields for p in parts]) if parts else np.zeros((0, 9), np.int32)
    pools, toffs, base = [], [], 0
    for p in parts:
        toffs.append(p.toff + base)
        pl = p.pool[:int((p.toff + p.fields[:, 8]).max())] if len(p) else np.zeros(0, np.uint8)
        pools.append(pl)
        base += len(pl)
    toff = np.concatenate(toffs) if toffs else np.zeros(0, np.int64)
    pool = np.concatenate(pools) if pools else np.zeros(1, np.uint8)
    order = np.lexsort((fields[:, 0], fields[:, 2], fields[:, 3], fields[:, 1]))
    return Alignments(fields[order], toff[order], pool if pool.size else np.zeros(1, np.uint8),
                      sum(p.nraw for p in parts))


# ---------------------------------------------------------------------------------------------
#  k-mer-space sharding (the N > 1 path of bench.py): nothing is replicated.
#    1. every rank scans ITS contigs of both genomes (syncmer scan + record build);
#    2. the k-mer records travel to the rank that owns their prefix range (all-to-all #1);
#    3. every rank sorts + indexes its slice of both tables and merges them -> seeds;
#    4. the seeds travel to the rank that owns their A-contig (all-to-all #2);
#    5. every rank sorts its seeds and extends them; rank 0 gathers the records.
#  Both exchanges move 16-byte records between device buffers with NCCL (all_to_all_single).
# ---------------------------------------------------------------------------------------------

def owner_of_contigs(lengths, world):
    """greedy length balance, longest first: owner[c] for every contig (deterministic on every rank)"""
    order = np.argsort(-np.asarray(lengths, dtype=np.int64), kind="stable")
    load = [0] * world
    owner = np.zeros(len(lengths), dtype=np.int32)
    for i in order:
        r = int(np.argmin(load))
        owner[int(i)] = r
        load[r] += int(lengths[int(i)])
    return owner


def top_byte_cuts(world):
    """rank r owns the k-mers whose first four bases (top byte) lie in [cuts[r], cuts[r+1])"""
    return [(256 * r + world - 1) // world for r in range(world + 1)]


def exchange_rows(dist, rows, send_rows, async_op=False):
    """all-to-all of 16-byte records: `rows` is an (n,2) int64 tensor whose rows
    [sum(send_rows[:r]), +send_rows[r]) go to rank r.  Returns the (m,2) tensor of received rows, in
    source-rank order (NCCL on GPUs, gloo in the CPU tests).  async_op: returns (tensor, work) with the
    transfer still in flight -- work.wait() before the tensor is read (and keep `rows` alive until then)."""
    import torch
    world = dist.get_world_size()
    device = rows.device
    sr = torch.tensor([int(v) for v in send_rows], dtype=torch.int64, device=device)
    rr = torch.empty(world, dtype=torch.int64, device=device)
    dist.all_to_all_single(rr, sr)
    recv_rows = [int(v) for v in rr.tolist()]
    n_send, n_recv = int(sum(send_rows)), int(sum(recv_rows))
    dst = torch.empty((max(n_recv, 1), 2), dtype=torch.int64, device=device)[:n_recv]
    work = dist.all_to_all_single(dst, rows[:n_send].contiguous(), output_split_sizes=recv_rows,
                                  input_split_sizes=[int(v) for v in send_rows], async_op=async_op)
    return (dst, work) if async_op else dst


def align_sharded(dA, dB, freqA, dist, device, **kw):
    """The whole path on world GPUs from device-resident genomes (every rank holds both genomes:
    2 bits per base).  Returns (Alignments of this rank's A-contigs with GLOBAL contig numbers, stats)."""
    import torch
    from . import lib
    rank, world = dist.get_rank(), dist.get_world_size()
    gA, gB = dA.genome, dB.genome
    p = dict(lib.DEFAULTS)
    p.update(kw)
    import os, sys, time
    trace = [] if os.environ.get("FGB_SHARD_TRACE") else None

    def mark(what):                      # phase wall clock per rank (diagnostics only: it synchronizes)
        if trace is not None:
            torch.cuda.synchronize()
            trace.append((what, time.perf_counter()))
    mark("start")
    ownA = owner_of_contigs(gA.clen, world)
    ownB = owner_of_contigs(gB.clen, world)
    cuts = top_byte_cuts(world)
    plo, phi = cuts[rank] << 16, cuts[rank + 1] << 16
    from .formats import gix_bytes
    #  The two tables are pipelined: while the k-mer records of one travel (NCCL's stream), this rank's
    #  stream scans / groups the other genome or sorts the slice that already arrived.
    nk, flight = [], []
    owner256 = np.zeros(256, dtype=np.int32)
    for r in range(world):
        owner256[cuts[r]:cuts[r + 1]] = r
    for dg, own, fwd in ((dA, ownA, True), (dB, ownB, False)):
        ptr, n = lib.kmers_scan(dg, own == rank, fwd)
        mark("scan")
        grouped = torch.empty((max(n, 1), 2), dtype=torch.int64, device=device)
        bounds = lib.records_group_by_owner(ptr, n, owner256, world, grouped.data_ptr())
        lib.device_free(ptr)
        mark("group k-mers")
        send = [int(bounds[r + 1] - bounds[r]) for r in range(world)]
        recv, work = exchange_rows(dist, grouped, send, async_op=True)
        flight.append((recv, work, grouped))
        mark("exchange k-mers (issued)")
    tables = []
    for (recv, work, grouped), dg, fwd in zip(flight, (dA, dB), (True, False)):
        work.wait()
        del grouped
        pb, cb = gix_bytes(dg.genome)
        if phi > plo:
            x = lib.gix_from_records(recv.data_ptr() if recv.shape[0] else 0, int(recv.shape[0]), plo, phi, fwd,
                                     pb, cb, dg.genome.ncontig)
        else:
            x = None
        mark("sort+index slice")
        tables.append(x)
        nk.append(int(recv.shape[0]))
        del recv
    del flight
    xA, xB = tables
    amx, bmx = int(gA.clen.max()), int(gB.clen.max())
    if xA is not None:
        sptr, ns, bits, sumlen, n1m = lib.seeds_merge(xA, xB, amx, bmx, p["freq"])
        xA.close()
        xB.close()
    else:
        sptr, ns, sumlen, n1m = 0, 0, 0, 0
        ab = int(amx + bmx).bit_length()
        bits = (ab, max(ab - 6, 1), max(1, (gB.ncontig - 1).bit_length()), max(1, (gA.ncontig - 1).bit_length()))
    mark("merge")
    # owner of every A-contig RANK (the icont field of a seed)
    own_by_rank = ownA[dA.perm]
    grouped = torch.empty((max(ns, 1), 2), dtype=torch.int64, device=device)
    bounds = lib.seeds_group_by_owner(sptr, ns, bits, own_by_rank, world, grouped.data_ptr())
    if sptr:
        lib.device_free(sptr)
    mark("group seeds")
    send = [int(bounds[r + 1] - bounds[r]) for r in range(world)]
    recv = exchange_rows(dist, grouped, send)
    mark("exchange seeds")
    del grouped
    S = lib.seeds_from_records(recv.data_ptr() if recv.shape[0] else 0, int(recv.shape[0]), bits, amx, bmx)
    nseeds_mine = int(recv.shape[0])
    del recv
    mark("sort seeds")
    ov = lib.DeviceOverlaps.extend(S, dA, dB, freqA, p["chain_break"], p["chain_min"], p["align_min"], p["align_rate"])
    cnt = ov.counters()
    mark("extend")
    alns = lib.filter_overlaps(ov.h, dA.perm, dB.perm, bits[2], bits[3])
    ov.close()
    S.close()
    mark("filter")
    if trace is not None:
        sys.stderr.write("[shard %d] " % rank + " | ".join("%s %.2f" % (w, 1e3 * (t - trace[i][1]))
                                                          for i, (w, t) in enumerate(trace[1:])) + "\n")
    stats = {"nkmers1_fwd": nk[0], "nkmers2": nk[1], "nseeds_merged": ns, "nseeds": nseeds_mine, "sumlen": sumlen,
             "nhits": cnt["hits"], "nla": cnt["la_calls"], "nwaves": cnt["waves"], "ncells": cnt["cells"],
             "nseg": cnt["nseg"], "nwork": cnt["nwork"], "warp_cycles": cnt["warp_cycles"],
             "wave_cycles": cnt["wave_cycles"], "extract_cycles": cnt["extract_cycles"],
             "slow_cycles": cnt["slowest_warp"]["cycles"], "slow_waves": cnt["slowest_warp"]["waves"],
             "paired_waves": cnt["paired_waves"], "pairings": cnt["pairings"]}
    return alns, stats
