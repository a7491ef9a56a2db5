#!/usr/bin/env python
"""bench.py -- Gbp aligned/s of the FastGA seed-and-extend hot path on B200 (BASELINE.json metric).

One "step" = one pass of the whole path over one synthetic genome pair:
  GIX build of both genomes (syncmer scan, record build, bucketed k-mer sort, prefix index) ->
  adaptamer merge -> seed sort -> chain scan + wave extension -> D2H of the raw alignments -> host
  redundancy filter.
`value`  : inputs (the staged 2-bit genomes) already resident in HBM when the timed region starts.
`e2e`    : the reference-facing C-ABI call fgb_fastga on HOST buffers (.bps images in pinned
           memory), H2D of both images and D2H of the records inside the timed region.
`roofline`: the seed-merge kernel (the kernel SURVEY 8d grades), algorithmic bytes on the on-disk
           widths over its own CUDA-event time; `other_kernels` the sort stages; the extension
           kernel is latency-bound and reported as cell updates/s.
N > 1    : genome-1 contigs are sharded over the ranks; the table of genome 2 is built
           cooperatively (each rank sorts one slice of the k-mer prefix space, NCCL all-gather);
           per-rank results are gathered to rank 0 with torch.distributed.
--impl reference : the UNMODIFIED reference (oracle/_ref: GIXmake x2 + FastGA -T<cores>) on the
           IDENTICAL pair the GPU arm runs at this N (same generator, same seed, same size), from
           the .1gdb/.bps the reference's own FAtoGDB wrote (FASTA parsing is outside both arms'
           timed regions) to the .1aln, temp files on /dev/shm.  One run takes 10 s .. minutes, so
           the number of timed runs is capped (config.reference_runs says how many).
Parity on the bench pair: both arms put the canonical md5 of their alignment records
           (ONEview form, sorted) into the line; at N=1 the GPU arm's cpu_baseline leg runs the
           reference once on the same pair and records whether the two md5s are equal.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20260924
PER_GPU_BP = 100_000_000          # BASELINE.json configs[1]: 100 Mbp genome vs 5 %-diverged copy
DIV = 0.05
NCONTIG = 8
SV_EVERY = 200_000


def workload(n_gpus, per_gpu_bp=PER_GPU_BP):
    from fastga_b200 import synth
    return synth.make_pair(SEED, per_gpu_bp * n_gpus, NCONTIG * n_gpus, DIV, sv_every=SV_EVERY)


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region, through NVML in-process (spawning
    nvidia-smi five times a second stalls the CUDA driver calls of the measured process)."""
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.samples = []
        self.reasons = set()
        self.max_mhz = None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            getr = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception:
            return
        while not self.stop_flag:
            try:
                self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                r = int(getr(h))
                for bit, name in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def other_kernels(stats, dev_ms, peak, seed_passes, nk_sorted):
    """achieved HBM GB/s of the sort stages from their CUDA-event times on THIS rank
    (bytes = records this rank sorted x 16 B x 2 per pass)"""
    out = []
    if dev_ms.get("ksort_ms", 0) > 0:
        b = nk_sorted * 32 * 3
        out.append({"stage": "k-mer table sort (sort_onesweep_kernel x2 + kmer_bucket_sort_kernel), records sorted "
                             "by this rank: %d" % nk_sorted, "bound": "hbm",
                    "bytes": b, "ms": dev_ms["ksort_ms"], "achieved": b / dev_ms["ksort_ms"] / 1e6,
                    "frac": b / dev_ms["ksort_ms"] / 1e6 / peak})
    if dev_ms.get("ssort_ms", 0) > 0:
        passes = seed_passes
        b = stats["nseeds"] * 32 * passes
        out.append({"stage": "seed sort (sort_onesweep_kernel, %d 8-bit passes)" % passes, "bound": "hbm",
                    "bytes": b, "ms": dev_ms["ssort_ms"], "achieved": b / dev_ms["ssort_ms"] / 1e6,
                    "frac": b / dev_ms["ssort_ms"] / 1e6 / peak})
    return out


def ncu_traffic_bytes():
    """DRAM bytes of one adaptamer_merge_kernel launch on this workload from the committed ncu
    --set full capture of the CURRENT kernel (profiles/r02_ncu_merge_kernel.json); None if no
    capture of this round's kernel is committed."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_merge_kernel.json")
    try:
        d = json.load(open(p))
        tot = 0.0
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            v, u = d[k].split()
            tot += float(v) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[u]
        return tot
    except Exception:
        return None


REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def canonical_md5(lines):
    import hashlib
    h = hashlib.md5()
    for l in sorted(lines):
        h.update(l.encode() + b"\n")
    return h.hexdigest()


def oneview_lines(path):
    """one text line per alignment of a .1aln ('A .. | R | D .. | T .. | X ..'), through the
    reference's own ONEview (SURVEY 8c canonical form)"""
    out = subprocess.run([os.path.join(REF_DIR, "ONEview"), path], stdout=subprocess.PIPE, text=True,
                         check=True).stdout
    recs, cur = [], None
    for line in out.split("\n"):
        if line.startswith("A "):
            if cur is not None:
                recs.append(cur)
            cur = line
        elif cur is not None and line[:1] in ("R", "D", "T", "X") and (len(line) == 1 or line[1] == " "):
            cur += " | " + line
    if cur is not None:
        recs.append(cur)
    return recs


def run_reference(A, B, threads, max_runs, warmup, budget_s=240.0):
    """times the unmodified reference on the pair (A, B): FAtoGDB once (untimed, like the staging of
    the .bps images on the GPU side), then per run GIXmake A, GIXmake B, FastGA -1:ref A B from the
    .1gdb.  Returns a dict with the per-run wall seconds, the phase split and the canonical md5."""
    import re
    from fastga_b200 import formats, synth
    if not os.path.exists(os.path.join(REF_DIR, "FastGA")):
        raise RuntimeError("oracle/_ref/FastGA missing: run __graft_entry__.build() where /root/reference exists")
    env = dict(os.environ)
    env["PATH"] = REF_DIR + os.pathsep + env.get("PATH", "")
    gbp = (sum(len(a) for a in A) + sum(len(b) for b in B)) / 1e9
    times, gix_s, proper_s = [], [], []
    info = {}

    def sh(cmd, wd):
        r = subprocess.run(cmd, cwd=wd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError("reference command failed: %s\n%s" % (" ".join(cmd), r.stdout[-2000:]))
        return r.stdout

    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as wd:
        formats.write_fasta(os.path.join(wd, "A.fasta"), synth.scaffolds_of(A, "sa", 1))
        formats.write_fasta(os.path.join(wd, "B.fasta"), synth.scaffolds_of(B, "sb", 1))
        sh(["FAtoGDB", "A.fasta"], wd)
        sh(["FAtoGDB", "B.fasta"], wd)
        os.remove(os.path.join(wd, "A.fasta"))
        os.remove(os.path.join(wd, "B.fasta"))
        run = 0
        while True:
            for f in os.listdir(wd):
                if ".ktab." in f or f.endswith(".gix") or f.endswith(".1aln"):
                    os.remove(os.path.join(wd, f))
            t0 = time.time()
            sh(["GIXmake", "-T%d" % threads, "-P" + wd, "A"], wd)
            sh(["GIXmake", "-T%d" % threads, "-P" + wd, "B"], wd)
            t1 = time.time()
            log = sh(["FastGA", "-v", "-T%d" % threads, "-P" + wd, "-1:ref", "A", "B"], wd)
            t2 = time.time()
            timed = run >= warmup
            if timed:
                times.append(t2 - t0)
                gix_s.append(t1 - t0)
                proper_s.append(t2 - t1)
            run += 1
            ntimed = len(times)
            if ntimed >= max_runs:
                break
            if timed and (ntimed + 1) * (t2 - t0) > budget_s:
                break
            if not timed and (t2 - t0) > budget_s / 3:      # a single run is already long: count it
                times.append(t2 - t0); gix_s.append(t1 - t0); proper_s.append(t2 - t1)
                break
        log = log.replace("\r", "\n")
        m = re.search(r"Total seeds = ([\d,]+)", log)
        if m:
            info["seeds"] = int(m.group(1).replace(",", ""))
        m = re.search(r"Total hits over \d+bp = (\d+), (\d+) aln's, (\d+) non-redundant", log)
        if m:
            info["hits"], info["alns"], info["kept"] = int(m.group(1)), int(m.group(2)), int(m.group(3))
        lines = oneview_lines(os.path.join(wd, "ref.1aln"))
        info["alignments"] = len(lines)
        info["aln_md5"] = canonical_md5(lines)
    s = float(np.mean(times))
    info.update({"gbp": gbp, "threads": threads, "runs": len(times), "s_per_run": s,
                 "gix_s": float(np.mean(gix_s)), "fastga_proper_s": float(np.mean(proper_s)),
                 "value": gbp / s, "value_proper": gbp / float(np.mean(proper_s))})
    return info


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, alns):
    """Writes the alignment records a caller of the timed path receives, so that two builds can be
    compared record for record on the same seeded pair:
      fields.npy       (n, 9) float64, columns lib.ALN_FIELDS, in the order the path returns them
      trace.npy        float32, the trace bytes of all n records concatenated
      trace_offset.npy (n + 1,) float64, record i's trace is trace[offset[i]:offset[i + 1]]
      rows.npy         (n,) float64, which records of the step these are
    Above DUMP_BYTES in all, a fixed seeded sample of the records is written (rows says which)."""
    n = len(alns)
    tlen = alns.fields[:, 8].astype(np.int64)

    def nbytes(rows):
        return len(rows) * (9 * 8 + 8 + 8) + 8 + 4 * int(tlen[rows].sum())

    rows = np.arange(n)
    k = n
    while nbytes(rows) > DUMP_BYTES:
        k = k * 9 // 10
        rows = np.sort(np.random.default_rng(SEED).permutation(n)[:k])
    toff = np.concatenate([[0], np.cumsum(tlen[rows])])
    trace = np.zeros(int(toff[-1]), dtype=np.float32)
    for j, i in enumerate(rows):
        trace[toff[j]:toff[j + 1]] = alns.trace(i)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "fields.npy"), alns.fields[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "trace.npy"), trace)
    np.save(os.path.join(out_dir, "trace_offset.npy"), toff.astype(np.float64))
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


def workload_text(per_gpu_bp, n):
    return ("synthetic %d Mbp genome (%d contigs) vs 5%%-diverged copy%s, SV breaks every ~%d kbp, seed %d; "
            "FastGA defaults -f10 -c85 -s1000 -l100 -i.7"
            % (per_gpu_bp * n // 1_000_000, NCONTIG * n, " (100 Mbp per GPU x %d GPUs)" % n if n > 1 else "",
               SV_EVERY // 1000, SEED))


def main():
    #  stdout carries exactly ONE line (the JSON): libraries that chat on fd 1 (NCCL prints its
    #  version there) are pointed at stderr for the duration of the run
    sys.stdout.flush()
    real_out = os.dup(1)
    os.dup2(2, 1)
    try:
        line = run()
    finally:
        sys.stdout.flush()
        os.dup2(real_out, 1)
    if line is not None:
        os.write(1, (json.dumps(line) + "\n").encode())


def run():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--per-gpu-bp", type=int, default=PER_GPU_BP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the alignment records of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return None
        threads = min(cores, 32)          # GIXmake refuses -T > 32 (GIXmake.c:1723)
        A, B = workload(args.gpus, args.per_gpu_bp)
        info = run_reference(A, B, threads, max(1, args.steps), min(args.warmup, 1))
        val, ms = info["value"], 1000.0 * info["s_per_run"]
        line = {"impl": "reference", "metric": "Gbp aligned/sec (genome x genome)", "value": val,
                "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32", "data": "synthetic",
                "config": {"workload": workload_text(args.per_gpu_bp, args.gpus),
                           "scope": "from the .1gdb/.bps (FAtoGDB outside the timed region) to the .1aln: "
                                    "GIXmake -T%d x2 + FastGA -T%d, temp on /dev/shm" % (threads, threads),
                           "reference_runs": info["runs"],
                           "phase_s": {"gix_build": info["gix_s"], "fastga_proper": info["fastga_proper_s"]},
                           "value_fastga_proper": info["value_proper"],
                           "alignments": info.get("alignments"), "aln_md5": info.get("aln_md5"),
                           "seeds": info.get("seeds"), "hits": info.get("hits")},
                "cpu_baseline": {"value": val, "unit": "Gbp/s", "cores": threads, "kind": "reference",
                                 "sample": "the whole %.3f Gbp pair (same config as the GPU arm), %d run(s) of %.1f s"
                                           % (info["gbp"], info["runs"], info["s_per_run"])},
                "e2e": {"value": val, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        return line

    import torch
    import torch.distributed as dist
    from fastga_b200 import formats, lib

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    A, B = workload(world, args.per_gpu_bp)
    from fastga_b200 import shard
    #  every rank holds both genomes (2 bits per base: 50 MB per 100 Mbp pair member); the WORK is
    #  sharded -- scanning by contig, index + merge by k-mer prefix range, extension by A-contig
    gA = formats.genome_from_arrays(A)
    gB = formats.genome_from_arrays(B)
    freqA = gA.freq
    total_gbp = (sum(len(a) for a in A) + sum(len(b) for b in B)) / 1e9

    dA = lib.DeviceGenome(gA, want_revcomp=True)
    dB = lib.DeviceGenome(gB)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_step_ms = []

    def timed(fn, steps, keep=None):
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        outs = []
        for i in range(steps):
            outs.append(fn())
            evs[i + 1].record()
        torch.cuda.synchronize()
        ms = torch.tensor([evs[0].elapsed_time(evs[steps])], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if keep is not None:
            keep.extend(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))
        barrier()
        return float(ms.item()) / steps, outs

    if world > 1:
        dev = torch.device("cuda", local_rank)
        step = lambda: shard.align_sharded(dA, dB, freqA, dist, dev)
    else:
        step = lambda: lib.align_resident(dA, dB, freqA)
    for _ in range(args.warmup):
        step()

    sampler = ClockSampler(local_rank)
    sampler.start()
    lib.timings_reset()
    ms_step, outs = timed(step, args.steps, per_step_ms)
    tm = lib.timings_get()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    alns, stats = outs[-1]

    # end to end through the reference-facing call on HOST buffers: the .bps images sit in pinned
    # host memory (what a caller that wants full PCIe rate does), every step copies them to the
    # device and reads the alignment records back
    def pinned(g):
        t = torch.empty(g.bps.size, dtype=torch.uint8).pin_memory()
        t.numpy()[:] = g.bps
        q = formats.Genome(g.clen, t.numpy())
        q._pin = t
        q._freq = g.freq
        return q
    pA, pB = pinned(gA), pinned(gB)
    if world > 1:
        def e2e_step():
            # the sharded call on host buffers: every rank stages both .bps images (H2D), runs its
            # share, reads its records back; the gather of the records to rank 0 is part of the step
            eA = lib.DeviceGenome(pA, want_revcomp=True)
            eB = lib.DeviceGenome(pB)
            out = shard.align_sharded(eA, eB, freqA, dist, dev)
            shard.gather_alignments(out[0], None, dist, dev)
            h2d = pA.bps.size + pB.bps.size
            out[1]["h2d_bytes"] = int(h2d)
            out[1]["d2h_bytes"] = int(out[0].pool.size + out[0].fields.nbytes)
            eA.close()
            eB.close()
            return out
    else:
        e2e_step = lambda: lib.fastga(pA, pB)
    e2e_step()
    ms_e2e, outs2 = timed(e2e_step, args.steps)
    st2 = outs2[-1][1]

    # gather the per-rank record streams on rank 0 (variable length; the path's only collective)
    nrec = len(alns)
    final = alns
    if world > 1:
        merged = shard.gather_alignments(alns, None, dist, torch.device("cuda", local_rank))
        if rank == 0:
            nrec = len(merged)
            final = merged

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, final)
    gpu_md5 = canonical_md5(final.canonical_lines_unsorted())
    steps = args.steps
    # roofline of the seed-merge kernel (the kernel north_star grades): algorithmic bytes on the
    # on-disk widths, B = (N1 + N2)*E + H*R (SURVEY 8d), N1 / N2 = the entries of the two tables the
    # reference's merge walks (both strands of table 1, as in round 1).  This implementation reads only
    # the forward-strand entries of table 1 (reverse entries never seed, FastGA.c:921-928, and the fused
    # path does not build them): `frac_forward_n1` is the same time against that smaller B.
    pb = max(1, (int(max(gA.clen.max(), gB.clen.max())).bit_length() + 7) // 8)
    E1 = 9 + pb + 1
    R = 1 + 2 * (pb + 1)
    #  (N > 1: this rank's slices of the two tables and the seeds ITS merge produced)
    merged_seeds = stats.get("nseeds_merged", stats["nseeds"])
    algo = (stats["nkmers1_fwd"] + stats["nkmers2"]) * E1 + merged_seeds * R
    algo_ondisk = (stats.get("nkmers1", 2 * stats["nkmers1_fwd"]) + stats["nkmers2"]) * E1 + merged_seeds * R
    merge_ms = tm["merge_ms"] / max(1, tm["merge_launches"])
    # byte passes of the seed sort: key = lcp(6) drem(6) anti band jcont icont strand (api.cu:fgb_seeds_find)
    abits = int(gA.clen.max() + gB.clen.max()).bit_length()
    kb = 12 + abits + max(1, abits - 6) + max(1, (gB.ncontig - 1).bit_length()) + max(1, (gA.ncontig - 1).bit_length()) + 1
    seed_passes = (kb - 6 + 7) // 8          # 8-bit digits from bit 6 up (the lcp field never breaks a tie)
    peak, peak_src = measured_peak_hbm()
    ach = algo_ondisk / (merge_ms * 1e-3) / 1e9 if merge_ms > 0 else 0.0
    dev_ms = {k: v / steps for k, v in tm.items() if k.endswith("_ms")}
    # records this rank's k-mer sorts handled per step: table 1 forward-only + its share of table 2
    nk_sorted = stats["nkmers1_fwd"] + stats["nkmers2"]
    step_ms = sorted(per_step_ms)

    line = {"metric": "Gbp aligned/sec (genome x genome)", "value": total_gbp / (ms_step / 1000.0),
            "unit": "Gbp/s", "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic",
            "config": {"workload": workload_text(args.per_gpu_bp, world) +
                                   "; k-mer tables and seed sets are larger than L2 (no flush needed)",
                       "sharding": ("k-mer space: every rank scans its contigs, k-mer records go to the owner of "
                                    "their prefix range and seeds to the owner of their A-contig (two NCCL "
                                    "all-to-alls of 16-byte records), nothing replicated; counts below are rank 0's share")
                                   if world > 1 else "single GPU",
                       "alignments": nrec, "aln_md5": gpu_md5,
                       "seeds": stats["nseeds"], "kmers": [stats.get("nkmers1"), stats["nkmers2"]],
                       "kmers1_forward": stats["nkmers1_fwd"],
                       "hits": stats["nhits"], "la_calls": stats["nla"], "waves": stats["nwaves"],
                       "wave_cells": stats["ncells"], "stage_ms": dev_ms,
                       "step_ms_min_med_max": [step_ms[0], step_ms[len(step_ms) // 2], step_ms[-1]],
                       "triples": [stats["nseg"], stats["nwork"]],
                       "host_wall_us": {k: stats.get(k) for k in ("us_gix", "us_seeds", "us_extend", "us_filter")},
                       "extend_cycles": {k: stats[k] for k in ("warp_cycles", "wave_cycles", "extract_cycles", "slow_cycles",
                                                                "slow_waves", "paired_waves", "pairings")}},
            "roofline": {"bound": "hbm", "kernel": "adaptamer_merge_kernel", "achieved": ach, "peak": peak,
                         "unit": "GB/s", "frac": ach / peak,
                         "traffic": ncu_traffic_bytes() if (world == 1 and args.per_gpu_bp == PER_GPU_BP) else None,
                         "peak_source": peak_src,
                         "algorithmic_bytes": algo_ondisk, "kernel_ms": merge_ms,
                         "algorithmic_bytes_forward_n1": algo,
                         "frac_forward_n1": (algo / (merge_ms * 1e-3) / 1e9 / peak) if merge_ms > 0 else 0.0},
            # the other HBM-side stages against the same measured peak (16-byte device records;
            # k-mer sort = 2 Onesweep passes + 1 shared-memory bucket pass, seed sort = ceil(keybits/8) passes)
            "other_kernels": other_kernels(stats, dev_ms, peak, seed_passes, nk_sorted),
            "extend_kernel": {"ms": tm["extend_ms"] / steps, "launches_per_step": tm["extend_launches"] / steps,
                              "cell_updates_per_s":
                              stats["ncells"] / max(1e-9, tm["extend_ms"] / steps / 1000.0)},
            "clocks": sampler.summary(),
            "e2e": {"value": total_gbp / (ms_e2e / 1000.0), "unit": "Gbp/s",
                    "h2d_bytes_per_step": st2["h2d_bytes"], "d2h_bytes_per_step": st2["d2h_bytes"],
                    "ms_per_step": ms_e2e},
            "gpu_launches": tm["launches"]}

    if not args.no_cpu_baseline and world == 1:
        # the reference on the SAME pair (one run, ~10-20 s at -T32): baseline and parity in one go
        try:
            threads = min(cores, 32)
            info = run_reference(A, B, threads, 1, 0)
            line["cpu_baseline"] = {"value": info["value"], "unit": "Gbp/s", "cores": threads, "kind": "reference",
                                    "sample": "the whole %.3f Gbp pair (same config): GIXmake x2 %.1f s + FastGA "
                                              "-T%d %.1f s from the .1gdb, 1 run"
                                              % (info["gbp"], info["gix_s"], threads, info["fastga_proper_s"]),
                                    "value_fastga_proper": info["value_proper"]}
            line["parity"] = {"pair": "the bench pair itself", "reference_md5": info["aln_md5"], "gpu_md5": gpu_md5,
                              "equal": info["aln_md5"] == gpu_md5,
                              "reference_counts": {k: info.get(k) for k in ("seeds", "hits", "alns", "kept")},
                              "gpu_counts": {"seeds": stats["nseeds"], "hits": stats["nhits"],
                                             "alns": final.nraw, "kept": nrec}}
        except Exception as ex:      # the reference arm must never sink the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "Gbp/s", "cores": cores, "kind": "reference",
                                    "sample": "failed: %s" % str(ex)[:200]}
    if world > 1:
        dist.destroy_process_group()
    return line


if __name__ == "__main__":
    main()
