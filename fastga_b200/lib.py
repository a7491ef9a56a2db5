"""ctypes binding of the C-ABI in include/fastga_b200.h (host buffers in, host buffers out)."""
import ctypes as C

import numpy as np

from . import load_library

c_void_p, c_int, c_ll = C.c_void_p, C.c_int, C.c_longlong

ERRORS = {-1: "CUDA runtime error", -2: "bad argument", -3: "input exceeds a device-layout limit",
          -4: "device arena overflow"}


class FgbError(RuntimeError):
    pass


def _check(rc, what):
    if rc != 0:
        raise FgbError("%s failed: %s (%d)" % (what, ERRORS.get(rc, "?"), rc))


class Timings(C.Structure):
    _fields_ = [(n, C.c_float) for n in
                ("h2d_ms", "stage_ms", "scan_ms", "ksort_ms", "index_ms", "merge_ms", "ssort_ms",
                 "triples_ms", "extend_ms", "d2h_ms", "filter_ms")] + \
               [("merge_launches", C.c_int), ("extend_launches", C.c_int), ("launches", C.c_int)]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


def _ptr(a):
    return a.ctypes.data_as(c_void_p)


def timings_reset():
    load_library().fgb_timings_reset()


def timings_get():
    t = Timings()
    load_library().fgb_timings_get(C.byref(t))
    return t.asdict()


def device_ready():
    return bool(load_library().fgb_device_ready())


class DeviceGenome:
    """fgb_genome handle: the staged 2-bit contigs of one genome in HBM."""

    def __init__(self, genome, want_revcomp=False, stream=None):
        L = load_library()
        self.genome = genome
        self.h = c_void_p()
        L.fgb_genome_create.argtypes = [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_int,
                                        C.POINTER(c_void_p), c_void_p]
        _check(L.fgb_genome_create(_ptr(genome.bps), genome.bps.size, genome.ncontig,
                                   _ptr(genome.clen), _ptr(genome.boff), int(want_revcomp),
                                   C.byref(self.h), stream), "fgb_genome_create")
        self.perm = np.zeros(genome.ncontig, dtype=np.int32)
        L.fgb_genome_perm.argtypes = [c_void_p, c_void_p]
        L.fgb_genome_perm(self.h, _ptr(self.perm))
        self.crank = np.empty_like(self.perm)
        self.crank[self.perm] = np.arange(genome.ncontig, dtype=np.int32)

    def download(self, rev=False):
        L = load_library()
        L.fgb_genome_words.restype = c_ll
        L.fgb_genome_words.argtypes = [c_void_p]
        n = L.fgb_genome_words(self.h)
        words = np.zeros(n, dtype=np.uint64)
        woff = np.zeros(self.genome.ncontig + 1, dtype=np.int64)
        L.fgb_genome_download.argtypes = [c_void_p, c_int, c_void_p, c_void_p]
        _check(L.fgb_genome_download(self.h, int(rev), _ptr(words), _ptr(woff)), "fgb_genome_download")
        return words, woff

    def close(self):
        if self.h:
            L = load_library()
            L.fgb_genome_free.argtypes = [c_void_p]
            L.fgb_genome_free(self.h)
            self.h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceGix:
    """fgb_gix handle: sorted 128-bit k-mer records + 2^24 prefix index in HBM."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def build(cls, dgenome, stream=None):
        L = load_library()
        h = c_void_p()
        L.fgb_gix_build.argtypes = [c_void_p, C.POINTER(c_void_p), c_void_p]
        _check(L.fgb_gix_build(dgenome.h, C.byref(h), stream), "fgb_gix_build")
        return cls(h)

    @classmethod
    def build_forward(cls, dgenome, stream=None):
        """forward-strand entries only (the adaptamer side of a merge)"""
        L = load_library()
        h = c_void_p()
        L.fgb_gix_build_forward.argtypes = [c_void_p, C.POINTER(c_void_p), c_void_p]
        _check(L.fgb_gix_build_forward(dgenome.h, C.byref(h), stream), "fgb_gix_build_forward")
        return cls(h)

    @classmethod
    def import_ktab(cls, gixfile, stream=None):
        L = load_library()
        h = c_void_p()
        L.fgb_gix_import_ktab.argtypes = [c_void_p, c_ll, c_int, c_int, c_void_p, c_int,
                                          C.POINTER(c_void_p), c_void_p]
        ent = np.ascontiguousarray(gixfile.entries)
        idx = np.ascontiguousarray(gixfile.index, dtype=np.int64)
        _check(L.fgb_gix_import_ktab(_ptr(ent), gixfile.n, gixfile.post_bytes, gixfile.cont_bytes,
                                     _ptr(idx), gixfile.ncontig, C.byref(h), stream),
               "fgb_gix_import_ktab")
        return cls(h)

    @property
    def n(self):
        L = load_library()
        L.fgb_gix_size.restype = c_ll
        L.fgb_gix_size.argtypes = [c_void_p]
        return L.fgb_gix_size(self.h)

    @property
    def post_bytes(self):
        L = load_library()
        L.fgb_gix_post_bytes.argtypes = [c_void_p]
        return L.fgb_gix_post_bytes(self.h)

    @property
    def cont_bytes(self):
        L = load_library()
        L.fgb_gix_cont_bytes.argtypes = [c_void_p]
        return L.fgb_gix_cont_bytes(self.h)

    def download(self, want_index=True):
        L = load_library()
        n = self.n
        tab = np.zeros((n, 2), dtype=np.uint64)
        pstart = np.zeros((1 << 24) + 1, dtype=np.uint32) if want_index else None
        buck = np.zeros(1024, dtype=np.uint64)
        L.fgb_gix_download.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
        _check(L.fgb_gix_download(self.h, _ptr(tab), _ptr(pstart) if want_index else None, _ptr(buck)),
               "fgb_gix_download")
        return tab, pstart, buck

    def export_ktab(self, part_first, stream=None):
        L = load_library()
        E = 9 + self.post_bytes + self.cont_bytes
        out = np.zeros(self.n * E, dtype=np.uint8)
        pf = np.ascontiguousarray(part_first, dtype=np.int64)
        L.fgb_gix_export_ktab.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_void_p]
        _check(L.fgb_gix_export_ktab(self.h, _ptr(pf), len(pf), _ptr(out), stream), "fgb_gix_export_ktab")
        return out

    def close(self):
        if self.h:
            L = load_library()
            L.fgb_gix_free.argtypes = [c_void_p]
            L.fgb_gix_free(self.h)
            self.h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceSeeds:
    """fgb_seeds handle: sorted adaptive-seed records in HBM."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def find(cls, gix1, gix2, amxpos, bmxpos, freq=10, stream=None):
        L = load_library()
        h = c_void_p()
        L.fgb_seeds_find.argtypes = [c_void_p, c_void_p, c_ll, c_ll, c_int, C.POINTER(c_void_p), c_void_p]
        _check(L.fgb_seeds_find(gix1.h, gix2.h, amxpos, bmxpos, freq, C.byref(h), stream), "fgb_seeds_find")
        return cls(h)

    @property
    def n(self):
        L = load_library()
        L.fgb_seeds_size.restype = c_ll
        L.fgb_seeds_size.argtypes = [c_void_p]
        return L.fgb_seeds_size(self.h)

    @property
    def sumlen(self):
        L = load_library()
        L.fgb_seeds_sumlen.restype = c_ll
        L.fgb_seeds_sumlen.argtypes = [c_void_p]
        return L.fgb_seeds_sumlen(self.h)

    @property
    def layout(self):
        L = load_library()
        bits = (c_int * 4)()
        L.fgb_seeds_layout.argtypes = [c_void_p, c_void_p]
        L.fgb_seeds_layout(self.h, bits)
        return tuple(bits)

    def download(self):
        L = load_library()
        rec = np.zeros((self.n, 2), dtype=np.uint64)
        L.fgb_seeds_download.argtypes = [c_void_p, c_void_p]
        _check(L.fgb_seeds_download(self.h, _ptr(rec)), "fgb_seeds_download")
        return rec

    def close(self):
        if self.h:
            L = load_library()
            L.fgb_seeds_free.argtypes = [c_void_p]
            L.fgb_seeds_free(self.h)
            self.h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sort128_host(recs, byte_lo, byte_hi, stream=None):
    """In-place device sort of an (n,2) uint64 array of 128-bit records on key bytes [lo,hi)."""
    L = load_library()
    assert recs.dtype == np.uint64 and recs.flags.c_contiguous and recs.shape[1] == 2
    L.fgb_sort128_host.argtypes = [c_void_p, c_ll, c_int, c_int, c_void_p]
    _check(L.fgb_sort128_host(_ptr(recs), recs.shape[0], byte_lo, byte_hi, stream), "fgb_sort128_host")
    return recs


OVL_DT = np.dtype([("triple", "i4"), ("seq", "i4"), ("pairkey", "i4"), ("abpos", "i4"), ("bbpos", "i4"),
                   ("aepos", "i4"), ("bepos", "i4"), ("diffs", "i4"), ("tlen", "i4"), ("toff", "i8")])


def align_spec(ave_corr, freq):
    """(tables[65536] int16, ave_path) of New_Align_Spec (align.c:222-268)"""
    L = load_library()
    tables = np.zeros(65536, dtype=np.int16)
    ave = c_int()
    f = np.ascontiguousarray(freq, dtype=np.float32)
    L.fgb_align_spec.argtypes = [C.c_double, c_void_p, c_void_p, C.POINTER(c_int)]
    _check(L.fgb_align_spec(float(ave_corr), _ptr(f), _ptr(tables), C.byref(ave)), "fgb_align_spec")
    return tables, ave.value


class DeviceOverlaps:
    """fgb_overlaps handle: raw local alignments (before the redundancy filter), host resident."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def extend(cls, seeds, dgenomeA, dgenomeB, freq, chain_break=2000, chain_min=170, align_min=100,
               align_rate=0.3, tspace=100, stream=None):
        L = load_library()
        tables, ave = align_spec(1.0 - align_rate, freq)
        h = c_void_p()
        L.fgb_extend.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, C.c_double, c_void_p,
                                 c_int, c_int, C.POINTER(c_void_p), c_void_p]
        _check(L.fgb_extend(seeds.h, dgenomeA.h, dgenomeB.h, chain_break, chain_min, align_min,
                            float(align_rate), _ptr(tables), ave, tspace, C.byref(h), stream), "fgb_extend")
        return cls(h)

    def counters(self):
        L = load_library()
        out = (C.c_ulonglong * 16)()
        L.fgb_overlaps_counters.argtypes = [c_void_p, c_void_p]
        L.fgb_overlaps_counters(self.h, out)
        v = list(out)
        return {"hits": v[0], "la_calls": v[1], "waves": v[2], "cells": v[3], "nseg": v[5], "nwork": v[6],
                "warp_cycles": v[8], "wave_cycles": v[9], "extract_cycles": v[10], "paired_waves": v[11], "pairings": v[12],
                "front_wait": v[4], "front_total": v[7], "back_wait": v[13],
                "max_warp_cycles": v[14],
                "slowest_warp": {"cycles": (v[15] >> 40) << 12, "waves": (v[15] >> 16) & 0xffffff, "la_calls": v[15] & 0xffff}}

    def records(self):
        """(structured array sorted in reference discovery order, trace byte pool)"""
        L = load_library()
        L.fgb_overlaps_bytes.restype = c_ll
        L.fgb_overlaps_bytes.argtypes = [c_void_p]
        L.fgb_overlaps_data.restype = c_void_p
        L.fgb_overlaps_data.argtypes = [c_void_p]
        nb = L.fgb_overlaps_bytes(self.h)
        if nb == 0:
            return np.zeros(0, dtype=OVL_DT), np.zeros(0, dtype=np.uint8)
        buf = np.ctypeslib.as_array(C.cast(L.fgb_overlaps_data(self.h), C.POINTER(C.c_uint8)), shape=(nb,)).copy()
        recs = []
        off = 0
        while off < nb:
            h = np.frombuffer(buf[off:off + 40].tobytes(), dtype=np.int32)
            recs.append((h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], off + 40))
            off += 40 + ((int(h[8]) + 7) & ~7)
        arr = np.array(recs, dtype=OVL_DT)
        order = np.lexsort((arr["seq"], arr["triple"]))
        return arr[order], buf

    def close(self):
        if self.h:
            L = load_library()
            L.fgb_overlaps_free.argtypes = [c_void_p]
            L.fgb_overlaps_free(self.h)
            self.h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


ALN_FIELDS = ("comp", "aread", "bread", "abpos", "bbpos", "aepos", "bepos", "diffs", "tlen")


class Alignments:
    """Final local alignments (after the redundancy filter, in .1aln order)."""

    def __init__(self, fields, toff, pool, nraw):
        self.fields = fields        # (n, 9) int32, columns ALN_FIELDS
        self.toff = toff
        self.pool = pool
        self.nraw = nraw

    def __len__(self):
        return self.fields.shape[0]

    def trace(self, i):
        return self.pool[int(self.toff[i]):int(self.toff[i]) + int(self.fields[i, 8])]

    def canonical_lines(self):
        """One text line per alignment in ONEview's form 'A .. | R | D .. | T .. | X ..', sorted."""
        return sorted(self.canonical_lines_unsorted())

    def canonical_lines_unsorted(self):
        out = []
        for i in range(len(self)):
            comp, ar, br, ab, bb, ae, be, df, tl = (int(x) for x in self.fields[i])
            t = self.trace(i)
            line = "A %d %d %d %d %d %d" % (ar, ab, ae, br, bb, be)
            if comp:
                line += " | R"
            line += " | D %d" % df
            line += " | T %d" % (tl // 2) + "".join(" %d" % v for v in t[1::2])
            line += " | X %d" % (tl // 2) + "".join(" %d" % v for v in t[0::2])
            out.append(line)
        return out


def filter_overlaps(ovl_handle, perm1, perm2, jc_bits, ic_bits, do_filter=True):
    L = load_library()
    h = c_void_p()
    p1 = np.ascontiguousarray(perm1, dtype=np.int32)
    p2 = np.ascontiguousarray(perm2, dtype=np.int32)
    L.fgb_filter.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, C.POINTER(c_void_p)]
    _check(L.fgb_filter(ovl_handle, _ptr(p1), _ptr(p2), jc_bits, ic_bits, int(do_filter), C.byref(h)),
           "fgb_filter")
    return _alns_out(h)


def overlaps_from_buffer(buf):
    L = load_library()
    h = c_void_p()
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    L.fgb_overlaps_from_buffer.argtypes = [c_void_p, c_ll, C.POINTER(c_void_p)]
    _check(L.fgb_overlaps_from_buffer(_ptr(buf), buf.size, C.byref(h)), "fgb_overlaps_from_buffer")
    return DeviceOverlaps(h)


class RunStats(C.Structure):
    _fields_ = [(n, c_ll) for n in ("nkmers1", "nkmers2", "nseeds", "sumlen", "nhits", "nla", "nwaves",
                                    "ncells", "nraw", "h2d_bytes", "d2h_bytes", "nseg", "nwork", "warp_cycles",
                                    "wave_cycles", "extract_cycles", "us_gix", "us_seeds", "us_extend", "us_filter",
                                    "nkmers1_fwd", "slow_cycles", "slow_waves", "paired_waves", "pairings")]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


DEFAULTS = dict(freq=10, chain_break=2000, chain_min=170, align_min=100, align_rate=0.3)


def _alns_out(h):
    L = load_library()
    for f in ("fgb_alns_count", "fgb_alns_raw_count", "fgb_alns_pool_bytes"):
        getattr(L, f).restype = c_ll
        getattr(L, f).argtypes = [c_void_p]
    n, nraw, pb = L.fgb_alns_count(h), L.fgb_alns_raw_count(h), L.fgb_alns_pool_bytes(h)
    fields = np.zeros((n, 9), dtype=np.int32)
    toff = np.zeros(n, dtype=np.int64)
    pool = np.zeros(max(pb, 1), dtype=np.uint8)
    L.fgb_alns_get.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
    _check(L.fgb_alns_get(h, _ptr(fields), _ptr(toff), _ptr(pool)), "fgb_alns_get")
    L.fgb_alns_free.argtypes = [c_void_p]
    L.fgb_alns_free(h)
    return Alignments(fields, toff, pool, nraw)


def align_resident(dA, dB, freqA, stream=None, **kw):
    """Whole path from device-resident genomes: returns (Alignments, stats dict)"""
    p = dict(DEFAULTS)
    p.update(kw)
    L = load_library()
    h = c_void_p()
    st = RunStats()
    f = np.ascontiguousarray(freqA, dtype=np.float32)
    L.fgb_align_resident.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, C.c_double,
                                     C.POINTER(c_void_p), C.POINTER(RunStats), c_void_p]
    _check(L.fgb_align_resident(dA.h, dB.h, _ptr(f), p["freq"], p["chain_break"], p["chain_min"],
                                p["align_min"], float(p["align_rate"]), C.byref(h), C.byref(st), stream),
           "fgb_align_resident")
    return _alns_out(h), st.asdict()


def fastga_self(g, stream=None, **kw):
    """SELF mode, `FastGA A` with one source (formats.Genome) -> (Alignments, stats)"""
    p = dict(DEFAULTS)
    p.update(kw)
    L = load_library()
    h = c_void_p()
    st = RunStats()
    f = np.ascontiguousarray(g.freq, dtype=np.float32)
    L.fgb_fastga_self.argtypes = [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, C.c_double,
                                  C.POINTER(c_void_p), C.POINTER(RunStats), c_void_p]
    _check(L.fgb_fastga_self(_ptr(g.bps), g.bps.size, g.ncontig, _ptr(g.clen), _ptr(g.boff), _ptr(f),
                             p["freq"], p["chain_break"], p["chain_min"], p["align_min"], float(p["align_rate"]),
                             C.byref(h), C.byref(st), stream), "fgb_fastga_self")
    return _alns_out(h), st.asdict()


def fastga(gA, gB, stream=None, **kw):
    """The reference-facing call on host buffers (formats.Genome x2) -> (Alignments, stats)"""
    p = dict(DEFAULTS)
    p.update(kw)
    L = load_library()
    h = c_void_p()
    st = RunStats()
    f = np.ascontiguousarray(gA.freq, dtype=np.float32)
    L.fgb_fastga.argtypes = [c_void_p, c_ll, c_int, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_ll, c_int, c_void_p, c_void_p,
                             c_int, c_int, c_int, c_int, C.c_double,
                             C.POINTER(c_void_p), C.POINTER(RunStats), c_void_p]
    _check(L.fgb_fastga(_ptr(gA.bps), gA.bps.size, gA.ncontig, _ptr(gA.clen), _ptr(gA.boff), _ptr(f),
                        _ptr(gB.bps), gB.bps.size, gB.ncontig, _ptr(gB.clen), _ptr(gB.boff),
                        p["freq"], p["chain_break"], p["chain_min"], p["align_min"], float(p["align_rate"]),
                        C.byref(h), C.byref(st), stream), "fgb_fastga")
    return _alns_out(h), st.asdict()


def compute_trace_pts(dA, dB, alns, tspace=100, stream=None):
    """Compute_Trace_PTS for every alignment of `alns` (an Alignments): returns (soff, script, diffs) --
    script[soff[i]:soff[i+1]] is the edit script the reference leaves in path->trace, diffs[i] its
    path->diffs (-1: trace points inconsistent with the sequences).  dB needs want_revcomp=True when
    strand-C records are present."""
    L = load_library()
    h = c_void_p()
    fields = np.ascontiguousarray(alns.fields, dtype=np.int32)
    toff = np.ascontiguousarray(alns.toff, dtype=np.int64)
    pool = np.ascontiguousarray(alns.pool, dtype=np.uint8)
    L.fgb_compute_trace_pts.argtypes = [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_void_p, c_int,
                                        C.POINTER(c_void_p), c_void_p]
    _check(L.fgb_compute_trace_pts(dA.h, dB.h, len(alns), _ptr(fields), _ptr(toff), _ptr(pool), tspace,
                                   C.byref(h), stream), "fgb_compute_trace_pts")
    L.fgb_scripts_total.restype = c_ll
    L.fgb_scripts_total.argtypes = [c_void_p]
    n, tot = len(alns), L.fgb_scripts_total(h)
    soff = np.zeros(n + 1, dtype=np.int64)
    script = np.zeros(max(tot, 1), dtype=np.int32)
    diffs = np.zeros(max(n, 1), dtype=np.int32)
    L.fgb_scripts_get.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
    _check(L.fgb_scripts_get(h, _ptr(soff), _ptr(script), _ptr(diffs)), "fgb_scripts_get")
    L.fgb_scripts_free.argtypes = [c_void_p]
    L.fgb_scripts_free(h)
    return soff, script[:tot], diffs[:n]


# ---- building blocks of the k-mer-space sharded path (several GPUs; orchestrated by shard.py) ----

def hit_groups_host(hrange, tinfo, hits, bands=1, slack=1000, gap=-1):
    """The host rule of fgb_extend that cuts every work triple's chain list into independently extended
    groups (no device needed).  hrange: (nwork,2) (first hit, count | bit 31); tinfo: (nwork,2) (key,
    band); hits: (nhits,2) (alow, ahgh).  Returns (items (n,4): triple, first hit, hits, number of the
    first hit in its triple -- in launch order; next (n,2): first hit of the next group or INT64_MAX)."""
    L = load_library()
    hr = np.ascontiguousarray(hrange, dtype=np.uint32).reshape(-1, 2)
    ti = np.ascontiguousarray(tinfo, dtype=np.int32).reshape(-1, 2)
    hh = np.ascontiguousarray(hits, dtype=np.int64).reshape(-1, 2)
    cap = len(hh) + len(hr) + 1
    items = np.zeros((cap, 4), dtype=np.uint32)
    nxt = np.zeros((cap, 2), dtype=np.int64)
    L.fgb_hit_groups_host.restype = c_ll
    L.fgb_hit_groups_host.argtypes = [c_int, c_void_p, c_void_p, c_void_p, c_ll, c_int, c_ll, c_ll, c_void_p, c_void_p]
    n = L.fgb_hit_groups_host(len(hr), _ptr(hr), _ptr(ti), _ptr(hh), len(hh), bands, slack, gap, _ptr(items), _ptr(nxt))
    return items[:n].copy(), nxt[:n].copy()


def device_free(ptr):
    L = load_library()
    L.fgb_device_free.argtypes = [c_void_p]
    L.fgb_device_free(c_void_p(ptr))


def kmers_scan(dgenome, mask, fwd_only, stream=None):
    """unsorted k-mer records of the contigs with mask[c] != 0 -> (device pointer, n); free with device_free"""
    L = load_library()
    ptr, n = c_void_p(), c_ll()
    m = np.ascontiguousarray(mask, dtype=np.uint8)
    L.fgb_kmers_scan.argtypes = [c_void_p, c_void_p, c_int, C.POINTER(c_void_p), C.POINTER(c_ll), c_void_p]
    _check(L.fgb_kmers_scan(dgenome.h, _ptr(m), int(fwd_only), C.byref(ptr), C.byref(n), stream), "fgb_kmers_scan")
    return ptr.value, n.value


def records_group_by_owner(src_ptr, n, owner256, world, dst_ptr, stream=None):
    """groups n k-mer records by the rank owning their first four bases (owner256[top byte]) into dst;
    returns bounds[world+1]"""
    L = load_library()
    bounds = np.zeros(world + 1, dtype=np.int64)
    own = np.ascontiguousarray(owner256, dtype=np.int32)
    assert own.shape == (256,)
    L.fgb_records_group_by_owner.argtypes = [c_void_p, c_ll, c_void_p, c_int, c_void_p, c_void_p, c_void_p]
    _check(L.fgb_records_group_by_owner(c_void_p(src_ptr), n, _ptr(own), world, c_void_p(dst_ptr), _ptr(bounds),
                                        stream), "fgb_records_group_by_owner")
    return bounds


def gix_from_records(ptr, n, plo, phi, fwd_only, post_bytes, cont_bytes, ncontig, stream=None):
    L = load_library()
    h = c_void_p()
    L.fgb_gix_from_records.argtypes = [c_void_p, c_ll, C.c_uint, C.c_uint, c_int, c_int, c_int, c_int,
                                       C.POINTER(c_void_p), c_void_p]
    _check(L.fgb_gix_from_records(c_void_p(ptr), n, plo, phi, int(fwd_only), post_bytes, cont_bytes, ncontig,
                                  C.byref(h), stream), "fgb_gix_from_records")
    return DeviceGix(h)


def seeds_merge(gix1, gix2, amxpos, bmxpos, freq=10, stream=None):
    """unsorted seeds of gix1 x gix2 -> (device pointer, n, bits[4], sumlen, n1_merged); free with device_free"""
    L = load_library()
    ptr, n = c_void_p(), c_ll()
    bits = (c_int * 4)()
    info = (c_ll * 2)()
    L.fgb_seeds_merge.argtypes = [c_void_p, c_void_p, c_ll, c_ll, c_int, C.POINTER(c_void_p), C.POINTER(c_ll),
                                  c_void_p, c_void_p, c_void_p]
    _check(L.fgb_seeds_merge(gix1.h, gix2.h, amxpos, bmxpos, freq, C.byref(ptr), C.byref(n), bits, info, stream),
           "fgb_seeds_merge")
    return ptr.value, n.value, tuple(bits), info[0], info[1]


def seeds_group_by_owner(src_ptr, n, bits, owner_by_rank, world, dst_ptr, stream=None):
    L = load_library()
    bounds = np.zeros(world + 1, dtype=np.int64)
    b = (c_int * 4)(*bits)
    ow = np.ascontiguousarray(owner_by_rank, dtype=np.int32)
    L.fgb_seeds_group_by_owner.argtypes = [c_void_p, c_ll, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
    _check(L.fgb_seeds_group_by_owner(c_void_p(src_ptr), n, b, _ptr(ow), len(ow), world, c_void_p(dst_ptr),
                                      _ptr(bounds), stream), "fgb_seeds_group_by_owner")
    return bounds


def seeds_from_records(ptr, n, bits, amxpos, bmxpos, sumlen=0, stream=None):
    L = load_library()
    h = c_void_p()
    b = (c_int * 4)(*bits)
    L.fgb_seeds_from_records.argtypes = [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_ll, C.POINTER(c_void_p), c_void_p]
    _check(L.fgb_seeds_from_records(c_void_p(ptr), n, b, amxpos, bmxpos, sumlen, C.byref(h), stream),
           "fgb_seeds_from_records")
    return DeviceSeeds(h)


def local_alignments(dA, dB, jobs, freq, align_rate=0.3, tspace=100, stream=None):
    """Local_Alignment (align.h) for a batch: jobs (n,8) int32 = (A contig, B contig, comp, low, hgh, anti,
    lbord, hbord).  Returns (paths (n,7) int32: abpos bbpos aepos bepos diffs tlen status, toff, traces)."""
    L = load_library()
    jobs = np.ascontiguousarray(jobs, dtype=np.int32).reshape(-1, 8)
    n = jobs.shape[0]
    tables, ave = align_spec(1.0 - align_rate, freq)
    paths = np.zeros((max(n, 1), 7), dtype=np.int32)
    toff = np.zeros(max(n, 1), dtype=np.int64)
    cap = 1 << 20
    L.fgb_local_alignments.argtypes = [c_void_p, c_void_p, c_ll, c_void_p, c_void_p, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_ll, C.POINTER(c_ll), c_void_p]
    while True:
        traces = np.zeros(cap, dtype=np.uint8)
        used = c_ll()
        rc = L.fgb_local_alignments(dA.h, dB.h, n, _ptr(jobs), _ptr(tables), ave, tspace, _ptr(paths), _ptr(toff),
                                    _ptr(traces), cap, C.byref(used), stream)
        if rc == -4 and used.value > cap:
            cap = used.value + 1024
            continue
        _check(rc, "fgb_local_alignments")
        return paths[:n], toff[:n], traces[:used.value]
