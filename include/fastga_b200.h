/* fastga_b200.h -- C-ABI of libfastga_b200.so, the B200 (sm_100a) implementation of FastGA's
 * seed-and-extend hot path.  Plain pointers and sizes only; every function returns 0 (FGB_OK) or a
 * negative FGB_ERR_* code, and prints CUDA errors to stderr.  There is no CPU fallback: without a
 * CUDA device every compute entry point fails.
 *
 * FASTGA (the reference) has no plugin/FFI layer: its seams are ordinary C calls between
 * FastGA.c / GIXmake.c and MSDsort.c / RSDsort.c / align.c, plus the files.  Each entry point
 * below names the reference interface it replaces (file:line in thegenemyers/FASTGA).  The
 * reference-side stubs a maintainer would add are in INTEGRATION.md.
 *
 * `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream); all work of a
 * call is issued on it and the call returns after the stream has drained.
 *
 * Threading contract: ONE calling thread and ONE device per process at a time (what `FastGA`, one
 * process, and `torchrun`, one process per GPU, do).  The library keeps process-wide state -- a cache
 * of device blocks without a device id, per-stage timers, a pinned staging buffer, kernel attributes
 * set on first use -- and does not lock around it.
 */
#ifndef FASTGA_B200_H
#define FASTGA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FGB_OK            0
#define FGB_ERR_CUDA     -1   /* a CUDA runtime call failed                                     */
#define FGB_ERR_ARG      -2   /* bad argument                                                   */
#define FGB_ERR_LIMIT    -3   /* input exceeds a device-layout limit (see DESIGN.md "Limits")   */
#define FGB_ERR_OVERFLOW -4   /* a device arena overflowed even after the retry ladder          */

typedef struct fgb_genome   fgb_genome;    /* staged 2-bit contigs of one genome in HBM        */
typedef struct fgb_gix      fgb_gix;       /* sorted k-mer table + 2^24 prefix index in HBM    */
typedef struct fgb_seeds    fgb_seeds;     /* sorted adaptive-seed records in HBM              */
typedef struct fgb_overlaps fgb_overlaps;  /* raw local alignments, host resident              */
typedef struct fgb_alns     fgb_alns;      /* final alignments in .1aln order, host resident   */
typedef struct fgb_scripts  fgb_scripts;   /* explicit edit scripts of alignments, host resident */

typedef struct
{ long long nkmers1, nkmers2, nseeds, sumlen, nhits, nla, nwaves, ncells, nraw, h2d_bytes, d2h_bytes,
            nseg, nwork, warp_cycles, wave_cycles, extract_cycles,
            us_gix, us_seeds, us_extend, us_filter,      /* host wall microseconds per phase */
            nkmers1_fwd,                                 /* forward-strand entries of table 1 (what the merge reads) */
            slow_cycles, slow_waves,                     /* the extension warp that finished last: its cycles and waves */
            paired_waves, pairings;                      /* waves run by front/back warp pairs, passes handed to a pair */
} fgb_run_stats;

typedef struct
{ float h2d_ms, stage_ms, scan_ms, ksort_ms, index_ms, merge_ms, ssort_ms, triples_ms, extend_ms,
        d2h_ms, filter_ms;
  int   merge_launches, extend_launches, launches;
} fgb_timings;

/* ---- the whole path -----------------------------------------------------------------------
 * Replaces, inside `FastGA -1:<out> A B`, everything between Read_GDB and la_merge
 * (FastGA.c:4927-5205): GIXmake's k_sort/distribute for both genomes (GIXmake.c:616-716,
 * :1300-1596), adaptamer_merge (FastGA.c:2281), pair_sort_search (FastGA.c:4135) incl.
 * rmsd_sort, search_seeds/align_contigs and Local_Alignment, and la_sort's order.
 * Inputs are the GDB as Read_GDB leaves it: the .bps image, per contig clen and boff
 * (GDB.h:28-34) and the base frequencies gdb1->freq (GDB.h:72).  Defaults of the reference CLI:
 * freq 10, chain_break 2000, chain_min 170, align_min 100, align_rate .3 (FastGA.c:4451-4459). */
int fgb_fastga(const unsigned char *bpsA, long long bps_bytesA, int ncontigA, const long long *clenA,
               const long long *boffA, const float *freqA,
               const unsigned char *bpsB, long long bps_bytesB, int ncontigB, const long long *clenB,
               const long long *boffB,
               int freq, int chain_break, int chain_min, int align_min, double align_rate,
               fgb_alns **out, fgb_run_stats *stats, void *stream);

/* SELF mode, `FastGA A` with one source (FastGA.c:4867-4931): T2 = T1 and BMXPOS = AMXPOS; the
 * merge follows new_self_merge_thread (FastGA.c:1616: every entry, both strands, against the other
 * members of its own block); a contig against itself, forward strand, is aligned strictly above or
 * strictly below the main diagonal (Local_Alignment's lbord / hbord, FastGA.c:3247-3262). */
int fgb_fastga_self(const unsigned char *bps, long long bps_bytes, int ncontig, const long long *clen,
                    const long long *boff, const float *freq4,
                    int freq, int chain_break, int chain_min, int align_min, double align_rate,
                    fgb_alns **out, fgb_run_stats *stats, void *stream);

/* Same from device-resident genomes (bench.py's timed step). */
int fgb_align_resident(const fgb_genome *A, const fgb_genome *B, const float *freqA,
                       int freq, int chain_break, int chain_min, int align_min, double align_rate,
                       fgb_alns **out, fgb_run_stats *stats, void *stream);

/* ---- genome (GDB.h:28-72; Get_Contig / Get_Contig_Piece GDB.c:1739,1841; Complement_Seq) ---- */
int  fgb_genome_create(const unsigned char *bps, long long bps_bytes, int ncontig,
                       const long long *clen, const long long *boff, int want_revcomp,
                       fgb_genome **out, void *stream);
void fgb_genome_free(fgb_genome *g);
int  fgb_genome_perm(const fgb_genome *g, int *perm_out);   /* Perm of GIXmake.c:1950-1963 */
int  fgb_genome_download(const fgb_genome *g, int rev, unsigned long long *words, long long *woff_out);
long long fgb_genome_words(const fgb_genome *g);

/* ---- GIX (GIXmake.c distribute + k_sort; MSDsort.c msd_sort; libfastk.c Kmer_Stream) ----
 * The table is sorted by the 40-mer; entries with EQUAL k-mers follow each other by
 * (strand|contig rank, post).  msd_sort leaves that order to its unstable in-place permutation
 * (MSDsort.c:211-360); no consumer depends on it (seeds are fully re-sorted, FastGA.c:4320). */
int  fgb_gix_build(const fgb_genome *g, fgb_gix **out, void *stream);
/* forward-strand entries only: enough for the genome that supplies the adaptamers (its reverse
   entries never seed, FastGA.c:921-928); fgb_seeds_find compacts a both-strand table itself */
int  fgb_gix_build_forward(const fgb_genome *g, fgb_gix **out, void *stream);
/* entries = concatenated .ktab parts, index = the stub's cumulative 2^24 table (libfastk.c:815-840) */
int  fgb_gix_import_ktab(const unsigned char *entries, long long n, int post_bytes, int cont_bytes,
                         const long long *index, int ncontig, fgb_gix **out, void *stream);
/* on-disk entries (GIXmake.c:1235-1261); part_first[p] = first entry index of .ktab part p+1 */
int  fgb_gix_export_ktab(const fgb_gix *x, const long long *part_first, int nparts,
                         unsigned char *out, void *stream);
int  fgb_gix_download(const fgb_gix *x, void *tab, unsigned *pstart, unsigned long long *buck1024);
long long fgb_gix_size(const fgb_gix *x);
int  fgb_gix_post_bytes(const fgb_gix *x);
int  fgb_gix_cont_bytes(const fgb_gix *x);
void fgb_gix_free(fgb_gix *x);

/* ---- seeds (adaptamer_merge FastGA.c:2281 + new_merge_thread :610; reimport_thread :2641;
 *             rmsd_sort RSDsort.c:292) ---- */
int  fgb_seeds_find(const fgb_gix *x1, const fgb_gix *x2, long long amxpos, long long bmxpos,
                    int freq, fgb_seeds **out, void *stream);
/* SELF mode: the table against itself (self_adaptamer_merge FastGA.c:2496, new_self_merge_thread :1616);
   fgb_extend on these seeds applies the self rules of align_contigs */
int  fgb_seeds_find_self(const fgb_gix *x, long long amxpos, int freq, fgb_seeds **out, void *stream);
long long fgb_seeds_size(const fgb_seeds *s);
long long fgb_seeds_sumlen(const fgb_seeds *s);
int  fgb_seeds_layout(const fgb_seeds *s, int *bits /* anti, band, jcont, icont */);
int  fgb_seeds_download(const fgb_seeds *s, void *rec);
void fgb_seeds_free(fgb_seeds *s);

/* ---- extension (search_seeds / align_contigs FastGA.c:3716,2973; Local_Alignment align.c:1423;
 *                 New_Align_Spec align.c:222; Compress_TraceTo8 align.c:3892) ---- */
int  fgb_align_spec(double ave_corr, const float *freq, short *tables /* 65536 */, int *ave_path);
int  fgb_extend(const fgb_seeds *S, const fgb_genome *A, const fgb_genome *B,
                int chain_break, int chain_min, int align_min, double align_rate,
                const short *tables, int ave_path, int tspace, fgb_overlaps **out, void *stream);
/* the align.h seam proper: Local_Alignment (align.c:1423; align.h:262-298) for a batch of call tuples.
 * jobs: n x 8 ints (A contig, B contig, comp, low, hgh, anti, lbord, hbord) = the arguments
 * align_contigs passes with aseq/bseq = those contigs (comp: A reverse-complemented + ACOMP_FLAG,
 * FastGA.c:3184-3260).  paths: n x 7 ints (abpos bbpos aepos bepos diffs tlen status; status != 0: the
 * call did not fit the device arenas); traces: uint8 (diff, B-advance) pairs at toff[i], as
 * Compress_TraceTo8 leaves them.  FGB_ERR_OVERFLOW with *traces_used set: call again with more room. */
int  fgb_local_alignments(const fgb_genome *A, const fgb_genome *B, long long n, const int *jobs,
                          const short *tables, int ave_path, int tspace,
                          int *paths, long long *toff, unsigned char *traces, long long traces_cap,
                          long long *traces_used, void *stream);
int  fgb_overlaps_from_buffer(const unsigned char *buf, long long nbytes, fgb_overlaps **out);
long long fgb_overlaps_bytes(const fgb_overlaps *o);
long long fgb_overlaps_count(const fgb_overlaps *o);
const unsigned char *fgb_overlaps_data(const fgb_overlaps *o);
void fgb_overlaps_counters(const fgb_overlaps *o, unsigned long long *out /* 16 */);
void fgb_overlaps_free(fgb_overlaps *o);

/* ---- redundancy filter + final order (FastGA.c:3407-3685, :2818 entwine, :3800 SORT_MAP) ---- */
int  fgb_filter(const fgb_overlaps *O, const int *perm1, const int *perm2, int jc_bits, int ic_bits,
                int do_filter, fgb_alns **out);
long long fgb_alns_count(const fgb_alns *a);
long long fgb_alns_raw_count(const fgb_alns *a);
long long fgb_alns_pool_bytes(const fgb_alns *a);
/* fields: n x 9 ints (comp aread bread abpos bbpos aepos bepos diffs tlen); toff: n; pool: traces */
int  fgb_alns_get(const fgb_alns *a, int *fields, long long *toff, unsigned char *pool);
void fgb_alns_free(fgb_alns *a);

/* ---- trace points -> edit scripts (Compute_Trace_PTS align.c:6171 with iter_np :5584, mode
 *      GREEDIEST, band unbounded: the call of ALNtoPAF.c:272 / ALNtoPSL.c:193 / ALNshow) ----
 * fields/toff/pool as fgb_alns_get returns them (B coordinates of strand-C records in complemented
 * B, as in the .1aln).  B needs its reverse complement (fgb_genome_create want_revcomp) when any
 * record is strand C.  Script of alignment i = script[soff[i]..soff[i+1]): the int list
 * Compute_Trace_PTS leaves in path->trace (align.h:330-349: -(A position+1) = a dash goes into A
 * before that base, +(B position+1) likewise for B); diffs[i] = path->diffs, -1 when the trace
 * points contradict the sequences (the reference exits there, align.c:5655). */
int  fgb_compute_trace_pts(const fgb_genome *A, const fgb_genome *B, long long n, const int *fields,
                           const long long *toff, const unsigned char *pool, int tspace,
                           fgb_scripts **out, void *stream);
long long fgb_scripts_count(const fgb_scripts *s);
long long fgb_scripts_total(const fgb_scripts *s);
long long fgb_scripts_bad(const fgb_scripts *s);
int  fgb_scripts_get(const fgb_scripts *s, long long *soff /* n+1 */, int *script, int *diffs /* n */);
void fgb_scripts_free(fgb_scripts *s);

/* ---- sort seam (building block of msd_sort / rmsd_sort, MSDsort.c:404 / RSDsort.c:292) ---- */
int  fgb_sort128_host(void *recs, long long n, int byte_lo, int byte_hi, void *stream);
int  fgb_sort128_device(void *d_a, void *d_b, long long n, int byte_lo, int byte_hi,
                        void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream);
long long fgb_sort128_tmp_bytes(long long n);

/* ---- the reference's own extern sort entry points, same signatures, host byte records in
 *      place (MSDsort.c:404 built -DLCPs, GIXmake.c:117; RSDsort.c:292, FastGA.c:149) ---- */
typedef struct { int beg; int end; long long off; } fgb_range;      /* Range, RSDsort.c:254-258 */
void fgb_msd_sort(unsigned char *array, long long nelem, int rsize, int ksize,
                  long long *part, int beg, int end, int nthreads);
int  fgb_rmsd_sort(unsigned char *array, long long nelem, int rsize, int ksize, int nparts,
                   long long *part, int nthreads, fgb_range *range);

/* ---- building blocks of the several-GPU path (one process per GPU; fastga_b200/shard.py issues
 *      them with two all-to-alls of 16-byte device records in between).  The k-mer space is cut by
 *      the top byte of the k-mer (first four bases), the seed space by the A contig: the same cuts
 *      the reference makes across threads (GIXmake.c:1426 panels by first byte; FastGA.c:4144, :4320
 *      Range[] of contigs per thread).  Device pointers are plain CUDA pointers on the calling process's
 *      current device; buffers handed out are released with fgb_device_free. ---- */
int  fgb_device_alloc(long long bytes, void **out, void *stream);
void fgb_device_free(void *p);
/* unsorted k-mer records of the contigs with mask[c] != 0; fwd_only drops reverse-strand entries */
int  fgb_kmers_scan(const fgb_genome *g, const unsigned char *mask, int fwd_only,
                    void **d_recs, long long *n, void *stream);
/* records grouped by destination: owner256[b] = rank owning top k-mer byte b; d_out[bounds[w] .. bounds[w+1])
   = the records of rank w */
int  fgb_records_group_by_owner(const void *d_recs, long long n, const int *owner256, int world,
                                void *d_out, long long *bounds, void *stream);
/* sorted + indexed table over records whose 12-base prefix lies in [plo,phi) (one rank's slice) */
int  fgb_gix_from_records(const void *d_recs, long long n, unsigned plo, unsigned phi, int fwd_only,
                          int post_bytes, int cont_bytes, int ncontig, fgb_gix **out, void *stream);
/* adaptamer merge without the seed sort: unsorted seed records, bits[4] = anti/band/jcont/icont
 * widths, info[2] = sum of seed lengths, T1 entries merged */
int  fgb_seeds_merge(const fgb_gix *x1, const fgb_gix *x2, long long amxpos, long long bmxpos, int freq,
                     void **d_seeds, long long *n, int *bits, long long *info, void *stream);
/* d_out[bounds[w] .. bounds[w+1]) = the seeds whose A contig (rank order) belongs to owner[.] == w */
int  fgb_seeds_group_by_owner(const void *d_seeds, long long n, const int *bits, const int *owner,
                              int nrank_contigs, int world, void *d_out, long long *bounds, void *stream);
/* sorted seed set over received records: input of fgb_extend on the owning rank */
int  fgb_seeds_from_records(const void *d_recs, long long n, const int *bits, long long amxpos,
                            long long bmxpos, long long sumlen, fgb_seeds **out, void *stream);

/* ---- diagnostics: the host rule that cuts a band-pair triple's chain list into independently
 *      extended groups (fgb_extend; DESIGN.md 3b), callable without a device.  hrange / tinfo: 2 ints per
 *      work triple ((first hit, count | bit 31 = no list), ((strand, contig pair) key, band)); hits:
 *      (alow, ahgh) per chain; gap < 0: the component rule with `bands` / `slack`, else cut at gaps >= gap.
 *      items_out: 4 words per item (triple, first hit, hits, number of the first hit in its triple) in
 *      launch order; next_out: (alow, ahgh) of the next group's first hit (INT64_MAX: none). ---- */
long long fgb_hit_groups_host(int nwork, const unsigned *hrange, const int *tinfo, const long long *hits,
                              long long nhits, int bands, long long slack, long long gap,
                              unsigned *items_out, long long *next_out);

/* ---- housekeeping ---- */
int  fgb_device_ready(void);
void fgb_release_cache(void);      /* return cached device blocks to the driver */
void fgb_timings_reset(void);
void fgb_timings_get(fgb_timings *out);

#ifdef __cplusplus
}
#endif
#endif
