// C-ABI of libfastga_b200.so: opaque handles (genome / GIX / seed set) over device memory and the
// host-buffer entry points the reference-side host code binds (see include/fastga_b200.h and
// INTEGRATION.md).  No torch types, no CPU fallback: every call runs the sm_100a kernels.
#include "common.cuh"
#include "handles.h"
#include <vector>
#include <algorithm>
#include <string.h>
#include <chrono>

typedef unsigned long long u64;

static inline long long now_us()
{ return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

extern "C" {
int fgb_kmer_sort_range_device(void *d_a, void *d_b, long long n, unsigned plo, unsigned phi,
                               void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream);
int fgb_sort128_bits_device(void *d_a, void *d_b, long long n, int bit_lo, int bit_hi,
                            void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream);
int fgb_sort128_device(void *d_a, void *d_b, long long n, int byte_lo, int byte_hi,
                       void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream);
long long fgb_sort128_tmp_bytes(long long n);
int fgb_stage_genome_device(const void *d_bps, const long long *d_boff, const long long *d_clen,
                            const long long *d_woff, int ncontig, long long total_words,
                            void *d_seq, void *d_rseq, void *stream);
int fgb_syncmer_count_device(const void *d_seq, const long long *d_clen, const long long *d_woff,
                             const int *d_crank, const int *d_tile_contig, const int *d_tile_start,
                             int ntiles, unsigned *d_tile_count, unsigned long long *d_buck1024,
                             unsigned long long *d_total, void *d_tmp, long long tmp_bytes,
                             int fwd_only, void *stream);
int fgb_syncmer_emit_device(const void *d_seq, const long long *d_clen, const long long *d_woff,
                            const int *d_crank, const int *d_tile_contig, const int *d_tile_start,
                            int ntiles, unsigned *d_tile_offset, void *d_records, int fwd_only,
                            void *stream);
int fgb_kix_index_device(const void *d_tab, long long n, unsigned *d_pstart, unsigned char *d_adj, void *stream);
int fgb_ktab_export_device(const void *d_tab, long long n, int pbytes, int cbytes,
                           const long long *d_part_first, int nparts, void *d_out, void *stream);
int fgb_ktab_import_device(const void *d_ent, long long n, int pbytes, int cbytes,
                           const long long *d_index, void *d_tab, void *stream);
int fgb_sc_tile();
int fgb_owner_count_device(const void *d_seeds, long long n, int p_ic, int ic_bits, const int *d_owner, int nrc,
                           int world, unsigned long long *d_cnt, void *stream);
int fgb_owner_scatter_device(const void *d_seeds, long long n, int p_ic, int ic_bits, const int *d_owner, int nrc,
                             int world, unsigned long long *d_base, void *d_out, void *stream);
int fgb_self_merge_device(const void *d_T, long long n, const unsigned *d_pstart, int freq,
                          int anti_bits, int band_bits, int jc_bits, int ic_bits,
                          long long amxpos, void *d_seeds, long long capacity,
                          unsigned long long *d_counters, unsigned long long *h_nseeds,
                          unsigned long long *h_sumlen, void *stream);
int fgb_forward_view_device(const void *d_T, long long n, void *d_out, long long *h_nfwd, void *stream);
int fgb_merge_device(const void *d_T1, long long n1, const void *d_T2, long long n2, const unsigned *d_pstart2,
                     const unsigned char *d_adj2, int freq, int anti_bits, int band_bits, int jc_bits, int ic_bits,
                     long long amxpos, long long bmxpos, void *d_seeds, long long capacity,
                     unsigned long long *d_counters, unsigned long long *h_nseeds,
                     unsigned long long *h_sumlen, void *stream);
}

fgb_timings g_timings;

void fgb_count_launch(int n) { g_timings.launches += n; }

//  Device memory for the stages comes from a process-wide caching allocator: blocks are rounded
//  to size classes, kept on a free list when released and handed out again on the next step, so
//  the steady state of a repeated workload makes no cudaMalloc/cudaFree calls at all (both stall
//  the device; the stream-ordered pool turned out to take 1-800 ms for the multi-GB arenas).
//  All work of a call is issued on one stream, so reuse after release is stream-ordered.

#include <map>
#include <unordered_map>
#include <mutex>

static std::multimap<size_t,void *> g_free;
static std::unordered_map<void *,size_t> g_live;
static std::mutex g_mem_lock;

static size_t size_class(size_t b)
{ if (b < 4096) return 4096;
  size_t p = 4096;
  while (p < b) p <<= 1;                 // p/2 < b <= p
  size_t step = p >> 4;                  // 8 classes per octave
  return ((b + step - 1) / step) * step;
}

cudaError_t fgb_dmalloc(void **p, size_t bytes, cudaStream_t st)
{ (void) st;
  size_t c = size_class(bytes);
  std::lock_guard<std::mutex> g(g_mem_lock);
  auto it = g_free.lower_bound(c);
  if (it != g_free.end() && it->first <= c + (c >> 2))
    { *p = it->second;
      g_live[*p] = it->first;
      g_free.erase(it);
      return cudaSuccess;
    }
  cudaError_t e = cudaMalloc(p,c);
  if (e != cudaSuccess)                  // out of memory: drop the cache and retry once
    { cudaGetLastError();
      for (auto &kv : g_free) cudaFree(kv.second);
      g_free.clear();
      e = cudaMalloc(p,c);
      if (e != cudaSuccess) return e;
    }
  g_live[*p] = c;
  return cudaSuccess;
}

void fgb_dfree(void *p, cudaStream_t st)
{ (void) st;
  if (p == NULL) return;
  std::lock_guard<std::mutex> g(g_mem_lock);
  auto it = g_live.find(p);
  if (it == g_live.end()) { cudaFree(p); return; }
  g_free.insert(std::make_pair(it->second,p));
  g_live.erase(it);
}

//  Gives every cached block back to the driver.
extern "C" void fgb_release_cache()
{ std::lock_guard<std::mutex> g(g_mem_lock);
  for (auto &kv : g_free) cudaFree(kv.second);
  g_free.clear();
}

extern "C" void fgb_timings_reset() { memset(&g_timings,0,sizeof(g_timings)); }
extern "C" void fgb_timings_get(fgb_timings *out) { *out = g_timings; }

/***********************************************************************************************
 *  Genome: the GDB as the path sees it (GDB.h:28-34 GDB_CONTIG {clen, boff} + the .bps image)
 **********************************************************************************************/

extern "C" void fgb_genome_free(fgb_genome *g)
{ cudaStream_t st = 0;
  if (!g) return;
  fgb_dfree(g->d_clen,st); fgb_dfree(g->d_woff,st); fgb_dfree(g->d_crank,st); fgb_dfree(g->d_perm,st);
  fgb_dfree(g->d_seq,st); fgb_dfree(g->d_rseq,st);
  delete g;
}

static const long long *g_sort_len;
static int LSORT(const void *l, const void *r)          // GIXmake.c:1628-1633: decreasing length
{ int x = *((const int *) l), y = *((const int *) r);
  return (int) (g_sort_len[y] - g_sort_len[x]);
}

extern "C" int fgb_genome_create(const unsigned char *bps, long long bps_bytes, int ncontig,
                                 const long long *clen, const long long *boff, int want_revcomp,
                                 fgb_genome **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (ncontig <= 0 || ncontig > 0x7fff) return FGB_ERR_LIMIT;   // contig rank is a 15-bit field
  owner<fgb_genome> own(new fgb_genome(),fgb_genome_free);
  fgb_genome *g = own.get();
  g->ncontig = ncontig;
  g->clen.assign(clen,clen+ncontig);
  g->boff.assign(boff,boff+ncontig);
  g->woff.resize(ncontig+1);
  g->seqtot = 0; g->maxlen = 0;
  long long w = 2;                             // 16 zero bytes ahead of the first contig too
  for (int c = 0; c < ncontig; c++)
    { if (clen[c] >= 0x7fffffffll) return FGB_ERR_LIMIT;
      g->woff[c] = w;
      w += ((clen[c] + 31) >> 5) + 2;          // zero pad so 64-bit window reads stay inside
      w = (w + 1) & ~1ll;                      // 16-byte alignment of every contig
      g->seqtot += clen[c];
      if (clen[c] > g->maxlen) g->maxlen = clen[c];
    }
  g->woff[ncontig] = w;
  g->total_words = w;

  g->perm.resize(ncontig); g->crank.resize(ncontig);
  for (int c = 0; c < ncontig; c++) g->perm[c] = c;
  g_sort_len = clen;
  qsort(g->perm.data(),ncontig,sizeof(int),LSORT);     // same libc call as GIXmake.c:1959
  for (int c = 0; c < ncontig; c++) g->crank[g->perm[c]] = c;

  unsigned char *d_bps = NULL;
  long long *d_boff = NULL;
  dev_scope S(st); S.own(d_bps); S.own(d_boff);
  CUDA_TRY(fgb_dmalloc((void **) &d_bps,bps_bytes + 16,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_boff,sizeof(long long)*ncontig,st));
  CUDA_TRY(fgb_dmalloc((void **) &g->d_clen,sizeof(long long)*ncontig,st));
  CUDA_TRY(fgb_dmalloc((void **) &g->d_woff,sizeof(long long)*(ncontig+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &g->d_crank,sizeof(int)*ncontig,st));
  CUDA_TRY(fgb_dmalloc((void **) &g->d_perm,sizeof(int)*ncontig,st));
  CUDA_TRY(fgb_dmalloc((void **) &g->d_seq,sizeof(u64)*(w + 1024),st));      // slack: the extension stages 1 KB tiles that may start near a contig end
  if (want_revcomp) CUDA_TRY(fgb_dmalloc((void **) &g->d_rseq,sizeof(u64)*(w + 1024),st));
  { stage_timer t(&g_timings.h2d_ms,st);
    CUDA_TRY(cudaMemcpyAsync(d_bps,bps,bps_bytes,cudaMemcpyHostToDevice,st));
    CUDA_TRY(cudaMemcpyAsync(d_boff,boff,sizeof(long long)*ncontig,cudaMemcpyHostToDevice,st));
    CUDA_TRY(cudaMemcpyAsync(g->d_clen,clen,sizeof(long long)*ncontig,cudaMemcpyHostToDevice,st));
    CUDA_TRY(cudaMemcpyAsync(g->d_woff,g->woff.data(),sizeof(long long)*(ncontig+1),cudaMemcpyHostToDevice,st));
    CUDA_TRY(cudaMemcpyAsync(g->d_crank,g->crank.data(),sizeof(int)*ncontig,cudaMemcpyHostToDevice,st));
    CUDA_TRY(cudaMemcpyAsync(g->d_perm,g->perm.data(),sizeof(int)*ncontig,cudaMemcpyHostToDevice,st));
  }
  g->h2d_bytes = bps_bytes + (long long) ncontig*(3*8+2*4) + 8;
  int rc;
  { stage_timer t(&g_timings.stage_ms,st);
    rc = fgb_stage_genome_device(d_bps,d_boff,g->d_clen,g->d_woff,ncontig,w,g->d_seq,g->d_rseq,st);
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  if (rc) return rc;
  *out = own.release();
  return FGB_OK;
}

extern "C" int fgb_genome_perm(const fgb_genome *g, int *perm_out)
{ memcpy(perm_out,g->perm.data(),sizeof(int)*g->ncontig); return FGB_OK; }

//  staged words back to the host (tests): seq (rev=0) or its reverse complement (rev=1)
extern "C" int fgb_genome_download(const fgb_genome *g, int rev, unsigned long long *words,
                                   long long *woff_out)
{ const u64 *src = rev ? g->d_rseq : g->d_seq;
  if (src == NULL) return FGB_ERR_ARG;
  CUDA_TRY(cudaMemcpy(words,src,sizeof(u64)*g->total_words,cudaMemcpyDeviceToHost));
  memcpy(woff_out,g->woff.data(),sizeof(long long)*(g->ncontig+1));
  return FGB_OK;
}
extern "C" long long fgb_genome_words(const fgb_genome *g) { return g->total_words; }

/***********************************************************************************************
 *  GIX
 **********************************************************************************************/

extern "C" void fgb_gix_free(fgb_gix *x)
{ cudaStream_t st = 0;
  if (!x) return;
  fgb_dfree(x->d_tab,st); fgb_dfree(x->d_pstart,st); fgb_dfree(x->d_adj,st);
  delete x;
}

static void gix_bytes(const fgb_genome *g, fgb_gix *x)        // GIXmake.c:1888-1901
{ long long cum;
  x->post_bytes = 0;
  for (cum = 1; cum < g->maxlen; cum *= 256) x->post_bytes += 1;
  x->cont_bytes = 0;
  for (cum = 1; cum < 2ll*g->ncontig; cum *= 256) x->cont_bytes += 1;
}

//  K1..K4: syncmer scan -> 128-bit records -> 10-pass byte radix sort on the 80-bit k-mer ->
//  2^24 prefix index.

//  K1/K2: syncmer scan + record build of the contigs selected by `mask` (NULL: all) into a fresh
//  device buffer of *n unsorted records (room for n+1).  fwd_only: forward-strand entries only,
//  *nrev = reverse entries left out.
static int gix_scan(const fgb_genome *g, const unsigned char *mask, bool fwd_only,
                    rec128 **d_recs, long long *n_out, long long *nrev, unsigned long long *buck1024, cudaStream_t st)
{ int T = fgb_sc_tile();
  std::vector<int> tc, ts;
  for (int c = 0; c < g->ncontig; c++)
    if (g->clen[c] >= 12 && g->boff[c] >= 0 && (mask == NULL || mask[c]))
      for (long long t0 = 0; t0 + 12 <= g->clen[c]; t0 += T)
        { tc.push_back(c); ts.push_back((int) t0); }
  int ntiles = (int) tc.size();
  int *d_tc = NULL, *d_ts = NULL; unsigned *d_cnt = NULL;
  u64 *d_buck = NULL, *d_total = NULL; void *d_tmp = NULL;
  rec128 *d_a = NULL;
  dev_scope S(st); S.own(d_tc); S.own(d_ts); S.own(d_cnt); S.own(d_buck); S.own(d_total); S.own(d_tmp); S.own(d_a);
  long long tmpb = fgb_dev_scan_tmp_bytes(ntiles);
  int rc;
  u64 total = 0, rdropped = 0;
  CUDA_TRY(fgb_dmalloc((void **) &d_tc,sizeof(int)*(ntiles+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_ts,sizeof(int)*(ntiles+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_cnt,sizeof(unsigned)*(ntiles+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_buck,8*1025,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_total,8,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_tmp,tmpb,st));
  CUDA_TRY(cudaMemcpyAsync(d_tc,tc.data(),sizeof(int)*ntiles,cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemcpyAsync(d_ts,ts.data(),sizeof(int)*ntiles,cudaMemcpyHostToDevice,st));
  { stage_timer t(&g_timings.scan_ms,st);
    rc = fgb_syncmer_count_device(g->d_seq,g->d_clen,g->d_woff,g->d_crank,d_tc,d_ts,ntiles,d_cnt,
                                  d_buck,d_total,d_tmp,tmpb,fwd_only,st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(&total,d_total,8,cudaMemcpyDeviceToHost,st));
    if (buck1024) CUDA_TRY(cudaMemcpyAsync(buck1024,d_buck,8*1024,cudaMemcpyDeviceToHost,st));
    CUDA_TRY(cudaMemcpyAsync(&rdropped,d_buck + 1024,8,cudaMemcpyDeviceToHost,st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  if (total >= 0xfffffff0ull) return FGB_ERR_LIMIT;
  CUDA_TRY(fgb_dmalloc((void **) &d_a,sizeof(rec128)*(total+1),st));
  { stage_timer t(&g_timings.scan_ms,st);
    rc = fgb_syncmer_emit_device(g->d_seq,g->d_clen,g->d_woff,g->d_crank,d_tc,d_ts,ntiles,d_cnt,d_a,fwd_only,st);
  }
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));                      // tc/ts must outlive the copies
  *d_recs = d_a; d_a = NULL;                                // handed to the caller
  *n_out = (long long) total; *nrev = (long long) rdropped;
  return FGB_OK;
}

//  K3/K4: sorts the records in d_a whose 12-base prefixes lie in [plo,phi) and, with `index`, builds
//  the prefix index and the LCP bytes.  d_a is consumed: it ends up inside the handle or is released,
//  and the caller's pointer is cleared either way.
static int gix_finish(fgb_gix *x, rec128 *&d_a, long long n, unsigned plo, unsigned phi, bool index, cudaStream_t st)
{ rec128 *d_b = NULL; void *d_stmp = NULL;
  dev_scope S(st); S.own(d_a); S.own(d_b); S.own(d_stmp);
  long long stmpb = fgb_sort128_tmp_bytes(n);
  int rc, inb = 0;
  x->n = n;
  CUDA_TRY(fgb_dmalloc((void **) &d_b,sizeof(rec128)*(n+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_stmp,stmpb,st));
  if (index)
    { CUDA_TRY(fgb_dmalloc((void **) &x->d_pstart,sizeof(unsigned)*((1<<24)+1+8),st));
      CUDA_TRY(fgb_dmalloc((void **) &x->d_adj,(size_t) n + 32,st));
    }
  { stage_timer t(&g_timings.ksort_ms,st);
    rc = fgb_kmer_sort_range_device(d_a,d_b,n,plo,phi,d_stmp,stmpb,&inb,st);
  }
  if (rc) return rc;
  x->d_tab = inb ? d_b : d_a;
  if (inb) d_b = NULL; else d_a = NULL;                     // ownership moved to the handle
  if (index)
    { stage_timer t(&g_timings.index_ms,st);
      rc = fgb_kix_index_device(x->d_tab,n,x->d_pstart,x->d_adj,st);
    }
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));
  return FGB_OK;
}

//  fwd_only: forward-strand entries only; index: false = the table alone, no prefix index and no LCP
//  bytes (the T1 side of a merge reads neither)
static int gix_build(const fgb_genome *g, bool fwd_only, bool index, fgb_gix **out, cudaStream_t st)
{ owner<fgb_gix> own(new fgb_gix(),fgb_gix_free);
  fgb_gix *x = own.get();
  gix_bytes(g,x);
  x->ncontig = g->ncontig;
  x->fwd_only = fwd_only ? 1 : 0;
  rec128 *d_a = NULL; long long n = 0, nrev = 0;
  int rc = gix_scan(g,NULL,fwd_only,&d_a,&n,&nrev,x->buck1024,st);
  if (rc) return rc;
  x->n_both = n + nrev;
  if ((rc = gix_finish(x,d_a,n,0u,1u << 24,index,st))) return rc;
  *out = own.release();
  return FGB_OK;
}

extern "C" int fgb_gix_build(const fgb_genome *g, fgb_gix **out, void *stream)
{ return gix_build(g,false,true,out,(cudaStream_t) stream); }

//  Forward-strand entries only: the table of the genome that supplies the adaptamers.  Reverse
//  entries of T1 never seed (FastGA.c:921-928), so the fused path does not build, sort or read them.
extern "C" int fgb_gix_build_forward(const fgb_genome *g, fgb_gix **out, void *stream)
{ return gix_build(g,true,true,out,(cudaStream_t) stream); }

/***********************************************************************************************
 *  Building blocks of the k-mer-space sharded path (several GPUs, fastga_b200/shard.py): every rank
 *  scans ITS contigs of both genomes, the k-mer records travel to the rank that owns their prefix
 *  range, each rank merges its slice of the two tables, and the seeds travel to the rank that owns
 *  their A-contig.  Nothing is replicated; the two exchanges are all-to-alls of 16-byte records.
 **********************************************************************************************/

extern "C" int fgb_device_alloc(long long bytes, void **out, void *stream)
{ CUDA_TRY(fgb_dmalloc(out,(size_t) (bytes > 0 ? bytes : 16),(cudaStream_t) stream)); return FGB_OK; }
extern "C" void fgb_device_free(void *p) { fgb_dfree(p,0); }

//  unsorted k-mer records of the contigs with mask[c] != 0 (device buffer handed to the caller:
//  fgb_device_free); fwd_only: forward-strand entries only (the adaptamer side)
extern "C" int fgb_kmers_scan(const fgb_genome *g, const unsigned char *mask, int fwd_only,
                              void **d_recs, long long *n, void *stream)
{ rec128 *d = NULL; long long nrev = 0;
  int rc = gix_scan(g,mask,fwd_only != 0,&d,n,&nrev,NULL,(cudaStream_t) stream);
  if (rc) return rc;
  *d_recs = d;
  return FGB_OK;
}

//  a table over n unsorted device records (copied) whose 12-base prefixes lie in [plo,phi): one
//  rank's slice of a k-mer-space sharded table
extern "C" int fgb_gix_from_records(const void *d_recs, long long n, unsigned plo, unsigned phi, int fwd_only,
                                    int post_bytes, int cont_bytes, int ncontig, fgb_gix **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n < 0 || n >= 0xfffffff0ll || plo >= phi || phi > (1u << 24)) return FGB_ERR_ARG;
  owner<fgb_gix> own(new fgb_gix(),fgb_gix_free);
  fgb_gix *x = own.get();
  x->n_both = n; x->post_bytes = post_bytes; x->cont_bytes = cont_bytes; x->ncontig = ncontig;
  x->fwd_only = fwd_only ? 1 : 0;
  rec128 *d_a = NULL;
  dev_scope S(st); S.own(d_a);
  CUDA_TRY(fgb_dmalloc((void **) &d_a,sizeof(rec128)*(n+1),st));
  if (n > 0) CUDA_TRY(cudaMemcpyAsync(d_a,d_recs,sizeof(rec128)*n,cudaMemcpyDeviceToDevice,st));
  int rc = gix_finish(x,d_a,n,plo,phi,true,st);
  if (rc) return rc;
  *out = own.release();
  return FGB_OK;
}

extern "C" long long fgb_gix_size(const fgb_gix *x) { return x->n; }
extern "C" int fgb_gix_post_bytes(const fgb_gix *x) { return x->post_bytes; }
extern "C" int fgb_gix_cont_bytes(const fgb_gix *x) { return x->cont_bytes; }

extern "C" int fgb_gix_download(const fgb_gix *x, void *tab /* n x 16 B */, unsigned *pstart /* 2^24+1 */,
                                unsigned long long *buck1024)
{ if (tab) CUDA_TRY(cudaMemcpy(tab,x->d_tab,sizeof(rec128)*x->n,cudaMemcpyDeviceToHost));
  if (pstart) CUDA_TRY(cudaMemcpy(pstart,x->d_pstart,sizeof(unsigned)*((1<<24)+1),cudaMemcpyDeviceToHost));
  if (buck1024) memcpy(buck1024,x->buck1024,8*1024);
  return FGB_OK;
}

//  A GIX from the reference's on-disk form: concatenated .ktab entries (all parts, in order) and
//  the stub's cumulative 2^24 index (libfastk.c:815-840).
extern "C" int fgb_gix_import_ktab(const unsigned char *entries, long long n, int post_bytes,
                                   int cont_bytes, const long long *index, int ncontig,
                                   fgb_gix **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n >= 0xfffffff0ll || post_bytes > 4 || cont_bytes > 2) return FGB_ERR_LIMIT;
  owner<fgb_gix> own(new fgb_gix(),fgb_gix_free);
  fgb_gix *x = own.get();
  x->n = n; x->n_both = n; x->post_bytes = post_bytes; x->cont_bytes = cont_bytes; x->ncontig = ncontig;
  long long E = 9 + post_bytes + cont_bytes;
  unsigned char *d_ent = NULL; long long *d_index = NULL;
  dev_scope S(st); S.own(d_ent); S.own(d_index);
  CUDA_TRY(fgb_dmalloc((void **) &d_ent,E*n + 16,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_index,8ll<<24,st));
  CUDA_TRY(fgb_dmalloc((void **) &x->d_tab,sizeof(rec128)*(n+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &x->d_pstart,sizeof(unsigned)*((1<<24)+1+8),st));
  CUDA_TRY(fgb_dmalloc((void **) &x->d_adj,(size_t) x->n + 32,st));
  CUDA_TRY(cudaMemcpyAsync(d_ent,entries,E*n,cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemcpyAsync(d_index,index,8ll<<24,cudaMemcpyHostToDevice,st));
  int rc = fgb_ktab_import_device(d_ent,n,post_bytes,cont_bytes,d_index,x->d_tab,st);
  if (!rc) rc = fgb_kix_index_device(x->d_tab,n,x->d_pstart,x->d_adj,st);
  CUDA_TRY(cudaStreamSynchronize(st));
  if (rc) return rc;
  *out = own.release();
  return FGB_OK;
}

//  On-disk entries for the whole table (host buffer of n*(9+pb+cb) bytes); part_first = entry
//  index at which each .ktab part starts (its LCP byte is 0, MSDsort.c:485-488).
extern "C" int fgb_gix_export_ktab(const fgb_gix *x, const long long *part_first, int nparts,
                                   unsigned char *out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  long long E = 9 + x->post_bytes + x->cont_bytes;
  unsigned char *d_out = NULL; long long *d_pf = NULL;
  dev_scope S(st); S.own(d_out); S.own(d_pf);
  CUDA_TRY(fgb_dmalloc((void **) &d_out,E*x->n + 16,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_pf,8*(nparts+1),st));
  CUDA_TRY(cudaMemcpyAsync(d_pf,part_first,8*nparts,cudaMemcpyHostToDevice,st));
  int rc = fgb_ktab_export_device(x->d_tab,x->n,x->post_bytes,x->cont_bytes,d_pf,nparts,d_out,st);
  if (!rc) CUDA_TRY(cudaMemcpyAsync(out,d_out,E*x->n,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return rc;
}

/***********************************************************************************************
 *  Seeds: adaptamer merge + seed sort
 **********************************************************************************************/

static int bitlen(long long v) { int b = 0; while (v > 0) { b += 1; v >>= 1; } return b; }

extern "C" void fgb_seeds_free(fgb_seeds *s)
{ cudaStream_t st = 0;
  if (!s) return;
  fgb_dfree(s->d_rec,st);
  delete s;
}

static int seeds_find_impl(const fgb_gix *x1, const fgb_gix *x2, long long amxpos,
                           long long bmxpos, int freq, bool self, fgb_seeds **out, void *stream);

extern "C" int fgb_seeds_find(const fgb_gix *x1, const fgb_gix *x2, long long amxpos,
                              long long bmxpos, int freq, fgb_seeds **out, void *stream)
{ return seeds_find_impl(x1,x2,amxpos,bmxpos,freq,false,out,stream); }

//  SELF mode (FastGA A): the table against itself (new_self_merge_thread, FastGA.c:1616)
extern "C" int fgb_seeds_find_self(const fgb_gix *x, long long amxpos, int freq, fgb_seeds **out, void *stream)
{ return seeds_find_impl(x,x,amxpos,amxpos,freq,true,out,stream); }

struct seed_bits { int anti, band, jc, ic, key; };

static int seed_layout_of(const fgb_gix *x1, const fgb_gix *x2, long long amxpos, long long bmxpos, seed_bits *L)
{ L->anti = bitlen(amxpos + bmxpos);
  L->band = L->anti > 6 ? L->anti - 6 : 1;
  L->jc   = bitlen(x2->ncontig > 1 ? x2->ncontig-1 : 1);
  L->ic   = bitlen(x1->ncontig > 1 ? x1->ncontig-1 : 1);
  L->key  = 12 + L->anti + L->band + L->jc + L->ic + 1;
  return L->key > 128 ? FGB_ERR_LIMIT : FGB_OK;
}

//  K5: the unsorted seed records of x1 against x2 in a fresh device buffer (room for n+1)
static int seeds_merge_impl(const fgb_gix *x1, const fgb_gix *x2, long long amxpos, long long bmxpos, int freq,
                            bool self, const seed_bits &L, rec128 **d_out, long long *nseeds_out,
                            long long *sumlen_out, long long *n1m_out, cudaStream_t st)
{ if (self && x1->fwd_only) return FGB_ERR_ARG;                // SELF mode needs both strands
  u64 *d_counters = NULL; rec128 *d_fwd = NULL, *d_a = NULL;
  dev_scope S(st); S.own(d_counters); S.own(d_fwd); S.own(d_a);
  int rc;
  u64 nseeds = 0, sumlen = 0;
  //  the adaptamer side must be a forward-strand table (reverse entries never seed): a both-strand
  //  table (imported .ktab, fgb_gix_build) is compacted once; the fused path builds it forward-only
  const rec128 *t1 = x1->d_tab; long long n1 = x1->n;
  CUDA_TRY(fgb_dmalloc((void **) &d_counters,16,st));
  if (!self && !x1->fwd_only && n1 > 0)
    { CUDA_TRY(fgb_dmalloc((void **) &d_fwd,sizeof(rec128)*(n1+1),st));
      if ((rc = fgb_forward_view_device(x1->d_tab,n1,d_fwd,&n1,st))) return rc;
      t1 = d_fwd;
    }
  long long cap = (self ? 2*x1->n : 2*n1 + (n1 >> 1)) + 1024;
  for (int attempt = 0; ; attempt++)
    { CUDA_TRY(fgb_dmalloc((void **) &d_a,sizeof(rec128)*(cap+1),st));
      if (self)
        rc = fgb_self_merge_device(x1->d_tab,x1->n,x1->d_pstart,freq,L.anti,L.band,L.jc,L.ic,amxpos,
                                   d_a,cap,d_counters,&nseeds,&sumlen,st);
      else
        rc = fgb_merge_device(t1,n1,x2->d_tab,x2->n,x2->d_pstart,x2->d_adj,freq,L.anti,L.band,L.jc,L.ic,
                              amxpos,bmxpos,d_a,cap,d_counters,&nseeds,&sumlen,st);
      if (rc == FGB_OK) break;
      fgb_dfree(d_a,st); d_a = NULL;                          // the retry allocates it anew
      if (rc != FGB_ERR_OVERFLOW || attempt > 0) return rc;
      cap = (long long) nseeds + 1024;
      g_timings.merge_ms = 0; g_timings.merge_launches = 0;   // only the successful launch is reported
    }
  if (nseeds >= 0xfffffff0ull) return FGB_ERR_LIMIT;
  *d_out = d_a; d_a = NULL;                                   // handed to the caller
  *nseeds_out = (long long) nseeds; *sumlen_out = (long long) sumlen; *n1m_out = n1;
  return FGB_OK;
}

//  K6: sorts n seed records in d_a into a handle.  d_a is consumed: it ends up inside the handle or
//  is released, and the caller's pointer is cleared either way.
static int seeds_sort_impl(rec128 *&d_a, long long n, const seed_bits &L, long long amxpos, long long bmxpos,
                           bool self, long long sumlen, long long n1m, fgb_seeds **out, cudaStream_t st)
{ owner<fgb_seeds> own(new fgb_seeds(),fgb_seeds_free);
  rec128 *d_b = NULL; void *d_tmp = NULL;
  dev_scope S(st); S.own(d_a); S.own(d_b); S.own(d_tmp);
  fgb_seeds *s = own.get();
  s->self_mode = self ? 1 : 0;
  s->anti_bits = L.anti; s->band_bits = L.band; s->jc_bits = L.jc; s->ic_bits = L.ic;
  s->amxpos = amxpos; s->bmxpos = bmxpos;
  s->n = n; s->sumlen = sumlen; s->n1_merged = n1m;
  long long tmpb = fgb_sort128_tmp_bytes(n);
  int rc, inb = 0;
  CUDA_TRY(fgb_dmalloc((void **) &d_b,sizeof(rec128)*(n+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_tmp,tmpb,st));
  { stage_timer t(&g_timings.ssort_ms,st);
    //  from bit 6: the lcp field (bits 0..5) cannot break a tie -- two seeds that agree on strand,
    //  contigs, band, anti-diagonal and diagonal remainder are the same pair of positions
    rc = fgb_sort128_bits_device(d_a,d_b,n,6,L.key,d_tmp,tmpb,&inb,st);
  }
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));
  s->d_rec = inb ? d_b : d_a;
  if (inb) d_b = NULL; else d_a = NULL;                       // ownership moved to the handle
  *out = own.release();
  return FGB_OK;
}

static int seeds_find_impl(const fgb_gix *x1, const fgb_gix *x2, long long amxpos,
                           long long bmxpos, int freq, bool self, fgb_seeds **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  seed_bits L;
  int rc = seed_layout_of(x1,x2,amxpos,bmxpos,&L);
  if (rc) return rc;
  rec128 *d_a = NULL; long long n = 0, sumlen = 0, n1m = 0;
  if ((rc = seeds_merge_impl(x1,x2,amxpos,bmxpos,freq,self,L,&d_a,&n,&sumlen,&n1m,st))) return rc;
  return seeds_sort_impl(d_a,n,L,amxpos,bmxpos,self,sumlen,n1m,out,st);
}

//  ---- sharded path: seeds leave the merge unsorted, travel to their A-contig's owner, are sorted there ----

//  unsorted seed records of x1 against x2 (device buffer handed to the caller: fgb_device_free);
//  bits[4] = anti, band, jcont, icont field widths; info[2] = sum of seed lengths, T1 entries merged
extern "C" int fgb_seeds_merge(const fgb_gix *x1, const fgb_gix *x2, long long amxpos, long long bmxpos, int freq,
                               void **d_seeds, long long *n, int *bits, long long *info, void *stream)
{ seed_bits L;
  int rc = seed_layout_of(x1,x2,amxpos,bmxpos,&L);
  if (rc) return rc;
  rec128 *d_a = NULL; long long sumlen = 0, n1m = 0;
  if ((rc = seeds_merge_impl(x1,x2,amxpos,bmxpos,freq,false,L,&d_a,n,&sumlen,&n1m,(cudaStream_t) stream))) return rc;
  *d_seeds = d_a;
  bits[0] = L.anti; bits[1] = L.band; bits[2] = L.jc; bits[3] = L.ic;
  if (info) { info[0] = sumlen; info[1] = n1m; }
  return FGB_OK;
}

//  d_out[bounds[w] .. bounds[w+1]) are the records with owner[f] == w, f = the field_bits wide field
//  at bit field_pos of the record (f >= nowner: owner 0).  Count + scatter, order inside a group free.
static int group_by_owner(const void *d_in, long long n, int field_pos, int field_bits, const int *owner,
                          int nowner, int world, void *d_out, long long *bounds, cudaStream_t st)
{ if (world < 1 || world > 64) return FGB_ERR_ARG;
  for (int w = 0; w <= world; w++) bounds[w] = 0;
  if (n <= 0) return FGB_OK;
  int *d_owner = NULL; u64 *d_cnt = NULL;
  dev_scope S(st); S.own(d_owner); S.own(d_cnt);
  int rc;
  u64 cnt[64], base[65];
  CUDA_TRY(fgb_dmalloc((void **) &d_owner,sizeof(int)*(size_t) nowner,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_cnt,8*64*2,st));
  CUDA_TRY(cudaMemcpyAsync(d_owner,owner,sizeof(int)*(size_t) nowner,cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemsetAsync(d_cnt,0,8*64*2,st));
  if ((rc = fgb_owner_count_device(d_in,n,field_pos,field_bits,d_owner,nowner,world,d_cnt,st))) return rc;
  CUDA_TRY(cudaMemcpyAsync(cnt,d_cnt,8*64,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  base[0] = 0;
  for (int w = 0; w < world; w++) base[w+1] = base[w] + cnt[w];
  CUDA_TRY(cudaMemcpyAsync(d_cnt + 64,base,8*64,cudaMemcpyHostToDevice,st));
  if ((rc = fgb_owner_scatter_device(d_in,n,field_pos,field_bits,d_owner,nowner,world,d_cnt + 64,d_out,st))) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));
  for (int w = 0; w <= world; w++) bounds[w] = (long long) base[w];
  return FGB_OK;
}

//  seeds grouped by the rank that owns their A-contig: owner[r] for contig RANK r (the icont field)
extern "C" int fgb_seeds_group_by_owner(const void *d_seeds, long long n, const int *bits, const int *owner,
                                        int nrank_contigs, int world, void *d_out, long long *bounds,
                                        void *stream)
{ return group_by_owner(d_seeds,n,12 + bits[0] + bits[1] + bits[2],bits[3],owner,nrank_contigs,world,d_out,bounds,
                        (cudaStream_t) stream); }

//  k-mer records grouped by the rank that owns their first four bases: owner256[b] for top byte b
extern "C" int fgb_records_group_by_owner(const void *d_recs, long long n, const int *owner256, int world,
                                          void *d_out, long long *bounds, void *stream)
{ return group_by_owner(d_recs,n,120,8,owner256,256,world,d_out,bounds,(cudaStream_t) stream); }

//  sorted seed set over n unsorted device records (copied); bits as fgb_seeds_merge returns them
extern "C" int fgb_seeds_from_records(const void *d_recs, long long n, const int *bits, long long amxpos,
                                      long long bmxpos, long long sumlen, fgb_seeds **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n < 0 || n >= 0xfffffff0ll) return FGB_ERR_LIMIT;
  seed_bits L;
  L.anti = bits[0]; L.band = bits[1]; L.jc = bits[2]; L.ic = bits[3];
  L.key = 12 + L.anti + L.band + L.jc + L.ic + 1;
  if (L.key > 128) return FGB_ERR_LIMIT;
  rec128 *d_a = NULL;
  dev_scope S(st); S.own(d_a);
  CUDA_TRY(fgb_dmalloc((void **) &d_a,sizeof(rec128)*(n+1),st));
  if (n > 0) CUDA_TRY(cudaMemcpyAsync(d_a,d_recs,sizeof(rec128)*n,cudaMemcpyDeviceToDevice,st));
  return seeds_sort_impl(d_a,n,L,amxpos,bmxpos,false,sumlen,0,out,st);
}

extern "C" long long fgb_seeds_size(const fgb_seeds *s) { return s->n; }
extern "C" long long fgb_seeds_sumlen(const fgb_seeds *s) { return s->sumlen; }
extern "C" int fgb_seeds_layout(const fgb_seeds *s, int *bits /* anti, band, jc, ic */)
{ bits[0] = s->anti_bits; bits[1] = s->band_bits; bits[2] = s->jc_bits; bits[3] = s->ic_bits; return FGB_OK; }
extern "C" int fgb_seeds_download(const fgb_seeds *s, void *rec)
{ CUDA_TRY(cudaMemcpy(rec,s->d_rec,sizeof(rec128)*s->n,cudaMemcpyDeviceToHost)); return FGB_OK; }

//  Plain host-buffer sort of 16-byte records on key bytes [byte_lo,byte_hi): the building block
//  behind both drop-in sort seams.
extern "C" int fgb_sort128_host(void *recs, long long n, int byte_lo, int byte_hi, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  rec128 *d_a = NULL, *d_b = NULL; void *d_tmp = NULL;
  dev_scope S(st); S.own(d_a); S.own(d_b); S.own(d_tmp);
  long long tmpb = fgb_sort128_tmp_bytes(n);
  CUDA_TRY(fgb_dmalloc((void **) &d_a,sizeof(rec128)*(n+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_b,sizeof(rec128)*(n+1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_tmp,tmpb,st));
  CUDA_TRY(cudaMemcpyAsync(d_a,recs,sizeof(rec128)*n,cudaMemcpyHostToDevice,st));
  int inb = 0;
  int rc = fgb_sort128_device(d_a,d_b,n,byte_lo,byte_hi,d_tmp,tmpb,&inb,st);
  if (!rc) CUDA_TRY(cudaMemcpyAsync(recs,inb ? d_b : d_a,sizeof(rec128)*n,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return rc;
}

extern "C" int fgb_device_ready()
{ int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return 0;
  return 1;
}

/***********************************************************************************************
 *  Whole path, host buffers in / host records out: what `FastGA -1:<out> A B` computes between
 *  Read_GDB and la_merge (FastGA.c:4927-5205), GIX construction included.
 **********************************************************************************************/

struct fgb_overlaps;
struct fgb_alns;
extern "C" {
int fgb_extend(const fgb_seeds *S, const fgb_genome *A, const fgb_genome *B, int chain_break,
               int chain_min, int align_min, double align_rate, const short *tables, int ave_path,
               int tspace, fgb_overlaps **out, void *stream);
int fgb_align_spec(double ave_corr, const float *freq, short *tables, int *ave_path);
void fgb_overlaps_free(fgb_overlaps *o);
long long fgb_overlaps_bytes(const fgb_overlaps *o);
void fgb_overlaps_counters(const fgb_overlaps *o, unsigned long long *out);
int fgb_filter(const fgb_overlaps *O, const int *perm1, const int *perm2, int jc_bits, int ic_bits,
               int do_filter, fgb_alns **out);
}

struct fgb_run_stats
{ long long nkmers1, nkmers2, nseeds, sumlen, nhits, nla, nwaves, ncells, nraw, h2d_bytes, d2h_bytes,
            nseg, nwork, warp_cycles, wave_cycles, extract_cycles,
            us_gix, us_seeds, us_extend, us_filter, nkmers1_fwd,
            slow_cycles, slow_waves, paired_waves, pairings; };

//  The tail of both whole-path calls: extension of the seeds (released here), redundancy filter, and
//  the seed and overlap counters of *stats (nseeds, sumlen, nhits .. nraw, nseg .. extract_cycles,
//  slow_cycles .. pairings).  Where not NULL: *t_extended = host clock when the extension is done,
//  *ovl_bytes = bytes of raw records read back from the device.
static int extend_and_filter(fgb_seeds *sd, const fgb_genome *A, const fgb_genome *B, const float *freqA,
                             int chain_break, int chain_min, int align_min, double align_rate,
                             fgb_alns **out, fgb_run_stats *stats, long long *t_extended, long long *ovl_bytes,
                             void *stream)
{ fgb_overlaps *ov = NULL;
  short *tables = (short *) malloc(65536*sizeof(short));
  int ave = 0;
  fgb_align_spec(1.-align_rate,freqA,tables,&ave);           // FastGA.c:3760
  int rc = fgb_extend(sd,A,B,chain_break,chain_min,align_min,align_rate,tables,ave,100,&ov,stream);
  free(tables);
  if (t_extended) *t_extended = now_us();
  const long long nseeds = sd->n, sumlen = sd->sumlen;
  const int jb = sd->jc_bits, ib = sd->ic_bits;
  fgb_seeds_free(sd);
  if (rc) return rc;
  owner<fgb_overlaps> own(ov,fgb_overlaps_free);
  rc = fgb_filter(ov,A->perm.data(),B->perm.data(),jb,ib,1,out);
  if (ovl_bytes) *ovl_bytes = fgb_overlaps_bytes(ov);
  if (stats)
    { unsigned long long c[16];
      fgb_overlaps_counters(ov,c);
      stats->nseeds = nseeds; stats->sumlen = sumlen;
      stats->nhits = (long long) c[0]; stats->nla = (long long) c[1]; stats->nwaves = (long long) c[2];
      stats->ncells = (long long) c[3]; stats->nraw = 0;
      stats->nseg = (long long) c[5]; stats->nwork = (long long) c[6];
      stats->warp_cycles = (long long) c[8]; stats->wave_cycles = (long long) c[9];
      stats->extract_cycles = (long long) c[10];
      stats->slow_cycles = (long long) ((c[15] >> 40) << 12); stats->slow_waves = (long long) ((c[15] >> 16) & 0xffffff);
      stats->paired_waves = (long long) c[11]; stats->pairings = (long long) c[12];
    }
  return rc;
}

//  Device-resident genomes in, final alignments out (the timed "step" of bench.py).
extern "C" int fgb_align_resident(const fgb_genome *A, const fgb_genome *B, const float *freqA,
                                  int freq, int chain_break, int chain_min, int align_min,
                                  double align_rate, fgb_alns **out, fgb_run_stats *stats, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  fgb_gix *x1 = NULL, *x2 = NULL;
  int rc;
  long long t0 = now_us();
  //  adaptamer side: forward strand only, and only the table (the merge reads the OTHER table's index)
  if ((rc = gix_build(A,true,false,&x1,st))) return rc;
  owner<fgb_gix> own1(x1,fgb_gix_free);
  if ((rc = gix_build(B,false,true,&x2,st))) return rc;
  owner<fgb_gix> own2(x2,fgb_gix_free);
  long long t1 = now_us();
  const long long n1 = x1->n_both, n2 = x2->n;
  seed_bits L;
  rec128 *d_a = NULL; long long n = 0, sumlen = 0, n1m = 0;
  rc = seed_layout_of(x1,x2,A->maxlen,B->maxlen,&L);
  if (!rc) rc = seeds_merge_impl(x1,x2,A->maxlen,B->maxlen,freq,false,L,&d_a,&n,&sumlen,&n1m,st);
  //  the tables go back to the allocator as soon as the merge has read them (two tables + seeds +
  //  sort buffer of a multi-Gbp pair do not fit side by side)
  own1.reset(); own2.reset();
  if (rc) return rc;
  fgb_seeds *sd = NULL;
  if ((rc = seeds_sort_impl(d_a,n,L,A->maxlen,B->maxlen,false,sumlen,n1m,&sd,st))) return rc;
  long long t2 = now_us(), t3 = t2, ovl_bytes = 0;
  rc = extend_and_filter(sd,A,B,freqA,chain_break,chain_min,align_min,align_rate,out,stats,&t3,&ovl_bytes,stream);
  long long t4 = now_us();
  if (rc) return rc;
  if (stats)
    { stats->us_gix = t1-t0; stats->us_seeds = t2-t1; stats->us_extend = t3-t2; stats->us_filter = t4-t3;
      stats->nkmers1 = n1; stats->nkmers2 = n2; stats->nkmers1_fwd = n1m;
      stats->h2d_bytes = A->h2d_bytes + B->h2d_bytes + 65536*2;
      stats->d2h_bytes = ovl_bytes + 16 + 8*1024*2 + 64;
    }
  return FGB_OK;
}

//  The reference-facing call: host .bps images + contig tables in, alignments out; every
//  host<->device copy happens inside.
//  SELF mode: `FastGA A` (one source).  Same path with T2 = T1, BMXPOS = AMXPOS, the self block rule
//  in the merge and the band borders of align_contigs for a contig against itself.
extern "C" int fgb_fastga_self(const unsigned char *bps, long long nb, int nc, const long long *clen,
                               const long long *boff, const float *freq4,
                               int freq, int chain_break, int chain_min, int align_min, double align_rate,
                               fgb_alns **out, fgb_run_stats *stats, void *stream)
{ fgb_genome *A = NULL; fgb_gix *x = NULL; fgb_seeds *sd = NULL;
  int rc;
  if ((rc = fgb_genome_create(bps,nb,nc,clen,boff,1,&A,stream))) return rc;
  owner<fgb_genome> own(A,fgb_genome_free);
  if ((rc = fgb_gix_build(A,&x,stream))) return rc;
  rc = fgb_seeds_find_self(x,A->maxlen,freq,&sd,stream);
  const long long n1 = x->n;
  fgb_gix_free(x);
  if (rc) return rc;
  if (stats) memset(stats,0,sizeof(*stats));
  rc = extend_and_filter(sd,A,A,freq4,chain_break,chain_min,align_min,align_rate,out,stats,NULL,NULL,stream);
  if (rc) return rc;
  if (stats) stats->nkmers1 = stats->nkmers2 = n1;
  return FGB_OK;
}

extern "C" int fgb_fastga(const unsigned char *bpsA, long long nbA, int ncA, const long long *clenA,
                          const long long *boffA, const float *freqA,
                          const unsigned char *bpsB, long long nbB, int ncB, const long long *clenB,
                          const long long *boffB,
                          int freq, int chain_break, int chain_min, int align_min, double align_rate,
                          fgb_alns **out, fgb_run_stats *stats, void *stream)
{ fgb_genome *A = NULL, *B = NULL;
  int rc;
  if ((rc = fgb_genome_create(bpsA,nbA,ncA,clenA,boffA,1,&A,stream))) return rc;
  if ((rc = fgb_genome_create(bpsB,nbB,ncB,clenB,boffB,0,&B,stream))) { fgb_genome_free(A); return rc; }
  rc = fgb_align_resident(A,B,freqA,freq,chain_break,chain_min,align_min,align_rate,out,stats,stream);
  fgb_genome_free(A); fgb_genome_free(B);
  return rc;
}
