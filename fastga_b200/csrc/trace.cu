// Trace points -> explicit edit scripts on the device.
//
// Replaces (reference file:line):
//   Compute_Trace_PTS              align.c:6171-6308   (mode GREEDIEST, unbounded band: every caller
//                                                       of the path uses it that way, ALNtoPAF.c:272)
//   iter_np                        align.c:5584-5903   the O(NP) aligner run on every trace-point tile
//
// A .1aln record pins its alignment every 100 A-bases (trace points); between two trace points the
// exact edit script is recomputed on demand.  Tiles are independent (about 100 x 100 bases, as many
// waves as the tile has differences), and inside a tile the O(NP) recurrence is a serial chain -- a
// furthest point depends on its neighbour of the SAME wave -- so the unit of parallel work is one
// THREAD per tile: millions of tiles, each a few thousand instructions.  A tile keeps its waves
// (furthest B-index per diagonal, int16) and move codes (int8) in a private slab of HBM sized from
// the tile's own difference count (the optimum never needs more waves than the trace point
// recorded differences), reads the 2-bit staged contigs through L1, and leaves its indel positions
// in a per-tile slot; the host strings the slots of an alignment together in order.
//
// What must be reproduced exactly (it decides WHERE an indel is placed among equal-cost scripts):
// the order in which a wave is filled (above the end diagonal downwards, below it upwards, the end
// diagonal last), the tie order of the three-way choice, and the pointer-reversal read-out.
#include "common.cuh"
#include "handles.h"
#include <vector>
#include <string.h>

typedef unsigned long long u64;

struct TileJob                      // one trace-point tile
{ unsigned aln;                     // alignment it belongs to
  int a0, m;                        // A interval [a0,a0+m) in contig coordinates
  int b0, n;                        // B interval (complemented-B coordinates for strand C)
  int dcap;                         // waves available: recorded differences - |m-n|
  unsigned out;                     // first slot of its script entries
  u64 slab;                         // byte offset of its wave slab
};

struct AlnSeq { long long aw, bw; int alen, blen; };      // word offsets of the two contigs (B: of the strand's copy)

static __device__ __forceinline__ int base2(const unsigned *__restrict__ w, int i)
{ return (int) (__ldg(w + (i >> 4)) >> ((i & 15) << 1)) & 3; }

//  slab layout: rows D = -2 .. dcap of `width` int16 furthest points, then rows 0 .. dcap of int8
//  move codes; column of diagonal k is k - kmin
static __host__ __device__ __forceinline__ int tile_width(int m, int n, int dcap)
{ int del = m - n; if (del < 0) del = -del;
  return del + 2*(dcap/2 + 1) + 4;
}
static __host__ __device__ __forceinline__ u64 tile_slab_bytes(int m, int n, int dcap)
{ u64 w = (u64) tile_width(m,n,dcap);
  return (((u64) (dcap+3)*w*2 + (u64) (dcap+1)*w) + 15) & ~15ull;
}

__global__ void __launch_bounds__(128)
trace_tiles_kernel(const TileJob *__restrict__ jobs, int njobs, const AlnSeq *__restrict__ seqs,
                   const u64 *__restrict__ aseq, const u64 *__restrict__ bseq, const u64 *__restrict__ brseq,
                   const unsigned char *__restrict__ comp, unsigned char *__restrict__ slabs,
                   int *__restrict__ script, int *__restrict__ count, int *__restrict__ tdiffs)
{ const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= njobs) return;
  const TileJob J = jobs[t];
  const AlnSeq  S = seqs[J.aln];
  const unsigned *A = (const unsigned *) (aseq + S.aw);
  const unsigned *B = (const unsigned *) ((comp[J.aln] ? brseq : bseq) + S.bw);
  const int M = J.m, N = J.n, del = M - N;
  const int W = tile_width(M,N,J.dcap);
  int lo = del < 0 ? del : 0, hi = del < 0 ? 0 : del;
  const int kmin = lo - (J.dcap/2 + 1) - 1;
  short *F = (short *) (slabs + J.slab);
  signed char *H = (signed char *) (F + (size_t) (J.dcap+3) * W);
#define FROW(D) (F + (size_t) ((D)+2) * W - kmin)
#define HROW(D) (H + (size_t) (D) * W - kmin)

  { short *f2 = FROW(-2), *f1 = FROW(-1);
    for (int k = lo-1; k <= hi+1; k++) f2[k] = f1[k] = -2;
    f1[0] = -1;
  }
  lo += 1; hi -= 1;
  int D;
  for (D = 0; ; D++)
    { if (D > J.dcap) { count[t] = -1; tdiffs[t] = 0; return; }      // trace point inconsistent with the sequences
      const short *f2 = FROW(D-2), *f1 = FROW(D-1);
      short *f0 = FROW(D);
      signed char *hf = HROW(D);
      if ((D & 1) == 0) { lo -= 1; hi += 1; }
      f0[hi+1] = f0[lo-1] = -2;
      //  one furthest point: best of (k-1 | k | k+1) in the wave's tie order, then slide
#define CELL(K,AM,AP,MDIR,PDIR)                                               \
      { const int ac = f1[K] + 1, am = (AM), ap = (AP); int code;             \
        if (ac < am) { if (ap < am) { code = MDIR; j = am; } else { code = PDIR; j = ap; } } \
        else         { if (ap < ac) { code = 0;    j = ac; } else { code = PDIR; j = ap; } } \
        const int lim = (N < M - (K)) ? N : M - (K);                          \
        while (j < lim && base2(B,J.b0 + j) == base2(A,J.a0 + (K) + j)) j += 1; \
        hf[K] = (signed char) code; f0[K] = (short) j;                        \
      }
      int j = -2;
      for (int k = hi; k > del; k--)  CELL(k,f2[k-1],j+1,-1,4)
      j = -2;
      for (int k = lo; k < del; k++)  CELL(k,j,f2[k+1]+1,2,1)
      CELL(del,j,f0[del+1]+1,2,4)
#undef CELL
      if (f0[del] >= N) break;
    }

  //  read-out: reverse the move pointers from the end cell back to the origin ...
  HROW(0)[0] = 3;
  int k = del, e = HROW(D)[k];
  HROW(D)[k] = 3;
  while (e != 3)
    { int h = k + e;
      if (e > 1) h -= 3; else if (e == 0) D -= 1; else D -= 2;
      const int nx = HROW(D)[h];
      HROW(D)[h] = (signed char) e;
      e = nx; k = h;
    }
  //  ... then walk them forward, one script entry per change of diagonal (align.c:5865-5895):
  //  +(B position + 1) where A has an extra base ahead of it, -(A position + 1) where B has one
  int *out = script + J.out, no = 0;
  k = 0; D = 0; e = HROW(0)[0];
  while (e != 3)
    { int h = k - e;
      const int c = FROW(D)[k];
      if (e > 1) h += 3; else if (e == 0) D += 1; else D += 2;
      if (h > k)      out[no++] = J.b0 + 1 + c;
      else if (h < k) out[no++] = -(J.a0 + 1) - (c + k);
      k = h;
      e = HROW(D)[h];
    }
  count[t] = no;
  tdiffs[t] = D + (del < 0 ? -del : del);
#undef FROW
#undef HROW
}

struct fgb_scripts
{ long long n = 0;
  std::vector<long long> soff;      // n+1 offsets into script
  std::vector<int> script, diffs;
  long long bad = 0;                // alignments whose trace points contradict the sequences
};

extern "C" void fgb_scripts_free(fgb_scripts *s) { delete s; }
extern "C" long long fgb_scripts_count(const fgb_scripts *s) { return s->n; }
extern "C" long long fgb_scripts_total(const fgb_scripts *s) { return (long long) s->script.size(); }
extern "C" long long fgb_scripts_bad(const fgb_scripts *s) { return s->bad; }
extern "C" int fgb_scripts_get(const fgb_scripts *s, long long *soff, int *script, int *diffs)
{ memcpy(soff,s->soff.data(),sizeof(long long)*s->soff.size());
  if (!s->script.empty()) memcpy(script,s->script.data(),sizeof(int)*s->script.size());
  if (!s->diffs.empty()) memcpy(diffs,s->diffs.data(),sizeof(int)*s->diffs.size());
  return FGB_OK;
}

//  fields / toff / pool: alignments as fgb_alns_get returns them (n x 9 ints: comp aread bread abpos
//  bbpos aepos bepos diffs tlen; B coordinates of strand-C records in complemented B, as in the
//  .1aln).  B must have been created with its reverse complement when any record is strand C.
//  The script of alignment i is script[soff[i] .. soff[i+1]): what Compute_Trace_PTS leaves in
//  path->trace (align.h:330-349), diffs[i] what it leaves in path->diffs (-1: bad trace points).
extern "C" int fgb_compute_trace_pts(const fgb_genome *A, const fgb_genome *B, long long n, const int *fields,
                                     const long long *toff, const unsigned char *pool, int tspace,
                                     fgb_scripts **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n < 0 || tspace <= 0) return FGB_ERR_ARG;
  owner<fgb_scripts> own(new fgb_scripts(),fgb_scripts_free);
  fgb_scripts *R = own.get();
  R->n = n;
  R->soff.assign(n+1,0);
  R->diffs.assign(n,0);
  if (n == 0) { *out = own.release(); return FGB_OK; }

  std::vector<TileJob> jobs;
  std::vector<AlnSeq> seqs(n);
  std::vector<unsigned char> comp(n);
  std::vector<long long> first(n+1);            // first tile of every alignment
  u64 slab = 0; unsigned long long slots = 0;
  for (long long i = 0; i < n; i++)
    { const int *f = fields + 9*i;
      const unsigned char *tr = pool + toff[i];
      const int ar = f[1], br = f[2], tlen = f[8];
      if (ar < 0 || ar >= A->ncontig || br < 0 || br >= B->ncontig) return FGB_ERR_ARG;
      if (f[0] && B->d_rseq == NULL) return FGB_ERR_ARG;
      comp[i] = (unsigned char) (f[0] != 0);
      seqs[i].aw = A->woff[ar]; seqs[i].bw = B->woff[br];
      seqs[i].alen = (int) A->clen[ar]; seqs[i].blen = (int) B->clen[br];
      first[i] = (long long) jobs.size();
      const int ntile = tlen >= 2 ? tlen/2 : 1;
      int a = f[3], b = f[4];
      for (int t = 0; t < ntile; t++)
        { const bool last = (t == ntile-1);
          const int ae = last ? f[5] : (f[3]/tspace)*tspace + (t+1)*tspace;
          const int be = last ? f[6] : b + tr[2*t+1];
          const int d  = tlen >= 2 ? tr[2*t] : f[7];
          TileJob J;
          J.aln = (unsigned) i; J.a0 = a; J.m = ae - a; J.b0 = b; J.n = be - b;
          if (J.m < 0 || J.n < 0 || ae > seqs[i].alen || be > seqs[i].blen) return FGB_ERR_ARG;
          int del = J.m - J.n; if (del < 0) del = -del;
          J.dcap = d > del ? d - del : 0;
          J.out = (unsigned) slots; J.slab = slab;
          slots += (unsigned long long) (J.dcap + del);
          slab += tile_slab_bytes(J.m,J.n,J.dcap);
          jobs.push_back(J);
          a = ae; b = be;
        }
    }
  first[n] = (long long) jobs.size();
  if (slots >= 0xfffffff0ull || jobs.size() >= 0x7ffffff0ull) return FGB_ERR_LIMIT;

  const int nj = (int) jobs.size();
  TileJob *d_jobs = NULL; AlnSeq *d_seqs = NULL; unsigned char *d_comp = NULL, *d_slab = NULL;
  int *d_script = NULL, *d_count = NULL, *d_td = NULL;
  dev_scope S(st); S.own(d_jobs); S.own(d_seqs); S.own(d_comp); S.own(d_slab); S.own(d_script); S.own(d_count); S.own(d_td);
  std::vector<int> cnt(nj), td(nj), scr((size_t) slots + 1);
  CUDA_TRY(fgb_dmalloc((void **) &d_jobs,sizeof(TileJob)*(size_t) nj,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_seqs,sizeof(AlnSeq)*(size_t) n,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_comp,(size_t) n,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_slab,(size_t) slab + 16,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_script,sizeof(int)*((size_t) slots + 1),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_count,sizeof(int)*(size_t) nj,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_td,sizeof(int)*(size_t) nj,st));
  CUDA_TRY(cudaMemcpyAsync(d_jobs,jobs.data(),sizeof(TileJob)*(size_t) nj,cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemcpyAsync(d_seqs,seqs.data(),sizeof(AlnSeq)*(size_t) n,cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemcpyAsync(d_comp,comp.data(),(size_t) n,cudaMemcpyHostToDevice,st));
  trace_tiles_kernel<<<(nj + 127)/128,128,0,st>>>(d_jobs,nj,d_seqs,A->d_seq,B->d_seq,B->d_rseq,d_comp,d_slab,
                                                  d_script,d_count,d_td);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(cnt.data(),d_count,sizeof(int)*(size_t) nj,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaMemcpyAsync(td.data(),d_td,sizeof(int)*(size_t) nj,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaMemcpyAsync(scr.data(),d_script,sizeof(int)*(size_t) slots,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  //  string the tiles of every alignment together
  R->script.reserve((size_t) slots);
  for (long long i = 0; i < n; i++)
    { int diffs = 0; bool bad = false;
      R->soff[i] = (long long) R->script.size();
      for (long long t = first[i]; t < first[i+1]; t++)
        { if (cnt[t] < 0) { bad = true; break; }
          R->script.insert(R->script.end(),scr.begin() + jobs[t].out,scr.begin() + jobs[t].out + cnt[t]);
          diffs += td[t];
        }
      if (bad) { R->script.resize((size_t) R->soff[i]); diffs = -1; R->bad += 1; }
      R->diffs[i] = diffs;
    }
  R->soff[n] = (long long) R->script.size();
  *out = own.release();
  return FGB_OK;
}
