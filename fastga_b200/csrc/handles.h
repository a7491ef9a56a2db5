// Opaque handle layouts behind the C-ABI (include/fastga_b200.h only forward-declares them), and
// the per-stage device timings.
#pragma once
#include <cuda_runtime.h>
#include <vector>

struct fgb_timings            // device milliseconds per stage (CUDA events on the call's stream)
{ float h2d_ms, stage_ms, scan_ms, ksort_ms, index_ms, merge_ms, ssort_ms, triples_ms, extend_ms,
        d2h_ms, filter_ms;
  int   merge_launches, extend_launches, launches;
};

extern fgb_timings g_timings;             // fgb_timings_get / fgb_timings_reset

//  Adds the device time of the work issued on `s` during its lifetime to *d (one of the g_timings
//  fields); waits for that work when it ends.
struct stage_timer
{ cudaEvent_t a, b; cudaStream_t st; float *dst;
  stage_timer(float *d, cudaStream_t s) : st(s), dst(d)
    { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a,st); }
  ~stage_timer()
    { cudaEventRecord(b,st); cudaEventSynchronize(b);
      float ms = 0; cudaEventElapsedTime(&ms,a,b); *dst += ms;
      cudaEventDestroy(a); cudaEventDestroy(b);
    }
};

struct fgb_genome
{ int ncontig = 0;
  long long seqtot = 0, maxlen = 0, total_words = 0, h2d_bytes = 0;
  std::vector<long long> clen, boff, woff;
  std::vector<int> perm, crank;            // perm[rank] = contig, crank[contig] = rank
  long long *d_clen = nullptr, *d_woff = nullptr;
  int *d_crank = nullptr, *d_perm = nullptr;
  unsigned long long *d_seq = nullptr, *d_rseq = nullptr;
};

struct fgb_gix
{ long long n = 0;
  struct rec128 *d_tab = nullptr;
  unsigned *d_pstart = nullptr;            // [2^24+1] lower-bound index by 12-base prefix
  unsigned char *d_adj = nullptr;          // [n+32] LCP in bases of entries i-1 and i (0 at the table ends)
  unsigned long long buck1024[1024] = {0}; // sampler histogram (decides the .ktab part split)
  int post_bytes = 0, cont_bytes = 0, ncontig = 0;
  int fwd_only = 0;                        // forward-strand entries only (adaptamer side of a merge)
  long long n_both = 0;                    // entries of the both-strand table (= n unless fwd_only)
};

struct fgb_seeds
{ long long n = 0, sumlen = 0;
  struct rec128 *d_rec = nullptr;          // sorted seed records
  int anti_bits = 0, band_bits = 0, jc_bits = 0, ic_bits = 0;
  long long amxpos = 0, bmxpos = 0;
  int self_mode = 0;                       // seeds of a genome against itself (FastGA A)
  long long n1_merged = 0;                 // forward-strand T1 entries the merge consumed
};
