// GIX construction on the device: genome staging, closed (12,8)-syncmer scan, k-mer record
// build, prefix index + LCP, and conversion from/to the on-disk .ktab entry format.
//
// Replaces (reference file:line):
//   sample_thread / scan_thread      GIXmake.c:164-328, 406-611    -> syncmer_{count,emit}_kernel
//   setup_thread_plain               GIXmake.c:802-980             -> emit of 128-bit records
//   msd_sort                         MSDsort.c:404                 -> sort128.cu (10 byte passes)
//   compress_thread / k_sort writer  GIXmake.c:1211-1278,1300-1596 -> kix_index/ktab_export kernels
//   Kmer_Stream reader               libfastk.c:785-1313           -> ktab_import_kernel
#include "common.cuh"

// 4-mer hash map of the syncmer sampler.  This is data, not code: it defines which positions
// are indexed, so it must be value-identical to GIXmake.c:92-109 (TMap) for on-disk parity.
static const unsigned char h_TMap[256] =
  { 0xff,0xd4,0xf5,0xfd,0xe4,0xad,0x21,0xa5,0xed,0x64,0xbf,0xa9,0xf3,0x70,0xd6,0xf0,
    0xca,0x89,0xcb,0xc9,0x82,0x9d,0x13,0x79,0x0a,0x0f,0x25,0x19,0x3e,0x47,0xa3,0xa8,
    0xf9,0x5e,0xe8,0xa1,0xb0,0x71,0x1d,0x8c,0xde,0x69,0xe7,0x7c,0x56,0x3f,0x90,0xa4,
    0xeb,0x45,0x59,0xf1,0x97,0x4c,0x08,0xa0,0xb8,0x4a,0x86,0xc8,0xcd,0x98,0x7d,0xfc,
    0xef,0x4d,0x83,0x7e,0xdc,0x66,0x2b,0x8e,0xe0,0xa7,0xd0,0xa2,0x88,0x5f,0x7f,0xd9,
    0x9b,0x78,0xd1,0x8b,0xc3,0x8f,0x2d,0xe6,0x18,0x27,0x2c,0x24,0x94,0xb7,0xce,0xbd,
    0x0d,0x04,0x1c,0x09,0x16,0x23,0x00,0x1e,0x1a,0x29,0x2e,0x15,0x01,0x10,0x2a,0x20,
    0xbe,0x31,0x43,0x58,0xc2,0xaa,0x1f,0xe5,0xc5,0x9e,0xcf,0xc6,0x68,0xb2,0x80,0xf4,
    0xf8,0x53,0xb6,0x93,0x76,0x37,0x11,0x40,0xda,0x51,0xba,0x46,0x42,0x30,0x60,0x6d,
    0x5c,0x39,0x9f,0x48,0x6c,0x62,0x28,0x67,0x06,0x12,0x26,0x0e,0x33,0x50,0xa6,0x63,
    0xdd,0x3b,0xab,0x4b,0x72,0x5b,0x22,0x6f,0xb4,0x61,0x92,0x99,0x36,0x38,0x65,0xac,
    0x4f,0x2f,0x32,0x44,0x54,0x3c,0x03,0x5d,0x73,0x3a,0x77,0x84,0x8d,0x4e,0x49,0xd2,
    0xfb,0x91,0x6a,0xcc,0x8a,0x35,0x02,0x55,0x7a,0x34,0x96,0x3d,0xd3,0x41,0x85,0xf2,
    0xb1,0x75,0xc4,0xb5,0xbb,0xb3,0x1b,0xd5,0x07,0x05,0x17,0x0b,0x7b,0xd7,0xdf,0xea,
    0xe3,0x57,0xc0,0x95,0x9c,0x6e,0x14,0xae,0xb9,0x6b,0xc1,0x81,0x87,0x74,0xd8,0xe2,
    0xec,0x52,0xbc,0xe9,0xe1,0xdb,0x0c,0xf7,0xaf,0x5a,0x9a,0xc7,0xfa,0xf6,0xee,0xfe };

// Tables indexed by a little-endian packed 4-mer x (first base in the LOW two bits, as in .bps):
//   c_TN[x] = TMap[first-base-high packing of the 4-mer]
//   c_TC[x] = TMap[first-base-high packing of its reverse complement]
__constant__ unsigned char c_TN[256];
__constant__ unsigned char c_TC[256];

static int tables_ready = 0;

static int init_tables()
{ if (tables_ready) return FGB_OK;
  unsigned char tn[256], tc[256];
  for (int x = 0; x < 256; x++)
    { int b0 = x & 3, b1 = (x>>2) & 3, b2 = (x>>4) & 3, b3 = (x>>6) & 3;    // bases in order
      int fwd = (b0<<6) | (b1<<4) | (b2<<2) | b3;
      int rc  = ((3-b3)<<6) | ((3-b2)<<4) | ((3-b1)<<2) | (3-b0);
      tn[x] = h_TMap[fwd];
      tc[x] = h_TMap[rc];
    }
  CUDA_TRY(cudaMemcpyToSymbol(c_TN,tn,256));
  CUDA_TRY(cudaMemcpyToSymbol(c_TC,tc,256));
  tables_ready = 1;
  return FGB_OK;
}

typedef unsigned long long u64;

//  64 bits (32 bases) of a packed contig starting at base offset boff (may be < 0 or run past
//    the end: bases outside [0,32*nw) read as 0).  w = contig's first 64-bit word.

static __device__ __forceinline__ u64 bases64(const u64 *__restrict__ w, long long nw, long long boff)
{ long long q = boff >> 5;              // floor
  int s = (int) (boff & 31) << 1;
  u64 a = (q >= 0 && q < nw) ? w[q] : 0ull;
  if (s == 0) return a;
  u64 b = (q+1 >= 0 && q+1 < nw) ? w[q+1] : 0ull;
  return (a >> s) | (b << (64-s));
}

//  reverse the order of the 32 two-bit groups of x
static __device__ __forceinline__ u64 rev2(u64 x)
{ x = __brevll(x);
  return ((x & 0x5555555555555555ull) << 1) | ((x >> 1) & 0x5555555555555555ull);
}

/***********************************************************************************************
 *  Genome staging: .bps image (contig c at byte boff[c], COMPRESSED_LEN(len) bytes,
 *  gene_core.c:349-400) -> 16-byte aligned, zero-padded 64-bit words per contig; optional
 *  reverse-complement copy (what Complement_Seq + Get_Contig give align_contigs for strand C,
 *  FastGA.c:3179-3185).
 **********************************************************************************************/

__global__ void stage_contigs_kernel(const unsigned char *__restrict__ bps,
                                     const long long *__restrict__ boff,
                                     const long long *__restrict__ clen,
                                     const long long *__restrict__ woff, int ncontig,
                                     u64 *__restrict__ seq, long long total_words)
{ long long g = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total_words) return;
  int lo = 0, hi = ncontig-1;                     // last contig with woff <= g
  while (lo < hi)
    { int m = (lo+hi+1) >> 1;
      if (woff[m] <= g) lo = m; else hi = m-1;
    }
  long long q = g - woff[lo];
  long long nbytes = (clen[lo]+3) >> 2;
  long long b0 = q*8;
  u64 v = 0;
  if (boff[lo] >= 0 && q >= 0)
    { const unsigned char *p = bps + boff[lo];
      for (int i = 0; i < 8; i++)
        if (b0+i < nbytes)
          v |= (u64) p[b0+i] << (8*i);
      long long lim = clen[lo] - q*32;            // valid bases in this word
      if (lim < 32) v &= (lim <= 0) ? 0ull : ((1ull << (2*lim)) - 1);
    }
  seq[g] = v;
}

__global__ void revcomp_contigs_kernel(const u64 *__restrict__ seq, const long long *__restrict__ clen,
                                       const long long *__restrict__ woff, int ncontig,
                                       u64 *__restrict__ rseq, long long total_words)
{ long long g = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= total_words) return;
  int lo = 0, hi = ncontig-1;
  while (lo < hi)
    { int m = (lo+hi+1) >> 1;
      if (woff[m] <= g) lo = m; else hi = m-1;
    }
  long long q = g - woff[lo];
  long long L = clen[lo];
  long long nw = (lo+1 < ncontig ? woff[lo+1] : total_words) - woff[lo];
  if (q < 0) { rseq[g] = 0; return; }
  //  output bases i = 32q .. 32q+31 : out[i] = 3 - in[L-1-i]  ->  in bases L-32-32q .. L-1-32q
  u64 e = bases64(seq + woff[lo],nw,L - 32 - 32*q);
  u64 v = ~rev2(e);
  long long lim = L - q*32;
  if (lim < 32) v &= (lim <= 0) ? 0ull : ((1ull << (2*lim)) - 1);
  rseq[g] = v;
}

/***********************************************************************************************
 *  Syncmer scan.  A 12-mer at j is sampled iff the minimum of the canonical hashes of its five
 *  8-mers sits at the first or the last one, ties included -- the local form of the running
 *  min4/pos4 automaton of GIXmake.c:516-567.  Forward 40-mer seq[j,j+40) if j <= len-40
 *  (:571-578); reverse entry = revcomp(seq[j-28,j+12)) with post j+12 if j >= 28 (:579-586,
 *  :929-940).  One thread handles SC_PPT consecutive positions out of one 64-bit window.
 **********************************************************************************************/

#define SC_THREADS 256
#define SC_PPT     16
#define SC_TILE    (SC_THREADS*SC_PPT)          // 4096 positions per block
#define SC_WORDS   (SC_TILE/32 + 3)             // staged 64-bit words: [t0-32, t0+SC_TILE+64)

static __device__ __forceinline__ u64 sm_bases64(const u64 *sw, int boff)   // boff >= 0, staged
{ int q = boff >> 5, s = (boff & 31) << 1;
  u64 a = sw[q];
  if (s == 0) return a;
  return (a >> s) | (sw[q+1] << (64-s));
}

//  select mask (bit i set iff position p+i is a sampled syncmer start), i < SC_PPT

static __device__ __forceinline__ unsigned syncmer_mask(u64 E, const unsigned char *tn,
                                                        const unsigned char *tc)
{ unsigned hn[SC_PPT+8], hc[SC_PPT+8];
#pragma unroll
  for (int i = 0; i < SC_PPT+8; i++)
    { unsigned x = (unsigned) (E >> (2*i)) & 0xff;
      hn[i] = tn[x];
      hc[i] = tc[x];
    }
  unsigned mz[SC_PPT+4];
#pragma unroll
  for (int i = 0; i < SC_PPT+4; i++)
    { unsigned mn = (hn[i] << 8) | hn[i+4];
      unsigned mc = hc[i] | (hc[i+4] << 8);
      mz[i] = mn < mc ? mn : mc;
    }
  unsigned sel = 0;
#pragma unroll
  for (int i = 0; i < SC_PPT; i++)
    { unsigned m = min(min(min(mz[i],mz[i+1]),min(mz[i+2],mz[i+3])),mz[i+4]);
      if (mz[i] == m || mz[i+4] == m) sel |= 1u << i;
    }
  return sel;
}

template<int EMIT> __global__ void __launch_bounds__(SC_THREADS)
syncmer_kernel(const u64 *__restrict__ seq, const long long *__restrict__ clen,
               const long long *__restrict__ woff, const int *__restrict__ crank,
               const int *__restrict__ tile_contig, const int *__restrict__ tile_start,
               unsigned *__restrict__ tile_count,       // EMIT=0: out counts; EMIT=1: in offsets
               unsigned long long *__restrict__ buck1024,
               rec128 *__restrict__ out, int fwd_only)
{ __shared__ u64 sw[SC_WORDS+1];
  __shared__ unsigned char tn[256], tc[256];
  __shared__ unsigned wsum[SC_THREADS/32];
  __shared__ unsigned hist[1024];

  int tid = threadIdx.x;
  int c   = tile_contig[blockIdx.x];
  int t0  = tile_start[blockIdx.x];
  long long L  = clen[c];
  const u64 *w = seq + woff[c];
  long long nw = (L + 31) >> 5;

  tn[tid] = c_TN[tid];
  tc[tid] = c_TC[tid];
  if (EMIT == 0)
    for (int i = tid; i < 1024; i += SC_THREADS) hist[i] = 0;
  for (int i = tid; i < SC_WORDS+1; i += SC_THREADS)
    { long long gw = (t0 >> 5) - 1 + i;
      sw[i] = (gw >= 0 && gw < nw) ? w[gw] : 0ull;
    }
  __syncthreads();

  int p = t0 + tid*SC_PPT;                     // first position of this thread
  int sb = 32 + tid*SC_PPT;                    // its base offset inside the staged window
  unsigned sel = 0;
  if ((long long) p + 12 <= L)
    { sel = syncmer_mask(sm_bases64(sw,sb),tn,tc);
      long long lastok = L - 12 - p;           // positions p+i valid for i <= lastok
      if (lastok < SC_PPT-1) sel &= (2u << lastok) - 1;
    }

  //  how many records does this thread emit (fwd if j <= L-40, rev if j >= 28)
  unsigned fmask = sel, rmask = sel;
  { long long fl = L - 40 - p;                 // fwd ok for i <= fl
    if (fl < 0) fmask = 0; else if (fl < SC_PPT-1) fmask &= (2u << fl) - 1;
    int rl = 28 - p;                           // rev ok for i >= rl
    if (rl > 0) rmask = (rl >= SC_PPT) ? 0 : (rmask & ~((1u << rl) - 1));
  }
  //  fwd_only: forward-strand entries only (the table is only ever the adaptamer side of a merge,
  //  where reverse entries never seed, FastGA.c:921-928)
  unsigned rdropped = 0;                       // reverse entries a forward-only table leaves out
  if (fwd_only) { rdropped = __popc(rmask); rmask = 0; }
  unsigned cnt = __popc(fmask) + __popc(rmask);

  int lane = tid & 31, wp = tid >> 5;
  unsigned inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
    { unsigned t = __shfl_up_sync(0xffffffffu,inc,o);
      if (lane >= o) inc += t;
    }
  if (lane == 31) wsum[wp] = inc;
  __syncthreads();
  unsigned pre = 0, tot = 0;
  for (int i = 0; i < SC_THREADS/32; i++)
    { if (i < wp) pre += wsum[i];
      tot += wsum[i];
    }

  if (EMIT == 0)
    { //  10-bit first-5-bases histogram over ALL sampled positions, both strands, as
      //  sample_thread does (GIXmake.c:318-320); decides the .ktab part split (:669-691).
      unsigned m = sel;
      while (m)
        { int i = __ffs(m)-1;
          m &= m-1;
          u64 f = sm_bases64(sw,sb+i);                        // bases j..j+31
          unsigned fb = (unsigned) (rev2(f) >> 54);           // first five bases, base j high
          u64 r = sm_bases64(sw,sb+i+7);                      // bases j+7..
          unsigned rb = (unsigned) ((~r) & 0x3ff);            // comp of bases j+7..j+11, j+11 high
          //  revcomp first five = comp(j+11),comp(j+10),...,comp(j+7): base j+11 in top bits
          unsigned rr = 0;
#pragma unroll
          for (int k = 0; k < 5; k++)
            rr |= ((rb >> (2*k)) & 3) << (2*k);               // LE: j+7 low ... j+11 high == wanted
          atomicAdd(&hist[fb],1u);
          atomicAdd(&hist[rr],1u);
        }
      __syncthreads();
      for (int i = tid; i < 1024; i += SC_THREADS)
        if (hist[i]) atomicAdd(&buck1024[i],(unsigned long long) hist[i]);
      if (fwd_only)                            // slot 1024: size of the both-strand table minus this one
        { rdropped = __reduce_add_sync(0xffffffffu,rdropped);
          if (lane == 0 && rdropped) atomicAdd(&buck1024[1024],(unsigned long long) rdropped);
        }
      if (tid == 0) tile_count[blockIdx.x] = tot;
      return;
    }

  long long o = (long long) tile_count[blockIdx.x] + pre + inc - cnt;
  unsigned cr = (unsigned) crank[c];
  unsigned m = fmask | rmask;
  while (m)
    { int i = __ffs(m)-1;
      m &= m-1;
      int j = p + i;
      if (fmask >> i & 1)
        { u64 e0 = sm_bases64(sw,sb+i);
          u64 e1 = sm_bases64(sw,sb+i+32);
          rec128 r;
          r.hi = rev2(e0);
          r.lo = (rev2(e1) & 0xffff000000000000ull) | ((u64) cr << 32) | (unsigned) j;
          st_rec(out + o,r);
          o += 1;
        }
      if (rmask >> i & 1)
        { u64 e0 = sm_bases64(sw,sb+i-28);                    // bases s..s+31, s = j-28
          u64 e1 = sm_bases64(sw,sb+i+4) & 0xffffull;         // bases s+32..s+39
          rec128 r;
          r.hi = ~((e1 << 48) | (e0 >> 16));
          r.lo = ((~e0 & 0xffffull) << 48) | ((u64) (cr | 0x8000u) << 32) | (unsigned) (j+12);
          st_rec(out + o,r);
          o += 1;
        }
    }
}

/***********************************************************************************************
 *  Prefix index + LCP over the sorted table (compress_thread, GIXmake.c:1235-1261):
 *    pstart[x] = first entry whose 12-base prefix is >= x, pstart[2^24] = n.
 **********************************************************************************************/

__global__ void kix_index_kernel(const rec128 *__restrict__ tab, long long n,
                                 unsigned *__restrict__ pstart, unsigned char *__restrict__ adj)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  rec128 a, b;
  a.lo = a.hi = b.lo = b.hi = 0;
  if (i > 0) a = ld_rec(tab + i - 1);
  if (i < n) b = ld_rec(tab + i);
  //  the two open ends (everything up to the first prefix, everything above the last one) are
  //  filled by kix_ends_kernel with full parallelism: a slice of a sharded table covers only part
  //  of the prefix space, and one thread writing millions of index entries would take 60 ms
  if (i > 0 && i < n)
    { long long plo = (long long) KREC_PREFIX24(a.hi), phi = (long long) KREC_PREFIX24(b.hi);
      for (long long x = plo+1; x <= phi; x++)
        pstart[x] = (unsigned) i;
    }
  //  adj[i] = LCP in bases of entries i-1 and i (the LCP byte of the reference's .ktab entries,
  //  GIXmake.c:1249-1254), 0 at both ends of the table: the merge takes block extents from it
  int l = 0;
  if (i > 0 && i < n)
    { unsigned long long x = a.hi ^ b.hi;
      if (x) l = __clzll(x) >> 1;
      else
        { unsigned y = (unsigned) ((a.lo ^ b.lo) >> 48);
          l = y ? 32 + ((__clz(y) - 16) >> 1) : 40;
        }
    }
  adj[i] = (unsigned char) l;
}

static __device__ __forceinline__ int krec_lcp(const rec128 &a, const rec128 &b)
{ u64 x = a.hi ^ b.hi;
  if (x) return __clzll(x) >> 1;
  unsigned y = (unsigned) ((a.lo ^ b.lo) >> 48);
  if (y) return 32 + ((__clz(y) - 16) >> 1);
  return 40;
}

//  .ktab entry (GIXmake.c:1235-1261): [7 B bases 12..39][mask prefix len][lcp][post LE][contig LE
//    | strand in the top bit of the last byte].  LCP is the true LCP in bases with the previous
//    entry of the same part, 40 for an exact duplicate, and 0 for the first entry of a part
//    (MSDsort.c:485-506); part_first marks those (sorted list of entry indices).

__global__ void ktab_export_kernel(const rec128 *__restrict__ tab, long long n, int pbytes,
                                   int cbytes, const long long *__restrict__ part_first, int nparts,
                                   unsigned char *__restrict__ out)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rec128 r = tab[i];
  int lcp = 0;
  bool first = false;
  for (int p = 0; p < nparts; p++)
    if (part_first[p] == i) first = true;
  if (!first)
    lcp = krec_lcp(tab[i-1],r);
  int E = 9 + pbytes + cbytes;
  unsigned char *o = out + i*E;
  u64 suf = KREC_SUFFIX56(r);
  for (int k = 0; k < 7; k++)
    o[k] = (unsigned char) (suf >> (8*(6-k)));
  o[7] = 0;
  o[8] = (unsigned char) lcp;
  unsigned post = (unsigned) r.lo;
  for (int k = 0; k < pbytes; k++)
    o[9+k] = (unsigned char) (post >> (8*k));
  unsigned cs = (unsigned) (r.lo >> 32) & 0xffff;
  unsigned cv = (cs & 0x7fff) | ((cs >> 15) << (8*cbytes-1));
  for (int k = 0; k < cbytes; k++)
    o[9+pbytes+k] = (unsigned char) (cv >> (8*k));
}

//  Inverse: entries + cumulative index (stub layout libfastk.c:815-840) -> device records.

__global__ void ktab_import_kernel(const unsigned char *__restrict__ ent, long long n, int pbytes,
                                   int cbytes, const long long *__restrict__ index /* [2^24] cumulative */,
                                   rec128 *__restrict__ tab)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int lo = 0, hi = (1<<24)-1;                      // smallest x with index[x] > i
  while (lo < hi)
    { int m = (lo+hi) >> 1;
      if (index[m] > i) hi = m; else lo = m+1;
    }
  int E = 9 + pbytes + cbytes;
  const unsigned char *e = ent + i*E;
  u64 suf = 0;
  for (int k = 0; k < 7; k++)
    suf = (suf << 8) | e[k];
  unsigned post = 0;
  for (int k = 0; k < pbytes; k++)
    post |= (unsigned) e[9+k] << (8*k);
  unsigned cv = 0;
  for (int k = 0; k < cbytes; k++)
    cv |= (unsigned) e[9+pbytes+k] << (8*k);
  unsigned sign = cv >> (8*cbytes-1);
  unsigned cs = (cv & ((1u << (8*cbytes-1)) - 1)) | (sign << 15);
  rec128 r;
  r.hi = ((u64) lo << 40) | (suf >> 16);
  r.lo = ((suf & 0xffffull) << 48) | ((u64) cs << 32) | post;
  st_rec(tab + i,r);
}

/***********************************************************************************************
 *  Host-callable pieces (device pointers in, device pointers out).
 **********************************************************************************************/

extern "C" int fgb_sort128_device(void *d_a, void *d_b, long long n, int byte_lo, int byte_hi,
                                  void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream);
extern "C" long long fgb_sort128_tmp_bytes(long long n);

extern "C" int fgb_stage_genome_device(const void *d_bps, const long long *d_boff,
                                       const long long *d_clen, const long long *d_woff,
                                       int ncontig, long long total_words, void *d_seq,
                                       void *d_rseq /* may be NULL */, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (total_words <= 0) return FGB_OK;
  int nb = (int) ((total_words + 255) / 256);
  stage_contigs_kernel<<<nb,256,0,st>>>((const unsigned char *) d_bps,d_boff,d_clen,d_woff,ncontig,
                                        (u64 *) d_seq,total_words);
  if (d_rseq != NULL)
    revcomp_contigs_kernel<<<nb,256,0,st>>>((const u64 *) d_seq,d_clen,d_woff,ncontig,
                                            (u64 *) d_rseq,total_words);
  fgb_count_launch(d_rseq != NULL ? 2 : 1);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}

//  Pass 1 of the scan: per-tile record counts (then scanned in place to offsets), 1024-bin
//  sampler histogram, and the total number of records in *h_total.

extern "C" int fgb_syncmer_count_device(const void *d_seq, const long long *d_clen,
                                        const long long *d_woff, const int *d_crank,
                                        const int *d_tile_contig, const int *d_tile_start, int ntiles,
                                        unsigned *d_tile_count, unsigned long long *d_buck1024,
                                        unsigned long long *d_total, void *d_tmp, long long tmp_bytes,
                                        int fwd_only, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  int rc = init_tables();
  if (rc) return rc;
  CUDA_TRY(cudaMemsetAsync(d_buck1024,0,1025*8,st));
  if (ntiles > 0)
    syncmer_kernel<0><<<ntiles,SC_THREADS,0,st>>>((const u64 *) d_seq,d_clen,d_woff,d_crank,
                                                   d_tile_contig,d_tile_start,d_tile_count,
                                                   d_buck1024,NULL,fwd_only);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  return fgb_dev_exclusive_scan_u32(d_tile_count,ntiles,d_total,d_tmp,tmp_bytes,st);
}

extern "C" int fgb_syncmer_emit_device(const void *d_seq, const long long *d_clen,
                                       const long long *d_woff, const int *d_crank,
                                       const int *d_tile_contig, const int *d_tile_start, int ntiles,
                                       unsigned *d_tile_offset, void *d_records, int fwd_only,
                                       void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (ntiles > 0)
    syncmer_kernel<1><<<ntiles,SC_THREADS,0,st>>>((const u64 *) d_seq,d_clen,d_woff,d_crank,
                                                   d_tile_contig,d_tile_start,d_tile_offset,
                                                   NULL,(rec128 *) d_records,fwd_only);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}

//  d_adj: n + 32 bytes (entries past n are zeroed: the merge's slice loads run up to 31 bytes over)
__global__ void kix_ends_kernel(const rec128 *__restrict__ tab, long long n, unsigned *__restrict__ pstart)
{ long long x = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (x > (1ll << 24)) return;
  if (n == 0) { pstart[x] = 0; return; }
  long long p0 = (long long) KREC_PREFIX24(tab[0].hi), pl = (long long) KREC_PREFIX24(tab[n-1].hi);
  if (x <= p0) pstart[x] = 0;
  else if (x > pl) pstart[x] = (unsigned) n;
}

extern "C" int fgb_kix_index_device(const void *d_tab, long long n, unsigned *d_pstart, unsigned char *d_adj,
                                    void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  int nb = (int) ((n + 1 + 255) / 256);
  CUDA_TRY(cudaMemsetAsync(d_adj + n,0,32,st));
  kix_index_kernel<<<nb,256,0,st>>>((const rec128 *) d_tab,n,d_pstart,d_adj);
  kix_ends_kernel<<<((1 << 24) + 256)/256,256,0,st>>>((const rec128 *) d_tab,n,d_pstart);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}

extern "C" int fgb_ktab_export_device(const void *d_tab, long long n, int pbytes, int cbytes,
                                      const long long *d_part_first, int nparts, void *d_out,
                                      void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n <= 0) return FGB_OK;
  int nb = (int) ((n + 255) / 256);
  ktab_export_kernel<<<nb,256,0,st>>>((const rec128 *) d_tab,n,pbytes,cbytes,d_part_first,nparts,
                                      (unsigned char *) d_out);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}

extern "C" int fgb_ktab_import_device(const void *d_ent, long long n, int pbytes, int cbytes,
                                      const long long *d_index, void *d_tab, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n <= 0) return FGB_OK;
  int nb = (int) ((n + 255) / 256);
  ktab_import_kernel<<<nb,256,0,st>>>((const unsigned char *) d_ent,n,pbytes,cbytes,d_index,
                                      (rec128 *) d_tab);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}

extern "C" int fgb_sc_tile() { return SC_TILE; }
