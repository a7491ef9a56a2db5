// Adaptive-seed ("adaptamer") merge of two sorted k-mer tables, fused with the seed-record
// transform of the re-import step.
//
// Replaces new_merge_thread (FastGA.c:610-1025) + adaptamer_merge (:2281-2493) and the per-pair
// arithmetic of reimport_thread (:2703-2721).  The reference co-walks T1 and a per-12-mer cache
// of T2 with an LCP-driven state machine; its result is the declarative rule (SURVEY A.3):
//   for every forward-strand T1 entry e1 whose 12-base panel is non-empty in T2,
//     plen  = max over the panel of LCP(e1,e2)            (12..40)
//     R(e1) = the block of T2 entries with LCP(e1,e2) >= plen
//     if |R| < FREQ emit (plen, e1, e2) for every e2 in R, strand C iff e2 is a reverse entry.
//
// Tiled co-scan: T1 is a FORWARD-STRAND-ONLY table (reverse entries never seed; the fused path
// builds it that way, any other table is compacted once).  A CTA owns TILE consecutive T1 entries;
// because both tables are sorted, the T2 entries they can match are ONE contiguous slice.  Both the
// tile and the slice arrive by TMA bulk copy on one mbarrier and stay in record form (the 128-bit
// record orders as (k-mer, payload), so a probe is one 128-bit shared-memory load and compare);
// every T1 entry finds its insertion point with a few probes inside its panel (bounds from the
// 2^24 prefix index, read through L1); a neighbour sharing fewer than 12 bases is "no partner".
// Seeds are expanded load-balanced: each entry drops one 32-bit descriptor per seed into shared
// memory, then every thread builds one 128-bit seed record per step and the stores of the CTA are
// one contiguous run reserved with ONE atomic.
#include "common.cuh"
#include "handles.h"

typedef unsigned long long u64;

struct seed_layout                 // bit positions inside the 128-bit seed record
{ int anti_bits;                   // lcp [0,6) drem [6,12) anti [12,12+anti_bits) band ... jcont ... icont ... comp
  int band_bits;
  int jc_bits;
  int ic_bits;
  long long amxpos, bmxpos;        // longest contig of genome 1 / genome 2 (FastGA.c:5023-5041)
};

static __host__ __device__ __forceinline__ int seed_key_bits(const seed_layout &L)
{ return 12 + L.anti_bits + L.band_bits + L.jc_bits + L.ic_bits + 1; }

#define MG_THREADS 256
#define MG_WARPS   (MG_THREADS/32)
#ifndef MG_T2CAP
#define MG_T2CAP   1152                   // staged T2 entries per CTA (18 KB)
#endif
#ifndef MG_DCAP
#define MG_DCAP    1536                   // seed descriptors per CTA (3 per T1 entry; crowded tiles write entry-wise)
#endif
#ifndef MG_MINBLK
#define MG_MINBLK  6
#define MG_PCAP    512                    // staged words of the prefix index per CTA (the tile's prefix span + 2)
#endif
//  lcp (in bases, 0..28) of two 56-bit suffixes
static __device__ __forceinline__ int lcp56(u64 a, u64 b)
{ u64 x = a ^ b;
  return x ? ((__clzll(x) - 8) >> 1) : 28;
}

//  lcp (in bases, 0..40) of the k-mers of two records
static __device__ __forceinline__ int lcp_rec(const rec128 &a, const rec128 &b)
{ u64 x = a.hi ^ b.hi;
  if (x) return __clzll(x) >> 1;
  unsigned y = (unsigned) ((a.lo ^ b.lo) >> 48);
  return y ? 32 + ((__clz(y) - 16) >> 1) : 40;
}

static __device__ __forceinline__ u64 suffix_of(const rec128 *__restrict__ T, unsigned i)
{ uint4 v = *reinterpret_cast<const uint4 *>(T + i);
  u64 lo = (u64) v.x | ((u64) v.y << 32);
  u64 hi = (u64) v.z | ((u64) v.w << 32);
  return ((hi & 0xffffffffffull) << 16) | (lo >> 48);
}

struct seed_pack                          // kernel-uniform packing constants
{ int p_band, s_jc, s_ic, s_cp;           // band position; shifts inside the upper word
  long long amxpos, bmxpos, maxdag;
};

//  seed record of (plen, T1 payload, T2 payload); payload = post | (contig rank | strand<<15) << 32
//  (reimport_thread, FastGA.c:2703-2721)
static __device__ __forceinline__ rec128 make_seed(unsigned plen, u64 pay, u64 p2, const seed_pack &K)
{ long long ipost = (long long) (unsigned) pay, jpost = (long long) (unsigned) p2;
  unsigned icont = (unsigned) (pay >> 32) & 0x7fff;
  unsigned cs = (unsigned) (p2 >> 32) & 0xffff;
  unsigned comp = cs >> 15, jcont = cs & 0x7fff;
  long long diag, anti;
  if (comp) { diag = K.maxdag - (ipost + jpost); anti = K.amxpos - (ipost - jpost); }
  else      { diag = K.bmxpos + (ipost - jpost); anti = ipost + jpost; }
  u64 X = (u64) plen | ((u64) (diag & 63) << 6) | ((u64) anti << 12);
  u64 Y = (u64) (diag >> 6) | ((u64) jcont << K.s_jc) | ((u64) icont << K.s_ic)
                            | ((u64) comp << K.s_cp);
  rec128 sd;
  sd.lo = X | (Y << K.p_band);
  sd.hi = Y >> (64 - K.p_band);
  return sd;
}

template<int TILE> struct mg_stage
{ rec128   t2[MG_T2CAP];                  // the T2 slice (TMA destination)
  rec128   t1[TILE];                      // the T1 tile (TMA destination)
  unsigned desc[MG_DCAP];                 // per seed: T2 slot (11) | T1 slot (9) << 11 | (plen-12) << 20
  unsigned wtot[2*MG_WARPS], wsum[2*MG_WARPS];
  unsigned char adj[MG_T2CAP+48];         // LCP bytes of the slice (TMA destination; starts at the 16-byte boundary below the slice)
  unsigned pst[MG_PCAP];                  // prefix index of the tile's prefix span (TMA destination)
  unsigned rng[4];
  unsigned long long gbase;
  unsigned long long bar;
};

//  Adaptamer of one T1 entry against the staged slice: |R| (0 if no seed), first slice slot of R, plen.
//  Written for the WARP, not the lane: the panel search runs a warp-uniform number of predicated
//  halving steps (no divergent loop), and the extent of R comes from the table's adjacent-entry LCP
//  bytes (adj[i] = LCP(t2[i-1],t2[i]), the LCP byte of the reference's .ktab entries; T2 is sorted, so
//  t2[i-1] belongs to R iff t2[i] does and adj[i] >= plen): two predicated steps per side, then a
//  warp-uniform loop.  The bytes either side of the slice belong to other panels (< 12) and end every walk.
static __device__ __forceinline__ unsigned adaptamer_staged(const rec128 *__restrict__ t2,
                                                            const unsigned char *__restrict__ adj, unsigned nsl,
                                                            const rec128 &r1, unsigned lo, unsigned hi, int freq,
                                                            unsigned &lowi, int &plen)
{ const unsigned k1 = (unsigned) (r1.lo >> 48);
  const u64 *t2w = reinterpret_cast<const u64 *>(t2);
  unsigned a = lo, b = hi;                                    // lower bound of r1's k-mer inside its panel [lo,hi)
  for (unsigned w = __reduce_max_sync(0xffffffffu,hi - lo); w > 0; w >>= 1)
    { const unsigned m = (a + b) >> 1;                        // a == b: a probe with no effect
      const u64 qh = t2w[2*m+1];
      const unsigned ql = (unsigned) (t2w[2*m] >> 48);
      const bool less = (qh < r1.hi) || (qh == r1.hi && ql < k1);
      const bool live = a < b;
      if (live && less) a = m+1;
      if (live && !less) b = m;
    }
  //  the neighbours of the insertion point decide plen; a neighbour in another panel (the slice only
  //  holds the tile's panels, so this covers the slice ends too) shares fewer than 12 bases
  int ll = 0, lr = 0;
  if (lo < hi)
    { if (a > 0)   ll = lcp_rec(r1,ld_rec(t2 + a - 1));
      if (a < nsl) lr = lcp_rec(r1,ld_rec(t2 + a));
    }
  const int m = ll > lr ? ll : lr;
  const unsigned fq = (unsigned) freq;
  unsigned lft = a, rgt = a;
  bool goL = (m >= 12 && ll == m), goR = (m >= 12 && lr == m);
  if (goL) lft = a-1;
  if (goR) rgt = a+1;
  //  each side on its own up to FREQ members: |R| >= FREQ is all that matters beyond that (:799-823)
#pragma unroll
  for (int u = 0; u < 2; u++)
    { goL = goL && a - lft < fq && (int) adj[lft] >= m;
      if (goL) lft -= 1;
      goR = goR && rgt - a < fq && (int) adj[rgt] >= m;
      if (goR) rgt += 1;
    }
  while (__any_sync(0xffffffffu,goL || goR))
    { goL = goL && a - lft < fq && (int) adj[lft] >= m;
      if (goL) lft -= 1;
      goR = goR && rgt - a < fq && (int) adj[rgt] >= m;
      if (goR) rgt += 1;
    }
  lowi = lft; plen = m;
  return (m >= 12 && rgt - lft < fq) ? rgt - lft : 0u;
}

//  eight bytes from a byte address in shared memory (three aligned words, two funnel shifts)
static __device__ __forceinline__ u64 adj8(const unsigned char *p)
{ const unsigned sa = smem_u32((const void *) p);
  const unsigned *w = reinterpret_cast<const unsigned *>(p - (sa & 3u));
  const unsigned sh = (sa & 3u) << 3;
  const unsigned w0 = w[0], w1 = w[1], w2 = w[2];
  return (u64) __funnelshift_r(w0,w1,sh) | ((u64) __funnelshift_r(w1,w2,sh) << 32);
}

//  The same for N entries per lane at once (the CTA's rounds): the N searches advance in lock step, so
//  every dependent shared-memory probe of one has the probes of the others to overlap with.
template<int N>
static __device__ __forceinline__ void adaptamer_staged_n(const rec128 *__restrict__ t2,
                                                          const unsigned char *__restrict__ adj, unsigned nsl,
                                                          const rec128 (&r1)[N], const unsigned (&lo)[N],
                                                          const unsigned (&hi)[N], int freq,
                                                          unsigned (&cnt)[N], unsigned (&lowi)[N], int (&plen)[N])
{ const u64 *t2w = reinterpret_cast<const u64 *>(t2);
  const unsigned fq = (unsigned) freq;
  unsigned a[N], b[N], wmax = 0;
  u64 k1[N];
#pragma unroll
  for (int r = 0; r < N; r++)
    { a[r] = lo[r]; b[r] = hi[r]; wmax = max(wmax,hi[r] - lo[r]);
      k1[r] = (r1[r].hi << 24) | ((r1[r].lo >> 48) << 8);
    }
  for (unsigned w = __reduce_max_sync(0xffffffffu,wmax); w > 0; w >>= 1)
    {
#pragma unroll
      for (int r = 0; r < N; r++)
        { const unsigned m = (a[r] + b[r]) >> 1;                // a == b: a probe with no effect
          //  inside a panel the first 12 bases agree: the other 28 (56 bits) order the entries
          const u64 qk = (t2w[2*m+1] << 24) | ((t2w[2*m] >> 48) << 8);
          const bool less = qk < k1[r];
          const bool live = a[r] < b[r];
          if (live && less) a[r] = m+1;
          if (live && !less) b[r] = m;
        }
    }
  int m[N]; unsigned lft[N], rgt[N]; bool goL[N], goR[N], any = false;
#pragma unroll
  for (int r = 0; r < N; r++)
    { int ll = 0, lr = 0;
      if (lo[r] < hi[r])
        { if (a[r] > 0)   ll = lcp_rec(r1[r],ld_rec(t2 + a[r] - 1));
          if (a[r] < nsl) lr = lcp_rec(r1[r],ld_rec(t2 + a[r]));
        }
      m[r] = ll > lr ? ll : lr;
      lft[r] = rgt[r] = a[r];
      goL[r] = (m[r] >= 12 && ll == m[r]); goR[r] = (m[r] >= 12 && lr == m[r]);
      if (goL[r]) lft[r] = a[r]-1;
      if (goR[r]) rgt[r] = a[r]+1;
    }
  //  Extent of the block either side of the insertion point, EIGHT LCP bytes at a time: t2[i-1] is in R
  //  iff t2[i] is and adj[i] >= m, so a side extends by the run of bytes >= m next to it (one SIMD byte
  //  compare + a bit scan; the bytes beyond a panel end are < 12 and stop every run, whatever lies
  //  past them), capped at FREQ members a side (|R| >= FREQ is all that matters beyond, :799-823).
#pragma unroll
  for (int r = 0; r < N; r++)
    { const unsigned mm = (unsigned) m[r] * 0x01010101u;
      unsigned L = 0, R = 0;
      { const u64 v = adj8(adj + (int) a[r] - 8);                      // bytes a-8 .. a-1, the nearest on top
        const u64 ge = (u64) __vcmpgeu4((unsigned) v,mm) | ((u64) __vcmpgeu4((unsigned) (v >> 32),mm) << 32);
        L = (~ge) ? (unsigned) (__clzll((long long) ~ge) >> 3) : 8u;
      }
      { const u64 v = adj8(adj + a[r] + 1);                            // bytes a+1 .. a+8, the nearest at the bottom
        const u64 ge = (u64) __vcmpgeu4((unsigned) v,mm) | ((u64) __vcmpgeu4((unsigned) (v >> 32),mm) << 32);
        R = (~ge) ? (unsigned) ((__ffsll((long long) ~ge) - 1) >> 3) : 8u;
      }
      if (goL[r]) lft[r] -= min(L,fq - 1);
      if (goR[r]) rgt[r] += min(R,fq - 1);
      goL[r] = goL[r] && L == 8 && fq > 9;                              // a longer run: the loop below (rare)
      goR[r] = goR[r] && R == 8 && fq > 9;
    }
#pragma unroll
  for (int r = 0; r < N; r++) any = any || goL[r] || goR[r];
  while (__any_sync(0xffffffffu,any))
    { any = false;
#pragma unroll
      for (int r = 0; r < N; r++)
        { goL[r] = goL[r] && a[r] - lft[r] < fq && (int) adj[lft[r]] >= m[r];
          if (goL[r]) lft[r] -= 1;
          goR[r] = goR[r] && rgt[r] - a[r] < fq && (int) adj[rgt[r]] >= m[r];
          if (goR[r]) rgt[r] += 1;
          any = any || goL[r] || goR[r];
        }
    }
#pragma unroll
  for (int r = 0; r < N; r++)
    { lowi[r] = lft[r]; plen[r] = m[r];
      cnt[r] = (m[r] >= 12 && rgt[r] - lft[r] < fq) ? rgt[r] - lft[r] : 0u;
    }
}

//  Same straight from HBM (a tile whose slice does not fit the staging buffers: long repeats).
static __device__ __forceinline__ unsigned adaptamer_direct(const rec128 *__restrict__ T2,
                                                            const unsigned *__restrict__ pstart, const rec128 &r1,
                                                            int freq, unsigned &lowi, int &plen)
{ unsigned p  = KREC_PREFIX24(r1.hi);
  unsigned lo = pstart[p], hi = pstart[p+1];
  lowi = 0; plen = 0;
  if (lo >= hi) return 0;
  u64 s1 = KREC_SUFFIX56(r1);
  unsigned a = lo, b = hi;
  while (a < b)
    { unsigned m = (a + b) >> 1;
      if (suffix_of(T2,m) < s1) a = m+1; else b = m;
    }
  int ll = (a > lo) ? lcp56(s1,suffix_of(T2,a-1)) : -1;
  int lr = (a < hi) ? lcp56(s1,suffix_of(T2,a))   : -1;
  int m  = ll > lr ? ll : lr;
  plen = 12 + m;
  unsigned lft = a, rgt = a;
  int sh = 56 - 2*m;
  u64 key = s1 >> sh;
  while (lft > lo && rgt - lft < (unsigned) freq)
    { if ((suffix_of(T2,lft-1) >> sh) != key) break;
      lft -= 1;
    }
  while (rgt < hi && rgt - lft < (unsigned) freq)
    { if ((suffix_of(T2,rgt) >> sh) != key) break;
      rgt += 1;
    }
  if (rgt - lft >= (unsigned) freq) return 0;
  lowi = lft;
  return rgt - lft;
}

//  Per CTA of the merge: the prefix span of its T1 tile and the T2 slice it can match, found ahead
//  of the merge with full parallelism (inside the merge this would be a chain of two dependent HBM
//  round trips made by one lane while 255 threads wait).
__global__ void merge_ranges_kernel(const rec128 *__restrict__ T1, unsigned n1, const unsigned *__restrict__ pstart2,
                                    unsigned per_block, unsigned nblocks, uint4 *__restrict__ rng)
{ unsigned b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nblocks) return;
  unsigned long long b0 = (unsigned long long) b * per_block, b1 = b0 + per_block - 1;
  if (b1 >= n1) b1 = n1 - 1;
  unsigned pA = KREC_PREFIX24(T1[b0].hi), pB = KREC_PREFIX24(T1[b1].hi);
  unsigned lo2 = pstart2[pA], hi2 = pstart2[pB+1];
  rng[b] = make_uint4(pA,pB - pA,lo2,hi2 - lo2);
}

template<int TILE>
__global__ void __launch_bounds__(MG_THREADS,MG_MINBLK)
adaptamer_merge_kernel(const rec128 *__restrict__ T1, unsigned n1,
                       const rec128 *__restrict__ T2, const unsigned *__restrict__ pstart2,
                       const unsigned char *__restrict__ adj2, const uint4 *__restrict__ rng, int freq, seed_pack K,
                       rec128 *__restrict__ seeds, unsigned long long capacity,
                       unsigned long long *__restrict__ counters /* [0]=nseeds [1]=sum plen */)
{ extern __shared__ __align__(16) unsigned char mg_smem[];
  mg_stage<TILE> *S = reinterpret_cast<mg_stage<TILE> *>(mg_smem);
  constexpr int ROUNDS = (TILE >= MG_THREADS) ? TILE/MG_THREADS : 1;
  const int tid = threadIdx.x, lane = tid & 31, wp = tid >> 5;
  const unsigned long long b0 = (unsigned long long) blockIdx.x * TILE;
  const unsigned nt1 = (n1 - b0 < (unsigned long long) TILE) ? (unsigned) (n1 - b0) : (unsigned) TILE;

  if (tid == 0)
    { const uint4 r = rng[blockIdx.x];                      // pA, pB-pA, first T2 entry, #T2 entries
      S->rng[0] = r.x; S->rng[1] = r.y; S->rng[2] = r.z; S->rng[3] = r.w;
      mbar_init(&S->bar,1);
      const bool st = (r.w <= MG_T2CAP);
      //  LCP bytes of the slice and one beyond, from the 16-byte boundary at or below the slice start
      const unsigned ab = ((r.z & 15u) + r.w + 1u + 15u) & ~15u;
      //  prefix index words pA .. pB+1 (panel bounds of every tile entry), from the 16-byte boundary below pA
      const unsigned pw = ((r.x & 3u) + r.y + 2u + 3u) & ~3u;
      const bool sp = (pw <= MG_PCAP);
      mbar_expect_tx(&S->bar,nt1*16u + ((st && r.w) ? r.w*16u + ab + (sp ? pw*4u : 0u) : 0u));
      tma_copy_1d(S->t1,T1 + b0,nt1*16u,&S->bar);
      if (st && r.w)
        { tma_copy_1d(S->t2,T2 + r.z,r.w*16u,&S->bar);
          tma_copy_1d(S->adj,adj2 + (r.z & ~15u),ab,&S->bar);
          if (sp) tma_copy_1d(S->pst,pstart2 + (r.x & ~3u),pw*4u,&S->bar);
        }
    }
  __syncthreads();
  const unsigned lo2 = S->rng[2], nsl = S->rng[3];
  const bool staged = (nsl <= MG_T2CAP);
  mbar_wait(&S->bar,0);
  const unsigned char *const adj = S->adj + (lo2 & 15u);       // adj[i]: slice entries i-1 and i

  //  search: thread tid owns tile entries tid, tid+256, ...
  const u64 *t2k = reinterpret_cast<const u64 *>(S->t2);
  const u64 *t1k = reinterpret_cast<const u64 *>(S->t1);
  const u64 PAY = 0xffffffffffffull;
  unsigned cnt[ROUNDS], lowi[ROUNDS], excl[ROUNDS]; int plen[ROUNDS];
  if (staged)
    { //  all 32 lanes take part (warp-uniform search steps); lanes past the tile search nothing
      rec128 r1[ROUNDS]; unsigned lo[ROUNDS], hi[ROUNDS];
      const unsigned pbase = S->rng[0] & ~3u;
      const bool sp = nsl > 0 && (((S->rng[0] & 3u) + S->rng[1] + 2u + 3u) & ~3u) <= MG_PCAP;   // prefix span staged (else: HBM)
#pragma unroll
      for (int r = 0; r < ROUNDS; r++)
        { const unsigned j = r*MG_THREADS + tid;
          r1[r].lo = r1[r].hi = 0; lo[r] = hi[r] = 0;
          if (j < nt1)
            { r1[r] = ld_rec(&S->t1[j]);
              const unsigned p = KREC_PREFIX24(r1[r].hi);
              if (sp) { lo[r] = S->pst[p - pbase] - lo2; hi[r] = S->pst[p - pbase + 1] - lo2; }
              else    { lo[r] = __ldg(pstart2 + p) - lo2; hi[r] = __ldg(pstart2 + p + 1) - lo2; }
            }
        }
      adaptamer_staged_n<ROUNDS>(S->t2,adj,nsl,r1,lo,hi,freq,cnt,lowi,plen);
    }
  else
    {
#pragma unroll
      for (int r = 0; r < ROUNDS; r++)
        { const unsigned j = r*MG_THREADS + tid;
          cnt[r] = 0; lowi[r] = 0; plen[r] = 0;
          if (j < nt1) cnt[r] = adaptamer_direct(T2,pstart2,ld_rec(&S->t1[j]),freq,lowi[r],plen[r]);
        }
    }
  //  Offsets of every entry's seeds inside the CTA's run (round 0 of all warps, then round 1).  The counts
  //  of the two rounds ride one register through the scans, 16 bits each: an entry yields < FREQ <= 255
  //  seeds (FastGA.c:4960), a round of the CTA < 256 * 255.
  static_assert(ROUNDS <= 2,"two packed rounds at most");
  unsigned total = 0;
  { unsigned pk = cnt[0], sl = cnt[0] * (unsigned) plen[0];
    if (ROUNDS == 2) { pk |= cnt[ROUNDS-1] << 16; sl += cnt[ROUNDS-1] * (unsigned) plen[ROUNDS-1]; }
    unsigned inc = pk;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
      { const unsigned t = __shfl_up_sync(0xffffffffu,inc,o);
        if (lane >= o) inc += t;
      }
    sl = __reduce_add_sync(0xffffffffu,sl);
    if (lane == 31) S->wtot[wp] = inc;
    if (lane == 0)  S->wsum[wp] = sl;
    __syncthreads();
    //  across the warps: eight packed totals scanned by the first eight lanes of every warp
    const unsigned v = (lane < MG_WARPS) ? S->wtot[lane] : 0u;
    unsigned winc = v;
#pragma unroll
    for (int o = 1; o < MG_WARPS; o <<= 1)
      { const unsigned t = __shfl_up_sync(0xffffffffu,winc,o);
        if (lane >= o) winc += t;
      }
    const unsigned all = __shfl_sync(0xffffffffu,winc,MG_WARPS-1);     // CTA totals of the two rounds
    const unsigned mine = __shfl_sync(0xffffffffu,winc - v,wp);        // ... of the warps before this one
    const unsigned t0 = all & 0xffffu;
    total = t0 + (all >> 16);
    excl[0] = (inc & 0xffffu) - cnt[0] + (mine & 0xffffu);
    if (ROUNDS == 2) excl[ROUNDS-1] = (inc >> 16) - cnt[ROUNDS-1] + t0 + (mine >> 16);
  }
  const bool fast = staged && total <= MG_DCAP;
  if (fast)
    {
#pragma unroll
      for (int r = 0; r < ROUNDS; r++)
        { const unsigned d = lowi[r] | ((unsigned) (r*MG_THREADS + tid) << 11) | ((unsigned) (plen[r] - 12) << 20);
          for (unsigned k = 0; k < cnt[r]; k++) S->desc[excl[r] + k] = d + k;
        }
    }
  //  ONE atomic per CTA reserves its output run (per-warp atomics on the single counter serialise in L2)
  if (tid == 0)
    { unsigned long long q = 0, g = 0;
      for (int k = 0; k < MG_WARPS; k++) q += S->wsum[k];
      if (total) { g = atomicAdd(&counters[0],(unsigned long long) total); atomicAdd(&counters[1],q); }
      S->gbase = g;
    }
  __syncthreads();
  if (total == 0) return;
  const unsigned long long gbase = S->gbase;
  if (fast)
    { for (unsigned o = tid; o < total; o += MG_THREADS)
        { const unsigned d = S->desc[o];
          const u64 p2 = t2k[2*(d & 2047u)] & PAY, p1 = t1k[2*((d >> 11) & 511u)] & PAY;
          if (gbase + o < capacity) st_rec(seeds + gbase + o,make_seed(12u + (d >> 20),p1,p2,K));
        }
      return;
    }
  //  slow path (unstaged tile or more seeds than descriptors): every entry writes its own seeds
#pragma unroll
  for (int r = 0; r < ROUNDS; r++)
    { const unsigned j = r*MG_THREADS + tid;
      if (cnt[r] == 0) continue;
      const u64 p1 = t1k[2*j] & PAY;
      for (unsigned k = 0; k < cnt[r]; k++)
        { const u64 p2 = (staged ? t2k[2*(lowi[r]+k)] : T2[lowi[r]+k].lo) & PAY;
          const unsigned long long o = gbase + excl[r] + k;
          if (o < capacity) st_rec(seeds + o,make_seed((unsigned) plen[r],p1,p2,K));
        }
    }
}

//  Forward-strand view of a both-strand table (order kept): flags -> exclusive scan -> scatter.
__global__ void fwd_flag_kernel(const rec128 *__restrict__ T, long long n, unsigned *__restrict__ flag)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = (unsigned) (((T[i].lo >> 47) & 1) ^ 1);
}
__global__ void fwd_scatter_kernel(const rec128 *__restrict__ T, long long n, const unsigned *__restrict__ pos,
                                   rec128 *__restrict__ out)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rec128 r = ld_rec(T + i);
  if (((r.lo >> 47) & 1) == 0) st_rec(out + pos[i],r);
}

//  d_out: room for n records.  *h_nfwd = number of forward-strand entries written.
extern "C" int fgb_forward_view_device(const void *d_T, long long n, void *d_out, long long *h_nfwd, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  *h_nfwd = 0;
  if (n <= 0) return FGB_OK;
  unsigned *d_flag = NULL; void *d_tmp = NULL; unsigned long long *d_total = NULL;
  dev_scope S(st); S.own(d_flag); S.own(d_tmp); S.own(d_total);
  long long tmpb = fgb_dev_scan_tmp_bytes(n);
  CUDA_TRY(fgb_dmalloc((void **) &d_flag,sizeof(unsigned)*(n+1),st));
  CUDA_TRY(fgb_dmalloc(&d_tmp,tmpb,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_total,8,st));
  int nb = (int) ((n + 255) / 256);
  fwd_flag_kernel<<<nb,256,0,st>>>((const rec128 *) d_T,n,d_flag);
  int rc = fgb_dev_exclusive_scan_u32(d_flag,n,d_total,d_tmp,tmpb,st);
  if (rc) return rc;
  fwd_scatter_kernel<<<nb,256,0,st>>>((const rec128 *) d_T,n,d_flag,(rec128 *) d_out);
  fgb_count_launch(2);
  unsigned long long tot = 0;
  CUDA_TRY(cudaMemcpyAsync(&tot,d_total,8,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  *h_nfwd = (long long) tot;
  return FGB_OK;
}

/***********************************************************************************************
 *  SELF mode (FastGA A): new_self_merge_thread (FastGA.c:1616-1909).  One table; EVERY entry,
 *  either strand, is an i.  plen = its longest prefix shared with another entry of its 12-base
 *  panel = max of the LCPs with its two neighbours; block = the run of entries sharing those plen
 *  bases, the entry included; if the block has < FREQ members, one seed (i, p) for every OTHER
 *  member p, strand C iff the signs differ.  One thread per entry: no search, its own index is
 *  the insertion point.  Output run of a block reserved with one atomic.
 **********************************************************************************************/

static __device__ __forceinline__ int lcp_full(const rec128 &a, const rec128 &b)      // bases, 0..40
{ u64 x = a.hi ^ b.hi;
  if (x) return __clzll(x) >> 1;
  unsigned y = (unsigned) ((a.lo ^ b.lo) >> 48);
  if (y) return 32 + ((__clz(y) - 16) >> 1);
  return 40;
}

__global__ void __launch_bounds__(256)
self_merge_kernel(const rec128 *__restrict__ T, unsigned n, const unsigned *__restrict__ pstart,
                  int freq, seed_pack K, rec128 *__restrict__ seeds, unsigned long long capacity,
                  unsigned long long *__restrict__ counters)
{ __shared__ unsigned s_w[8], s_l[8];
  __shared__ unsigned long long s_base;
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const unsigned i = blockIdx.x * 256u + threadIdx.x;
  unsigned lo = i, hi = i, cnt = 0;
  int plen = 0;
  rec128 e; e.lo = e.hi = 0;
  if (i < n)
    { e = ld_rec(T + i);
      unsigned p = KREC_PREFIX24(e.hi);
      unsigned cbeg = pstart[p], cend = pstart[p+1];
      int lp = (i > cbeg)   ? lcp_full(ld_rec(T + i - 1),e) : 11;
      int ls = (i+1 < cend) ? lcp_full(e,ld_rec(T + i + 1)) : 11;
      plen = lp > ls ? lp : ls;
      if (plen >= 12)
        { lo = i; hi = i+1;
          while (lo > cbeg && i - lo < (unsigned) freq && lcp_full(ld_rec(T + lo - 1),ld_rec(T + lo)) >= plen) lo -= 1;
          while (hi < cend && hi - lo < (unsigned) freq && lcp_full(ld_rec(T + hi - 1),ld_rec(T + hi)) >= plen) hi += 1;
          if (hi - lo < (unsigned) freq) cnt = hi - lo - 1;
        }
    }
  unsigned inc = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
    { unsigned t = __shfl_up_sync(0xffffffffu,inc,o);
      if (lane >= o) inc += t;
    }
  unsigned slen = __reduce_add_sync(0xffffffffu,cnt * (unsigned) plen);
  if (lane == 31) { s_w[wp] = inc; s_l[wp] = slen; }
  __syncthreads();
  if (threadIdx.x == 0)
    { unsigned long long t = 0, q = 0;
      for (int k = 0; k < 8; k++) { t += s_w[k]; q += s_l[k]; }
      s_base = t ? atomicAdd(&counters[0],t) : 0ull;
      if (q) atomicAdd(&counters[1],q);
    }
  __syncthreads();
  if (cnt == 0) return;
  unsigned long long o = s_base + (inc - cnt);
  for (int k = 0; k < wp; k++) o += s_w[k];
  const long long ipost = (long long) (unsigned) e.lo;
  const unsigned icont = (unsigned) (e.lo >> 32) & 0x7fff, isign = (unsigned) (e.lo >> 47) & 1;
  for (unsigned q = lo; q < hi; q++)
    { if (q == i) continue;
      rec128 r2 = ld_rec(T + q);
      long long jpost = (long long) (unsigned) r2.lo;
      unsigned cs = (unsigned) (r2.lo >> 32) & 0xffff;
      unsigned comp = (cs >> 15) ^ isign, jcont = cs & 0x7fff;
      long long diag, anti;
      if (comp) { diag = K.maxdag - (ipost + jpost); anti = K.amxpos - (ipost - jpost); }
      else      { diag = K.bmxpos + (ipost - jpost); anti = ipost + jpost; }
      u64 X = (u64) (unsigned) plen | ((u64) (diag & 63) << 6) | ((u64) anti << 12);
      u64 Y = (u64) (diag >> 6) | ((u64) jcont << K.s_jc) | ((u64) icont << K.s_ic)
                                | ((u64) comp << K.s_cp);
      rec128 sd;
      sd.lo = X | (Y << K.p_band);
      sd.hi = Y >> (64 - K.p_band);
      if (o < capacity) st_rec(seeds + o,sd);
      o += 1;
    }
}

extern "C" int fgb_self_merge_device(const void *d_T, long long n, const unsigned *d_pstart, int freq,
                                     int anti_bits, int band_bits, int jc_bits, int ic_bits,
                                     long long amxpos, void *d_seeds, long long capacity,
                                     unsigned long long *d_counters, unsigned long long *h_nseeds,
                                     unsigned long long *h_sumlen, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  seed_layout L;
  L.anti_bits = anti_bits; L.band_bits = band_bits; L.jc_bits = jc_bits; L.ic_bits = ic_bits;
  L.amxpos = amxpos; L.bmxpos = amxpos;
  if (seed_key_bits(L) > 128 || freq < 1 || freq > 255) return FGB_ERR_LIMIT;
  if (n >= 0xffffffffll) return FGB_ERR_LIMIT;
  CUDA_TRY(cudaMemsetAsync(d_counters,0,16,st));
  seed_pack K;
  K.p_band = 12 + anti_bits;
  K.s_jc = band_bits; K.s_ic = band_bits + jc_bits; K.s_cp = band_bits + jc_bits + ic_bits;
  K.amxpos = amxpos; K.bmxpos = amxpos; K.maxdag = 2*amxpos;
  if (K.s_cp + 1 > 64 || K.p_band >= 64 || K.p_band < 13) return FGB_ERR_LIMIT;
  if (n > 0)
    { self_merge_kernel<<<(unsigned) ((n + 255) / 256),256,0,st>>>((const rec128 *) d_T,(unsigned) n,d_pstart,freq,K,
                                                                  (rec128 *) d_seeds,(unsigned long long) capacity,d_counters);
      fgb_count_launch(1);
    }
  CUDA_TRY(cudaGetLastError());
  unsigned long long h[2];
  CUDA_TRY(cudaMemcpyAsync(h,d_counters,16,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  *h_nseeds = h[0];
  if (h_sumlen) *h_sumlen = h[1];
  return (h[0] > (unsigned long long) capacity) ? FGB_ERR_OVERFLOW : FGB_OK;
}

//  T1: sorted FORWARD-STRAND-ONLY device table; T2: sorted device table, pstart2: its [2^24+1]
//  lower-bound index.  Appends seed records to d_seeds (capacity records).  d_counters: 2 x u64 on
//  the device, zeroed here.  On return *h_nseeds is the number of seeds FOUND; if it exceeds
//  capacity the buffer content is incomplete and the caller must retry with a larger buffer
//  (FGB_ERR_OVERFLOW).

template<int TILE>
static int merge_launch(const rec128 *T1, unsigned n1, const rec128 *T2, const unsigned *pstart2,
                        const unsigned char *adj2, int freq,
                        const seed_pack &K, rec128 *seeds, unsigned long long capacity,
                        unsigned long long *counters, cudaStream_t st)
{ const int smem = (int) sizeof(mg_stage<TILE>);
  CUDA_TRY(cudaFuncSetAttribute(adaptamer_merge_kernel<TILE>,cudaFuncAttributeMaxDynamicSharedMemorySize,smem));
  unsigned nb = (unsigned) (((unsigned long long) n1 + TILE - 1) / TILE);
  uint4 *d_rng = NULL;
  CUDA_TRY(fgb_dmalloc((void **) &d_rng,sizeof(uint4)*(size_t) nb,st));
  { stage_timer t(&g_timings.merge_ms,st);
    merge_ranges_kernel<<<(nb + 255)/256,256,0,st>>>(T1,n1,pstart2,(unsigned) TILE,nb,d_rng);
    adaptamer_merge_kernel<TILE><<<nb,MG_THREADS,smem,st>>>(T1,n1,T2,pstart2,adj2,d_rng,freq,K,seeds,capacity,counters);
  }
  g_timings.merge_launches += 1;
  fgb_count_launch(2);
  fgb_dfree(d_rng,st);
  return FGB_OK;
}

extern "C" int fgb_merge_device(const void *d_T1, long long n1, const void *d_T2, long long n2,
                                const unsigned *d_pstart2, const unsigned char *d_adj2, int freq,
                                int anti_bits, int band_bits, int jc_bits, int ic_bits,
                                long long amxpos, long long bmxpos,
                                void *d_seeds, long long capacity, unsigned long long *d_counters,
                                unsigned long long *h_nseeds, unsigned long long *h_sumlen,
                                void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  seed_layout L;
  L.anti_bits = anti_bits; L.band_bits = band_bits; L.jc_bits = jc_bits; L.ic_bits = ic_bits;
  L.amxpos = amxpos; L.bmxpos = bmxpos;
  if (seed_key_bits(L) > 128 || freq < 1 || freq > 255) return FGB_ERR_LIMIT;
  if (n1 >= 0xffffffffll) return FGB_ERR_LIMIT;
  CUDA_TRY(cudaMemsetAsync(d_counters,0,16,st));
  seed_pack K;
  K.p_band = 12 + anti_bits;
  K.s_jc = band_bits; K.s_ic = band_bits + jc_bits; K.s_cp = band_bits + jc_bits + ic_bits;
  K.amxpos = amxpos; K.bmxpos = bmxpos; K.maxdag = amxpos + bmxpos;
  if (K.s_cp + 1 > 64 || K.p_band >= 64 || K.p_band < 13) return FGB_ERR_LIMIT;
  if (n1 > 0)
    { //  tile = T1 entries per CTA: the denser T2 is relative to T1 (a shard of genome 1 against
      //  all of genome 2), the smaller the tile, so that the CTA's T2 slice fits the staging buffer
      double ratio = (double) (n2 > 0 ? n2 : 1) / (double) n1;
      int rc;
#define MG_ARGS (const rec128 *) d_T1,(unsigned) n1,(const rec128 *) d_T2,d_pstart2,d_adj2,freq,K,(rec128 *) d_seeds, \
                (unsigned long long) capacity,d_counters,st
      if (ratio <= 2.1)       rc = merge_launch<512>(MG_ARGS);
      else if (ratio <= 4.2)  rc = merge_launch<256>(MG_ARGS);
      else if (ratio <= 8.4)  rc = merge_launch<128>(MG_ARGS);
      else                    rc = merge_launch<64>(MG_ARGS);
#undef MG_ARGS
      if (rc) return rc;
    }
  CUDA_TRY(cudaGetLastError());
  unsigned long long h[2];
  CUDA_TRY(cudaMemcpyAsync(h,d_counters,16,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  *h_nseeds = h[0];
  if (h_sumlen) *h_sumlen = h[1];
  return (h[0] > (unsigned long long) capacity) ? FGB_ERR_OVERFLOW : FGB_OK;
}

/***********************************************************************************************
 *  Seeds to their A-contig's owner (k-mer-space sharded path): count per owner, then scatter.
 *  A CTA counts / places its 2048 seeds in shared memory first, so the global counters see one
 *  atomic per owner and CTA.
 **********************************************************************************************/

static __device__ __forceinline__ unsigned seed_icont(const rec128 &r, int p_ic, int ic_bits)
{ u64 v = (p_ic >= 64) ? (r.hi >> (p_ic - 64)) : ((r.lo >> p_ic) | (p_ic ? (r.hi << (64 - p_ic)) : 0ull));
  return (unsigned) (v & ((1ull << ic_bits) - 1));
}

#define OW_ITEMS 8
template<bool SCATTER>
__global__ void __launch_bounds__(256)
seed_owner_kernel(const rec128 *__restrict__ seeds, long long n, int p_ic, int ic_bits,
                  const int *__restrict__ owner, int nrc, int world, unsigned long long *__restrict__ cnt_or_base,
                  rec128 *__restrict__ out)
{ __shared__ unsigned s_cnt[64];
  __shared__ unsigned long long s_base[64];
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const long long t0 = (long long) blockIdx.x * (256*OW_ITEMS);
  rec128 r[OW_ITEMS]; int w[OW_ITEMS]; unsigned slot[OW_ITEMS];
#pragma unroll
  for (int it = 0; it < OW_ITEMS; it++)
    { const long long i = t0 + it*256 + threadIdx.x;
      w[it] = -1;
      if (i < n)
        { r[it] = ld_rec(seeds + i);
          const unsigned ic = seed_icont(r[it],p_ic,ic_bits);
          w[it] = (ic < (unsigned) nrc) ? owner[ic] : 0;
          slot[it] = atomicAdd(&s_cnt[w[it]],1u);
        }
    }
  __syncthreads();
  if (threadIdx.x < world && s_cnt[threadIdx.x])
    s_base[threadIdx.x] = atomicAdd(&cnt_or_base[threadIdx.x],(unsigned long long) s_cnt[threadIdx.x]);
  if (!SCATTER) return;
  __syncthreads();
#pragma unroll
  for (int it = 0; it < OW_ITEMS; it++)
    if (w[it] >= 0) st_rec(out + s_base[w[it]] + slot[it],r[it]);
}

extern "C" int fgb_owner_count_device(const void *d_seeds, long long n, int p_ic, int ic_bits, const int *d_owner,
                                      int nrc, int world, unsigned long long *d_cnt, void *stream)
{ unsigned nb = (unsigned) ((n + 256*OW_ITEMS - 1) / (256*OW_ITEMS));
  seed_owner_kernel<false><<<nb,256,0,(cudaStream_t) stream>>>((const rec128 *) d_seeds,n,p_ic,ic_bits,d_owner,nrc,
                                                              world,d_cnt,NULL);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}
extern "C" int fgb_owner_scatter_device(const void *d_seeds, long long n, int p_ic, int ic_bits, const int *d_owner,
                                        int nrc, int world, unsigned long long *d_base, void *d_out, void *stream)
{ unsigned nb = (unsigned) ((n + 256*OW_ITEMS - 1) / (256*OW_ITEMS));
  seed_owner_kernel<true><<<nb,256,0,(cudaStream_t) stream>>>((const rec128 *) d_seeds,n,p_ic,ic_bits,d_owner,nrc,
                                                             world,d_base,(rec128 *) d_out);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}
