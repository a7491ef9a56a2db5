// LSD radix sort of 128-bit records on a byte range of the key, hand-written for sm_100a.
//
// Replaces the reference's two CPU sorts on the hot path:
//   msd_sort   (MSDsort.c:404)  -- k-mer records of the GIX build, key = 40-mer (80 bits)
//   rmsd_sort  (RSDsort.c:292)  -- adaptive-seed records, key = (jcont, band, anti, drem, lcp)
// Both are in-place American-flag MSD sorts on byte-packed records (MSDsort.c:211-360); on the
// device every record is widened to one 16-byte word so each pass is a perfectly coalesced
// stream (read 16 B, write 16 B per record).  One pass = one Onesweep kernel: a stable scatter
// that ranks records inside a 4096-record tile with a warp multi-split (ballots), finds the tile's
// bases by decoupled look-back, stages the tile in shared memory in digit order and writes digit
// runs back coalesced, while counting the next pass's histogram.  HBM-bound integer work: no
// tensor cores.
#include "common.cuh"
#include <stdlib.h>
#include <vector>

#define SORT_THREADS 512
#ifndef SORT_ITEMS
#define SORT_ITEMS   8
#endif
#ifndef SORT_MINBLK
#define SORT_MINBLK  2
#endif
#define SORT_TILE    (SORT_THREADS*SORT_ITEMS)
#define SORT_WARPS   (SORT_THREADS/32)

static __device__ __forceinline__ unsigned warp_incl_scan(unsigned v, int lane)
{
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
    { unsigned t = __shfl_up_sync(0xffffffffu,v,o);
      if (lane >= o) v += t;
    }
  return v;
}


/***********************************************************************************************
 *  Onesweep pass: one kernel per key byte reads every record once and writes it once.
 *   - the GLOBAL digit histogram of a pass is produced by the previous pass (each tile counts
 *     the next byte while it holds the records; the first pass has a small histogram kernel);
 *   - the tile's base inside each digit bucket comes from a decoupled look-back over the
 *     per-tile digit counts (status word = count | flag<<62; 1 = tile aggregate, 2 = inclusive
 *     prefix), tiles being handed out by an atomic ticket so every predecessor is running.
 **********************************************************************************************/

//  Lanes of the warp holding the same 8-bit digit as this lane (among valid lanes).  MATCH.ANY
//  costs one internal round per distinct value in the warp (~30 for random digits); nine ballots
//  are a fixed, much smaller cost.
static __device__ __forceinline__ unsigned match_digit(unsigned d, bool valid)
{ unsigned peers = __ballot_sync(0xffffffffu,valid);
#pragma unroll
  for (int k = 0; k < 8; k++)
    { bool bit = (d >> k) & 1;
      unsigned bk = __ballot_sync(0xffffffffu,bit);
      peers &= bit ? bk : ~bk;
    }
  return peers;
}


#define ST_AGG  (1ull << 62)
#define ST_INC  (2ull << 62)
#define ST_MASK ((1ull << 62) - 1)

__global__ void __launch_bounds__(SORT_THREADS)
sort_ghist_kernel(const rec128 *__restrict__ in, long long n, int dsh /* digit = bits [dsh,dsh+8) */, unsigned long long *__restrict__ ghist)
{ __shared__ unsigned h[256];
  int tid = threadIdx.x;
  if (tid < 256) h[tid] = 0;
  __syncthreads();
  //  a digit inside one 64-bit half is counted from that half alone (half the traffic)
  const bool one = (dsh >= 64 || dsh <= 56);
  const unsigned long long *half = reinterpret_cast<const unsigned long long *>(in) + (dsh >= 64);
  const int sh = dsh & 63;
  for (long long tile0 = (long long) blockIdx.x * SORT_TILE; tile0 < n; tile0 += (long long) gridDim.x * SORT_TILE)
    {
#pragma unroll
      for (int it = 0; it < SORT_ITEMS; it++)
        { long long idx = tile0 + it*SORT_THREADS + tid;
          bool valid = idx < n;
          unsigned d = 0;
          if (valid) d = one ? (unsigned) ((half[2*idx] >> sh) & 0xff) : rec_dig(ld_rec(in + idx),dsh);
          unsigned peers = match_digit(d,valid);             // one atomic per distinct digit of the warp
          if (valid && (tid & 31) == __ffs(peers)-1) atomicAdd(&h[d],__popc(peers));
        }
    }
  __syncthreads();
  if (tid < 256 && h[tid]) atomicAdd(&ghist[tid],(unsigned long long) h[tid]);
}

//  exclusive scan of a 256-bin global histogram -> bin bases; zeroes the histogram of the pass
//  after it and the tile ticket.
__global__ void sort_bins_kernel(const unsigned long long *__restrict__ ghist, unsigned long long *__restrict__ binbase,
                                 unsigned long long *__restrict__ nexthist, unsigned *__restrict__ ticket)
{ __shared__ unsigned long long ws[8];
  int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  unsigned long long v = ghist[tid], inc = v;
  for (int o = 1; o < 32; o <<= 1)
    { unsigned long long t = __shfl_up_sync(0xffffffffu,inc,o);
      if (lane >= o) inc += t;
    }
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  unsigned long long pre = 0;
  for (int i = 0; i < w; i++) pre += ws[i];
  binbase[tid] = pre + inc - v;
  nexthist[tid] = 0;
  if (tid == 0) *ticket = 0;
}

__global__ void __launch_bounds__(SORT_THREADS,SORT_MINBLK)
sort_onesweep_kernel(const rec128 *__restrict__ in, rec128 *__restrict__ out, long long n, int byte /* bit offset of the digit */,
                     int next_byte /* bit offset of the next pass's digit, -1: none */, const unsigned long long *__restrict__ binbase,
                     unsigned long long *__restrict__ nexthist, unsigned long long *status /* [ntiles][256] */,
                     unsigned *__restrict__ ticket)
{ extern __shared__ __align__(16) unsigned char smem_raw[];
  rec128   *tile   = reinterpret_cast<rec128 *>(smem_raw);
  unsigned *wcount = reinterpret_cast<unsigned *>(tile + SORT_TILE);   // [SORT_WARPS][256]
  unsigned *bexcl  = wcount + SORT_WARPS*256;                           // [256]
  unsigned *nhist  = bexcl + 256;                                       // [256] next byte
  unsigned *wtot   = nhist + 256;                                       // [8]
  unsigned long long *gbase = reinterpret_cast<unsigned long long *>(wtot + 8);   // [256]
  __shared__ unsigned tile_s;
  __shared__ __align__(8) unsigned long long tbar;

  int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0)
    { unsigned t = atomicAdd(ticket,1u);
      tile_s = t;
      //  the tile is 4096 consecutive 128-bit records: fetched by one TMA bulk copy (UBLKCP)
      //  into the staging buffer while the block zeroes its counters
      long long t0 = (long long) t * SORT_TILE, rm = n - t0;
      unsigned nb = (unsigned) (rm < SORT_TILE ? rm : SORT_TILE) * 16u;
      mbar_init(&tbar,1);
      tma_load_1d(tile,in + t0,nb,&tbar);
    }
  for (int i = tid; i < SORT_WARPS*256; i += SORT_THREADS) wcount[i] = 0;
  if (tid < 256) nhist[tid] = 0;
  __syncthreads();
  const unsigned tileid = tile_s;
  long long tile0 = (long long) tileid * SORT_TILE;
  long long rem = n - tile0;
  int cnt = rem < SORT_TILE ? (int) rem : SORT_TILE;

  rec128   r[SORT_ITEMS];
  unsigned rank[SORT_ITEMS];
  int base = w*(32*SORT_ITEMS);
  unsigned *myc = wcount + w*256;
  mbar_wait(&tbar,0);
#pragma unroll
  for (int it = 0; it < SORT_ITEMS; it++)
    { int idx = base + it*32 + lane;
      bool valid = idx < cnt;
      unsigned d = 0;
      if (valid)
        { r[it] = ld_rec(tile + idx);
          d = rec_dig(r[it],byte);
        }
      unsigned peers = match_digit(d,valid);
      int leader = valid ? __ffs(peers)-1 : lane;
      unsigned b = 0;
      if (valid && lane == leader)
        { b = myc[d];
          myc[d] = b + __popc(peers);
        }
      b = __shfl_sync(0xffffffffu,b,leader);
      rank[it] = b + __popc(peers & lanemask_lt());
      if (next_byte >= 0 && valid) atomicAdd(&nhist[rec_dig(r[it],next_byte)],1u);
      __syncwarp();
    }
  __syncthreads();

  //  Order of the rest: publish the tile's digit counts at once (the tiles after this one add them up
  //  while it works on), place the records in digit order inside the tile, and only THEN look back for
  //  this tile's own bases -- by which time the tiles before it have had the whole placement phase to
  //  publish theirs, so the walk is short and rarely spins.
  unsigned c = 0, inc = 0;
  unsigned long long *mine = status + (unsigned long long) tileid*256 + tid;
  if (tid < 256)
    { unsigned sum = 0;
#pragma unroll
      for (int ww = 0; ww < SORT_WARPS; ww++)
        { unsigned t = wcount[ww*256+tid];
          wcount[ww*256+tid] = sum;
          sum += t;
        }
      c = sum;
      if (tileid == 0)
        atomicExch(mine,ST_INC | c);
      else
        atomicExch(mine,ST_AGG | c);
      inc = warp_incl_scan(c,lane);
      if (lane == 31) wtot[w] = inc;
    }
  __syncthreads();
  if (tid < 256)
    { unsigned pre = 0;
      for (int i = 0; i < w; i++) pre += wtot[i];
      bexcl[tid] = pre + inc - c;
    }
  __syncthreads();

#pragma unroll
  for (int it = 0; it < SORT_ITEMS; it++)
    { int idx = base + it*32 + lane;
      if (idx < cnt)
        { unsigned d = rec_dig(r[it],byte);
          st_rec(tile + (bexcl[d] + myc[d] + rank[it]),r[it]);
        }
    }
  if (tid < 256)
    { //  four predecessors per round trip (the status words of consecutive tiles are independent loads;
      //  a serial walk pays one L2 latency per tile, and the walk is as deep as the tiles in flight)
      volatile unsigned long long *stt = status;
      unsigned long long excl = 0;
      for (long long t = (long long) tileid - 1; t >= 0; )
        { unsigned long long v[4];
#pragma unroll
          for (int q = 0; q < 4; q++)
            v[q] = (t - q >= 0) ? stt[(unsigned long long) (t - q)*256 + tid] : ST_INC;
          bool done = false;
#pragma unroll
          for (int q = 0; q < 4; q++)
            { if (done || (v[q] >> 62) == 0) break;            // not there yet: spin from this tile on
              excl += v[q] & ST_MASK;
              t -= 1;
              if (v[q] & ST_INC) done = true;
            }
          if (done) break;
        }
      if (tileid != 0) atomicExch(mine,ST_INC | (excl + c));
      gbase[tid] = binbase[tid] + excl - bexcl[tid];
      if (next_byte >= 0 && nhist[tid]) atomicAdd(&nexthist[tid],(unsigned long long) nhist[tid]);
    }
  __syncthreads();

  for (int p = tid; p < cnt; p += SORT_THREADS)
    { rec128 v = ld_rec(tile + p);
      unsigned d = rec_dig(v,byte);
      st_rec(out + (gbase[d] + p),v);
    }
}

static const size_t ONESWEEP_SMEM = SORT_TILE*sizeof(rec128) + (SORT_WARPS*256 + 256 + 256 + 8)*sizeof(unsigned)
                                    + 256*sizeof(unsigned long long);

extern "C" long long fgb_sort128_tmp_bytes(long long n)
{ long long ntiles = (n + SORT_TILE - 1) / SORT_TILE;
  if (ntiles < 1) ntiles = 1;
  return 256*ntiles*8 + (3*256 + 16)*8;          // look-back status + 2 histograms + bin bases + ticket
}

//  Sorts n records on key bytes [byte_lo,byte_hi) of the 128-bit little-endian value, stable.
//  d_a holds the input; d_b is a same-size scratch.  Returns via *result_in_b where the sorted
//  data landed (0 = d_a, 1 = d_b).  All pointers are device pointers.

//  LSD passes on the 8-bit digits at bit offsets bit_lo, bit_lo+8, ... below bit_hi (the last digit may
//  reach past bit_hi: the bits above a key are part of the order, zero in every record sorted here)
extern "C" int fgb_sort128_bits_device(void *d_a, void *d_b, long long n, int bit_lo, int bit_hi,
                                       void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n < 0 || bit_lo < 0 || bit_hi > 128 || bit_lo > bit_hi) return FGB_ERR_ARG;
  if (n >= 0xffffffffll) return FGB_ERR_LIMIT;
  *result_in_b = 0;
  if (n <= 1 || bit_lo == bit_hi) return FGB_OK;
  if (tmp_bytes < fgb_sort128_tmp_bytes(n)) return FGB_ERR_ARG;

  int ntiles = (int) ((n + SORT_TILE - 1) / SORT_TILE);
  unsigned long long *status = (unsigned long long *) d_tmp;
  unsigned long long *hist[2] = { status + 256ull*ntiles, status + 256ull*ntiles + 256 };
  unsigned long long *binbase = status + 256ull*ntiles + 512;
  unsigned *ticket = (unsigned *) (binbase + 256);

  static bool attr_set = false;
  if (!attr_set)
    { CUDA_TRY(cudaFuncSetAttribute(sort_onesweep_kernel,cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int) ONESWEEP_SMEM));
      attr_set = true;
    }

  rec128 *src = (rec128 *) d_a, *dst = (rec128 *) d_b;
  CUDA_TRY(cudaMemsetAsync(hist[0],0,256*8,st));
  { int nb = ntiles < 1184 ? ntiles : 1184;
    sort_ghist_kernel<<<nb,SORT_THREADS,0,st>>>(src,n,bit_lo,hist[0]);
    fgb_count_launch(1);
  }
  int cur = 0;
  for (int b = bit_lo; b < bit_hi; b += 8)
    { sort_bins_kernel<<<1,256,0,st>>>(hist[cur],binbase,hist[cur^1],ticket);
      CUDA_TRY(cudaMemsetAsync(status,0,256ull*ntiles*8,st));
      sort_onesweep_kernel<<<ntiles,SORT_THREADS,ONESWEEP_SMEM,st>>>(src,dst,n,b,(b+8 < bit_hi) ? b+8 : -1,
                                                                   binbase,hist[cur^1],status,ticket);
      fgb_count_launch(2);
      cur ^= 1;
      rec128 *t = src; src = dst; dst = t;
      *result_in_b ^= 1;
    }
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}

extern "C" int fgb_sort128_device(void *d_a, void *d_b, long long n, int byte_lo, int byte_hi,
                                  void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream)
{ if (byte_lo < 0 || byte_hi > 16 || byte_lo > byte_hi) return FGB_ERR_ARG;
  return fgb_sort128_bits_device(d_a,d_b,n,8*byte_lo,8*byte_hi,d_tmp,tmp_bytes,result_in_b,stream);
}

/***********************************************************************************************
 *  k-mer table sort (msd_sort's job in GIXmake.c:1436): by the 40-mer (bytes 6..15), equal
 *  k-mers by (strand|contig rank, post), i.e. by the whole 128-bit value.
 *
 *  Ten full Onesweep passes move 10 x 32 bytes per record through HBM.  Instead:
 *    1. two Onesweep passes on the two MOST significant key bytes (byte 14 then 15) leave the
 *       records partitioned into 65536 prefix bins;
 *    2. consecutive bins are packed into groups of at most BK_CAP records and BK_SPAN bins; one
 *       CTA per group pulls the group into shared memory with one TMA bulk copy, sorts it there
 *       (kmer_bucket_sort_kernel) and writes it back once;
 *    3. bins larger than BK_CAP (repeats) are compacted, sorted with the generic Onesweep sort and
 *       copied back.
 *  HBM traffic per record: 2 x 32 + 32 bytes instead of 10 x 32.
 **********************************************************************************************/

#define BK_THREADS SORT_THREADS
#define BK_ITEMS   8
#define BK_CAP     (BK_THREADS*BK_ITEMS)
#define BK_WARPS   SORT_WARPS
#define BK_SPAN    4                     // a group covers at most this many consecutive 16-bit bins
#define BK_SUBBITS 10
#define BK_NSUB    (BK_SPAN << BK_SUBBITS)
#define BK_MAXSUB  32                    // a sub-bin longer than this sends the group down the LSD path

//  bin_start[p] = first record whose bin ((hi >> binshift) - base) is >= p, p in [0,nbins]
__global__ void kmer_bins_kernel(const rec128 *__restrict__ tab, long long n, int binshift, unsigned long long base,
                                 unsigned *__restrict__ bin_start, long long nbins)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  long long lo = (i == 0) ? -1 : (long long) ((tab[i-1].hi >> binshift) - base);
  long long hi = (i == n) ? nbins : (long long) ((tab[i].hi >> binshift) - base);
  if (hi > nbins) hi = nbins;
  for (long long p = lo+1; p <= hi; p++) bin_start[p] = (unsigned) i;
}

//  One CTA sorts one group (<= BK_CAP records of <= BK_SPAN consecutive bins) by the full 128-bit
//  value.  Fast path: a counting split on the next 10 key bits (shared-memory atomics) leaves
//  sub-bins of one or two records, and every record finds its place by comparing itself with its
//  sub-bin.  A group with a crowded sub-bin (repeats) runs sixteen LSD byte passes instead.

__global__ void __launch_bounds__(BK_THREADS,2)
kmer_bucket_sort_kernel(const rec128 *__restrict__ in, rec128 *__restrict__ out,
                        const uint2 *__restrict__ groups /* start, count */, int binshift)
{ extern __shared__ __align__(16) unsigned char smem_raw[];
  rec128   *tile   = reinterpret_cast<rec128 *>(smem_raw);
  unsigned *cnt    = reinterpret_cast<unsigned *>(tile + BK_CAP);        // [BK_NSUB+1]; LSD path: wcount[BK_WARPS][256]
  unsigned *bexcl  = cnt + BK_NSUB + 32;                                  // [256]
  unsigned *wtot   = bexcl + 256;                                         // [BK_WARPS]
  __shared__ __align__(8) unsigned long long tbar;

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const uint2 g = groups[blockIdx.x];
  const int count = (int) g.y;
  if (tid == 0)
    { mbar_init(&tbar,1);
      tma_load_1d(tile,in + g.x,(unsigned) count * 16u,&tbar);
    }
  for (int i = tid; i <= BK_NSUB; i += BK_THREADS) cnt[i] = 0;
  __syncthreads();
  mbar_wait(&tbar,0);

  rec128   r[BK_ITEMS];
  unsigned sub[BK_ITEMS], off[BK_ITEMS];
  const int base = w*(32*BK_ITEMS);
  const unsigned b0 = (unsigned) (tile[0].hi >> binshift);
  const int subshift = binshift - BK_SUBBITS;
#pragma unroll
  for (int it = 0; it < BK_ITEMS; it++)
    { int idx = base + it*32 + lane;
      if (idx < count)
        { r[it] = ld_rec(tile + idx);
          sub[it] = ((((unsigned) (r[it].hi >> binshift)) - b0) << BK_SUBBITS) | ((unsigned) (r[it].hi >> subshift) & ((1u << BK_SUBBITS)-1));
          off[it] = atomicAdd(&cnt[sub[it]],1u);
        }
    }
  __syncthreads();
  //  exclusive scan of the sub-bin counts (8 per thread), crowded sub-bin detection
  bool big = false;
  { unsigned v[8], sum = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { v[i] = cnt[8*tid+i]; big |= (v[i] > BK_MAXSUB); sum += v[i]; }
    unsigned inc = warp_incl_scan(sum,lane);
    if (lane == 31) wtot[w] = inc;
    __syncthreads();
    unsigned pre = inc - sum;
    for (int i = 0; i < w; i++) pre += wtot[i];
#pragma unroll
    for (int i = 0; i < 8; i++) { cnt[8*tid+i] = pre; pre += v[i]; }
    if (tid == BK_THREADS-1) cnt[BK_NSUB] = pre;
  }
  big = __syncthreads_or(big);

  if (!big)
    {
#pragma unroll
      for (int it = 0; it < BK_ITEMS; it++)
        { int idx = base + it*32 + lane;
          if (idx < count) st_rec(tile + (cnt[sub[it]] + off[it]),r[it]);
        }
      __syncthreads();
      for (int p = tid; p < count; p += BK_THREADS)
        { rec128 R = ld_rec(tile + p);
          unsigned sb = ((((unsigned) (R.hi >> binshift)) - b0) << BK_SUBBITS) | ((unsigned) (R.hi >> subshift) & ((1u << BK_SUBBITS)-1));
          int s = (int) cnt[sb], e = (int) cnt[sb+1], rank = 0;
          for (int q = s; q < e; q++)
            { rec128 Q = ld_rec(tile + q);
              bool less = (Q.hi < R.hi) || (Q.hi == R.hi && (Q.lo < R.lo || (Q.lo == R.lo && q < p)));
              rank += less;
            }
          st_rec(out + (g.x + s + rank),R);
        }
      return;
    }

  //  LSD path: all sixteen bytes, records still in registers in load order
  unsigned *wcount = cnt;
  unsigned *myc = wcount + w*256;
  unsigned rank[BK_ITEMS];
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; i++) myc[i*32 + lane] = 0;
  __syncwarp();
  for (int byte = 0; byte < 16; byte++)
    {
#pragma unroll
      for (int it = 0; it < BK_ITEMS; it++)
        { int idx = base + it*32 + lane;
          bool valid = idx < count;
          unsigned d = valid ? rec_byte(r[it],byte) : 0;
          unsigned peers = match_digit(d,valid);
          int leader = valid ? __ffs(peers)-1 : lane;
          unsigned b = 0;
          if (valid && lane == leader)
            { b = myc[d];
              myc[d] = b + __popc(peers);
            }
          b = __shfl_sync(0xffffffffu,b,leader);
          rank[it] = b + __popc(peers & lanemask_lt());
          __syncwarp();
        }
      __syncthreads();
      unsigned c = 0, inc = 0;
      if (tid < 256)
        { unsigned sum = 0;
#pragma unroll
          for (int ww = 0; ww < BK_WARPS; ww++)
            { unsigned t = wcount[ww*256+tid];
              wcount[ww*256+tid] = sum;
              sum += t;
            }
          c = sum;
          inc = warp_incl_scan(c,lane);
          if (lane == 31) wtot[w] = inc;
        }
      __syncthreads();
      if (tid < 256)
        { unsigned pre = 0;
          for (int i = 0; i < w; i++) pre += wtot[i];
          bexcl[tid] = pre + inc - c;
        }
      __syncthreads();
#pragma unroll
      for (int it = 0; it < BK_ITEMS; it++)
        { int idx = base + it*32 + lane;
          if (idx < count)
            { unsigned d = rec_byte(r[it],byte);
              st_rec(tile + (bexcl[d] + myc[d] + rank[it]),r[it]);
            }
        }
      __syncthreads();
      if (byte + 1 < 16)
        {
#pragma unroll
          for (int it = 0; it < BK_ITEMS; it++)
            { int idx = base + it*32 + lane;
              if (idx < count) r[it] = ld_rec(tile + idx);
            }
#pragma unroll
          for (int i = 0; i < 8; i++) myc[i*32 + lane] = 0;
          __syncwarp();
        }
    }
  for (int p = tid; p < count; p += BK_THREADS)
    st_rec(out + (g.x + p),ld_rec(tile + p));
}

//  copies record segments: src[sfrom[k] .. +len[k]) -> dst[dfrom[k] ..); pre[] = prefix sums of len
__global__ void kmer_copy_segments_kernel(const rec128 *__restrict__ src, rec128 *__restrict__ dst,
                                          const unsigned *__restrict__ sfrom, const unsigned *__restrict__ dfrom,
                                          const unsigned *__restrict__ pre, int nseg, long long total)
{ for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long) gridDim.x * blockDim.x)
    { int lo = 0, hi = nseg;                                  // last k with pre[k] <= i
      while (hi - lo > 1) { int md = (lo+hi) >> 1; if (pre[md] <= i) lo = md; else hi = md; }
      unsigned o = (unsigned) (i - pre[lo]);
      st_rec(dst + (dfrom[lo] + o),ld_rec(src + (sfrom[lo] + o)));
    }
}

static const size_t BUCKET_SMEM = BK_CAP*sizeof(rec128) + (BK_NSUB + 32 + 256 + BK_WARPS)*sizeof(unsigned);

//  d_a: n records in emit order; d_b: scratch of the same size.  Sorted table lands in d_a or d_b
//  (*result_in_b).  d_tmp as for fgb_sort128_device.  Synchronises the stream once (the bin
//  boundaries come to the host to pack the groups).

//  [plo,phi): the range of 12-base prefixes the records come from (the whole space, or one
//  rank's slice of a k-mer-space sharded table).  The 65536 bins always tile THAT range, so a share
//  is binned as finely as a whole table of the same size (bins of 16 + log2(2^24/range) top bits;
//  one more partition pass when that exceeds two bytes).

extern "C" int fgb_kmer_sort_range_device(void *d_a, void *d_b, long long n, unsigned plo, unsigned phi,
                                          void *d_tmp, long long tmp_bytes, int *result_in_b, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  *result_in_b = 0;
  if (n <= 1) return FGB_OK;
  if (n >= 0xffffffffll) return FGB_ERR_LIMIT;
  if (phi <= plo || phi > (1u << 24)) return FGB_ERR_ARG;
  //  as many bins as keep the average bin near 1.5 K records (a CTA sorts <= BK_CAP in shared memory):
  //  65536 up to ~100 M records, one more power of two per doubling beyond (a 1 Gbp genome: 2^19)
  long long maxbins = 65536, target = 1536;
  if (getenv("FGB_KSORT_BIN_TARGET") != NULL) target = atoll(getenv("FGB_KSORT_BIN_TARGET"));   // tests: force more bins
  if (target < 1) target = 1;
  while (maxbins < (1ll << 24) && n / maxbins > target) maxbins <<= 1;
  int sh = 0;                                            // bins = ((prefix24 - plo') >> sh), plo' = plo rounded down
  while ((long long) ((((unsigned long long) (phi - 1) >> sh) - ((unsigned long long) plo >> sh))) >= maxbins) sh += 1;
  const int binshift = 40 + sh;                          // prefix24 = hi >> 40
  const unsigned long long base = (unsigned long long) plo >> sh;
  const long long nbins = (long long) (((unsigned long long) (phi - 1) >> sh) - base) + 1;
  int inb = 0;
  //  partition passes: 8-bit digits over the bins' bits (the top 24 - sh bits of the k-mer)
  int rc = fgb_sort128_bits_device(d_a,d_b,n,64 + binshift,128,d_tmp,tmp_bytes,&inb,st);
  if (rc) return rc;
  rec128 *src = (rec128 *) (inb ? d_b : d_a), *dst = (rec128 *) (inb ? d_a : d_b);

  static bool attr_set = false;
  if (!attr_set)
    { CUDA_TRY(cudaFuncSetAttribute(kmer_bucket_sort_kernel,cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int) BUCKET_SMEM));
      attr_set = true;
    }

  unsigned *d_bins = NULL;
  uint2 *d_groups = NULL;
  dev_scope S(st); S.own(d_bins); S.own(d_groups);
  CUDA_TRY(fgb_dmalloc((void **) &d_bins,sizeof(unsigned)*(size_t) (nbins+1),st));
  { int nb = (int) ((n + 1 + 255) / 256);
    kmer_bins_kernel<<<nb,256,0,st>>>(src,n,binshift,base,d_bins,nbins);
    fgb_count_launch(1);
  }
  std::vector<unsigned> bins((size_t) nbins + 1);
  CUDA_TRY(cudaMemcpyAsync(bins.data(),d_bins,sizeof(unsigned)*(size_t) (nbins+1),cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));

  std::vector<uint2> groups;
  std::vector<unsigned> ofrom, opre;                    // oversized bins: start, prefix of lengths
  unsigned ototal = 0;
  { unsigned gs = bins[0], gc = 0; long long gp = 0;           // group start record, size, first bin
    for (long long p = 0; p < nbins; p++)
      { unsigned len = bins[p+1] - bins[p];
        if (len == 0) continue;
        if (len > BK_CAP)
          { if (gc) { groups.push_back(make_uint2(gs,gc)); gc = 0; }
            ofrom.push_back(bins[p]); opre.push_back(ototal); ototal += len;
            continue;
          }
        if (gc != 0 && (gc + len > BK_CAP || p - gp >= BK_SPAN))
          { groups.push_back(make_uint2(gs,gc)); gc = 0; }
        if (gc == 0) { gs = bins[p]; gp = p; }
        gc += len;
      }
    if (gc) groups.push_back(make_uint2(gs,gc));
  }

  if (!groups.empty())
    { CUDA_TRY(fgb_dmalloc((void **) &d_groups,sizeof(uint2)*groups.size(),st));
      CUDA_TRY(cudaMemcpyAsync(d_groups,groups.data(),sizeof(uint2)*groups.size(),cudaMemcpyHostToDevice,st));
      kmer_bucket_sort_kernel<<<(unsigned) groups.size(),BK_THREADS,BUCKET_SMEM,st>>>(src,dst,d_groups,binshift);
      fgb_count_launch(1);
      CUDA_TRY(cudaGetLastError());
    }
  if (ototal > 0)
    { int nseg = (int) ofrom.size();
      opre.push_back(ototal);
      std::vector<unsigned> cfrom(opre.begin(),opre.end()-1);            // position in the compact array
      rec128 *d_c1 = NULL, *d_c2 = NULL; void *d_ctmp = NULL; unsigned *d_seg = NULL;
      dev_scope C(st); C.own(d_c1); C.own(d_c2); C.own(d_ctmp); C.own(d_seg);
      long long ctb = fgb_sort128_tmp_bytes(ototal);
      CUDA_TRY(fgb_dmalloc((void **) &d_c1,sizeof(rec128)*((size_t) ototal+1),st));
      CUDA_TRY(fgb_dmalloc((void **) &d_c2,sizeof(rec128)*((size_t) ototal+1),st));
      CUDA_TRY(fgb_dmalloc(&d_ctmp,ctb,st));
      CUDA_TRY(fgb_dmalloc((void **) &d_seg,sizeof(unsigned)*(3*(size_t) nseg+1),st));
      CUDA_TRY(cudaMemcpyAsync(d_seg,ofrom.data(),sizeof(unsigned)*nseg,cudaMemcpyHostToDevice,st));
      CUDA_TRY(cudaMemcpyAsync(d_seg+nseg,cfrom.data(),sizeof(unsigned)*nseg,cudaMemcpyHostToDevice,st));
      CUDA_TRY(cudaMemcpyAsync(d_seg+2*nseg,opre.data(),sizeof(unsigned)*(nseg+1),cudaMemcpyHostToDevice,st));
      int nb = (int) ((ototal + 255) / 256); if (nb > 4736) nb = 4736;
      kmer_copy_segments_kernel<<<nb,256,0,st>>>(src,d_c1,d_seg,d_seg+nseg,d_seg+2*nseg,nseg,ototal);
      int cinb = 0;
      rc = fgb_sort128_device(d_c1,d_c2,ototal,0,16,d_ctmp,ctb,&cinb,st);
      if (rc) return rc;
      kmer_copy_segments_kernel<<<nb,256,0,st>>>(cinb ? d_c2 : d_c1,dst,d_seg+nseg,d_seg,d_seg+2*nseg,nseg,ototal);
      fgb_count_launch(2);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaStreamSynchronize(st));                // the staging vectors above must outlive the copies
    }
  CUDA_TRY(cudaStreamSynchronize(st));
  *result_in_b = inb ^ 1;
  return FGB_OK;
}

/***********************************************************************************************
 *  Generic exclusive scan of a u32 array (reduce / scan-of-sums / downsweep), used for stream
 *  compaction of syncmer posts, seeds and work lists.
 **********************************************************************************************/

#define SCAN_THREADS 1024
#define SCAN_ITEMS   8
#define SCAN_TILE    (SCAN_THREADS*SCAN_ITEMS)

__global__ void __launch_bounds__(SCAN_THREADS)
scan_reduce_kernel(const unsigned *__restrict__ data, long long n, unsigned long long *__restrict__ sums)
{ __shared__ unsigned long long ws[32];
  long long t0 = (long long) blockIdx.x * SCAN_TILE;
  unsigned long long s = 0;
  for (int i = 0; i < SCAN_ITEMS; i++)
    { long long idx = t0 + i*SCAN_THREADS + threadIdx.x;
      if (idx < n) s += data[idx];
    }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu,s,o);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32)
    { s = ws[threadIdx.x];
      for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu,s,o);
      if (threadIdx.x == 0) sums[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(1024)
scan_sums_kernel(unsigned long long *__restrict__ sums, int nb, unsigned long long *__restrict__ total)
{ __shared__ unsigned long long ws[32];
  __shared__ unsigned long long carry_s;
  int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += 1024)
    { int i = base + tid;
      unsigned long long v = (i < nb) ? sums[i] : 0, inc = v;
      for (int o = 1; o < 32; o <<= 1)
        { unsigned long long t = __shfl_up_sync(0xffffffffu,inc,o);
          if (lane >= o) inc += t;
        }
      if (lane == 31) ws[w] = inc;
      __syncthreads();
      if (w == 0)
        { unsigned long long s = ws[lane], si = s;
          for (int o = 1; o < 32; o <<= 1)
            { unsigned long long t = __shfl_up_sync(0xffffffffu,si,o);
              if (lane >= o) si += t;
            }
          ws[lane] = si - s;
        }
      __syncthreads();
      unsigned long long ex = carry_s + ws[w] + inc - v;
      if (i < nb) sums[i] = ex;
      __syncthreads();
      if (tid == 1023) carry_s = ex + v;
      __syncthreads();
    }
  if (tid == 0 && total != NULL) *total = carry_s;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_down_kernel(unsigned *__restrict__ data, long long n, const unsigned long long *__restrict__ sums)
{ __shared__ unsigned ws[32];
  int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  long long t0 = (long long) blockIdx.x * SCAN_TILE + (long long) tid * SCAN_ITEMS;
  unsigned v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++)
    { v[i] = (t0 + i < n) ? data[t0+i] : 0;
      s += v[i];
    }
  unsigned inc = warp_incl_scan(s,lane);
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0)
    { unsigned x = ws[lane];
      unsigned xi = warp_incl_scan(x,lane);
      ws[lane] = xi - x;
    }
  __syncthreads();
  unsigned ex = (unsigned) sums[blockIdx.x] + ws[w] + inc - s;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++)
    { if (t0 + i < n) data[t0+i] = ex;
      ex += v[i];
    }
}

long long fgb_dev_scan_tmp_bytes(long long n)
{ long long nb = (n + SCAN_TILE - 1) / SCAN_TILE;
  if (nb < 1) nb = 1;
  return nb * 8 + 64;
}

//  In-place exclusive scan (values mod 2^32); *d_total (device, may be NULL) gets the 64-bit sum.

int fgb_dev_exclusive_scan_u32(unsigned *d_data, long long n, unsigned long long *d_total,
                               void *d_tmp, long long tmp_bytes, cudaStream_t st)
{ if (n <= 0)
    { if (d_total) CUDA_TRY(cudaMemsetAsync(d_total,0,8,st));
      return FGB_OK;
    }
  if (tmp_bytes < fgb_dev_scan_tmp_bytes(n)) return FGB_ERR_ARG;
  int nb = (int) ((n + SCAN_TILE - 1) / SCAN_TILE);
  unsigned long long *sums = (unsigned long long *) d_tmp;
  scan_reduce_kernel<<<nb,SCAN_THREADS,0,st>>>(d_data,n,sums);
  scan_sums_kernel<<<1,1024,0,st>>>(sums,nb,d_total);
  scan_down_kernel<<<nb,SCAN_THREADS,0,st>>>(d_data,n,sums);
  fgb_count_launch(3);
  CUDA_TRY(cudaGetLastError());
  return FGB_OK;
}
