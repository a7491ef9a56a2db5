// Seed-chain detection and wave-based local alignment extension on the device.
//
// Replaces (reference file:line):
//   search_seeds / align_contigs, search part   FastGA.c:3716-3798, 2973-3403
//   Local_Alignment, forward_wave, reverse_wave align.c:1423-1576, 352-874, 878-1418
//   Compress_TraceTo8                           align.c:3892
//
// Unit of parallel work = one TRIPLE (two adjacent 64-wide diagonal bands of one
// (strand, A-contig, B-contig) group): inside a triple the reference carries `alast` from chain
// to chain and the next Local_Alignment starts where the previous ended, so a triple is a
// sequential program; triples are independent (FastGA.c:3087).  One warp PAIR owns one triple:
//   * the chain scan is warp-parallel on the front warp (32 merged seeds per step);
//   * a wave is data-parallel over its diagonals.  While the band fits a warp the state
//     (V, T, HA, HM, NA) lives in registers of the lane owning the diagonal and the pass is split
//     between the front warp (V recurrence, snake, band trim) and the back warp (bit-vectors, trim
//     tests, pebbles) through a ring in shared memory (struct PairBox); wider or bordered bands run
//     on the front warp alone, in 32-diagonal chunks over circular arrays in shared memory / HBM;
//   * the running maxima besta/lasta/trim* (strict '>' in descending-k order) are reproduced
//     with redux.max + ballots, a warp prefix-max when the best cell fails its quality test;
//   * pebbles (trace-point crossings) go to a per-warp arena in HBM, allocated by ballot;
//   * the two wave routines are one direction-normalised routine (see oracle/fastga_oracle.c D);
//   * SELF mode (a genome against itself): band borders for a contig against itself (handle_hit).
// Sequences are the 2-bit staged contigs (gix.cu); a snake step compares 32 bases per 64-bit XOR.
// Integer / branch work: no tensor cores.
#include "common.cuh"
#include "handles.h"
#include <limits.h>
#include <string.h>
#include <vector>
#include <algorithm>

typedef unsigned long long u64;

#ifndef EX_WARPS
#define EX_WARPS     12                  // four triples at a time per CTA, three warps each (front, T, P)
#endif
#define EX_TEAM      3
#ifndef EX_MINBLK
#define EX_MINBLK    1
#endif
#define EX_W         256                 // diagonals of wave state per warp (shared memory)
#define FULL         0xffffffffu

#define TRIM_LEN     15
#define DUB_TRIM     45
#define PATH_INT     0x0fffffffffffffffull
#define PATH_WIN     0x1fffffffffffffffull
#define TRIM_MASK    0x7fff
#define TRIM_MLAG    250
#define WAVE_LAG     70
#define BUCK_SHIFT   6
#define BUCK_WIDTH   64
#define BUCK_ANTI    128

#define ST_OK        0
#define ST_BAND      1                   // band wider than the state capacity
#define ST_CELLS     2                   // pebble arena full
#define ST_STAGE     3                   // trace staging full
#define ST_SPEC      4                   // a hit group could not run on its own: the triple is re-run in one piece

struct __align__(16) Peb { int ptr, diag, diff, mark; };

struct ChainHit;
//  Work item of the first launch: hits [h0,h0+hn) of work triple w, whose first hit is number g of
//  its triple (hn bit 31: no hit list, the triple is scanned in the kernel).
struct ExItem { unsigned w, h0, hn, g; };
#define SPEC_SEQ_BITS 14                 // records of a hit group are numbered (g << 14) + 0, 1, ...
struct ext_params
{ const rec128 *seeds; long long nseeds;
  int p_anti, anti_bits, p_band, band_bits, p_jc, jc_bits, p_ic, ic_bits, p_cp;
  long long amxpos, bmxpos;
  const unsigned *seg_start; int nseg;
  const unsigned *work; int nwork; unsigned *queue;
  const unsigned *widx;                                // retry launches: position of work[w] in the first launch's list
  const ChainHit *hits; const uint2 *hit_range;        // pre-scanned chains of every triple of the first list (NULL: scan here)
  unsigned *failed_w;                                  // positions (first list) of the triples in failed[]
  unsigned *need;                                      // bit ST_* set when a triple failed for that reason
  unsigned long long *wlog;                            // diagnostics (FGB_WLOG): 4 words per work item, or NULL
  const ExItem *items;                                 // first launch: hit groups (NULL: work[] holds whole triples)
  long long *galast;                                   //   per item: where the tube stood after its last hit
  int attempt;                                         // launch number, stamped on every record
  const u64 *aseq, *arseq; const long long *awoff, *aclen; const int *aperm;
  const u64 *bseq;         const long long *bwoff, *bclen; const int *bperm;
  int chain_break, chain_min, aln_min; double aln_rate;
  int tspace, path_ave, dscore; const short *score, *table;
  Peb *cells; long long cells_per_warp;
  unsigned char *stage; int stage_bytes;               // per warp: 2 x stage_bytes
  unsigned char *out; u64 out_cap; u64 *out_used;
  u64 *counters;                                       // 0 hits 1 LA calls 2 waves 3 cells 4 records
  unsigned *failed; unsigned *nfailed;                 // triples that overflowed an arena
  unsigned char *bigstate;                             // wide-band kernel: per-warp wave state in HBM
  int self_mode;                                       // FastGA A: genome against itself (align_contigs :3030)
};

struct Ctx
{ const unsigned *A, *B; int alen, blen; long long anw, bnw;
  int *V, *HA, *HM, *NA; u64 *T; int *carry;
  Peb *cells; int cmax, avail;
  unsigned char *fstage, *rstage; int smax;
  int tspace, path_ave; const short *score, *table; const short *ttab; int sc15;
  u64 nwaves, ncells, cyc_wave, cyc_extract, pwaves, npairs, fwait, ftot, bwait, btot;
  struct PairBox *box;                   // front/back warp pair mailbox (NULL: this warp runs waves alone)
  unsigned box_off;                      //   and its offset inside the dynamic shared memory
  Peb *pwin; int pwin_n;                 // pwin_n pebbles of shared memory: the window of the trace read-out
};

//  Front/back pairing of a wave pass.  The recurrence that makes a pass serial is only the
//  furthest-point recurrence V (three-way max + snake) and the band trim that follows from it;
//  the match bit-vectors, the trim-point tests and the trace pebbles hang off it without feeding
//  back, except for the loop's stop test.  So a pass is split over two warps of a block: the FRONT
//  warp runs V and the band, and streams each wave (the 32 new V values + a header) through a ring
//  in shared memory; the BACK warp replays the predecessor choice from the V values, carries
//  T / HA / HM / NA in its registers, tests trim points, drops pebbles, and raises `stop` when
//  lasta falls TRIM_MLAG behind.  The front may run ahead by at most EX_RING waves; what it
//  computes past the stop wave is discarded.  Anything unusual (band wider than 31 diagonals,
//  a wave that does not advance the best point, an empty band) is handed back: the back warp
//  spills its state and the front warp finishes the pass alone on the code below.

#ifndef EX_PAIR
#define EX_PAIR 1
#endif
#ifndef EX_NOREG
#define EX_NOREG 0                       // 1 (debug): never use the register path of the single-warp waves
#endif
#define EX_RING 32
#define EX_TILEW 256                     // 32-bit words per staged sequence tile: 4096 bases
#define EX_TILEB (16*EX_TILEW)

struct __align__(16) RingEnt
{ int cmd, top, lowk, mx;                // cmd 1 wave, 2 last wave (more == 0), 3 hand back; band [lowk,top] of the wave
  int lowk_after, hghk_after, pad0, pad1;
  int cc[32];
};

struct __align__(16) PairBox
{ volatile int seq, cmd;                 // front -> back: seq bumps per request; cmd 1 / 2 = forward / reverse pass, 9 exit
  volatile int head, tail;               // last wave pushed / consumed by the pebble warp (ring slots are free up to here)
  volatile int stop;                     // T warp -> front, P warp: 0 running, 1 pass finished, 2 handed back
  volatile int tailt, stopp;             // last wave the T warp finished (P may process up to here); P warp done (1 / 2)
  int pstatus;                           // ST_* of the P warp
  int lowk, hghk, besta, lasta, trima, trimx, trimd, trimha, avail;
  int tspace, path_ave, cmax, wmask, dif0;
  Peb *cells; int *V, *HA, *HM, *NA; u64 *T;
  int status, r_lasta, r_trima, r_trimx, r_trimd, r_trimha, r_avail, r_dif; u64 r_ncell;
  long long r_bwait, r_btot;             // diagnostics: T warp cycles waiting for the front / P warp cycles waiting for T
  long long r_fwait, r_ffast;            //   front: cycles waiting for ring space, waves on the fast path
  int tring[EX_RING];                    // T -> P: lane holding the new trim point of a wave, -1 none
  unsigned tileA[EX_TILEW], tileB[EX_TILEW];   // 2-bit sequence tiles of the two contigs around the band (front warp)
  RingEnt ring[EX_RING];
};

#define SPIN_LIMIT (1 << 27)
#ifndef EX_DIAG
#define EX_DIAG 0                        // 1: per-wave wait-cycle accounting of the pair (slows the waves by ~5 %)
#endif
#define DIAG_CLOCK() (EX_DIAG ? clock64() : 0ll)

//  The trace read-out walks a pebble chain from the trim point back to the start: every hop used to be
//  a dependent L2 / HBM round trip (0.5-1 us x thousands of trace points, three walks per alignment:
//  8 % of the kernel's cycles, all of them on the critical path of an item).  Pebbles are appended in
//  wave order and a chain only points backwards, a few cells at a time (all diagonals of a band drop
//  theirs between two of one path's): the walk pulls the c.pwin_n cells ending at the current one into
//  shared memory with one coalesced load and hops inside that window until the chain leaves it.
struct PebWalk
{ const Peb *cells; Peb *win; int lo, hi, n;             // window = cells[lo..hi] (at most n cells), lo > hi: empty
  __device__ __forceinline__ void init(const Peb *c, Peb *w, int cap) { cells = c; win = w; n = cap; lo = 0; hi = -1; }
  __device__ __forceinline__ Peb at(int idx)              // idx is warp-uniform
  { if (idx < lo || idx > hi)
      { const int lane = threadIdx.x & 31;
        __syncwarp();
        hi = idx; lo = idx - (n-1); if (lo < 0) lo = 0;
#pragma unroll 4
        for (int q = lane; lo + q <= hi; q += 32)
          *reinterpret_cast<int4 *>(win + q) = __ldcg(reinterpret_cast<const int4 *>(cells + lo + q));
        __syncwarp();
      }
    const int4 v = *reinterpret_cast<const int4 *>(win + (idx - lo));
    Peb r; r.ptr = v.x; r.diag = v.y; r.diff = v.z; r.mark = v.w;
    return r;
  }
};

#define EX_WBIG      8192                // diagonals of wave state per warp in the wide-band retry kernel (HBM)

//  The kernel's dynamic shared memory.  Device functions address the pair mailboxes as offsets from
//  THIS symbol, so the compiler knows the state space (LDS/STS instead of generic loads).
extern __shared__ __align__(16) unsigned char ex_smem[];

//  flag hand-off between the two warps of a pair: release store (fence + STS) / acquire load (LDS)
static __device__ __forceinline__ void st_release_smem(volatile int *p, int v)
{ asm volatile("st.release.cta.shared.b32 [%0], %1;" :: "r"(smem_u32((const void *) p)), "r"(v) : "memory"); }
static __device__ __forceinline__ int ld_acquire_smem_a(unsigned a)          // a = shared-window address
{ int v;
  asm volatile("ld.acquire.cta.shared.b32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
static __device__ __forceinline__ void st_release_smem_a(unsigned a, int v)
{ asm volatile("st.release.cta.shared.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
static __device__ __forceinline__ int ld_acquire_smem(const volatile int *p)
{ int v;
  asm volatile("ld.acquire.cta.shared.b32 %0, [%1];" : "=r"(v) : "r"(smem_u32((const void *) p)) : "memory");
  return v;
}
#define IX(k) ((k) & (W-1))

static __device__ __forceinline__ u64 get_bits(const rec128 &r, int pos, int n)
{ u64 v;
  if (pos >= 64) v = r.hi >> (pos-64);
  else if (pos == 0) v = r.lo;
  else v = (r.lo >> pos) | (r.hi << (64-pos));
  return n >= 64 ? v : (v & ((1ull << n) - 1));
}

//  32 bases starting at base offset boff of a staged contig (32-bit word view).  Contigs are
//  zero-padded by 16 bytes on both sides (fgb_genome_create), so boff in [-32, len+32) needs no
//  bounds test: three aligned loads and two funnel shifts.

static __device__ __forceinline__ u64 win(const unsigned *__restrict__ w, int boff)
{ int q = boff >> 4, s = (boff & 15) << 1;
  unsigned w0 = __ldg(w+q), w1 = __ldg(w+q+1), w2 = __ldg(w+q+2);      // staged contigs are read-only: LDG through L1
  return (u64) __funnelshift_r(w0,w1,s) | ((u64) __funnelshift_r(w1,w2,s) << 32);
}

static __device__ __forceinline__ int base_at(const unsigned *__restrict__ w, int len, int i)
{ if (i < 0 || i >= len) return 4;
  return (int) (__ldg(w + (i >> 4)) >> ((i & 15) << 1)) & 3;
}

template<int S, class CX> static __device__ __forceinline__ int a_at(const CX &c, int xn)
{ return base_at(c.A,c.alen,(S > 0) ? xn : -xn-1); }
template<int S, class CX> static __device__ __forceinline__ int b_at(const CX &c, int yn)
{ return base_at(c.B,c.blen,(S > 0) ? yn : -yn-1); }

//  slide along diagonal kk from normalised xn; returns #matches, flag 0 mismatch / 1 B end / 2 A end
//    (B is tested first, align.c:683-697)

template<int S, class CX>
static __device__ __forceinline__ int snake(const CX &c, int xn, int kk, int &flag)
{ int yn = xn - kk, t = 0, tmax;
  if (S > 0)
    { const int x = xn, y = yn;
      tmax = min(c.alen - x,c.blen - y);
      if ((x | y) < 0 || tmax <= 0)                        // off a sequence end (rare): B first, then A
        { flag = (y < 0 || y >= c.blen) ? 1 : 2; return 0; }
      while (t < tmax)
        { u64 d = win(c.A,x+t) ^ win(c.B,y+t);
          if (d) { t += (__ffsll((long long) d)-1) >> 1; break; }
          t += 32;
        }
      if (t >= tmax) { t = tmax; flag = (y + t == c.blen) ? 1 : 2; }
      else flag = 0;
    }
  else
    { const int x = -xn, y = -yn;
      tmax = min(x,y);
      if (tmax <= 0 || y > c.blen || x > c.alen)
        { flag = (y <= 0 || y > c.blen) ? 1 : 2; return 0; }
      while (t < tmax)
        { u64 d = win(c.A,x-t-32) ^ win(c.B,y-t-32);
          if (d) { t += __clzll((long long) d) >> 1; break; }
          t += 32;
        }
      if (t >= tmax) { t = tmax; flag = (y - t == 0) ? 1 : 2; }
      else flag = 0;
    }
  return t;
}

//  TABLE[x] / SCORE[x] of align.c:207-220 for a 15-bit column pattern x.  TABLE (64 KB of int16)
//  stays in HBM and is read through L1 (the patterns met in practice are almost all ones: a few
//  hundred hot rows), which leaves the shared memory for a second CTA per SM;
//  SCORE[x] = popc(x)*1000 - 15*dscore needs no table.

struct SeqV { const unsigned *A, *B; int alen, blen; };       // the two contigs of a pass, by value (registers)
struct TrimV { const short *ttab; int sc15; };

template<class CX>
static __device__ __forceinline__ bool trim_ok(const CX &c, u64 b)
{ int lo15 = (int) (b & TRIM_MASK), hi15 = (int) ((b >> TRIM_LEN) & TRIM_MASK);
  int tl = __ldg(c.ttab + lo15), th = __ldg(c.ttab + hi15);       // 64 KB table in HBM, its hot rows live in L1
  int sl = __popc(lo15)*1000 - c.sc15;
  return tl >= 0 && th + sl >= 0;                        // TABLE[lo] >= 0 && TABLE[hi] + SCORE[lo] >= 0
}

static __device__ __forceinline__ int warp_prefix_max_excl(int v, int lane)
{ int r = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
    { int t = __shfl_up_sync(FULL,r,o);
      if (lane >= o) r = max(r,t);
    }
  int e = __shfl_up_sync(FULL,r,1);
  return lane == 0 ? INT_MIN : e;
}

//  One wave pass (direction s) from anti-diagonal mida over diagonals [low,hgh].
//  Outputs the trim point (original coordinates), its diffs and the pebble chain head.
//
//  Wave state per diagonal: V (furthest anti-diagonal), T (match bit-vector of the last 64
//  columns), HA/HM (head pebble and its mark), NA (next trace-point anti-diagonal).  While the
//  band fits one warp (<= 32 diagonals, the normal case: the WAVE_LAG trim keeps ~8) the state
//  lives in REGISTERS of the lane that owns the diagonal (lane = -kk mod 32, fixed for the whole
//  pass), neighbours are read with shuffles and a wave is one straight-line pass with no shared
//  memory traffic and no barrier.  Wider bands spill to the arrays in c (shared memory, or HBM in
//  the wide-band retry kernel) and are processed in 32-diagonal chunks.

static __device__ __forceinline__ unsigned rotr32(unsigned x, int r) { return __funnelshift_r(x,x,r); }

//  BACK warp of a pair: one wave pass (direction s) from the state the front warp left after
//  wave 0.  Returns when the pass is finished (stop = 1) or handed back (stop = 2).

//  The BACK of a pass is two warps.  Both replay the predecessor choice from consecutive V's (two
//  shuffles); the T warp carries the match bit-vectors, tests trim points and decides when the pass
//  stops; the P warp, one or more waves behind it, carries the pebble lists (HA / HM / NA), drops
//  pebbles and picks up the pebble head of every trim point the T warp announces (tring).  Per wave
//  each executes about half of what one back warp did, and the wave rate of a pass is set by the
//  slowest of the three warps.

//  T warp: one wave pass (direction s) from the state the front warp left after wave 0.
template<int s>
static __device__ __noinline__ void wave_T(const unsigned box_off, const short *__restrict__ ttab, const int sc15)
{ PairBox *const bx = reinterpret_cast<PairBox *>(ex_smem + box_off);
  const TrimV c = { ttab, sc15 };
  const int lane = threadIdx.x & 31;
  const int FRESH = (s > 0) ? -1 : -INT_MAX;
  const int lane_up = (lane + 31) & 31, lane_dn = (lane + 1) & 31;
  int lowk = bx->lowk, hghk = bx->hghk, besta = bx->besta, lasta = bx->lasta, trima = bx->trima;
  int trimx = bx->trimx, trimd = bx->trimd;
  const int path_ave = bx->path_ave, wmask = bx->wmask, dif0 = bx->dif0;
  int rV; u64 rT;
  { const int kk = hghk - ((hghk + lane) & 31);
    const int ix = kk & wmask;
    rV = (kk >= lowk) ? bx->V[ix] : FRESH;
    rT = bx->T[ix];
  }
  int d = 0, head_seen = 0, fin = 0;                         // fin: 1 pass finished, 2 handed back
  long long dg_wait = 0;
  const unsigned head_a = smem_u32((const void *) &bx->head), tailt_a = smem_u32((const void *) &bx->tailt);
  while (true)
    { d += 1;
      if (d > head_seen)
        { int spin = 0; const long long w0 = DIAG_CLOCK();
          while ((head_seen = ld_acquire_smem_a(head_a)) < d)
            if (bx->stopp != 0 || ++spin > SPIN_LIMIT) { fin = 1; break; }     // the P warp gave up (arena full)
          dg_wait += DIAG_CLOCK() - w0;
          if (fin) { d -= 1; break; }
        }
      const RingEnt *e = &bx->ring[d & (EX_RING-1)];
      const int4 hd = *(const int4 *) e;                       // cmd, top, lowk, mx
      if (hd.x == 3)
        { //  hand back: the band of the last wave goes to the front warp's arrays
          const int kk = hghk - ((hghk + lane) & 31);
          if (kk >= lowk) { const int ix = kk & wmask; bx->V[ix] = rV; bx->T[ix] = rT; }
          d -= 1; fin = 2;
          break;
        }
      const int2 af = *(const int2 *) &e->lowk_after;
      const int top = hd.y, lowb = hd.z, mx = hd.w, la = af.x, ha_ = af.y;
      const int cc = e->cc[lane];
      const int ltop = (-top) & 31;
      const int kk = top - ((top + lane) & 31);
      const bool act = kk >= lowb;
      //  replay the predecessor choice (align.c:625-660): out-of-band lanes hold FRESH
      const int ap = __shfl_sync(FULL,rV,lane_up), am = __shfl_sync(FULL,rV,lane_dn), ac = rV;
      int pred, cp;
      if (ap > max(ac,am)) { pred = 1;  cp = ap+1; }
      else if (am > ac)    { pred = -1; cp = am+1; }
      else                 { pred = 0;  cp = ac+2; }
      u64 b = __shfl_sync(FULL,rT,(lane - pred) & 31);
      const int xn = (cc + kk) >> 1;
      { const int t = xn - ((cp + kk) >> 1);                   // matches the snake slid over
        b <<= 1;
        b = (t >= 64) ? ~0ull : ((b << t) | ((1ull << t) - 1));
      }
      //  the front warp only pushes waves that advance the best point (mx > besta)
      int tlane = -1;                                          // lane of this wave's new trim point
      { const int cm = act ? cc : INT_MIN;
        unsigned eq = rotr32(__ballot_sync(FULL,cm == mx),ltop);
        int Lb = (ltop + __ffs(eq) - 1) & 31;
        bool qual = act && cc > besta && __popcll(b & PATH_WIN) >= path_ave;
        bool tq = qual && trim_ok(c,b);
        //  Lb = highest diagonal reaching the wave maximum = the last record setter of the sequential
        //  scan: if it passes both tests it alone decides (one shuffle); else the full prefix-max
        const int tqL = __shfl_sync(FULL,(int) tq,Lb), xL = __shfl_sync(FULL,xn,Lb);
        if (tqL)
          { lasta = mx; trima = mx; trimd = dif0+d;
            trimx = xL;
            tlane = Lb;
          }
        else
          { unsigned ql = __ballot_sync(FULL,qual), tl = __ballot_sync(FULL,tq);
            int cpos = __shfl_sync(FULL,cm,(ltop + lane) & 31);   // value at position = lane
            int ex = max(warp_prefix_max_excl(cpos,lane),besta);
            unsigned rm = __ballot_sync(FULL,cpos > ex);
            unsigned qm = rm & rotr32(ql,ltop), tm = rm & rotr32(tl,ltop);
            if (qm) lasta = __shfl_sync(FULL,cc,(ltop + 31 - __clz(qm)) & 31);
            if (tm)
              { int L3 = (ltop + 31 - __clz(tm)) & 31;
                trima = __shfl_sync(FULL,cc,L3);
                trimx = __shfl_sync(FULL,xn,L3);
                trimd = dif0+d;
                tlane = L3;
              }
          }
        besta = mx;
      }
      if (act) rT = b;
      rV = (kk >= la && kk <= ha_ && act) ? cc : FRESH;
      lowk = la; hghk = ha_;
      __syncwarp();
      if (lane == 0)
        { bx->tring[d & (EX_RING-1)] = tlane;
          st_release_smem_a(tailt_a,d);
        }
      if (hd.x == 2 || lasta < besta - TRIM_MLAG) { fin = 1; break; }
    }
  __syncwarp();
  if (lane == 0)
    { bx->status = ST_OK; bx->r_lasta = lasta; bx->r_trima = trima; bx->r_trimx = trimx; bx->r_trimd = trimd;
      bx->r_dif = dif0 + d;
      if (EX_DIAG) bx->r_bwait = dg_wait;
      st_release_smem(&bx->stop,fin);
    }
  __syncwarp();
}

//  P warp: the pebble side of the same pass, following the T warp.
template<int s>
static __device__ __noinline__ void wave_P(const unsigned box_off)
{ PairBox *const bx = reinterpret_cast<PairBox *>(ex_smem + box_off);
  const int lane = threadIdx.x & 31;
  const unsigned lt = lanemask_lt();
  const int FRESH = (s > 0) ? -1 : -INT_MAX;
  const int lane_up = (lane + 31) & 31, lane_dn = (lane + 1) & 31;
  int lowk = bx->lowk, hghk = bx->hghk, trimha = bx->trimha, avail = bx->avail;
  const int tspace = bx->tspace, cmax = bx->cmax, wmask = bx->wmask, dif0 = bx->dif0;
  Peb *cells = bx->cells;
  u64 ncell = 0;
  int rV, rHA, rHM, rNA;
  { const int kk = hghk - ((hghk + lane) & 31);
    const int ix = kk & wmask;
    rV = (kk >= lowk) ? bx->V[ix] : FRESH;
    rHA = bx->HA[ix]; rHM = bx->HM[ix]; rNA = bx->NA[ix];
  }
  int d = 0, seen = 0, fin = 0, status = ST_OK;
  long long dg_wait = 0;
  const unsigned tailt_a = smem_u32((const void *) &bx->tailt), stop_a = smem_u32((const void *) &bx->stop);
  const unsigned tail_a = smem_u32((const void *) &bx->tail);
  while (true)
    { d += 1;
      if (d > seen)
        { int spin = 0; const long long w0 = DIAG_CLOCK();
          while ((seen = ld_acquire_smem_a(tailt_a)) < d)
            { const int st = ld_acquire_smem_a(stop_a);
              if (st != 0)
                { seen = ld_acquire_smem_a(tailt_a);             // T published its last wave before it stopped
                  if (seen < d) { fin = st; break; }
                }
              if (++spin > SPIN_LIMIT) { fin = 1; status = ST_STAGE; break; }
            }
          dg_wait += DIAG_CLOCK() - w0;
          if (fin) { d -= 1; break; }
        }
      const RingEnt *e = &bx->ring[d & (EX_RING-1)];
      const int4 hd = *(const int4 *) e;                       // cmd, top, lowk, mx
      const int2 af = *(const int2 *) &e->lowk_after;
      const int top = hd.y, lowb = hd.z, la = af.x, ha_ = af.y;
      const int cc = e->cc[lane];
      const int tln = bx->tring[d & (EX_RING-1)];
      const int kk = top - ((top + lane) & 31);
      const bool act = kk >= lowb;
      const bool fresh = (kk == top || kk == lowb);
      const int ap = __shfl_sync(FULL,rV,lane_up), am = __shfl_sync(FULL,rV,lane_dn), ac = rV;
      int pred;
      if (ap > max(ac,am)) pred = 1;
      else if (am > ac)    pred = -1;
      else                 pred = 0;
      const int src = (lane - pred) & 31;
      int ha = __shfl_sync(FULL,rHA,src), hm = __shfl_sync(FULL,rHM,src);
      int nn = __shfl_sync(FULL,rNA,src);
      int nan = fresh ? nn : rNA;
      const int xn = (cc + kk) >> 1, k = s*kk;
      bool need = act && xn >= nan;
      while (__any_sync(FULL,need))
        { bool create = need && (s*hm < nan);
          if (avail + 32 > cmax) { fin = 1; status = ST_CELLS; break; }
          unsigned m = __ballot_sync(FULL,create);
          int idx = avail + __popc(m & lt);
          avail += __popc(m);
          if (create)
            { Peb p; p.ptr = ha; p.diag = k; p.diff = dif0+d; p.mark = s*nan;
              cells[idx] = p;
              ha = idx; hm = s*nan;
            }
          if (need) nan += tspace;
          need = act && xn >= nan;
        }
      if (fin) { d -= 1; break; }
      if (tln >= 0) trimha = __shfl_sync(FULL,ha,tln);         // pebble head of the new trim point
      if (act) { rHA = ha; rHM = hm; rNA = nan; }
      rV = (kk >= la && kk <= ha_ && act) ? cc : FRESH;
      lowk = la; hghk = ha_;
      ncell += (u64) (top - lowb + 1);
      __syncwarp();
      if (lane == 0) st_release_smem_a(tail_a,d);
    }
  if (fin == 2)
    { //  handed back after wave d: the pebble state of the band goes to the front warp's arrays
      const int kk = hghk - ((hghk + lane) & 31);
      if (kk >= lowk) { const int ix = kk & wmask; bx->HA[ix] = rHA; bx->HM[ix] = rHM; bx->NA[ix] = rNA; }
    }
  __syncwarp();
  if (lane == 0)
    { bx->pstatus = status; bx->r_trimha = trimha; bx->r_avail = avail; bx->r_ncell = ncell;
      if (EX_DIAG) bx->r_btot = dg_wait;
      __threadfence();                                         // pebbles (HBM) before the flag
      st_release_smem(&bx->stopp,fin);
    }
  __syncwarp();
}

//  FRONT warp of a pair: the waves of one pass from the band [lowk,hghk] (V of the last wave in rV,
//  lane (-kk & 31) owning diagonal kk) until the pass ends, the back warp stops it, or a wave is
//  not a plain one (then it is undone and handed back).  Everything a wave needs lives in
//  registers; the control flow is warp-uniform by construction (the branches test ballots, redux
//  results and band scalars only), so there is no divergence bookkeeping on the chain V -> snake
//  -> maximum -> band trim -> V that bounds how fast one alignment can grow.
//  Returns (lowk, hghk, besta, 1 if the pass must finish on the single-warp code without pairing).

template<int s>
static __device__ __forceinline__ int snake_u(const unsigned *__restrict__ A, const unsigned *__restrict__ B,
                                              const int alen, const int blen, const bool act, const int xn,
                                              const int kk, bool &ended)
{ //  direction-normalised coordinates -> contig coordinates; `lim` = bases left on the diagonal
  const int x = (s > 0) ? xn : -xn, y = (s > 0) ? xn - kk : kk - xn;
  const int lim = (s > 0) ? min(alen - x,blen - y) : min(x,y);
  const bool ok = (s > 0) ? (act && (x | y) >= 0 && lim > 0) : (act && lim > 0 && y <= blen && x <= alen);
  const int xo = ok ? x : ((s > 0) ? 0 : 32), yo = ok ? y : ((s > 0) ? 0 : 32);     // idle lanes read a valid window
  int t;
  { const u64 dd = (s > 0) ? (win(A,xo) ^ win(B,yo)) : (win(A,xo-32) ^ win(B,yo-32));
    t = dd ? ((s > 0) ? ((__ffsll((long long) dd)-1) >> 1) : (__clzll((long long) dd) >> 1)) : 32;
  }
  bool cont = ok && t == 32 && 32 < lim;
  while (__any_sync(FULL,cont))                                   // a run of 32+ matches (one lane in five at 5 %)
    { const int o = cont ? t : 0;
      const u64 dd = (s > 0) ? (win(A,xo+o) ^ win(B,yo+o)) : (win(A,xo-o-32) ^ win(B,yo-o-32));
      const int m = dd ? ((s > 0) ? ((__ffsll((long long) dd)-1) >> 1) : (__clzll((long long) dd) >> 1)) : 32;
      if (cont) t += m;
      cont = cont && m == 32 && t < lim;
    }
  ended = act && (!ok || t >= lim);
  return ok ? min(t,lim) : 0;
}

//  which end stopped the slide: 1 = B's, 2 = A's (B is tested first, align.c:683-697)
template<int s>
static __device__ __forceinline__ int end_flag(const int alen, const int blen, const int xn0, const int kk, const int t)
{ const int x = (s > 0) ? xn0 : -xn0, y = (s > 0) ? xn0 - kk : kk - xn0;
  const int lim = (s > 0) ? min(alen - x,blen - y) : min(x,y);
  if (s > 0)
    { if ((x | y) < 0 || lim <= 0) return (y < 0 || y >= blen) ? 1 : 2;
      return (y + t == blen) ? 1 : 2;
    }
  if (lim <= 0 || y > blen || x > alen) return (y <= 0 || y > blen) ? 1 : 2;
  return (y - t == 0) ? 1 : 2;
}

//  32 bases at base offset off (>= 0) of a staged sequence tile (shared memory)
static __device__ __forceinline__ u64 win_t(const unsigned *tile, int off)
{ const int q = off >> 4, sh = (off & 15) << 1;
  const unsigned w0 = tile[q], w1 = tile[q+1], w2 = tile[q+2];
  return (u64) __funnelshift_r(w0,w1,sh) | ((u64) __funnelshift_r(w1,w2,sh) << 32);
}

//  stages 4096 bases of a contig from base t0 (a multiple of 64: 16-byte aligned; >= -64: the zero
//  pad ahead of every contig) into a tile: two 128-bit read-only loads and stores per lane
static __device__ __forceinline__ void tile_fill(unsigned *tile, const unsigned *__restrict__ G, int t0, int lane)
{ const uint4 *src = reinterpret_cast<const uint4 *>(G + (t0 >> 4));
  uint4 *dst = reinterpret_cast<uint4 *>(tile);
  dst[lane] = __ldg(src + lane);
  dst[lane + 32] = __ldg(src + lane + 32);
  __syncwarp();
}

//  Can the next EX_FASTN waves run on the interior fast path?  Every lane of those waves slides from
//  x in [xlo,xhi] / y in [ylo,yhi] (direction-normalised; from the band scalars: a live diagonal has
//  V >= besta - WAVE_LAG, besta grows by at most 2*65 a wave, the band by one diagonal each side);
//  the fast path needs both 32-base windows of every slide inside the staged tiles and inside the
//  contigs.  Re-stages a tile when the band has moved out of it.  Warp-uniform.
#define EX_FASTN 8
template<int s>
static __device__ __forceinline__ bool fast_window(unsigned *tA, unsigned *tB, const unsigned *__restrict__ A,
                                                   const unsigned *__restrict__ B, int alen, int blen,
                                                   int besta, int lowk, int hghk, int &a0, int &b0, int lane)
{ const int clo = besta - WAVE_LAG, chi = besta + 2 + EX_FASTN*130;
  const int xlo = (clo + lowk - EX_FASTN) >> 1, xhi = ((chi + hghk + EX_FASTN) >> 1) + 1;
  const int ylo = (clo - hghk - EX_FASTN) >> 1, yhi = ((chi - lowk + EX_FASTN) >> 1) + 1;
  //  real coordinates touched: s > 0 [lo, hi+64+48);  s < 0: positions -hi-64-16 .. -lo+48
  const int ra0 = (s > 0) ? xlo : -xhi - 80, ra1 = (s > 0) ? xhi + 112 : -xlo + 48;
  const int rb0 = (s > 0) ? ylo : -yhi - 80, rb1 = (s > 0) ? yhi + 112 : -ylo + 48;
  if (s > 0) { if (xlo < 0 || ylo < 0 || xhi + 64 > alen || yhi + 64 > blen) return false; }
  else       { if (-xhi - 64 < 0 || -yhi - 64 < 0 || -xlo > alen || -ylo > blen) return false; }
  if (ra0 < a0 || ra1 > a0 + EX_TILEB)
    { a0 = (s > 0) ? ((ra0 - 64) & ~63) : (((ra1 + 64 + 63) & ~63) - EX_TILEB);
      if (a0 < -64) a0 = -64;
      if (ra0 < a0 || ra1 > a0 + EX_TILEB) return false;
      tile_fill(tA,A,a0,lane);
    }
  if (rb0 < b0 || rb1 > b0 + EX_TILEB)
    { b0 = (s > 0) ? ((rb0 - 64) & ~63) : (((rb1 + 64 + 63) & ~63) - EX_TILEB);
      if (b0 < -64) b0 = -64;
      if (rb0 < b0 || rb1 > b0 + EX_TILEB) return false;
      tile_fill(tB,B,b0,lane);
    }
  return true;
}

template<int s>
static __device__ __noinline__ int4 front_run(const unsigned box_off, const unsigned *__restrict__ A,
                                              const unsigned *__restrict__ B, const int alen, const int blen,
                                              int lowk, int hghk, int besta, int rV)
{ PairBox *const bx = reinterpret_cast<PairBox *>(ex_smem + box_off);
  const SeqV q = { A, B, alen, blen };
  const int lane = threadIdx.x & 31;
  const int FRESH = (s > 0) ? -1 : -INT_MAX;
  const int lane_up = (lane + 31) & 31, lane_dn = (lane + 1) & 31;      // owners of kk+1 / kk-1
  int d = 0, tail_seen = 0, alone = 0;
  long long dg_wait = 0, dg_fast = 0;                        // EX_DIAG: cycles waiting for ring space, fast-path waves
  int a0 = INT_MAX/2, b0 = INT_MAX/2, fleft = 0;             // staged tiles (none yet); waves until the next fast-path check
  bool fok = false;
  const unsigned head_a = smem_u32((const void *) &bx->head);
  while (true)
    { const int lowk0 = lowk, hghk0 = hghk;
      lowk -= 1; hghk += 1;
      const int top = hghk, ltop = (-top) & 31;
      const int kk = top - ((top + lane) & 31);
      const bool act = kk >= lowk;
      bool bail = (hghk - lowk > 30);
      const bool wide = bail;
      int cc = 0, mx = 0, nmore = 1;
      unsigned m = 0;
      //  ---- interior fast path: both contigs' 2-bit windows come from tiles staged in shared memory,
      //  no contig end within reach, at most two 32-base windows per slide.  Anything else (a longer
      //  run, a wave that does not advance the best point) is recomputed by the general code below.
      if (fleft == 0)
        { fok = (hghk - lowk <= 24 - EX_FASTN) && fast_window<s>(bx->tileA,bx->tileB,A,B,alen,blen,besta,lowk,hghk,a0,b0,lane);
          fleft = EX_FASTN;
        }
      fleft -= 1;
      bool fast = false;
      if (fok)
        { const int vp = __shfl_sync(FULL,rV,lane_up), vm = __shfl_sync(FULL,rV,lane_dn);
          const int c0 = max(max(vp,vm)+1,rV+2);
          const int xn0 = (c0 + kk) >> 1, yn0 = xn0 - kk;
          const int oa = act ? ((s > 0) ? xn0 - a0 : -xn0 - 32 - a0) : 64;    // idle lanes read a valid spot
          const int ob = act ? ((s > 0) ? yn0 - b0 : -yn0 - 32 - b0) : 64;
          u64 dd = win_t(bx->tileA,oa) ^ win_t(bx->tileB,ob);
          int t = dd ? ((s > 0) ? ((__ffsll((long long) dd)-1) >> 1) : (__clzll((long long) dd) >> 1)) : 32;
          bool lng = act && t == 32;
          if (__any_sync(FULL,lng))                                  // one more window for the 32-base runs
            { dd = win_t(bx->tileA,(s > 0) ? oa+32 : oa-32) ^ win_t(bx->tileB,(s > 0) ? ob+32 : ob-32);
              const int t2 = dd ? ((s > 0) ? ((__ffsll((long long) dd)-1) >> 1) : (__clzll((long long) dd) >> 1)) : 32;
              if (lng) t += t2;
              lng = lng && t2 == 32;
            }
          cc = c0 + 2*t;                                             // c0 + kk is even on every live diagonal
          mx = __reduce_max_sync(FULL,act ? cc : INT_MIN);
          m = rotr32(__ballot_sync(FULL,act && cc >= mx - WAVE_LAG),ltop);
          fast = !__any_sync(FULL,lng) && mx > besta;                // else: this wave over again, the general way
        }
      if (!fast && !bail)
        { fleft = 0;                                                 // a general wave may slide any distance: re-check
          const int vp = __shfl_sync(FULL,rV,lane_up), vm = __shfl_sync(FULL,rV,lane_dn);
          const int c0 = max(max(vp,vm)+1,rV+2);
          const int xn0 = (c0 + kk) >> 1;
          bool ended;
          const int t = snake_u<s>(A,B,alen,blen,act,xn0,kk,ended);
          const int xn = xn0 + t;
          cc = 2*xn - kk;
          mx = __reduce_max_sync(FULL,act ? cc : INT_MIN);
          int nlow = lowk, nhgh = hghk;
          if (mx <= besta) bail = true;
          else
            { const unsigned en = __ballot_sync(FULL,ended);
              if (en)                                              // a slide reached a contig end (rare)
                { const int flag = ended ? end_flag<s>(alen,blen,xn0,kk,t) : 0;
                  const unsigned hb = rotr32(__ballot_sync(FULL,flag == 1),ltop);
                  const unsigned hq = rotr32(__ballot_sync(FULL,flag == 2),ltop);
                  const unsigned eq = rotr32(__ballot_sync(FULL,act && cc == mx),ltop);
                  const int bx_ = __shfl_sync(FULL,xn,(ltop + __ffs(eq) - 1) & 31);
                  if (hb) { const int bcl = top - (__ffs(hb)-1);     if (nlow <= bcl) nlow = bcl+1; }
                  if (hq) { const int acl = top - (31 - __clz(hq));  if (nhgh >= acl) nhgh = acl-1; }
                  nmore = (b_at<s>(q,mx-bx_) != 4 && a_at<s>(q,bx_) != 4);
                }
              m = rotr32(__ballot_sync(FULL,kk >= nlow && kk <= nhgh && cc >= mx - WAVE_LAG),ltop);
              if (m == 0) bail = true;
            }
        }
      if (bail)
        { //  not a plain wave: undo it, let the back warp spill, finish alone
          lowk = lowk0; hghk = hghk0;
          if (!wide) alone = 1;                          // pathological wave: stay alone for the rest of the pass
          int spin = 0;
          while (d + 1 - bx->tail > EX_RING-1 && (bx->stop | bx->stopp) == 0) if (++spin > SPIN_LIMIT) break;
          __syncwarp();
          if (lane == 0)
            { bx->ring[(d+1) & (EX_RING-1)].cmd = 3;
              st_release_smem(&bx->head,d+1);
            }
          break;
        }
      d += 1;
      besta = mx;
      hghk = top - (__ffs(m)-1); lowk = top - (31 - __clz(m));
      rV = (kk >= lowk && kk <= hghk) ? cc : FRESH;
      if (EX_DIAG && fast) dg_fast += 1;
      if (d - tail_seen > EX_RING-1)
        { int spin = 0; const long long w0 = DIAG_CLOCK();
          while (d - (tail_seen = bx->tail) > EX_RING-1 && (bx->stop | bx->stopp) == 0) if (++spin > SPIN_LIMIT) break;
          dg_wait += DIAG_CLOCK() - w0;
        }
      RingEnt *e = &bx->ring[d & (EX_RING-1)];
      e->cc[lane] = cc;
      if (lane == 0)
        { *(int4 *) e = make_int4(nmore ? 1 : 2,top,lowk0-1,mx);
          *(int2 *) &e->lowk_after = make_int2(lowk,hghk);
        }
      if (!nmore || (d & 1) == 0)                        // publish every other wave
        { __syncwarp();
          if (lane == 0) st_release_smem_a(head_a,d);
        }
      if (!nmore || ((d & 7) == 0 && (bx->stop | bx->stopp) != 0)) break;
    }
  if (EX_DIAG && lane == 0) { bx->r_fwait = dg_wait; bx->r_ffast = dg_fast; }
  return make_int4(lowk,hghk,besta,alone);
}

template<int s, int W>
static __device__ __noinline__ int wave(Ctx &c, int low, int hgh, const int mida, int minp, int maxp,
                           const int aoff, int &endx, int &endy, int &diffs, int &trimha_out)
{ const int lane = threadIdx.x & 31;
  const unsigned lt = lanemask_lt();
  const int FRESH = (s > 0) ? -1 : -INT_MAX;
  const int tspace = c.tspace;
  int lowk, hghk, minpn, maxpn;

  if (s > 0) { lowk = low;  hghk = hgh;  minpn = minp;  maxpn = maxp; }
  else       { lowk = -hgh; hghk = -low; minpn = -maxp; maxpn = -minp; }
  if (hghk - lowk + 5 > W) return ST_BAND;

  c.avail = 0;
  int dif = 0, more = 1;
  int besta = s*mida, trima = besta, lasta = besta;
  int bestx = s*((mida+hgh)>>1), trimx = bestx;
  int trimd = 0, trimha = 0;
  int aclip = INT_MAX, bclip = -INT_MAX;
  bool anyhit = false;
  u64 ncell = 0;

  //  wave 0 (align.c:426-507 / :956-1036)
  for (int top = hghk; top >= lowk; top -= 32)
    { int kk = top - lane;
      bool act = kk >= lowk;
      int k = s*kk, x = (mida+k)>>1;
      int na, mark0, nan;
      if (s > 0)
        { na = ((x+(tspace-aoff))/tspace-1)*tspace+aoff; mark0 = na; nan = na + tspace; }
      else
        { na = ((x+(tspace-aoff)-1)/tspace-1)*tspace+aoff; mark0 = x; nan = -na; }
      if (c.avail + 32 > c.cmax) return ST_CELLS;
      unsigned am = __ballot_sync(FULL,act);
      int ha = c.avail + __popc(am & lt);
      c.avail += __popc(am);
      int hm = mark0;
      if (act)
        { Peb p; p.ptr = -1; p.diag = k; p.diff = 0; p.mark = mark0;
          c.cells[ha] = p;
        }
      int xn = s*x, flag = 0;
      if (act) xn += snake<s>(c,xn,kk,flag);
      int cc = 2*xn - kk;
      bool need = act && xn >= nan;
      while (__any_sync(FULL,need))
        { if (c.avail + 32 > c.cmax) return ST_CELLS;
          unsigned m = __ballot_sync(FULL,need);
          int idx = c.avail + __popc(m & lt);
          c.avail += __popc(m);
          if (need)
            { Peb p; p.ptr = ha; p.diag = k; p.diff = 0; p.mark = s*nan;
              c.cells[idx] = p;
              ha = idx; hm = s*nan; nan += tspace;
            }
          need = act && xn >= nan;
        }
      //  running maximum, descending kk = ascending lane
      int ex = max(warp_prefix_max_excl(act ? cc : INT_MIN,lane),besta);
      unsigned rm = __ballot_sync(FULL,act && cc > ex);
      if (rm)
        { int L = 31 - __clz(rm);
          besta = trima = lasta = __shfl_sync(FULL,cc,L);
          bestx = trimx = __shfl_sync(FULL,xn,L);
          trimha = __shfl_sync(FULL,ha,L);
        }
      unsigned hb = __ballot_sync(FULL,act && flag == 1);
      unsigned hq = __ballot_sync(FULL,act && flag == 2);
      if (hb) { anyhit = true; int v = top - (__ffs(hb)-1); if (bclip < v) bclip = v; }
      if (hq) { anyhit = true; aclip = top - (31 - __clz(hq)); }
      if (act)
        { c.V[IX(kk)] = cc; c.T[IX(kk)] = PATH_INT; c.HA[IX(kk)] = ha; c.HM[IX(kk)] = hm;
          c.NA[IX(kk)] = nan;
        }
    }
  __syncwarp();
  if (anyhit)
    { more = (b_at<s>(c,besta-bestx) != 4 && a_at<s>(c,bestx) != 4);
      if (hghk >= aclip) hghk = aclip-1;
      if (lowk <= bclip) lowk = bclip+1;
      aclip = INT_MAX; bclip = -INT_MAX; anyhit = false;
    }

  //  successive waves (align.c:546-800 / :1077-1330)
  bool inreg = false;                          // state of the band is in the r* registers
  int rV = 0, rHA = 0, rHM = 0, rNA = 0; u64 rT = 0;
  const int lane_up = (lane + 31) & 31, lane_dn = (lane + 1) & 31;      // owners of kk+1 / kk-1

  bool pair_ok = EX_PAIR && c.box != NULL && minp == -INT_MAX && maxp == INT_MAX;
  while (more && lasta >= besta - TRIM_MLAG)
    {
      //  ---- front/back pairing (see PairBox): this warp keeps only V and the band ----
      if (EX_PAIR && pair_ok && hghk >= lowk && hghk - lowk <= 24)
        { PairBox *const bx = reinterpret_cast<PairBox *>(ex_smem + c.box_off);
          const SeqV q = { c.A, c.B, c.alen, c.blen };
          if (inreg)                                   // the band of the last wave goes to the arrays
            { const int kk = hghk - ((lane - ((-hghk) & 31)) & 31);
              if (kk >= lowk)
                { c.V[IX(kk)] = rV; c.T[IX(kk)] = rT; c.HA[IX(kk)] = rHA; c.HM[IX(kk)] = rHM; c.NA[IX(kk)] = rNA; }
              inreg = false;
            }
          __syncwarp();
          if (lane == 0)
            { bx->lowk = lowk; bx->hghk = hghk; bx->besta = besta; bx->lasta = lasta; bx->trima = trima;
              bx->trimx = trimx; bx->trimd = trimd; bx->trimha = trimha; bx->avail = c.avail;
              bx->tspace = tspace; bx->path_ave = c.path_ave; bx->cmax = c.cmax; bx->wmask = W-1; bx->dif0 = dif;
              bx->cells = c.cells; bx->V = c.V; bx->HA = c.HA; bx->HM = c.HM; bx->NA = c.NA; bx->T = c.T;
              bx->head = 0; bx->tail = 0; bx->stop = 0; bx->tailt = 0; bx->stopp = 0;
              bx->cmd = (s > 0) ? 1 : 2;
              st_release_smem(&bx->seq,bx->seq + 1);
            }
          __syncwarp();
          { const int kk = hghk - ((lane - ((-hghk) & 31)) & 31);
            rV = (kk >= lowk) ? c.V[IX(kk)] : FRESH;
          }
          int stp = 0;
          long long fwait = 0; const long long ft0 = DIAG_CLOCK();
          { const int4 fr = front_run<s>(c.box_off,q.A,q.B,q.alen,q.blen,lowk,hghk,besta,rV);
            lowk = fr.x; hghk = fr.y; besta = fr.z;
            if (fr.w) pair_ok = false;
          }
          { int spin = 0; long long w0 = DIAG_CLOCK();
            while ((stp = ld_acquire_smem(&bx->stop)) == 0) if (++spin > SPIN_LIMIT) { stp = 1; break; }
            spin = 0;
            while (ld_acquire_smem(&bx->stopp) == 0) if (++spin > SPIN_LIMIT) break;      // the pebble warp too
            fwait += DIAG_CLOCK() - w0;
            (void) fwait; (void) ft0;
          }
          const int bst = bx->pstatus != ST_OK ? bx->pstatus : bx->status;
          lasta = bx->r_lasta; trima = bx->r_trima; trimx = bx->r_trimx; trimd = bx->r_trimd; trimha = bx->r_trimha;
          if (EX_DIAG) { c.bwait += (u64) bx->r_bwait; c.btot += (u64) bx->r_btot; c.fwait += (u64) bx->r_fwait; c.ftot += (u64) bx->r_ffast; }
          c.avail = bx->r_avail; c.pwaves += (u64) (bx->r_dif - dif); c.npairs += 1; dif = bx->r_dif; ncell += bx->r_ncell;
          __syncwarp();
          if (bst != ST_OK) return bst;
          if (stp == 1) more = 0;                        // the pass ended in the back warp
          //  stp == 2: handed back after wave dif; lowk/hghk/besta are this warp's own
          continue;
        }


      lowk -= 1; hghk += 1;
      if (hghk - lowk + 5 > W) return ST_BAND;
      if (dif > c.alen + c.blen + 1000) return ST_STAGE;     // cannot happen (every wave is one more difference): hang guard
      //  new band edges (align.c:611-622): a fresh diagonal copies its neighbour's NA and counts as
      //  FRESH; done with predicates on the owning lanes instead of stores + a warp barrier
      const bool newlow = (lowk >= minpn), newhgh = (hghk <= maxpn);
      if (!newlow) lowk += 1;
      if (!newhgh) hghk -= 1;
      dif += 1;
      ncell += (u64) (hghk - lowk + 1);

      if (!EX_NOREG && hghk - lowk < 32)
        { //  ---- register path: lane (-kk & 31) owns diagonal kk ----
          const int top = hghk, ltop = (-top) & 31;
          const int kk = top - ((lane - ltop) & 31);
          const bool act = kk >= lowk;
          if (!inreg)
            { rV = c.V[IX(kk)]; rT = c.T[IX(kk)]; rHA = c.HA[IX(kk)]; rHM = c.HM[IX(kk)]; rNA = c.NA[IX(kk)];
              inreg = true;
            }
          const bool flo = newlow && kk == lowk, fhi = newhgh && kk == top;
          int vp = __shfl_sync(FULL,rV,lane_up), vm = __shfl_sync(FULL,rV,lane_dn);
          //  a fresh edge diagonal is FRESH for itself AND for the neighbour that looks at it
          int ap = (kk == top  || (newhgh && kk+1 == top))  ? FRESH : vp;
          int ac = (flo || fhi) ? FRESH : rV;
          int am = (kk == lowk || (newlow && kk-1 == lowk)) ? FRESH : vm;
          int pred, cc;
          if (ac < am) { if (am < ap) { pred = 1; cc = ap+1; } else { pred = -1; cc = am+1; } }
          else         { if (ac < ap) { pred = 1; cc = ap+1; } else { pred = 0;  cc = ac+2; } }
          const int src = (lane - pred) & 31;
          u64 b  = __shfl_sync(FULL,rT,src);
          int ha = __shfl_sync(FULL,rHA,src), hm = __shfl_sync(FULL,rHM,src);
          int nn = __shfl_sync(FULL,rNA,src);            // a fresh edge always descends from its one neighbour
          int nan = (flo || fhi) ? nn : rNA;

          b <<= 1;
          int xn = (cc + kk) >> 1, flag = 0, k = s*kk;
          if (act)
            { int t = snake<s>(c,xn,kk,flag);
              xn += t;
              b = (t >= 64) ? ~0ull : ((b << t) | ((1ull << t) - 1));
            }
          cc = 2*xn - kk;

          bool need = act && xn >= nan;
          while (__any_sync(FULL,need))
            { bool create = need && (s*hm < nan);
              if (c.avail + 32 > c.cmax) return ST_CELLS;
              unsigned m = __ballot_sync(FULL,create);
              int idx = c.avail + __popc(m & lt);
              c.avail += __popc(m);
              if (create)
                { Peb p; p.ptr = ha; p.diag = k; p.diff = dif; p.mark = s*nan;
                  c.cells[idx] = p;
                  ha = idx; hm = s*nan;
                }
              if (need) nan += tspace;
              need = act && xn >= nan;
            }
          if (act) { rV = cc; rT = b; rHA = ha; rHM = hm; rNA = nan; }

          //  masks below are rotated into "position" space: bit p = diagonal top-p
          int cm = act ? cc : INT_MIN;
          int mx = __reduce_max_sync(FULL,cm);
          if (mx > besta)
            { //  Pb = highest diagonal reaching the wave maximum = the last record setter of the
              //  sequential scan.  If it passes both quality tests it alone decides lasta and the
              //  trim point; otherwise fall back to the full prefix-max.
              unsigned eq = rotr32(__ballot_sync(FULL,cm == mx),ltop);
              int Lb = (ltop + __ffs(eq) - 1) & 31;
              bool qual = act && cc > besta && __popcll(b & PATH_WIN) >= c.path_ave;
              bool tq = qual && trim_ok(c,b);
              unsigned ql = __ballot_sync(FULL,qual), tl = __ballot_sync(FULL,tq);
              if ((tl >> Lb) & 1)
                { lasta = mx; trima = mx; trimd = dif;
                  trimx  = __shfl_sync(FULL,xn,Lb);
                  trimha = __shfl_sync(FULL,ha,Lb);
                }
              else
                { int cp = __shfl_sync(FULL,cm,(ltop + lane) & 31);      // value at position = lane
                  int ex = max(warp_prefix_max_excl(cp,lane),besta);
                  unsigned rm = __ballot_sync(FULL,cp > ex);
                  unsigned qm = rm & rotr32(ql,ltop), tm = rm & rotr32(tl,ltop);
                  if (qm) lasta = __shfl_sync(FULL,cc,(ltop + 31 - __clz(qm)) & 31);
                  if (tm)
                    { int L3 = (ltop + 31 - __clz(tm)) & 31;
                      trima  = __shfl_sync(FULL,cc,L3);
                      trimx  = __shfl_sync(FULL,xn,L3);
                      trimha = __shfl_sync(FULL,ha,L3);
                      trimd  = dif;
                    }
                }
              besta = mx;
              bestx = __shfl_sync(FULL,xn,Lb);
            }
          if (__any_sync(FULL,act && flag != 0))
            { unsigned hb = rotr32(__ballot_sync(FULL,act && flag == 1),ltop);
              unsigned hq = rotr32(__ballot_sync(FULL,act && flag == 2),ltop);
              if (hb) { int v = top - (__ffs(hb)-1); if (bclip < v) bclip = v; }
              if (hq) aclip = top - (31 - __clz(hq));
              more = (b_at<s>(c,besta-bestx) != 4 && a_at<s>(c,bestx) != 4);
              if (hghk >= aclip) hghk = aclip-1;
              if (lowk <= bclip) lowk = bclip+1;
              aclip = INT_MAX; bclip = -INT_MAX;
            }
          //  trim the band to points within WAVE_LAG of the best (align.c:782-790)
          unsigned m = rotr32(__ballot_sync(FULL,kk >= lowk && kk <= hghk && cc >= besta - WAVE_LAG),ltop);
          if (m == 0) hghk = lowk-1;
          else { hghk = top - (__ffs(m)-1); lowk = top - (31 - __clz(m)); }
          continue;
        }

      //  ---- wide band: state in the arrays of c, 32-diagonal chunks ----
      if (inreg)
        { const int otop = hghk - (newhgh ? 1 : 0), olow = lowk + (newlow ? 1 : 0);   // band of the last wave
          const int kk = otop - ((lane - ((-otop) & 31)) & 31);
          if (kk >= olow)
            { c.V[IX(kk)] = rV; c.T[IX(kk)] = rT; c.HA[IX(kk)] = rHA; c.HM[IX(kk)] = rHM; c.NA[IX(kk)] = rNA; }
          inreg = false;
          __syncwarp();
        }
      for (int top = hghk; top >= lowk; top -= 32)
        { int kk = top - lane;
          bool act = kk >= lowk;
          const bool flo = newlow && kk == lowk, fhi = newhgh && kk == hghk;
          int ap = (kk == hghk || (newhgh && kk+1 == hghk)) ? FRESH
                                                            : ((lane == 0) ? c.carry[0] : c.V[IX(kk+1)]);
          int ac = (flo || fhi) ? FRESH : c.V[IX(kk)];
          int am = (kk == lowk || (newlow && kk-1 == lowk)) ? FRESH : c.V[IX(kk-1)];
          int pred, cc;
          if (ac < am) { if (am < ap) { pred = 1; cc = ap+1; } else { pred = -1; cc = am+1; } }
          else         { if (ac < ap) { pred = 1; cc = ap+1; } else { pred = 0;  cc = ac+2; } }
          u64 b; int ha, hm;
          if (pred == 1 && lane == 0)
            { b  = (u64) (unsigned) c.carry[1] | ((u64) (unsigned) c.carry[2] << 32);
              ha = c.carry[3]; hm = c.carry[4];
            }
          else
            { int si = IX(kk+pred);
              b = c.T[si]; ha = c.HA[si]; hm = c.HM[si];
            }
          int nan = c.NA[IX(flo ? kk+1 : (fhi ? kk-1 : kk))];
          //  the fresh low edge copies the OLD NA of the diagonal above it (align.c:611-613, before
          //  the wave): if that diagonal closed the previous chunk it has been updated already
          if (flo && lane == 0 && top != hghk) nan = c.carry[5];
          //  lane 31's own old state is the next chunk's "kk+1"
          int  o_v = 0, o_ha = 0, o_hm = 0, o_na = 0; u64 o_t = 0;
          const bool morechunks = (top - 32 >= lowk);
          if (lane == 31 && morechunks)
            { o_v = ac; o_t = c.T[IX(kk)]; o_ha = c.HA[IX(kk)]; o_hm = c.HM[IX(kk)]; o_na = c.NA[IX(kk)]; }
          __syncwarp();                              // all reads of old state done
          if (lane == 31 && morechunks)
            { c.carry[0] = o_v; c.carry[1] = (int) (unsigned) o_t; c.carry[2] = (int) (o_t >> 32);
              c.carry[3] = o_ha; c.carry[4] = o_hm; c.carry[5] = o_na;
            }

          b <<= 1;
          int xn = (cc + kk) >> 1, flag = 0, k = s*kk;
          if (act)
            { int t = snake<s>(c,xn,kk,flag);
              xn += t;
              b = (t >= 64) ? ~0ull : ((b << t) | ((1ull << t) - 1));
            }
          cc = 2*xn - kk;

          bool need = act && xn >= nan;
          while (__any_sync(FULL,need))
            { bool create = need && (s*hm < nan);
              if (c.avail + 32 > c.cmax) return ST_CELLS;
              unsigned m = __ballot_sync(FULL,create);
              int idx = c.avail + __popc(m & lt);
              c.avail += __popc(m);
              if (create)
                { Peb p; p.ptr = ha; p.diag = k; p.diff = dif; p.mark = s*nan;
                  c.cells[idx] = p;
                  ha = idx; hm = s*nan;
                }
              if (need) nan += tspace;
              need = act && xn >= nan;
            }

          int cm = act ? cc : INT_MIN;
          int mx = __reduce_max_sync(FULL,cm);
          if (mx > besta)
            { unsigned eq = __ballot_sync(FULL,cm == mx);
              int Lb = __ffs(eq) - 1;
              bool qual = act && cc > besta && __popcll(b & PATH_WIN) >= c.path_ave;
              bool tq = qual && trim_ok(c,b);
              unsigned ql = __ballot_sync(FULL,qual), tl = __ballot_sync(FULL,tq);
              if ((tl >> Lb) & 1)
                { lasta = mx; trima = mx; trimd = dif;
                  trimx  = __shfl_sync(FULL,xn,Lb);
                  trimha = __shfl_sync(FULL,ha,Lb);
                }
              else
                { int ex = max(warp_prefix_max_excl(cm,lane),besta);
                  unsigned rm = __ballot_sync(FULL,act && cc > ex);
                  unsigned qm = rm & ql, tm = rm & tl;
                  if (qm) lasta = __shfl_sync(FULL,cc,31 - __clz(qm));
                  if (tm)
                    { int L3 = 31 - __clz(tm);
                      trima  = __shfl_sync(FULL,cc,L3);
                      trimx  = __shfl_sync(FULL,xn,L3);
                      trimha = __shfl_sync(FULL,ha,L3);
                      trimd  = dif;
                    }
                }
              besta = mx;
              bestx = __shfl_sync(FULL,xn,Lb);
            }
          if (__any_sync(FULL,act && flag != 0))
            { unsigned hb = __ballot_sync(FULL,act && flag == 1);
              unsigned hq = __ballot_sync(FULL,act && flag == 2);
              anyhit = true;
              if (hb) { int v = top - (__ffs(hb)-1); if (bclip < v) bclip = v; }
              if (hq) aclip = top - (31 - __clz(hq));
            }
          if (act)
            { c.V[IX(kk)] = cc; c.T[IX(kk)] = b; c.HA[IX(kk)] = ha; c.HM[IX(kk)] = hm;
              c.NA[IX(kk)] = nan;
            }
          __syncwarp();
        }

      if (anyhit)
        { more = (b_at<s>(c,besta-bestx) != 4 && a_at<s>(c,bestx) != 4);
          if (hghk >= aclip) hghk = aclip-1;
          if (lowk <= bclip) lowk = bclip+1;
          aclip = INT_MAX; bclip = -INT_MAX; anyhit = false;
        }

      //  trim the band to points within WAVE_LAG of the best (align.c:782-790)
      { int n = besta - WAVE_LAG, nh = lowk-1;
        for (int top = hghk; top >= lowk; top -= 32)
          { int kk = top - lane;
            unsigned m = __ballot_sync(FULL,kk >= lowk && c.V[IX(kk)] >= n);
            if (m) { nh = top - (__ffs(m)-1); break; }
          }
        hghk = nh;
        for (int bot = lowk; bot <= hghk; bot += 32)
          { int kk = bot + lane;
            unsigned m = __ballot_sync(FULL,kk <= hghk && c.V[IX(kk)] >= n);
            if (m) { lowk = bot + (__ffs(m)-1); break; }
          }
      }
    }

  c.nwaves += (u64) dif; c.ncells += ncell;
  endx = s*trimx;
  endy = s*(trima - trimx);
  diffs = trimd;
  trimha_out = trimha;
  return ST_OK;
}

//  Forward read-out (align.c:805-870) into c.fstage as bytes.  Warp-uniform; lane 0 stores.

static __device__ int fwd_extract(Ctx &c, int trimha, int mida, int trimx, int trimy, int trimd,
                                  int &tlen, int &root_diag)
{ const int lane = threadIdx.x & 31;
  //  ONE walk of the pebble chain (each hop is a dependent L2 round trip): the pairs come out last
  //  to first, so they are written downwards from the top of the staging buffer and moved to its
  //  start afterwards (warp-parallel) instead of counting the chain first.
  PebWalk W; W.init(c.cells,c.pwin,c.pwin_n);
  Peb tip = W.at(trimha);
  int kt = tip.diag, bt, et;
  if (tip.ptr < 0) { bt = (mida - kt) >> 1; et = 0; }
  else             { bt = tip.mark - kt;    et = tip.diff; }
  int extra = (bt + kt != trimx);
  int pos = c.smax & ~1;                                  // next pair goes to [pos-2,pos)
  int addd = 0, addb = 0;                                 // adjustment of the last pair
  if (extra)
    { if (pos < 2) return ST_STAGE;
      if (lane == 0)
        { c.fstage[pos-2] = (unsigned char) (trimd - et);
          c.fstage[pos-1] = (unsigned char) (trimy - bt);
        }
      pos -= 2;
    }
  else if (bt != trimy)
    { addd = trimd - et; addb = trimy - bt; }
  bool first = true;
  Peb cur = tip;
  root_diag = kt;
  while (cur.ptr >= 0)
    { Peb prv = W.at(cur.ptr);
      int a = cur.mark - cur.diag, d = cur.diff, bp, ep;
      if (prv.ptr < 0) { bp = (mida - prv.diag) >> 1; ep = 0; }
      else             { bp = prv.mark - prv.diag;    ep = prv.diff; }
      int pd = d - ep, pb = a - bp;
      if (first) { pd += addd; pb += addb; first = false; }
      if (pos < 2) return ST_STAGE;
      if (lane == 0)
        { c.fstage[pos-2] = (unsigned char) pd;
          c.fstage[pos-1] = (unsigned char) pb;
        }
      pos -= 2;
      cur = prv;
      root_diag = cur.diag;
    }
  const int top = c.smax & ~1, len = top - pos;
  __syncwarp();
  if (pos > 0)
    for (int o = 0; o < len; o += 32)                     // move down; reads stay ahead of writes
      { unsigned char v = 0;
        if (o + lane < len) v = c.fstage[pos + o + lane];
        __syncwarp();
        if (o + lane < len) c.fstage[o + lane] = v;
        __syncwarp();
      }
  tlen = len;
  return ST_OK;
}

//  Reverse read-out (align.c:1334-1414): pairs in FINAL order (tip first) into c.rstage; the
//  start-not-on-a-trace-point case folds its pair into the first forward pair (c.fstage[0..1]).

static __device__ int rev_extract(Ctx &c, const Peb *cells, int trimha, int aoff, int trimx, int trimy,
                                  int trimd, int ftlen, int &rtlen)
{ const int lane = threadIdx.x & 31;
  int n = 0, h, root = trimha;
  PebWalk W; W.init(cells,c.pwin,c.pwin_n);
  for (h = trimha; h >= 0; h = W.at(h).ptr) { n += 1; root = h; }
  Peb r0 = W.at(root);
  int b0 = r0.mark - r0.diag;
  bool offpt = ((b0 + r0.diag) % c.tspace != aoff);
  int wr = 0;                                        // bytes written to rstage so far

  if (n == 1)
    { if (offpt)                                     // single pair (trimd, b0 - trimy), h < 0 after
        { int pd = trimd, pb = b0 - trimy;
          if (ftlen == 0)
            { if (2 > c.smax) return ST_STAGE;
              if (lane == 0) { c.rstage[0] = (unsigned char) pd; c.rstage[1] = (unsigned char) pb; }
              wr = 2;
            }
          else if (lane == 0)
            { c.fstage[0] = (unsigned char) (c.fstage[0] + pd);
              c.fstage[1] = (unsigned char) (c.fstage[1] + pb);
            }
        }
      else
        { int k = r0.diag, b = b0, e = 0;
          if (b + k != trimx)
            { if (2 > c.smax) return ST_STAGE;
              if (lane == 0)
                { c.rstage[0] = (unsigned char) (trimd - e); c.rstage[1] = (unsigned char) (b - trimy); }
              wr = 2;
            }
          else if (b != trimy && lane == 0)          // adjusts the first forward pair (atrace[atlen])
            { c.fstage[0] = (unsigned char) (c.fstage[0] + (trimd - e));
              c.fstage[1] = (unsigned char) (c.fstage[1] + (b - trimy));
            }
        }
      __syncwarp();
      rtlen = wr;
      return ST_OK;
    }

  //  n >= 2: pairs i = n-1 .. 1 between chain cells c_i and c_(i-1); pair 1 is merged into the
  //  forward trace when the root is off a trace point and a forward trace exists.
  Peb tip = W.at(trimha);
  int kt = tip.diag, bt = tip.mark - kt, et = tip.diff;
  bool extra = (bt + kt != trimx);
  int addd = 0, addb = 0;
  bool merged = offpt && ftlen != 0;
  int npairs = (n-1) - (merged ? 1 : 0) + (extra ? 1 : 0);
  if (2*npairs > c.smax) return ST_STAGE;
  if (extra)
    { if (lane == 0)
        { c.rstage[0] = (unsigned char) (trimd - et); c.rstage[1] = (unsigned char) (bt - trimy); }
      wr = 2;
    }
  else if (bt != trimy)
    { addd = trimd - et; addb = bt - trimy; }        // onto the most recently generated pair
  Peb cur = tip;
  int idx = n-1;
  while (cur.ptr >= 0)
    { Peb prv = W.at(cur.ptr);
      int a = cur.mark - cur.diag, d = cur.diff;
      int bp = prv.mark - prv.diag, ep = (prv.ptr < 0) ? 0 : prv.diff;
      int pd = d - ep, pb = bp - a;
      if (idx == n-1) { pd += addd; pb += addb; }
      if (idx == 1 && merged)
        { if (lane == 0)
            { c.fstage[0] = (unsigned char) (c.fstage[0] + pd);
              c.fstage[1] = (unsigned char) (c.fstage[1] + pb);
            }
        }
      else
        { if (lane == 0) { c.rstage[wr] = (unsigned char) pd; c.rstage[wr+1] = (unsigned char) pb; }
          wr += 2;
        }
      idx -= 1;
      cur = prv;
    }
  __syncwarp();
  rtlen = wr;
  return ST_OK;
}

struct LAres { int abpos, bbpos, aepos, bepos, diffs, ftlen, rtlen; };

//  Local_Alignment (align.c:1423-1576), lbord = hbord = -1 and A != B (non-self).

//  lbord / hbord >= 0 confine the band to [low-lbord, hgh+hbord] (align.c:1466-1481; aseq != bseq
//  always here, so the "selfie" defaults never apply): used for a contig against itself.
template<int W>
static __device__ int local_alignment(Ctx &c, int acomp, int low, int hgh, int anti, LAres &R,
                                      int lbord = -1, int hbord = -1)
{ int aoff = acomp ? (c.alen % c.tspace) : 0;
  int ex, ey, df, tha, st, rootd = 0;

  while (((anti-hgh)>>1) < 0) hgh -= 1;
  const int minp = (lbord < 0) ? -INT_MAX : low - lbord;
  const int maxp = (hbord < 0) ?  INT_MAX : hgh + hbord;

  R.ftlen = R.rtlen = 0; R.diffs = 0;
  long long tk = clock64();
  st = wave<1,W>(c,low,hgh,anti,minp,maxp,aoff,ex,ey,df,tha);
  c.cyc_wave += (u64) (clock64() - tk); tk = clock64();
  int st2 = st ? 0 : fwd_extract(c,tha,anti,ex,ey,df,R.ftlen,rootd);
  c.cyc_extract += (u64) (clock64() - tk);
  __syncwarp();
  if (st) return st;
  if (st2) return st2;
  R.aepos = ex; R.bepos = ey; R.diffs = df;
  low = rootd;
  bool fshort = ((R.aepos + R.bepos) - anti < DUB_TRIM);

  tk = clock64();
  st = wave<-1,W>(c,low,low,anti,minp,maxp,aoff,ex,ey,df,tha);
  if (st) return st;
  c.cyc_wave += (u64) (clock64() - tk); tk = clock64();
  st = rev_extract(c,c.cells,tha,aoff,ex,ey,df,R.ftlen,R.rtlen);
  if (st) return st;
  c.cyc_extract += (u64) (clock64() - tk);
  R.abpos = ex; R.bbpos = ey; R.diffs += df;
  bool rshort = (anti - (R.abpos + R.bbpos) < DUB_TRIM);

  if (fshort)
    { if (rshort)
        { R.aepos = R.abpos = (R.abpos + R.aepos) >> 1;
          R.bepos = R.bbpos = (R.bbpos + R.bepos) >> 1;
          R.ftlen = R.rtlen = 0;
        }
      else
        { low  = R.abpos - R.bbpos;
          anti = R.abpos + R.bbpos;
          R.ftlen = R.rtlen = 0;
          st = wave<1,W>(c,low,low,anti,minp,maxp,aoff,ex,ey,df,tha);
          if (st) return st;
          st = fwd_extract(c,tha,anti,ex,ey,df,R.ftlen,rootd);
          if (st) return st;
          R.aepos = ex; R.bepos = ey; R.diffs = df;
        }
    }
  else if (rshort)
    { low  = R.aepos - R.bepos;
      anti = R.aepos + R.bepos;
      R.ftlen = R.rtlen = 0; R.diffs = 0;
      st = wave<-1,W>(c,low,low,anti,minp,maxp,aoff,ex,ey,df,tha);
      if (st) return st;
      st = rev_extract(c,c.cells,tha,aoff,ex,ey,df,0,R.rtlen);
      if (st) return st;
      R.abpos = ex; R.bbpos = ey; R.diffs += df;
    }
  __syncwarp();
  return ST_OK;
}

#define OUT_HDR 40        // bytes: triple, seq, pairkey, abpos, bbpos, aepos, bepos, diffs, tlen, 0

//  Appends one alignment record; ACOMP flip of coordinates and trace order (align.c:1534-1557).

static __device__ void emit_record(const ext_params &P, Ctx &c, const LAres &R, int acomp,
                                   unsigned triple, int seq, unsigned pairkey)
{ const int lane = threadIdx.x & 31;
  int tlen = R.rtlen + R.ftlen;
  u64 need = OUT_HDR + ((tlen + 7) & ~7);
  u64 off = 0;
  if (lane == 0) off = atomicAdd(P.out_used,need);
  off = __shfl_sync(FULL,off,0);
  if (off + need > P.out_cap) return;                 // host sees out_used > cap and retries
  unsigned char *o = P.out + off;
  if (lane == 0)
    { int *h = (int *) o;
      int ab = R.abpos, bb = R.bbpos, ae = R.aepos, be = R.bepos;
      if (acomp)
        { ab = c.alen - R.aepos; ae = c.alen - R.abpos;
          bb = c.blen - R.bepos; be = c.blen - R.bbpos;
        }
      h[0] = (int) triple; h[1] = seq; h[2] = (int) pairkey;
      h[3] = ab; h[4] = bb; h[5] = ae; h[6] = be; h[7] = R.diffs; h[8] = tlen; h[9] = P.attempt;
    }
  unsigned char *t = o + OUT_HDR;
  for (int i = lane*2; i < tlen; i += 64)             // pair i/2 of the un-flipped trace
    { const unsigned char *src = (i < R.rtlen) ? (c.rstage + i) : (c.fstage + (i - R.rtlen));
      int dst = acomp ? (tlen - 2 - i) : i;
      t[dst] = src[0]; t[dst+1] = src[1];
    }
}

//  Walks one triple: chain scan (FastGA.c:3087-3162), tube stepping (:3205-3340).
//  ALIGN = false: count qualifying chains only (prefilter).

//  Sequential reader over the sorted seeds.  STAGED (warp-uniform callers): a 32-record window
//  is staged in shared memory with one coalesced 512-byte load, so the serial chain scan sees
//  shared-memory latency instead of a dependent HBM/L2 round trip per seed.

template<bool STAGED> struct SeedRd
{ const rec128 *S; rec128 *buf; unsigned base, n;
  __device__ __forceinline__ void init(const rec128 *s, rec128 *b, unsigned nn)
    { S = s; buf = b; n = nn; base = 0xffffffffu; }
  __device__ __forceinline__ rec128 get(unsigned i)
    { if (!STAGED) return S[i];
      if (i - base >= 32u)
        { __syncwarp();
          base = i;
          unsigned k = i + (threadIdx.x & 31);
          if (k < n) st_rec(buf + (threadIdx.x & 31),ld_rec(S + k));
          __syncwarp();
        }
      return buf[i - base];
    }
};

template<bool ALIGN>
static __device__ int scan_triple(const ext_params &P, Ctx &c, unsigned j, unsigned &nhit_out,
                                  u64 &nla, rec128 *stagebuf)
{ const rec128 *S = P.seeds;
  unsigned b = P.seg_start[j], m = P.seg_start[j+1];
  SeedRd<ALIGN> RL, RU;
  RL.init(S,stagebuf,(unsigned) P.nseeds);
  RU.init(S,stagebuf + 32,(unsigned) P.nseeds);
  rec128 r0 = S[b];
  u64 grp = get_bits(r0,P.p_jc,P.jc_bits + P.ic_bits + 1);
  long long cdiag = (long long) get_bits(r0,P.p_band,P.band_bits);
  bool isnew = true, aux = false;
  if (j > 0)
    { rec128 rp = S[P.seg_start[j-1]];
      if (get_bits(rp,P.p_jc,P.jc_bits + P.ic_bits + 1) == grp &&
          (long long) get_bits(rp,P.p_band,P.band_bits) == cdiag-1)
        isnew = false;
    }
  unsigned e = m;
  if (j+1 < (unsigned) P.nseg)
    { rec128 rn = S[m];
      if (get_bits(rn,P.p_jc,P.jc_bits + P.ic_bits + 1) == grp &&
          (long long) get_bits(rn,P.p_band,P.band_bits) == cdiag+1)
        { aux = true; e = P.seg_start[j+2]; }
    }
  nhit_out = 0;
  if (!isnew && !aux) return ST_OK;

  int comp = (int) get_bits(r0,P.p_cp,1);
  unsigned pairkey = (unsigned) get_bits(r0,P.p_jc,P.jc_bits + P.ic_bits + 1);
  long long alen = 0, blen = 0, mlen = 0, doffset = 0, aoffset = 0;
  if (ALIGN)
    { int ctg1 = P.aperm[get_bits(r0,P.p_ic,P.ic_bits)];
      int ctg2 = P.bperm[get_bits(r0,P.p_jc,P.jc_bits)];
      alen = P.aclen[ctg1]; blen = P.bclen[ctg2]; mlen = alen + blen;
      doffset = alen - (P.amxpos + P.bmxpos); aoffset = alen - P.amxpos;
      c.A = (const unsigned *) ((comp ? P.arseq : P.aseq) + P.awoff[ctg1]);
      c.B = (const unsigned *) (P.bseq + P.bwoff[ctg2]);
      c.alen = (int) alen; c.blen = (int) blen;
      c.anw = (alen + 31) >> 5; c.bnw = (blen + 31) >> 5;
    }

  const long long LMAX = 0x7fffffffffffffffll;
  long long alast = -1, ahgh, alow, amid, anti, eant, ipost, apost;
  unsigned s = b, t = m;
  int go = 1, lcp, wch, mix = 0, cov = 0, dgmin, dgmax, dg, seq = 0;

  ipost = (long long) get_bits(RL.get(s),P.p_anti,P.anti_bits);
  apost = aux ? (long long) get_bits(RU.get(t),P.p_anti,P.anti_bits) : LMAX;
  dgmin = 2*BUCK_WIDTH; dgmax = 0;
  ahgh  = -P.chain_break;
  alow  = (apost < ipost) ? apost : ipost;
  while (go)
    { if (apost < ipost)
        { rec128 r = RU.get(t);
          lcp = (int) (r.lo & 63); dg = (int) ((r.lo >> 6) & 63) + BUCK_WIDTH;
          anti = apost;
          t += 1;
          apost = (t >= e) ? LMAX : (long long) get_bits(RU.get(t),P.p_anti,P.anti_bits);
          wch = 2;
        }
      else
        { if (s < m) { rec128 r = RL.get(s); lcp = (int) (r.lo & 63); dg = (int) ((r.lo >> 6) & 63); }
          else       { lcp = 0; dg = 0; }
          anti = ipost;
          s += 1;
          if (s >= m) { if (s > m) go = 0; else ipost = LMAX; }
          else ipost = (long long) get_bits(RL.get(s),P.p_anti,P.anti_bits);
          wch = 1;
        }
      lcp <<= 1;

      if (anti < ahgh + P.chain_break)
        { long long cps = anti + lcp;
          if (cps > ahgh)
            { if (anti >= ahgh) cov += lcp; else cov += (int) (cps - ahgh);
              ahgh = cps;
            }
          mix |= wch;
          if (dg < dgmin) dgmin = dg; else if (dg > dgmax) dgmax = dg;
        }
      else
        { if (cov >= P.chain_min && (mix != 1 || isnew))
            { nhit_out += 1;
              if (ALIGN)
                { dgmin += (int) (cdiag << BUCK_SHIFT);
                  dgmax += (int) (cdiag << BUCK_SHIFT);
                  if (comp)
                    { dgmin += (int) doffset; dgmax += (int) doffset; alow += aoffset; ahgh += aoffset; }
                  else
                    { dgmin -= (int) P.bmxpos; dgmax -= (int) P.bmxpos; }
                  if (ahgh > alast)
                    { if (alow < alast) alow = alast;
                      ahgh -= BUCK_ANTI;
                      do
                        { amid = alow + BUCK_ANTI;
                          if (amid > ahgh)
                            { amid = ahgh;
                              if (amid + dgmin < 0)
                                { dgmin = (int) -amid;
                                  if (dgmin > dgmax) break;
                                }
                            }
                          LAres R;
                          int st = local_alignment<EX_W>(c,comp,dgmin,dgmax,(int) amid,R);
                          if (st) return st;
                          nla += 1;
                          int ab = R.abpos, bb = R.bbpos, ae = R.aepos, be = R.bepos;
                          int rlen = ae - ab;              // same after the ACOMP flip
                          if (rlen >= P.aln_min && P.aln_rate*rlen >= (double) R.diffs)
                            { emit_record(P,c,R,comp,j,seq,pairkey);
                              seq += 1;
                            }
                          //  eant in the flipped frame (FastGA.c:3309-3312) == un-flipped end
                          if (comp) eant = mlen - ((alen - ae) + (blen - be));
                          else      eant = (long long) ae + be;
                          (void) ab; (void) bb;
                          if (eant <= alow) alow = amid; else alow = eant;
                        }
                      while (alow < ahgh);
                      alast = alow;
                    }
                }
            }
          if (go)
            { cov = lcp; ahgh = anti + lcp; mix = wch; alow = anti; dgmin = dgmax = dg; }
        }
    }
  return ST_OK;
}

/***********************************************************************************************
 *  Warp-parallel chain scan of one triple (the extension stage's version of the loop above).
 *
 *  The serial scan keeps ahgh = running maximum of anti+2*lcp over the current chain and breaks
 *  the chain when anti >= ahgh + CHAIN_BREAK.  Because seeds arrive in anti order and one seed
 *  spans at most 80 anti-diagonals, every seed of an earlier chain ends more than CHAIN_BREAK-80
 *  below the current one, so the chain-local running maximum equals the running maximum over
 *  ALL earlier seeds of the triple.  Breaks, the coverage increments, and the per-chain
 *  reductions (cov, mix, dgmin, dgmax, alow, ahgh) therefore come from warp prefix-max /
 *  prefix-sum / ballots over 32 merged seeds at a time; only completed chains that qualify
 *  (cov >= CHAIN_MIN) enter the sequential tube stepping, in order, exactly as FastGA.c:3157-3340.
 **********************************************************************************************/

struct TripleCtx
{ unsigned j, pairkey; int comp, seq; bool isnew, selfpair, spec;
  long long cdiag, alen, blen, mlen, doffset, aoffset, alast;
};

template<int W>
static __device__ int handle_hit(const ext_params &P, Ctx &c, TripleCtx &T, long long alow,
                                 long long ahgh, int dgmin, int dgmax, u64 &nla)
{ long long amid, eant;
  dgmin += (int) (T.cdiag << BUCK_SHIFT);
  dgmax += (int) (T.cdiag << BUCK_SHIFT);
  if (T.comp)
    { dgmin += (int) T.doffset; dgmax += (int) T.doffset; alow += T.aoffset; ahgh += T.aoffset; }
  else
    { dgmin -= (int) P.bmxpos; dgmax -= (int) P.bmxpos; }
  if (ahgh > T.alast)
    { if (alow < T.alast) alow = T.alast;
      ahgh -= BUCK_ANTI;
      do
        { amid = alow + BUCK_ANTI;
          if (amid > ahgh)
            { amid = ahgh;
              if (amid + dgmin < 0)
                { dgmin = (int) -amid;
                  if (dgmin > dgmax) break;
                }
            }
          LAres R;
          int st = ST_OK;
          if (T.selfpair)
            { //  a contig against itself, forward strand: strictly above or strictly below the main
              //  diagonal, nothing across it (FastGA.c:3247-3262; there the tube then advances with
              //  the stale bepos of the previous alignment of the thread -- here with 0)
              if (dgmin > 0)      st = local_alignment<W>(c,T.comp,dgmin,dgmax,(int) amid,R,dgmin-1,-1);
              else if (dgmax < 0) st = local_alignment<W>(c,T.comp,dgmin,dgmax,(int) amid,R,-1,-(dgmax+1));
              else { R.abpos = R.aepos = R.bbpos = R.bepos = 0; R.diffs = 0; R.ftlen = R.rtlen = 0; }
            }
          else
            st = local_alignment<W>(c,T.comp,dgmin,dgmax,(int) amid,R);
          if (st) return st;
          nla += 1;
          int rlen = R.aepos - R.abpos;                    // same after the ACOMP flip
          if (rlen >= P.aln_min && P.aln_rate*rlen >= (double) R.diffs)
            { emit_record(P,c,R,T.comp,T.j,T.seq,T.pairkey);
              T.seq += 1;
              if (T.spec && (T.seq & ((1 << SPEC_SEQ_BITS) - 1)) == 0) return ST_SPEC;   // numbering exhausted
            }
          eant = (long long) R.aepos + R.bepos;            // un-flipped end (FastGA.c:3309-3312)
          if (eant <= alow) alow = amid; else alow = eant;
        }
      while (alow < ahgh);
      T.alast = alow;
    }
  return ST_OK;
}

#define SCAN_SMEM 1536          // per warp: La Ua (32 x i64) Lm Um (32 x int) Ma (64 x i64) Mm (64 x int)

//  Bands of a triple: L = [b,m) (band c), U = [m,e) (band c+1, if present).  False: nothing to scan.
static __device__ bool triple_setup(const ext_params &P, unsigned j, TripleCtx &T, unsigned &b, unsigned &m, unsigned &e)
{ const rec128 *S = P.seeds;
  b = P.seg_start[j]; m = P.seg_start[j+1]; e = m;
  rec128 r0 = S[b];
  u64 grp = get_bits(r0,P.p_jc,P.jc_bits + P.ic_bits + 1);
  T.cdiag = (long long) get_bits(r0,P.p_band,P.band_bits);
  T.isnew = true;
  bool aux = false;
  if (j > 0)
    { rec128 rp = S[P.seg_start[j-1]];
      if (get_bits(rp,P.p_jc,P.jc_bits + P.ic_bits + 1) == grp &&
          (long long) get_bits(rp,P.p_band,P.band_bits) == T.cdiag-1)
        T.isnew = false;
    }
  if (j+1 < (unsigned) P.nseg)
    { rec128 rn = S[m];
      if (get_bits(rn,P.p_jc,P.jc_bits + P.ic_bits + 1) == grp &&
          (long long) get_bits(rn,P.p_band,P.band_bits) == T.cdiag+1)
        { aux = true; e = P.seg_start[j+2]; }
    }
  if (!T.isnew && !aux) return false;
  T.j = j; T.seq = 0; T.alast = -1; T.spec = false;
  T.comp = (int) get_bits(r0,P.p_cp,1);
  T.pairkey = (unsigned) grp;
  return true;
}

static __device__ void triple_contigs(const ext_params &P, Ctx &c, TripleCtx &T)
{ rec128 r0 = P.seeds[P.seg_start[T.j]];
  int ctg1 = P.aperm[get_bits(r0,P.p_ic,P.ic_bits)];
  int ctg2 = P.bperm[get_bits(r0,P.p_jc,P.jc_bits)];
  T.selfpair = (P.self_mode != 0 && ctg1 == ctg2 && T.comp == 0);
  T.alen = P.aclen[ctg1]; T.blen = P.bclen[ctg2]; T.mlen = T.alen + T.blen;
  T.doffset = T.alen - (P.amxpos + P.bmxpos); T.aoffset = T.alen - P.amxpos;
  c.A = (const unsigned *) ((T.comp ? P.arseq : P.aseq) + P.awoff[ctg1]);
  c.B = (const unsigned *) (P.bseq + P.bwoff[ctg2]);
  c.alen = (int) T.alen; c.blen = (int) T.blen;
  c.anw = (T.alen + 31) >> 5; c.bnw = (T.blen + 31) >> 5;
}

//  The open chain at the end of a scanned range, and the running maximum of anti + 2*lcp
struct ChainOpen { long long alow, carryP; int cov, mix, dgmin, dgmax, cnt; bool head; };

//  Chain detection over the merged seeds of L[s,m) and U[t,e), 32 at a time, starting from the
//  running maximum carryP of everything before the range.  sink.closed(alow,ahgh,cov,mix,dmin,dmax,
//  cnt,head) is called for every chain a break closes (head: the chain contains the range's start;
//  cnt: its seeds inside the range); O returns the chain left open.
template<class Sink>
static __device__ int scan_core(const ext_params &P, unsigned s, unsigned m, unsigned t, unsigned e,
                                long long carryP, unsigned char *wsm, Sink &sink, ChainOpen &O)
{ const int lane = threadIdx.x & 31;
  const rec128 *S = P.seeds;
  long long *La = (long long *) wsm, *Ua = La + 32, *Ma = Ua + 32;
  int *Lm = (int *) (Ma + 64), *Um = Lm + 32, *Mm = Um + 32;
  const long long NEG = -0x7fffffffffffffffll;
  const long long CB = P.chain_break;
  long long c_alow = 0;
  int c_cov = 0, c_mix = 0, c_dgmin = 2*BUCK_WIDTH, c_dgmax = 0, c_cnt = 0;
  bool head = true;

  while (s < m || t < e)
    { int nl = (int) min(32u,m - s), nu = (int) min(32u,e - t);
      __syncwarp();
      if (lane < nl)
        { rec128 r = ld_rec(S + s + lane);
          La[lane] = (long long) get_bits(r,P.p_anti,P.anti_bits);
          Lm[lane] = (int) ((r.lo & 63) << 1) | (int) (((r.lo >> 6) & 63) << 8) | (1 << 16);
        }
      if (lane < nu)
        { rec128 r = ld_rec(S + t + lane);
          Ua[lane] = (long long) get_bits(r,P.p_anti,P.anti_bits);
          Um[lane] = (int) ((r.lo & 63) << 1) | (int) ((((r.lo >> 6) & 63) + BUCK_WIDTH) << 8) | (2 << 16);
        }
      __syncwarp();
      //  merged rank of every window element (ties: lower band first, FastGA.c:3111)
      int rankL = 0x7fffffff, rankU = 0x7fffffff;
      if (lane < nl)
        { long long a = La[lane]; int lo = 0, hi = nu;             // # U with anti < a
          while (lo < hi) { int md = (lo+hi) >> 1; if (Ua[md] < a) lo = md+1; else hi = md; }
          rankL = lane + lo;
        }
      if (lane < nu)
        { long long a = Ua[lane]; int lo = 0, hi = nl;             // # L with anti <= a
          while (lo < hi) { int md = (lo+hi) >> 1; if (La[md] <= a) lo = md+1; else hi = md; }
          rankU = lane + lo;
        }
      //  only ranks up to the end of the first exhausted window are final
      int valid = nl + nu;
      if (nl > 0 && s + nl < m) valid = min(valid,__shfl_sync(FULL,rankL,nl-1) + 1);
      if (nu > 0 && t + nu < e) valid = min(valid,__shfl_sync(FULL,rankU,nu-1) + 1);
      if (rankL < valid) { Ma[rankL] = La[lane]; Mm[rankL] = Lm[lane]; }
      if (rankU < valid) { Ma[rankU] = Ua[lane]; Mm[rankU] = Um[lane]; }
      s += __popc(__ballot_sync(FULL,rankL < valid));
      t += __popc(__ballot_sync(FULL,rankU < valid));
      __syncwarp();

      for (int base = 0; base < valid; base += 32)
        { int n = min(32,valid - base);
          bool act = lane < n;
          long long anti = act ? Ma[base+lane] : 0;
          int meta = act ? Mm[base+lane] : 0;
          int lcp2 = meta & 0xff, dg = (meta >> 8) & 0xff, wch = meta >> 16;
          long long cps = act ? anti + lcp2 : NEG;
          long long pm = cps;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1)
            { long long v = __shfl_up_sync(FULL,pm,o);
              if (lane >= o && v > pm) pm = v;
            }
          long long pe = __shfl_up_sync(FULL,pm,1);
          if (lane == 0) pe = NEG;
          long long Pl = pe > carryP ? pe : carryP;             // ahgh seen by this seed
          bool brk = act && anti >= Pl + CB;
          int inc = 0;
          if (act)
            { if (brk) inc = lcp2;
              else if (cps > Pl) inc = (anti >= Pl) ? lcp2 : (int) (cps - Pl);
            }
          int Ssum = inc;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1)
            { int v = __shfl_up_sync(FULL,Ssum,o);
              if (lane >= o) Ssum += v;
            }
          const unsigned bm = __ballot_sync(FULL,brk);
          const unsigned w1 = __ballot_sync(FULL,act && wch == 1), w2 = __ballot_sync(FULL,act && wch == 2);
          //  Segments between breaks: the first continues the carried chain, the last stays open, the
          //  ones in between are whole chains.  Nearly all of those are stray seeds below chain_min:
          //  every break lane sizes its own segment, only the ones that reach chain_min are visited.
          const unsigned above = bm & ~((2u << lane) - 1u);
          const int qn = above ? (__ffs(above) - 1) : n;              // end of the segment this lane starts (if brk)
          const int segcov = __shfl_sync(FULL,Ssum,qn > 0 ? qn-1 : 0) - (Ssum - inc);
          unsigned todo = __ballot_sync(FULL,brk && above != 0 && segcov >= P.chain_min);
          const int nbrk = __popc(bm);
          //  visit order: [0,first break) | qualifying middle segments | [last break,n)
          int stage = 0;
          while (true)
            { int seglo, q; bool cont, last;
              if (stage == 0)
                { seglo = 0; q = bm ? (__ffs(bm) - 1) : n; cont = true; last = (bm == 0); stage = 1; }
              else if (todo)
                { seglo = __ffs(todo) - 1; todo &= todo - 1;
                  q = __shfl_sync(FULL,qn,seglo); cont = false; last = false;
                }
              else
                { seglo = 31 - __clz(bm); q = n; cont = false; last = true; }
              const unsigned R = ((q >= 32) ? 0xffffffffu : ((1u << q) - 1)) & ~((1u << seglo) - 1);
              int cov = (q > 0 ? __shfl_sync(FULL,Ssum,q-1) : 0) - (seglo > 0 ? __shfl_sync(FULL,Ssum,seglo-1) : 0);
              int mix = ((w1 & R) ? 1 : 0) | ((w2 & R) ? 2 : 0);
              int cnt = __popc(R);
              const bool inR = (R >> lane) & 1;
              int dmin = __reduce_min_sync(FULL,inR ? dg : 255);
              int dmax = __reduce_max_sync(FULL,inR ? dg : -1);
              long long alow = c_alow;
              if (cont)
                { cov += c_cov; mix |= c_mix; cnt += c_cnt;
                  dmin = min(dmin,c_dgmin); dmax = max(dmax,c_dgmax);
                }
              else
                alow = __shfl_sync(FULL,anti,seglo);
              if (last)                                           // open chain -> carry
                { c_cov = cov; c_mix = mix; c_dgmin = dmin; c_dgmax = dmax; c_alow = alow; c_cnt = cnt;
                  break;
                }
              const long long ahgh = __shfl_sync(FULL,Pl,q);
              int st = sink.closed(alow,ahgh,cov,mix,dmin,dmax,cnt,head);
              if (st) return st;
              head = false;
            }
          if (nbrk > 1) head = false;                             // skipped chains closed too
          long long pmx = __shfl_sync(FULL,pm,n-1);
          if (pmx > carryP) carryP = pmx;
        }
    }
  O.alow = c_alow; O.carryP = carryP; O.cov = c_cov; O.mix = c_mix; O.dgmin = c_dgmin; O.dgmax = c_dgmax;
  O.cnt = c_cnt; O.head = head;
  return ST_OK;
}

//  in-kernel scan of a whole triple (triples whose pre-scanned chunks overflowed): chains go straight
//  to the tube stepping
template<int W> struct HitNow
{ const ext_params &P; Ctx &c; TripleCtx &T; u64 &nla; unsigned &nhit;
  __device__ int closed(long long alow, long long ahgh, int cov, int mix, int dmin, int dmax, int, bool)
  { if (cov >= P.chain_min && (mix != 1 || T.isnew))
      { nhit += 1;
        return handle_hit<W>(P,c,T,alow,ahgh,dmin,dmax,nla);
      }
    return ST_OK;
  }
};

template<int W>
static __device__ int scan_triple_warp(const ext_params &P, Ctx &c, unsigned j, unsigned &nhit_out,
                                       u64 &nla, unsigned char *wsm)
{ TripleCtx T;
  unsigned b, m, e;
  nhit_out = 0;
  if (!triple_setup(P,j,T,b,m,e)) return ST_OK;
  triple_contigs(P,c,T);
  HitNow<W> sink = { P, c, T, nla, nhit_out };
  ChainOpen O;
  int st = scan_core(P,b,m,m,e,-(long long) P.chain_break,wsm,sink,O);
  if (st) return st;
  //  the scan's final iteration (anti = MAX) closes the last chain
  return sink.closed(O.alow,O.carryP,O.cov,O.mix,O.dgmin,O.dgmax,O.cnt,false);
}

/***********************************************************************************************
 *  Chain detection ahead of the extension, in parallel over CHUNKS of a triple.  A long triple's
 *  chain scan is a serial walk over up to millions of seeds; inside extend_kernel it sat on the
 *  critical path of the kernel's longest triple.  Chain breaks only depend on the running maximum
 *  of anti + 2*lcp, and a seed spans at most 80 anti-diagonals, so that maximum at any cut point is
 *  found by looking back a few dozen seeds: the merged seed sequence is cut at anti values
 *  (chain_plan_kernel), every chunk is scanned by its own warp (chain_chunk_kernel: chains inside
 *  the chunk become hits, the pieces touching its two ends are returned as partial sums), and one
 *  thread per triple stitches the partial chains of consecutive chunks (chain_stitch_kernel).
 *  extend_kernel then only walks the hit list of its triple (run_hits).
 **********************************************************************************************/

#define CH_SEEDS 1024            // seeds per chunk (both bands), x1.5
#define CH_HCAP  48              // hits recorded per chunk (more: the triple is scanned in extend_kernel)
#ifndef CH_TOPK
#define CH_TOPK  (1 << 30)             // only the largest triples are pre-scanned: theirs is the scan that sits on the kernel's
#endif                           //   critical path; the others are scanned inside extend_kernel, which has idle warps to spare

struct ChainHit { long long alow, ahgh; int dgmin, dgmax; };

struct ChunkPlan { unsigned w, j, k, nch, sL, sU; };            // work-list position, triple, chunk number, chunks of the triple, band starts

struct ChunkOut
{ int nhit, over, first_break, head_closed, tail_valid, empty;
  int h_cov, h_mix, h_dgmin, h_dgmax;
  int t_cov, t_mix, t_dgmin, t_dgmax;
  long long h_ahgh, t_alow, carry_start, carry_end;
  ChainHit hits[CH_HCAP];
};

__global__ void chain_plan_kernel(ext_params P, ChunkPlan *__restrict__ plan, int nplan)
{ int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nplan) return;
  ChunkPlan c = plan[i];
  c.j = P.work[c.w];
  TripleCtx T; unsigned b, m, e;
  if (!triple_setup(P,c.j,T,b,m,e)) { c.sL = P.seg_start[c.j+1]; c.sU = c.sL; plan[i] = c; return; }
  if (c.k == 0) { c.sL = b; c.sU = m; plan[i] = c; return; }
  //  cut k sits after the first k/nch of the MERGED sequence (lower band first on equal anti, the
  //  order scan_core merges in): a merge-path search over the two bands, so a chunk holds the same
  //  number of seeds whichever band they crowd in
  const rec128 *S = P.seeds;
  const unsigned nL = m - b, nU = e - m;
  const unsigned long long tgt = (unsigned long long) c.k * ((nL + nU + c.nch - 1) / c.nch);
  if (tgt >= (unsigned long long) nL + nU) { c.sL = m; c.sU = e; plan[i] = c; return; }   // an empty chunk at the end
  const unsigned t = (unsigned) tgt;
  unsigned lo = t > nU ? t - nU : 0u, hi = t < nL ? t : nL;        // L seeds among the first t
  while (lo < hi)
    { const unsigned md = (lo + hi) >> 1;
      const long long al = (long long) get_bits(S[b + md],P.p_anti,P.anti_bits);
      const long long au = (long long) get_bits(S[m + (t - 1 - md)],P.p_anti,P.anti_bits);
      if (al <= au) lo = md + 1; else hi = md;
    }
  c.sL = b + lo; c.sU = m + (t - lo);
  plan[i] = c;
}

struct ChunkSink
{ const ext_params &P; ChunkOut *out; bool isnew; int lane; int nhit;
  __device__ int closed(long long alow, long long ahgh, int cov, int mix, int dmin, int dmax, int cnt, bool head)
  { if (head)
      { if (lane == 0)
          { out->first_break = (cnt == 0); out->head_closed = 1;
            out->h_cov = cov; out->h_mix = mix; out->h_dgmin = dmin; out->h_dgmax = dmax; out->h_ahgh = ahgh;
          }
        return ST_OK;
      }
    if (cov >= P.chain_min && (mix != 1 || isnew))
      { if (lane == 0 && nhit < CH_HCAP)
          { ChainHit h; h.alow = alow; h.ahgh = ahgh; h.dgmin = dmin; h.dgmax = dmax; out->hits[nhit] = h; }
        nhit += 1;
      }
    return ST_OK;
  }
};

__global__ void __launch_bounds__(128)
chain_chunk_kernel(ext_params P, const ChunkPlan *__restrict__ plan, int nplan, ChunkOut *__restrict__ outs)
{ __shared__ __align__(16) unsigned char sm[4*SCAN_SMEM];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const int i = blockIdx.x * 4 + wp;
  if (i >= nplan) return;
  const ChunkPlan c = plan[i];
  ChunkOut *out = outs + i;
  TripleCtx T; unsigned b, m, e;
  const bool ok = triple_setup(P,c.j,T,b,m,e);
  unsigned sL = c.sL, sU = c.sU, eL = m, eU = e;
  if (ok && c.k + 1 < c.nch) { eL = plan[i+1].sL; eU = plan[i+1].sU; }
  if (lane == 0)
    { out->nhit = 0; out->over = 0; out->first_break = 0; out->head_closed = 0; out->tail_valid = 0;
      out->empty = (!ok || (sL >= eL && sU >= eU));
    }
  __syncwarp();
  if (!ok || (sL >= eL && sU >= eU)) return;
  const rec128 *S = P.seeds;
  //  running maximum of anti + 2*lcp over everything before the chunk: only seeds within 80
  //  anti-diagonals of the last one can hold it
  long long carry = -(long long) P.chain_break;
  if (c.k > 0)
    { long long best = -0x7fffffffffffffffll, top = -0x7fffffffffffffffll;
      for (int band = 0; band < 2; band++)
        { const unsigned lo = band ? m : b, hi = band ? sU : sL;
          if (hi > lo) { long long a = (long long) get_bits(S[hi-1],P.p_anti,P.anti_bits); if (a > top) top = a; }
        }
      for (int band = 0; band < 2; band++)
        { const unsigned lo = band ? m : b; unsigned hi = band ? sU : sL;
          while (hi > lo)
            { long long a = -0x7fffffffffffffffll, v = -0x7fffffffffffffffll;
              if (hi >= lo + 1 + (unsigned) lane)
                { rec128 r = ld_rec(S + hi - 1 - lane);
                  a = (long long) get_bits(r,P.p_anti,P.anti_bits);
                  v = a + (long long) ((r.lo & 63) << 1);
                }
              for (int o = 16; o > 0; o >>= 1)
                { long long w = __shfl_xor_sync(FULL,v,o); if (w > v) v = w; }
              if (v > best) best = v;
              const long long amin = __shfl_sync(FULL,a,31);       // the farthest seed looked at (NEG if fewer than 32)
              if (hi < lo + 32 || amin < top - 80) break;
              hi -= 32;
            }
        }
      if (best > carry) carry = best;
    }
  if (lane == 0) out->carry_start = carry;
  ChunkSink sink = { P, out, T.isnew, lane, 0 };
  ChainOpen O;
  scan_core(P,sL,eL,sU,eU,carry,sm + wp*SCAN_SMEM,sink,O);
  if (lane == 0)
    { out->carry_end = O.carryP;
      out->nhit = sink.nhit; out->over = (sink.nhit > CH_HCAP);
      if (O.head)                                                 // no break inside: the whole chunk continues the open chain
        { out->h_cov = O.cov; out->h_mix = O.mix; out->h_dgmin = O.dgmin; out->h_dgmax = O.dgmax; }
      else
        { out->tail_valid = 1; out->t_alow = O.alow;
          out->t_cov = O.cov; out->t_mix = O.mix; out->t_dgmin = O.dgmin; out->t_dgmax = O.dgmax;
        }
    }
}

//  one thread per work triple: its chunks in order -> the ordered hit list of the triple
__global__ void chain_stitch_kernel(ext_params P, const ChunkPlan *__restrict__ plan, const ChunkOut *__restrict__ outs,
                                    const unsigned *__restrict__ first_chunk, int ntrip, ChainHit *__restrict__ hits,
                                    unsigned long long *__restrict__ hit_used, unsigned long long hit_cap,
                                    uint2 *__restrict__ hit_range /* start, count | 0x80000000: scan in extend_kernel */,
                                    int2 *__restrict__ tinfo /* (strand, contig pair) key and band of the triple */)
{ int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= ntrip) return;
  tinfo[w] = make_int2(-1,0);
  const unsigned c0 = first_chunk[w], c1 = first_chunk[w+1];
  TripleCtx T; unsigned b, m, e;
  if (c1 == c0) { hit_range[w] = make_uint2(0u,0x80000000u); return; }          // not pre-scanned
  if (!triple_setup(P,plan[c0].j,T,b,m,e)) { hit_range[w] = make_uint2(0u,0u); return; }
  tinfo[w] = make_int2((int) T.pairkey,(int) T.cdiag);
  unsigned long long total = 0; bool over = false;
  for (unsigned k = c0; k < c1; k++) { total += (unsigned long long) outs[k].nhit + 1; over |= (outs[k].over != 0); }
  total += 1;
  unsigned long long base = atomicAdd(hit_used,total);
  if (over || base + total > hit_cap) { hit_range[w] = make_uint2(0u,0x80000000u); return; }
  ChainHit *H = hits + base;
  unsigned n = 0;
  bool open = false; long long o_alow = 0; int o_cov = 0, o_mix = 0, o_dmin = 2*BUCK_WIDTH, o_dmax = 0;
  long long last_carry = -(long long) P.chain_break;
#define CH_EMIT(AHGH) do { if (open && o_cov >= P.chain_min && (o_mix != 1 || T.isnew)) \
                             { ChainHit h; h.alow = o_alow; h.ahgh = (AHGH); h.dgmin = o_dmin; h.dgmax = o_dmax; H[n++] = h; } \
                           open = false; } while (0)
  for (unsigned k = c0; k < c1; k++)
    { const ChunkOut &C = outs[k];
      if (C.empty) continue;
      if (C.first_break) CH_EMIT(C.carry_start);
      else
        { //  the chunk's head continues the open chain (an open chain always exists: chunk 0 starts with a break)
          o_cov += C.h_cov; o_mix |= C.h_mix;
          if (C.h_dgmin < o_dmin) o_dmin = C.h_dgmin;
          if (C.h_dgmax > o_dmax) o_dmax = C.h_dgmax;
          if (C.head_closed) CH_EMIT(C.h_ahgh);
        }
      for (int q = 0; q < C.nhit; q++) H[n++] = C.hits[q];
      if (C.tail_valid)
        { open = true; o_alow = C.t_alow; o_cov = C.t_cov; o_mix = C.t_mix; o_dmin = C.t_dgmin; o_dmax = C.t_dgmax; }
      last_carry = C.carry_end;
    }
  CH_EMIT(last_carry);                                             // the scan's final iteration closes the last chain
#undef CH_EMIT
  hit_range[w] = make_uint2((unsigned) base,n);
}

//  extend_kernel's side: the tube stepping of every pre-scanned chain of a triple, in order
template<int W>
static __device__ int run_hits(const ext_params &P, Ctx &c, unsigned j, const ChainHit *__restrict__ H, unsigned n,
                               unsigned &nhit_out, u64 &nla, const unsigned g, const bool spec, long long &alast_out)
{ TripleCtx T;
  unsigned b, m, e;
  nhit_out = 0;
  alast_out = -0x7fffffffffffffffll;
  if (n == 0 || !triple_setup(P,j,T,b,m,e)) return ST_OK;
  triple_contigs(P,c,T);
  //  a hit group starts as if nothing of its triple had been aligned before it (the host checks that
  //  afterwards, fgb_extend); its records are numbered from (g << SPEC_SEQ_BITS)
  T.spec = spec; T.seq = (int) (g << SPEC_SEQ_BITS);
  for (unsigned q = 0; q < n; q++)
    { const ChainHit h = H[q];
      nhit_out += 1;
      int st = handle_hit<W>(P,c,T,h.alow,h.ahgh,h.dgmin,h.dgmax,nla);
      if (st) return st;
    }
  if (T.alast >= 0) alast_out = T.alast - (T.comp ? T.aoffset : 0);       // in the hits' own coordinates
  return ST_OK;
}

static __device__ __forceinline__ bool upper_differs(const rec128 &a, const rec128 &b, int pos)
{ if (pos < 64) return a.hi != b.hi || (a.lo >> pos) != (b.lo >> pos);
  return (a.hi >> (pos-64)) != (b.hi >> (pos-64));
}

//  K7: marks the start of every band segment: seeds i-1 and i differ above the anti field.

__global__ void seg_flag_kernel(const rec128 *__restrict__ seeds, long long n, int p_band,
                                unsigned *__restrict__ flag)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned f = 1;
  if (i > 0)
    { rec128 a = seeds[i-1], b = seeds[i];
      f = upper_differs(a,b,p_band);
    }
  flag[i] = f;
}

//  (heads are recomputed from the seeds, so the scan can run in place on the flag array)
__global__ void seg_fill2_kernel(const rec128 *__restrict__ seeds, long long n, int p_band,
                                 const unsigned *__restrict__ pos, unsigned *__restrict__ seg_start,
                                 unsigned nseg)
{ long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { seg_start[nseg] = (unsigned) n; return; }
  bool head = true;
  if (i > 0)
    { rec128 a = seeds[i-1], b = seeds[i];
      head = upper_differs(a,b,p_band);
    }
  if (head) seg_start[pos[i]] = (unsigned) i;
}

//  K7 prefilter: one thread per band segment.  A chain needs cov >= chain_min and one seed covers
//  at most 80 anti-diagonals, so triples with too few seeds are dropped outright; short triples
//  are scanned exactly by their thread; long ones (their serial scan would be a straggler) go
//  to the warp stage unconditionally -- it scans them with staged, coalesced seed loads.

#define PREF_LONG 64

__global__ void prefilter_kernel(ext_params P, unsigned *__restrict__ work_long, unsigned *__restrict__ work_short,
                                 unsigned *__restrict__ nwork /* [0] long [1] short */,
                                 unsigned *__restrict__ long_size)
{ unsigned j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= (unsigned) P.nseg) return;
  const rec128 *S = P.seeds;
  unsigned b = P.seg_start[j], m = P.seg_start[j+1], e = m;
  unsigned minseeds = (unsigned) ((P.chain_min + 79) / 80);
  rec128 r0 = S[b];
  u64 grp = get_bits(r0,P.p_jc,P.jc_bits + P.ic_bits + 1);
  long long cdiag = (long long) get_bits(r0,P.p_band,P.band_bits);
  if (j+1 < (unsigned) P.nseg)
    { rec128 rn = S[m];
      if (get_bits(rn,P.p_jc,P.jc_bits + P.ic_bits + 1) == grp &&
          (long long) get_bits(rn,P.p_band,P.band_bits) == cdiag+1)
        e = P.seg_start[j+2];
    }
  if (e - b < minseeds) return;
  if (e - b > PREF_LONG)
    { bool isnew = true;
      if (j > 0)
        { rec128 rp = S[P.seg_start[j-1]];
          if (get_bits(rp,P.p_jc,P.jc_bits + P.ic_bits + 1) == grp &&
              (long long) get_bits(rp,P.p_band,P.band_bits) == cdiag-1)
            isnew = false;
        }
      if (isnew || e != m)
        { unsigned o = atomicAdd(nwork,1u);
          work_long[o] = j; long_size[o] = e - b;
        }
      return;
    }
  Ctx c; u64 nla = 0; unsigned nh = 0;
  scan_triple<false>(P,c,j,nh,nla,NULL);
  if (nh > 0)
    work_short[atomicAdd(nwork+1,1u)] = j;
}

#define WSTATE_BYTES(W) ((W)*(4*4+8) + 32)
#define STATE_BYTES (WSTATE_BYTES(EX_W) + SCAN_SMEM)
#define BIG_SMEM_PER_WARP (SCAN_SMEM)
#define TT_BYTES    (32768*2)
#define EX_NFRONT   (EX_PAIR ? EX_WARPS/EX_TEAM : EX_WARPS)  // warps of a block that take triples
#define BOX_BYTES   (EX_PAIR ? (EX_WARPS/EX_TEAM)*((int) sizeof(PairBox)) : 0)

template<int W>
__global__ void __launch_bounds__(EX_WARPS*32,EX_MINBLK)
extend_kernel(ext_params P)
{ unsigned char *const smem = ex_smem;
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const long long gw = (long long) blockIdx.x * EX_WARPS + wp;
  const size_t per_warp = (W == EX_W) ? STATE_BYTES : BIG_SMEM_PER_WARP;
  unsigned char *sb = (W == EX_W) ? (smem + (size_t) wp * STATE_BYTES)
                                  : (P.bigstate + (size_t) gw * WSTATE_BYTES(EX_WBIG));
  Ctx c;
  c.T  = (u64 *) sb;
  c.V  = (int *) (sb + W*8);
  c.HA = c.V + W; c.HM = c.HA + W; c.NA = c.HM + W;
  c.carry = c.NA + W;
  rec128 *stagebuf = (W == EX_W) ? (rec128 *) (sb + WSTATE_BYTES(EX_W))
                                 : (rec128 *) (smem + (size_t) wp * BIG_SMEM_PER_WARP);
  c.ttab = P.table; c.sc15 = TRIM_LEN * P.dscore;
  //  read-out window: the state slot of the team's T warp (T and P keep their state in registers; the
  //  front warp's own scan buffer is live while a triple scanned here calls into an alignment)
  c.pwin = EX_PAIR ? (Peb *) (smem + (size_t) (wp + 1) * per_warp) : (Peb *) stagebuf;
  c.pwin_n = (EX_PAIR && W == EX_W) ? 256 : 64;
  c.box = NULL; c.box_off = 0;
  if (EX_PAIR)
    { c.box_off = (unsigned) ((size_t) EX_WARPS * per_warp + (size_t) (wp / EX_TEAM) * sizeof(PairBox));
      c.box = (PairBox *) (smem + c.box_off);
      if ((wp % EX_TEAM) == 0 && lane == 0) { c.box->seq = 0; c.box->cmd = 0; c.box->stop = 0; c.box->stopp = 0; }
    }
  __syncthreads();
  if (EX_PAIR && (wp % EX_TEAM))
    { //  T warp (1) / P warp (2) of team wp/3: serve the passes their front warp starts
      PairBox *bx = c.box;
      const int role = wp % EX_TEAM;
      int myseq = 0;
      while (true)
        { int sq;
          while ((sq = ld_acquire_smem(&bx->seq)) == myseq) __nanosleep(100);
          myseq = sq;
          int cm = bx->cmd;
          if (cm == 9) break;
          if (role == 1) { if (cm == 1) wave_T<1>(c.box_off,c.ttab,c.sc15); else wave_T<-1>(c.box_off,c.ttab,c.sc15); }
          else           { if (cm == 1) wave_P<1>(c.box_off); else wave_P<-1>(c.box_off); }
          __syncwarp();
        }
      return;
    }
  long long t_start = clock64();
  c.cells = P.cells + gw * P.cells_per_warp;
  c.cmax  = (int) P.cells_per_warp;
  c.avail = 0;
  c.fstage = P.stage + gw * 2ll * P.stage_bytes;
  c.rstage = c.fstage + P.stage_bytes;
  c.smax = P.stage_bytes;
  c.tspace = P.tspace; c.path_ave = P.path_ave; c.score = P.score; c.table = P.table;
  c.nwaves = 0; c.ncells = 0; c.cyc_wave = 0; c.cyc_extract = 0; c.pwaves = 0; c.npairs = 0; c.fwait = 0; c.ftot = 0; c.bwait = 0; c.btot = 0;
  u64 nla = 0, nhits = 0;

  while (true)
    { unsigned w = 0;
      if (lane == 0) w = atomicAdd(P.queue,1u);
      w = __shfl_sync(FULL,w,0);
      if (w >= (unsigned) P.nwork) break;
      unsigned j, w0, nh = 0;
      uint2 hr = make_uint2(0u,0x80000000u);
      unsigned grp = 0; bool spec = false;
      if (P.items != NULL)
        { const ExItem it = P.items[w];
          w0 = it.w; j = P.work[w0]; hr = make_uint2(it.h0,it.hn); grp = it.g; spec = true;
        }
      else
        { j = P.work[w];
          w0 = P.widx ? P.widx[w] : w;
          if (P.hit_range != NULL) hr = P.hit_range[w0];
        }
      const u64 lg_w = c.nwaves, lg_l = nla; const long long lg_t = clock64();
      int st; long long alast_out = -0x7fffffffffffffffll;
      if (hr.y & 0x80000000u) st = scan_triple_warp<W>(P,c,j,nh,nla,(unsigned char *) stagebuf);
      else                    st = run_hits<W>(P,c,j,P.hits + hr.x,hr.y,nh,nla,grp,spec,alast_out);
      if (P.items != NULL && lane == 0) P.galast[w] = alast_out;
      if (st != ST_OK)
        { if (lane == 0)
            { unsigned o = atomicAdd(P.nfailed,1u);
              P.failed[o] = j; P.failed_w[o] = w0;
              atomicOr(P.need,1u << st);
            }
        }
      else if (!spec || (hr.y & 0x80000000u))
        nhits += nh;                                                // (hit groups are counted by the host)
      if (P.wlog != NULL && lane == 0)
        { unsigned long long *L = P.wlog + 4ull*w;
          L[0] = ((u64) gw << 32) | j; L[1] = ((c.nwaves - lg_w) << 24) | ((nla - lg_l) << 8) | (u64) (st & 0xff);
          L[2] = (u64) (lg_t - t_start); L[3] = (u64) (clock64() - t_start);
        }
      __syncwarp();
    }
  if (EX_PAIR && lane == 0)
    { c.box->cmd = 9;                              // release the back warp
      st_release_smem(&c.box->seq,c.box->seq + 1);
    }
  if (lane == 0)
    { atomicAdd(&P.counters[0],nhits);
      atomicAdd(&P.counters[1],nla);
      atomicAdd(&P.counters[2],c.nwaves);
      atomicAdd(&P.counters[3],c.ncells);
      atomicAdd(&P.counters[8],(u64) (clock64() - t_start));
      atomicAdd(&P.counters[9],c.cyc_wave);
      atomicAdd(&P.counters[10],c.cyc_extract);
      atomicAdd(&P.counters[11],c.pwaves);
      if (EX_DIAG)                                                    // slowest warp: cycles, of which in waves / read-outs (all >> 12)
        atomicMax(&P.counters[12],(((u64) (clock64() - t_start) >> 12) << 40) | ((c.cyc_wave >> 12) << 20) | (c.cyc_extract >> 12));
      else atomicAdd(&P.counters[12],c.npairs);
      atomicAdd(&P.counters[4],c.fwait); atomicAdd(&P.counters[7],c.ftot);
      atomicAdd(&P.counters[13],c.bwait);
      if (EX_DIAG) atomicAdd(&P.counters[14],c.btot);                 // P warp wait cycles (diagnostic builds)
      else atomicMax(&P.counters[14],(u64) (clock64() - t_start));
      { u64 cy = (u64) (clock64() - t_start) >> 12, wv = c.nwaves > 0xffffff ? 0xffffff : c.nwaves;
        u64 la = nla > 0xffff ? 0xffff : nla;
        atomicMax(&P.counters[15],(cy << 40) | (wv << 16) | la);      // the slowest warp: cycles/4096, waves, LA calls
      }
    }
}

/***********************************************************************************************
 *  The align.h seam: Local_Alignment (align.c:1423, align.h:262-298) as a batched export.  One
 *  warp per call tuple (contig pair, strand, low, hgh, anti, lbord, hbord) on the single-warp wave
 *  code; the Path comes back as Local_Alignment leaves it (ACOMP flip applied), the trace as bytes.
 **********************************************************************************************/

struct la_job { int actg, bctg, comp, low, hgh, anti, lbord, hbord; };

__global__ void __launch_bounds__(EX_WARPS*32,EX_MINBLK)
la_batch_kernel(ext_params P, const la_job *__restrict__ jobs, int njobs, int *__restrict__ status)
{ unsigned char *const smem = ex_smem;
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const long long gw = (long long) blockIdx.x * EX_WARPS + wp;
  unsigned char *sb = smem + (size_t) wp * STATE_BYTES;
  Ctx c;
  c.T  = (u64 *) sb;
  c.V  = (int *) (sb + EX_W*8);
  c.HA = c.V + EX_W; c.HM = c.HA + EX_W; c.NA = c.HM + EX_W;
  c.carry = c.NA + EX_W;
  c.pwin = (Peb *) (sb + WSTATE_BYTES(EX_W)); c.pwin_n = 64;
  c.ttab = P.table; c.sc15 = TRIM_LEN * P.dscore;
  c.box = NULL; c.box_off = 0;
  c.cells = P.cells + gw * P.cells_per_warp;
  c.cmax  = (int) P.cells_per_warp;
  c.avail = 0;
  c.fstage = P.stage + gw * 2ll * P.stage_bytes;
  c.rstage = c.fstage + P.stage_bytes;
  c.smax = P.stage_bytes;
  c.tspace = P.tspace; c.path_ave = P.path_ave; c.score = P.score; c.table = P.table;
  c.nwaves = 0; c.ncells = 0; c.cyc_wave = 0; c.cyc_extract = 0; c.pwaves = 0; c.npairs = 0; c.fwait = 0; c.ftot = 0; c.bwait = 0; c.btot = 0;
  while (true)
    { unsigned w = 0;
      if (lane == 0) w = atomicAdd(P.queue,1u);
      w = __shfl_sync(FULL,w,0);
      if (w >= (unsigned) njobs) break;
      const la_job J = jobs[w];
      c.A = (const unsigned *) ((J.comp ? P.arseq : P.aseq) + P.awoff[J.actg]);
      c.B = (const unsigned *) (P.bseq + P.bwoff[J.bctg]);
      c.alen = (int) P.aclen[J.actg]; c.blen = (int) P.bclen[J.bctg];
      c.anw = (c.alen + 31) >> 5; c.bnw = (c.blen + 31) >> 5;
      LAres R;
      int st = local_alignment<EX_W>(c,J.comp,J.low,J.hgh,J.anti,R,J.lbord,J.hbord);
      if (st == ST_OK) emit_record(P,c,R,J.comp,w,0,0u);
      if (lane == 0) status[w] = st;
      __syncwarp();
    }
}

/***********************************************************************************************
 *  Host side of the stage
 **********************************************************************************************/

struct fgb_overlaps
{ long long nrec = 0, nbytes = 0;
  unsigned char *h_buf = nullptr;          // packed records (OUT_HDR + trace padded to 8)
  unsigned long long counters[16] = {0};
  long long nseg = 0, nwork = 0;
  bool pinned = false;
};

extern "C" void fgb_overlaps_free(fgb_overlaps *o)
{ if (!o) return;
  if (o->h_buf) { if (o->pinned) cudaFreeHost(o->h_buf); else free(o->h_buf); }
  delete o;
}
//  Wraps packed records produced elsewhere (tests feed the host filter without a GPU).
extern "C" int fgb_overlaps_from_buffer(const unsigned char *buf, long long nbytes, fgb_overlaps **out)
{ fgb_overlaps *o = new fgb_overlaps();
  o->h_buf = (unsigned char *) malloc(nbytes + 64);
  memcpy(o->h_buf,buf,nbytes);
  o->nbytes = nbytes;
  *out = o;
  return FGB_OK;
}
extern "C" long long fgb_overlaps_bytes(const fgb_overlaps *o) { return o->nbytes; }
extern "C" const unsigned char *fgb_overlaps_data(const fgb_overlaps *o) { return o->h_buf; }
extern "C" void fgb_overlaps_counters(const fgb_overlaps *o, unsigned long long *out)
{ for (int i = 0; i < 16; i++) out[i] = o->counters[i];          /* out: 16 entries */
  out[5] = (unsigned long long) o->nseg; out[6] = (unsigned long long) o->nwork;
}


#include <chrono>
static long long tr_t0 = 0;
static void tr_mark(const char *what)
{ static int on = -1;
  if (on < 0) on = (getenv("FGB_TRACE") != NULL);
  if (!on) return;
  long long t = std::chrono::duration_cast<std::chrono::microseconds>(
                  std::chrono::steady_clock::now().time_since_epoch()).count();
  fprintf(stderr,"[fgb_trace] %-28s +%8.3f ms\n",what,tr_t0 ? (t - tr_t0)/1000.0 : 0.0);
  tr_t0 = t;
}

static bool tr_on() { static int on = -1; if (on < 0) on = (getenv("FGB_TRACE") != NULL); return on != 0; }
#define TR_SYNC(what) do { if (tr_on()) { cudaStreamSynchronize(st); tr_mark(what); } } while (0)

//  tables: 2 x 32768 int16 (score, then table) and ave_path from New_Align_Spec's arithmetic,
//  computed by the host caller (align.c:222-268 is float/double set-up, kept on the host).

//  Hit groups of the work triples (host): see the comment in fgb_extend.  hrange[w] = (first hit, count |
//  bit 31: no list) into hh[0..hused); tinfo[w] = ((strand, contig pair) key, band); items come out in launch
//  order (largest estimated cost first) with, for each, the first hit of the next group of its triple.
static void build_hit_groups(unsigned nwork, const uint2 *hrange, const int2 *tinfo, const ChainHit *hh,
                             unsigned long long hused, int SPEC_BANDS, long long SPEC_SLACK, long long SPEC_GAP,
                             std::vector<ExItem> &items, std::vector<long long> &nxt_alow,
                             std::vector<long long> &nxt_ahgh, std::vector<unsigned> &hcount)
{ hcount.assign(nwork,0u);
  for (unsigned w = 0; w < nwork; w++)
    if (!(hrange[w].y & 0x80000000u)) hcount[w] = hrange[w].y;

  //  components of chains (index = position in hh; only listed triples' ranges are used)
  std::vector<unsigned> comp((size_t) hused + 1);
  for (size_t q = 0; q <= hused; q++) comp[q] = (unsigned) q;
  auto find = [&](unsigned x) { while (comp[x] != x) { comp[x] = comp[comp[x]]; x = comp[x]; } return x; };
  auto unite = [&](unsigned x, unsigned y) { x = find(x); y = find(y); if (x != y) comp[x < y ? y : x] = (x < y ? x : y); };
  if (SPEC_GAP < 0)
    { std::vector<std::pair<std::pair<int,int>,unsigned> > byband;       // ((key, band), w)
      for (unsigned w = 0; w < nwork; w++)
        if (hcount[w] > 0) byband.push_back(std::make_pair(std::make_pair(tinfo[w].x,tinfo[w].y),w));
      std::sort(byband.begin(),byband.end());
      for (size_t i = 0; i < byband.size(); i++)
        { const unsigned w1 = byband[i].second;
          const ChainHit *H1 = hh + hrange[w1].x; const unsigned n1 = hcount[w1];
          for (unsigned q = 1; q < n1; q++)                                   // neighbours in its own list
            if (H1[q].alow - H1[q-1].ahgh < SPEC_SLACK) unite(hrange[w1].x + q - 1,hrange[w1].x + q);
          for (size_t k = i + 1; k < byband.size(); k++)
            { if (byband[k].first.first != byband[i].first.first ||
                  byband[k].first.second - byband[i].first.second > SPEC_BANDS) break;
              const unsigned w2 = byband[k].second;
              const ChainHit *H2 = hh + hrange[w2].x; const unsigned n2 = hcount[w2];
              unsigned a = 0, b = 0;                                          // interval join of two sorted lists
              while (a < n1 && b < n2)
                { if (H1[a].ahgh + SPEC_SLACK < H2[b].alow) a += 1;
                  else if (H2[b].ahgh + SPEC_SLACK < H1[a].alow) b += 1;
                  else
                    { unite(hrange[w1].x + a,hrange[w2].x + b);
                      if (H1[a].ahgh < H2[b].ahgh) a += 1; else b += 1;
                    }
                }
            }
        }
    }
  //  extent of every component: how long the alignment of its block will be (launch order)
  std::vector<long long> clo((size_t) hused + 1,0x7fffffffffffffffll), chi((size_t) hused + 1,-0x7fffffffffffffffll);
  for (unsigned w = 0; w < nwork; w++)
    for (unsigned q = 0; q < hcount[w]; q++)
      { const unsigned x = hrange[w].x + q, r = find(x);
        if (hh[x].alow < clo[r]) clo[r] = hh[x].alow;
        if (hh[x].ahgh > chi[r]) chi[r] = hh[x].ahgh;
      }

  struct Grp { ExItem it; long long span, na, nh; };
  std::vector<Grp> G;
  const long long INF = 0x7fffffffffffffffll;
  std::vector<unsigned> lastof;                                    // scratch: last list position of a component
  for (unsigned w = 0; w < nwork; w++)
    { const uint2 hr = hrange[w];
      if (hr.y & 0x80000000u)
        { Grp g; g.it.w = w; g.it.h0 = 0; g.it.hn = 0x80000000u; g.it.g = 0; g.span = INF; g.na = g.nh = INF;
          G.push_back(g); continue;
        }
      if (hr.y == 0) continue;
      const ChainHit *H = hh + hr.x;
      const bool one = (hr.y >= (1u << (31 - SPEC_SEQ_BITS)));        // too many hits to number by group
      //  reach[q] = last position holding a hit of the component of hit q
      lastof.assign(hr.y,0u);
      { std::vector<std::pair<unsigned,unsigned> > cq(hr.y);
        for (unsigned q = 0; q < hr.y; q++) cq[q] = std::make_pair(find(hr.x + q),q);
        std::sort(cq.begin(),cq.end());
        for (unsigned q = hr.y; q-- > 0; )
          lastof[cq[q].second] = (q + 1 < hr.y && cq[q+1].first == cq[q].first) ? lastof[cq[q+1].second] : cq[q].second;
      }
      unsigned a = 0;
      while (a < hr.y)
        { unsigned b = a + 1, reach = lastof[a];
          long long span = 0; unsigned lastc = 0xffffffffu;
          while (b < hr.y && (one || b <= reach || (SPEC_GAP >= 0 && H[b].alow - H[b-1].ahgh < SPEC_GAP)))
            { if (lastof[b] > reach) reach = lastof[b];
              b += 1;
            }
          for (unsigned q = a; q < b; q++)
            { const unsigned r = find(hr.x + q);
              if (r != lastc) { span += chi[r] - clo[r]; lastc = r; }
            }
          Grp g; g.it.w = w; g.it.h0 = hr.x + a; g.it.hn = b - a; g.it.g = a; g.span = span;
          g.na = (b < hr.y) ? H[b].alow : INF; g.nh = (b < hr.y) ? H[b].ahgh : INF;
          G.push_back(g);
          a = b;
        }
    }
  std::stable_sort(G.begin(),G.end(),[](const Grp &x, const Grp &y) { return x.span > y.span; });
  items.resize(G.size()); nxt_alow.resize(G.size()); nxt_ahgh.resize(G.size());
  for (size_t q = 0; q < G.size(); q++) { items[q] = G[q].it; nxt_alow[q] = G[q].na; nxt_ahgh[q] = G[q].nh; }
}

//  The grouping rule on its own (no device needed): hrange / tinfo as 2 x nwork ints, hits as (alow, ahgh) pairs;
//  items_out: 4 words per item (work triple, first hit, hits | bit 31, number of the first hit in its triple),
//  next_out: (alow, ahgh) of the next group's first hit or INT64_MAX.  Returns the number of items
//  (at most one per hit plus one per triple without a list).
extern "C" long long fgb_hit_groups_host(int nwork, const unsigned *hrange, const int *tinfo, const long long *hits,
                                         long long nhits, int bands, long long slack, long long gap,
                                         unsigned *items_out, long long *next_out)
{ std::vector<uint2> hr((size_t) nwork); std::vector<int2> ti((size_t) nwork);
  for (int w = 0; w < nwork; w++) { hr[w] = make_uint2(hrange[2*w],hrange[2*w+1]); ti[w] = make_int2(tinfo[2*w],tinfo[2*w+1]); }
  std::vector<ChainHit> hh((size_t) nhits + 1);
  for (long long q = 0; q < nhits; q++) { hh[q].alow = hits[2*q]; hh[q].ahgh = hits[2*q+1]; hh[q].dgmin = hh[q].dgmax = 0; }
  std::vector<ExItem> items; std::vector<long long> na, nh; std::vector<unsigned> hc;
  build_hit_groups((unsigned) nwork,hr.data(),ti.data(),hh.data(),(unsigned long long) nhits,bands,slack,gap,items,na,nh,hc);
  for (size_t q = 0; q < items.size(); q++)
    { items_out[4*q] = items[q].w; items_out[4*q+1] = items[q].h0; items_out[4*q+2] = items[q].hn; items_out[4*q+3] = items[q].g;
      next_out[2*q] = na[q]; next_out[2*q+1] = nh[q];
    }
  return (long long) items.size();
}

extern "C" int fgb_extend(const fgb_seeds *S, const fgb_genome *A, const fgb_genome *B,
                          int chain_break, int chain_min, int align_min, double align_rate,
                          const short *tables, int ave_path, int tspace,
                          fgb_overlaps **out, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (A->d_rseq == NULL) return FGB_ERR_ARG;
  if (S->n >= 0xfffffff0ll) return FGB_ERR_LIMIT;
  owner<fgb_overlaps> Oown(new fgb_overlaps(),fgb_overlaps_free);
  fgb_overlaps *O = Oown.get();
  long long n = S->n;
  tr_mark("extend: enter");

  ext_params P;
  memset(&P,0,sizeof(P));
  P.seeds = S->d_rec; P.nseeds = n;
  P.p_anti = 12; P.anti_bits = S->anti_bits;
  P.p_band = P.p_anti + S->anti_bits; P.band_bits = S->band_bits;
  P.p_jc = P.p_band + S->band_bits; P.jc_bits = S->jc_bits;
  P.p_ic = P.p_jc + S->jc_bits; P.ic_bits = S->ic_bits;
  P.p_cp = P.p_ic + S->ic_bits;
  P.amxpos = S->amxpos; P.bmxpos = S->bmxpos;
  P.aseq = A->d_seq; P.arseq = A->d_rseq; P.awoff = A->d_woff; P.aclen = A->d_clen; P.aperm = A->d_perm;
  P.bseq = B->d_seq; P.bwoff = B->d_woff; P.bclen = B->d_clen; P.bperm = B->d_perm;
  P.chain_break = chain_break; P.chain_min = chain_min;
  P.aln_min = align_min - 50; P.aln_rate = align_rate + .05;      // FastGA.c:3013-3014
  P.tspace = tspace; P.path_ave = ave_path;
  P.self_mode = S->self_mode;
  P.dscore = -tables[0] / TRIM_LEN;                     // SCORE[0] = -15 * dscore

  short *d_tables = NULL;
  u64 *d_counters = NULL, *d_total = NULL;
  unsigned *d_flag = NULL, *d_seg = NULL, *d_work = NULL, *d_misc = NULL, *d_failed = NULL;
  void *d_tmp = NULL;
  ChunkPlan *d_plan = NULL; ChunkOut *d_couts = NULL; unsigned *d_first = NULL, *d_failed_w = NULL;
  ChainHit *d_hits = NULL; uint2 *d_hrange = NULL;
  //  hit groups (first launch): items in launch order, and for each the first hit of the NEXT group of
  //  its triple (what its tube must not have reached for the groups to have been independent)
  ExItem *d_items = NULL; long long *d_galast = NULL; int2 *d_tinfo = NULL;
  unsigned char *d_out = NULL;
  dev_scope G(st);
  G.own(d_tables); G.own(d_counters); G.own(d_total); G.own(d_flag); G.own(d_seg); G.own(d_work);
  G.own(d_misc); G.own(d_failed); G.own(d_tmp);
  G.own(d_plan); G.own(d_couts); G.own(d_first); G.own(d_failed_w); G.own(d_hits); G.own(d_hrange);
  G.own(d_items); G.own(d_galast); G.own(d_tinfo);
  G.own(d_out);
  CUDA_TRY(fgb_dmalloc((void **) &d_tables,65536*sizeof(short),st));
  CUDA_TRY(cudaMemcpyAsync(d_tables,tables,65536*sizeof(short),cudaMemcpyHostToDevice,st));
  P.score = d_tables; P.table = d_tables + 32768;
  CUDA_TRY(fgb_dmalloc((void **) &d_counters,16*8,st));
  CUDA_TRY(cudaMemsetAsync(d_counters,0,16*8,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_total,8,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_misc,64,st));
  CUDA_TRY(cudaMemsetAsync(d_misc,0,64,st));
  P.counters = d_counters;

  unsigned nseg = 0, nwork = 0;
  std::vector<unsigned> wsize; bool sizes_known = false;
  unsigned long long hit_cap = 0;
  std::vector<ExItem> items; std::vector<long long> nxt_alow, nxt_ahgh;
  std::vector<unsigned> hwork, hcount;                 // work triples; hits of each pre-scanned one
  unsigned long long hits_done = 0;                    // hits of the pre-scanned triples the first launch completed
  if (n > 0)
    { stage_timer t(&g_timings.triples_ms,st);
      long long tmpb = fgb_dev_scan_tmp_bytes(n);
      CUDA_TRY(fgb_dmalloc((void **) &d_flag,sizeof(unsigned)*(n+1),st));
      CUDA_TRY(fgb_dmalloc((void **) &d_tmp,tmpb,st));
      int nb = (int) ((n + 255) / 256);
      seg_flag_kernel<<<nb,256,0,st>>>(S->d_rec,n,P.p_band,d_flag);
      int rc = fgb_dev_exclusive_scan_u32(d_flag,n,d_total,d_tmp,tmpb,st);
      if (rc) return rc;
      u64 tot = 0;
      CUDA_TRY(cudaMemcpyAsync(&tot,d_total,8,cudaMemcpyDeviceToHost,st));
      CUDA_TRY(cudaStreamSynchronize(st));
      nseg = (unsigned) tot;
      TR_SYNC("  seg flags + scan");
      CUDA_TRY(fgb_dmalloc((void **) &d_seg,sizeof(unsigned)*(nseg+2),st));
      CUDA_TRY(fgb_dmalloc((void **) &d_work,sizeof(unsigned)*(3ll*nseg+3),st));
      nb = (int) ((n + 1 + 255) / 256);
      seg_fill2_kernel<<<nb,256,0,st>>>(S->d_rec,n,P.p_band,d_flag,d_seg,nseg);
      P.seg_start = d_seg; P.nseg = (int) nseg;
      prefilter_kernel<<<(nseg + 127)/128,128,0,st>>>(P,d_work,d_work + nseg + 1,d_misc + 6,d_work + 2ll*nseg + 2);
      fgb_count_launch(3);
      CUDA_TRY(cudaGetLastError());
      unsigned nw2[2];
      CUDA_TRY(cudaMemcpyAsync(nw2,d_misc + 6,8,cudaMemcpyDeviceToHost,st));
      CUDA_TRY(cudaStreamSynchronize(st));
      TR_SYNC("  seg fill + prefilter");
      //  long triples first, largest first (the kernel's makespan is its longest triple, so it
      //  must not start late), then the exact short hits
      if (nw2[0] >= 1 && nw2[0] <= (1u << 20))
        { std::vector<unsigned> lj(nw2[0]), ls(nw2[0]), ord(nw2[0]);
          CUDA_TRY(cudaMemcpyAsync(lj.data(),d_work,4ull*nw2[0],cudaMemcpyDeviceToHost,st));
          CUDA_TRY(cudaMemcpyAsync(ls.data(),d_work + 2ll*nseg + 2,4ull*nw2[0],cudaMemcpyDeviceToHost,st));
          CUDA_TRY(cudaStreamSynchronize(st));
          for (unsigned q = 0; q < nw2[0]; q++) ord[q] = q;
          std::sort(ord.begin(),ord.end(),[&](unsigned a, unsigned b)
                    { return ls[a] != ls[b] ? ls[a] > ls[b] : lj[a] < lj[b]; });
          std::vector<unsigned> sj(nw2[0]);
          wsize.resize(nw2[0]);
          for (unsigned q = 0; q < nw2[0]; q++) { sj[q] = lj[ord[q]]; wsize[q] = ls[ord[q]]; }
          CUDA_TRY(cudaMemcpyAsync(d_work,sj.data(),4ull*nw2[0],cudaMemcpyHostToDevice,st));
          CUDA_TRY(cudaStreamSynchronize(st));
          sizes_known = true;
        }
      else if (nw2[0] == 0) sizes_known = true;
      CUDA_TRY(cudaMemcpyAsync(d_work + nw2[0],d_work + nseg + 1,sizeof(unsigned)*nw2[1],
                               cudaMemcpyDeviceToDevice,st));
      nwork = nw2[0] + nw2[1];
      TR_SYNC("  work list ordered");

      //  chain detection of every work triple, chunk-parallel (chain_plan / chain_chunk / chain_stitch)
      if (sizes_known && nwork > 0)
        { std::vector<ChunkPlan> plan;
          std::vector<unsigned> first(nwork + 1);
          for (unsigned w = 0; w < nwork; w++)
            { unsigned size = w < wsize.size() ? wsize[w] : 0;
              unsigned nch = (unsigned) (((unsigned long long) size + CH_SEEDS + CH_SEEDS/2 - 1) / (CH_SEEDS + CH_SEEDS/2));
              if (nch < 1) nch = 1;
              if (w >= CH_TOPK || w >= wsize.size()) nch = 0;          // scanned inside extend_kernel
              first[w] = (unsigned) plan.size();
              for (unsigned k = 0; k < nch; k++)
                { ChunkPlan c; c.w = w; c.j = 0; c.k = k; c.nch = nch; c.sL = c.sU = 0; plan.push_back(c); }
            }
          first[nwork] = (unsigned) plan.size();
          const int nplan = (int) plan.size();
          if (nplan > 0) {
          hit_cap = (unsigned long long) nplan * (CH_HCAP + 1) + nwork + 16;
          CUDA_TRY(fgb_dmalloc((void **) &d_plan,sizeof(ChunkPlan)*(size_t) nplan,st));
          CUDA_TRY(fgb_dmalloc((void **) &d_couts,sizeof(ChunkOut)*(size_t) nplan,st));
          CUDA_TRY(fgb_dmalloc((void **) &d_first,sizeof(unsigned)*(size_t) (nwork + 1),st));
          CUDA_TRY(fgb_dmalloc((void **) &d_hits,sizeof(ChainHit)*(size_t) hit_cap,st));
          CUDA_TRY(fgb_dmalloc((void **) &d_hrange,sizeof(uint2)*(size_t) nwork,st));
          CUDA_TRY(fgb_dmalloc((void **) &d_tinfo,sizeof(int2)*(size_t) nwork,st));
          CUDA_TRY(cudaMemcpyAsync(d_plan,plan.data(),sizeof(ChunkPlan)*(size_t) nplan,cudaMemcpyHostToDevice,st));
          CUDA_TRY(cudaMemcpyAsync(d_first,first.data(),sizeof(unsigned)*(size_t) (nwork + 1),cudaMemcpyHostToDevice,st));
          CUDA_TRY(cudaMemsetAsync(d_misc + 8,0,8,st));
          P.work = d_work; P.nwork = (int) nwork;
          TR_SYNC("  chain: plan uploaded");
          chain_plan_kernel<<<(nplan + 127)/128,128,0,st>>>(P,d_plan,nplan);
          TR_SYNC("  chain: plan kernel");
          chain_chunk_kernel<<<(nplan + 3)/4,128,0,st>>>(P,d_plan,nplan,d_couts);
          if (tr_on()) { cudaStreamSynchronize(st); fprintf(stderr,"[fgb_trace]   nwork %u nplan %d\n",nwork,nplan); tr_mark("  chain: chunk kernel"); }
          chain_stitch_kernel<<<(nwork + 127)/128,128,0,st>>>(P,d_plan,d_couts,d_first,(int) nwork,d_hits,
                                                             (unsigned long long *) (d_misc + 8),hit_cap,d_hrange,d_tinfo);
          fgb_count_launch(3);
          CUDA_TRY(cudaGetLastError());
          CUDA_TRY(cudaStreamSynchronize(st));                 // plan / first are host vectors
          TR_SYNC("  chain: stitch kernel");
          P.hits = d_hits; P.hit_range = d_hrange;

          //  Hit groups.  Inside a triple a hit is clipped or skipped by the end of the alignments
          //  before it (alast, FastGA.c:3262-3318), which chains its hits serially.  In practice a hit is
          //  only ever touched by an alignment of ITS aligned block: the block's seed chains in this band
          //  pair and in the neighbouring ones, overlapping end to end while the path drifts across
          //  bands.  Chains of one (strand, contig pair) within SPEC_BANDS bands whose anti-diagonal
          //  intervals (+- SPEC_SLACK) overlap are joined into components (union-find); a triple's hit list is cut
          //  wherever the components before and after the cut are disjoint.  Every group is a work
          //  item of its own that starts with a clear tube; after the launch the host checks that no
          //  group's tube reached the next group's first hit -- else the triple is re-run in one piece
          //  (retry ladder below), so a wrong guess costs time, never the result.
          { int SPEC_BANDS = 1; long long SPEC_SLACK = 1000;
            if (getenv("FGB_SPEC_BANDS") != NULL) SPEC_BANDS = atoi(getenv("FGB_SPEC_BANDS"));
            if (getenv("FGB_SPEC_SLACK") != NULL) SPEC_SLACK = atoll(getenv("FGB_SPEC_SLACK"));
            long long SPEC_GAP = -1;                                   // tests: cut at every gap >= this instead
            if (getenv("FGB_SPEC_GAP") != NULL) SPEC_GAP = atoll(getenv("FGB_SPEC_GAP"));
            //  the small result arrays come back through one pinned scratch buffer (grow-only): four copies in
            //  flight and one synchronisation instead of a staged, synchronous copy each
            static unsigned char *hpin = NULL; static size_t hpin_cap = 0;
            auto pinned = [&](size_t bytes) -> unsigned char *
              { if (bytes > hpin_cap)
                  { if (hpin) cudaFreeHost(hpin);
                    hpin = NULL; hpin_cap = 0;
                    if (cudaMallocHost(&hpin,bytes*2 + 4096) != cudaSuccess) return NULL;
                    hpin_cap = bytes*2 + 4096;
                  }
                return hpin;
              };
            unsigned long long hused = 0;
            std::vector<uint2> hrange(nwork);
            std::vector<int2> tinfo(nwork);
            hwork.resize(nwork); hcount.assign(nwork,0u);
            { const size_t o1 = 16, o2 = o1 + sizeof(uint2)*(size_t) nwork, o3 = o2 + sizeof(int2)*(size_t) nwork,
                           o4 = o3 + sizeof(unsigned)*(size_t) nwork;
              unsigned char *hp = pinned(o4);
              if (hp == NULL) return FGB_ERR_CUDA;
              CUDA_TRY(cudaMemcpyAsync(hp,d_misc + 8,8,cudaMemcpyDeviceToHost,st));
              CUDA_TRY(cudaMemcpyAsync(hp + o1,d_hrange,sizeof(uint2)*(size_t) nwork,cudaMemcpyDeviceToHost,st));
              CUDA_TRY(cudaMemcpyAsync(hp + o2,d_tinfo,sizeof(int2)*(size_t) nwork,cudaMemcpyDeviceToHost,st));
              CUDA_TRY(cudaMemcpyAsync(hp + o3,d_work,sizeof(unsigned)*(size_t) nwork,cudaMemcpyDeviceToHost,st));
              CUDA_TRY(cudaStreamSynchronize(st));
              memcpy(&hused,hp,8);
              memcpy(hrange.data(),hp + o1,sizeof(uint2)*(size_t) nwork);
              memcpy(tinfo.data(),hp + o2,sizeof(int2)*(size_t) nwork);
              memcpy(hwork.data(),hp + o3,sizeof(unsigned)*(size_t) nwork);
            }
            if (hused > hit_cap) hused = hit_cap;
            std::vector<ChainHit> hh((size_t) hused + 1);
            if (hused > 0)
              { unsigned char *hp = pinned(sizeof(ChainHit)*(size_t) hused);
                if (hp == NULL) return FGB_ERR_CUDA;
                CUDA_TRY(cudaMemcpyAsync(hp,d_hits,sizeof(ChainHit)*(size_t) hused,cudaMemcpyDeviceToHost,st));
                CUDA_TRY(cudaStreamSynchronize(st));
                memcpy(hh.data(),hp,sizeof(ChainHit)*(size_t) hused);
              }
            build_hit_groups(nwork,hrange.data(),tinfo.data(),hh.data(),hused,SPEC_BANDS,SPEC_SLACK,SPEC_GAP,
                             items,nxt_alow,nxt_ahgh,hcount);
            if (!items.empty())
              { CUDA_TRY(fgb_dmalloc((void **) &d_items,sizeof(ExItem)*items.size(),st));
                CUDA_TRY(fgb_dmalloc((void **) &d_galast,sizeof(long long)*items.size(),st));
                CUDA_TRY(cudaMemcpyAsync(d_items,items.data(),sizeof(ExItem)*items.size(),cudaMemcpyHostToDevice,st));
              }                                                      // (`items` lives until the launches are over)
            TR_SYNC("  chain: hit groups");
          }
          }
        }
    }
  O->nseg = nseg; O->nwork = nwork;
  tr_mark("extend: triples+prefilter");

  u64 out_cap = 0, out_used = 0;
  if (nwork > 0)
    { int dev = 0, nsm = 148;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&nsm,cudaDevAttrMultiProcessorCount,dev);
      size_t smem = (size_t) EX_WARPS * STATE_BYTES + BOX_BYTES;
      size_t smem_big = (size_t) EX_WARPS * BIG_SMEM_PER_WARP + BOX_BYTES;
      CUDA_TRY(cudaFuncSetAttribute(extend_kernel<EX_W>,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem));
      CUDA_TRY(cudaFuncSetAttribute(extend_kernel<EX_WBIG>,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem_big));
      int bps = 0;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps,extend_kernel<EX_W>,EX_WARPS*32,smem));
      if (bps < 1) bps = 1;
      long long nblocks = (long long) nsm * bps;
      bool use_items = (P.hit_range != NULL);              // first launch over hit groups
      long long want = ((long long) (use_items ? items.size() : nwork) + EX_NFRONT - 1) / EX_NFRONT;
      if (want < 1) want = 1;
      if (nblocks > want) nblocks = want;
      long long nwarps = nblocks * EX_WARPS;

      CUDA_TRY(fgb_dmalloc((void **) &d_failed,sizeof(unsigned)*(nwork+1),st));
      CUDA_TRY(fgb_dmalloc((void **) &d_failed_w,sizeof(unsigned)*(nwork+1),st));
      P.work = d_work; P.nwork = (int) nwork;
      P.queue = d_misc + 1; P.nfailed = d_misc + 2; P.failed = d_failed; P.failed_w = d_failed_w; P.widx = NULL; P.need = d_misc + 10;
      P.out_used = (u64 *) (d_misc + 4);

      long long cells_per_warp = 1ll << 17;          // 128 K pebbles = 2 MB per warp
      int stage_bytes = 1 << 15;
      out_cap = (u64) nwork * 512 + (64ull << 20);
      std::vector<std::pair<unsigned,int> > todo;    // (triple, launch number) of every re-run
      unsigned *d_list = d_work; unsigned nlist = use_items ? (unsigned) items.size() : nwork;
      unsigned *d_work2 = NULL;
      dev_scope G2(st); G2.own(d_work2);
      u64 used_before = 0;
      for (int attempt = 0; nlist > 0; attempt++)
        { unsigned misc[12];
          { Peb *d_cells = NULL; unsigned char *d_stage = NULL; unsigned char *d_big = NULL;
            unsigned long long *d_wlog = NULL;
            dev_scope L(st); L.own(d_wlog); L.own(d_cells); L.own(d_stage); L.own(d_big);    // arenas of this launch
            CUDA_TRY(fgb_dmalloc((void **) &d_cells,sizeof(Peb)*cells_per_warp*nwarps,st));
            CUDA_TRY(fgb_dmalloc((void **) &d_stage,2ll*stage_bytes*nwarps,st));
            if (d_out == NULL) CUDA_TRY(fgb_dmalloc((void **) &d_out,out_cap,st));
            P.cells = d_cells; P.cells_per_warp = cells_per_warp;
            P.stage = d_stage; P.stage_bytes = stage_bytes;
            P.out = d_out; P.out_cap = out_cap;
            P.work = d_list; P.nwork = (int) nlist;
            P.items = use_items ? d_items : NULL; P.galast = d_galast; P.attempt = attempt;
            if (attempt > 0)                                     // retries: wide-band kernel, state in HBM
              { CUDA_TRY(fgb_dmalloc((void **) &d_big,(size_t) nwarps * WSTATE_BYTES(EX_WBIG),st));
                P.bigstate = d_big;
              }
            tr_mark("extend: arenas allocated");
            if (attempt == 0 && getenv("FGB_WLOG") != NULL)
              { CUDA_TRY(fgb_dmalloc((void **) &d_wlog,32ull*(nlist+1),st));
                CUDA_TRY(cudaMemsetAsync(d_wlog,0,32ull*(nlist+1),st));
              }
            P.wlog = d_wlog;
            CUDA_TRY(cudaMemsetAsync(d_misc+1,0,8,st));          // queue, nfailed
            CUDA_TRY(cudaMemsetAsync(d_misc+10,0,4,st));         // reasons of this attempt's failures
            { stage_timer t(&g_timings.extend_ms,st);
              if (attempt == 0)
                extend_kernel<EX_W><<<(unsigned) nblocks,EX_WARPS*32,smem,st>>>(P);
              else
                extend_kernel<EX_WBIG><<<(unsigned) nblocks,EX_WARPS*32,smem_big,st>>>(P);
            }
            g_timings.extend_launches += 1;
            fgb_count_launch(1);
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaMemcpyAsync(misc,d_misc,48,cudaMemcpyDeviceToHost,st));
            CUDA_TRY(cudaStreamSynchronize(st));
            tr_mark("extend: kernel done");
            if (d_wlog != NULL)
              { std::vector<unsigned long long> lg(4ull*nlist);
                CUDA_TRY(cudaMemcpy(lg.data(),d_wlog,32ull*nlist,cudaMemcpyDeviceToHost));
                FILE *f = fopen(getenv("FGB_WLOG"),"w");
                if (f != NULL)
                  { for (unsigned q = 0; q < nlist; q++)
                      fprintf(f,"%u %llu %llu %llu %llu %llu %llu %llu %u %u %u\n",q,lg[4*q] >> 32,lg[4*q] & 0xffffffffull,
                              lg[4*q+1] >> 24,(lg[4*q+1] >> 8) & 0xffff,lg[4*q+1] & 0xff,lg[4*q+2],lg[4*q+3],
                              (P.items != NULL ? (items[q].w < wsize.size() ? wsize[items[q].w] : 0u)
                                               : (q < wsize.size() ? wsize[q] : 0u)),
                              P.items != NULL ? (items[q].hn & 0x7fffffffu) : 0u,P.items != NULL ? items[q].g : 0u);
                    fclose(f);
                  }
              }
          }
          out_used = ((u64) misc[5] << 32) | misc[4];
          unsigned nfailed = misc[2];
          if (out_used > out_cap)
            { //  record buffer too small: grow it (keeping earlier attempts' records) and
              //  repeat this attempt
              if (attempt > 12) return FGB_ERR_OVERFLOW;
              unsigned char *d_new = NULL;
              u64 ncap = out_used * 2 + (64ull << 20);
              CUDA_TRY(fgb_dmalloc((void **) &d_new,ncap,st));
              if (used_before) CUDA_TRY(cudaMemcpy(d_new,d_out,used_before,cudaMemcpyDeviceToDevice));
              fgb_dfree(d_out,st); d_out = d_new; out_cap = ncap;
              CUDA_TRY(cudaMemcpy(d_misc+4,&used_before,8,cudaMemcpyHostToDevice));
              out_used = used_before;
              for (size_t q = 0; q < todo.size(); q++)            // the repeat runs under the next launch number
                if (todo[q].second == attempt) todo[q].second = attempt + 1;
              continue;
            }
          used_before = out_used;
          //  failed triples (and their positions in the first list, which index the hit lists)
          std::vector<unsigned> f(nfailed), fw(nfailed);
          if (nfailed > 0)
            { CUDA_TRY(cudaMemcpy(f.data(),d_failed,sizeof(unsigned)*nfailed,cudaMemcpyDeviceToHost));
              CUDA_TRY(cudaMemcpy(fw.data(),d_failed_w,sizeof(unsigned)*nfailed,cudaMemcpyDeviceToHost));
            }
          if (use_items)
            { //  were the hit groups independent?  a group's tube must have stopped short of the next group's first hit
              std::vector<long long> ga(items.size());
              CUDA_TRY(cudaMemcpy(ga.data(),d_galast,sizeof(long long)*items.size(),cudaMemcpyDeviceToHost));
              for (size_t q = 0; q < items.size(); q++)
                if (ga[q] > nxt_alow[q] || ga[q] >= nxt_ahgh[q])
                  { f.push_back(hwork[items[q].w]); fw.push_back(items[q].w); }
              //  several groups of a triple may have failed: one re-run each
              std::vector<std::pair<unsigned,unsigned> > u(f.size());
              for (size_t q = 0; q < f.size(); q++) u[q] = std::make_pair(fw[q],f[q]);
              std::sort(u.begin(),u.end());
              u.erase(std::unique(u.begin(),u.end()),u.end());
              f.resize(u.size()); fw.resize(u.size());
              for (size_t q = 0; q < u.size(); q++) { fw[q] = u[q].first; f[q] = u[q].second; }
              if (tr_on()) fprintf(stderr,"[fgb_trace]   hit groups %zu, triples to re-run %zu (%u arena overflows)\n",items.size(),u.size(),nfailed);
              nfailed = (unsigned) f.size();
              use_items = false;
              //  hit count (the -v line, FastGA.c:4371): the groups do not count their hits, a triple
              //  that completed in this launch contributes its whole list, a re-run counts for itself
              for (size_t q = 0; q < hcount.size(); q++) hits_done += hcount[q];
              for (size_t q = 0; q < fw.size(); q++) hits_done -= hcount[fw[q]];
            }
          if (nfailed == 0) break;
          if (attempt > 12 || cells_per_warp > (1ll << 27)) return FGB_ERR_OVERFLOW;
          //  rerun only the failed triples (whole, hit after hit) with larger arenas on fewer warps; the
          //  records of their earlier launches are dropped by the host below.
          for (size_t q = 0; q < f.size(); q++) todo.push_back(std::make_pair(f[q],attempt + 1));
          if (d_work2 == NULL) CUDA_TRY(fgb_dmalloc((void **) &d_work2,sizeof(unsigned)*2*(nwork+1),st));
          CUDA_TRY(cudaMemcpy(d_work2,f.data(),sizeof(unsigned)*nfailed,cudaMemcpyHostToDevice));
          CUDA_TRY(cudaMemcpy(d_work2 + nwork + 1,fw.data(),sizeof(unsigned)*nfailed,cudaMemcpyHostToDevice));
          P.widx = d_work2 + nwork + 1;
          d_list = d_work2; nlist = nfailed;
          //  grow only what overflowed: a band too wide for the register / shared-memory state (ST_BAND)
          //  just moves to the wide-band kernel below with the same arenas
          if (attempt > 0 || (misc[10] & (1u << ST_CELLS))) cells_per_warp *= 8;
          if (attempt > 0 || (misc[10] & (1u << ST_STAGE))) stage_bytes *= 4;
          long long nb2 = ((long long) nfailed + EX_NFRONT - 1) / EX_NFRONT;
          long long maxb = (24ll << 30) / ((long long) sizeof(Peb) * cells_per_warp * EX_WARPS);
          if (maxb < 1) maxb = 1;
          nblocks = nb2 < maxb ? nb2 : maxb;
          nwarps = nblocks * EX_WARPS;
        }

      //  bring the records back and drop partial output of triples that were re-run
      O->nbytes = (long long) out_used;
      tr_mark("extend: attempts done");
      //  D2H through a grow-only pinned staging buffer (cudaMallocHost per step costs ms)
      static unsigned char *pin = NULL; static u64 pin_cap = 0;
      if (out_used + 64 > pin_cap)
        { if (pin) cudaFreeHost(pin);
          pin_cap = out_used * 2 + (8ull << 20);
          CUDA_TRY(cudaMallocHost(&pin,pin_cap));
        }
      O->h_buf = (unsigned char *) malloc(out_used + 64);
      O->pinned = false;
      { stage_timer t(&g_timings.d2h_ms,st);
        CUDA_TRY(cudaMemcpyAsync(pin,d_out,out_used,cudaMemcpyDeviceToHost,st));
      }
      CUDA_TRY(cudaStreamSynchronize(st));
      memcpy(O->h_buf,pin,out_used);
      tr_mark("extend: d2h");
      if (!todo.empty())
        { //  a re-run triple may have emitted records in earlier launches: keep only those of its
          //  LAST launch (every record carries its launch number)
          std::sort(todo.begin(),todo.end());
          std::vector<std::pair<unsigned,int> > last;
          for (size_t q = 0; q < todo.size(); q++)
            if (q + 1 == todo.size() || todo[q+1].first != todo[q].first) last.push_back(todo[q]);
          std::vector<long long> offs;
          for (long long off = 0; off < O->nbytes; )
            { int *h = (int *) (O->h_buf + off);
              offs.push_back(off);
              off += OUT_HDR + ((h[8] + 7) & ~7);
            }
          std::vector<char> keep(offs.size(),1);
          for (size_t i = 0; i < offs.size(); i++)
            { int *h = (int *) (O->h_buf + offs[i]);
              auto it = std::lower_bound(last.begin(),last.end(),std::make_pair((unsigned) h[0],INT_MIN));
              if (it != last.end() && it->first == (unsigned) h[0] && it->second != h[9]) keep[i] = 0;
            }
          long long w = 0;
          for (size_t i = 0; i < offs.size(); i++)
            { int *h = (int *) (O->h_buf + offs[i]);
              long long sz = OUT_HDR + ((h[8] + 7) & ~7);
              if (keep[i])
                { if (w != offs[i]) memmove(O->h_buf + w,O->h_buf + offs[i],sz);
                  w += sz;
                }
            }
          O->nbytes = w;
        }
    }
  CUDA_TRY(cudaMemcpy(O->counters,d_counters,16*8,cudaMemcpyDeviceToHost));
  O->counters[0] += hits_done;
  { long long cnt = 0;
    for (long long off = 0; off < O->nbytes; )
      { int *h = (int *) (O->h_buf + off);
        off += OUT_HDR + ((h[8] + 7) & ~7);
        cnt += 1;
      }
    O->nrec = cnt;
  }
  tr_mark("extend: leave");
  *out = Oown.release();                                     // (the device blocks go back as G leaves scope)
  return FGB_OK;
}

//  jobs: n x 8 ints (A contig, B contig, comp, low, hgh, anti, lbord, hbord) -- the arguments of
//  Local_Alignment with aseq/bseq = those contigs (A reverse-complemented and ACOMP_FLAG set when comp,
//  as align_contigs calls it, FastGA.c:3184-3260).  paths: n x 7 ints (abpos bbpos aepos bepos diffs tlen
//  status), status 0 or the ST_* code of a call that did not fit the device arenas; toff: n offsets into
//  `traces` (uint8 pairs, what Compress_TraceTo8 leaves).  traces_cap bytes are available; *traces_used
//  returns the bytes needed (call again with a larger buffer if it exceeds the capacity).
extern "C" int fgb_local_alignments(const fgb_genome *A, const fgb_genome *B, long long n, const int *jobs,
                                    const short *tables, int ave_path, int tspace,
                                    int *paths, long long *toff, unsigned char *traces, long long traces_cap,
                                    long long *traces_used, void *stream)
{ cudaStream_t st = (cudaStream_t) stream;
  if (n < 0 || n > 0x7fffffff) return FGB_ERR_ARG;
  *traces_used = 0;
  if (n == 0) return FGB_OK;
  for (long long i = 0; i < n; i++)
    { const int *j = jobs + 8*i;
      if (j[0] < 0 || j[0] >= A->ncontig || j[1] < 0 || j[1] >= B->ncontig) return FGB_ERR_ARG;
      if (j[2] && A->d_rseq == NULL) return FGB_ERR_ARG;
    }
  ext_params P;
  memset(&P,0,sizeof(P));
  P.aseq = A->d_seq; P.arseq = A->d_rseq; P.awoff = A->d_woff; P.aclen = A->d_clen; P.aperm = A->d_perm;
  P.bseq = B->d_seq; P.bwoff = B->d_woff; P.bclen = B->d_clen; P.bperm = B->d_perm;
  P.tspace = tspace; P.path_ave = ave_path;
  P.dscore = -tables[0] / TRIM_LEN;
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm,cudaDevAttrMultiProcessorCount,dev);
  long long nblocks = (n + EX_WARPS - 1) / EX_WARPS;
  if (nblocks > nsm) nblocks = nsm;
  const long long nwarps = nblocks * EX_WARPS;
  const long long cells_per_warp = 1ll << 18;
  const int stage_bytes = 1 << 16;
  const size_t smem = (size_t) EX_WARPS * STATE_BYTES;
  short *d_tables = NULL; la_job *d_jobs = NULL; int *d_status = NULL; unsigned *d_misc = NULL;
  Peb *d_cells = NULL; unsigned char *d_stage = NULL, *d_out = NULL;
  dev_scope S(st); S.own(d_tables); S.own(d_jobs); S.own(d_status); S.own(d_misc); S.own(d_cells); S.own(d_stage);
  S.own(d_out);
  std::vector<unsigned char> h;
  std::vector<int> hs(n);
  u64 out_cap = (u64) n * 256 + (u64) traces_cap + (1ull << 20), out_used = 0;
  CUDA_TRY(cudaFuncSetAttribute(la_batch_kernel,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem));
  CUDA_TRY(fgb_dmalloc((void **) &d_tables,65536*sizeof(short),st));
  CUDA_TRY(fgb_dmalloc((void **) &d_jobs,sizeof(la_job)*(size_t) n,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_status,sizeof(int)*(size_t) n,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_misc,64,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_cells,sizeof(Peb)*cells_per_warp*nwarps,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_stage,2ll*stage_bytes*nwarps,st));
  CUDA_TRY(fgb_dmalloc((void **) &d_out,out_cap,st));
  CUDA_TRY(cudaMemcpyAsync(d_tables,tables,65536*sizeof(short),cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemcpyAsync(d_jobs,jobs,sizeof(la_job)*(size_t) n,cudaMemcpyHostToDevice,st));
  CUDA_TRY(cudaMemsetAsync(d_misc,0,64,st));
  P.score = d_tables; P.table = d_tables + 32768;
  P.cells = d_cells; P.cells_per_warp = cells_per_warp;
  P.stage = d_stage; P.stage_bytes = stage_bytes;
  P.out = d_out; P.out_cap = out_cap; P.out_used = (u64 *) (d_misc + 4);
  P.queue = d_misc + 1;
  la_batch_kernel<<<(unsigned) nblocks,EX_WARPS*32,smem,st>>>(P,d_jobs,(int) n,d_status);
  fgb_count_launch(1);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(&out_used,d_misc + 4,8,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaMemcpyAsync(hs.data(),d_status,sizeof(int)*(size_t) n,cudaMemcpyDeviceToHost,st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (out_used > out_cap) return FGB_ERR_OVERFLOW;
  h.resize((size_t) out_used + 64);
  CUDA_TRY(cudaMemcpy(h.data(),d_out,out_used,cudaMemcpyDeviceToHost));
  { long long used = 0;
    for (long long i = 0; i < n; i++)
      { int *p = paths + 7*i;
        p[0] = p[1] = p[2] = p[3] = p[4] = p[5] = 0; p[6] = hs[i];
        toff[i] = 0;
      }
    for (u64 off = 0; off < out_used; )
      { const int *r = (const int *) (h.data() + off);
        const long long i = r[0];
        int *p = paths + 7*i;
        p[0] = r[3]; p[1] = r[4]; p[2] = r[5]; p[3] = r[6]; p[4] = r[7]; p[5] = r[8];
        toff[i] = used;
        if (used + r[8] <= traces_cap) memcpy(traces + used,h.data() + off + OUT_HDR,(size_t) r[8]);
        used += r[8];
        off += OUT_HDR + ((r[8] + 7) & ~7);
      }
    *traces_used = used;
    if (used > traces_cap) return FGB_ERR_OVERFLOW;
  }
  return FGB_OK;
}

extern "C" long long fgb_overlaps_count(const fgb_overlaps *o) { return o->nrec; }

/***********************************************************************************************
 *  Alignment specification: New_Align_Spec's float/double arithmetic (align.c:222-268) stays
 *  on the host; the two 32768-entry int16 tables (score, then table) and ave_path go to HBM.
 **********************************************************************************************/

static void spec_table(int bit, int prefix, int score, int mx, int mscore, int dscore,
                       short *table, short *sc)
{ if (bit >= TRIM_LEN)
    { table[prefix] = (short) (score - mx);
      sc[prefix]    = (short) score;
    }
  else
    { if (score > mx) mx = score;
      spec_table(bit+1,(prefix << 1),    score - dscore,mx,mscore,dscore,table,sc);
      spec_table(bit+1,(prefix << 1) | 1,score + mscore,mx,mscore,dscore,table,sc);
    }
}

extern "C" int fgb_align_spec(double ave_corr, const float *freq, short *tables, int *ave_path)
{ static const double bias_factor[10] = { .690, .690, .690, .690, .780, .850, .900, .933, .966, 1.000 };
  double match = freq[0] + freq[3];
  if ((match <= 0.) == (match > 0.)) match = .5;
  if (match > .5) match = 1. - match;
  int bias = (int) ((match + .025)*20. - 1.);
  if (match < .2) bias = 3;
  *ave_path  = (int) (60 * (1. - bias_factor[bias] * (1. - ave_corr)));
  int mscore = (int) (1000 * bias_factor[bias] * (1. - ave_corr));
  int dscore = 1000 - mscore;
  spec_table(0,0,0,0,mscore,dscore,tables + 32768,tables);
  return FGB_OK;
}
