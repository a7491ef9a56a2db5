// Shared device/host helpers for the fastga_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <memory>
#include <vector>

#define FGB_OK            0
#define FGB_ERR_CUDA     -1   // a CUDA runtime call failed (message on stderr)
#define FGB_ERR_ARG      -2   // bad argument
#define FGB_ERR_LIMIT    -3   // input exceeds a documented device-layout limit
#define FGB_ERR_OVERFLOW -4   // a device work arena overflowed even after retry

#define CUDA_TRY(call)                                                                   \
  do { cudaError_t _e = (call);                                                          \
       if (_e != cudaSuccess)                                                            \
         { fprintf(stderr,"fastga_b200: CUDA error %s at %s:%d: %s\n",                   \
                   cudaGetErrorName(_e),__FILE__,__LINE__,cudaGetErrorString(_e));       \
           return FGB_ERR_CUDA; } } while (0)

// 128-bit record, little-endian: value = hi:lo.  All sorts are on byte ranges of this value.
struct __align__(16) rec128 { unsigned long long lo, hi; };

static __device__ __forceinline__ rec128 ld_rec(const rec128 *p)
{ uint4 v = *reinterpret_cast<const uint4 *>(p);
  rec128 r;
  r.lo = (unsigned long long) v.x | ((unsigned long long) v.y << 32);
  r.hi = (unsigned long long) v.z | ((unsigned long long) v.w << 32);
  return r;
}

static __device__ __forceinline__ void st_rec(rec128 *p, rec128 r)
{ uint4 v;
  v.x = (unsigned) r.lo; v.y = (unsigned) (r.lo >> 32);
  v.z = (unsigned) r.hi; v.w = (unsigned) (r.hi >> 32);
  *reinterpret_cast<uint4 *>(p) = v;
}

static __device__ __forceinline__ unsigned rec_byte(const rec128 &r, int b)
{ return (b < 8) ? (unsigned) ((r.lo >> (8*b)) & 0xff) : (unsigned) ((r.hi >> (8*(b-8))) & 0xff); }

//  the 8-bit digit at bit offset sh of the 128-bit value (sh is uniform over a kernel: no divergence)
static __device__ __forceinline__ unsigned rec_dig(const rec128 &r, int sh)
{ if (sh >= 64) return (unsigned) ((r.hi >> (sh - 64)) & 0xff);
  if (sh <= 56) return (unsigned) ((r.lo >> sh) & 0xff);
  return (unsigned) (((r.lo >> sh) | (r.hi << (64 - sh))) & 0xff);
}

static __device__ __forceinline__ unsigned lanemask_lt()
{ unsigned m; asm volatile("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

// k-mer table record (GIX entry in HBM):
//   hi           = bases 0..31 of the 40-mer, base 0 in the top two bits
//   lo[63:48]    = bases 32..39
//   lo[47:32]    = contig rank | strand<<15      (GIXmake.c:896-953: InvP rank, sign flag)
//   lo[31:0]     = post (contig-relative; start+12 for reverse-strand entries)
#define KREC_PREFIX24(hi)   ((unsigned) ((hi) >> 40))
#define KREC_SUFFIX56(r)    ((((r).hi & 0xffffffffffull) << 16) | ((r).lo >> 48))      // bases 12..39

int fgb_dev_exclusive_scan_u32(unsigned *d_data, long long n, unsigned long long *d_total,
                               void *d_tmp, long long tmp_bytes, cudaStream_t st);
long long fgb_dev_scan_tmp_bytes(long long n);

void fgb_count_launch(int n);                 // kernels launched (bench.py gpu_launches)

//  stream-ordered device allocation from a retained pool (no cudaMalloc/cudaFree stalls per step)
cudaError_t fgb_dmalloc(void **p, size_t bytes, cudaStream_t st);
void fgb_dfree(void *p, cudaStream_t st);

//  Device blocks of a call go back on EVERY way out of it, error returns included: the pointer
//  variables are registered once (declare the scope after them), whatever they hold when the scope
//  ends is released, in registration order.  A block handed to a handle or to the caller is
//  cleared from its variable first.
struct dev_scope
{ cudaStream_t st; std::vector<void **> slots;
  explicit dev_scope(cudaStream_t s) : st(s) {}
  template<class T> void own(T *&p) { slots.push_back((void **) &p); }
  ~dev_scope() { for (void **s : slots) if (*s != NULL) { fgb_dfree(*s,st); *s = NULL; } }
};

//  A handle released by its free function unless handed out with release().
template<class T> using owner = std::unique_ptr<T,void (*)(T *)>;

//  TMA 1-D bulk copy global -> shared (cp.async.bulk, SASS UBLKCP) completed on an mbarrier.
//  dst/src 16-byte aligned, bytes a multiple of 16.  One elected thread issues; every thread of
//  the CTA may wait on the barrier phase.
static __device__ __forceinline__ unsigned smem_u32(const void *p)
{ return (unsigned) __cvta_generic_to_shared(p); }

static __device__ __forceinline__ void mbar_init(unsigned long long *bar, int count)
{ asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

static __device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, unsigned bytes,
                                                   unsigned long long *bar)
{ asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
               :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

//  several bulk copies completing on ONE barrier phase: announce the byte total once, then issue the copies
static __device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{ asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
               :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}

static __device__ __forceinline__ void tma_copy_1d(void *smem_dst, const void *gmem_src, unsigned bytes,
                                                   unsigned long long *bar)
{ asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

static __device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned phase)
{ unsigned ok;
  do
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(phase) : "memory");
  while (!ok);
}
