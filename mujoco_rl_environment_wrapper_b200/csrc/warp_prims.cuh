// warp_prims.cuh — the handful of warp-level primitives the step kernel is written against.
// Under nvcc they are the CUDA intrinsics.  Under MJB_HOST_EMU (tests/emu, g++) the same kernel
// source runs on a fibre-based SIMT emulator (32 lanes = 32 ucontext fibres, round-robin at every
// sync / shuffle) so the device code can be debugged in a container without a GPU.  The emulator
// is test tooling; the product only ever runs the nvcc build.
#pragma once
#if !defined(__CUDACC_RTC__)
#include <math.h>
#include <stdint.h>
#include <string.h>
#endif

#if defined(MJB_HOST_EMU)
#include "../../tests/emu/simt_emu.h"
#define MJB_DEV inline
#define MJB_DEV_NOINLINE inline
#define MJB_NOUNROLL
#define MJB_LANE() (simt::lane())
#define MJB_SYNC() simt::barrier()
#define MJB_SHFL(v, src) simt::shfl((v), (src))
#define MJB_SHFL_XOR(v, m) simt::shfl_xor((v), (m))
#define MJB_BALLOT(p) simt::ballot(p)
#define MJB_POPC(x) __builtin_popcount(x)
#define MJB_FFS(x) __builtin_ffs(x)
#define MJB_RSQRT(x) (1.0f / sqrtf(x))
inline uint32_t mjb_f2u(float x) { uint32_t u; memcpy(&u, &x, 4); return u; }
#define MJB_F2U(x) mjb_f2u(x)
#define MJB_G2S(dst, src) (*(dst) = *(src))
#define MJB_G2S_WAIT() ((void)0)
#define MJB_CTA_SYNC(nthreads) ((void)0)
#else
#define MJB_DEV __device__ __forceinline__
#define MJB_DEV_NOINLINE __device__ __noinline__
#define MJB_NOUNROLL _Pragma("unroll 1")
#define MJB_LANE() ((int)(threadIdx.x & 31))
#define MJB_SYNC() __syncwarp()
#define MJB_SHFL(v, src) __shfl_sync(0xffffffffu, (v), (src))
#define MJB_SHFL_XOR(v, m) __shfl_xor_sync(0xffffffffu, (v), (m))
#define MJB_BALLOT(p) __ballot_sync(0xffffffffu, (p))
#define MJB_POPC(x) __popc(x)
#define MJB_FFS(x) __ffs(x)
#define MJB_RSQRT(x) rsqrtf(x)
#define MJB_F2U(x) __float_as_uint(x)
// asynchronous 4-byte global -> shared copy (LDGSTS): the loads of a whole state row are in flight together and
// the warp waits once (MJB_G2S_WAIT) instead of once per array
__device__ __forceinline__ void mjb_g2s4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
#define MJB_G2S(dst, src) mjb_g2s4((dst), (src))
#define MJB_G2S_WAIT() asm volatile("cp.async.wait_all;" ::: "memory")
// CTA-level alignment of the env-warps that are busy in this round (named barrier 1 with an explicit
// thread count, so idle warps of a partial round do not take part).  nthreads == 0 disables it.
__device__ __forceinline__ void mjb_cta_sync(int nthreads) {
  if (nthreads > 32) asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}
#define MJB_CTA_SYNC(nthreads) mjb_cta_sync(nthreads)
#endif

// block-placement hints: rarely taken paths move out of the straight-line instruction stream
#define MJB_UNLIKELY(x) __builtin_expect(!!(x), 0)
#define MJB_LIKELY(x) __builtin_expect(!!(x), 1)

namespace mjb {

MJB_DEV float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += MJB_SHFL_XOR(v, o);
  return v;
}
MJB_DEV float wmin(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, MJB_SHFL_XOR(v, o));
  return v;
}
MJB_DEV float wmax(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, MJB_SHFL_XOR(v, o));
  return v;
}

}  // namespace mjb
