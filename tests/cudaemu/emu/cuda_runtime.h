// tests/cudaemu/emu/cuda_runtime.h — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// A minimal stand-in for the CUDA runtime and the device execution model so that the SAME kernel sources the product
// compiles with nvcc (the vcs_*.cuh kernels, comp.cu, ars.cu and the glue in vcs.cu) can be compiled with g++ and have
// their indexing and integer arithmetic checked against the oracle on a machine without a GPU.  "Device memory" is host
// memory; a launch runs the blocks of the grid one after another, each block as real threads with a barrier behind
// __syncthreads().  Warp shuffles, ballots and mma.sync are emulated lane by lane (b200emu::warp_gather / warp_mma_*);
// inline PTX is not, so kernels that use it take their plain-C branch under B200_CUDA_EMU.  The one kernel left out
// is vcs_l2tc_kernel (tcgen05 / tensor memory).  Nothing in gstreamer_b200/ loads the library built from this;
// libb200dsp.so has no CPU fallback.
#pragma once

#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <functional>
#include <vector>

#define B200_CUDA_EMU 1
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __grid_constant__
#define __align__(n) alignas (n)

struct uint3_emu { unsigned x, y, z; };
struct dim3 {
  unsigned x, y, z;
  dim3 (unsigned a = 1, unsigned b = 1, unsigned c = 1) : x (a), y (b), z (c) {}
};
// CUDA's own alignments (vector_types.h): a load or store of one of these through a pointer that is not a multiple of
// its alignment faults on the device, and the UBSan build (build_emu.build ("ubsan")) reports it here
struct alignas (8) uint2 { unsigned x, y; };
struct alignas (16) uint4 { unsigned x, y, z, w; };
struct alignas (16) int4 { int x, y, z, w; };
struct alignas (8) int2 { int x, y; };
struct alignas (8) float2 { float x, y; };
struct alignas (16) float4 { float x, y, z, w; };
struct alignas (16) double2 { double x, y; };
struct alignas (4) short2 { short x, y; };
struct alignas (8) short4 { short x, y, z, w; };

extern thread_local uint3_emu threadIdx, blockIdx;
extern thread_local dim3 blockDim, gridDim;

namespace b200emu {
extern uint8_t *dyn_smem;         // the launch's dynamic shared memory: a heap block of exactly the requested size
void barrier ();
// runs body once per thread of every block of the grid
void launch (dim3 grid, dim3 block, size_t smem_bytes, const std::function<void ()> & body);
}

inline void __syncthreads () { b200emu::barrier (); }

namespace b200emu {
// mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 for the calling thread's warp (warp = 32 consecutive thread ids of
// the block; every lane must call it).  Fragment layouts as in the PTX ISA: A 16x32 u8 row-major - a0: row g, k 4t..4t+3;
// a1: row g+8, same k; a2: row g, k 16+4t..; a3: row g+8, k 16+4t.. - B 32x8 s8 column-major - b0: k 4t..4t+3, n g;
// b1: k 16+4t.., n g - C/D 16x8 s32 - d0: (g, 2t), d1: (g, 2t+1), d2: (g+8, 2t), d3: (g+8, 2t+1); g = lane >> 2, t = lane & 3.
void warp_mma_u8s8 (int d[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0, unsigned b1, const int c[4]);
void warp_mma_s8u8 (int d[4], unsigned a0, unsigned a1, unsigned a2, unsigned a3, unsigned b0, unsigned b1, const int c[4]);   // A s8, B u8
// every lane of the calling thread's warp contributes `v`; returns the 32 values (all lanes must call it)
void warp_gather (unsigned v, unsigned out[32]);
unsigned lane_id ();
}

inline unsigned __shfl_sync (unsigned, unsigned v, int src) { unsigned a[32]; b200emu::warp_gather (v, a); return a[src & 31]; }
inline int __shfl_sync (unsigned m, int v, int src) { return (int) __shfl_sync (m, (unsigned) v, src); }
inline unsigned __shfl_up_sync (unsigned, unsigned v, unsigned delta)
{
  unsigned a[32]; b200emu::warp_gather (v, a);
  const unsigned l = b200emu::lane_id ();
  return l >= delta ? a[l - delta] : v;
}
inline unsigned __shfl_down_sync (unsigned, unsigned v, unsigned delta)
{
  unsigned a[32]; b200emu::warp_gather (v, a);
  const unsigned l = b200emu::lane_id ();
  return l + delta < 32 ? a[l + delta] : v;
}
inline unsigned __ballot_sync (unsigned, int pred)
{
  unsigned a[32], m = 0; b200emu::warp_gather (pred ? 1u : 0u, a);
  for (int i = 0; i < 32; i++) m |= a[i] << i;
  return m;
}
inline int __popc (unsigned v) { return __builtin_popcount (v); }
inline unsigned __umulhi (unsigned a, unsigned b) { return (unsigned) (((unsigned long long) a * b) >> 32); }
inline unsigned __funnelshift_r (unsigned lo, unsigned hi, unsigned sh)
{
  return (unsigned) ((((unsigned long long) hi << 32) | lo) >> (sh & 31));
}
// IEEE single operations, no contraction (the build passes -ffp-contract=off; x86-64 SSE arithmetic rounds each operation)
inline float __fadd_rn (float a, float b) { volatile float r = a + b; return r; }
inline float __fsub_rn (float a, float b) { volatile float r = a - b; return r; }
inline float __fmul_rn (float a, float b) { volatile float r = a * b; return r; }
inline float __fdiv_rn (float a, float b) { volatile float r = a / b; return r; }
inline float __int2float_rn (int a) { return (float) a; }
inline double __dadd_rn (double a, double b) { volatile double r = a + b; return r; }
inline double __dsub_rn (double a, double b) { volatile double r = a - b; return r; }
inline double __dmul_rn (double a, double b) { volatile double r = a * b; return r; }
inline double __ddiv_rn (double a, double b) { volatile double r = a / b; return r; }
inline uint4 make_uint4 (unsigned x, unsigned y, unsigned z, unsigned w) { return uint4 {x, y, z, w}; }
inline uint2 make_uint2 (unsigned x, unsigned y) { return uint2 {x, y}; }
inline float4 make_float4 (float x, float y, float z, float w) { return float4 {x, y, z, w}; }
inline int4 make_int4 (int x, int y, int z, int w) { return int4 {x, y, z, w}; }

using std::max;
using std::min;

template <typename T> inline T __ldg (const T *p) { return *p; }
inline unsigned __byte_perm (unsigned a, unsigned b, unsigned s)
{
  const unsigned long long v = ((unsigned long long) b << 32) | a;
  unsigned r = 0;
  for (int i = 0; i < 4; i++) {
    const unsigned sel = (s >> (4 * i)) & 0xf;
    unsigned byte = (unsigned) (v >> (8 * (sel & 7))) & 0xff;
    if (sel & 8) byte = (byte & 0x80) ? 0xff : 0x00;              // msb replication mode
    r |= byte << (8 * i);
  }
  return r;
}
inline unsigned __vavgu4 (unsigned a, unsigned b)
{
  unsigned r = 0;
  for (int i = 0; i < 4; i++) r |= ((((a >> (8 * i)) & 0xff) + ((b >> (8 * i)) & 0xff) + 1) >> 1) << (8 * i);
  return r;
}

// ---- runtime API subset -----------------------------------------------------------------------------------------------
typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorNoDevice = 100, cudaErrorInsufficientDriver = 35 };
typedef void *cudaStream_t;
typedef void *cudaEvent_t;
enum cudaMemcpyKind { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3 };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2, cudaHostAllocPortable = 1, cudaHostRegisterPortable = 1 };
enum { cudaFuncAttributeMaxDynamicSharedMemorySize = 8, cudaDevAttrMultiProcessorCount = 16, cudaDevAttrMaxSharedMemoryPerBlockOptin = 97 };

inline cudaError_t cudaMalloc (void **p, size_t n) { *p = malloc (n ? n : 1); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
inline cudaError_t cudaFree (void *p) { free (p); return cudaSuccess; }
inline cudaError_t cudaMemcpy (void *d, const void *s, size_t n, cudaMemcpyKind) { memcpy (d, s, n); return cudaSuccess; }
inline cudaError_t cudaMemset (void *d, int v, size_t n) { memset (d, v, n); return cudaSuccess; }
inline cudaError_t cudaMemsetAsync (void *d, int v, size_t n, cudaStream_t) { memset (d, v, n); return cudaSuccess; }
inline cudaError_t cudaDeviceSynchronize () { return cudaSuccess; }
inline cudaError_t cudaMemcpyAsync (void *d, const void *s, size_t n, cudaMemcpyKind, cudaStream_t) { memcpy (d, s, n); return cudaSuccess; }
inline cudaError_t cudaGetLastError () { return cudaSuccess; }
inline const char *cudaGetErrorName (cudaError_t) { return "emu"; }
inline const char *cudaGetErrorString (cudaError_t) { return "emu"; }
inline cudaError_t cudaGetDevice (int *d) { *d = 0; return cudaSuccess; }
inline cudaError_t cudaSetDevice (int) { return cudaSuccess; }
inline cudaError_t cudaGetDeviceCount (int *n) { *n = 1; return cudaSuccess; }
inline cudaError_t cudaDeviceGetAttribute (int *v, int a, int) { *v = a == cudaDevAttrMaxSharedMemoryPerBlockOptin ? 232448 : 148; return cudaSuccess; }
inline cudaError_t cudaStreamCreateWithFlags (cudaStream_t *s, unsigned) { *s = nullptr; return cudaSuccess; }
inline cudaError_t cudaStreamDestroy (cudaStream_t) { return cudaSuccess; }
inline cudaError_t cudaStreamSynchronize (cudaStream_t) { return cudaSuccess; }
inline cudaError_t cudaStreamWaitEvent (cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
inline cudaError_t cudaEventCreateWithFlags (cudaEvent_t *e, unsigned) { *e = nullptr; return cudaSuccess; }
inline cudaError_t cudaEventDestroy (cudaEvent_t) { return cudaSuccess; }
inline cudaError_t cudaEventRecord (cudaEvent_t, cudaStream_t) { return cudaSuccess; }
inline cudaError_t cudaEventSynchronize (cudaEvent_t) { return cudaSuccess; }
inline cudaError_t cudaHostAlloc (void **p, size_t n, unsigned) { *p = malloc (n); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
inline cudaError_t cudaFreeHost (void *p) { free (p); return cudaSuccess; }
inline cudaError_t cudaHostRegister (void *, size_t, unsigned) { return cudaSuccess; }
inline cudaError_t cudaHostUnregister (void *) { return cudaSuccess; }
inline cudaError_t cudaDeviceGetPCIBusId (char *b, int n, int) { if (n > 0) b[0] = 0; return cudaErrorNoDevice; }
template <typename F> inline cudaError_t cudaFuncSetAttribute (F, int, int) { return cudaSuccess; }
struct cudaFuncAttributes { size_t sharedSizeBytes = 0; };
template <typename F> inline cudaError_t cudaFuncGetAttributes (cudaFuncAttributes *a, F) { a->sharedSizeBytes = 0; return cudaSuccess; }
