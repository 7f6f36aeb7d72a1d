// Shared device helpers for libgpode (sm_100a only).
//  * packed-FP32 math: FFMA2 / FADD2 / FMUL2 (two fp32 lanes per issue slot, Blackwell-only SASS)
//  * MUFU wrappers (ex2 / cos / sin approximations)
//  * parameter-tile pipeline: 1-D TMA bulk copy (cp.async.bulk -> UBLKCP) + mbarrier, double buffered
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "chunk_geom.h"
#include "gpode.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libgpode is written for sm_100a (B200) only"
#endif

namespace gpode {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr int kMaxD = 16;          // largest GP input dimension compiled
constexpr int kMaxSamples = 65535;  // largest L: the launches put the sample index on grid y or z
constexpr int kMaxStages = 4;
constexpr int kSmemLimit = 227 * 1024;

// ---- packed fp32 ------------------------------------------------------------------------------
__device__ __forceinline__ float2 bc(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 lo(float4 v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi(float4 v) { return make_float2(v.z, v.w); }

// ---- MUFU ---------------------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float2 ex2_2(float2 v) { return make_float2(ex2_approx(v.x), ex2_approx(v.y)); }
__device__ __forceinline__ float2 cos_2(float2 v) { return make_float2(__cosf(v.x), __cosf(v.y)); }
__device__ __forceinline__ float2 sin_2(float2 v) { return make_float2(__sinf(v.x), __sinf(v.y)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- mbarrier + bulk async copy (TMA 1-D) -------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
// (the mbarrier / bulk-copy helpers below take either a pointer or a ready 32-bit shared-window address: kernels under register pressure
//  keep ONE opaque base address and add constants -- the compiler otherwise re-derives every address from the generic pointer, each
//  time through S2R SR_CgaCtaId)
__device__ __forceinline__ uint32_t smem_u32(uint32_t a) { return a; }

template <class B>
__device__ __forceinline__ void mbar_init(B bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
template <class B>
__device__ __forceinline__ void mbar_expect_tx(B bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Every mbarrier wait in the library is bounded in TIME, not in polls: a lost arrival (a bug) traps after kWaitTimeoutNs of no
// progress instead of hanging the GPU, while slow progress (compute-sanitizer, cuda-gdb, a shared SM) never reaches the bound.
// -DGPODE_WAIT_TIMEOUT_NS=0 compiles the bound out.
#ifndef GPODE_WAIT_TIMEOUT_NS
#define GPODE_WAIT_TIMEOUT_NS 20000000000ull   /* 20 s */
#endif
template <class B>
__device__ __forceinline__ bool mbar_try(B bar, uint32_t parity) {   // non-blocking phase test
  uint32_t ok;
  // (the last operand is the suspend-time hint in ns: the thread may sleep in hardware until the phase completes instead of re-polling)
  asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, 2000;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// mbarrier.try_wait may suspend the thread for a hardware time slice when the phase is not complete; test_wait never does: use it
// where the caller has other work to do (the MMA issuer polling for drained ring slots)
template <class B>
__device__ __forceinline__ bool mbar_test(B bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  const unsigned long long t0 = global_ns();
  while (!mbar_try(bar, parity)) {
    __nanosleep(128);
#ifdef GPODE_DEBUG_WAIT   // development aid: name the barrier that never completed and carry on (results are garbage) instead of trapping
    if (global_ns() - t0 > 300000000ull) {
      printf("gpode wait timeout: barrier smem+%u parity %u thread %d block (%d,%d)\n", bar, parity, static_cast<int>(threadIdx.x),
             static_cast<int>(blockIdx.x), static_cast<int>(blockIdx.y));
      return;
    }
#else
    if (GPODE_WAIT_TIMEOUT_NS != 0ull && global_ns() - t0 > GPODE_WAIT_TIMEOUT_NS) __trap();
#endif
  }
}
template <class B>
__device__ __forceinline__ void mbar_wait(B bar, uint32_t parity) {
  // fast path: a PTX-level poll loop (3 instructions per wake-up; the address and the parity stay in registers -- the C++ loop this
  // replaces re-derived both on every iteration, ~15 instructions per poll and a third of all instructions the fused reverse sweep
  // issued).  try_wait suspends the thread in hardware until the barrier is touched or the hint expires.
  uint32_t done;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .u32 n;\n"
      "mov.u32 n, 0;\n"
      "GPODE_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, 2000;\n"
      "@p bra GPODE_DONE;\n"
      "add.u32 n, n, 1;\n"
      "setp.lt.u32 p, n, 65536;\n"
      "@p bra GPODE_WAIT;\n"
      "setp.ne.u32 p, n, n;\n"
      "GPODE_DONE:\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  if (!done) mbar_wait_slow(smem_u32(bar), parity);
}
// Wait of a warp that is AHEAD of the others (ring slot / buffer not drained yet): polls at intervals of ~`ns` instead of spinning.
// mbarrier.try_wait's hardware suspend returns on every barrier event of the CTA -- with ~30 busy barriers that is a spin loop (measured
// on the fused reverse sweep: 29 polls per wait, a third of all issued instructions, taken from the schedulers of the warps being waited for).
template <class B>
__device__ __forceinline__ void mbar_wait_sleepy(B bar, uint32_t parity, uint32_t ns) {
  uint32_t done;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .u32 n;\n"
      "mov.u32 n, 0;\n"
      "GPODE_SWAIT:\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "@p bra GPODE_SDONE;\n"
      "nanosleep.u32 %3;\n"
      "add.u32 n, n, 1;\n"
      "setp.lt.u32 p, n, 65536;\n"
      "@p bra GPODE_SWAIT;\n"
      "setp.ne.u32 p, n, n;\n"
      "GPODE_SDONE:\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  if (!done) mbar_wait_slow(smem_u32(bar), parity);
}
// global -> shared bulk copy, completion counted in bytes on `bar`; bytes % 16 == 0, both 16-B aligned
template <class Dst, class B>
__device__ __forceinline__ void bulk_g2s(Dst dst, const void* src, uint32_t bytes, B bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- packed RBF parameter layout (floats) -------------------------------------------------------
// per sample l:  headers [D_out][HDR]   : c_kd = -log2(e) / (2 ell_kd^2), d < DP, zero padded to HDR
//                rows    [D_out][NR][ROW]: NR = SP2 + MP2 rows of (DP+2) float2 = (DP+2)/2 float4
//                   feature rows  j < SP2 : {omega(2j,d), omega(2j+1,d)}_d<DP, {b, b}, {w', w'}
//                   inducing rows j >= SP2: {G(2m,d), G(2m+1,d)}_d<DP, {H, H}, {ln2 nu', ln2 nu'}
// DP = D_in rounded up to even.  Rows stream through shared memory in chunks of <= RC rows that never
// straddle the feature / inducing boundary.
__host__ __device__ constexpr int rbf_hdr_floats(int DP) { return ((DP + 3) / 4) * 4; }
__host__ __device__ constexpr int rbf_row_floats(int DP) { return (DP + 2) * 2; }
constexpr int kChunkBytes = 12 * 1024;
constexpr int kPipeStages = 3;

// Streams the row chunks of one sample through a ring of shared-memory stages with 1-D TMA bulk
// copies (cp.async.bulk -> UBLKCP) completing on mbarriers.  The chunk sequence is cyclic over
// (k = 0..D_out-1) x (feature chunks, inducing chunks) and repeats for every field evaluation.  One
// elected thread issues copies; all threads wait.  release() is a CTA-wide barrier, so every thread of
// the CTA walks the same sequence.
struct ChunkPipe {
  float* buf0;
  uint64_t* bar;       // kPipeStages mbarriers, then 4 ints of producer state (thread 0 only)
  const float* rows;   // rows region of this sample
  int stage;           // consumer ring position
  uint32_t phase;

  __device__ __forceinline__ void issue_next(const ChunkGeom& cg, long total) {
    int* ps = reinterpret_cast<int*>(bar + kPipeStages);  // {issued (long), pk, pc, pstage}
    long issued = *reinterpret_cast<long*>(ps);
    if (issued < total) {
      int pk = ps[2], pc = ps[3], pstage = ps[4];
      const bool in_m = cg.tail ? (pk == cg.K) : (pc >= cg.NCs);
      int n, rowf;
      size_t off;
      if (!in_m) {
        const int r0 = pc * cg.RCs;
        n = min(cg.RCs, cg.SP2 - r0);
        rowf = cg.rowf_s;
        off = static_cast<size_t>(pk) * cg.blk_floats + static_cast<size_t>(r0) * cg.rowf_s;
      } else {
        const int r0 = (cg.tail ? pc : pc - cg.NCs) * cg.RCm;
        n = min(cg.RCm, cg.MP2 - r0);
        rowf = cg.rowf_m;
        off = (cg.tail ? static_cast<size_t>(cg.K) * cg.blk_floats : static_cast<size_t>(pk) * cg.blk_floats + static_cast<size_t>(cg.SP2) * cg.rowf_s) +
              static_cast<size_t>(r0) * cg.rowf_m;
      }
      const uint32_t bytes = static_cast<uint32_t>(n * rowf) * 4u;
      mbar_expect_tx(bar + pstage, bytes);
      bulk_g2s(buf0 + pstage * cg.stage_floats, rows + off, bytes, bar + pstage);
      pstage = (pstage + 1 == kPipeStages) ? 0 : pstage + 1;
      const int limit = cg.tail ? (pk == cg.K ? cg.NCm : cg.NCs) : cg.NCs + cg.NCm;
      if (++pc == limit) {
        pc = 0;
        ++pk;
        if (pk == (cg.tail ? cg.K + 1 : cg.K)) pk = 0;
      }
      *reinterpret_cast<long*>(ps) = issued + 1;
      ps[2] = pk;
      ps[3] = pc;
      ps[4] = pstage;
    }
  }
  __device__ __forceinline__ void init(float* smem_stages, uint64_t* bars, const float* sample_rows, const ChunkGeom& cg, long total) {
    buf0 = smem_stages;
    bar = bars;
    rows = sample_rows;
    stage = 0;
    phase = 0;
    if (threadIdx.x == 0) {
#pragma unroll
      for (int i = 0; i < kPipeStages; ++i) mbar_init(bar + i, 1);
      int* ps = reinterpret_cast<int*>(bar + kPipeStages);
      ps[0] = ps[1] = ps[2] = ps[3] = ps[4] = 0;
      mbar_fence_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
      for (int i = 0; i < kPipeStages; ++i) issue_next(cg, total);
    }
  }
  __device__ __forceinline__ const float* acquire(const ChunkGeom& cg) {
    mbar_wait(bar + stage, phase);
    return buf0 + stage * cg.stage_floats;
  }
  __device__ __forceinline__ void release(const ChunkGeom& cg, long total) {
    __syncthreads();  // every warp is done reading the stage
    if (threadIdx.x == 0) issue_next(cg, total);
    if (++stage == kPipeStages) {
      stage = 0;
      phase ^= 1u;
    }
  }
};

// Butcher tableaux of the fixed-grid methods (strictly lower A, weights b), see oracle/solvers.py
struct Tableau {
  int stages;
  float a[kMaxStages][kMaxStages];
  float b[kMaxStages];
};
__host__ __device__ inline Tableau make_tableau(int method) {
  Tableau t = {};
  if (method == GPODE_EULER) {
    t.stages = 1;
    t.b[0] = 1.f;
  } else if (method == GPODE_MIDPOINT) {
    t.stages = 2;
    t.a[1][0] = 0.5f;
    t.b[1] = 1.f;
  } else {
    t.stages = 4;
    t.a[1][0] = 1.f / 3.f;
    t.a[2][0] = -1.f / 3.f;
    t.a[2][1] = 1.f;
    t.a[3][0] = 1.f;
    t.a[3][1] = -1.f;
    t.a[3][2] = 1.f;
    t.b[0] = 0.125f;
    t.b[1] = 0.375f;
    t.b[2] = 0.375f;
    t.b[3] = 0.125f;
  }
  return t;
}
inline int method_stages(int method) { return method == GPODE_EULER ? 1 : (method == GPODE_MIDPOINT ? 2 : 4); }

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace gpode
