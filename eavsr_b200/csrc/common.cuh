// Shared device/host helpers for the eavsr_b200 alignment kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/eavsr_b200.h"

namespace eavsr {

// ---- host-side error plumbing (C ABI returns int, message via eavsr_last_error) ----
void set_error(const char* fmt, ...);
int  check_launch(const char* what);

#define EAVSR_REQUIRE(cond, ...)                      \
  do {                                                \
    if (!(cond)) {                                    \
      ::eavsr::set_error(__VA_ARGS__);                \
      return EAVSR_ERR_INVALID;                       \
    }                                                 \
  } while (0)

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// element strides of an (n, c, h, w) tensor
struct Strides4 { long long n, c, h, w; };
// DCNv2 geometry (HO/WO derived)
struct DcnGeom {
  int N, Cin, H, W, Cout, KH, KW, SH, SW, PH, PW, DH, DW, G, DG, HO, WO;
};
size_t strided_extent_elems(const int64_t s[4], int n, int c, int h, int w);
// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda); returns false when unavailable / rejected.
// dims / box / element strides have `rank` entries, strides_bytes rank - 1 (dimension 0 is contiguous).
bool encode_tensor_map(void* tensor_map /* CUtensorMap* */, int dtype /* EAVSR_F32 | EAVSR_BF16 */, int rank, const void* base,
                       const unsigned long long* dims, const unsigned long long* strides_bytes, const unsigned* box,
                       int swizzle /* CUtensorMapSwizzle */);

// ---- element access helpers -------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16lo_to_f32(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16hi_to_f32(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// Load NV consecutive channels (16 bytes for bf16 NV=8 / fp32 NV=4) and widen to fp32.
template <typename T, int NV> struct VecLoad;
template <> struct VecLoad<__nv_bfloat16, 8> {
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float* f) {
    uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
    f[0] = bf16lo_to_f32(u.x); f[1] = bf16hi_to_f32(u.x);
    f[2] = bf16lo_to_f32(u.y); f[3] = bf16hi_to_f32(u.y);
    f[4] = bf16lo_to_f32(u.z); f[5] = bf16hi_to_f32(u.z);
    f[6] = bf16lo_to_f32(u.w); f[7] = bf16hi_to_f32(u.w);
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float* f) {
    uint4 u;
    u.x = pack_bf16x2(f[0], f[1]); u.y = pack_bf16x2(f[2], f[3]);
    u.z = pack_bf16x2(f[4], f[5]); u.w = pack_bf16x2(f[6], f[7]);
    *reinterpret_cast<uint4*>(p) = u;
  }
};
template <> struct VecLoad<__nv_bfloat16, 4> {
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float* f) {
    uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    f[0] = bf16lo_to_f32(u.x); f[1] = bf16hi_to_f32(u.x);
    f[2] = bf16lo_to_f32(u.y); f[3] = bf16hi_to_f32(u.y);
  }
};
template <> struct VecLoad<float, 4> {
  static __device__ __forceinline__ void ld(const float* p, float* f) {
    float4 u = __ldg(reinterpret_cast<const float4*>(p));
    f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
  }
  static __device__ __forceinline__ void st(float* p, const float* f) {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  }
};
template <> struct VecLoad<float, 8> {
  static __device__ __forceinline__ void ld(const float* p, float* f) {
    VecLoad<float, 4>::ld(p, f);
    VecLoad<float, 4>::ld(p + 4, f + 4);
  }
};

// Packed register image of CPI consecutive channels (kept packed while loads are in flight).
template <typename XT, int CPI> struct RawVec {
  static constexpr int NW = CPI * (int)sizeof(XT) / 4;
  static __device__ __forceinline__ void ld(const XT* p, uint32_t* w) {
    if constexpr (NW == 2) {
      uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
      w[0] = u.x; w[1] = u.y;
    } else if constexpr (NW == 4) {
      uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
      w[0] = u.x; w[1] = u.y; w[2] = u.z; w[3] = u.w;
    } else {
      uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
      uint4 v = __ldg(reinterpret_cast<const uint4*>(p) + 1);
      w[0] = u.x; w[1] = u.y; w[2] = u.z; w[3] = u.w;
      w[4] = v.x; w[5] = v.y; w[6] = v.z; w[7] = v.w;
    }
  }
  static __device__ __forceinline__ float get(const uint32_t* w, int e) {
    if constexpr (sizeof(XT) == 4) return __uint_as_float(w[e]);
    else return (e & 1) ? bf16hi_to_f32(w[e >> 1]) : bf16lo_to_f32(w[e >> 1]);
  }
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- cp.async ---------------------------------------------------------------------
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_8(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// ---- mbarrier / tcgen05 (sm_100a) ---------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::);
}
// Bounded wait (~2 s of SM clocks): a descriptor / protocol bug must surface as a trap, never as a
// hung GPU.
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    __nanosleep(64);   // polling warps must not steal issue slots from the warps they wait for
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
// 1-D bulk copy global -> shared (TMA engine, no tensor map), completion counted on an mbarrier.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}
// One lane of a converged warp.  Unlike `lane == 0`, the compiler knows that exactly one thread is
// active inside `if (elect_one())`, so warp-level instructions with uniform-register operands
// (tcgen05.mma / commit, bulk copies) are emitted straight instead of inside an ELECT / BRA.U.ANY loop
// that re-issues them once per possibly-active thread.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
}
template <int NCOLS> __device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_dst), "n"(NCOLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
}
template <int NCOLS> __device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(NCOLS));
}
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate, single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar)
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (lane i <-> TMEM lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 consecutive columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 4 consecutive columns
__device__ __forceinline__ void tmem_ld_32x4(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile: rows of 128 B, 8-row atoms of 1024 B (SBO),
// base 1024 B aligned.  cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout SWIZZLE_128B=2 [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128_kmajor(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// cute::UMMA::InstrDescriptor for kind::f16: D=f32 (bit4), A=B=bf16 (bits 7,10), K-major A/B,
// N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// byte offset of (row r, byte kb<128) inside a K-major SW128 tile
__device__ __forceinline__ uint32_t sw128_offset(uint32_t r, uint32_t kb) {
  return (r >> 3) * 1024u + (r & 7u) * 128u + ((((kb >> 4) ^ (r & 7u)) << 4) | (kb & 15u));
}

}  // namespace eavsr
