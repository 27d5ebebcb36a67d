// Fused producers / consumers around the alignment hot path (inference, sm_100a).
//
// ncu launch list of the full EAVSR+ forward (profiles/): once DCNv2 and the warps run on this
// library, 75 % of the device time is PyTorch glue between them -- cuDNN's grouped-direct kernel for
// the two tiny grouped 3x3 convolutions in every AdaptBlock (403 us per call), TensorIterator
// broadcast kernels for the affine offset expansion, and a reduce + four small launches per channel
// attention.  These kernels replace that glue:
//
//   adapt_mix        concat2(concat(cat[x, ref]))            models/networks.py:289-290,299 / 327-328,334
//                    = depthwise 3x3 (128 ch) + LeakyReLU(0.2) + grouped 3x3 (2 -> 1, 64 groups) +
//                    LeakyReLU(0.2) in ONE pass over the two inputs (50 MB instead of ~200 MB + 2 launches)
//   affine_offsets   T*R - R + t expansion + sigmoid(mask)   models/networks.py:302-313
//   channel_sum /    CALayer (global mean -> 1x1 -> ReLU -> 1x1 -> sigmoid -> scale) + residual add
//   ca_scale_residual                                        models/networks.py:449-465 (RCABlock)
#include <cuda.h>

#include "common.cuh"

namespace eavsr {
namespace {

// ---------------------------------------------------------------------------------------------
// adapt_mix
// ---------------------------------------------------------------------------------------------
// Persistent: each CTA stages both halves' weights once, then walks work items (image, tile, half) with a stride of
// the grid.  A tile's input (2-pixel halo, zero outside the image) arrives as one 4-D TMA tensor load into a
// two-deep mbarrier ring: the load of item j + 2 is issued as soon as item j's stage 1 has read its buffer, so it
// overlaps two items of math.  bf16 tiles stay small enough for two CTAs per SM (16 warps): the two __syncthreads
// of an item stall one CTA while the other computes.
constexpr int MX_C = 64;                        // channels of each input
constexpr int MX_NS = 2;                        // input ring depth

// output tile, threads and CTAs per SM of each instantiation
template <typename T> struct MixTile;
template <> struct MixTile<__nv_bfloat16> { static constexpr int TH = 8, TW = 16, THREADS = 256, MINB = 2; };
// fp32: the 8x16 tile's ring + y (178 KB) leaves one CTA per SM; measured faster than two CTAs on 8x8 tiles, which
// pay 1.56x stage-1 recompute and twice the per-item overhead
template <> struct MixTile<float> { static constexpr int TH = 8, TW = 16, THREADS = 256, MINB = 1; };

template <typename T> struct MixSmem {
  static constexpr int TH = MixTile<T>::TH, TW = MixTile<T>::TW;
  static constexpr int IH = TH + 4, IW = TW + 4, YH = TH + 2, YW = TW + 2;
  static constexpr uint32_t STAGE_BYTES = IH * IW * MX_C * sizeof(T);
  T in[MX_NS][IH * IW][MX_C];
  T y[YH * YW][MX_C];
  T w1[2][9][MX_C];                             // [half][tap][c]: depthwise weight of cat channel half * 64 + c
  T w2[2][9][MX_C];                             // [half][tap][c]: weight of y channel c into out channel half * 32 + c / 2
  float b1[2 * MX_C];
  float b2[MX_C];
  uint64_t full[MX_NS];
};
static_assert(MixSmem<__nv_bfloat16>::STAGE_BYTES % 128 == 0 && MixSmem<float>::STAGE_BYTES % 128 == 0,
              "ring stages must stay 128-byte aligned for the tensor loads");

struct MixParams {
  // (64 ch, W, H, N) views of a and b, box (64, TW + 4, TH + 4, 1), no swizzle, out-of-image pixels zero-filled
  alignas(64) CUtensorMap ta;
  alignas(64) CUtensorMap tb;
  const void* w1;
  const void* b1;
  const void* w2;
  const void* b2;
  void* out;
  int H, W, tiles_x, tiles_y, total;
  float slope;
};

// 8 consecutive channels as 32-bit registers and one multiply-add of channel e.  bf16 keeps the channels packed
// (4 registers) and multiplies them as they are: fma.rn.f32.bf16 (FHFMA.BF16 reading either half of a register)
// forms the exact product of two bf16 values and rounds its fp32 sum once, the same bits as widening both operands
// and issuing FFMA, without the 96 widening instructions per 144 FMAs that bound the kernel before.
template <typename T> struct MixMath;
template <> struct MixMath<__nv_bfloat16> {
  static constexpr int NR = 4;
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, uint32_t* r) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    r[0] = u.x; r[1] = u.y; r[2] = u.z; r[3] = u.w;
  }
  static __device__ __forceinline__ float fma(const uint32_t* w, const uint32_t* v, int e, float c) {
    const uint32_t a = w[e >> 1], b = v[e >> 1];
    const unsigned short x = (e & 1) ? (unsigned short)(a >> 16) : (unsigned short)(a & 0xffffu);
    const unsigned short y = (e & 1) ? (unsigned short)(b >> 16) : (unsigned short)(b & 0xffffu);
    float d;
    asm("fma.rn.f32.bf16 %0, %1, %2, %3;" : "=f"(d) : "h"(x), "h"(y), "f"(c));
    return d;
  }
  static __device__ __forceinline__ void st8(__nv_bfloat16* p, const float* f) { VecLoad<__nv_bfloat16, 8>::st(p, f); }
  static __device__ __forceinline__ void st4(__nv_bfloat16* p, const float* f) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]));
  }
};
template <> struct MixMath<float> {
  static constexpr int NR = 8;
  static __device__ __forceinline__ void ld(const float* p, uint32_t* r) {
    const uint4 a = *reinterpret_cast<const uint4*>(p), b = *reinterpret_cast<const uint4*>(p + 4);
    r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
  }
  static __device__ __forceinline__ float fma(const uint32_t* w, const uint32_t* v, int e, float c) {
    return fmaf(__uint_as_float(w[e]), __uint_as_float(v[e]), c);
  }
  static __device__ __forceinline__ void st8(float* p, const float* f) {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
  }
  static __device__ __forceinline__ void st4(float* p, const float* f) {
    *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  }
};

template <typename T>
__global__ void __launch_bounds__(MixTile<T>::THREADS, MixTile<T>::MINB) adapt_mix_kernel(const __grid_constant__ MixParams P) {
  using S_ = MixSmem<T>;
  using M = MixMath<T>;
  constexpr int TH = S_::TH, TW = S_::TW, IW = S_::IW, YH = S_::YH, YW = S_::YW, NR = M::NR;
  constexpr int NT = MixTile<T>::THREADS;
  extern __shared__ uint8_t mix_smem_raw[];
  S_& S = *reinterpret_cast<S_*>(mix_smem_raw + ((128u - (smem_u32(mix_smem_raw) & 127u)) & 127u));
  const int tid = threadIdx.x;
  const int my_items = (P.total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  // item j of this CTA: half fastest, so the a and b tiles of one place run side by side and the two 64-byte
  // halves of an output pixel reach L2 together
  auto item_at = [&](int j, int& n, int& half, int& y0, int& x0) {
    int t = (int)blockIdx.x + j * (int)gridDim.x;
    half = t & 1;
    t >>= 1;
    const int tx = t % P.tiles_x;
    t /= P.tiles_x;
    y0 = (t % P.tiles_y) * TH;
    n = t / P.tiles_y;
    x0 = tx * TW;
  };
  auto issue = [&](int j) {
    int n, half, y0, x0;
    item_at(j, n, half, y0, x0);
    const uint32_t bar = smem_u32(&S.full[j % MX_NS]);
    mbar_arrive_expect_tx(bar, S_::STAGE_BYTES);
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];\n" ::
            "r"(smem_u32(&S.in[j % MX_NS][0][0])),
        "l"(reinterpret_cast<uint64_t>(half ? &P.tb : &P.ta)), "r"(0), "r"(x0 - 2), "r"(y0 - 2), "r"(n), "r"(bar)
        : "memory");
  };

  if (tid == 0) {
    for (int s = 0; s < MX_NS; ++s) mbar_init(smem_u32(&S.full[s]), 1);
    fence_mbar_init();
    for (int j = 0; j < MX_NS && j < my_items; ++j) issue(j);
  }
  {
    const T* w1g = static_cast<const T*>(P.w1);
    const T* w2g = static_cast<const T*>(P.w2);
    for (int i = tid; i < 2 * 9 * MX_C; i += NT) {
      const int half = i / (9 * MX_C), tap = (i / MX_C) % 9, c = i % MX_C;
      S.w1[half][tap][c] = w1g[(size_t)(half * MX_C + c) * 9 + tap];
      S.w2[half][tap][c] = w2g[((size_t)(half * (MX_C / 2) + (c >> 1)) * 2 + (c & 1)) * 9 + tap];
    }
    for (int i = tid; i < 2 * MX_C; i += NT) S.b1[i] = to_f32<T>(static_cast<const T*>(P.b1)[i]);
    for (int i = tid; i < MX_C; i += NT) S.b2[i] = to_f32<T>(static_cast<const T*>(P.b2)[i]);
  }
  __syncthreads();

  // Every thread works on ONE 8-channel chunk for the whole kernel (NT % 8 == 0), so its 9 x 8 weights of a
  // stage live in registers and every tap is one 16-byte LDS + 8 FMAs per pixel.  Each thread computes TWO
  // horizontally adjacent pixels per step: 3 x 4 chunk loads feed 2 x 72 FMAs.
  const int c0 = (tid & 7) * 8;
  static_assert(YW % 2 == 0 && TW % 2 == 0 && NT % 8 == 0, "pixel pairs, whole chunk groups");
  T* out = static_cast<T*>(P.out);
  for (int j = 0; j < my_items; ++j) {
    int n, half, y0, x0;
    item_at(j, n, half, y0, x0);
    const int s = j % MX_NS;
    uint32_t wr[9][NR];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) M::ld(&S.w1[half][tap][c0], wr[tap]);
    mbar_wait(smem_u32(&S.full[s]), (j / MX_NS) & 1);

    // stage 1: y = lrelu(b1 + depthwise3x3(in)) on the (TH+2)x(TW+2) ring, rounded to T, 0 outside the image
    for (int i = tid; i < YH * (YW / 2) * (MX_C / 8); i += NT) {
      const int pp = i / (MX_C / 8);
      const int yy = pp / (YW / 2), xx = (pp % (YW / 2)) * 2;
      float acc[2][8];
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[0][e] = acc[1][e] = S.b1[half * MX_C + c0 + e];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        uint32_t v[4][NR];
#pragma unroll
        for (int c = 0; c < 4; ++c) M::ld(&S.in[s][(yy + r) * IW + xx + c][c0], v[c]);
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            acc[0][e] = M::fma(wr[r * 3 + t], v[t], e, acc[0][e]);
            acc[1][e] = M::fma(wr[r * 3 + t], v[t + 1], e, acc[1][e]);
          }
      }
      const int gy = y0 - 1 + yy;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int gx = x0 - 1 + xx + k;
        const bool inside = gy >= 0 && gy < P.H && gx >= 0 && gx < P.W;
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float v = acc[k][e] > 0.f ? acc[k][e] : acc[k][e] * P.slope;
          o[e] = inside ? v : 0.f;
        }
        M::st8(&S.y[yy * YW + xx + k][c0], o);
      }
    }
    __syncthreads();                            // y complete; every thread is done reading in[s]
    if (tid == 0 && j + MX_NS < my_items) issue(j + MX_NS);

    // stage 2: out[o] = lrelu(b2[o] + sum_tap w2[tap][2o] y[2o] + w2[tap][2o+1] y[2o+1])
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) M::ld(&S.w2[half][tap][c0], wr[tap]);
    for (int i = tid; i < TH * (TW / 2) * (MX_C / 8); i += NT) {
      const int pp = i / (MX_C / 8);
      const int yy = pp / (TW / 2), xx = (pp % (TW / 2)) * 2;
      const int gy = y0 + yy, gx = x0 + xx;
      if (gy >= P.H || gx >= P.W) continue;
      float acc[2][4];
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[0][e] = acc[1][e] = S.b2[half * (MX_C / 2) + (c0 >> 1) + e];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        uint32_t v[4][NR];
#pragma unroll
        for (int c = 0; c < 4; ++c) M::ld(&S.y[(yy + r) * YW + xx + c][c0], v[c]);
#pragma unroll
        for (int t = 0; t < 3; ++t)
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            acc[0][e >> 1] = M::fma(wr[r * 3 + t], v[t], e, acc[0][e >> 1]);
            acc[1][e >> 1] = M::fma(wr[r * 3 + t], v[t + 1], e, acc[1][e >> 1]);
          }
      }
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (gx + k >= P.W) continue;
        float o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = acc[k][e] > 0.f ? acc[k][e] : acc[k][e] * P.slope;
        M::st4(out + ((size_t)n * P.H * P.W + (size_t)gy * P.W + gx + k) * MX_C + half * (MX_C / 2) + (c0 >> 1), o);
      }
    }
    __syncthreads();                            // y is rewritten by the next item's stage 1
  }
}

// ---------------------------------------------------------------------------------------------
// affine offsets + sigmoid mask.  One thread per (pixel, group); outputs are fp32 NCHW planes
// (lanes along pixels -> coalesced), exactly the layout eavsr_dcn_forward consumes.
// offset[(g*9+k)*2+i] = T[g][i][0]*R0[k] + T[g][i][1]*R1[k] - R_i[k] + t[g][i]
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
affine_offsets_kernel(const T* __restrict__ tm, Strides4 ts, const T* __restrict__ tr, Strides4 rs,
                      const T* __restrict__ ml, Strides4 ms, const T* __restrict__ tm_bias,
                      const T* __restrict__ tr_bias, const T* __restrict__ ml_bias, float* __restrict__ offset,
                      float* __restrict__ mask, int N, int D, int H, int W) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long HW = (long long)H * W;
  if (idx >= (long long)N * D * HW) return;
  const int pix = (int)(idx % HW);
  const int g = (int)((idx / HW) % D);
  const int n = (int)(idx / (HW * D));
  const int y = pix / W, x = pix % W;
  const T* tp = tm + n * ts.n + y * ts.h + x * ts.w + (long long)(g * 4) * ts.c;
  const T* rp = tr + n * rs.n + y * rs.h + x * rs.w + (long long)(g * 2) * rs.c;
  float a = to_f32<T>(tp[0]), b = to_f32<T>(tp[ts.c]), c = to_f32<T>(tp[2 * ts.c]), d = to_f32<T>(tp[3 * ts.c]);
  float t0 = to_f32<T>(rp[0]), t1 = to_f32<T>(rp[rs.c]);
  if (tm_bias) {   // biases of the bias-free convolutions that produced T / t / logits
    a += to_f32<T>(tm_bias[g * 4]); b += to_f32<T>(tm_bias[g * 4 + 1]);
    c += to_f32<T>(tm_bias[g * 4 + 2]); d += to_f32<T>(tm_bias[g * 4 + 3]);
  }
  if (tr_bias) { t0 += to_f32<T>(tr_bias[g * 2]); t1 += to_f32<T>(tr_bias[g * 2 + 1]); }
  float* op = offset + ((size_t)(n * D + g) * 18) * HW + pix;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const float r0 = (float)(k / 3 - 1), r1 = (float)(k % 3 - 1);
    op[(size_t)(2 * k) * HW] = a * r0 + b * r1 - r0 + t0;
    op[(size_t)(2 * k + 1) * HW] = c * r0 + d * r1 - r1 + t1;
  }
  if (mask) {
    const T* mp = ml + n * ms.n + y * ms.h + x * ms.w + (long long)(g * 9) * ms.c;
    float* mo = mask + ((size_t)(n * D + g) * 9) * HW + pix;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const float lg = to_f32<T>(mp[k * ms.c]) + (ml_bias ? to_f32<T>(ml_bias[g * 9 + k]) : 0.f);
      mo[(size_t)k * HW] = 1.f / (1.f + __expf(-lg));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// channel attention: sums over H*W (NHWC), then out = res * sigmoid(MLP(mean)) + skip
// ---------------------------------------------------------------------------------------------
constexpr int CS_THREADS = 256;
constexpr int CS_PIX = 512;   // pixels per CTA

template <typename T, int C, bool PROD = false>
__global__ void __launch_bounds__(CS_THREADS)
channel_sum_kernel(const T* __restrict__ x, float* __restrict__ sums, int HW, const T* __restrict__ x2 = nullptr) {
  constexpr int VEC = 16 / sizeof(T);
  constexpr int CPP = C / VEC;
  constexpr int PPI = CS_THREADS / CPP;          // pixels per iteration
  __shared__ float red[PPI][C];
  const int n = blockIdx.y;
  const int ch = threadIdx.x % CPP, pl = threadIdx.x / CPP;
  const int p0 = blockIdx.x * CS_PIX;
  const int p1 = min(p0 + CS_PIX, HW);
  float acc[VEC];
#pragma unroll
  for (int e = 0; e < VEC; ++e) acc[e] = 0.f;
  const T* xn = x + (size_t)n * HW * C;
  for (int p = p0 + pl; p < p1; p += PPI) {
    float v[VEC];
    VecLoad<T, VEC>::ld(xn + (size_t)p * C + ch * VEC, v);
    if (PROD) {                                    // sums of the element-wise product of two tensors
      float u[VEC];
      VecLoad<T, VEC>::ld(x2 + (size_t)n * HW * C + (size_t)p * C + ch * VEC, u);
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[e] += v[e] * u[e];
    } else {
#pragma unroll
      for (int e = 0; e < VEC; ++e) acc[e] += v[e];
    }
  }
#pragma unroll
  for (int e = 0; e < VEC; ++e) red[pl][ch * VEC + e] = acc[e];
  __syncthreads();
  if (threadIdx.x < C) {
    float s = 0.f;
#pragma unroll 4
    for (int i = 0; i < PPI; ++i) s += red[i][threadIdx.x];
    atomicAdd(sums + n * C + threadIdx.x, s);
  }
}

template <typename T, int C, int R>
__global__ void __launch_bounds__(256)
ca_scale_residual_kernel(const T* __restrict__ res, const T* __restrict__ skip, const float* __restrict__ sums,
                         const T* __restrict__ w1, const T* __restrict__ b1, const T* __restrict__ w2,
                         const T* __restrict__ b2, const T* __restrict__ res_bias, T* __restrict__ out, int HW,
                         float inv_hw, int chunks_per_img) {
  constexpr int VEC = 16 / sizeof(T);
  constexpr int CPP = C / VEC;
  __shared__ float part[8];
  __shared__ float hid[R];
  __shared__ float scale[C];
  __shared__ float rb[C];                       // bias of the conv that produced `res` (0 if none)
  static_assert(R * C == 256, "one thread per (hidden unit, channel) product");
  const int n = blockIdx.y;
  // The squeeze-excite MLP is a prologue every CTA pays before it can stream: all 256 products of the
  // first layer are loaded and multiplied in parallel (one global round trip) and reduced with shuffles,
  // instead of four threads walking 64 dependent loads each (~3 us of a 12 us kernel).
  {
    const int r = threadIdx.x >> 6, i = threadIdx.x & 63;
    const float bi = res_bias ? to_f32<T>(res_bias[i]) : 0.f;
    if (r == 0) rb[i] = bi;
    float p = to_f32<T>(w1[r * C + i]) * (sums[n * C + i] * inv_hw + bi);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) p += __shfl_xor_sync(0xffffffffu, p, off);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = p;
  }
  __syncthreads();
  if (threadIdx.x < R) hid[threadIdx.x] = fmaxf(to_f32<T>(b1[threadIdx.x]) + part[2 * threadIdx.x] + part[2 * threadIdx.x + 1], 0.f);
  __syncthreads();
  if (threadIdx.x < C) {
    float a = to_f32<T>(b2[threadIdx.x]);
#pragma unroll
    for (int j = 0; j < R; ++j) a += to_f32<T>(w2[threadIdx.x * R + j]) * hid[j];
    scale[threadIdx.x] = 1.f / (1.f + __expf(-a));
  }
  __syncthreads();
  const size_t base = (size_t)n * HW * C;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < chunks_per_img; i += gridDim.x * 256) {
    const int ch = i % CPP;
    float r[VEC], s[VEC], o[VEC];
    VecLoad<T, VEC>::ld(res + base + (size_t)i * VEC, r);
    VecLoad<T, VEC>::ld(skip + base + (size_t)i * VEC, s);
#pragma unroll
    for (int e = 0; e < VEC; ++e) o[e] = (r[e] + rb[ch * VEC + e]) * scale[ch * VEC + e] + s[e];
    VecLoad<T, VEC>::st(out + base + (size_t)i * VEC, o);
  }
}

// x[p][c] = act(x[p][c] + bias[c]) in place on a dense NHWC tensor; act = LeakyReLU(slope)
// (slope 1 = identity, 0 = ReLU).  PyTorch adds a cuDNN convolution's bias with a broadcast
// TensorIterator kernel (not vectorised for channels_last: 17.6 us on a 64x272x480 bf16 map) and the
// activation with another launch; this is one 16-byte-vectorised pass.
template <typename T>
__global__ void __launch_bounds__(256)
bias_act_kernel(T* __restrict__ x, const T* __restrict__ bias, int C, long long nchunks, float slope) {
  constexpr int VEC = 16 / sizeof(T);
  const int cpp = C / VEC;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < nchunks; i += (long long)gridDim.x * 256) {
    const int ch = (int)(i % cpp);
    float v[VEC], b[VEC];
    VecLoad<T, VEC>::ld(x + i * VEC, v);
    VecLoad<T, VEC>::ld(bias + ch * VEC, b);
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      const float t = v[e] + b[e];
      v[e] = t > 0.f ? t : t * slope;
    }
    VecLoad<T, VEC>::st(x + i * VEC, v);
  }
}

// PixelShuffle(2) of a dense NHWC tensor with the producing convolution's bias and LeakyReLU folded
// in: out[n, 2h+i, 2w+j, c] = act(x[n, h, w, 4c + 2i + j] + bias[4c + 2i + j]).  One thread reads the
// 4*VEC consecutive input channels that make VEC output channels of the four output pixels (64 B)
// and writes four 16-byte vectors.  Replaces bias add + activation + pixel_shuffle + two layout copies
// (1.2 ms per 544x960 -> 1088x1920 frame in the ATen path).
template <typename T>
__global__ void __launch_bounds__(256)
bias_act_shuffle_kernel(const T* __restrict__ x, const T* __restrict__ bias, T* __restrict__ out, int Cout, int H,
                        int W, long long items, float slope) {
  constexpr int VEC = 16 / sizeof(T);
  const int cpp = Cout / VEC;                     // output chunks per input pixel
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < items; i += (long long)gridDim.x * 256) {
    const int ch = (int)(i % cpp);
    const long long pix = i / cpp;
    const int w = (int)(pix % W);
    const long long nh = pix / W;                 // n * H + h
    const T* ip = x + pix * (4 * Cout) + ch * (4 * VEC);
    float v[4 * VEC], b[4 * VEC];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      VecLoad<T, VEC>::ld(ip + k * VEC, v + k * VEC);
      if (bias) VecLoad<T, VEC>::ld(bias + ch * (4 * VEC) + k * VEC, b + k * VEC);
    }
#pragma unroll
    for (int e = 0; e < 4 * VEC; ++e) {
      const float t = v[e] + (bias ? b[e] : 0.f);
      v[e] = t > 0.f ? t : t * slope;
    }
#pragma unroll
    for (int ij = 0; ij < 4; ++ij) {
      float o[VEC];
#pragma unroll
      for (int e = 0; e < VEC; ++e) o[e] = v[e * 4 + ij];
      const long long orow = nh * 2 + (ij >> 1);  // n * 2H + 2h + i
      T* op = out + ((orow * (2 * W)) + 2 * w + (ij & 1)) * Cout + ch * VEC;
      VecLoad<T, VEC>::st(op, o);
    }
  }
}

bool dense_nhwc(const int64_t s[4], int c, int h, int w) {
  return s[1] == 1 && s[3] == c && s[2] == (int64_t)w * c && s[0] == (int64_t)h * w * c;
}
bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <typename T>
int mix_launch(const void* a, const void* b, const void* w1, const void* b1, const void* w2, const void* b2,
               void* out, int n, int h, int w, float slope, cudaStream_t st) {
  using S_ = MixSmem<T>;
  const int dt = sizeof(T) == 2 ? EAVSR_BF16 : EAVSR_F32;
  const long long total = 2ll * n * ceil_div(h, S_::TH) * ceil_div(w, S_::TW);
  EAVSR_REQUIRE(total < (1ll << 31), "adapt_mix: too many tiles");
  MixParams P;
  const unsigned long long dims[4] = {MX_C, (unsigned long long)w, (unsigned long long)h, (unsigned long long)n};
  const unsigned long long str[3] = {MX_C * sizeof(T), (unsigned long long)w * MX_C * sizeof(T),
                                     (unsigned long long)h * w * MX_C * sizeof(T)};
  const unsigned box[4] = {MX_C, S_::IW, S_::IH, 1};
  if (!encode_tensor_map(&P.ta, dt, 4, a, dims, str, box, 0 /* CU_TENSOR_MAP_SWIZZLE_NONE */) ||
      !encode_tensor_map(&P.tb, dt, 4, b, dims, str, box, 0)) {
    set_error("adapt_mix: the tensor maps of the inputs were rejected");
    return EAVSR_ERR_UNSUPPORTED;
  }
  P.w1 = w1; P.b1 = b1; P.w2 = w2; P.b2 = b2; P.out = out;
  P.H = h; P.W = w;
  P.tiles_x = ceil_div(w, S_::TW); P.tiles_y = ceil_div(h, S_::TH);
  P.total = (int)total;
  P.slope = slope;
  auto k = adapt_mix_kernel<T>;
  const int smem = (int)sizeof(S_) + 128;       // + alignment slack of the ring
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) { set_error("adapt_mix: smem attr: %s", cudaGetErrorString(e)); return EAVSR_ERR_CUDA; }
  int dev = 0, sms = 148, per_sm = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, MixTile<T>::THREADS, smem);
  if (e != cudaSuccess || per_sm < 1) { set_error("adapt_mix: occupancy: %s", cudaGetErrorString(e)); return EAVSR_ERR_CUDA; }
  const long long grid = total < (long long)sms * per_sm ? total : (long long)sms * per_sm;
  k<<<(unsigned)grid, MixTile<T>::THREADS, smem, st>>>(P);
  return check_launch("adapt_mix");
}

}  // namespace
}  // namespace eavsr

using namespace eavsr;

extern "C" int eavsr_adapt_mix_forward(const void* a, const void* b, const void* w1, const void* b1,
                                       const void* w2, const void* b2, void* out, int n, int c, int h, int w,
                                       float negative_slope, int dtype, void* stream) {
  EAVSR_REQUIRE(a && b && w1 && b1 && w2 && b2 && out, "adapt_mix: null pointer");
  EAVSR_REQUIRE(n > 0 && h > 0 && w > 0, "adapt_mix: empty tensor");
  if (c != MX_C) { set_error("adapt_mix: only %d-channel inputs are fused (got %d)", MX_C, c); return EAVSR_ERR_UNSUPPORTED; }
  EAVSR_REQUIRE(al16(a) && al16(b) && al16(out), "adapt_mix: tensors must be 16-byte aligned dense NHWC");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == EAVSR_F32) return mix_launch<float>(a, b, w1, b1, w2, b2, out, n, h, w, negative_slope, st);
  if (dtype == EAVSR_BF16) return mix_launch<__nv_bfloat16>(a, b, w1, b1, w2, b2, out, n, h, w, negative_slope, st);
  set_error("adapt_mix: bad dtype %d", dtype);
  return EAVSR_ERR_INVALID;
}

extern "C" int eavsr_affine_offsets_forward(const void* transform, const int64_t transform_strides[4],
                                            const void* translation, const int64_t translation_strides[4],
                                            const void* mask_logits, const int64_t mask_strides[4],
                                            const void* transform_bias, const void* translation_bias,
                                            const void* mask_bias, float* offset, float* mask, int n,
                                            int deform_groups, int h, int w, int dtype, void* stream) {
  EAVSR_REQUIRE(transform && translation && offset && transform_strides && translation_strides,
                "affine_offsets: null pointer");
  EAVSR_REQUIRE(!mask || (mask_logits && mask_strides), "affine_offsets: mask output without logits");
  EAVSR_REQUIRE(n > 0 && deform_groups > 0 && h > 0 && w > 0, "affine_offsets: empty tensor");
  cudaStream_t st = (cudaStream_t)stream;
  Strides4 ts{transform_strides[0], transform_strides[1], transform_strides[2], transform_strides[3]};
  Strides4 rs{translation_strides[0], translation_strides[1], translation_strides[2], translation_strides[3]};
  Strides4 ms{0, 0, 0, 0};
  if (mask) ms = Strides4{mask_strides[0], mask_strides[1], mask_strides[2], mask_strides[3]};
  const long long total = (long long)n * deform_groups * h * w;
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (dtype == EAVSR_F32)
    affine_offsets_kernel<float><<<blocks, 256, 0, st>>>((const float*)transform, ts, (const float*)translation, rs,
                                                         (const float*)mask_logits, ms, (const float*)transform_bias,
                                                         (const float*)translation_bias, (const float*)mask_bias,
                                                         offset, mask, n, deform_groups, h, w);
  else if (dtype == EAVSR_BF16)
    affine_offsets_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(
        (const __nv_bfloat16*)transform, ts, (const __nv_bfloat16*)translation, rs,
        (const __nv_bfloat16*)mask_logits, ms, (const __nv_bfloat16*)transform_bias,
        (const __nv_bfloat16*)translation_bias, (const __nv_bfloat16*)mask_bias, offset, mask, n, deform_groups, h, w);
  else { set_error("affine_offsets: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("affine_offsets");
}

extern "C" int eavsr_ca_residual_forward(const void* res, const void* skip, const void* w1, const void* b1,
                                         const void* w2, const void* b2, const void* res_bias, void* out,
                                         float* sums_workspace, int n, int c, int h, int w, int reduction, int dtype,
                                         void* stream) {
  EAVSR_REQUIRE(res && skip && w1 && b1 && w2 && b2 && out && sums_workspace, "ca_residual: null pointer");
  EAVSR_REQUIRE(n > 0 && h > 0 && w > 0, "ca_residual: empty tensor");
  if (c != 64 || reduction != 16) {
    set_error("ca_residual: only C=64, reduction=16 is fused (got C=%d, r=%d)", c, reduction);
    return EAVSR_ERR_UNSUPPORTED;
  }
  EAVSR_REQUIRE(al16(res) && al16(skip) && al16(out), "ca_residual: tensors must be 16-byte aligned dense NHWC");
  EAVSR_REQUIRE(n <= 65535, "ca_residual: batch too large");
  cudaStream_t st = (cudaStream_t)stream;
  const int HW = h * w;
  cudaError_t e = cudaMemsetAsync(sums_workspace, 0, (size_t)n * c * sizeof(float), st);
  if (e != cudaSuccess) { set_error("ca_residual: memset: %s", cudaGetErrorString(e)); return EAVSR_ERR_CUDA; }
  dim3 g1(ceil_div(HW, CS_PIX), n);
  int rc;
  if (dtype == EAVSR_F32) {
    channel_sum_kernel<float, 64><<<g1, CS_THREADS, 0, st>>>((const float*)res, sums_workspace, HW);
    rc = check_launch("ca_residual(sum)");
    if (rc) return rc;
    const int chunks = HW * 64 / 4;
    dim3 g2(min(ceil_div(chunks, 256 * 4), 148 * 8), n);
    ca_scale_residual_kernel<float, 64, 4><<<g2, 256, 0, st>>>((const float*)res, (const float*)skip, sums_workspace,
                                                             (const float*)w1, (const float*)b1, (const float*)w2,
                                                             (const float*)b2, (const float*)res_bias, (float*)out, HW,
                                                             1.f / (float)HW, chunks);
  } else if (dtype == EAVSR_BF16) {
    using B = __nv_bfloat16;
    channel_sum_kernel<B, 64><<<g1, CS_THREADS, 0, st>>>((const B*)res, sums_workspace, HW);
    rc = check_launch("ca_residual(sum)");
    if (rc) return rc;
    const int chunks = HW * 64 / 8;
    dim3 g2(min(ceil_div(chunks, 256 * 4), 148 * 8), n);
    ca_scale_residual_kernel<B, 64, 4><<<g2, 256, 0, st>>>((const B*)res, (const B*)skip, sums_workspace, (const B*)w1,
                                                         (const B*)b1, (const B*)w2, (const B*)b2, (const B*)res_bias,
                                                         (B*)out, HW, 1.f / (float)HW, chunks);
  } else { set_error("ca_residual: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("ca_residual(scale)");
}

extern "C" int eavsr_bias_act_forward(void* x, const void* bias, int c, long long pixels, float negative_slope,
                                      int dtype, void* stream) {
  EAVSR_REQUIRE(x && bias, "bias_act: null pointer");
  EAVSR_REQUIRE(c > 0 && pixels > 0, "bias_act: empty tensor");
  const int vec = dtype == EAVSR_F32 ? 4 : 8;
  if (c % vec != 0 || !al16(x) || !al16(bias)) {
    set_error("bias_act: needs C %% %d == 0 and 16-byte aligned dense NHWC data (C=%d)", vec, c);
    return EAVSR_ERR_UNSUPPORTED;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const long long nchunks = pixels * (c / vec);
  long long blocks = (nchunks + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (dtype == EAVSR_F32)
    bias_act_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((float*)x, (const float*)bias, c, nchunks, negative_slope);
  else if (dtype == EAVSR_BF16)
    bias_act_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, st>>>((__nv_bfloat16*)x, (const __nv_bfloat16*)bias, c,
                                                                    nchunks, negative_slope);
  else { set_error("bias_act: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("bias_act");
}

// ---------------------------------------------------------------------------------------------
// nhwc_cat: torch.cat(dim=1) of dense NHWC tensors into (a channel slice of) an NHWC buffer
// ---------------------------------------------------------------------------------------------
// The concatenations in front of the fusion / backbone / reconstruction convolutions (models/eavsrp_model.py:
// 271-324, 350-364; 128..320 channels at full resolution) ran at ~1 TB/s in ATen's generic cat kernel (it does
// not know the tensors are channels_last) and were 6.5 % of the device time.  Here every thread moves 16-byte
// chunks: consecutive threads read consecutive chunks of one source pixel and write consecutive chunks of the
// output pixel, both fully coalesced.
constexpr int CAT_MAX = 8;
struct CatParams {
  const uint4* src[CAT_MAX];
  int cpp[CAT_MAX];          // 16-byte chunks per pixel of each source
  int first[CAT_MAX + 1];    // prefix sums of cpp
  int nsrc;
  int out_cpp;               // chunks per pixel of the OUTPUT buffer (its pixel stride)
  int out_off;               // first chunk written inside an output pixel
};

__global__ void __launch_bounds__(256)
nhwc_cat_kernel(const __grid_constant__ CatParams P, uint4* __restrict__ out, long long pixels) {
  const int total_cpp = P.first[P.nsrc];
  const long long n = pixels * total_cpp;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const float rcp = 1.f / (float)total_cpp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    long long px;
    int ch;
    if (n < (1ll << 22)) {                       // float reciprocal + one correction: exact below 2^22
      int q = __float2int_rz((float)(int)i * rcp), r = (int)i - q * total_cpp;
      if (r < 0) { r += total_cpp; --q; }
      if (r >= total_cpp) { r -= total_cpp; ++q; }
      px = q; ch = r;
    } else {
      px = i / total_cpp; ch = (int)(i - px * total_cpp);
    }
    int s = 0;
#pragma unroll
    for (int k = 1; k < CAT_MAX; ++k) s += (k < P.nsrc && ch >= P.first[k]) ? 1 : 0;
    const uint4 v = __ldg(P.src[s] + px * P.cpp[s] + (ch - P.first[s]));
    out[px * P.out_cpp + P.out_off + ch] = v;
  }
}

// Scale + residual only, with channel sums that were produced elsewhere (the epilogue of
// eavsr_conv3x3_forward): out = (res + res_bias) * sigmoid(MLP(sums / HW + res_bias)) + skip.
extern "C" int eavsr_ca_scale_forward(const void* res, const void* skip, const float* sums, const void* w1,
                                      const void* b1, const void* w2, const void* b2, const void* res_bias, void* out,
                                      int n, int c, int h, int w, int reduction, int dtype, void* stream) {
  EAVSR_REQUIRE(res && skip && sums && w1 && b1 && w2 && b2 && out, "ca_scale: null pointer");
  EAVSR_REQUIRE(n > 0 && h > 0 && w > 0 && n <= 65535, "ca_scale: bad shape");
  if (c != 64 || reduction != 16) {
    set_error("ca_scale: only C=64, reduction=16 is fused (got C=%d, r=%d)", c, reduction);
    return EAVSR_ERR_UNSUPPORTED;
  }
  EAVSR_REQUIRE(al16(res) && al16(skip) && al16(out), "ca_scale: tensors must be 16-byte aligned dense NHWC");
  cudaStream_t st = (cudaStream_t)stream;
  const int HW = h * w;
  if (dtype == EAVSR_F32) {
    const int chunks = HW * 64 / 4;
    dim3 g2(min(ceil_div(chunks, 256 * 4), 148 * 8), n);
    ca_scale_residual_kernel<float, 64, 4><<<g2, 256, 0, st>>>((const float*)res, (const float*)skip, sums,
                                                             (const float*)w1, (const float*)b1, (const float*)w2,
                                                             (const float*)b2, (const float*)res_bias, (float*)out, HW,
                                                             1.f / (float)HW, chunks);
  } else if (dtype == EAVSR_BF16) {
    using B = __nv_bfloat16;
    const int chunks = HW * 64 / 8;
    dim3 g2(min(ceil_div(chunks, 256 * 4), 148 * 8), n);
    ca_scale_residual_kernel<B, 64, 4><<<g2, 256, 0, st>>>((const B*)res, (const B*)skip, sums, (const B*)w1,
                                                         (const B*)b1, (const B*)w2, (const B*)b2, (const B*)res_bias,
                                                         (B*)out, HW, 1.f / (float)HW, chunks);
  } else { set_error("ca_scale: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("ca_scale");
}

extern "C" int eavsr_bias_act_shuffle_forward(const void* x, const void* bias, void* out, int n, int c_out, int h,
                                              int w, float negative_slope, int dtype, void* stream) {
  EAVSR_REQUIRE(x && out, "bias_act_shuffle: null pointer");
  EAVSR_REQUIRE(n > 0 && c_out > 0 && h > 0 && w > 0, "bias_act_shuffle: empty tensor");
  const int vec = dtype == EAVSR_F32 ? 4 : 8;
  if (c_out % vec != 0 || !al16(x) || !al16(out) || (bias && !al16(bias))) {
    set_error("bias_act_shuffle: needs C_out %% %d == 0 and 16-byte aligned dense NHWC data (C_out=%d)", vec, c_out);
    return EAVSR_ERR_UNSUPPORTED;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const long long items = (long long)n * h * w * (c_out / vec);
  long long blocks = (items + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (dtype == EAVSR_F32)
    bias_act_shuffle_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((const float*)x, (const float*)bias, (float*)out,
                                                                    c_out, h, w, items, negative_slope);
  else if (dtype == EAVSR_BF16)
    bias_act_shuffle_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, st>>>(
        (const __nv_bfloat16*)x, (const __nv_bfloat16*)bias, (__nv_bfloat16*)out, c_out, h, w, items, negative_slope);
  else { set_error("bias_act_shuffle: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("bias_act_shuffle");
}

extern "C" int eavsr_nhwc_cat_forward(const void* const* srcs, const int* src_channels, int nsrc, void* out,
                                      int out_channels, int out_channel_offset, long long pixels, int dtype,
                                      void* stream) {
  EAVSR_REQUIRE(srcs && src_channels && out, "nhwc_cat: null pointer");
  EAVSR_REQUIRE(nsrc >= 1 && nsrc <= CAT_MAX, "nhwc_cat: 1..%d sources (got %d)", CAT_MAX, nsrc);
  EAVSR_REQUIRE(pixels > 0, "nhwc_cat: empty tensor");
  if (dtype != EAVSR_F32 && dtype != EAVSR_BF16) { set_error("nhwc_cat: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  const int vec = dtype == EAVSR_F32 ? 4 : 8;
  CatParams P;
  P.nsrc = nsrc;
  P.first[0] = 0;
  for (int i = 0; i < nsrc; ++i) {
    EAVSR_REQUIRE(srcs[i], "nhwc_cat: null source %d", i);
    if (src_channels[i] <= 0 || src_channels[i] % vec != 0 || !al16(srcs[i])) {
      set_error("nhwc_cat: source %d needs C %% %d == 0 and 16-byte alignment (C=%d)", i, vec, src_channels[i]);
      return EAVSR_ERR_UNSUPPORTED;
    }
    P.src[i] = (const uint4*)srcs[i];
    P.cpp[i] = src_channels[i] / vec;
    P.first[i + 1] = P.first[i] + P.cpp[i];
  }
  for (int i = nsrc; i < CAT_MAX; ++i) { P.src[i] = nullptr; P.cpp[i] = 0; P.first[i + 1] = P.first[nsrc]; }
  if (out_channels % vec != 0 || out_channel_offset % vec != 0 || out_channel_offset < 0 || !al16(out) ||
      out_channel_offset / vec + P.first[nsrc] > out_channels / vec) {
    set_error("nhwc_cat: output slice [%d, +%d) of %d channels must be 16-byte aligned and inside the buffer",
              out_channel_offset, P.first[nsrc] * vec, out_channels);
    return EAVSR_ERR_INVALID;
  }
  P.out_cpp = out_channels / vec;
  P.out_off = out_channel_offset / vec;
  const long long n = pixels * P.first[nsrc];
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 32) blocks = 148 * 32;
  nhwc_cat_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(P, (uint4*)out, pixels);
  return check_launch("nhwc_cat");
}

// Per-(n, channel) sums over H*W of a dense NHWC tensor with 64 channels, fp32 (sums is zero-filled here): the
// bias gradient of the 64-output convolutions and the global average pooling of CALayer in the training step, where
// ATen's generic reduction of a channels_last tensor took 30 us per 4 MB tensor.
extern "C" int eavsr_channel_sum_forward(const void* x, float* sums, int n, int c, long long hw, int dtype, void* stream) {
  EAVSR_REQUIRE(x && sums, "channel_sum: null pointer");
  EAVSR_REQUIRE(n > 0 && hw > 0 && hw < (1ll << 31) && n <= 65535, "channel_sum: bad shape");
  if (c != 64) { set_error("channel_sum: only C=64 (got %d)", c); return EAVSR_ERR_UNSUPPORTED; }
  EAVSR_REQUIRE(al16(x), "channel_sum: x must be 16-byte aligned dense NHWC");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)n * c * sizeof(float), st);
  if (e != cudaSuccess) { set_error("channel_sum: memset: %s", cudaGetErrorString(e)); return EAVSR_ERR_CUDA; }
  dim3 g1(ceil_div(hw, CS_PIX), n);
  if (dtype == EAVSR_F32) channel_sum_kernel<float, 64><<<g1, CS_THREADS, 0, st>>>((const float*)x, sums, (int)hw);
  else if (dtype == EAVSR_BF16) channel_sum_kernel<__nv_bfloat16, 64><<<g1, CS_THREADS, 0, st>>>((const __nv_bfloat16*)x, sums, (int)hw);
  else { set_error("channel_sum: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("channel_sum");
}


// sums(n, 64) = sum over the pixels of a * b (both (n, 64, h, w) dense NHWC): the gradient of the channel-attention
// scale in `res * scale + skip` (d scale = sum_hw(grad * res)), one pass instead of a multiply + ATen reduction.
extern "C" int eavsr_channel_dot_forward(const void* a, const void* b, float* sums, int n, int c, long long hw, int dtype,
                                         void* stream) {
  EAVSR_REQUIRE(a && b && sums, "channel_dot: null pointer");
  EAVSR_REQUIRE(n > 0 && hw > 0 && hw < (1ll << 31) && n <= 65535, "channel_dot: bad shape");
  if (c != 64) { set_error("channel_dot: only C=64 (got %d)", c); return EAVSR_ERR_UNSUPPORTED; }
  EAVSR_REQUIRE(al16(a) && al16(b), "channel_dot: tensors must be 16-byte aligned dense NHWC");
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(sums, 0, (size_t)n * c * sizeof(float), st);
  if (e != cudaSuccess) { set_error("channel_dot: memset: %s", cudaGetErrorString(e)); return EAVSR_ERR_CUDA; }
  dim3 g1(ceil_div(hw, CS_PIX), n);
  if (dtype == EAVSR_F32)
    channel_sum_kernel<float, 64, true><<<g1, CS_THREADS, 0, st>>>((const float*)a, sums, (int)hw, (const float*)b);
  else if (dtype == EAVSR_BF16)
    channel_sum_kernel<__nv_bfloat16, 64, true><<<g1, CS_THREADS, 0, st>>>((const __nv_bfloat16*)a, sums, (int)hw,
                                                                          (const __nv_bfloat16*)b);
  else { set_error("channel_dot: bad dtype %d", dtype); return EAVSR_ERR_INVALID; }
  return check_launch("channel_dot");
}
