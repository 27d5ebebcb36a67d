// Reconstruction tail of EAVSR+ as one tcgen05 kernel, writing 8-bit frames (models/eavsrp_model.py:350-364 followed
// by the visuals of models/base_model.py:146-150), or 16-bit ones (M = 2^bits - 1 in place of 255), or Y'CbCr 4:2:0
// planes of 8- or 16-bit samples, or the 8-bit frame's squared error against a ground-truth frame (the store types
// below):
//
//   out[n, y, x, c] = rint(clamp(255 * (b[c] + sum_{k,ci} W[c,ci,k] X[n,ci,y+ky-1,x+kx-1] + up_s(lr)[n,c,y,x]), 0, 255))
//
// X is the (n, 64, H, W) bf16 NHWC output of conv_hr + LeakyReLU, W / b are conv_last (64 -> 3, 3x3, pad 1), up_s is
// ATen's bilinear upsampling (align_corners=False, scale_factor=s) of the fp32 LR frame.  The composition it replaces
// reads the 128 B/px feature map with cuDNN, writes and re-reads an fp32 SR frame three times and converts last; here
// the features are read once and 3 bytes per pixel are written.
//
// The recipe of conv3x3_tc.cu (DESIGN.md 3.4, 3.7b): a 6 x 32-pixel halo tile of 64 channels arrives by one 4-D tensor
// load with 128-byte swizzle and zero fill (the convolution's padding) and is the K-major SW128 A operand of the MMAs
// through views advanced by whole halo rows.  One MMA per kernel row (M = 128 halo positions, N = 48): the B operand is
// the three taps of the row, each padded to 16 output rows (3 real, 13 zero), so accumulator block c (16 columns) holds
// D_c[m] = sum_r halo(32 r + m) . W(r, c) and the output at halo position p is D_0[p] + D_1[p + 1] + D_2[p + 2] -- two
// shfl.down in the epilogue.  A tile is a 4 x 32 block of which 4 x 30 are outputs.
//
// Warp roles (320 threads, 1 CTA / SM, persistent over tiles):
//   warp  0    one lane issues the halo tensor loads into a ST_NS-stage ring (re-requests a stage when the MMAs that
//              read it have completed)
//   warp  1    TMEM owner; one lane loads the 18 KB of packed weights, issues 12 MMAs per tile, commits to mbarriers
//   warps 2-9  two epilogue teams of four warps (one TMEM lane quadrant = one tile row each); team t drains accumulator
//              buffer t: bilinear base from the LR frame (loads issued before the accumulator wait), tcgen05.ld,
//              shifted sum, + bias, quantise, 3 byte stores per pixel (RgbSse: and the squared error against a
//              ground-truth frame, one 64-bit atomic per warp and image)
#include <cuda.h>

#include <type_traits>

#include "common.cuh"

namespace eavsr {
namespace {

constexpr int ST_CH = 64;
constexpr int ST_TR = 4, ST_TC = 30;            // real outputs per tile
constexpr int ST_PW = 32;                       // halo pitch in pixels (= MMA rows per output row)
constexpr int ST_HROWS = (ST_TR + 2) * ST_PW;   // 192 halo positions; row-shifted views read rows 0 .. 191
constexpr int ST_ASTAGE = ST_HROWS * 128;       // 24 KB (24 swizzle atoms: stages stay atom-aligned)
constexpr int ST_NS = 6;                        // halo stages
constexpr int ST_NPAD = 16;                     // output rows per tap in the packed weights (3 real)
constexpr int ST_BTAP = ST_NPAD * ST_CH * 2;    // 2 KB per tap
constexpr int ST_N = 3 * ST_NPAD;               // MMA N: the three taps of a kernel row
constexpr int ST_ACC = 64;                      // TMEM column stride of the two accumulator buffers
constexpr int ST_TMEM = 128;
constexpr int ST_THREADS = 320;

struct StSmem {
  static constexpr int B_OFF = 0;                                  // 9 x 2 KB, 1024-aligned
  static constexpr int A_OFF = B_OFF + 9 * ST_BTAP;                // 18 KB: still 1024-aligned
  static constexpr int BAR_OFF = A_OFF + ST_NS * ST_ASTAGE;
  // full[NS], empty[NS], accf[2], acce[2], wbar; then the tmem slot
  static constexpr int NBARS = 2 * ST_NS + 5;
  static constexpr int TOTAL = BAR_OFF + NBARS * 8 + 16;
  static constexpr int DYN = TOTAL + 1024;
};

// The epilogue's store, a template parameter of the kernel: interleaved RGB, or Y'CbCr 4:2:0 planes, of 8-bit samples
// or of 16-bit samples (10-, 12- or 16-bit codes).  T is the sample type; the 8-bit stores keep their constants as
// immediates, the 16-bit ones carry theirs.
struct RgbOut {
  using T = uint8_t;
  uint8_t* p;
  long long s_n, s_y, s_x, s_c;
};
struct Rgb16Out {
  using T = uint16_t;
  uint16_t* p;
  long long s_n, s_y, s_x, s_c;
  float m;                         // 2^bits - 1
};
template <class T>
struct PlaneOutT {
  T* p;
  long long s_n, s_y, s_x;
};
using PlaneOut = PlaneOutT<uint8_t>;
struct Yuv420Out {
  using T = uint8_t;
  PlaneOut y, u, v;                // u, v: (out_h / 2, out_w / 2)
  float kr, kg, kb, cu, cv;        // fp32 coefficients of eavsr_b200/yuv.py: cu = 112 / (1 - kb), cv = 112 / (1 - kr)
};
struct Yuv420Out16 {
  using T = uint16_t;
  PlaneOutT<uint16_t> y, u, v;
  float kr, kg, kb, cu, cv;        // with k = 2^(bits - 8): cu = 112k / (1 - kb), cv = 112k / (1 - kr)
  float ys, yo, co;                // 219k, 16k, 128k
  int shift;                       // codes are stored times 2^shift
};
// The 8-bit RGB codes of RgbOut measured against a ground-truth frame: sse[n * sse_s] += sum over the valid pixels
// of image n of (q - gt)^2, exact in integers.  The frame itself is stored only when p is set.
struct RgbSse {
  using T = uint8_t;
  const uint8_t* gt;
  long long g_n, g_y, g_x, g_c;
  uint8_t* p;                      // null: no store
  long long s_n, s_y, s_x, s_c;
  unsigned long long* sse;         // added to, never overwritten
  long long sse_s;
};
template <class Out>
constexpr bool is_yuv420 = std::is_same<Out, Yuv420Out>::value || std::is_same<Out, Yuv420Out16>::value;

template <class Out>
struct TailParams {
  // (64 ch, W, H, N) bf16 view of X, box (64, 32, 6, 1), 128-byte swizzle, out-of-image pixels zero-filled
  alignas(64) CUtensorMap tm;
  const uint8_t* wpacked;
  const __nv_bfloat16* bias;       // (3) or null
  const float* lr;
  long long ls_n, ls_c, ls_h, ls_w;
  Out out;
  int out_h, out_w, lr_h, lr_w, tiles_x, tiles_per_img, total_tiles;
  float inv_scale;
};

// 4:2:0: the odd-row warp of each (q, q + 1) pair hands its horizontal pair sums to the even-row warp through a
// double-buffered slot of 2 x 3 x 16 floats; one named barrier per pair (ids 1-4)
constexpr int ST_XCH = 4 * 2 * 3 * 16 * 4;
template <class Out>
constexpr int st_dyn() { return StSmem::DYN + (is_yuv420<Out> ? ST_XCH : 0); }

// packed[tap][o][ci] (o < 16, K-major SW128) = W[o, ci, tap] for o < 3, 0 otherwise
__global__ void sr_tail_pack_weight_kernel(const __nv_bfloat16* __restrict__ w, uint8_t* __restrict__ packed) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // (tap, o, ci)
  if (idx >= 9 * ST_NPAD * ST_CH) return;
  const int ci = idx % ST_CH, o = (idx / ST_CH) % ST_NPAD, t = idx / (ST_CH * ST_NPAD);
  *reinterpret_cast<__nv_bfloat16*>(packed + (size_t)t * ST_BTAP + sw128_offset(o, ci * 2)) =
      o < 3 ? w[((size_t)o * ST_CH + ci) * 9 + t] : __float2bfloat16_rn(0.f);
}

// RgbSse: the warp's sum of its lanes' running sums, added to image n's total by one 64-bit atomic
__device__ __forceinline__ void sse_flush(const RgbSse& o, int n, unsigned long long acc, int lane) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0 && acc != 0) atomicAdd(o.sse + n * o.sse_s, acc);
}

template <class Out>
__global__ void __launch_bounds__(ST_THREADS, 1) sr_tail_u8_kernel(const __grid_constant__ TailParams<Out> P) {
  constexpr bool YUV = is_yuv420<Out>;
  constexpr bool SSE = std::is_same<Out, RgbSse>::value;
  using T = typename Out::T;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sB = base + StSmem::B_OFF, sA = base + StSmem::A_OFF, bars = base + StSmem::BAR_OFF;
  const uint32_t bar_full = bars, bar_empty = bars + ST_NS * 8, bar_accf = bars + 2 * ST_NS * 8;
  const uint32_t bar_acce = bar_accf + 16, bar_w = bar_acce + 16;
  const uint32_t tmem_slot_addr = bars + StSmem::NBARS * 8;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + StSmem::BAR_OFF + StSmem::NBARS * 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int first = blockIdx.x;
  const int my_tiles = (P.total_tiles - first + (int)gridDim.x - 1) / (int)gridDim.x;
  if (tid == 0) {
    for (int s = 0; s < ST_NS; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_accf + 8 * b, 1);
      mbar_init(bar_acce + 8 * b, 4);                           // the four warps of the team that drains buffer b
    }
    mbar_init(bar_w, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<ST_TMEM>(tmem_slot_addr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_slot;

  auto tile_at = [&](int tl, int& n, int& ty, int& tx) {
    const int tile = first + tl * (int)gridDim.x;
    n = tile / P.tiles_per_img;
    const int rem = tile - n * P.tiles_per_img;
    ty = rem / P.tiles_x;
    tx = rem - ty * P.tiles_x;
  };

  if (warp == 0) {
    // ===================== halo loads =====================
    if (elect_one()) {
      for (int tl = 0; tl < my_tiles; ++tl) {
        const int s = tl % ST_NS;
        if (tl >= ST_NS) mbar_wait(bar_empty + 8 * s, ((tl / ST_NS) - 1) & 1);
        int n, ty, tx;
        tile_at(tl, n, ty, tx);
        mbar_arrive_expect_tx(bar_full + 8 * s, ST_ASTAGE);
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];\n" ::
                "r"(sA + s * ST_ASTAGE),
            "l"(reinterpret_cast<uint64_t>(&P.tm)), "r"(0), "r"(tx * ST_TC - 1), "r"(ty * ST_TR - 1), "r"(n),
            "r"(bar_full + 8 * s)
            : "memory");
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      mbar_arrive_expect_tx(bar_w, 9 * ST_BTAP);
      bulk_g2s(sB, P.wpacked, 9 * ST_BTAP, bar_w);
      mbar_wait(bar_w, 0);
      constexpr uint32_t IDESC = umma_idesc_bf16(128, ST_N);
      const uint64_t b_base = umma_desc_sw128_kmajor(sB);
      for (int tl = 0; tl < my_tiles; ++tl) {
        const int s = tl % ST_NS, buf = tl & 1;
        if (tl >= 2) mbar_wait(bar_acce + 8 * buf, ((tl >> 1) - 1) & 1);
        mbar_wait(bar_full + 8 * s, (tl / ST_NS) & 1);
        tc_fence_after();
        const uint64_t a_base = umma_desc_sw128_kmajor(sA + s * ST_ASTAGE);
        const uint32_t d = tmem_d + buf * ST_ACC;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // A: halo advanced by r rows of 32 pixels (4 whole swizzle atoms); B: taps (r, 0..2) = 48 rows, 6 atoms
            const uint64_t adesc = a_base + (uint64_t)((r * ST_PW * 128) >> 4) + 2 * k;
            const uint64_t bdesc = b_base + (uint64_t)((r * 3 * ST_BTAP) >> 4) + 2 * k;
            umma_bf16(d, adesc, bdesc, IDESC, (r | k) != 0);
          }
        }
        umma_commit(bar_empty + 8 * s);
        umma_commit(bar_accf + 8 * buf);
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue =====================
    const int team = (warp - 2) >> 2;
    const int q = warp & 3;                       // TMEM lane quadrant = output row of the tile
    float bias[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) bias[c] = P.bias ? __bfloat162float(P.bias[c]) : 0.f;
    // RgbSse: this lane's running sum over the tiles of image sse_n.  The team's tiles come in increasing order, so n
    // never decreases along them, and each image's sum leaves the warp once, when n changes and after the last tile
    unsigned long long sse_acc = 0;
    int sse_n = -1;
    for (int tl = team; tl < my_tiles; tl += 2) {
      int n, ty, tx;
      tile_at(tl, n, ty, tx);
      const int y = ty * ST_TR + q, x = tx * ST_TC + lane;
      const bool valid = lane < ST_TC && y < P.out_h && x < P.out_w;
      // bilinear base, ATen's upsample_bilinear2d (align_corners=False, scale_factor=s) in its order of operations
      float up[3] = {0.f, 0.f, 0.f};
      uint32_t gt[3] = {0u, 0u, 0u};
      if (valid) {
        if constexpr (SSE) {
          // the ground truth, loaded with the LR samples: both arrive while the MMAs finish
          const uint8_t* g = P.out.gt + n * P.out.g_n + (long long)y * P.out.g_y + (long long)x * P.out.g_x;
#pragma unroll
          for (int c = 0; c < 3; ++c) gt[c] = __ldg(g + c * P.out.g_c);
        }
        const float sy = fmaxf(P.inv_scale * ((float)y + 0.5f) - 0.5f, 0.f);
        const float sx = fmaxf(P.inv_scale * ((float)x + 0.5f) - 0.5f, 0.f);
        const int h1 = (int)sy, w1 = (int)sx;
        const long long dh = h1 < P.lr_h - 1 ? P.ls_h : 0, dw = w1 < P.lr_w - 1 ? P.ls_w : 0;
        const float l1y = sy - (float)h1, l0y = 1.f - l1y, l1x = sx - (float)w1, l0x = 1.f - l1x;
        const float* p = P.lr + n * P.ls_n + h1 * P.ls_h + w1 * P.ls_w;
        float v[3][4];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float* pc = p + c * P.ls_c;
          v[c][0] = __ldg(pc);
          v[c][1] = __ldg(pc + dw);
          v[c][2] = __ldg(pc + dh);
          v[c][3] = __ldg(pc + dh + dw);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) up[c] = l0y * (l0x * v[c][0] + l1x * v[c][1]) + l1y * (l0x * v[c][2] + l1x * v[c][3]);
      }
      mbar_wait(bar_accf + 8 * team, (tl >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + team * ST_ACC;
      uint32_t a0[4], a1[4], a2[4];
      tmem_ld_32x4(taddr, a0);
      tmem_ld_32x4(taddr + ST_NPAD, a1);
      tmem_ld_32x4(taddr + 2 * ST_NPAD, a2);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acce + 8 * team);          // accumulator drained: tile tl + 2 may start
      if constexpr (SSE) {
        if (n != sse_n) {                                       // n is the same for the whole warp
          if (sse_n >= 0) sse_flush(P.out, sse_n, sse_acc, lane);
          sse_n = n;
          sse_acc = 0;
        }
        const long long off = n * P.out.s_n + (long long)y * P.out.s_y + (long long)x * P.out.s_x;
        const bool store = valid && P.out.p != nullptr;
        // at most 3 * 255^2 per lane and tile: 32 bits hold it, the running sum is 64-bit
        uint32_t e = 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float t = __uint_as_float(a0[c]) + __shfl_down_sync(0xffffffffu, __uint_as_float(a1[c]), 1) +
                          __shfl_down_sync(0xffffffffu, __uint_as_float(a2[c]), 2);
          // RgbOut's codes, expression for expression
          const int code = __float2int_rn(fminf(fmaxf(255.f * ((t + bias[c]) + up[c]), 0.f), 255.f));
          if (store) P.out.p[off + c * P.out.s_c] = (uint8_t)code;
          const int d = code - (int)gt[c];
          e += (uint32_t)(d * d);
        }
        if (valid) sse_acc += e;
      } else if constexpr (!YUV) {
        T* op = P.out.p + n * P.out.s_n + (long long)y * P.out.s_y + (long long)x * P.out.s_x;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float t = __uint_as_float(a0[c]) + __shfl_down_sync(0xffffffffu, __uint_as_float(a1[c]), 1) +
                          __shfl_down_sync(0xffffffffu, __uint_as_float(a2[c]), 2);
          if constexpr (sizeof(T) == 1) {
            // the reference's visuals: clamp(sr * 255, 0, 255).round(), round half to even
            const float v = fminf(fmaxf(255.f * ((t + bias[c]) + up[c]), 0.f), 255.f);
            if (valid) op[c * P.out.s_c] = (uint8_t)__float2int_rn(v);
          } else {
            // the same at M = 2^bits - 1
            const float v = fminf(fmaxf(P.out.m * ((t + bias[c]) + up[c]), 0.f), P.out.m);
            if (valid) op[c * P.out.s_c] = (uint16_t)__float2int_rn(v);
          }
        }
      } else {
        // rgb_to_yuv420 of eavsr_b200/yuv.py in its fp32 order of operations (no contraction into FMAs)
        const Out& o = P.out;
        float v[3], s[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float t = __uint_as_float(a0[c]) + __shfl_down_sync(0xffffffffu, __uint_as_float(a1[c]), 1) +
                          __shfl_down_sync(0xffffffffu, __uint_as_float(a2[c]), 2);
          v[c] = fminf(fmaxf((t + bias[c]) + up[c], 0.f), 1.f);
          s[c] = __fadd_rn(v[c], __shfl_xor_sync(0xffffffffu, v[c], 1));      // p(x) + p(x + 1), x even
        }
        const float yc = __fadd_rn(__fadd_rn(__fmul_rn(o.kr, v[0]), __fmul_rn(o.kg, v[1])), __fmul_rn(o.kb, v[2]));
        if constexpr (sizeof(T) == 1) {
          if (valid)
            o.y.p[n * o.y.s_n + (long long)y * o.y.s_y + (long long)x * o.y.s_x] =
                (uint8_t)__float2int_rn(__fadd_rn(__fmul_rn(219.f, yc), 16.f));
        } else {
          if (valid)
            o.y.p[n * o.y.s_n + (long long)y * o.y.s_y + (long long)x * o.y.s_x] =
                (uint16_t)(__float2int_rn(__fadd_rn(__fmul_rn(o.ys, yc), o.yo)) << o.shift);
        }
        // tile origins are even and out_h, out_w are even: a 2x2 block is lanes (2k, 2k + 1) of warps q, q + 1 of
        // one team, and it is valid as a whole.  The slot is double-buffered over the team's tiles, so the write
        // for its next tile lands in the other buffer, and the one after that waits at the barrier for this read
        float* xch = reinterpret_cast<float*>(smem + StSmem::TOTAL) + ((team * 2 + (q >> 1)) * 2 + ((tl >> 1) & 1)) * 48;
        const int bar_id = 1 + team * 2 + (q >> 1);
        if (q & 1) {
          if (!(lane & 1))
#pragma unroll
            for (int c = 0; c < 3; ++c) xch[c * 16 + (lane >> 1)] = s[c];
          asm volatile("bar.sync %0, 64;\n" ::"r"(bar_id) : "memory");
        } else {
          asm volatile("bar.sync %0, 64;\n" ::"r"(bar_id) : "memory");
          if (valid && !(lane & 1)) {
            float m[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) m[c] = __fmul_rn(__fadd_rn(s[c], xch[c * 16 + (lane >> 1)]), 0.25f);
            const float ym = __fadd_rn(__fadd_rn(__fmul_rn(o.kr, m[0]), __fmul_rn(o.kg, m[1])), __fmul_rn(o.kb, m[2]));
            const long long yh = y >> 1, xh = x >> 1;
            if constexpr (sizeof(T) == 1) {
              o.u.p[n * o.u.s_n + yh * o.u.s_y + xh * o.u.s_x] =
                  (uint8_t)__float2int_rn(__fadd_rn(__fmul_rn(__fsub_rn(m[2], ym), o.cu), 128.f));
              o.v.p[n * o.v.s_n + yh * o.v.s_y + xh * o.v.s_x] =
                  (uint8_t)__float2int_rn(__fadd_rn(__fmul_rn(__fsub_rn(m[0], ym), o.cv), 128.f));
            } else {
              o.u.p[n * o.u.s_n + yh * o.u.s_y + xh * o.u.s_x] =
                  (uint16_t)(__float2int_rn(__fadd_rn(__fmul_rn(__fsub_rn(m[2], ym), o.cu), o.co)) << o.shift);
              o.v.p[n * o.v.s_n + yh * o.v.s_y + xh * o.v.s_x] =
                  (uint16_t)(__float2int_rn(__fadd_rn(__fmul_rn(__fsub_rn(m[0], ym), o.cv), o.co)) << o.shift);
            }
          }
        }
      }
    }
    if constexpr (SSE) {
      if (sse_n >= 0) sse_flush(P.out, sse_n, sse_acc, lane);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<ST_TMEM>(tmem_d);
}

// checks, tensor map and launch shared by the RGB, the 4:2:0 and the squared-error entry points
template <class Out>
int sr_tail_launch(const char* who, const void* x, const int64_t x_strides[4], const void* packed_weight,
                   const void* bias, const float* lr, const int64_t lr_strides[4], const Out& out, int n, int c, int h,
                   int w, int scale, int out_h, int out_w, int dtype, void* stream) {
  EAVSR_REQUIRE(c == ST_CH, "%s: the feature map must have 64 channels (got %d)", who, c);
  EAVSR_REQUIRE(scale == 2 || scale == 4, "%s: scale must be 2 or 4 (got %d)", who, scale);
  EAVSR_REQUIRE(n > 0 && h > 0 && w > 0 && h % scale == 0 && w % scale == 0,
                "%s: bad map %dx%dx%d for scale %d", who, n, h, w, scale);
  EAVSR_REQUIRE(out_h > 0 && out_w > 0 && out_h <= h && out_w <= w,
                "%s: crop %dx%d outside the %dx%d map", who, out_h, out_w, h, w);
  EAVSR_REQUIRE(x_strides[0] == (int64_t)h * w * ST_CH && x_strides[1] == 1 && x_strides[2] == (int64_t)w * ST_CH &&
                    x_strides[3] == ST_CH,
                "%s: x must be dense channels_last (NHWC)", who);
  EAVSR_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(packed_weight)) & 15u) == 0,
                "%s: x and the packed weights must be 16-byte aligned", who);
  if (dtype != EAVSR_BF16) {
    set_error("%s: only bf16 features are implemented (dtype %d)", who, dtype);
    return EAVSR_ERR_UNSUPPORTED;
  }
  const int tiles_x = ceil_div(out_w, ST_TC), tiles_y = ceil_div(out_h, ST_TR);
  const long long total = (long long)tiles_x * tiles_y * n;
  EAVSR_REQUIRE(total < (1ll << 31), "%s: too many tiles", who);
  static thread_local TailParams<Out> P;
  const unsigned long long dims[4] = {ST_CH, (unsigned long long)w, (unsigned long long)h, (unsigned long long)n};
  const unsigned long long str[3] = {ST_CH * 2ull, (unsigned long long)w * ST_CH * 2,
                                     (unsigned long long)h * w * ST_CH * 2};
  const unsigned box[4] = {ST_CH, ST_PW, ST_TR + 2, 1};
  if (!encode_tensor_map(&P.tm, EAVSR_BF16, 4, x, dims, str, box, 3 /* CU_TENSOR_MAP_SWIZZLE_128B */)) {
    set_error("%s: the tensor map of x was rejected", who);
    return EAVSR_ERR_UNSUPPORTED;
  }
  P.wpacked = (const uint8_t*)packed_weight;
  P.bias = (const __nv_bfloat16*)bias;
  P.lr = lr;
  P.ls_n = lr_strides[0]; P.ls_c = lr_strides[1]; P.ls_h = lr_strides[2]; P.ls_w = lr_strides[3];
  P.out = out;
  P.out_h = out_h; P.out_w = out_w; P.lr_h = h / scale; P.lr_w = w / scale;
  P.tiles_x = tiles_x; P.tiles_per_img = tiles_x * tiles_y; P.total_tiles = (int)total;
  P.inv_scale = 1.f / (float)scale;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaError_t e = cudaFuncSetAttribute(sr_tail_u8_kernel<Out>, cudaFuncAttributeMaxDynamicSharedMemorySize, st_dyn<Out>());
  if (e != cudaSuccess) { set_error("%s: smem attr: %s", who, cudaGetErrorString(e)); return EAVSR_ERR_CUDA; }
  sr_tail_u8_kernel<Out><<<(int)(total < sms ? total : sms), ST_THREADS, st_dyn<Out>(), (cudaStream_t)stream>>>(P);
  return check_launch(who);
}

}  // namespace
}  // namespace eavsr

using namespace eavsr;

extern "C" size_t eavsr_sr_tail_packed_weight_bytes(void) { return (size_t)9 * ST_BTAP; }

extern "C" int eavsr_sr_tail_pack_weight(const void* weight, void* packed, int cin, int cout, int dtype, void* stream) {
  EAVSR_REQUIRE(weight && packed, "sr_tail_pack_weight: null pointer");
  EAVSR_REQUIRE(cin == ST_CH && cout == 3, "sr_tail_pack_weight: only 64 -> 3 is implemented (got %d -> %d)", cin, cout);
  if (dtype != EAVSR_BF16) {
    set_error("sr_tail_pack_weight: only bf16 weights are implemented (dtype %d)", dtype);
    return EAVSR_ERR_UNSUPPORTED;
  }
  sr_tail_pack_weight_kernel<<<(9 * ST_NPAD * ST_CH + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)weight, (uint8_t*)packed);
  return check_launch("sr_tail_pack_weight");
}

extern "C" int eavsr_sr_tail_u8_forward(const void* x, const int64_t x_strides[4], const void* packed_weight,
                                        const void* bias, const float* lr, const int64_t lr_strides[4], void* out,
                                        const int64_t out_strides[4], int n, int c, int h, int w, int scale, int out_h,
                                        int out_w, int dtype, void* stream) {
  EAVSR_REQUIRE(x && x_strides && packed_weight && lr && lr_strides && out && out_strides,
                "sr_tail_u8_forward: null pointer");
  const RgbOut o = {(uint8_t*)out, out_strides[0], out_strides[1], out_strides[2], out_strides[3]};
  return sr_tail_launch("sr_tail_u8_forward", x, x_strides, packed_weight, bias, lr, lr_strides, o, n, c, h, w, scale,
                        out_h, out_w, dtype, stream);
}

extern "C" int eavsr_sr_tail_yuv420_forward(const void* x, const int64_t x_strides[4], const void* packed_weight,
                                            const void* bias, const float* lr, const int64_t lr_strides[4],
                                            void* out_y, const int64_t y_strides[4], void* out_u,
                                            const int64_t u_strides[4], void* out_v, const int64_t v_strides[4], int n,
                                            int c, int h, int w, int scale, int out_h, int out_w, float kr, float kb,
                                            int dtype, void* stream) {
  EAVSR_REQUIRE(x && x_strides && packed_weight && lr && lr_strides && out_y && y_strides && out_u && u_strides &&
                    out_v && v_strides,
                "sr_tail_yuv420_forward: null pointer");
  EAVSR_REQUIRE(out_h % 2 == 0 && out_w % 2 == 0, "sr_tail_yuv420_forward: 4:2:0 needs an even crop (got %dx%d)",
                out_h, out_w);
  EAVSR_REQUIRE(kr > 0.f && kb > 0.f && kr + kb < 1.f, "sr_tail_yuv420_forward: bad matrix (kr %g, kb %g)", kr, kb);
  Yuv420Out o;
  o.y = {(uint8_t*)out_y, y_strides[0], y_strides[2], y_strides[3]};
  o.u = {(uint8_t*)out_u, u_strides[0], u_strides[2], u_strides[3]};
  o.v = {(uint8_t*)out_v, v_strides[0], v_strides[2], v_strides[3]};
  // the fp32 coefficients of eavsr_b200/yuv.py, in its order
  o.kr = kr; o.kb = kb; o.kg = (1.f - kr) - kb;
  o.cu = 112.f / (1.f - kb); o.cv = 112.f / (1.f - kr);
  return sr_tail_launch("sr_tail_yuv420_forward", x, x_strides, packed_weight, bias, lr, lr_strides, o, n, c, h, w,
                        scale, out_h, out_w, dtype, stream);
}

static bool hbd_bits_ok(int bits) { return bits == 10 || bits == 12 || bits == 16; }

extern "C" int eavsr_sr_tail_u16_forward(const void* x, const int64_t x_strides[4], const void* packed_weight,
                                         const void* bias, const float* lr, const int64_t lr_strides[4], void* out,
                                         const int64_t out_strides[4], int n, int c, int h, int w, int scale,
                                         int out_h, int out_w, int bits, int dtype, void* stream) {
  EAVSR_REQUIRE(x && x_strides && packed_weight && lr && lr_strides && out && out_strides,
                "sr_tail_u16_forward: null pointer");
  EAVSR_REQUIRE(hbd_bits_ok(bits), "sr_tail_u16_forward: bits must be 10, 12 or 16 (got %d)", bits);
  EAVSR_REQUIRE((reinterpret_cast<uintptr_t>(out) & 1u) == 0, "sr_tail_u16_forward: out must be 2-byte aligned");
  const Rgb16Out o = {(uint16_t*)out, out_strides[0], out_strides[1], out_strides[2], out_strides[3],
                      (float)((1 << bits) - 1)};
  return sr_tail_launch("sr_tail_u16_forward", x, x_strides, packed_weight, bias, lr, lr_strides, o, n, c, h, w,
                        scale, out_h, out_w, dtype, stream);
}

extern "C" int eavsr_sr_tail_yuv420_u16_forward(const void* x, const int64_t x_strides[4], const void* packed_weight,
                                                const void* bias, const float* lr, const int64_t lr_strides[4],
                                                void* out_y, const int64_t y_strides[4], void* out_u,
                                                const int64_t u_strides[4], void* out_v, const int64_t v_strides[4],
                                                int n, int c, int h, int w, int scale, int out_h, int out_w, float kr,
                                                float kb, int bits, int shift, int dtype, void* stream) {
  EAVSR_REQUIRE(x && x_strides && packed_weight && lr && lr_strides && out_y && y_strides && out_u && u_strides &&
                    out_v && v_strides,
                "sr_tail_yuv420_u16_forward: null pointer");
  EAVSR_REQUIRE(hbd_bits_ok(bits), "sr_tail_yuv420_u16_forward: bits must be 10, 12 or 16 (got %d)", bits);
  EAVSR_REQUIRE(shift == 0 || shift == 16 - bits, "sr_tail_yuv420_u16_forward: shift must be 0 or %d (got %d)",
                16 - bits, shift);
  EAVSR_REQUIRE(((reinterpret_cast<uintptr_t>(out_y) | reinterpret_cast<uintptr_t>(out_u) |
                  reinterpret_cast<uintptr_t>(out_v)) & 1u) == 0,
                "sr_tail_yuv420_u16_forward: the planes must be 2-byte aligned");
  EAVSR_REQUIRE(out_h % 2 == 0 && out_w % 2 == 0,
                "sr_tail_yuv420_u16_forward: 4:2:0 needs an even crop (got %dx%d)", out_h, out_w);
  EAVSR_REQUIRE(kr > 0.f && kb > 0.f && kr + kb < 1.f, "sr_tail_yuv420_u16_forward: bad matrix (kr %g, kb %g)", kr,
                kb);
  Yuv420Out16 o;
  o.y = {(uint16_t*)out_y, y_strides[0], y_strides[2], y_strides[3]};
  o.u = {(uint16_t*)out_u, u_strides[0], u_strides[2], u_strides[3]};
  o.v = {(uint16_t*)out_v, v_strides[0], v_strides[2], v_strides[3]};
  // the fp32 coefficients of eavsr_b200/yuv.py at k = 2^(bits - 8); k is a power of two, so k * cu is exact
  const float k = (float)(1 << (bits - 8));
  o.kr = kr; o.kb = kb; o.kg = (1.f - kr) - kb;
  o.cu = k * (112.f / (1.f - kb)); o.cv = k * (112.f / (1.f - kr));
  o.ys = 219.f * k; o.yo = 16.f * k; o.co = 128.f * k;
  o.shift = shift;
  return sr_tail_launch("sr_tail_yuv420_u16_forward", x, x_strides, packed_weight, bias, lr, lr_strides, o, n, c, h,
                        w, scale, out_h, out_w, dtype, stream);
}

extern "C" int eavsr_sr_tail_u8_sse_forward(const void* x, const int64_t x_strides[4], const void* packed_weight,
                                            const void* bias, const float* lr, const int64_t lr_strides[4],
                                            const void* gt, const int64_t gt_strides[4], void* out,
                                            const int64_t out_strides[4], unsigned long long* sse,
                                            long long sse_stride, int n, int c, int h, int w, int scale, int out_h,
                                            int out_w, int dtype, void* stream) {
  EAVSR_REQUIRE(x && x_strides && packed_weight && lr && lr_strides && gt && gt_strides && sse && (!out || out_strides),
                "sr_tail_u8_sse_forward: null pointer");
  EAVSR_REQUIRE((reinterpret_cast<uintptr_t>(sse) & 7u) == 0, "sr_tail_u8_sse_forward: sse must be 8-byte aligned");
  RgbSse o;
  o.gt = (const uint8_t*)gt;
  o.g_n = gt_strides[0]; o.g_y = gt_strides[1]; o.g_x = gt_strides[2]; o.g_c = gt_strides[3];
  o.p = (uint8_t*)out;
  o.s_n = out ? out_strides[0] : 0; o.s_y = out ? out_strides[1] : 0;
  o.s_x = out ? out_strides[2] : 0; o.s_c = out ? out_strides[3] : 0;
  o.sse = sse;
  o.sse_s = sse_stride;
  return sr_tail_launch("sr_tail_u8_sse_forward", x, x_strides, packed_weight, bias, lr, lr_strides, o, n, c, h, w,
                        scale, out_h, out_w, dtype, stream);
}
