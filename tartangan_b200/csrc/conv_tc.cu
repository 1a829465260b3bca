// Tensor-core implicit-GEMM convolution for sm_100a: tcgen05.mma (bf16 x bf16 -> fp32 in TMEM).
// Replaces aten::convolution / convolution_backward for every nn.Conv2d of the residual blocks
// (reference models/blocks/generator.py:41,44,52; discriminator.py:63,66,78) whose channel
// counts are multiples of 16.  NHWC bf16 activations, k in {1,3}, stride 1, pad k/2.
//
// Tiling: one CTA = 16 rows x 8 cols = 128 output pixels of one image (UMMA M = 128).
// The input halo tile (18 x 10 pixels) is staged ONCE in shared memory as 16-byte units
// [channel/8][halo pixel][8 channels] — the SWIZZLE_NONE canonical layout — so that each of the
// 9 filter taps is just a shifted descriptor start address (no im2col copies, no re-reads):
//   fprop/dgrad: A = pixels x channels (K-major),  B = packed weights (K-major),  N = Cout
//   wgrad      : A = gy^T   (MN-major, K = pixels), B = shifted x (MN-major),     N = Cin
// Zero padding = zero-filled halo.
// The epilogue reads the fp32 accumulator from TMEM (tcgen05.ld 32x32b), adds the bias and
// writes NHWC rows (one thread = one pixel = Cout contiguous channels).
#include "tc_common.cuh"

#define TC_TH 16
#define TC_TW 8

// compile-time loop: f(std::integral_constant<int, 0>) ... f(std::integral_constant<int, N-1>)
#include <type_traits>
#include <utility>
template <int... Is, typename F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, Is...>, F&& f) { (f(std::integral_constant<int, Is>{}), ...); }
template <int N, typename F>
__device__ __forceinline__ void static_for(F&& f) { static_for_impl(std::make_integer_sequence<int, N>{}, f); }

// ------------------------------------------------------------------ weight packing
// mode 0 (fprop): wp[tap][ci/8][co][ci%8]            = w[co][ci][ky][kx]        (B: N=co, K=ci)
// mode 1 (dgrad): wp[tap'][co/8][ci][co%8]           = w[co][ci][k-1-ky][k-1-kx] (B: N=ci, K=co)
__global__ void pack_weight_tc_kernel(const float* __restrict__ w, bf16* __restrict__ wp, int Cout, int Cin, int k, int mode) {
  int total = Cout * Cin * k * k;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int kx = i % k, ky = (i / k) % k, ci = (i / (k * k)) % Cin, co = i / (k * k * Cin);
    bf16 v = __float2bfloat16_rn(w[i]);
    if (mode == 0) {
      int tap = ky * k + kx;
      wp[(((long long)tap * (Cin / 8) + ci / 8) * Cout + co) * 8 + (ci % 8)] = v;
    } else {
      int tap = (k - 1 - ky) * k + (k - 1 - kx);
      wp[(((long long)tap * (Cout / 8) + co / 8) * Cin + ci) * 8 + (co % 8)] = v;
    }
  }
}
extern "C" size_t ttg_pack_weight_tc_bytes(int Cout, int Cin, int ksize) { return (size_t)Cout * Cin * ksize * ksize * 2; }
extern "C" int ttg_pack_weight_tc(const float* w, void* wp, int Cout, int Cin, int ksize, int mode, void* stream) {
  TTG_REQUIRE(Cout % 16 == 0 && Cin % 16 == 0, "pack_weight_tc: channels must be multiples of 16 (%d,%d)", Cout, Cin);
  int total = Cout * Cin * ksize * ksize;
  pack_weight_tc_kernel<<<ttg_grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w, (bf16*)wp, Cout, Cin, ksize, mode);
  TTG_CHECK_LAUNCH("pack_weight_tc");
  return TTG_OK;
}

// ------------------------------------------------------------------ staging of an activation tile
// Writes the [halo row][C/8][halo col] x 16B image of the (TC_TH+2h) x (TC_TW+2h) halo tile at (y0-h, x0-h):
// unit index = (hy * C/8 + c8) * WH + hx.  Rows of 8 pixels are contiguous (one 8 x 16 B core matrix), the next
// channel group is WH units away and the next halo row C/8 * WH units away, so both the vertical filter taps
// and the channel groups are reachable with ONE uniform descriptor stride (used by wgrad to fold ky into N).
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int HALO>
__device__ __forceinline__ bool tile_src(int u, int c8n, int n, int y0, int x0, int H, int W, int C,
                                         long long& src_elem, uint32_t& dst_unit) {
  constexpr int WH = TC_TW + 2 * HALO;
  const int c8 = u % c8n, pix = u / c8n;
  const int hy = pix / WH, hx = pix - hy * WH;
  const int gy = y0 + hy - HALO, gx = x0 + hx - HALO;
  dst_unit = (uint32_t)((hy * c8n + c8) * WH + hx);
  const bool ok = gy >= 0 && gy < H && gx >= 0 && gx < W;
  src_elem = ok ? ((((long long)n * H + gy) * W + gx) * C + c8 * 8) : 0;
  return ok;
}

// asynchronous version (LDGSTS, zero-fill outside the image); caller waits with cp_async_wait_all()
template <int HALO>
__device__ __forceinline__ void stage_tile_async(uint8_t* sA, const bf16* __restrict__ x, int n, int y0, int x0, int H,
                                                 int W, int C, int nthr) {
  constexpr int HP = (TC_TW + 2 * HALO) * (TC_TH + 2 * HALO);
  const int c8n = C >> 3;
  const uint32_t base = smem_u32(sA);
  for (int u = threadIdx.x; u < HP * c8n; u += nthr) {
    long long se; uint32_t du;
    const bool ok = tile_src<HALO>(u, c8n, n, y0, x0, H, W, C, se, du);
    cp_async16(base + du * 16, x + se, ok ? 16u : 0u);
  }
}

// register version, 4 loads in flight per thread
template <int HALO>
__device__ __forceinline__ void stage_tile(uint8_t* sA, const bf16* __restrict__ x, int n, int y0, int x0, int H, int W,
                                           int C, int nthr) {
  constexpr int HP = (TC_TW + 2 * HALO) * (TC_TH + 2 * HALO);
  const int c8n = C >> 3;
  const int total = HP * c8n;
  for (int base = 0; base < total; base += 4 * nthr) {
    uint4 v[4]; uint32_t du[4]; bool live[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int u = base + j * nthr + threadIdx.x;
      live[j] = u < total;
      v[j] = make_uint4(0u, 0u, 0u, 0u);
      du[j] = 0;
      if (live[j]) {
        long long se;
        if (tile_src<HALO>(u, c8n, n, y0, x0, H, W, C, se, du[j])) v[j] = __ldg(reinterpret_cast<const uint4*>(x + se));
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (live[j]) *reinterpret_cast<uint4*>(sA + (size_t)du[j] * 16) = v[j];
  }
}

// Channel-padded variants for the RGB layers (Cin == 3 first D conv, Cout == 3 image gradients / last G conv):
// the tensors in HBM keep their real channel count, the shared-memory / weight images are padded to 16 with
// zeros, so these layers run on the same tensor-core kernels.
__global__ void pack_weight_tc_pad_kernel(const float* __restrict__ w, bf16* __restrict__ wp, int Cout, int Cin, int CoutP,
                                          int CinP, int k, int mode) {
  int total = Cout * Cin * k * k;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int kx = i % k, ky = (i / k) % k, ci = (i / (k * k)) % Cin, co = i / (k * k * Cin);
    bf16 v = __float2bfloat16_rn(w[i]);
    if (mode == 0) {
      int tap = ky * k + kx;
      wp[(((long long)tap * (CinP / 8) + ci / 8) * CoutP + co) * 8 + (ci % 8)] = v;
    } else {
      int tap = (k - 1 - ky) * k + (k - 1 - kx);
      wp[(((long long)tap * (CoutP / 8) + co / 8) * CinP + ci) * 8 + (co % 8)] = v;
    }
  }
}
extern "C" int ttg_pack_weight_tc_pad(const float* w, void* wp, int Cout, int Cin, int CoutP, int CinP, int ksize, int mode,
                                      void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(CoutP % 16 == 0 && CinP % 16 == 0 && Cout <= CoutP && Cin <= CinP, "pack_weight_tc_pad: bad padding");
  cudaMemsetAsync(wp, 0, (size_t)CoutP * CinP * ksize * ksize * 2, st);
  int total = Cout * Cin * ksize * ksize;
  pack_weight_tc_pad_kernel<<<ttg_grid_for(total, 256), 256, 0, st>>>(w, (bf16*)wp, Cout, Cin, CoutP, CinP, ksize, mode);
  TTG_CHECK_LAUNCH("pack_weight_tc_pad");
  return TTG_OK;
}

// stage a tile of a tensor with c_real (<= 8) channels into the C-channel (padded) shared-memory image
template <int HALO>
__device__ __forceinline__ void stage_tile_pad(uint8_t* sA, const bf16* __restrict__ x, int n, int y0, int x0, int H, int W,
                                               int C, int c_real, int nthr) {
  constexpr int WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO, HP = WH * HH;
  const int c8n = C >> 3;
  for (int pix = threadIdx.x; pix < HP; pix += nthr) {
    const int hy = pix / WH, hx = pix - hy * WH;
    const int gy = y0 + hy - HALO, gx = x0 + hx - HALO;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
      const unsigned short* src = reinterpret_cast<const unsigned short*>(x) + (((long long)n * H + gy) * W + gx) * c_real;
      for (int c = 0; c < c_real; ++c) w[c >> 1] |= (uint32_t)src[c] << (16 * (c & 1));
    }
    uint8_t* d = sA + (size_t)((hy * c8n) * WH + hx) * 16;
    *reinterpret_cast<uint4*>(d) = make_uint4(w[0], w[1], w[2], w[3]);
    for (int c8 = 1; c8 < c8n; ++c8) *reinterpret_cast<uint4*>(d + (size_t)c8 * WH * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
}

// Fast staging for the persistent kernel (units per halo row <= 128): every thread owns one fixed
// (column, channel-group) position of the halo row and walks down the rows, so all div/mod work is
// done once per kernel and a 16-byte unit costs ~10 instructions instead of ~70.
struct RowStager {
  int q_hx, q_c8, r0, rpp, active;     // fixed per thread
};
template <int HALO>
__device__ __forceinline__ RowStager make_row_stager(int C, int tid) {
  constexpr int WH = TC_TW + 2 * HALO;
  const int c8n = C >> 3, upr = WH * c8n;
  RowStager rs;
  rs.rpp = 128 / upr;
  const int q = tid % upr;
  rs.r0 = tid / upr;
  rs.active = tid < upr * rs.rpp;
  rs.q_hx = q / c8n;
  rs.q_c8 = q - rs.q_hx * c8n;
  return rs;
}
template <int HALO>
__device__ __forceinline__ void stage_rows(const RowStager& rs, uint8_t* sA, const bf16* __restrict__ x, int n, int y0,
                                           int x0, int H, int W, int C) {
  constexpr int WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO;
  if (!rs.active) return;
  const int gx = x0 + rs.q_hx - HALO;
  const bool xok = gx >= 0 && gx < W;
  const bf16* col = x + ((long long)n * H * W + gx) * C + rs.q_c8 * 8;
  const int c8n = C >> 3;
  uint32_t dst = smem_u32(sA) + (uint32_t)((rs.r0 * c8n + rs.q_c8) * WH + rs.q_hx) * 16;
  const uint32_t dstep = (uint32_t)(rs.rpp * c8n * WH) * 16;
  for (int r = rs.r0; r < HH; r += rs.rpp, dst += dstep) {
    const int gy = y0 + r - HALO;
    const bool ok = xok && gy >= 0 && gy < H;
    cp_async16(dst, ok ? col + (long long)gy * W * C : x, ok ? 16u : 0u);
  }
}

// ------------------------------------------------------------------ fprop / dgrad, persistent (weights resident)
// For layers whose packed filter fits in shared memory (C <= 64): one CTA loops over tiles with the
// filter loaded once, two activation buffers and two TMEM accumulators, so that per tile the
// cp.async loads of tile i+1, the MMAs of tile i and the epilogue of tile i-1 overlap.
template <int HALO>
__device__ __forceinline__ void conv_tc_epilogue(uint32_t tacc, int warp, int tid, int n, int y0, int x0, int H, int W,
                                                 int Cout, const float* __restrict__ bias, void* __restrict__ y, int out_f32,
                                                 int cout_real = 0) {
  if (cout_real && cout_real != Cout) {           // padded output channels: scalar stores of the real ones
    const int gy = y0 + (tid >> 3), gx = x0 + (tid & 7);
    const bool valid = gy < H && gx < W;
    const long long opix = ((long long)n * H + gy) * W + gx;
    uint32_t r[16];
    tmem_ld16(tacc + ((uint32_t)(warp * 32) << 16), r);
    tmem_ld_wait();
    if (valid) {
      for (int j = 0; j < cout_real; ++j) {
        const float f = __uint_as_float(r[j]) + (bias ? bias[j] : 0.f);
        if (out_f32) reinterpret_cast<float*>(y)[opix * cout_real + j] = f;
        else reinterpret_cast<bf16*>(y)[opix * cout_real + j] = __float2bfloat16_rn(f);
      }
    }
    return;
  }
  const int gy = y0 + (tid >> 3), gx = x0 + (tid & 7);
  const bool valid = gy < H && gx < W;
  const long long opix = ((long long)n * H + gy) * W + gx;
  for (int c0 = 0; c0 < Cout; c0 += 16) {
    uint32_t r[16];
    tmem_ld16(tacc + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, r);
    tmem_ld_wait();
    if (valid) {
      float f[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(r[j]) + (bias ? bias[c0 + j] : 0.f);
      if (out_f32) {
        float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + opix * Cout + c0);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
      } else {
        uint4 o[2];
        __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) h[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
        uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(y) + opix * Cout + c0);
        dst[0] = o[0]; dst[1] = o[1];
      }
    }
  }
}

// Coalescing epilogue (bf16 NHWC output, Cout a multiple of 16): every warp stages its 32 pixels x (<= 64 channels)
// in a private, padded shared-memory strip and writes it back with consecutive lanes on consecutive 16-byte units,
// so a store instruction covers whole 32-byte sectors / 128-byte lines instead of 16 B out of every pixel.
//   strip pitch = chunk bytes + 16  ->  both the pixel-major writes and the unit-major reads are conflict free.
#define TC_EPI_CHUNK 64
static inline int tc_epi_strip_bytes(int Cout) { return 4 * 32 * ((Cout < TC_EPI_CHUNK ? Cout : TC_EPI_CHUNK) * 2 + 16); }
// strips + per-CTA BatchNorm statistics accumulators (sum, sum of squares: 2 x Cout floats)
static inline int tc_epi_bytes(int Cout) { return tc_epi_strip_bytes(Cout) + 2 * Cout * 4; }
__device__ __forceinline__ int tc_epi_strip_bytes_dev(int Cout) { return 4 * 32 * ((Cout < TC_EPI_CHUNK ? Cout : TC_EPI_CHUNK) * 2 + 16); }

// Sum of 16 per-lane values over the 32 lanes of a warp, for all 16 values at once (butterfly that halves the
// number of values a lane carries at every exchange: 8+4+2+1+1 shuffles instead of 16 x 5).  On return v[0] holds the
// warp total of value index ((lane>>4)&1)*8 + ((lane>>3)&1)*4 + ((lane>>2)&1)*2 + ((lane>>1)&1).
__device__ __forceinline__ void warp_reduce16(float (&v)[16], int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float keep = (lane & 16) ? v[j + 8] : v[j], send = (lane & 16) ? v[j] : v[j + 8];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float keep = (lane & 8) ? v[j + 4] : v[j], send = (lane & 8) ? v[j] : v[j + 4];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const float keep = (lane & 4) ? v[j + 2] : v[j], send = (lane & 4) ? v[j] : v[j + 2];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  {
    const float keep = (lane & 2) ? v[1] : v[0], send = (lane & 2) ? v[0] : v[1];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}
// `Cout` = channels stored per pixel (row pitch of y): the accumulator width, or 8 for the 8-channel staging tensors
// of the RGB layers (accumulator columns 8..15 are padding and are dropped).
// Per-lane statistics accumulators for layers whose pixels are one chunk wide (Cout <= 64, Cout / 8 a power of two):
// in the write-back loop a lane always handles the same 8-channel group (u % (Cout/8) == lane % (Cout/8)), so it sums
// the units it is storing anyway and the cross-lane reduction happens ONCE per CTA (epi_stats_flush), not per tile.
struct EpiStats { float s[8], q[8]; };
__device__ __forceinline__ bool epi_stats_in_regs(int Cout) { const int u = Cout >> 3; return Cout <= TC_EPI_CHUNK && (u & (u - 1)) == 0; }
__device__ __forceinline__ void epi_stats_flush(EpiStats& e, int lane, int Cout, float* s_stats) {
  const int up = Cout >> 3, j = lane % up;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    float a = e.s[k], b = e.q[k];
    for (int o = 16; o >= up; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    if (lane < up) { atomicAdd(&s_stats[j * 8 + k], a); atomicAdd(&s_stats[Cout + j * 8 + k], b); }
  }
}
// Lean write-back for the common case (bf16 NHWC output, compile-time Cout in {16, 32, 64}, tile completely inside
// the image): everything that the generic routine below derives at run time (chunking, swizzle shifts, bounds) is a
// constant here.  The small-channel layers are bound by the instruction count per 128-pixel tile (round 2, ncu:
// ~1100 warp instructions per tile in the generic epilogue, issue slots 67 % busy at 2.6 TB/s), not by HBM.
template <int COUT, bool STATS>
__device__ __forceinline__ void conv_tc_epilogue_lean(uint32_t tacc, uint8_t* sE, int warp, int lane, long long pix0, int W,
                                                      const float* __restrict__ bias, bf16* __restrict__ y, EpiStats* est) {
  constexpr int UPP = COUT / 8, LOG = UPP == 2 ? 1 : UPP == 4 ? 2 : 3, FSH = 3 - LOG, PITCH = COUT * 2;
  const uint32_t strip = smem_u32(sE + (size_t)warp * 32 * (PITCH + 16));
  const int key = (lane >> FSH) & (UPP - 1);
  const uint32_t mine = strip + (uint32_t)(lane * PITCH);
#pragma unroll
  for (int c1 = 0; c1 < COUT; c1 += 16) {
    uint32_t r[16];
    tmem_ld16(tacc + ((uint32_t)(warp * 32) << 16) + (uint32_t)c1, r);
    tmem_ld_wait();
    if (bias) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + c1) + q);
        r[4 * q] = __float_as_uint(__uint_as_float(r[4 * q]) + b4.x);
        r[4 * q + 1] = __float_as_uint(__uint_as_float(r[4 * q + 1]) + b4.y);
        r[4 * q + 2] = __float_as_uint(__uint_as_float(r[4 * q + 2]) + b4.z);
        r[4 * q + 3] = __float_as_uint(__uint_as_float(r[4 * q + 3]) + b4.w);
      }
    }
    uint32_t o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
      o[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    const int u0 = c1 >> 3;
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(mine + (uint32_t)((u0 ^ key) << 4)), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(mine + (uint32_t)(((u0 + 1) ^ key) << 4)), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < UPP; ++i) {
    const int u = lane + 32 * i, p = u >> LOG, j = u & (UPP - 1);      // j == lane & (UPP - 1): a lane always owns the same channel group
    const int slot = j ^ ((p >> FSH) & (UPP - 1));
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "r"(strip + (uint32_t)(p * PITCH + (slot << 4))));
    *reinterpret_cast<uint4*>(y + (pix0 + (long long)(warp * 4 + (p >> 3)) * W + (p & 7)) * COUT + j * 8) = v;
    if constexpr (STATS) {
      const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float f0 = __uint_as_float(w4[k] << 16), f1 = __uint_as_float(w4[k] & 0xffff0000u);
        est->s[2 * k] += f0; est->q[2 * k] += f0 * f0;
        est->s[2 * k + 1] += f1; est->q[2 * k + 1] += f1 * f1;
      }
    }
  }
  __syncwarp();
}
__device__ __forceinline__ void conv_tc_epilogue_coalesced(uint32_t tacc, uint8_t* sE, int warp, int lane, int n, int y0, int x0,
                                                           int H, int W, int Cout, const float* __restrict__ bias,
                                                           bf16* __restrict__ y, float* s_stats = nullptr,
                                                           EpiStats* est = nullptr) {
  if (y0 + TC_TH <= H && x0 + TC_TW <= W && (s_stats == nullptr || est != nullptr) && (Cout == 16 || Cout == 32 || Cout == 64)) {
    const long long pix0 = ((long long)n * H + y0) * W + x0;
    if (est) {
      if (Cout == 16) conv_tc_epilogue_lean<16, true>(tacc, sE, warp, lane, pix0, W, bias, y, est);
      else if (Cout == 32) conv_tc_epilogue_lean<32, true>(tacc, sE, warp, lane, pix0, W, bias, y, est);
      else conv_tc_epilogue_lean<64, true>(tacc, sE, warp, lane, pix0, W, bias, y, est);
    } else {
      if (Cout == 16) conv_tc_epilogue_lean<16, false>(tacc, sE, warp, lane, pix0, W, bias, y, nullptr);
      else if (Cout == 32) conv_tc_epilogue_lean<32, false>(tacc, sE, warp, lane, pix0, W, bias, y, nullptr);
      else conv_tc_epilogue_lean<64, false>(tacc, sE, warp, lane, pix0, W, bias, y, nullptr);
    }
    return;
  }
  if (Cout == 8) {                       // one 16-byte unit per pixel: lanes are already on consecutive units
    uint32_t r[16];
    tmem_ld16(tacc + ((uint32_t)(warp * 32) << 16), r);
    tmem_ld_wait();
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float f0 = __uint_as_float(r[2 * j]), f1 = __uint_as_float(r[2 * j + 1]);
      if (bias) { f0 += bias[2 * j]; f1 += bias[2 * j + 1]; }
      __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);
      o[j] = *reinterpret_cast<uint32_t*>(&h);
    }
    const int gy = y0 + warp * 4 + (lane >> 3), gx = x0 + (lane & 7);
    if (gy < H && gx < W) *reinterpret_cast<uint4*>(y + (((long long)n * H + gy) * W + gx) * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    return;
  }
  const int cc = Cout < TC_EPI_CHUNK ? Cout : TC_EPI_CHUNK;     // channels per chunk (16, 32, 48 or 64)
  const int upp = cc >> 3;                                       // 16-byte units per pixel in a chunk
  // Strip layout: power-of-two `upp`: dense pixels, unit j of pixel p stored at slot j ^ ((p / (8/upp)) % upp) -- both the
  // pixel-major 16-byte writes (lane = pixel) and the unit-major reads (lane = unit) then touch 8 distinct 16-byte
  // bank groups per quarter warp.  Other widths (48 channels): padded pitch.
  const bool swz = (upp & (upp - 1)) == 0;
  const int pitch = swz ? cc * 2 : cc * 2 + 16;
  const int fsh = swz ? 3 - (__ffs(upp) - 1) : 0;                // log2(8 / upp)
  uint8_t* strip = sE + (size_t)warp * 32 * (cc * 2 + 16);
  const uint32_t strip_addr = smem_u32(strip);
  const int wkey = swz ? ((lane >> fsh) & (upp - 1)) : 0;        // this lane's pixel (= lane) swizzle key
  for (int c0 = 0; c0 < Cout; c0 += cc) {
    const int ccur = min(cc, Cout - c0);
    for (int c1 = 0; c1 < ccur; c1 += 16) {
      uint32_t r[16];
      tmem_ld16(tacc + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c0 + c1), r);
      tmem_ld_wait();
      uint32_t o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float f0 = __uint_as_float(r[2 * j]), f1 = __uint_as_float(r[2 * j + 1]);
        if (bias) { f0 += bias[c0 + c1 + 2 * j]; f1 += bias[c0 + c1 + 2 * j + 1]; }
        __nv_bfloat162 h = __floats2bfloat162_rn(f0, f1);
        o[j] = *reinterpret_cast<uint32_t*>(&h);
      }
      const int u0 = c1 >> 3;                                    // first of the two units written here
      const uint32_t d0 = strip_addr + (uint32_t)(lane * pitch + ((u0 ^ wkey) << 4));
      const uint32_t d1 = strip_addr + (uint32_t)(lane * pitch + (((u0 + 1) ^ wkey) << 4));
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(d0), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(d1), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
      if (s_stats && !est) {
        // BatchNorm statistics of the tensor being written (the bf16-rounded values, pixels inside the image only)
        const bool inside = (y0 + warp * 4 + (lane >> 3)) < H && (x0 + (lane & 7)) < W;
        float v[16], q[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[2 * j] = inside ? __uint_as_float(o[j] << 16) : 0.f;
          v[2 * j + 1] = inside ? __uint_as_float(o[j] & 0xffff0000u) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) q[j] = v[j] * v[j];
        warp_reduce16(v, lane);
        warp_reduce16(q, lane);
        const int ch = c0 + c1 + ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
        atomicAdd(&s_stats[(lane & 1) ? Cout + ch : ch], (lane & 1) ? q[0] : v[0]);
      }
    }
    __syncwarp();
    const int up_cur = ccur >> 3;
    const int units = 32 * up_cur;
    const int sh = (up_cur & (up_cur - 1)) == 0 ? __ffs(up_cur) - 1 : -1;
    for (int u = lane; u < units; u += 32) {
      const int p = sh >= 0 ? (u >> sh) : u / up_cur, j = u - p * up_cur;
      const int gy = y0 + warp * 4 + (p >> 3), gx = x0 + (p & 7);
      const int slot = swz ? (j ^ ((p >> fsh) & (upp - 1))) : j;
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                   : "r"(strip_addr + (uint32_t)(p * pitch + (slot << 4))));
      if (gy < H && gx < W) {
        *reinterpret_cast<uint4*>(y + (((long long)n * H + gy) * W + gx) * Cout + c0 + j * 8) = v;
        if (est) {
          const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float f0 = __uint_as_float(w4[k] << 16), f1 = __uint_as_float(w4[k] & 0xffff0000u);
            est->s[2 * k] += f0; est->q[2 * k] += f0 * f0;
            est->s[2 * k + 1] += f1; est->q[2 * k + 1] += f1 * f1;
          }
        }
      }
    }
    __syncwarp();
  }
  (void)upp;
}

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }


// Warp-specialised persistent kernel: warps 0-3 stage tiles (cp.async, NBUF-deep ring) and run the
// epilogue; warp 4 only issues tcgen05.mma.  Hand-offs are mbarriers (full/empty per activation slot,
// full/empty per TMEM accumulator), so loads of tile i+NBUF-1, MMAs of tile i and the epilogue of
// tile i-1 are in flight together and nobody waits for the single MMA-issuing thread.
// Serves the channel-padded layers that the TMA kernels do not cover: <= 8 real input channels read with scalar
// loads, or a 16-channel accumulator of which only cout_real channels are stored (the fp32 RGB output conv).
template <int K, int NBUF>
__global__ void __launch_bounds__(160) conv_tc_persist_kernel(const bf16* __restrict__ x, const bf16* __restrict__ wp,
                                                              const float* __restrict__ bias, void* __restrict__ y,
                                                              int out_f32, int H, int W, int Cin, int Cout,
                                                              int total_tiles, int tmem_cols, int cin_real, int cout_real) {
  constexpr int HALO = K / 2, WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO, HP = WH * HH;
  // DIST tiles are prefetched ahead; NBUF - DIST >= 2 leaves a slot of slack so that re-using a slot never
  // waits on MMAs issued in the previous iteration.  The epilogue runs LAG tiles behind over 4 accumulators.
  constexpr int DIST = NBUF > 2 ? NBUF - 2 : 1;
  constexpr int LAG = 2, NACC = 4;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int k16n = Cin >> 4;
  const uint32_t slice_bytes = (uint32_t)Cout * 32;
  const uint32_t w_bytes = (uint32_t)(K * K * k16n) * slice_bytes;
  const uint32_t a_bytes = (uint32_t)(Cin >> 3) * HP * 16;
  uint8_t* sW = smem;
  uint8_t* sA = smem + w_bytes;                                               // NBUF slots
  uint64_t* full = reinterpret_cast<uint64_t*>(sA + NBUF * (size_t)a_bytes);  // slot staged (128 arrivals)
  uint64_t* empty = full + NBUF;                                              // slot consumed by the MMAs (commit)
  uint64_t* acc_full = empty + NBUF;                                          // accumulator ready (commit)
  uint64_t* acc_empty = acc_full + NACC;                                      // accumulator drained (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + NACC);

  const int tiles_x = (W + TC_TW - 1) / TC_TW, tiles_y = (H + TC_TH - 1) / TC_TH, tiles_img = tiles_x * tiles_y;
  const int T = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA
  auto tile_coords = [&](int j, int& n, int& y0, int& x0) {
    const int tile = blockIdx.x + j * gridDim.x;
    n = tile / tiles_img;
    const int t2 = tile - n * tiles_img;
    y0 = (t2 / tiles_x) * TC_TH;
    x0 = (t2 % tiles_x) * TC_TW;
  };

  if (warp == 4) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  if (tid == 0) {
    for (int i = 0; i < NBUF; ++i) { mbar_init(&full[i], 128); mbar_init(&empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 128); }
    mbar_fence_init();
  }
  if (warp < 4)
    for (int i = tid; i < (int)(w_bytes / 16); i += 128)
      reinterpret_cast<uint4*>(sW)[i] = __ldg(reinterpret_cast<const uint4*>(wp) + i);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ------------------------------------------------------------ loaders + epilogue (128 threads)
    const bool fast_stage = WH * (Cin >> 3) <= 128;
    const RowStager rs = make_row_stager<HALO>(fast_stage ? Cin : 16, tid);
    auto stage = [&](int j) {           // always commits one cp.async group (possibly empty)
      if (j < T) {
        const int s = j % NBUF;
        if (j >= NBUF) mbar_wait(&empty[s], (uint32_t)((j / NBUF) - 1) & 1u);   // MMAs of tile j-NBUF done with the slot
        int n, y0, x0;
        tile_coords(j, n, y0, x0);
        uint8_t* dst = sA + (size_t)s * a_bytes;
        if (cin_real != Cin) stage_tile_pad<HALO>(dst, x, n, y0, x0, H, W, Cin, cin_real, 128);
        else if (fast_stage) stage_rows<HALO>(rs, dst, x, n, y0, x0, H, W, Cin);
        else stage_tile_async<HALO>(dst, x, n, y0, x0, H, W, Cin, 128);
      }
      cp_async_commit();
    };
    auto epilogue = [&](int j) {
      const int acc = j & (NACC - 1);
      int n, y0, x0;
      tile_coords(j, n, y0, x0);
      mbar_wait(&acc_full[acc], (uint32_t)(j / NACC) & 1u);
      tc_fence_after_sync();
      if (!out_f32 && cout_real == Cout)
        conv_tc_epilogue_coalesced(tmem_base + (uint32_t)(acc * Cout), reinterpret_cast<uint8_t*>(full) + 256, warp, lane, n, y0, x0, H, W,
                                   Cout, bias, reinterpret_cast<bf16*>(y));
      else
      conv_tc_epilogue<HALO>(tmem_base + (uint32_t)(acc * Cout), warp, tid, n, y0, x0, H, W, Cout, bias, y, out_f32, cout_real);
      tc_fence_before_sync();
      mbar_arrive(&acc_empty[acc]);
    };
#pragma unroll
    for (int d = 0; d < DIST; ++d) stage(d);
    for (int it = 0; it < T; ++it) {
      stage(it + DIST);
      cp_async_wait_group<DIST>();       // this thread's part of tile `it` has landed
      fence_proxy_async_smem();          // ... and is visible to the tensor-core proxy
      mbar_arrive(&full[it % NBUF]);
      if (it >= LAG) epilogue(it - LAG);
    }
    for (int j = T > LAG ? T - LAG : 0; j < T; ++j) epilogue(j);
    cp_async_wait_all();
  } else {
    // ------------------------------------------------------------ MMA issuer (warp 4)
    const uint32_t idesc = umma_idesc_bf16(128, Cout, 0, 0);
    const uint64_t b0 = umma_desc(smem_u32(sW), (uint32_t)Cout * 16, 128);
    const uint32_t b_step = slice_bytes >> 4;
    for (int it = 0; it < T; ++it) {
      const int s = it % NBUF, acc = it & (NACC - 1);
      mbar_wait(&full[s], (uint32_t)(it / NBUF) & 1u);
      if (it >= NACC) mbar_wait(&acc_empty[acc], (uint32_t)((it / NACC) - 1) & 1u);
      tc_fence_after_sync();
      if (elect_one()) {
        const int c8n = Cin >> 3;
        const uint64_t a0 = umma_desc(smem_u32(sA + (size_t)s * a_bytes), WH * 16, c8n * WH * 16);
        const uint32_t dacc = tmem_base + (uint32_t)(acc * Cout);
        uint32_t sl = 0;
#pragma unroll
        for (int tap = 0; tap < K * K; ++tap) {
          const int ky = tap / K, kx = tap % K;
          for (int j = 0; j < k16n; ++j, ++sl)
            umma_bf16(dacc, a0 + (uint64_t)((ky * c8n * WH + kx) + 2 * j * WH), b0 + (uint64_t)(sl * b_step), idesc, sl > 0 ? 1u : 0u);
        }
        umma_commit(&empty[s]);
        umma_commit(&acc_full[acc]);
      }
      __syncwarp();
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

template <int K, int NBUF>
static int launch_conv_tc_persist(const void* x, const void* wp, const float* bias, void* y, int out_f32, int H, int W,
                                  int Cin, int Cout, long long tiles, int psmem, int pcols, int per_sm, int cin_real,
                                  int cout_real, cudaStream_t st) {
  static int smem_set = 0;
  if (psmem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_persist_kernel<K, NBUF>, cudaFuncAttributeMaxDynamicSharedMemorySize, psmem);
    if (e != cudaSuccess) return ttg_set_error(TTG_ERR_CUDA, "conv2d_tc: smem attribute: %s", cudaGetErrorString(e));
    smem_set = psmem;
  }
  long long grid = (long long)ttg_num_sms() * per_sm;
  if (grid > tiles) grid = tiles;
  conv_tc_persist_kernel<K, NBUF><<<(unsigned)grid, 160, psmem, st>>>((const bf16*)x, (const bf16*)wp, bias, y, out_f32, H, W, Cin,
                                                               Cout, (int)tiles, pcols, cin_real, cout_real);
  TTG_CHECK_LAUNCH("conv2d_tc_persist");
  return TTG_OK;
}

#define TC_RESIDENT_W_BYTES (80 * 1024)

// ------------------------------------------------------------------ fprop / dgrad, TMA-fed (weights resident)
// Same pipeline as conv_tc_persist_kernel, but the activation halo tile is fetched by ONE
// cp.async.bulk.tensor (TMA) instruction per tile: a rank-5 tensor map over the NHWC tensor viewed as
// (8 channels, W, C/8, H, N) with box (8, WH, C/8, HH, 1) lands in shared memory exactly as the
// [halo row][channel group][halo col] x 16 B image the UMMA descriptors expect, zero-filled outside the
// image (the conv padding), completion counted in bytes on the slot's mbarrier.  Layers with a compile-time
// input channel count (CIN in {16, 32, 64}) use the pixel-major swizzled tile instead (see umma_desc_swz).
// warp 5 = TMA producer, warp 4 = MMA issuer, warps 0-3 = epilogue only.
#include <cuda.h>
typedef CUresult (*ttg_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static ttg_encode_tiled_fn ttg_get_encode_tiled() {
  static ttg_encode_tiled_fn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (ttg_encode_tiled_fn)p;
  }
  return fn;
}
// Every driver that runs sm_100a exports cuTensorMapEncodeTiled; all tensor-core convolutions fetch their tiles with it.
static int ttg_no_encode_tiled(const char* who) {
  return ttg_set_error(TTG_ERR_UNSUPPORTED, "%s: the CUDA driver does not provide cuTensorMapEncodeTiled", who);
}

// accumulate flag as an immediate: with a compile-time input channel count every A descriptor of a tile is base + constant
template <bool ACC>
__device__ __forceinline__ void umma_bf16_imm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  if constexpr (ACC)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
}

// Pixel-major ("NHWC as it lies in memory") activation tile for the A operand: halo pixel (hy, hx) at
// (hy * WH + hx) * CIN * 2 bytes, its CIN channels contiguous -- the K-major canonical layout with a
// SWIZZLE_{32,64,128}B row of CIN * 2 bytes, written by ONE tensor-map load whose inner box dimension is the whole
// pixel (32-128 bytes per L2 request instead of the 16-byte requests of the [row][channel group][col] image: ncu of
// the 16->16 layers showed 8.4 M L2 read requests for 134 MB and the L2 request pipe, not HBM, near its limit).
// The swizzle XOR is a function of the absolute shared-memory address for both the TMA write and the UMMA read, so
// tap (ky, kx) is still just a shifted start address (rows are pixels) and a K step is +32 bytes inside the row.
__device__ __forceinline__ uint64_t umma_desc_swz(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t layout_type) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) |
         ((uint64_t)layout_type << 61);
}
__device__ __forceinline__ uint64_t umma_desc_sw(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | ((uint64_t)layout_type << 61);
}
__host__ __device__ __forceinline__ uint32_t umma_swz_layout_for(int channels) { return channels == 16 ? 6u : channels == 32 ? 4u : 2u; }
// all K*K*CIN/16 MMAs of one tile, statically unrolled (weights resident: B advances by b_step per slice)
template <int K, int CIN, int SL = 0>
__device__ __forceinline__ void resident_issue_tile_swz(uint32_t dacc, uint64_t a0, uint64_t b, uint32_t b_step, uint32_t idesc) {
  constexpr int K16N = CIN / 16, WH = TC_TW + 2 * (K / 2);
  if constexpr (SL < K * K * K16N) {
    constexpr int tap = SL / K16N, j = SL % K16N, ky = tap / K, kx = tap % K;
    umma_bf16_imm<(SL > 0)>(dacc, a0 + (uint64_t)((ky * WH + kx) * (CIN / 8) + 2 * j), b, idesc);
    resident_issue_tile_swz<K, CIN, SL + 1>(dacc, a0, b + b_step, b_step, idesc);
  }
}

template <int K, int NBUF, int CIN, bool STATS>
__global__ void __launch_bounds__(192) conv_tc_tma_kernel(const __grid_constant__ CUtensorMap tmap, const bf16* __restrict__ wp,
                                                          const float* __restrict__ bias, void* __restrict__ y, int out_f32,
                                                          int H, int W, int Cin_rt, int Cout, int total_tiles, int tmem_cols,
                                                          int cstore, double* __restrict__ stats) {
  constexpr int HALO = K / 2, WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO, HP = WH * HH;
  constexpr int NACC = 4;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int Cin = CIN > 0 ? CIN : Cin_rt;
  const int k16n = Cin >> 4, c8n = Cin >> 3;
  const uint32_t slice_bytes = (uint32_t)Cout * 32;
  const uint32_t w_bytes = (uint32_t)(K * K * k16n) * slice_bytes;
  const uint32_t a_bytes = (uint32_t)c8n * HP * 16;
  uint8_t* sW = smem;
  uint8_t* sA = smem + ((w_bytes + 127) & ~127u);                             // NBUF slots, 128-B aligned for TMA
  uint64_t* full = reinterpret_cast<uint64_t*>(sA + NBUF * (size_t)a_bytes);
  uint64_t* empty = full + NBUF;
  uint64_t* acc_full = empty + NBUF;
  uint64_t* acc_empty = acc_full + NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + NACC);

  const int tiles_x = (W + TC_TW - 1) / TC_TW, tiles_y = (H + TC_TH - 1) / TC_TH, tiles_img = tiles_x * tiles_y;
  const int T = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  auto tile_coords = [&](int j, int& n, int& y0, int& x0) {
    const int tile = blockIdx.x + j * gridDim.x;
    n = tile / tiles_img;
    const int t2 = tile - n * tiles_img;
    y0 = (t2 / tiles_x) * TC_TH;
    x0 = (t2 % tiles_x) * TC_TW;
  };

  float* s_stats = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full) + 512 + tc_epi_strip_bytes_dev(Cout));
  if constexpr (STATS)
    for (int i = tid; i < 2 * Cout; i += blockDim.x) s_stats[i] = 0.f;
  if (warp == 4) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  if (tid == 0) {
    for (int i = 0; i < NBUF; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 128); }
    mbar_fence_init();
  }
  if (warp < 4)
    for (int i = tid; i < (int)(w_bytes / 16); i += 128)
      reinterpret_cast<uint4*>(sW)[i] = __ldg(reinterpret_cast<const uint4*>(wp) + i);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ------------------------------------------------------------ epilogue (LAG tiles behind)
    EpiStats est;
    if constexpr (STATS) {
#pragma unroll
      for (int k = 0; k < 8; ++k) est.s[k] = est.q[k] = 0.f;
    }
    const bool reg_stats = STATS && epi_stats_in_regs(Cout) && cstore == Cout;
    for (int j = 0; j < T; ++j) {
      const int acc = j & (NACC - 1);
      int n, y0, x0;
      tile_coords(j, n, y0, x0);
      // one warp polls the mbarrier, the other three park on a hardware barrier: spinning warps cost issue slots
      if (warp == 0) mbar_wait(&acc_full[acc], (uint32_t)(j / NACC) & 1u);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      tc_fence_after_sync();
      if (!out_f32)
        conv_tc_epilogue_coalesced(tmem_base + (uint32_t)(acc * Cout), reinterpret_cast<uint8_t*>(full) + 512, warp, lane, n, y0, x0, H, W,
                                   cstore, bias, reinterpret_cast<bf16*>(y), STATS ? s_stats : nullptr,
                                   (STATS && reg_stats) ? &est : nullptr);
      else
      conv_tc_epilogue<HALO>(tmem_base + (uint32_t)(acc * Cout), warp, tid, n, y0, x0, H, W, Cout, bias, y, out_f32);
      tc_fence_before_sync();
      mbar_arrive(&acc_empty[acc]);
    }
    if constexpr (STATS) { if (reg_stats) epi_stats_flush(est, lane, Cout, s_stats); }
  } else if (warp == 4) {
    // ------------------------------------------------------------ MMA issuer
    const uint32_t idesc = umma_idesc_bf16(128, Cout, 0, 0);
    const uint64_t b0 = umma_desc(smem_u32(sW), (uint32_t)Cout * 16, 128);
    const uint32_t b_step = slice_bytes >> 4;
    for (int it = 0; it < T; ++it) {
      const int s = it % NBUF, acc = it & (NACC - 1);
      mbar_wait(&full[s], (uint32_t)(it / NBUF) & 1u);
      if (it >= NACC) mbar_wait(&acc_empty[acc], (uint32_t)((it / NACC) - 1) & 1u);
      tc_fence_after_sync();
      if (elect_one()) {
        const uint32_t dacc = tmem_base + (uint32_t)(acc * Cout);
        if constexpr (CIN > 0) {
          const uint64_t a0 = umma_desc_swz(smem_u32(sA + (size_t)s * a_bytes), (uint32_t)(WH * CIN * 2), umma_swz_layout_for(CIN));
          resident_issue_tile_swz<K, CIN>(dacc, a0, b0, b_step, idesc);
        } else {
          const uint64_t a0 = umma_desc(smem_u32(sA + (size_t)s * a_bytes), WH * 16, c8n * WH * 16);
          uint32_t sl = 0;
#pragma unroll
          for (int tap = 0; tap < K * K; ++tap) {
            const int ky = tap / K, kx = tap % K;
            for (int j = 0; j < k16n; ++j, ++sl)
              umma_bf16(dacc, a0 + (uint64_t)((ky * c8n * WH + kx) + 2 * j * WH), b0 + (uint64_t)(sl * b_step), idesc, sl > 0 ? 1u : 0u);
          }
        }
        umma_commit(&empty[s]);
        umma_commit(&acc_full[acc]);
      }
      __syncwarp();
    }
  } else if (warp == 5 && elect_one()) {
    // ------------------------------------------------------------ TMA producer (warp 5, one lane)
    for (int j = 0; j < T; ++j) {
      const int s = j % NBUF;
      if (j >= NBUF) mbar_wait(&empty[s], (uint32_t)((j / NBUF) - 1) & 1u);
      int n, y0, x0;
      tile_coords(j, n, y0, x0);
      const uint32_t bar = smem_u32(&full[s]);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(a_bytes) : "memory");
      if constexpr (CIN > 0)
      asm volatile(
          "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
          ::"r"(smem_u32(sA + (size_t)s * a_bytes)), "l"(&tmap), "r"(0), "r"(x0 - HALO), "r"(y0 - HALO), "r"(n), "r"(bar)
          : "memory");
      else
      asm volatile(
          "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
          ::"r"(smem_u32(sA + (size_t)s * a_bytes)), "l"(&tmap), "r"(0), "r"(x0 - HALO), "r"(0), "r"(y0 - HALO), "r"(n), "r"(bar)
          : "memory");
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  if constexpr (STATS)
    for (int i = tid; i < 2 * Cout; i += blockDim.x) atomicAdd(&stats[i], (double)s_stats[i]);
}

template <int K, int NBUF, int CIN>
static int launch_conv_tc_tma(const void* x, const void* wp, const float* bias, void* y, int out_f32, int N, int H, int W,
                              int Cin, int Cout, int cin_mem, int cstore, long long tiles, int w_bytes, int a_bytes, int pcols,
                              double* stats, cudaStream_t st) {
  const ttg_encode_tiled_fn enc = ttg_get_encode_tiled();
  if (!enc) return ttg_no_encode_tiled("conv2d_tc");
  constexpr int HALO = K / 2;
  CUtensorMap tmap;
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r;
  if constexpr (CIN > 0) {
    // pixel-major swizzled tile (see umma_desc_swz).  cin_mem = channels per pixel in memory (Cin, or 8 for the RGB
    // staging tensors: the box still asks for Cin channels and those that do not exist are zero-filled by the TMA
    // engine, like the spatial halo)
    const cuuint64_t d4[4] = {(cuuint64_t)cin_mem, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t s4[3] = {(cuuint64_t)cin_mem * 2, (cuuint64_t)W * cin_mem * 2, (cuuint64_t)H * W * cin_mem * 2};
    const cuuint32_t b4[4] = {(cuuint32_t)Cin, (cuuint32_t)(TC_TW + 2 * HALO), (cuuint32_t)(TC_TH + 2 * HALO), 1};
    r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), d4, s4, b4, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CIN == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CIN == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    const cuuint64_t gdim[5] = {8, (cuuint64_t)W, (cuuint64_t)(cin_mem / 8), (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t gstr[4] = {(cuuint64_t)cin_mem * 2, 16, (cuuint64_t)W * cin_mem * 2, (cuuint64_t)H * W * cin_mem * 2};
    const cuuint32_t box[5] = {8, (cuuint32_t)(TC_TW + 2 * HALO), (cuuint32_t)(Cin / 8), (cuuint32_t)(TC_TH + 2 * HALO), 1};
    r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x), gdim, gstr, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r != CUDA_SUCCESS) return ttg_set_error(TTG_ERR_CUDA, "conv2d_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
  const int smem = ((w_bytes + 127) & ~127) + NBUF * a_bytes + 512 + tc_epi_bytes(Cout);     // 512: mbarriers (up to 8 slots) + TMEM slot
  static int smem_set = 0;
  if (smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_tma_kernel<K, NBUF, CIN, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_tma_kernel<K, NBUF, CIN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return ttg_set_error(TTG_ERR_CUDA, "conv2d_tc: smem attribute: %s", cudaGetErrorString(e));
    smem_set = smem;
  }
  int per_sm = (200 * 1024) / smem;
  if (per_sm > 512 / pcols) per_sm = 512 / pcols;
  if (per_sm > 8) per_sm = 8;
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)ttg_num_sms() * per_sm;
  if (grid > tiles) grid = tiles;
  if (stats)
    conv_tc_tma_kernel<K, NBUF, CIN, true><<<(unsigned)grid, 192, smem, st>>>(tmap, (const bf16*)wp, bias, y, out_f32, H, W, Cin, Cout,
                                                                        (int)tiles, pcols, cstore, stats);
  else
    conv_tc_tma_kernel<K, NBUF, CIN, false><<<(unsigned)grid, 192, smem, st>>>(tmap, (const bf16*)wp, bias, y, out_f32, H, W, Cin, Cout,
                                                                         (int)tiles, pcols, cstore, stats);
  TTG_CHECK_LAUNCH("conv2d_tc_tma");
  return TTG_OK;
}

// ------------------------------------------------------------------ fprop / dgrad, filters too large for shared memory
// (128->128, 256->256 ...): persistent, warp-specialised, weights STREAMED.  warps 0-3 run the epilogue; warp 4 issues
// tcgen05.mma; warp 5 fetches the activation tiles (tensor-map loads, NA slots) and streams the packed filter from L2
// through a ring of NW 16 KB stages for every tile.  These layers are tensor/L2 bound, not HBM bound.
#define TC_WSTAGE_BYTES (16 * 1024)
#ifdef TTG_TRACE
// development build only: per-event clock64() stamps of CTA 0 (role, index, t0, t1)
__device__ long long ttg_trace_buf[16 * 256 * 2];
__device__ __forceinline__ void ttg_trace(int role, int idx, long long t0, long long t1) {
  if (blockIdx.x != 0 || idx >= 256) return;
  ttg_trace_buf[(role * 256 + idx) * 2] = t0;          // fire-and-forget stores: no round trip in the traced path
  ttg_trace_buf[(role * 256 + idx) * 2 + 1] = t1;
}
extern "C" int ttg_trace_read(long long* host, int reset) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(host, ttg_trace_buf, sizeof(ttg_trace_buf));
  if (reset) { static long long z[16 * 256 * 2]; cudaMemcpyToSymbol(ttg_trace_buf, z, sizeof(z)); }
  return 16 * 256;
}
#define TTG_T0() long long t0__ = clock64()
#define TTG_T1(role, idx) ttg_trace(role, idx, t0__, clock64())
#else
#define TTG_T0()
#define TTG_T1(role, idx)
#endif
// One chunk (= one weight stage) of the statically unrolled MMA sequence of a 3x3 tile.
template <int CIN, int COUT, int CHUNK, int C, int I = 0>
__device__ __forceinline__ void stream_issue_chunk(uint32_t dacc, uint64_t a0, uint64_t b, uint32_t idesc) {
  constexpr int K16N = CIN / 16, C8N = CIN / 8, WH = TC_TW + 2, TOTAL = 9 * K16N;
  constexpr int slice = C * CHUNK + I;
  if constexpr (I < CHUNK && slice < TOTAL) {
    constexpr int tap = slice / K16N, j = slice % K16N, ky = tap / 3, kx = tap % 3;
    constexpr uint32_t aoff = (uint32_t)(ky * C8N * WH + kx + 2 * j * WH);
    umma_bf16_imm<(slice > 0)>(dacc, a0 + (uint64_t)aoff, b + (uint64_t)(I * (COUT * 32 / 16)), idesc);
    stream_issue_chunk<CIN, COUT, CHUNK, C, I + 1>(dacc, a0, b, idesc);
  }
}

// CIN / COUT > 0: 3x3 layer with compile-time channel counts (lean, fully unrolled issue sequence);
// CIN == 0: any supported layer, runtime walk.
template <int K, int NA, int CIN, int COUT>
__global__ void __launch_bounds__(192) conv_tc_stream_ws_kernel(const bf16* __restrict__ wp,
                                                                const float* __restrict__ bias, void* __restrict__ y,
                                                                int out_f32, int H, int W, int Cin_rt, int Cout_rt,
                                                                int total_tiles, int tmem_cols, int chunk_slices_rt,
                                                                const __grid_constant__ CUtensorMap tmap,
                                                                double* __restrict__ stats) {
  constexpr int HALO = K / 2, WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO, HP = WH * HH;
  constexpr bool STATIC = CIN > 0;
  // weight ring: the issuing thread pays ~400 cycles of fixed cost per stage (mbarrier wait, fences, commit), so the
  // static variant uses 32 KB stages (8 MMAs of 128x128x16 = 512 tensor cycles per stage)
  constexpr int NW = STATIC ? 3 : 4, WSB = STATIC ? 2 * TC_WSTAGE_BYTES : TC_WSTAGE_BYTES, NACC = 2;
  constexpr int APIECES = K == 3 ? 6 : 4, AROWS = HH / APIECES;      // activation tile = APIECES tensor-map loads
  static_assert(!STATIC || K == 3, "static channel counts: 3x3 only");
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int Cin = STATIC ? CIN : Cin_rt, Cout = STATIC ? COUT : Cout_rt;
  const int k16n = Cin >> 4, c8n = Cin >> 3;
  const int total_slices = K * K * k16n;
  const int chunk_slices = STATIC ? WSB / (COUT > 0 ? COUT * 32 : 1) : chunk_slices_rt;
  const int nchunks = (total_slices + chunk_slices - 1) / chunk_slices;
  const uint32_t slice_bytes = (uint32_t)Cout * 32;
  const uint32_t a_bytes = (uint32_t)c8n * HP * 16;
  uint8_t* sA = smem;
  uint8_t* sW = smem + (size_t)NA * a_bytes;
  uint64_t* afull = reinterpret_cast<uint64_t*>(sW + (size_t)NW * WSB);
  uint64_t* aempty = afull + NA;
  uint64_t* wfull = aempty + NA;
  uint64_t* wempty = wfull + NW;
  uint64_t* acc_full = wempty + NW;
  uint64_t* acc_empty = acc_full + NACC;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + NACC);

  const int tiles_x = (W + TC_TW - 1) / TC_TW, tiles_y = (H + TC_TH - 1) / TC_TH, tiles_img = tiles_x * tiles_y;
  const int T = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  auto tile_coords = [&](int j, int& n, int& y0, int& x0) {
    const int tile = blockIdx.x + j * gridDim.x;
    n = tile / tiles_img;
    const int t2 = tile - n * tiles_img;
    y0 = (t2 / tiles_x) * TC_TH;
    x0 = (t2 % tiles_x) * TC_TW;
  };
  float* s_stats = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(afull) + 256 + tc_epi_strip_bytes_dev(Cout));
  if (stats)
    for (int i = tid; i < 2 * Cout; i += blockDim.x) s_stats[i] = 0.f;
  if (warp == 4) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  if (tid == 0) {
    for (int i = 0; i < NA; ++i) { mbar_init(&afull[i], 1); mbar_init(&aempty[i], 1); }
    for (int i = 0; i < NW; ++i) { mbar_init(&wfull[i], 1); mbar_init(&wempty[i], 1); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 128); }
    mbar_fence_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ------------------------------------------------------------ epilogue (tiles arrive by TMA, warp 5)
    for (int j = 0; j < T; ++j) {
      const int acc = j % NACC;
      int n, y0, x0;
      tile_coords(j, n, y0, x0);
      { TTG_T0(); mbar_wait(&acc_full[acc], (uint32_t)(j / NACC) & 1u); if (tid == 0) { TTG_T1(5, j); } }
      tc_fence_after_sync();
      TTG_T0();
      if (!out_f32)
        conv_tc_epilogue_coalesced(tmem_base + (uint32_t)(acc * Cout), reinterpret_cast<uint8_t*>(afull) + 256, warp, lane, n, y0, x0, H, W,
                                   Cout, bias, reinterpret_cast<bf16*>(y), stats ? s_stats : nullptr);
      else
        conv_tc_epilogue<HALO>(tmem_base + (uint32_t)(acc * Cout), warp, tid, n, y0, x0, H, W, Cout, bias, y, out_f32);
      tc_fence_before_sync();
      mbar_arrive(&acc_empty[acc]);
      if (tid == 0) { TTG_T1(6, j); }
    }
  } else if (warp == 4) {
    // ------------------------------------------------------------ MMA issuer
    // The issuing thread is a single in-order instruction stream: every instruction between two UTCHMMAs is
    // exposed latency, so the static variant folds all descriptor arithmetic into immediates.
    const uint32_t idesc = umma_idesc_bf16(128, Cout, 0, 0);
    const uint32_t sl_units = slice_bytes >> 4;
    const uint64_t bdesc0 = umma_desc(smem_u32(sW), (uint32_t)Cout * 16, 128);
    uint32_t g = 0;
    for (int it = 0; it < T; ++it) {
      const int s = it % NA, acc = it % NACC;
      { TTG_T0(); mbar_wait(&afull[s], (uint32_t)(it / NA) & 1u); if (lane == 0) { TTG_T1(2, it); } }
      { TTG_T0(); if (it >= NACC) mbar_wait(&acc_empty[acc], (uint32_t)((it / NACC) - 1) & 1u); if (lane == 0) { TTG_T1(3, it); } }
      const uint64_t a0 = umma_desc(smem_u32(sA + (size_t)s * a_bytes), WH * 16, c8n * WH * 16);
      const uint32_t dacc = tmem_base + (uint32_t)(acc * Cout);
      if constexpr (STATIC) {
        constexpr int CHUNK = WSB / (COUT * 32);
        static_assert(CHUNK >= 1, "stage smaller than one K slice");
        constexpr int NCH = (9 * (CIN / 16) + CHUNK - 1) / CHUNK;
        auto chunk = [&](auto cc) {
          constexpr int C = decltype(cc)::value;
          const uint32_t ws = (g + C) % NW;
          { TTG_T0(); mbar_wait(&wfull[ws], ((g + C) / NW) & 1u); if (lane == 0) { TTG_T1(1, (int)(g + C)); } }
          tc_fence_after_sync();
          if (elect_one()) {
            TTG_T0();
            stream_issue_chunk<CIN, COUT, CHUNK, C>(dacc, a0, bdesc0 + (uint64_t)(ws * (WSB >> 4)), idesc);
            TTG_T1(7, (int)(g + C));
            { TTG_T0();
            umma_commit(&wempty[ws]);
            if constexpr (C == NCH - 1) { umma_commit(&aempty[s]); umma_commit(&acc_full[acc]); }
            TTG_T1(8, (int)(g + C)); }
          }
          __syncwarp();
        };
        static_for<NCH>(chunk);
        g += NCH;
      } else {
        // runtime (tap, k16) walk kept incrementally: no division in the issue loop
        int j = 0, kx = 0;
        uint32_t a_row = 0;               // ky * c8n * WH
        uint32_t accum = 0;
        int left = total_slices;
        for (int c = 0; c < nchunks; ++c, ++g) {
          const uint32_t ws = g % NW;
          mbar_wait(&wfull[ws], (g / NW) & 1u);
          tc_fence_after_sync();
          {
            // every lane walks the indices (they are warp-uniform); one elected lane issues
            uint64_t b = bdesc0 + (uint64_t)(ws * (WSB >> 4));
            const int cnt = min(chunk_slices, left);
            const bool leader = elect_one();
            for (int i = 0; i < cnt; ++i) {
              if (leader) umma_bf16(dacc, a0 + (uint64_t)(a_row + (uint32_t)kx + (uint32_t)(2 * j * WH)), b, idesc, accum);
              accum = 1u;
              b += sl_units;
              if (++j == k16n) { j = 0; if (++kx == K) { kx = 0; a_row += (uint32_t)(c8n * WH); } }
            }
            if (leader) {
              umma_commit(&wempty[ws]);
              if (c == nchunks - 1) { umma_commit(&aempty[s]); umma_commit(&acc_full[acc]); }
            }
          }
          __syncwarp();
          left -= chunk_slices;
        }
      }
    }
  } else {
    // ------------------------------------------------------------ producer (warp 5, one lane)
    // weights: cp.async.bulk (TMA 1-D bulk copy), one instruction per 16 KB stage, completion counted in bytes on
    // the stage's mbarrier, NW stages in flight; activation halo tiles: one tensor-map load per tile.
    if (elect_one()) {
      const uint32_t G = (uint32_t)T * (uint32_t)nchunks;
      const uint32_t chunk_bytes = (uint32_t)chunk_slices * slice_bytes;
      const uint32_t last_bytes = (uint32_t)(total_slices - (nchunks - 1) * chunk_slices) * slice_bytes;
      const uint32_t sW_addr = smem_u32(sW);
      // An activation tile is fetched as APIECES row groups: the TMA engine serves requests in order and a halo tile is
      // thousands of 16-byte rows, so one big load would stall the weight stream queued behind it.  The pieces of tile
      // t+1 are slipped in between the weight stages of tile t (all pieces complete_tx on the slot's barrier).
      auto issue_a_piece = [&](int j, int piece) {
        const int s = j % NA;
        int n, y0, x0;
        tile_coords(j, n, y0, x0);
        const uint32_t bar = smem_u32(&afull[s]);
        if (piece == 0) {
          if (j >= NA) mbar_wait(&aempty[s], (uint32_t)((j / NA) - 1) & 1u);
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(a_bytes) : "memory");
        }
        const uint32_t dst = smem_u32(sA + (size_t)s * a_bytes) + (uint32_t)(piece * AROWS * c8n * WH * 16);
        asm volatile(
            "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
            ::"r"(dst), "l"(&tmap), "r"(0), "r"(x0 - HALO), "r"(0), "r"(y0 - HALO + piece * AROWS), "r"(n), "r"(bar)
            : "memory");
      };
      // pieces of the next tile start once the ring has turned over (its slot is then known to be free: NA == 2),
      // or after the last stage when there is a single activation slot
      const int c_first = NA > 1 ? min(NW, nchunks - 1) : nchunks - 1;
      if (T > 0)
        for (int pc = 0; pc < APIECES; ++pc) issue_a_piece(0, pc);
      int c = 0, tile = 0, piece = 0;
      for (uint32_t g = 0; g < G; ++g) {
        const uint32_t ws = g % NW;
        { TTG_T0(); if (g >= NW) mbar_wait(&wempty[ws], ((g / NW) - 1) & 1u); TTG_T1(4, (int)g); }
        const uint32_t bytes = c == nchunks - 1 ? last_bytes : chunk_bytes;
        const uint8_t* src = reinterpret_cast<const uint8_t*>(wp) + (size_t)c * chunk_bytes;
        const uint32_t bar = smem_u32(&wfull[ws]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(sW_addr + ws * WSB), "l"(src), "r"(bytes), "r"(bar) : "memory");
        if (tile + 1 < T && c >= c_first) {
          if (piece < APIECES) issue_a_piece(tile + 1, piece++);
          if (c == nchunks - 1)
            while (piece < APIECES) issue_a_piece(tile + 1, piece++);
        }
        if (++c == nchunks) { c = 0; ++tile; piece = 0; }
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  if (stats)
    for (int i = tid; i < 2 * Cout; i += blockDim.x) atomicAdd(&stats[i], (double)s_stats[i]);
}

template <int K, int NA, int CIN, int COUT>
static int launch_conv_tc_stream_ws(const void* x, const void* wp, const float* bias, void* y, int out_f32, int N, int H, int W,
                                    int Cin, int Cout, long long tiles, double* stats, cudaStream_t st) {
  const ttg_encode_tiled_fn enc = ttg_get_encode_tiled();
  if (!enc) return ttg_no_encode_tiled("conv2d_tc");
  constexpr int HALO = K / 2;
  const int HP = (TC_TW + 2 * HALO) * (TC_TH + 2 * HALO);
  constexpr int NW = CIN > 0 ? 3 : 4, WSB = CIN > 0 ? 2 * TC_WSTAGE_BYTES : TC_WSTAGE_BYTES;
  constexpr int APIECES = K == 3 ? 6 : 4;
  const int smem = NA * (Cin / 8) * HP * 16 + NW * WSB + 256 + tc_epi_bytes(Cout);
  CUtensorMap tmap;
  const cuuint64_t gdim[5] = {8, (cuuint64_t)W, (cuuint64_t)(Cin / 8), (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t gstr[4] = {(cuuint64_t)Cin * 2, 16, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2};
  const cuuint32_t box[5] = {8, (cuuint32_t)(TC_TW + 2 * HALO), (cuuint32_t)(Cin / 8), (cuuint32_t)((TC_TH + 2 * HALO) / APIECES), 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return ttg_set_error(TTG_ERR_CUDA, "conv2d_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
  static int smem_set = 0;
  if (smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_stream_ws_kernel<K, NA, CIN, COUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return ttg_set_error(TTG_ERR_CUDA, "conv2d_tc: smem attribute: %s", cudaGetErrorString(e));
    smem_set = smem;
  }
  int chunk_slices = WSB / (Cout * 32);
  if (chunk_slices < 1) chunk_slices = 1;
  const int cols = (int)tmem_cols_for(2 * Cout);
  long long grid = ttg_num_sms();
  if (grid > tiles) grid = tiles;
  conv_tc_stream_ws_kernel<K, NA, CIN, COUT><<<(unsigned)grid, 192, smem, st>>>(
      (const bf16*)wp, bias, y, out_f32, H, W, Cin, Cout, (int)tiles, cols, chunk_slices, tmap, stats);
  TTG_CHECK_LAUNCH("conv2d_tc_stream_ws");
  return TTG_OK;
}

// Cin / Cout are the (padded, multiple-of-16) GEMM channel counts; cin_real / cout_real the channel counts of the
// tensors in memory (equal to Cin / Cout except for the RGB layers).
// stats (optional): double[2 * Cout], zeroed by the caller; receives sum / sum of squares per output channel of the
// tensor written (BatchNorm statistics of the next layer, see ttg_conv2d_tc_stats).
static int conv2d_tc_core(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin,
                          int Cout, int cin_real, int cout_real, int ksize, int dtype_out, double* stats, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  // 8-channel staging tensors (ttg_pad_channels8) ride the TMA path: not "padded" in the scalar-access sense
  // (genuine 8-channel layers of the '512thin' config look the same; with an fp32 output they take the scalar-access
  // padded path below instead)
  const bool tma8 = dtype_out == TTG_BF16;
  const bool in8 = tma8 && cin_real == 8 && Cin == 16, out8 = tma8 && cout_real == 8 && Cout == 16;
  const bool padded = (cin_real != Cin && !in8) || (cout_real != Cout && !out8);
  TTG_REQUIRE(cin_real >= 1 && cin_real <= Cin && cout_real >= 1 && cout_real <= Cout, "conv2d_tc: bad real channel counts");
  TTG_REQUIRE(!padded || ((cin_real == Cin || cin_real <= 8) && (cout_real == Cout || (cout_real <= 16 && Cout == 16))),
              "conv2d_tc: channel padding supports <= 8 real input channels / Cout padded to 16");
  TTG_REQUIRE(ksize == 1 || ksize == 3, "conv2d_tc: ksize %d unsupported", ksize);
  TTG_REQUIRE(Cin % 16 == 0 && Cout % 16 == 0 && Cin >= 16 && Cout >= 16 && Cin <= 256 && Cout <= 256,
              "conv2d_tc: channels must be multiples of 16 in [16,256] (got %d -> %d)", Cin, Cout);
  TTG_REQUIRE(dtype_out == TTG_BF16 || dtype_out == TTG_F32, "conv2d_tc: bad output dtype");
  TTG_REQUIRE(padded || ((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0),
              "conv2d_tc: activation pointers must be 16-byte aligned");
  TTG_REQUIRE((reinterpret_cast<uintptr_t>(wp) & 15) == 0, "conv2d_tc: weight pointer must be 16-byte aligned");
  const int halo = ksize / 2;
  const int HP = (TC_TW + 2 * halo) * (TC_TH + 2 * halo);
  const int a_bytes = (Cin / 8) * HP * 16;
  const long long tiles = (long long)N * ((H + TC_TH - 1) / TC_TH) * ((W + TC_TW - 1) / TC_TW);
  TTG_REQUIRE(tiles > 0 && tiles < (1ll << 31), "conv2d_tc: bad problem size");
  const int w_bytes = ksize * ksize * (Cin / 16) * Cout * 32;
  TTG_REQUIRE(!padded || w_bytes <= TC_RESIDENT_W_BYTES, "conv2d_tc: padded layers must fit the resident-filter kernel");
  const int of32 = dtype_out == TTG_F32;
  if (w_bytes <= TC_RESIDENT_W_BYTES && !padded) {
    const int tcols = (int)tmem_cols_for(4 * Cout);
    const bool deep = a_bytes <= 12 * 1024;       // small tiles: 4 slots, else 3
#define TTG_TMA(KK, NB, CI) launch_conv_tc_tma<KK, NB, CI>(x, wp, bias, y, of32, N, H, W, Cin, Cout, cin_real, cout_real, tiles, w_bytes, a_bytes, tcols, stats, st)
    // activation slots that fit next to the resident filter (256 -> 128 1x1: 64 KB filter + 64 KB tiles -> 2 slots)
    const bool three = ((w_bytes + 127) & ~127) + 3 * a_bytes + 256 + tc_epi_bytes(Cout) <= 227 * 1024;
    // ring depth: the pipeline of one CTA is latency bound (one CTA per SM reaches half the throughput of three), so the
    // small tiles get 8 / 6 slots: 16->16 @128^2 80 -> 66 us, 32->32 @64^2 39 -> 37 us (round 2 sweep)
    const bool four64 = ((w_bytes + 127) & ~127) + 4 * a_bytes + 256 + tc_epi_bytes(Cout) <= 200 * 1024;
    if (ksize == 3) return Cin == 16 ? TTG_TMA(3, 8, 16) : Cin == 32 ? TTG_TMA(3, 6, 32) : Cin == 64 ? (four64 ? TTG_TMA(3, 4, 64) : TTG_TMA(3, 3, 64))
                                   : (deep ? TTG_TMA(3, 4, 0) : three ? TTG_TMA(3, 3, 0) : TTG_TMA(3, 2, 0));
    return Cin == 16 ? TTG_TMA(1, 8, 16) : Cin == 32 ? TTG_TMA(1, 8, 32) : Cin == 64 ? (four64 ? TTG_TMA(1, 4, 64) : TTG_TMA(1, 3, 64))
                     : (deep ? TTG_TMA(1, 4, 0) : three ? TTG_TMA(1, 3, 0) : TTG_TMA(1, 2, 0));
#undef TTG_TMA
  }
  if (padded) {
    TTG_REQUIRE(stats == nullptr, "conv2d_tc: output statistics need the TMA kernels (bf16 output, no padding)");
    const int nbuf = a_bytes <= 12 * 1024 ? 4 : (a_bytes <= 24 * 1024 ? 3 : 2);
    const int psmem = w_bytes + nbuf * a_bytes + 256 + tc_epi_bytes(Cout);
    const int pcols = (int)tmem_cols_for(4 * Cout);
    int per_sm = (200 * 1024) / psmem;
    if (per_sm > 512 / pcols) per_sm = 512 / pcols;
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
#define TTG_PERSIST(KK, NB) launch_conv_tc_persist<KK, NB>(x, wp, bias, y, of32, H, W, Cin, Cout, tiles, psmem, pcols, per_sm, \
                                                           cin_real, cout_real, st)
    if (ksize == 3) return nbuf == 4 ? TTG_PERSIST(3, 4) : nbuf == 3 ? TTG_PERSIST(3, 3) : TTG_PERSIST(3, 2);
    return nbuf == 4 ? TTG_PERSIST(1, 4) : nbuf == 3 ? TTG_PERSIST(1, 3) : TTG_PERSIST(1, 2);
#undef TTG_PERSIST
  }
  // filter streamed through shared memory: one K slice of it (Cout * 32 bytes) always fits a weight stage
  static_assert(256 * 32 <= TC_WSTAGE_BYTES, "weight stage smaller than one K slice");
  const bool two = 2 * a_bytes + 4 * TC_WSTAGE_BYTES + 256 + tc_epi_bytes(Cout) <= 200 * 1024;
#define TTG_STREAM(KK, NAA, CI, CO) launch_conv_tc_stream_ws<KK, NAA, CI, CO>(x, wp, bias, y, of32, N, H, W, Cin, Cout, tiles, stats, st)
  const bool two32 = 2 * a_bytes + 6 * TC_WSTAGE_BYTES + 256 + tc_epi_bytes(Cout) <= 224 * 1024;
  const bool one32 = a_bytes + 6 * TC_WSTAGE_BYTES + 256 + tc_epi_bytes(Cout) <= 224 * 1024;
  if (ksize == 3 && two32) {
    if (Cin == 128 && Cout == 128) return TTG_STREAM(3, 2, 128, 128);
    if (Cin == 128 && Cout == 64) return TTG_STREAM(3, 2, 128, 64);
    if (Cin == 64 && Cout == 128) return TTG_STREAM(3, 2, 64, 128);
    if (Cin == 128 && Cout == 256) return TTG_STREAM(3, 2, 128, 256);
  }
  if (ksize == 3 && !two32 && one32) {
    if (Cin == 256 && Cout == 256) return TTG_STREAM(3, 1, 256, 256);
    if (Cin == 256 && Cout == 128) return TTG_STREAM(3, 1, 256, 128);
  }
  if (ksize == 3) return two ? TTG_STREAM(3, 2, 0, 0) : TTG_STREAM(3, 1, 0, 0);
  return two ? TTG_STREAM(1, 2, 0, 0) : TTG_STREAM(1, 1, 0, 0);
#undef TTG_STREAM
}

extern "C" int ttg_conv2d_tc_ex(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin,
                                int Cout, int cin_real, int cout_real, int ksize, int dtype_out, void* stream) {
  return conv2d_tc_core(x, wp, bias, y, N, H, W, Cin, Cout, cin_real, cout_real, ksize, dtype_out, nullptr, stream);
}
// conv + BatchNorm statistics of its output in one pass: sums[0..Cout) = sum_pixels y, sums[Cout..2Cout) = sum y^2
// (fp64, of the bf16 values written).  The epilogue reduces the tile it holds in registers, so the statistics pass of
// the following nn.BatchNorm2d (native_batch_norm's first read of the tensor) disappears.
extern "C" int ttg_conv2d_tc_stats_supported(int Cin, int Cout, int ksize) {
  return Cin % 16 == 0 && Cout % 16 == 0 && Cin >= 16 && Cout >= 16 && Cin <= 256 && Cout <= 256 && (ksize == 1 || ksize == 3);
}
extern "C" int ttg_conv2d_tc_stats(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin,
                                   int Cout, int ksize, double* sums, void* stream) {
  TTG_REQUIRE(sums != nullptr, "conv2d_tc_stats: sums is required");
  TTG_REQUIRE(ttg_conv2d_tc_stats_supported(Cin, Cout, ksize), "conv2d_tc_stats: unsupported layer %d -> %d k%d", Cin, Cout, ksize);
  cudaMemsetAsync(sums, 0, sizeof(double) * 2 * (size_t)Cout, (cudaStream_t)stream);
  return conv2d_tc_core(x, wp, bias, y, N, H, W, Cin, Cout, Cin, Cout, ksize, TTG_BF16, sums, stream);
}
extern "C" int ttg_conv2d_tc(const void* x, const void* wp, const float* bias, void* y, int N, int H, int W, int Cin,
                             int Cout, int ksize, int dtype_out, void* stream) {
  return ttg_conv2d_tc_ex(x, wp, bias, y, N, H, W, Cin, Cout, Cin, Cout, ksize, dtype_out, stream);
}

// ------------------------------------------------------------------ wgrad
// gw[co][ci][ky][kx] += sum over the CTA's pixel tiles of gy[p,co] * x[p+tap,ci].
// grid = (pixel splits, tap groups, Cout halves).  Per tile and tap: 8 MMAs (K = 2 rows x 8 pixels),
// M = 128 output channels (rows >= Cout are padding), N = Cin, accumulators: taps_per_group x Cin columns.
template <int K>
__global__ void __launch_bounds__(128) conv_wgrad_tc_kernel(const bf16* __restrict__ x, const bf16* __restrict__ gy,
                                                            float* __restrict__ gw, int N, int H, int W, int Cin, int Cout,
                                                            int taps_per_group, int tmem_cols) {
  constexpr int HALO = K / 2, WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO, HP = WH * HH, NPIX = TC_TH * TC_TW;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t x_bytes = (uint32_t)(Cin >> 3) * HP * 16;
  uint8_t* sX = smem;
  uint8_t* sG = smem + x_bytes;                       // [16 co-groups][128 pixels] x 16 B (always 128 rows)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sG + 16 * NPIX * 16);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);

  const int tap0 = blockIdx.y * taps_per_group;
  const int ntaps = min(taps_per_group, K * K - tap0);
  const int co_base = blockIdx.z * 128;
  const int co_cnt = min(128, Cout - co_base);

  if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  if (tid == 32) { mbar_init(&bars[0], 1); mbar_fence_init(); }
  // zero the padding rows of the gy tile once (rows >= co_cnt are never rewritten)
  for (int u = tid; u < 16 * NPIX; u += blockDim.x) *reinterpret_cast<uint4*>(sG + (size_t)u * 16) = make_uint4(0u, 0u, 0u, 0u);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles_x = (W + TC_TW - 1) / TC_TW, tiles_y = (H + TC_TH - 1) / TC_TH;
  const long long total_tiles = (long long)N * tiles_x * tiles_y;
  const uint32_t idesc = umma_idesc_bf16(128, Cin, 1, 1);
  const uint32_t sX_addr = smem_u32(sX), sG_addr = smem_u32(sG);
  const int g8n = co_cnt >> 3;
  uint32_t phase = 0;
  bool first = true;
  for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int n = (int)(tile / (tiles_x * tiles_y)), t2 = (int)(tile - (long long)n * tiles_x * tiles_y);
    const int y0 = (t2 / tiles_x) * TC_TH, x0 = (t2 % tiles_x) * TC_TW;
    if (!first) { mbar_wait(&bars[0], phase); phase ^= 1u; }       // previous tile's MMAs have consumed the smem
    stage_tile<HALO>(sX, x, n, y0, x0, H, W, Cin, 128);
    for (int u = tid; u < NPIX * g8n; u += blockDim.x) {
      const int g8 = u % g8n, pix = u / g8n;
      const int py = y0 + (pix >> 3), px = x0 + (pix & 7);
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (py < H && px < W) v = *reinterpret_cast<const uint4*>(gy + (((long long)n * H + py) * W + px) * Cout + co_base + g8 * 8);
      *reinterpret_cast<uint4*>(sG + ((size_t)g8 * NPIX + pix) * 16) = v;
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after_sync();
      for (int t = 0; t < ntaps; ++t) {
        const int tap = tap0 + t, ky = tap / K, kx = tap - ky * K;
#pragma unroll 1
        for (int r = 0; r < TC_TH / 2; ++r) {
          // A = gy^T (MN-major): M groups of 8 channels (SBO = 128 pixels x 16 B), K = pixels: 8 per row (16 B apart), rows LBO apart
          const uint64_t adesc = umma_desc(sG_addr + (uint32_t)(2 * r * TC_TW) * 16, TC_TW * 16, NPIX * 16);
          // B = shifted x (MN-major): N groups of 8 channels (SBO = WH units), K = pixels of halo rows 2r+ky, 2r+1+ky
          const int c8n = Cin >> 3;
          const uint64_t bdesc = umma_desc(sX_addr + (uint32_t)((2 * r + ky) * c8n * WH + kx) * 16, c8n * WH * 16, WH * 16);
          umma_bf16(tmem_base + (uint32_t)(t * Cin), adesc, bdesc, idesc, (first && r == 0) ? 0u : 1u);
        }
      }
      umma_commit(&bars[0]);
    }
    first = false;
  }
  if (!first) {
    mbar_wait(&bars[0], phase);
    tc_fence_after_sync();
    const int co = co_base + tid;                     // TMEM lane = output channel
    for (int t = 0; t < ntaps; ++t) {
      const int tap = tap0 + t;
      for (int c0 = 0; c0 < Cin; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(t * Cin + c0), r);
        tmem_ld_wait();
        if (tid < co_cnt) {
#pragma unroll
          for (int j = 0; j < 16; ++j) atomicAdd(gw + ((long long)co * Cin + c0 + j) * (K * K) + tap, __uint_as_float(r[j]));
        }
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

// ------------------------------------------------------------------ wgrad, persistent + warp-specialised
// warp 7 loads (x halo tile, gy tile) pairs with tensor-map loads into an NBUF ring; warps 4-6 each issue the
// MMAs of a share of the accumulator "units" (disjoint TMEM columns, so the issuing threads never touch
// the same accumulator); accumulators stay in TMEM over all tiles of the CTA; warps 0-3 run one atomic epilogue.
// For Cin <= 80 a unit is a filter column kx with N = 3*Cin: the [row][c8][col] tile layout makes the
// three vertical taps one uniform-stride B operand, so gy^T (the A operand, mostly padding rows for
// small Cout) is read 3 instead of 9 times per K step; with Cout <= 64 the MMA uses M = 64.
template <int K, int NBUF>
__global__ void __launch_bounds__(256) conv_wgrad_tc_ws_kernel(float* __restrict__ gw, int N, int H, int W, int Cin,
                                                               int Cout, int units_per_group, int fuse,
                                                               int tmem_cols, int g_bytes, int cout_real,
                                                               const __grid_constant__ CUtensorMap tmap_x,
                                                               const __grid_constant__ CUtensorMap tmap_g,
                                                               float* __restrict__ gbias) {
  constexpr int HALO = K / 2, WH = TC_TW + 2 * HALO, HH = TC_TH + 2 * HALO, NPIX = TC_TH * TC_TW;
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int c8n = Cin >> 3;
  // fuse == 3 ("mfold"): the filter column kx is folded into M and the filter row ky into N, so a tile
  // costs 8 MMAs instead of 24:  D[(j, co), (ky, ci)] = sum_q gy[q + j - 1][co] * x[q + (ky-1) rows][ci],  kx = 2 - j.
  // Both tiles are PIXEL-MAJOR (NHWC as in memory: one TMA request per pixel, SWIZZLE_32B/64B/128B by channel count),
  // which is the MN-major canonical layout with one swizzle row per pixel:
  //   A = gy^T: the gy tile with a one-column halo, [16 rows][10 cols][Cout]; the M block j is the same tile one pixel
  //       further on (LBO = one pixel), K = the 8 pixels of a tile row (k-blocks SBO = one tile row apart);
  //   B = x without horizontal halo, [18 rows][8 cols][Cin]; N block ky = one row further down (LBO = one row).
  const bool mfold = fuse == 3;
  const int whx = mfold ? TC_TW : WH;                   // columns of the staged x tile
  const uint32_t x_bytes = (uint32_t)c8n * HH * whx * 16;
  uint8_t* sG = smem;                                   // NBUF gy tiles, [co/8][128 pixels] x 16 B
  uint8_t* sX = smem + (size_t)NBUF * g_bytes;          // NBUF x halo tiles
  // barriers live at the end of the allocation (the host pads so that an A descriptor that starts in
  // the last gy slot never leaves the allocation)
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)NBUF * (g_bytes + x_bytes));
  uint64_t* empty = full + NBUF;
  uint64_t* done = empty + NBUF;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  // fuse == 2: SWAPPED orientation for narrow inputs (3*Cin <= 128): A = shifted x with M = (ky, ci) rows,
  // B = gy^T with N = Cout, one unit per filter column kx.  The 128-row MMA floor is then filled with
  // 3*Cin useful rows instead of Cout, which cuts the tensor-pipe time of the 16/32-channel layers 3x.
  const bool swapped = fuse == 2;
  const int units_total = mfold ? 1 : (fuse ? K : K * K);
  const int NU = swapped ? Cout : (fuse ? K * Cin : Cin);     // accumulator columns per unit
  const int unit0 = blockIdx.y * units_per_group;
  const int nunits = min(units_per_group, units_total - unit0);
  const int n_issuers = min(3, nunits);
  const int co_base = blockIdx.z * 128;
  const int co_cnt = min(128, Cout - co_base);
  const bool m64 = swapped ? (K * Cin <= 64) : mfold ? (K * co_cnt <= 64) : (Cout <= 64);
  const int g8n = co_cnt >> 3;
  const int tiles_x = (W + TC_TW - 1) / TC_TW, tiles_y = (H + TC_TH - 1) / TC_TH, tiles_img = tiles_x * tiles_y;
  const int total_tiles = N * tiles_img;
  const int T = (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  auto tile_coords = [&](int j, int& n, int& y0, int& x0) {
    const int tile = blockIdx.x + j * gridDim.x;
    n = tile / tiles_img;
    const int t2 = tile - n * tiles_img;
    y0 = (t2 / tiles_x) * TC_TH;
    x0 = (t2 % tiles_x) * TC_TW;
  };

  // Bias gradient (sum over pixels of gy) for free: warps 0-3 are idle during the main loop, so they add up the gy
  // tile that sits in shared memory anyway (CTAs of the first tap group only).  Replaces the separate ttg_channel_sum
  // pass over gy.
  const bool do_bias = gbias != nullptr && blockIdx.y == 0;
  float* s_bias = reinterpret_cast<float*>(tmem_slot + 4);        // [128] floats after the barriers
  if (do_bias && tid < 128) s_bias[tid] = 0.f;
  if (warp == 4) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
  if (tid == 0) {
    for (int i = 0; i < NBUF; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], (uint32_t)n_issuers + (do_bias ? 4u : 0u)); }
    mbar_init(done, (uint32_t)n_issuers);
    mbar_fence_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    if (do_bias) {
      // thread -> one 8-channel group and every ppg-th pixel of the tile: consecutive lanes read consecutive pixels
      const int ppg = 128 / g8n, g8 = tid / ppg, p0 = tid - g8 * ppg;
      float bs[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) bs[k] = 0.f;
      for (int it = 0; it < T; ++it) {
        const int s = it % NBUF;
        mbar_wait(&full[s], (uint32_t)(it / NBUF) & 1u);
        if (mfold) {
          // pixel-major swizzled tile with a one-column halo: pixel (row, col) at halo index row * 10 + col + 1
          const uint32_t gs = smem_u32(sG + (size_t)s * g_bytes);
          for (int p = p0; p < NPIX; p += ppg) {
            const uint32_t pa = gs + (uint32_t)(((p >> 3) * (TC_TW + 2) + (p & 7) + 1) * co_cnt * 2);
            uint4 v;
            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                         : "r"(pa + (uint32_t)((g8 ^ (int)((pa >> 7) & (uint32_t)(g8n - 1))) << 4)));
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) { bs[2 * k] += __uint_as_float(w4[k] << 16); bs[2 * k + 1] += __uint_as_float(w4[k] & 0xffff0000u); }
          }
        } else {
        const uint8_t* gt = sG + (size_t)s * g_bytes + (size_t)g8 * NPIX * 16;
        for (int p = p0; p < NPIX; p += ppg) {
          const uint4 v = *reinterpret_cast<const uint4*>(gt + (size_t)p * 16);
          const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) { bs[2 * k] += __uint_as_float(w4[k] << 16); bs[2 * k + 1] += __uint_as_float(w4[k] & 0xffff0000u); }
        }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) atomicAdd(&s_bias[g8 * 8 + k], bs[k]);
    }
    if (T > 0) {
      { TTG_T0(); mbar_wait(done, 0); if (tid == 0) { TTG_T1(9, 0); } }
      tc_fence_after_sync();
      TTG_T0();
      // accumulator row -> TMEM lane: M=128: row = lane; M=64: rows 16w..16w+15 live in lanes 32w..32w+15.
      // The partial sums go to a PACKED fp32 image with 16 consecutive accumulator columns contiguous, so a thread
      // issues four 16-byte vector reductions per TMEM load instead of sixteen scattered scalar atomics:
      //   normal / fused : gwp[tap][co][ci]      (columns = ci)
      //   swapped        : gwp[tap][ci][co]      (columns = co)
      // ttg_wgrad_unpack_kernel turns it into OIHW.
      const int row = m64 ? (warp * 16 + lane) : tid;
      const bool valid = (m64 ? lane < 16 : true) && row < (swapped ? K * Cin : mfold ? K * co_cnt : co_cnt);
      const int co = co_base + row;
      for (int t = 0; t < nunits; ++t) {
        const int u = unit0 + t;
        for (int c0 = 0; c0 < NU; c0 += 16) {
          uint32_t r[16];
          tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(t * NU + c0), r);
          tmem_ld_wait();
          if (!valid) continue;
          float* dst;
          if (swapped) {                              // row = ky*Cin + ci, column = output channel, unit = kx
            const int ky = row / Cin, ci = row - ky * Cin;
            dst = gw + ((long long)(ky * K + u) * Cin + ci) * Cout + co_base + c0;
          } else if (mfold) {                         // row = kx*Cout + co, column = ky*Cin + ci
            const int jb = row / co_cnt, cc = row - jb * co_cnt;           // M block j <-> filter column kx = 2 - j
            const int ky = c0 / Cin, ci0 = c0 - ky * Cin;
            dst = gw + ((long long)(ky * K + (2 - jb)) * Cout + cc) * Cin + ci0;
          } else {
            const int ky = fuse ? c0 / Cin : 0, ci0 = fuse ? c0 - ky * Cin : c0;
            const int tap = fuse ? ky * K + u : u;
            dst = gw + ((long long)tap * Cout + co) * Cin + ci0;
          }
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            asm volatile("red.global.v4.f32.add [%0], {%1,%2,%3,%4};" ::"l"(dst + j), "r"(r[j]), "r"(r[j + 1]), "r"(r[j + 2]), "r"(r[j + 3])
                         : "memory");
        }
      }
      if (tid == 0) { TTG_T1(10, 0); }
    }
  } else if (warp - 4 < n_issuers) {
    const int me = warp - 4;
    const uint32_t idesc = umma_idesc_bf16(m64 ? 64 : 128, NU, 1, 1);
    for (int it = 0; it < T; ++it) {
      const int s = it % NBUF;
      { TTG_T0(); mbar_wait(&full[s], (uint32_t)(it / NBUF) & 1u); if (lane == 0 && me == 0) { TTG_T1(11, it); } }
      tc_fence_after_sync();
      TTG_T0();
      // K steps that only cover rows below the image (tiles taller than an 8x8 feature map) are skipped
      int n_, y0_, x0_;
      tile_coords(it, n_, y0_, x0_);
      const int rmax = min(TC_TH / 2, (H - y0_ + 1) >> 1);
      const bool leader = elect_one();
      if (leader && mfold) {
        const uint32_t gpix = (uint32_t)co_cnt * 2, grow = (uint32_t)(TC_TW + 2) * gpix;       // bytes per gy pixel / tile row
        const uint32_t xrow = (uint32_t)TC_TW * (uint32_t)Cin * 2;                             // bytes per x tile row
        const uint64_t a0 = umma_desc_sw(smem_u32(sG + (size_t)s * g_bytes), gpix, grow, umma_swz_layout_for(co_cnt));
        const uint64_t b0 = umma_desc_sw(smem_u32(sX + (size_t)s * x_bytes), xrow, xrow, umma_swz_layout_for(Cin));
#pragma unroll
        for (int r = 0; r < TC_TH / 2; ++r)
          if (r < rmax)
            umma_bf16(tmem_base, a0 + (uint64_t)((2 * r * grow) >> 4), b0 + (uint64_t)((2 * r * xrow) >> 4), idesc,
                      (it == 0 && r == 0) ? 0u : 1u);
        umma_commit(&empty[s]);
        if (it == T - 1) umma_commit(done);
      } else if (leader && swapped) {
        // A = shifted x (MN-major): M groups = (ky, c8) WH units apart; B = gy^T (MN-major): N groups = co/8
        const uint64_t a0 = umma_desc(smem_u32(sX + (size_t)s * x_bytes), (uint32_t)(c8n * WH) * 16, WH * 16);
        const uint64_t b0 = umma_desc(smem_u32(sG + (size_t)s * g_bytes), TC_TW * 16, NPIX * 16);
        for (int t = me; t < nunits; t += 3) {
          const int kx = unit0 + t;
          const uint32_t dcol = tmem_base + (uint32_t)(t * NU);
#pragma unroll
          for (int r = 0; r < TC_TH / 2; ++r)
            if (r < rmax)
              umma_bf16(dcol, a0 + (uint64_t)(2 * r * c8n * WH + kx), b0 + (uint64_t)(2 * r * TC_TW), idesc,
                        (it == 0 && r == 0) ? 0u : 1u);
        }
        umma_commit(&empty[s]);
        if (it == T - 1) umma_commit(done);
      } else if (leader) {
        // A = gy^T (MN-major): channel groups SBO = 128 px x 16 B apart, pixels 16 B apart, rows (8 px) LBO apart
        const uint64_t a0 = umma_desc(smem_u32(sG + (size_t)s * g_bytes), TC_TW * 16, NPIX * 16);
        // B = shifted x (MN-major): N groups (c8, and ky when fused) WH units apart, halo rows c8n*WH units apart
        const uint64_t b0 = umma_desc(smem_u32(sX + (size_t)s * x_bytes), (uint32_t)(c8n * WH) * 16, WH * 16);
        for (int t = me; t < nunits; t += 3) {
          const int u = unit0 + t;
          const int ky = fuse ? 0 : u / K, kx = fuse ? u : u - ky * K;
          const uint32_t dcol = tmem_base + (uint32_t)(t * NU);
          const uint64_t bt = b0 + (uint64_t)(ky * c8n * WH + kx);
#pragma unroll
          for (int r = 0; r < TC_TH / 2; ++r)
            if (r < rmax)
              umma_bf16(dcol, a0 + (uint64_t)(2 * r * TC_TW), bt + (uint64_t)(2 * r * c8n * WH), idesc,
                        (it == 0 && r == 0) ? 0u : 1u);
        }
        umma_commit(&empty[s]);
        if (it == T - 1) umma_commit(done);
        if (me == 0) { TTG_T1(12, it); }
      }
      __syncwarp();
    }
  } else if (warp == 7 && elect_one()) {
    // ---- TMA producer: one tensor-map load for the x halo tile, one for the gy tile, per slot
    for (int j = 0; j < T; ++j) {
      const int s = j % NBUF;
      { TTG_T0(); if (j >= NBUF) mbar_wait(&empty[s], (uint32_t)((j / NBUF) - 1) & 1u); TTG_T1(13, j); }
      int n, y0, x0;
      tile_coords(j, n, y0, x0);
      const uint32_t bar = smem_u32(&full[s]);
      const uint32_t gbytes_tile = (uint32_t)g8n * NPIX * 16;
      if (mfold) {
        const uint32_t gtile = (uint32_t)(TC_TH * (TC_TW + 2) * co_cnt * 2);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(x_bytes + gtile) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
            ::"r"(smem_u32(sX + (size_t)s * x_bytes)), "l"(&tmap_x), "r"(0), "r"(x0), "r"(y0 - HALO), "r"(n), "r"(bar) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
            ::"r"(smem_u32(sG + (size_t)s * g_bytes)), "l"(&tmap_g), "r"(0), "r"(x0 - 1), "r"(y0), "r"(n), "r"(bar) : "memory");
        continue;
      }
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(x_bytes + gbytes_tile) : "memory");
      asm volatile(
          "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
          ::"r"(smem_u32(sX + (size_t)s * x_bytes)), "l"(&tmap_x), "r"(0), "r"(x0 - HALO), "r"(0), "r"(y0 - HALO), "r"(n), "r"(bar)
          : "memory");
      asm volatile(
          "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
          ::"r"(smem_u32(sG + (size_t)s * g_bytes)), "l"(&tmap_g), "r"(0), "r"(x0), "r"(y0), "r"(co_base >> 3), "r"(n), "r"(bar)
          : "memory");
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  if (do_bias && tid < co_cnt && co_base + tid < cout_real) atomicAdd(&gbias[co_base + tid], s_bias[tid]);
}

template <int K, int NBUF>
static int launch_wgrad_ws(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout, int upg, int fuse,
                           int cols, int g_bytes, int smem, dim3 grid, int cin_real, int cout_real, float* gbias, cudaStream_t st) {
  const ttg_encode_tiled_fn enc = ttg_get_encode_tiled();
  if (!enc) return ttg_no_encode_tiled("conv2d_wgrad_tc");
  constexpr int HALO = K / 2;
  CUtensorMap tx, tg;
  CUresult r1, r2;
  if (fuse == 3) {
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const cuuint64_t xd[4] = {(cuuint64_t)cin_real, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t xs[3] = {(cuuint64_t)cin_real * 2, (cuuint64_t)W * cin_real * 2, (cuuint64_t)H * W * cin_real * 2};
    const cuuint32_t xb[4] = {(cuuint32_t)Cin, TC_TW, (cuuint32_t)(TC_TH + 2 * HALO), 1};
    const cuuint64_t gd[4] = {(cuuint64_t)cout_real, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t gs[3] = {(cuuint64_t)cout_real * 2, (cuuint64_t)W * cout_real * 2, (cuuint64_t)H * W * cout_real * 2};
    const cuuint32_t gb[4] = {(cuuint32_t)Cout, TC_TW + 2, TC_TH, 1};
    auto swz_of = [](int c) { return c == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : c == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B; };
    r1 = enc(&tx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), xd, xs, xb, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             swz_of(Cin), CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    r2 = enc(&tg, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(gy), gd, gs, gb, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             swz_of(Cout), CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  } else {
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const cuuint64_t xd[5] = {8, (cuuint64_t)W, (cuuint64_t)(cin_real / 8), (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t xs[4] = {(cuuint64_t)cin_real * 2, 16, (cuuint64_t)W * cin_real * 2, (cuuint64_t)H * W * cin_real * 2};
    const cuuint32_t xb[5] = {8, (cuuint32_t)(TC_TW + 2 * HALO), (cuuint32_t)(Cin / 8), (cuuint32_t)(TC_TH + 2 * HALO), 1};
    const int g8n = (Cout < 128 ? Cout : 128) / 8;
    const cuuint64_t gd[5] = {8, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)(cout_real / 8), (cuuint64_t)N};
    const cuuint64_t gs[4] = {(cuuint64_t)cout_real * 2, (cuuint64_t)W * cout_real * 2, 16, (cuuint64_t)H * W * cout_real * 2};
    const cuuint32_t gb[5] = {8, TC_TW, TC_TH, (cuuint32_t)g8n, 1};
    r1 = enc(&tx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x), xd, xs, xb, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    r2 = enc(&tg, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(gy), gd, gs, gb, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS)
    return ttg_set_error(TTG_ERR_CUDA, "conv2d_wgrad_tc: cuTensorMapEncodeTiled failed (%d, %d)", (int)r1, (int)r2);
  static int smem_set = 0;
  if (smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_tc_ws_kernel<K, NBUF>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return ttg_set_error(TTG_ERR_CUDA, "conv2d_wgrad_tc: smem attribute: %s", cudaGetErrorString(e));
    smem_set = smem;
  }
  conv_wgrad_tc_ws_kernel<K, NBUF><<<grid, 256, smem, st>>>(gw, N, H, W, Cin, Cout, upg, fuse, cols, g_bytes, cout_real, tx, tg, gbias);
  TTG_CHECK_LAUNCH("conv2d_wgrad_tc_ws");
  return TTG_OK;
}

static int g_wgrad_tc_smem[2] = {0, 0};

// packed partial-sum image -> OIHW fp32 (layout 0: gwp[tap][co][ci], 1: gwp[tap][ci][co]; padded sizes CoutP x CinP)
// acc != 0: added to gw (a view of the flat .grad buffer) instead of overwriting it
__global__ void ttg_wgrad_unpack_kernel(const float* __restrict__ gwp, float* __restrict__ gw, int Cout, int Cin, int CoutP, int CinP,
                                        int taps, int layout, int acc) {
  const int total = Cout * Cin * taps;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int tap = i % taps, ci = (i / taps) % Cin, co = i / (taps * Cin);
    const float v = layout == 0 ? gwp[((long long)tap * CoutP + co) * CinP + ci] : gwp[((long long)tap * CinP + ci) * CoutP + co];
    gw[i] = acc ? gw[i] + v : v;
  }
}
static inline int ttg_pad16(int c) { return c <= 8 ? 16 : c; }
extern "C" size_t ttg_conv2d_wgrad_tc_workspace_bytes(int Cin, int Cout, int ksize) {
  return sizeof(float) * (size_t)ttg_pad16(Cin) * ttg_pad16(Cout) * ksize * ksize + 16 + 8 * 256 + 16;   // + channel-sum scratch (fp64 [C])
}

extern "C" int ttg_channel_sum_acc(const void* x, long long M, int C, float* out, int accumulate, void* workspace, int dtype, void* stream);
static int wgrad_tc_core(const void* x, const void* gy, float* gw, float* gbias, int N, int H, int W, int Cin, int Cout,
                         int cin_real, int cout_real, int ksize, void* workspace, void* stream, int accumulate = 0);
extern "C" int ttg_conv2d_wgrad_tc_ex(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout,
                                      int cin_real, int cout_real, int ksize, void* workspace, void* stream) {
  return wgrad_tc_core(x, gy, gw, nullptr, N, H, W, Cin, Cout, cin_real, cout_real, ksize, workspace, stream);
}
extern "C" int ttg_conv2d_wgrad_tc(const void* x, const void* gy, float* gw, int N, int H, int W, int Cin, int Cout,
                                   int ksize, void* workspace, void* stream) {
  return ttg_conv2d_wgrad_tc_ex(x, gy, gw, N, H, W, Cin, Cout, Cin, Cout, ksize, workspace, stream);
}
// wgrad + bias gradient (gbias[co] = sum over pixels of gy[., co], fp32) in one pass over gy: the idle warps of the
// TMA-fed wgrad kernel add up the gy tiles while the tensor cores consume them (Conv2d bias gradient of
// convolution_backward).  The Cin = 256 layers (conv_wgrad_tc_kernel) use ttg_channel_sum internally instead.
extern "C" int ttg_conv2d_wgrad_bias_tc_ex(const void* x, const void* gy, float* gw, float* gbias, int N, int H, int W, int Cin,
                                           int Cout, int cin_real, int cout_real, int ksize, void* workspace, void* stream) {
  TTG_REQUIRE(gbias != nullptr, "conv2d_wgrad_bias_tc: gbias is required");
  return wgrad_tc_core(x, gy, gw, gbias, N, H, W, Cin, Cout, cin_real, cout_real, ksize, workspace, stream);
}
// gw += / gbias += variant: the weight (and optional bias) gradient is accumulated into the caller's buffers
// (views of the flat .grad buffer of the model), which removes autograd's per-parameter add kernels.
// flags: bit 0 = accumulate (always set by this entry point's callers), bit 1 = the workspace is already all zero
extern "C" int ttg_conv2d_wgrad_tc_acc(const void* x, const void* gy, float* gw, float* gbias, int N, int H, int W, int Cin,
                                       int Cout, int cin_real, int cout_real, int ksize, int flags, void* workspace,
                                       void* stream) {
  return wgrad_tc_core(x, gy, gw, gbias, N, H, W, Cin, Cout, cin_real, cout_real, ksize, workspace, stream, flags | 1);
}
static int wgrad_tc_core(const void* x, const void* gy, float* gw, float* gbias, int N, int H, int W, int Cin, int Cout,
                         int cin_real, int cout_real, int ksize, void* workspace, void* stream, int accumulate) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "conv2d_wgrad_tc: workspace must be 16-byte aligned");
  float* gwp = reinterpret_cast<float*>(workspace);
  const bool padded = cin_real != Cin || cout_real != Cout;
  TTG_REQUIRE((cin_real == Cin || (cin_real == 8 && Cin == 16)) && (cout_real == Cout || (cout_real == 8 && Cout == 16)),
              "conv2d_wgrad_tc: channel padding supports 8-channel staging tensors (ttg_pad_channels8) only");
  TTG_REQUIRE(ksize == 1 || ksize == 3, "conv2d_wgrad_tc: ksize %d unsupported", ksize);
  TTG_REQUIRE(Cin % 16 == 0 && Cout % 16 == 0 && Cin >= 16 && Cout >= 16 && Cin <= 256 && Cout <= 256,
              "conv2d_wgrad_tc: channels must be multiples of 16 in [16,256] (got %d -> %d)", Cin, Cout);
  const int taps = ksize * ksize;
  int tpg = 512 / Cin;                 // accumulator columns: taps_per_group * Cin <= 512
  if (tpg > taps) tpg = taps;
  const int groups = (taps + tpg - 1) / tpg;
  const int halves = (Cout + 127) / 128;
  const int halo = ksize / 2;
  const int HP = (TC_TW + 2 * halo) * (TC_TH + 2 * halo);
  const int smem = (Cin / 8) * HP * 16 + 16 * TC_TH * TC_TW * 16 + 64;
  const long long tiles = (long long)N * ((H + TC_TH - 1) / TC_TH) * ((W + TC_TW - 1) / TC_TW);
  int per_sm = (200 * 1024) / smem;
  const int cols = (int)tmem_cols_for(tpg * Cin);
  if (per_sm > 512 / cols) per_sm = 512 / cols;
  if (per_sm < 1) per_sm = 1;
  {
    // persistent warp-specialised variant when at least two (x, gy) slots fit in shared memory
    // measured: the swapped orientation only pays when the input is wider than the output (32->16: 204 -> 175 us);
    // for Cin <= Cout the MMA count, not the MMA shape, is what bounds these narrow layers
    // kx folded into M and ky into N (fuse 3): 8 MMAs per tile instead of 24 for the narrow layers, which are bound
    // by the MMA count (16->16 @128^2: 131 us with 24 small MMAs per 128 pixels)
    const bool mfold = ksize == 3 && (Cout == 16 || Cout == 32) && (Cin == 16 || Cin == 32 || Cin == 64);
    const bool swap_ok = !mfold && ksize == 3 && 3 * Cin <= 128 && Cout <= 128 && Cin > Cout;
    const int fuse = mfold ? 3 : swap_ok ? 2 : ((ksize == 3 && 3 * Cin <= 256) ? 1 : 0);
    const int units_total = mfold ? 1 : fuse ? 3 : taps;
    const int NU = swap_ok ? Cout : (fuse ? 3 * Cin : Cin);
    int upg = 512 / NU;
    if (upg > units_total) upg = units_total;
    const int wgroups = (units_total + upg - 1) / upg;
    upg = (units_total + wgroups - 1) / wgroups;                 // balance units over the groups
    const int wcols = (int)tmem_cols_for(upg * NU);
    const int x_bytes = mfold ? (Cin / 8) * (TC_TH + 2) * TC_TW * 16 : (Cin / 8) * HP * 16;
    const int g_bytes = mfold ? TC_TH * (TC_TW + 2) * Cout * 2 : ((Cout < 128 ? Cout : 128) / 8) * TC_TH * TC_TW * 16;
    // bytes an M=64 / M=128 A descriptor spans from the start of a gy slot (mfold: the tile plus the three extra pixels
    // the padding M block reaches past its end)
    const int reach = swap_ok ? 0 : mfold ? g_bytes + 4 * Cout * 2 : (Cout <= 64 ? 8 : 16) * TC_TH * TC_TW * 16;
    // swapped orientation: the padding rows of the A operand (ky = 3) reach one halo row past the last x slot
    const int xpad = swap_ok ? 2 * (Cin / 8) * (TC_TW + 2 * halo) * 16 : 0;
    int nbuf = (200 * 1024 - reach) / (x_bytes + g_bytes);
    const int nbuf_cap = mfold ? 8 : 4;     // the folded variant's pipeline is latency bound: deeper ring
    if (nbuf > nbuf_cap) nbuf = nbuf_cap;
    if (nbuf == 5) nbuf = 4;
    if (nbuf == 7) nbuf = 6;
    if (nbuf >= 2) {
      int wper_sm = 512 / wcols;
      int body = nbuf * (x_bytes + g_bytes);
      const int need = (nbuf - 1) * g_bytes + reach;
      if (body < need) body = need;
      const int wsmem = body + xpad + 1024;          // barriers + the bias partial sums
      if (wper_sm > (220 * 1024) / wsmem) wper_sm = (220 * 1024) / wsmem;
      if (wper_sm > 4) wper_sm = 4;
      if (wper_sm < 1) wper_sm = 1;
      long long wsplits = (long long)ttg_num_sms() * wper_sm / (wgroups * halves);
      if (wsplits < 1) wsplits = 1;
      if (wsplits > tiles) wsplits = tiles;
      if (!(accumulate & 2)) cudaMemsetAsync(gwp, 0, sizeof(float) * (size_t)Cout * Cin * taps, st);
      if (gbias && !(accumulate & 1)) cudaMemsetAsync(gbias, 0, sizeof(float) * (size_t)cout_real, st);
      dim3 wgrid((unsigned)wsplits, wgroups, halves);
#define TTG_WG(KK, NB) launch_wgrad_ws<KK, NB>(x, gy, gwp, N, H, W, Cin, Cout, upg, fuse, wcols, g_bytes, wsmem, wgrid, cin_real, cout_real, gbias, st)
      int rc;
      if (ksize == 3) rc = nbuf == 8 ? TTG_WG(3, 8) : nbuf == 6 ? TTG_WG(3, 6) : nbuf == 4 ? TTG_WG(3, 4) : nbuf == 3 ? TTG_WG(3, 3) : TTG_WG(3, 2);
      else rc = nbuf == 4 ? TTG_WG(1, 4) : nbuf == 3 ? TTG_WG(1, 3) : TTG_WG(1, 2);
#undef TTG_WG
      if (rc != TTG_OK) return rc;
      const int total = cout_real * cin_real * taps;
      ttg_wgrad_unpack_kernel<<<ttg_grid_for(total, 256), 256, 0, st>>>(gwp, gw, cout_real, cin_real, Cout, Cin, taps, swap_ok ? 1 : 0, accumulate & 1);
      TTG_CHECK_LAUNCH("conv2d_wgrad_unpack");
      return TTG_OK;
    }
  }
  TTG_REQUIRE(!padded, "conv2d_wgrad_tc: padded layers must fit the persistent kernel");
  long long splits = (long long)ttg_num_sms() * per_sm / (groups * halves);
  if (splits < 1) splits = 1;
  if (splits > tiles) splits = tiles;
  const int ki = ksize == 3 ? 1 : 0;
  if (smem > g_wgrad_tc_smem[ki]) {
    cudaError_t e = ksize == 3
        ? cudaFuncSetAttribute(conv_wgrad_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
        : cudaFuncSetAttribute(conv_wgrad_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return ttg_set_error(TTG_ERR_CUDA, "conv2d_wgrad_tc: smem attribute: %s", cudaGetErrorString(e));
    g_wgrad_tc_smem[ki] = smem;
  }
  if (!(accumulate & 1)) cudaMemsetAsync(gw, 0, sizeof(float) * (size_t)Cout * Cin * taps, st);
  dim3 grid((unsigned)splits, groups, halves);
  if (ksize == 3)
    conv_wgrad_tc_kernel<3><<<grid, 128, smem, st>>>((const bf16*)x, (const bf16*)gy, gw, N, H, W, Cin, Cout, tpg, cols);
  else
    conv_wgrad_tc_kernel<1><<<grid, 128, smem, st>>>((const bf16*)x, (const bf16*)gy, gw, N, H, W, Cin, Cout, tpg, cols);
  TTG_CHECK_LAUNCH("conv2d_wgrad_tc");
  if (gbias) {
    void* scratch = reinterpret_cast<uint8_t*>(workspace) + ((sizeof(float) * (size_t)Cout * Cin * taps + 15) & ~(size_t)15);
    return ttg_channel_sum_acc(gy, (long long)N * H * W, cout_real, gbias, accumulate, scratch, TTG_BF16, stream);
  }
  return TTG_OK;
}

// ------------------------------------------------------------------ 8-channel staging of the RGB tensors
// The image-like tensors (3 channels: D's first conv input, the image gradient, G's output conv) are copied into
// 8-channel pixels (channels >= c_real zero) so that the tensor-core kernels fetch / store them with the same TMA
// tiles and 16-byte stores as every other layer; the copy costs one extra pass over a tensor that is 5x smaller than
// its 16-channel neighbour.
__global__ void pad_channels8_kernel(const unsigned short* __restrict__ x, uint4* __restrict__ y, long long npix, int c_real) {
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (long long)gridDim.x * blockDim.x) {
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    const unsigned short* src = x + p * c_real;
    for (int c = 0; c < c_real; ++c) w[c >> 1] |= (uint32_t)src[c] << (16 * (c & 1));
    y[p] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
__global__ void unpad_channels8_kernel(const uint4* __restrict__ y8, unsigned short* __restrict__ y, long long npix, int c_real) {
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (long long)gridDim.x * blockDim.x) {
    const uint4 v = y8[p];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    unsigned short* dst = y + p * c_real;
    for (int c = 0; c < c_real; ++c) dst[c] = (unsigned short)(w[c >> 1] >> (16 * (c & 1)));
  }
}
extern "C" int ttg_pad_channels8(const void* x, void* y8, long long npix, int c_real, void* stream) {
  TTG_REQUIRE(c_real >= 1 && c_real <= 8 && npix >= 0, "pad_channels8: 1..8 channels");
  TTG_REQUIRE((reinterpret_cast<uintptr_t>(y8) & 15) == 0, "pad_channels8: destination must be 16-byte aligned");
  if (npix == 0) return TTG_OK;
  pad_channels8_kernel<<<ttg_grid_occ(pad_channels8_kernel, npix, 256), 256, 0, (cudaStream_t)stream>>>(
      (const unsigned short*)x, (uint4*)y8, npix, c_real);
  TTG_CHECK_LAUNCH("pad_channels8");
  return TTG_OK;
}
extern "C" int ttg_unpad_channels8(const void* y8, void* y, long long npix, int c_real, void* stream) {
  TTG_REQUIRE(c_real >= 1 && c_real <= 8 && npix >= 0, "unpad_channels8: 1..8 channels");
  TTG_REQUIRE((reinterpret_cast<uintptr_t>(y8) & 15) == 0, "unpad_channels8: source must be 16-byte aligned");
  if (npix == 0) return TTG_OK;
  unpad_channels8_kernel<<<ttg_grid_occ(unpad_channels8_kernel, npix, 256), 256, 0, (cudaStream_t)stream>>>(
      (const uint4*)y8, (unsigned short*)y, npix, c_real);
  TTG_CHECK_LAUNCH("unpad_channels8");
  return TTG_OK;
}

// ------------------------------------------------------------------ all filters of a model in one launch
// table: n_entries rows of 9 int64: {src offset (floats), dst offset (bytes), Cout, Cin, CoutP, CinP, k, mode,
// first block}; blocks [first block, next first block) pack entry e.  Replaces ~50 pack_weight launches per step
// (every filter, both operand orientations) by one launch after each optimiser update.
__global__ void pack_weights_multi_kernel(const float* __restrict__ flat, unsigned char* __restrict__ packed,
                                          const long long* __restrict__ table, int n_entries) {
  __shared__ int s_e;
  if (threadIdx.x == 0) {
    int e = 0;
    while (e + 1 < n_entries && (long long)blockIdx.x >= table[(e + 1) * 9 + 8]) ++e;
    s_e = e;
  }
  __syncthreads();
  const long long* t = table + (long long)s_e * 9;
  const float* w = flat + t[0];
  bf16* wp = reinterpret_cast<bf16*>(packed + t[1]);
  const int Cout = (int)t[2], Cin = (int)t[3], CoutP = (int)t[4], CinP = (int)t[5], k = (int)t[6], mode = (int)t[7];
  const int i = (int)((long long)blockIdx.x - t[8]) * blockDim.x + threadIdx.x;
  if (i >= Cout * Cin * k * k) return;
  const int kx = i % k, ky = (i / k) % k, ci = (i / (k * k)) % Cin, co = i / (k * k * Cin);
  const bf16 v = __float2bfloat16_rn(w[i]);
  if (mode == 0) {
    const int tap = ky * k + kx;
    wp[(((long long)tap * (CinP / 8) + ci / 8) * CoutP + co) * 8 + (ci % 8)] = v;
  } else {
    const int tap = (k - 1 - ky) * k + (k - 1 - kx);
    wp[(((long long)tap * (CoutP / 8) + co / 8) * CinP + ci) * 8 + (co % 8)] = v;
  }
}
extern "C" int ttg_pack_weights_multi(const float* flat, void* packed, const long long* table, int n_entries,
                                      int total_blocks, void* stream) {
  TTG_REQUIRE(n_entries >= 0 && total_blocks >= 0, "pack_weights_multi: bad table");
  if (n_entries == 0 || total_blocks == 0) return TTG_OK;
  pack_weights_multi_kernel<<<total_blocks, 256, 0, (cudaStream_t)stream>>>(flat, (unsigned char*)packed, table, n_entries);
  TTG_CHECK_LAUNCH("pack_weights_multi");
  return TTG_OK;
}
