// Spatial resampling and glue kernels over NHWC activations (all HBM streams):
//   2x2 sum-pool (nn.AvgPool2d(2), reference blocks/discriminator.py:67, and the
//   adjoint of nearest upsample), nearest x2 upsample (F.interpolate, reference
//   blocks/generator.py:58, and the adjoint of avg-pool), bilinear 1/2 with
//   align_corners=True and its transpose (blocks/discriminator.py:55-57,92),
//   residual add (generator.py:62, discriminator.py:95), sum over H,W
//   (discriminator.py:143,166), NCHW fp32 <-> NHWC conversions at the module
//   boundary, tanh (generator.py:126).
#include "chanops.cuh"

template <typename T, int V> struct Ld {
  static __device__ __forceinline__ void ld(const T* p, float* f) {
    if constexpr (V == 1) f[0] = to_f(*p); else { Vec<T> q; q.load(p); q.unpack(f); }
  }
  static __device__ __forceinline__ void st(T* p, const float* f) {
    if constexpr (V == 1) *p = from_f<T>(f[0]); else { Vec<T> q; q.pack(f); q.store(p); }
  }
};

template <typename T> static inline bool vec2_ok(int C, const void* a, const void* b) {
  return C % Vec<T>::N == 0 && !((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15);
}

// y[n,oy,ox,c] = scale * sum_{2x2} x[n,2oy+dy,2ox+dx,c]
template <typename T, int V>
__global__ void pool2_kernel(const T* __restrict__ x, T* __restrict__ y, int N, int Ho, int Wo, int C, float scale) {
  const int cv = C / V;
  const long long total = (long long)N * Ho * Wo * cv;
  const int Wi = Wo * 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % cv) * V; long long p = i / cv;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    const T* src = x + (((long long)n * Ho * 2 + oy * 2) * Wi + ox * 2) * C + c;
    float a[V], b[V], s[V];
    Ld<T, V>::ld(src, a); Ld<T, V>::ld(src + C, b);
#pragma unroll
    for (int j = 0; j < V; ++j) s[j] = a[j] + b[j];
    Ld<T, V>::ld(src + (long long)Wi * C, a); Ld<T, V>::ld(src + (long long)Wi * C + C, b);
#pragma unroll
    for (int j = 0; j < V; ++j) s[j] = (s[j] + a[j] + b[j]) * scale;
    Ld<T, V>::st(y + (((long long)n * Ho + oy) * Wo + ox) * C + c, s);
  }
}
__global__ void pool2_bf16x8_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, unsigned total, unsigned Wo, unsigned cv, float scale);
static inline bool ttg_bf16x8_ok(int dtype, int C, const void* a, const void* b, long long items);
extern "C" int ttg_pool2_sum(const void* x, void* y, int N, int Ho, int Wo, int C, float scale, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (ttg_bf16x8_ok(dtype, C, x, y, (long long)N * Ho * Wo * (C / 8) * 4)) {
    const long long total = (long long)N * Ho * Wo * (C / 8);
    if (total == 0) return TTG_OK;
    pool2_bf16x8_kernel<<<ttg_grid_occ(pool2_bf16x8_kernel, total, 256, 256), 256, 0, st>>>(
        (const uint4*)x, (uint4*)y, (unsigned)total, (unsigned)Wo, (unsigned)(C / 8), scale);
    TTG_CHECK_LAUNCH("pool2_sum");
    return TTG_OK;
  }
  TTG_DISPATCH(dtype, {
    if (vec2_ok<T>(C, x, y)) { pool2_kernel<T, Vec<T>::N><<<ttg_grid_occ(pool2_kernel<T, Vec<T>::N>, (long long)N * Ho * Wo * (C / Vec<T>::N), 256, 256), 256, 0, st>>>((const T*)x, (T*)y, N, Ho, Wo, C, scale); }
    else { pool2_kernel<T, 1><<<ttg_grid_occ(pool2_kernel<T, 1>, (long long)N * Ho * Wo * C, 256, 256), 256, 0, st>>>((const T*)x, (T*)y, N, Ho, Wo, C, scale); }
  });
  TTG_CHECK_LAUNCH("pool2_sum");
  return TTG_OK;
}

// y[n,oy,ox,c] = scale * x[n,oy/2,ox/2,c]
template <typename T, int V>
__global__ void upsample2_kernel(const T* __restrict__ x, T* __restrict__ y, int N, int Hi, int Wi, int C, float scale) {
  const int cv = C / V; const int Ho = Hi * 2, Wo = Wi * 2;
  const long long total = (long long)N * Ho * Wo * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % cv) * V; long long p = i / cv;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    float a[V];
    Ld<T, V>::ld(x + (((long long)n * Hi + (oy >> 1)) * Wi + (ox >> 1)) * C + c, a);
#pragma unroll
    for (int j = 0; j < V; ++j) a[j] *= scale;
    Ld<T, V>::st(y + (((long long)n * Ho + oy) * Wo + ox) * C + c, a);
  }
}
// bf16 fast path: one thread = one 16-byte INPUT unit -> four 16-byte stores (the 2x2 replicas), 32-bit index
// arithmetic, two units in flight per thread.  (The generic kernel spends ~300 instructions per unit on 64-bit
// div/mod and re-reads every input unit four times.)
__device__ __forceinline__ uint4 ttg_scale_bf16x8(uint4 v, float scale) {
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); h[i] = __floats2bfloat162_rn(f.x * scale, f.y * scale); }
  return v;
}
__global__ void __launch_bounds__(256) upsample2_bf16x8_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, unsigned total,
                                                               unsigned Wi, unsigned cv, float scale) {
  const unsigned stride = gridDim.x * blockDim.x, rowo = 2u * Wi * cv;
  for (unsigned i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < total; i0 += 2u * stride) {
    const unsigned i1 = i0 + stride;
    const bool two = i1 < total;
    uint4 v0 = x[i0], v1 = two ? x[i1] : make_uint4(0u, 0u, 0u, 0u);
    if (scale != 1.f) { v0 = ttg_scale_bf16x8(v0, scale); if (two) v1 = ttg_scale_bf16x8(v1, scale); }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (u == 1 && !two) break;
      const unsigned i = u ? i1 : i0;
      const uint4 v = u ? v1 : v0;
      const unsigned c8 = i % cv, p = i / cv, xi = p % Wi, q = p / Wi;          // q = n * Hi + yi
      uint4* o = y + ((size_t)q * 2u * rowo + (size_t)(2u * xi) * cv + c8);
      o[0] = v; o[cv] = v; o[rowo] = v; o[rowo + cv] = v;
    }
  }
}
__global__ void __launch_bounds__(256) pool2_bf16x8_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, unsigned total,
                                                           unsigned Wo, unsigned cv, float scale) {
  const unsigned stride = gridDim.x * blockDim.x, rowi = 2u * Wo * cv;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const unsigned c8 = i % cv, p = i / cv, xo = p % Wo, q = p / Wo;              // q = n * Ho + oy
    const uint4* src = x + ((size_t)q * 2u * rowi + (size_t)(2u * xo) * cv + c8);
    const uint4 a = src[0], b = src[cv], c = src[rowi], d = src[rowi + cv];
    const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&a);
    const __nv_bfloat162* hb = reinterpret_cast<const __nv_bfloat162*>(&b);
    const __nv_bfloat162* hc = reinterpret_cast<const __nv_bfloat162*>(&c);
    const __nv_bfloat162* hd = reinterpret_cast<const __nv_bfloat162*>(&d);
    uint4 o;
    __nv_bfloat162* ho = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fa = __bfloat1622float2(ha[j]), fb = __bfloat1622float2(hb[j]), fc = __bfloat1622float2(hc[j]), fd = __bfloat1622float2(hd[j]);
      ho[j] = __floats2bfloat162_rn((((fa.x + fb.x) + fc.x) + fd.x) * scale, (((fa.y + fb.y) + fc.y) + fd.y) * scale);
    }
    y[i] = o;
  }
}
static inline bool ttg_bf16x8_ok(int dtype, int C, const void* a, const void* b, long long items) {
  return dtype == TTG_BF16 && C % 8 == 0 && items < (1ll << 31) - (1ll << 24) &&
         !((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15);
}
extern "C" int ttg_upsample2(const void* x, void* y, int N, int Hi, int Wi, int C, float scale, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (ttg_bf16x8_ok(dtype, C, x, y, (long long)N * Hi * Wi * (C / 8) * 4)) {
    const long long total = (long long)N * Hi * Wi * (C / 8);
    if (total == 0) return TTG_OK;
    upsample2_bf16x8_kernel<<<ttg_grid_occ(upsample2_bf16x8_kernel, total, 512, 256), 256, 0, st>>>(
        (const uint4*)x, (uint4*)y, (unsigned)total, (unsigned)Wi, (unsigned)(C / 8), scale);
    TTG_CHECK_LAUNCH("upsample2");
    return TTG_OK;
  }
  TTG_DISPATCH(dtype, {
    if (vec2_ok<T>(C, x, y)) { upsample2_kernel<T, Vec<T>::N><<<ttg_grid_occ(upsample2_kernel<T, Vec<T>::N>, (long long)N * Hi * Wi * 4 * (C / Vec<T>::N), 256, 256), 256, 0, st>>>((const T*)x, (T*)y, N, Hi, Wi, C, scale); }
    else { upsample2_kernel<T, 1><<<ttg_grid_occ(upsample2_kernel<T, 1>, (long long)N * Hi * Wi * 4 * C, 256, 256), 256, 0, st>>>((const T*)x, (T*)y, N, Hi, Wi, C, scale); }
  });
  TTG_CHECK_LAUNCH("upsample2");
  return TTG_OK;
}

// Bilinear, output size = input/2, align_corners=True: src = dst * (in-1)/(out-1).
__device__ __forceinline__ void bil_src(int o, int in, int out, int& i0, int& i1, float& w1) {
  float scale = out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f;
  float s = scale * (float)o;
  i0 = (int)s; if (i0 > in - 1) i0 = in - 1;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  w1 = s - (float)i0;
}
template <typename T, int V>
__global__ void bilinear_down_kernel(const T* __restrict__ x, T* __restrict__ y, int N, int Hi, int Wi, int C) {
  const int cv = C / V; const int Ho = Hi / 2, Wo = Wi / 2;
  const long long total = (long long)N * Ho * Wo * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % cv) * V; long long p = i / cv;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    int y0, y1, x0, x1; float wy, wx;
    bil_src(oy, Hi, Ho, y0, y1, wy); bil_src(ox, Wi, Wo, x0, x1, wx);
    const T* b = x + (long long)n * Hi * Wi * C + c;
    float a00[V], a01[V], a10[V], a11[V], o[V];
    Ld<T, V>::ld(b + ((long long)y0 * Wi + x0) * C, a00); Ld<T, V>::ld(b + ((long long)y0 * Wi + x1) * C, a01);
    Ld<T, V>::ld(b + ((long long)y1 * Wi + x0) * C, a10); Ld<T, V>::ld(b + ((long long)y1 * Wi + x1) * C, a11);
#pragma unroll
    for (int j = 0; j < V; ++j)
      o[j] = (1.f - wy) * ((1.f - wx) * a00[j] + wx * a01[j]) + wy * ((1.f - wx) * a10[j] + wx * a11[j]);
    Ld<T, V>::st(y + (((long long)n * Ho + oy) * Wo + ox) * C + c, o);
  }
}
extern "C" int ttg_bilinear_down_fwd(const void* x, void* y, int N, int Hi, int Wi, int C, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(Hi % 2 == 0 && Wi % 2 == 0, "bilinear_down: odd input size %dx%d", Hi, Wi);
  TTG_DISPATCH(dtype, {
    if (vec2_ok<T>(C, x, y)) { bilinear_down_kernel<T, Vec<T>::N><<<ttg_grid_occ(bilinear_down_kernel<T, Vec<T>::N>, (long long)N * (Hi / 2) * (Wi / 2) * (C / Vec<T>::N), 256, 256), 256, 0, st>>>((const T*)x, (T*)y, N, Hi, Wi, C); }
    else { bilinear_down_kernel<T, 1><<<ttg_grid_occ(bilinear_down_kernel<T, 1>, (long long)N * (Hi / 2) * (Wi / 2) * C, 256, 256), 256, 0, st>>>((const T*)x, (T*)y, N, Hi, Wi, C); }
  });
  TTG_CHECK_LAUNCH("bilinear_down_fwd");
  return TTG_OK;
}

// Transpose of the above as a gather: gx[iy,ix] = sum over outputs whose footprint covers (iy,ix).
__device__ __forceinline__ int bil_candidates(int i, int in, int out, int* oidx, float* w) {
  // outputs o with i0(o)==i or i1(o)==i lie within +-1 of i*(out-1)/(in-1)
  int cnt = 0;
  int guess = in > 1 ? (int)((float)i * (float)(out - 1) / (float)(in - 1)) : 0;
  for (int o = guess - 1; o <= guess + 2; ++o) {
    if (o < 0 || o >= out) continue;
    int i0, i1; float w1; bil_src(o, in, out, i0, i1, w1);
    float ww = 0.f;
    if (i0 == i) ww += 1.f - w1;
    if (i1 == i) ww += w1;
    if (i0 == i || i1 == i) { oidx[cnt] = o; w[cnt] = ww; ++cnt; }
  }
  return cnt;
}
// one thread per input pixel: the (<= 3 x 3) contributing outputs and their weights are found once,
// then every channel vector of the pixel is gathered with them
// `add` (optional, same shape as gx): gx = add + B^T gy — the gradient fan-in of a D block's input (skip branch + conv
// branch, discriminator.py:90-95) without a separate add pass.
// The contributing outputs and weights of a pixel depend on its row and on its column only: every block first builds
// the two candidate tables ((Hi + Wi) entries) in shared memory, instead of 8 divisions per pixel (109 us for the RGB
// gradient of a 256 x 128 x 128 batch, where a pixel is only 3 elements).
template <typename T, int V>
__global__ void bilinear_down_bwd_kernel(const T* __restrict__ gy, const T* __restrict__ add, T* __restrict__ gx, int N, int Hi, int Wi, int C, int pervec) {
  extern __shared__ __align__(16) unsigned char bil_smem[];
  int* s_n = reinterpret_cast<int*>(bil_smem);                  // [Hi + Wi] candidate counts (rows first, then columns)
  int* s_o = s_n + (Hi + Wi);                                   // [Hi + Wi][4] output indices
  float* s_w = reinterpret_cast<float*>(s_o + 4 * (Hi + Wi));   // [Hi + Wi][4] weights
  const int cv = C / V; const int Ho = Hi / 2, Wo = Wi / 2;
  for (int e = threadIdx.x; e < Hi + Wi; e += blockDim.x) {
    int o[4]; float w[4];
    const int n = e < Hi ? bil_candidates(e, Hi, Ho, o, w) : bil_candidates(e - Hi, Wi, Wo, o, w);
    s_n[e] = n;
    for (int k = 0; k < 4; ++k) { s_o[4 * e + k] = k < n ? o[k] : 0; s_w[4 * e + k] = k < n ? w[k] : 0.f; }
  }
  __syncthreads();
  // pervec: one work item = one channel vector of one pixel, so that the small deep layers (8 x 8 x 128 channels: 16 K
  // pixels) spread over the whole GPU; otherwise one item = one pixel (few vectors per pixel: the table lookups are
  // shared; measured faster for C <= 16: 82.6 vs 120 us on the RGB gradient, 32 vs 41 us at 64 x 64 x 16)
  const int per = pervec ? cv : 1;
  const long long total = (long long)N * Hi * Wi * per;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long p = i / per;
    const int v0 = pervec ? (int)(i % per) : 0, v1 = pervec ? v0 + 1 : cv;
    const int ix = (int)(p % Wi); const long long q = p / Wi; const int iy = (int)(q % Hi); const int n = (int)(q / Hi);
    const int ny = s_n[iy], nx = s_n[Hi + ix];
    const int* oys = s_o + 4 * iy; const int* oxs = s_o + 4 * (Hi + ix);
    const float* wys = s_w + 4 * iy; const float* wxs = s_w + 4 * (Hi + ix);
    const T* gbase = gy + (long long)n * Ho * Wo * C;
    for (int v = v0; v < v1; ++v) {
      float acc[V];
      if (add) Ld<T, V>::ld(add + p * C + v * V, acc);
      else {
#pragma unroll
        for (int j = 0; j < V; ++j) acc[j] = 0.f;
      }
      for (int a = 0; a < ny; ++a)
        for (int b = 0; b < nx; ++b) {
          const float w = wys[a] * wxs[b];
          float g[V];
          Ld<T, V>::ld(gbase + ((long long)oys[a] * Wo + oxs[b]) * C + v * V, g);
#pragma unroll
          for (int j = 0; j < V; ++j) acc[j] += w * g[j];
        }
      Ld<T, V>::st(gx + p * C + v * V, acc);
    }
  }
}
extern "C" int ttg_bilinear_down_bwd_add(const void* gy, const void* add, void* gx, int N, int Hi, int Wi, int C, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const long long pixels = (long long)N * Hi * Wi;
  const size_t bsm = (size_t)(Hi + Wi) * 9 * sizeof(int);           // candidate tables of the thread-per-pixel kernel
  TTG_REQUIRE(bsm <= 48 * 1024, "bilinear_down_bwd: image too large for the candidate tables (%d x %d)", Hi, Wi);
  const int pv = C >= 32 ? 1 : 0;
  TTG_DISPATCH(dtype, {
    if (vec2_ok<T>(C, gy, gx) && (add == nullptr || vec2_ok<T>(C, add, gx))) { bilinear_down_bwd_kernel<T, Vec<T>::N><<<ttg_grid_occ(bilinear_down_bwd_kernel<T, Vec<T>::N>, pixels * (pv ? C / Vec<T>::N : 1), 128 * 4, 128, bsm), 128, bsm, st>>>((const T*)gy, (const T*)add, (T*)gx, N, Hi, Wi, C, pv); }
    else { bilinear_down_bwd_kernel<T, 1><<<ttg_grid_occ(bilinear_down_bwd_kernel<T, 1>, pixels * (C > 16 ? C : 1), 128 * 4, 128, bsm), 128, bsm, st>>>((const T*)gy, (const T*)add, (T*)gx, N, Hi, Wi, C, C > 16 ? 1 : 0); }
  });
  TTG_CHECK_LAUNCH("bilinear_down_bwd");
  return TTG_OK;
}
extern "C" int ttg_bilinear_down_bwd(const void* gy, void* gx, int N, int Hi, int Wi, int C, int dtype, void* stream) {
  return ttg_bilinear_down_bwd_add(gy, nullptr, gx, N, Hi, Wi, C, dtype, stream);
}

// BatchNorm statistics of the tensor a join kernel writes (sum / sum of squares per channel of the ROUNDED values):
// every thread owns one fixed 8-channel group (256 % (C/8) == 0), keeps 16 partial sums in registers, lanes of the
// same group are combined with shuffles, then one shared atomic per (warp, channel) and one fp64 atomic per
// (block, channel).  The residual blocks' outputs feed the next block's BatchNorm (generator.py:38, discriminator.py:60).
template <typename T> __device__ __forceinline__ float ttg_rounded(float v) { return to_f(from_f<T>(v)); }
template <int V>
__device__ __forceinline__ void join_stats_flush(float (&sa)[V], float (&sq)[V], int cv, int C, double* __restrict__ stats) {
  extern __shared__ float s_join[];            // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) s_join[i] = 0.f;
  __syncthreads();
  const int g = threadIdx.x % cv;
  const bool pow2 = (cv & (cv - 1)) == 0 && cv <= 32;
  if (pow2) {
#pragma unroll
    for (int j = 0; j < V; ++j)
      for (int o = 16; o >= cv; o >>= 1) {
        sa[j] += __shfl_xor_sync(0xffffffffu, sa[j], o);
        sq[j] += __shfl_xor_sync(0xffffffffu, sq[j], o);
      }
  }
  if (!pow2 || (threadIdx.x & 31) < cv) {
#pragma unroll
    for (int j = 0; j < V; ++j) { atomicAdd(&s_join[g * V + j], sa[j]); atomicAdd(&s_join[C + g * V + j], sq[j]); }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) atomicAdd(&stats[i], (double)s_join[i]);
}

// out[n,oy,ox,c] = h[n,oy,ox,c] + s[n,oy/2,ox/2,c]   (residual add with the nearest-upsampled skip folded in)
template <typename T, int V, bool STATS = false>
__global__ void add_up2_kernel(const T* __restrict__ h, const T* __restrict__ s, T* __restrict__ y, int N, int Ho, int Wo, int C,
                               double* __restrict__ stats = nullptr) {
  const int cv = C / V; const int Hi = Ho / 2, Wi = Wo / 2;
  const long long total = (long long)N * Ho * Wo * cv;
  float sa[V], sq[V];
#pragma unroll
  for (int j = 0; j < V; ++j) sa[j] = sq[j] = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % cv) * V; long long p = i / cv;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    float a[V], b[V];
    Ld<T, V>::ld(h + i * V, a);
    Ld<T, V>::ld(s + (((long long)n * Hi + (oy >> 1)) * Wi + (ox >> 1)) * C + c, b);
#pragma unroll
    for (int j = 0; j < V; ++j) a[j] += b[j];
    Ld<T, V>::st(y + i * V, a);
    if constexpr (STATS) {
#pragma unroll
      for (int j = 0; j < V; ++j) { const float r = ttg_rounded<T>(a[j]); sa[j] += r; sq[j] += r * r; }
    }
  }
  if constexpr (STATS) join_stats_flush<V>(sa, sq, cv, C, stats);
}
// join + BatchNorm statistics of its output (sums: double[2C], see join_stats_flush); 16-byte vector path only
extern "C" int ttg_join_stats_supported(int C) { return C % 8 == 0 && 256 % (C / 8) == 0 && C <= 256; }
extern "C" int ttg_add_up2_stats(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, double* sums, int dtype,
                                 void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(Ho % 2 == 0 && Wo % 2 == 0, "add_up2: odd output size");
  TTG_REQUIRE(sums != nullptr && ttg_join_stats_supported(C), "add_up2_stats: unsupported channel count %d", C);
  cudaMemsetAsync(sums, 0, sizeof(double) * 2 * (size_t)C, st);
  TTG_DISPATCH(dtype, {
    TTG_REQUIRE((vec2_ok<T>(C, h, s) && vec2_ok<T>(C, y, y)) && Vec<T>::N == 8, "add_up2_stats: bf16, 16-byte aligned tensors");
    constexpr int V = 8;
    const size_t smem = sizeof(float) * 2 * C;
    add_up2_kernel<T, V, true><<<ttg_grid_occ(add_up2_kernel<T, V, true>, (long long)N * Ho * Wo * (C / V), 512, 256, smem), 256, smem, st>>>(
        (const T*)h, (const T*)s, (T*)y, N, Ho, Wo, C, sums);
  });
  TTG_CHECK_LAUNCH("add_up2_stats");
  return TTG_OK;
}
extern "C" int ttg_add_up2(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(Ho % 2 == 0 && Wo % 2 == 0, "add_up2: odd output size");
  TTG_DISPATCH(dtype, {
    if (vec2_ok<T>(C, h, s) && vec2_ok<T>(C, y, y)) { add_up2_kernel<T, Vec<T>::N><<<ttg_grid_occ(add_up2_kernel<T, Vec<T>::N>, (long long)N * Ho * Wo * (C / Vec<T>::N), 512, 256), 256, 0, st>>>((const T*)h, (const T*)s, (T*)y, N, Ho, Wo, C); }
    else { add_up2_kernel<T, 1><<<ttg_grid_occ(add_up2_kernel<T, 1>, (long long)N * Ho * Wo * C, 1024, 256), 256, 0, st>>>((const T*)h, (const T*)s, (T*)y, N, Ho, Wo, C); }
  });
  TTG_CHECK_LAUNCH("add_up2");
  return TTG_OK;
}

// out[n,oy,ox,c] = scale * sum_{2x2} h + s[n,oy,ox,c]   (AvgPool2d(2) of the conv path + skip, one pass)
template <typename T, int V, bool STATS = false>
__global__ void pool2_add_kernel(const T* __restrict__ h, const T* __restrict__ s, T* __restrict__ y, int N, int Ho, int Wo, int C, float scale,
                                 double* __restrict__ stats = nullptr) {
  const int cv = C / V; const int Wi = Wo * 2;
  const long long total = (long long)N * Ho * Wo * cv;
  float sa[V], sq[V];
#pragma unroll
  for (int j = 0; j < V; ++j) sa[j] = sq[j] = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % cv) * V; long long p = i / cv;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    const T* src = h + (((long long)n * Ho * 2 + oy * 2) * Wi + ox * 2) * C + c;
    float a[V], b[V], acc[V], sk[V];
    Ld<T, V>::ld(src, a); Ld<T, V>::ld(src + C, b);
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = a[j] + b[j];
    Ld<T, V>::ld(src + (long long)Wi * C, a); Ld<T, V>::ld(src + (long long)Wi * C + C, b);
    Ld<T, V>::ld(s + i * V, sk);
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = (acc[j] + a[j] + b[j]) * scale + sk[j];
    Ld<T, V>::st(y + i * V, acc);
    if constexpr (STATS) {
#pragma unroll
      for (int j = 0; j < V; ++j) { const float r = ttg_rounded<T>(acc[j]); sa[j] += r; sq[j] += r * r; }
    }
  }
  if constexpr (STATS) join_stats_flush<V>(sa, sq, cv, C, stats);
}
extern "C" int ttg_pool2_add_stats(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, float scale, double* sums,
                                   int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(sums != nullptr && ttg_join_stats_supported(C), "pool2_add_stats: unsupported channel count %d", C);
  cudaMemsetAsync(sums, 0, sizeof(double) * 2 * (size_t)C, st);
  TTG_DISPATCH(dtype, {
    TTG_REQUIRE((vec2_ok<T>(C, h, s) && vec2_ok<T>(C, y, y)) && Vec<T>::N == 8, "pool2_add_stats: bf16, 16-byte aligned tensors");
    constexpr int V = 8;
    const size_t smem = sizeof(float) * 2 * C;
    pool2_add_kernel<T, V, true><<<ttg_grid_occ(pool2_add_kernel<T, V, true>, (long long)N * Ho * Wo * (C / V), 256, 256, smem), 256, smem, st>>>(
        (const T*)h, (const T*)s, (T*)y, N, Ho, Wo, C, scale, sums);
  });
  TTG_CHECK_LAUNCH("pool2_add_stats");
  return TTG_OK;
}
extern "C" int ttg_pool2_add(const void* h, const void* s, void* y, int N, int Ho, int Wo, int C, float scale, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_DISPATCH(dtype, {
    if (vec2_ok<T>(C, h, s) && vec2_ok<T>(C, y, y)) { pool2_add_kernel<T, Vec<T>::N><<<ttg_grid_occ(pool2_add_kernel<T, Vec<T>::N>, (long long)N * Ho * Wo * (C / Vec<T>::N), 256, 256), 256, 0, st>>>((const T*)h, (const T*)s, (T*)y, N, Ho, Wo, C, scale); }
    else { pool2_add_kernel<T, 1><<<ttg_grid_occ(pool2_add_kernel<T, 1>, (long long)N * Ho * Wo * C, 256, 256), 256, 0, st>>>((const T*)h, (const T*)s, (T*)y, N, Ho, Wo, C, scale); }
  });
  TTG_CHECK_LAUNCH("pool2_add");
  return TTG_OK;
}

// out = alpha*a + beta*b
template <typename T, int V>
__global__ void axpby_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ o, long long nvec, float alpha, float beta) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float x[V], y[V];
    Ld<T, V>::ld(a + i * V, x); Ld<T, V>::ld(b + i * V, y);
#pragma unroll
    for (int j = 0; j < V; ++j) x[j] = alpha * x[j] + beta * y[j];
    Ld<T, V>::st(o + i * V, x);
  }
}
struct AxpbyNoParams { template <int V> struct P {}; template <int V> __device__ __forceinline__ void load(int, P<V>&) const {} };
template <typename T> struct AxpbyOp : AxpbyNoParams {
  static constexpr int NIN = 2, NOUT = 1;
  const T* in[2]; T* out[1]; float alpha, beta;
  template <int V> __device__ __forceinline__ void apply(const float* v, int, const P<V>&, float* o) const { o[0] = alpha * v[0] + beta * v[1]; }
};
extern "C" int ttg_axpby(const void* a, const void* b, void* out, long long n, float alpha, float beta, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) return TTG_OK;
  if (dtype == TTG_BF16 && n % 8 == 0 &&
      !((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out)) & 15)) {
    // large bf16 tensors (gradient fan-in adds): the bulk-copy pipelined map of chanops.cuh
    AxpbyOp<bf16> op; op.in[0] = (const bf16*)a; op.in[1] = (const bf16*)b; op.out[0] = (bf16*)out; op.alpha = alpha; op.beta = beta;
    return launch_chan_map<bf16>("axpby", op, n, 8, st);
  }
  TTG_DISPATCH(dtype, {
    bool vec = n % Vec<T>::N == 0 && !((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out)) & 15);
    if (vec) axpby_kernel<T, Vec<T>::N><<<ttg_grid_occ(axpby_kernel<T, Vec<T>::N>, n / Vec<T>::N, 512, 256), 256, 0, st>>>((const T*)a, (const T*)b, (T*)out, n / Vec<T>::N, alpha, beta);
    else axpby_kernel<T, 1><<<ttg_grid_occ(axpby_kernel<T, 1>, n, 1024, 256), 256, 0, st>>>((const T*)a, (const T*)b, (T*)out, n, alpha, beta);
  });
  TTG_CHECK_LAUNCH("axpby");
  return TTG_OK;
}

// out = x * (host_scale * *dev_scale)   (dev_scale may be null); fp32 only (loss plumbing)
__global__ void scale_f32_kernel(const float* __restrict__ x, float* __restrict__ o, long long n, float hs, const float* ds) {
  float s = hs * (ds ? *ds : 1.f);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) o[i] = x[i] * s;
}
extern "C" int ttg_scale_f32(const float* x, float* out, long long n, float host_scale, const float* dev_scale, void* stream) {
  if (n == 0) return TTG_OK;
  scale_f32_kernel<<<ttg_grid_occ(scale_f32_kernel, n, 1024, 256), 256, 0, (cudaStream_t)stream>>>(x, out, n, host_scale, dev_scale);
  TTG_CHECK_LAUNCH("scale_f32");
  return TTG_OK;
}

// feats[n,c] = sum_{hw} x[n,hw,c]   (fp32 out);  one block per (n, channel group)
template <typename T>
__global__ void spatial_sum_kernel(const T* __restrict__ x, float* __restrict__ out, int HW, int C) {
  int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    const T* p = x + (long long)n * HW * C + c;
    for (int i = 0; i < HW; ++i) s += to_f(p[(long long)i * C]);
    out[(long long)n * C + c] = s;
  }
}
extern "C" int ttg_spatial_sum(const void* x, float* out, int N, int HW, int C, int dtype, void* stream) {
  TTG_DISPATCH(dtype, { spatial_sum_kernel<T><<<N, 128, 0, (cudaStream_t)stream>>>((const T*)x, out, HW, C); });
  TTG_CHECK_LAUNCH("spatial_sum");
  return TTG_OK;
}
template <typename T>
__global__ void spatial_bcast_kernel(const float* __restrict__ g, T* __restrict__ gx, long long total, int HW, int C) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C); long long n = i / ((long long)HW * C);
    gx[i] = from_f<T>(g[n * C + c]);
  }
}
extern "C" int ttg_spatial_bcast(const float* g, void* gx, int N, int HW, int C, int dtype, void* stream) {
  long long total = (long long)N * HW * C;
  TTG_DISPATCH(dtype, { spatial_bcast_kernel<T><<<ttg_grid_occ(spatial_bcast_kernel<T>, total, 1024, 256), 256, 0, (cudaStream_t)stream>>>(g, (T*)gx, total, HW, C); });
  TTG_CHECK_LAUNCH("spatial_bcast");
  return TTG_OK;
}

// NCHW fp32 (contiguous) -> NHWC T, and back.
template <typename T>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, T* __restrict__ y, int N, int C, int HW) {
  const long long total = (long long)N * HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long n = i / HW; int p = (int)(i % HW);
    const float* s = x + n * C * HW + p; T* d = y + i * C;
    for (int c = 0; c < C; ++c) d[c] = from_f<T>(s[(long long)c * HW]);
  }
}
template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ x, float* __restrict__ y, int N, int C, int HW) {
  const long long total = (long long)N * HW;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long n = i / HW; int p = (int)(i % HW);
    const T* s = x + i * C; float* d = y + n * C * HW + p;
    for (int c = 0; c < C; ++c) d[(long long)c * HW] = to_f(s[c]);
  }
}
// RGB images (C == 3, the layout boundary of every training step: real batch in, fake batch out, d/d(real) out): a
// thread converts 8 pixels -> three coalesced 32-byte reads per plane and three 16-byte stores (bf16) instead of 2-byte
// stores per element; 41 -> ~15 us for a 256 x 3 x 128 x 128 batch
__global__ void nchw_to_nhwc_rgb_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ y, int N, int HW) {
  const long long total = (long long)N * (HW / 8);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / (HW / 8); const int p = (int)(i % (HW / 8)) * 8;
    const float* s = x + n * 3 * HW + p;
    float v[3][8];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float4 a = *reinterpret_cast<const float4*>(s + (long long)c * HW), b = *reinterpret_cast<const float4*>(s + (long long)c * HW + 4);
      v[c][0] = a.x; v[c][1] = a.y; v[c][2] = a.z; v[c][3] = a.w; v[c][4] = b.x; v[c][5] = b.y; v[c][6] = b.z; v[c][7] = b.w;
    }
    float o[24];
#pragma unroll
    for (int e = 0; e < 24; ++e) o[e] = v[e % 3][e / 3];
    bf16* d = y + (n * HW + p) * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) { Vec<bf16> q; q.pack(o + 8 * k); q.store(d + 8 * k); }
  }
}
__global__ void nhwc_to_nchw_rgb_bf16_kernel(const bf16* __restrict__ x, float* __restrict__ y, int N, int HW) {
  const long long total = (long long)N * (HW / 8);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / (HW / 8); const int p = (int)(i % (HW / 8)) * 8;
    const bf16* s = x + (n * HW + p) * 3;
    float o[24];
#pragma unroll
    for (int k = 0; k < 3; ++k) { Vec<bf16> q; q.load(s + 8 * k); q.unpack(o + 8 * k); }
    float* d = y + n * 3 * HW + p;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      *reinterpret_cast<float4*>(d + (long long)c * HW) = make_float4(o[c], o[3 + c], o[6 + c], o[9 + c]);
      *reinterpret_cast<float4*>(d + (long long)c * HW + 4) = make_float4(o[12 + c], o[15 + c], o[18 + c], o[21 + c]);
    }
  }
}
static inline bool rgb_fast_ok(int C, int HW, int dtype, const void* a, const void* b) {
  return C == 3 && HW % 8 == 0 && dtype == TTG_BF16 && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0;
}
// wide-channel maps (the generator's (B, 128, 4, 4) base image): one thread per output element instead of one thread
// per pixel walking C strided reads one after the other (42 us for 0.5 M elements)
template <typename T>
__global__ void nchw_to_nhwc_elem_kernel(const float* __restrict__ x, T* __restrict__ y, int N, int C, int HW) {
  const long long total = (long long)N * HW * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C); const long long q = i / C; const int p = (int)(q % HW); const long long n = q / HW;
    y[i] = from_f<T>(x[(n * C + c) * HW + p]);
  }
}
extern "C" int ttg_nchw_to_nhwc(const float* x, void* y, int N, int C, int HW, int dtype, void* stream) {
  if (C >= 16 && HW <= 256) {      // (large maps: the per-pixel kernel below reads each plane coalesced)
    TTG_DISPATCH(dtype, { nchw_to_nhwc_elem_kernel<T><<<ttg_grid_occ(nchw_to_nhwc_elem_kernel<T>, (long long)N * HW * C, 256 * 4), 256, 0, (cudaStream_t)stream>>>(x, (T*)y, N, C, HW); });
    TTG_CHECK_LAUNCH("nchw_to_nhwc_elem");
    return TTG_OK;
  }
  if (rgb_fast_ok(C, HW, dtype, x, y)) {
    nchw_to_nhwc_rgb_bf16_kernel<<<ttg_grid_occ(nchw_to_nhwc_rgb_bf16_kernel, (long long)N * (HW / 8), 256, 256), 256, 0, (cudaStream_t)stream>>>(x, (bf16*)y, N, HW);
    TTG_CHECK_LAUNCH("nchw_to_nhwc_rgb");
    return TTG_OK;
  }
  TTG_DISPATCH(dtype, { nchw_to_nhwc_kernel<T><<<ttg_grid_occ(nchw_to_nhwc_kernel<T>, (long long)N * HW, 256, 256), 256, 0, (cudaStream_t)stream>>>(x, (T*)y, N, C, HW); });
  TTG_CHECK_LAUNCH("nchw_to_nhwc");
  return TTG_OK;
}
extern "C" int ttg_nhwc_to_nchw(const void* x, float* y, int N, int C, int HW, int dtype, void* stream) {
  if (rgb_fast_ok(C, HW, dtype, x, y)) {
    nhwc_to_nchw_rgb_bf16_kernel<<<ttg_grid_occ(nhwc_to_nchw_rgb_bf16_kernel, (long long)N * (HW / 8), 256, 256), 256, 0, (cudaStream_t)stream>>>((const bf16*)x, y, N, HW);
    TTG_CHECK_LAUNCH("nhwc_to_nchw_rgb");
    return TTG_OK;
  }
  TTG_DISPATCH(dtype, { nhwc_to_nchw_kernel<T><<<ttg_grid_occ(nhwc_to_nchw_kernel<T>, (long long)N * HW, 256, 256), 256, 0, (cudaStream_t)stream>>>((const T*)x, y, N, C, HW); });
  TTG_CHECK_LAUNCH("nhwc_to_nchw");
  return TTG_OK;
}

// dtype casts (flat)
template <typename S, typename D>
__global__ void cast_kernel(const S* __restrict__ x, D* __restrict__ y, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) y[i] = from_f<D>(to_f(x[i]));
}
extern "C" int ttg_cast(const void* x, int src_dtype, void* y, int dst_dtype, long long n, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) return TTG_OK;
  int grid = ttg_grid_for(n, 1024);
  if (src_dtype == TTG_F32 && dst_dtype == TTG_BF16) cast_kernel<float, bf16><<<grid, 256, 0, st>>>((const float*)x, (bf16*)y, n);
  else if (src_dtype == TTG_BF16 && dst_dtype == TTG_F32) cast_kernel<bf16, float><<<grid, 256, 0, st>>>((const bf16*)x, (float*)y, n);
  else if (src_dtype == TTG_F32 && dst_dtype == TTG_F32) cast_kernel<float, float><<<grid, 256, 0, st>>>((const float*)x, (float*)y, n);
  else if (src_dtype == TTG_BF16 && dst_dtype == TTG_BF16) cast_kernel<bf16, bf16><<<grid, 256, 0, st>>>((const bf16*)x, (bf16*)y, n);
  else return ttg_set_error(TTG_ERR_ARG, "cast: bad dtypes %d -> %d", src_dtype, dst_dtype);
  TTG_CHECK_LAUNCH("cast");
  return TTG_OK;
}

// ---------------------------------------------------------------- generator head: conv1x1(C -> 3) + tanh + layout boundary
// GeneratorOutput (generator.py:115-129) ends with conv1x1(C -> data_dims = 3) -> tanh, and the module boundary returns
// fp32 NCHW.  As a GEMM this layer has N = 3: on the tensor-core path it took 176 us (fp32 3-channel epilogue) + tanh +
// the NHWC -> NCHW pass.  It is a pure HBM stream (32 B read, 12 B written per pixel), so: one CUDA-core kernel, a thread
// per pixel, fp32 weights and accumulation, tanh, and the three fp32 planes written directly (coalesced over pixels).
// Backward in one kernel as well: gpre = g (1 - y^2); ga[p, ci] = sum_co gpre[co] w[co, ci] (bf16 NHWC); the 3 x C
// weight gradient and the bias gradient are reduced per thread -> warp -> block -> one fp64 atomic per value and block.
#define RGB_CO 3
template <int CIN>
__global__ void __launch_bounds__(256) rgb_head_fwd_kernel(const bf16* __restrict__ a, const float* __restrict__ w,
                                                           const float* __restrict__ bias, float* __restrict__ y, long long npix, int HW) {
  __shared__ float sw[RGB_CO * CIN + RGB_CO];
  for (int i = threadIdx.x; i < RGB_CO * CIN; i += blockDim.x) sw[i] = w[i];
  if (threadIdx.x < RGB_CO) sw[RGB_CO * CIN + threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
  __syncthreads();
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (long long)gridDim.x * blockDim.x) {
    float x[CIN];
#pragma unroll
    for (int v = 0; v < CIN / 8; ++v) { Vec<bf16> q; q.load(a + p * CIN + v * 8); q.unpack(x + v * 8); }
    const long long n = p / HW; const int pp = (int)(p % HW);
#pragma unroll
    for (int co = 0; co < RGB_CO; ++co) {
      float acc = sw[RGB_CO * CIN + co];
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) acc += x[ci] * sw[co * CIN + ci];
      y[(n * RGB_CO + co) * HW + pp] = tanhf(acc);
    }
  }
}
template <int CIN>
__global__ void __launch_bounds__(256) rgb_head_bwd_kernel(const bf16* __restrict__ a, const float* __restrict__ w,
                                                           const float* __restrict__ y, const float* __restrict__ g,
                                                           bf16* __restrict__ ga, double* __restrict__ sums, long long npix, int HW) {
  constexpr int NW = RGB_CO * CIN + RGB_CO;          // weight gradient [co][ci] then bias gradient [co]
  __shared__ float sw[RGB_CO * CIN];
  __shared__ float s_acc[NW];
  for (int i = threadIdx.x; i < RGB_CO * CIN; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < NW; i += blockDim.x) s_acc[i] = 0.f;
  __syncthreads();
  float gw[RGB_CO][CIN], gb[RGB_CO];
#pragma unroll
  for (int co = 0; co < RGB_CO; ++co) {
    gb[co] = 0.f;
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) gw[co][ci] = 0.f;
  }
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (long long)gridDim.x * blockDim.x) {
    const long long n = p / HW; const int pp = (int)(p % HW);
    float gp[RGB_CO];
#pragma unroll
    for (int co = 0; co < RGB_CO; ++co) {
      const long long o = (n * RGB_CO + co) * HW + pp;
      const float t = y[o];
      gp[co] = g[o] * (1.f - t * t);
      gb[co] += gp[co];
    }
    float x[CIN], o[CIN];
#pragma unroll
    for (int v = 0; v < CIN / 8; ++v) { Vec<bf16> q; q.load(a + p * CIN + v * 8); q.unpack(x + v * 8); }
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
      float acc = 0.f;
#pragma unroll
      for (int co = 0; co < RGB_CO; ++co) { acc += gp[co] * sw[co * CIN + ci]; gw[co][ci] += gp[co] * x[ci]; }
      o[ci] = acc;
    }
#pragma unroll
    for (int v = 0; v < CIN / 8; ++v) { Vec<bf16> q; q.pack(o + v * 8); q.store(ga + p * CIN + v * 8); }
  }
#pragma unroll
  for (int co = 0; co < RGB_CO; ++co) {
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
      float t = gw[co][ci];
      for (int s = 16; s >= 1; s >>= 1) t += __shfl_xor_sync(0xffffffffu, t, s);
      if ((threadIdx.x & 31) == 0) atomicAdd(&s_acc[co * CIN + ci], t);
    }
    float t = gb[co];
    for (int s = 16; s >= 1; s >>= 1) t += __shfl_xor_sync(0xffffffffu, t, s);
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_acc[RGB_CO * CIN + co], t);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NW; i += blockDim.x) atomicAdd(&sums[i], (double)s_acc[i]);
}
__global__ void rgb_head_finalize_kernel(const double* __restrict__ sums, float* __restrict__ gw, float* __restrict__ gb, int nw, int acc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nw) { if (acc) atomicAdd(&gw[i], (float)sums[i]); else gw[i] = (float)sums[i]; }
  else if (i < nw + RGB_CO && gb) { if (acc) atomicAdd(&gb[i - nw], (float)sums[i]); else gb[i - nw] = (float)sums[i]; }
}
extern "C" int ttg_rgb_head_supported(int Cin, int Cout) { return Cout == RGB_CO && (Cin == 8 || Cin == 16 || Cin == 32) ? 1 : 0; }
extern "C" size_t ttg_rgb_head_workspace_bytes(int Cin) { return sizeof(double) * (size_t)(RGB_CO * Cin + RGB_CO); }
// a: bf16 NHWC [N, HW, Cin]; w: fp32 [3][Cin]; y: fp32 NCHW [N, 3, HW] = tanh(conv1x1(a) + bias)
extern "C" int ttg_rgb_head_fwd(const void* a, const float* w, const float* bias, float* y, int N, int HW, int Cin, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(ttg_rgb_head_supported(Cin, RGB_CO), "rgb_head_fwd: Cin = %d unsupported", Cin);
  const long long npix = (long long)N * HW;
#define TTG_RGB_F(C) rgb_head_fwd_kernel<C><<<ttg_grid_occ(rgb_head_fwd_kernel<C>, npix, 256 * 2), 256, 0, st>>>((const bf16*)a, w, bias, y, npix, HW)
  if (Cin == 8) TTG_RGB_F(8); else if (Cin == 16) TTG_RGB_F(16); else TTG_RGB_F(32);
#undef TTG_RGB_F
  TTG_CHECK_LAUNCH("rgb_head_fwd");
  return TTG_OK;
}
// g: fp32 NCHW cotangent of y; ga: bf16 NHWC [N, HW, Cin]; gw [3][Cin] / gb [3] overwritten (accumulate = 0) or added to
extern "C" int ttg_rgb_head_bwd(const void* a, const float* w, const float* y, const float* g, void* ga, float* gw, float* gb,
                                int N, int HW, int Cin, int accumulate, void* workspace, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(ttg_rgb_head_supported(Cin, RGB_CO) && workspace != nullptr, "rgb_head_bwd: bad arguments (Cin = %d)", Cin);
  const long long npix = (long long)N * HW;
  double* sums = (double*)workspace;
  const int nw = RGB_CO * Cin;
  cudaMemsetAsync(sums, 0, sizeof(double) * (nw + RGB_CO), st);
#define TTG_RGB_B(C) rgb_head_bwd_kernel<C><<<ttg_grid_occ(rgb_head_bwd_kernel<C>, npix, 256 * 8), 256, 0, st>>>((const bf16*)a, w, y, g, (bf16*)ga, sums, npix, HW)
  if (Cin == 8) TTG_RGB_B(8); else if (Cin == 16) TTG_RGB_B(16); else TTG_RGB_B(32);
#undef TTG_RGB_B
  TTG_CHECK_LAUNCH("rgb_head_bwd");
  rgb_head_finalize_kernel<<<1, 128, 0, st>>>(sums, gw, gb, nw, accumulate);
  TTG_CHECK_LAUNCH("rgb_head_finalize");
  return TTG_OK;
}

// tanh forward / backward (fp32 image at the generator boundary)
__global__ void tanh_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) y[i] = tanhf(x[i]);
}
__global__ void tanh_bwd_kernel(const float* __restrict__ y, const float* __restrict__ g, float* __restrict__ gx, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) gx[i] = g[i] * (1.f - y[i] * y[i]);
}
extern "C" int ttg_tanh_fwd(const float* x, float* y, long long n, void* stream) {
  if (n == 0) return TTG_OK;
  tanh_fwd_kernel<<<ttg_grid_occ(tanh_fwd_kernel, n, 1024, 256), 256, 0, (cudaStream_t)stream>>>(x, y, n);
  TTG_CHECK_LAUNCH("tanh_fwd");
  return TTG_OK;
}
extern "C" int ttg_tanh_bwd(const float* y, const float* g, float* gx, long long n, void* stream) {
  if (n == 0) return TTG_OK;
  tanh_bwd_kernel<<<ttg_grid_occ(tanh_bwd_kernel, n, 1024, 256), 256, 0, (cudaStream_t)stream>>>(y, g, gx, n);
  TTG_CHECK_LAUNCH("tanh_bwd");
  return TTG_OK;
}

// ---------------------------------------------------------------- device-side input pipeline (SURVEY 8 f-3)
// The reference keeps its dataset as a uint8 stack (datasets/image_bytes_dataset.py:44-49: random crop, then
// ToTensor + Normalize(0.5, 0.5) = v / 127.5 - 1).  Here the stack [M][H][W][C] stays in HBM and one kernel crops
// and normalises a whole batch: out[b][c][y][x] = stack[index[b]][oy[b] + y][ox[b] + x][c] / 127.5 - 1, written
// either as fp32 NCHW (the reference's batch layout) or as the internal NHWC activation tensor.
template <typename T, bool NCHW>
__global__ void u8_crop_norm_kernel(const unsigned char* __restrict__ stack, const int* __restrict__ index,
                                    const int* __restrict__ oy, const int* __restrict__ ox, T* __restrict__ out, int B, int H,
                                    int W, int C, int S) {
  const long long total = (long long)B * S * S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % S); long long p = i / S;
    const int y = (int)(p % S); const int b = (int)(p / S);
    const unsigned char* src = stack + (((long long)index[b] * H + oy[b] + y) * W + ox[b] + x) * C;
    for (int c = 0; c < C; ++c) {
      const float v = (float)src[c] / 127.5f - 1.f;           // IEEE division: bit-identical to the host pipeline
      if (NCHW) out[(((long long)b * C + c) * S + y) * S + x] = from_f<T>(v);
      else out[i * C + c] = from_f<T>(v);
    }
  }
}
extern "C" int ttg_u8_crop_normalize(const unsigned char* stack, const int* index, const int* oy, const int* ox, void* out,
                                     int B, int H, int W, int C, int size, int dtype_out, int nchw_out, void* stream) {
  TTG_REQUIRE(B > 0 && C > 0 && size > 0 && size <= H && size <= W, "u8_crop_normalize: bad sizes");
  TTG_REQUIRE(!nchw_out || dtype_out == TTG_F32, "u8_crop_normalize: NCHW output is fp32 (the reference's batch layout)");
  const long long total = (long long)B * size * size;
  cudaStream_t st = (cudaStream_t)stream;
  if (nchw_out) {
    u8_crop_norm_kernel<float, true><<<ttg_grid_for(total, 256), 256, 0, st>>>(stack, index, oy, ox, (float*)out, B, H, W, C, size);
  } else {
    TTG_DISPATCH(dtype_out, { u8_crop_norm_kernel<T, false><<<ttg_grid_for(total, 256), 256, 0, st>>>(stack, index, oy, ox, (T*)out, B, H, W, C, size); });
  }
  TTG_CHECK_LAUNCH("u8_crop_normalize");
  return TTG_OK;
}
