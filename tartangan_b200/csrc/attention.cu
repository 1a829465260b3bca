// 2-D self-attention building blocks (reference models/blocks/attention.py:21-35) and the
// spectral-norm power iteration.  NHWC activations: a feature map is a [positions][channels]
// matrix per image, so theta^T phi is A*B^T and beta*g is A*B without any transposition copies.
//   maxpool2 fwd (+argmax byte), scatter (its backward), gather (backward of the backward)
//   bmm with fp32 accumulation (closed under differentiation via the transpose flags)
//   row softmax forward / backward / backward-of-backward (D-side attention under R1)
//   gamma*o scaling by a device scalar, dot product (d/dgamma)
#include "common.cuh"

// ---------------------------------------------------------------- max-pool 2x2
template <typename T>
__global__ void maxpool2_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, unsigned char* __restrict__ idx, int N,
                                    int Ho, int Wo, int C) {
  const long long total = (long long)N * Ho * Wo * C; const int Wi = Wo * 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C); long long p = i / C;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    const T* s = x + (((long long)n * Ho * 2 + oy * 2) * Wi + ox * 2) * C + c;
    // first maximum in window order; a NaN propagates and takes the index (the last NaN), like torch's max_pool2d
    float best = to_f(s[0]); int bi = 0;
    float v = to_f(s[C]); if (v > best || isnan(v)) { best = v; bi = 1; }
    v = to_f(s[(long long)Wi * C]); if (v > best || isnan(v)) { best = v; bi = 2; }
    v = to_f(s[(long long)Wi * C + C]); if (v > best || isnan(v)) { best = v; bi = 3; }
    y[i] = from_f<T>(best); idx[i] = (unsigned char)bi;
  }
}
// gx[window] = gy at the argmax position, 0 elsewhere
template <typename T>
__global__ void maxpool2_scatter_kernel(const T* __restrict__ gy, const unsigned char* __restrict__ idx, T* __restrict__ gx,
                                        int N, int Ho, int Wo, int C) {
  const long long total = (long long)N * Ho * Wo * C; const int Wi = Wo * 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C); long long p = i / C;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    T* d = gx + (((long long)n * Ho * 2 + oy * 2) * Wi + ox * 2) * C + c;
    int bi = idx[i]; T g = gy[i]; T z = from_f<T>(0.f);
    d[0] = bi == 0 ? g : z; d[C] = bi == 1 ? g : z;
    d[(long long)Wi * C] = bi == 2 ? g : z; d[(long long)Wi * C + C] = bi == 3 ? g : z;
  }
}
template <typename T>
__global__ void maxpool2_gather_kernel(const T* __restrict__ x, const unsigned char* __restrict__ idx, T* __restrict__ y,
                                       int N, int Ho, int Wo, int C) {
  const long long total = (long long)N * Ho * Wo * C; const int Wi = Wo * 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C); long long p = i / C;
    int ox = (int)(p % Wo); p /= Wo; int oy = (int)(p % Ho); int n = (int)(p / Ho);
    int bi = idx[i];
    y[i] = x[(((long long)n * Ho * 2 + oy * 2 + (bi >> 1)) * Wi + ox * 2 + (bi & 1)) * C + c];
  }
}
extern "C" int ttg_maxpool2_fwd(const void* x, void* y, unsigned char* idx, int N, int Ho, int Wo, int C, int dtype, void* stream) {
  long long total = (long long)N * Ho * Wo * C;
  TTG_DISPATCH(dtype, { maxpool2_fwd_kernel<T><<<ttg_grid_for(total, 512), 256, 0, (cudaStream_t)stream>>>((const T*)x, (T*)y, idx, N, Ho, Wo, C); });
  TTG_CHECK_LAUNCH("maxpool2_fwd");
  return TTG_OK;
}
extern "C" int ttg_maxpool2_scatter(const void* gy, const unsigned char* idx, void* gx, int N, int Ho, int Wo, int C, int dtype, void* stream) {
  long long total = (long long)N * Ho * Wo * C;
  TTG_DISPATCH(dtype, { maxpool2_scatter_kernel<T><<<ttg_grid_for(total, 512), 256, 0, (cudaStream_t)stream>>>((const T*)gy, idx, (T*)gx, N, Ho, Wo, C); });
  TTG_CHECK_LAUNCH("maxpool2_scatter");
  return TTG_OK;
}
extern "C" int ttg_maxpool2_gather(const void* x, const unsigned char* idx, void* y, int N, int Ho, int Wo, int C, int dtype, void* stream) {
  long long total = (long long)N * Ho * Wo * C;
  TTG_DISPATCH(dtype, { maxpool2_gather_kernel<T><<<ttg_grid_for(total, 512), 256, 0, (cudaStream_t)stream>>>((const T*)x, idx, (T*)y, N, Ho, Wo, C); });
  TTG_CHECK_LAUNCH("maxpool2_gather");
  return TTG_OK;
}

// ---------------------------------------------------------------- batched matmul, fp32 accumulate
// C[b][M,N] = op(A[b]) * op(B[b]); op(A) is [M,K] (stored [K,M] if transA), op(B) is [K,N] (stored [N,K] if transB).
// 64x64 block tile, 4x4 per thread, K staged 16 at a time.
template <typename T>
__global__ void __launch_bounds__(256) bmm_kernel(const T* __restrict__ A, const T* __restrict__ B, T* __restrict__ C, int M,
                                                  int N, int K, int ta, int tb) {
  __shared__ float sa[16][65], sb[16][65];
  const int b = blockIdx.z;
  A += (long long)b * M * K; B += (long long)b * K * N; C += (long long)b * M * N;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 16 * 64; i += 256) {
      int kk, mm;
      if (ta) { mm = i % 64; kk = i / 64; } else { kk = i % 16; mm = i / 16; }
      int gm = m0 + mm, gk = k0 + kk;
      sa[kk][mm] = (gm < M && gk < K) ? to_f(ta ? A[(long long)gk * M + gm] : A[(long long)gm * K + gk]) : 0.f;
      int nn;
      if (tb) { kk = i % 16; nn = i / 16; } else { nn = i % 64; kk = i / 64; }
      int gn = n0 + nn; gk = k0 + kk;
      sb[kk][nn] = (gn < N && gk < K) ? to_f(tb ? B[(long long)gn * K + gk] : B[(long long)gk * N + gn]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sa[kk][ty * 4 + i]; bb[i] = sb[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * bb[j];
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int gm = m0 + ty * 4 + i, gn = n0 + tx * 4 + j;
      if (gm < M && gn < N) C[(long long)gm * N + gn] = from_f<T>(acc[i][j]);
    }
}
extern "C" int ttg_bmm(const void* A, const void* B, void* C, int batch, int M, int N, int K, int transA, int transB,
                       int dtype, void* stream) {
  TTG_REQUIRE(batch > 0 && batch <= 65535 && M > 0 && N > 0 && K > 0, "bmm: bad sizes");
  dim3 grid((N + 63) / 64, (M + 63) / 64, batch);
  TTG_DISPATCH(dtype, { bmm_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)A, (const T*)B, (T*)C, M, N, K, transA, transB); });
  TTG_CHECK_LAUNCH("bmm");
  return TTG_OK;
}

// ---------------------------------------------------------------- row softmax (one warp per row)
template <typename T>
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, long long rows, int cols) {
  const int lane = threadIdx.x & 31; const long long warp = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  for (long long r = warp; r < rows; r += (long long)gridDim.x * 8) {
    const T* xr = x + r * cols; T* yr = y + r * cols;
    float mx = -INFINITY;
    for (int c = lane; c < cols; c += 32) mx = fmaxf(mx, to_f(xr[c]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) s += __expf(to_f(xr[c]) - mx);
    s = warp_sum(s);
    const float inv = 1.f / s;
    for (int c = lane; c < cols; c += 32) yr[c] = from_f<T>(__expf(to_f(xr[c]) - mx) * inv);
  }
}
// gx = y * (gy - sum(gy*y))
template <typename T>
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const T* __restrict__ y, const T* __restrict__ gy, T* __restrict__ gx,
                                                          long long rows, int cols) {
  const int lane = threadIdx.x & 31; const long long warp = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  for (long long r = warp; r < rows; r += (long long)gridDim.x * 8) {
    const T* yr = y + r * cols; const T* gr = gy + r * cols; T* o = gx + r * cols;
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) s += to_f(yr[c]) * to_f(gr[c]);
    s = warp_sum(s);
    for (int c = lane; c < cols; c += 32) o[c] = from_f<T>(to_f(yr[c]) * (to_f(gr[c]) - s));
  }
}
// given w = cotangent of gx:  cot_gy = y*(w - t),  cot_y = w*(gy - s) - gy*t,  s = sum(gy*y), t = sum(w*y)
template <typename T>
__global__ void __launch_bounds__(256) softmax_bwd2_kernel(const T* __restrict__ y, const T* __restrict__ gy, const T* __restrict__ w,
                                                           T* __restrict__ cot_gy, T* __restrict__ cot_y, long long rows, int cols) {
  const int lane = threadIdx.x & 31; const long long warp = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  for (long long r = warp; r < rows; r += (long long)gridDim.x * 8) {
    const T* yr = y + r * cols; const T* gr = gy + r * cols; const T* wr = w + r * cols;
    float s = 0.f, t = 0.f;
    for (int c = lane; c < cols; c += 32) { float yy = to_f(yr[c]); s += yy * to_f(gr[c]); t += yy * to_f(wr[c]); }
    s = warp_sum(s); t = warp_sum(t);
    for (int c = lane; c < cols; c += 32) {
      float yy = to_f(yr[c]), g = to_f(gr[c]), ww = to_f(wr[c]);
      cot_gy[r * cols + c] = from_f<T>(yy * (ww - t));
      cot_y[r * cols + c] = from_f<T>(ww * (g - s) - g * t);
    }
  }
}
extern "C" int ttg_softmax_fwd(const void* x, void* y, long long rows, int cols, int dtype, void* stream) {
  TTG_DISPATCH(dtype, { softmax_fwd_kernel<T><<<ttg_grid_for(rows, 8), 256, 0, (cudaStream_t)stream>>>((const T*)x, (T*)y, rows, cols); });
  TTG_CHECK_LAUNCH("softmax_fwd");
  return TTG_OK;
}
extern "C" int ttg_softmax_bwd(const void* y, const void* gy, void* gx, long long rows, int cols, int dtype, void* stream) {
  TTG_DISPATCH(dtype, { softmax_bwd_kernel<T><<<ttg_grid_for(rows, 8), 256, 0, (cudaStream_t)stream>>>((const T*)y, (const T*)gy, (T*)gx, rows, cols); });
  TTG_CHECK_LAUNCH("softmax_bwd");
  return TTG_OK;
}
extern "C" int ttg_softmax_bwd2(const void* y, const void* gy, const void* w, void* cot_gy, void* cot_y, long long rows,
                                int cols, int dtype, void* stream) {
  TTG_DISPATCH(dtype, { softmax_bwd2_kernel<T><<<ttg_grid_for(rows, 8), 256, 0, (cudaStream_t)stream>>>((const T*)y, (const T*)gy, (const T*)w, (T*)cot_gy, (T*)cot_y, rows, cols); });
  TTG_CHECK_LAUNCH("softmax_bwd2");
  return TTG_OK;
}

// ---------------------------------------------------------------- scale by device scalar, dot
template <typename T>
__global__ void scale_dev_kernel(const T* __restrict__ x, T* __restrict__ o, long long n, const float* __restrict__ s) {
  const float sc = s[0];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) o[i] = from_f<T>(to_f(x[i]) * sc);
}
extern "C" int ttg_scale_dev(const void* x, void* out, long long n, const float* dev_scale, int dtype, void* stream) {
  if (n == 0) return TTG_OK;
  TTG_DISPATCH(dtype, { scale_dev_kernel<T><<<ttg_grid_for(n, 1024), 256, 0, (cudaStream_t)stream>>>((const T*)x, (T*)out, n, dev_scale); });
  TTG_CHECK_LAUNCH("scale_dev");
  return TTG_OK;
}
template <typename T>
__global__ void __launch_bounds__(256) dot_kernel(const T* __restrict__ a, const T* __restrict__ b, double* __restrict__ ws, long long n) {
  __shared__ float s[8];
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) acc += to_f(a[i]) * to_f(b[i]);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < 8 ? s[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) atomicAdd(ws, (double)t);
  }
}
__global__ void dot_finalize_kernel(const double* ws, float* out) { out[0] = (float)ws[0]; }
extern "C" int ttg_dot_f32out(const void* a, const void* b, float* out, long long n, void* workspace, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  double* ws = (double*)workspace;
  cudaMemsetAsync(ws, 0, sizeof(double), st);
  TTG_DISPATCH(dtype, { dot_kernel<T><<<ttg_grid_for(n, 2048, 4), 256, 0, st>>>((const T*)a, (const T*)b, ws, n); });
  TTG_CHECK_LAUNCH("dot");
  dot_finalize_kernel<<<1, 1, 0, st>>>(ws, out);
  TTG_CHECK_LAUNCH("dot_finalize");
  return TTG_OK;
}

// ---------------------------------------------------------------- spectral norm power iteration
// W is [rows, cols] fp32 row-major (conv weight viewed (Cout, Cin*k*k), at most 256 x 2304 = 2.4 MB, L2 resident).
// ONE launch per call: a thread-block CLUSTER of 8 CTAs (the matrices are tiny, a launch costs more than the
// arithmetic, but one CTA alone reads 2.4 MB four times at ~50 GB/s: 217 us).  The phases are separated by cluster
// barriers; partial results travel through a small global workspace:
//   per iteration  v = normalize(W^T u)   (CTA = a slice of the columns; threads = column x row-group, fixed-order sums)
//                  u = normalize(W v)     (CTA = a slice of the rows; warp per row, shuffle reduction)
//   then sigma = u^T W v and w_out = W / sigma (CTA = a slice of the elements).
// Every sum has a fixed order: bitwise repeatable from run to run.
// workspace: 2 * SN_CL + rows + cols floats (ttg_spectral_norm_workspace_floats).
#include <cooperative_groups.h>
namespace cg = cooperative_groups;
#define SN_CL 8
#define SN_THREADS 512
__device__ __forceinline__ float sn_block_sum(float x, float* red) {      // all threads get the total
  x = warp_sum(x);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();                       // (red may still be read from the previous call)
  if (lane == 0) red[warp] = x;
  __syncthreads();
  float t = 0.f;
  for (int i = 0; i < nw; ++i) t += red[i];
  return t;
}
__device__ __forceinline__ void sn_cluster_barrier(cg::cluster_group& cl) { __threadfence(); cl.sync(); }
__device__ __forceinline__ float sn_sum_partials(const volatile float* p) {
  float t = 0.f;
  for (int i = 0; i < SN_CL; ++i) t += p[i];
  return t;
}
// n_iter == 0: eval mode, sigma from the stored u, v without updating them
__global__ void __cluster_dims__(SN_CL, 1, 1) __launch_bounds__(SN_THREADS)
sn_fused_kernel(const float* __restrict__ w, float* __restrict__ u_g, float* __restrict__ v_g, float* __restrict__ w_out,
                float* __restrict__ sigma_g, int rows, int cols, int n_iter, float eps, float* __restrict__ ws) {
  cg::cluster_group cl = cg::this_cluster();
  const int rank = (int)cl.block_rank();
  __shared__ float red[32];
  __shared__ float part[SN_THREADS];
  volatile float* pv = ws;                  // [SN_CL] partial |v|^2
  volatile float* pu = ws + SN_CL;          // [SN_CL] partial |u|^2 (or partial sigma)
  float* vraw = ws + 2 * SN_CL;             // [cols]
  float* uraw = vraw + cols;                // [rows]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = SN_THREADS / 32;
  const int c_per = (cols + SN_CL - 1) / SN_CL, c0 = rank * c_per, c1 = min(cols, c0 + c_per);
  const int r_per = (rows + SN_CL - 1) / SN_CL, r0 = rank * r_per, r1 = min(rows, r0 + r_per);
  float inv_v = 1.f, inv_u = 1.f;           // scale of vraw / uraw (1: they hold the stored, normalised vectors)
  if (n_iter == 0) {
    for (int c = c0 + tid; c < c1; c += SN_THREADS) vraw[c] = v_g[c];
    for (int r = r0 + tid; r < r1; r += SN_THREADS) uraw[r] = u_g[r];
    sn_cluster_barrier(cl);
  }
  for (int it = 0; it < n_iter; ++it) {
    // ---- v = W^T u over this CTA's columns: thread = (column, row group); the groups are summed in a fixed order
    float sq = 0.f;
    for (int cb = c0; cb < c1; cb += SN_THREADS) {
      const int ncs = min(SN_THREADS, c1 - cb);            // columns in this pass (all of the slice unless it is huge)
      const int rg = SN_THREADS / ncs;                      // row groups
      const int cl_ = tid % ncs, g = tid / ncs;
      float a = 0.f;
      if (g < rg)
        for (int r = g; r < rows; r += rg) a += w[(long long)r * cols + cb + cl_] * (it == 0 ? u_g[r] : __ldcg(&uraw[r]) * inv_u);
      __syncthreads();
      part[tid] = a;
      __syncthreads();
      if (tid < ncs) {
        float t = 0.f;
        for (int gg = 0; gg < rg; ++gg) t += part[gg * ncs + tid];
        vraw[cb + tid] = t; sq += t * t;
      }
    }
    const float sqb = sn_block_sum(sq, red);
    if (tid == 0) pv[rank] = sqb;
    sn_cluster_barrier(cl);
    inv_v = 1.f / fmaxf(sqrtf(sn_sum_partials(pv)), eps);
    // ---- u = W v over this CTA's rows: warp per row
    sq = 0.f;
    for (int r = r0 + warp; r < r1; r += nw) {
      const float* wr = w + (long long)r * cols;
      float a = 0.f;
      for (int c = lane; c < cols; c += 32) a += wr[c] * __ldcg(&vraw[c]);      // (written by other SMs: bypass L1)
      a = warp_sum(a) * inv_v;
      if (lane == 0) { uraw[r] = a; sq += a * a; }
    }
    const float squ = sn_block_sum(sq, red);
    if (tid == 0) pu[rank] = squ;
    sn_cluster_barrier(cl);
    inv_u = 1.f / fmaxf(sqrtf(sn_sum_partials(pu)), eps);
  }
  float sigma;
  if (n_iter > 0) {
    sigma = sn_sum_partials(pu) * inv_u;                    // u^T W v with u = W v / |W v|
  } else {
    float p = 0.f;
    for (int r = r0 + warp; r < r1; r += nw) {
      const float* wr = w + (long long)r * cols;
      float a = 0.f;
      for (int c = lane; c < cols; c += 32) a += wr[c] * __ldcg(&vraw[c]);
      a = warp_sum(a);
      if (lane == 0) p += a * __ldcg(&uraw[r]);
    }
    const float pb = sn_block_sum(p, red);
    if (tid == 0) pu[rank] = pb;
    sn_cluster_barrier(cl);
    sigma = sn_sum_partials(pu);
  }
  const float inv = 1.f / sigma;
  const long long n = (long long)rows * cols, per = (n + SN_CL - 1) / SN_CL, e0 = rank * per, e1 = min(n, e0 + per);
  for (long long i = e0 + tid; i < e1; i += SN_THREADS) w_out[i] = w[i] * inv;
  if (n_iter > 0) {
    for (int r = r0 + tid; r < r1; r += SN_THREADS) u_g[r] = uraw[r] * inv_u;
    for (int c = c0 + tid; c < c1; c += SN_THREADS) v_g[c] = vraw[c] * inv_v;
  }
  if (rank == 0 && tid == 0) sigma_g[0] = sigma;
}
extern "C" size_t ttg_spectral_norm_workspace_floats(int rows, int cols) { return (size_t)(2 * SN_CL + rows + cols + 16); }
static int sn_launch(const float* w, float* u, float* v, float* w_out, float* sigma, int rows, int cols, int n_iter, float eps,
                     float* ws, cudaStream_t st, const char* name) {
  TTG_REQUIRE(rows > 0 && cols > 0 && ws != nullptr, "spectral_norm: bad arguments");
  sn_fused_kernel<<<SN_CL, SN_THREADS, 0, st>>>(w, u, v, w_out, sigma, rows, cols, n_iter, eps, ws);
  TTG_CHECK_LAUNCH(name);
  return TTG_OK;
}
extern "C" int ttg_spectral_norm(const float* w, float* u, float* v, float* w_out, float* sigma, int rows, int cols,
                                 int n_iter, float eps, void* workspace, void* stream) {
  TTG_REQUIRE(n_iter >= 1, "spectral_norm: n_iter must be >= 1");
  return sn_launch(w, u, v, w_out, sigma, rows, cols, n_iter, eps, (float*)workspace, (cudaStream_t)stream, "spectral_norm");
}
// eval mode: sigma = u^T W v with the given (already normalised) u, v; no update
extern "C" int ttg_spectral_norm_sigma(const float* w, const float* u, const float* v, float* w_out, float* sigma, int rows,
                                       int cols, void* workspace, void* stream) {
  return sn_launch(w, (float*)u, (float*)v, w_out, sigma, rows, cols, 0, 0.f, (float*)workspace, (cudaStream_t)stream,
                   "spectral_norm_sigma");
}
// g_w = (g - dot(g, w_out) * u v^T) / sigma   (u, v constants: torch.nn.utils.spectral_norm detaches them); one launch
__global__ void __cluster_dims__(SN_CL, 1, 1) __launch_bounds__(SN_THREADS)
sn_bwd_fused_kernel(const float* __restrict__ g, const float* __restrict__ w_out, const float* __restrict__ u,
                    const float* __restrict__ v, const float* __restrict__ sigma, float* __restrict__ gw, int rows, int cols,
                    float* __restrict__ ws) {
  cg::cluster_group cl = cg::this_cluster();
  const int rank = (int)cl.block_rank();
  __shared__ float red[32];
  volatile float* pd = ws;
  const long long n = (long long)rows * cols, per = (n + SN_CL - 1) / SN_CL, e0 = rank * per, e1 = min(n, e0 + per);
  float part = 0.f;
  for (long long i = e0 + threadIdx.x; i < e1; i += SN_THREADS) part += g[i] * w_out[i];
  const float pb = sn_block_sum(part, red);
  if (threadIdx.x == 0) pd[rank] = pb;
  sn_cluster_barrier(cl);
  const float d = sn_sum_partials(pd);
  const float inv = 1.f / sigma[0];
  for (long long i = e0 + threadIdx.x; i < e1; i += SN_THREADS) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    gw[i] = (g[i] - d * u[r] * v[c]) * inv;
  }
}
extern "C" int ttg_spectral_norm_bwd(const float* g, const float* w_out, const float* u, const float* v, const float* sigma,
                                     float* gw, int rows, int cols, void* workspace, void* stream) {
  TTG_REQUIRE(workspace != nullptr, "spectral_norm_bwd: workspace missing");
  sn_bwd_fused_kernel<<<SN_CL, SN_THREADS, 0, (cudaStream_t)stream>>>(g, w_out, u, v, sigma, gw, rows, cols, (float*)workspace);
  TTG_CHECK_LAUNCH("spectral_norm_bwd");
  return TTG_OK;
}
