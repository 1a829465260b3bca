// Train-mode BatchNorm2d (+ fused LeakyReLU) over NHWC activations:
// statistics, forward, backward and backward-of-backward (needed by the R1
// gradient penalty, reference models/losses.py:17-30).  Replaces the ATen ops
// native_batch_norm / native_batch_norm_backward / NativeBatchNormBackwardBackward
// + leaky_relu(_backward) issued by every nn.BatchNorm2d + nn.LeakyReLU pair in
// reference models/blocks/{generator,discriminator}.py.
// All kernels are HBM streams: 16-byte vector loads, per-channel partial sums in
// registers -> shared -> one fp64 atomic per (block, channel).
#include "chanops.cuh"

// ---------------------------------------------------------------- statistics
struct NoParams { template <int V> struct P {}; template <int V> __device__ __forceinline__ void load(int, P<V>&) const {} };

template <typename T> struct StatsOp : NoParams {
  static constexpr int NIN = 1, NACC = 2;
  const T* in[1];
  template <int V> __device__ __forceinline__ void acc(const float* v, int, const P<V>&, float* a) const { a[0] += v[0]; a[1] += v[0] * v[0]; }
};

__global__ void bn_finalize_kernel(const double* __restrict__ sums, long long M, long long count_mult, int C, float eps, float momentum,
                                   float* __restrict__ mean, float* __restrict__ invstd,
                                   float* __restrict__ running_mean, float* __restrict__ running_var,
                                   long long* __restrict__ num_batches) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    double m = sums[c] / (double)M;
    double var = sums[C + c] / (double)M - m * m;
    if (var < 0) var = 0;
    mean[c] = (float)m;
    invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) {
      const double Mu = (double)M * (double)count_mult;     // element count the reference op would have seen
      double unbiased = Mu > 1 ? var * Mu / (Mu - 1.0) : var;
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)m;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
  }
  if (c == 0 && num_batches) *num_batches += 1;
}

extern "C" size_t ttg_bn_workspace_bytes(int C) { return sizeof(double) * 5 * (size_t)C; }

extern "C" int ttg_bn_stats(const void* x, long long M, int C, float eps, float momentum, float* mean, float* invstd,
                            float* running_mean, float* running_var, long long* num_batches, void* workspace,
                            long long count_mult, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(M > 0 && C > 0 && count_mult >= 1, "bn_stats: empty input");
  double* ws = (double*)workspace;
  TTG_DISPATCH(dtype, {
    StatsOp<T> op; op.in[0] = (const T*)x;
    int rc = launch_chan_reduce<T>("bn_stats", op, M, C, ws, st);
    if (rc) return rc;
  });
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(ws, M, count_mult, C, eps, momentum, mean, invstd, running_mean,
                                                       running_var, num_batches);
  TTG_CHECK_LAUNCH("bn_finalize");
  return TTG_OK;
}

// statistics already accumulated by the producer of x (ttg_conv2d_tc_stats): sums = {sum x, sum x^2} in fp64
extern "C" int ttg_bn_finalize(const double* sums, long long M, int C, float eps, float momentum, float* mean, float* invstd,
                               float* running_mean, float* running_var, long long* num_batches, long long count_mult,
                               void* stream) {
  TTG_REQUIRE(M > 0 && C > 0 && count_mult >= 1 && sums != nullptr, "bn_finalize: empty input");
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, M, count_mult, C, eps, momentum, mean, invstd,
                                                                       running_mean, running_var, num_batches);
  TTG_CHECK_LAUNCH("bn_finalize");
  return TTG_OK;
}

// eval-mode helper: mean/invstd from running statistics.
__global__ void bn_eval_stats_kernel(const float* rm, const float* rv, float eps, int C, float* mean, float* invstd) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) { mean[c] = rm[c]; invstd[c] = rsqrtf(rv[c] + eps); }
}
extern "C" int ttg_bn_eval_stats(const float* running_mean, const float* running_var, float eps, int C, float* mean,
                                 float* invstd, void* stream) {
  bn_eval_stats_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(running_mean, running_var, eps, C, mean, invstd);
  TTG_CHECK_LAUNCH("bn_eval_stats");
  return TTG_OK;
}

// ---------------------------------------------------------------- forward
template <typename T> struct BnActFwdOp {
  static constexpr int NIN = 1, NOUT = 1;
  const T* in[1]; T* out[1];
  const float *mean, *invstd, *gamma, *beta; float slope;
  template <int V> struct P { float a[V], b[V]; };     // y = x*a + b
  template <int V> __device__ __forceinline__ void load(int c0, P<V>& p) const {
#pragma unroll
    for (int j = 0; j < V; ++j) { float a = invstd[c0 + j] * gamma[c0 + j]; p.a[j] = a; p.b[j] = beta[c0 + j] - mean[c0 + j] * a; }
  }
  template <int V> __device__ __forceinline__ void apply(const float* v, int j, const P<V>& p, float* o) const {
    o[0] = lrelu(v[0] * p.a[j] + p.b[j], slope);
  }
};

extern "C" int ttg_bn_act_fwd(const void* x, void* y, long long M, int C, const float* mean, const float* invstd,
                              const float* gamma, const float* beta, float slope, int dtype, void* stream) {
  TTG_DISPATCH(dtype, {
    BnActFwdOp<T> op; op.in[0] = (const T*)x; op.out[0] = (T*)y;
    op.mean = mean; op.invstd = invstd; op.gamma = gamma; op.beta = beta; op.slope = slope;
    return launch_chan_map<T>("bn_act_fwd", op, M * C, C, (cudaStream_t)stream);
  });
  return TTG_OK;
}

// BatchNorm finalisation folded into the apply pass: every thread derives its channels' (mean, invstd) from the
// fp64 sums (same arithmetic as bn_finalize_kernel, so results are bit-identical), block 0 also stores them for the
// backward pass and updates the running statistics.
template <typename T> struct BnActFwdStatsOp {
  static constexpr int NIN = 1, NOUT = 1;
  const T* in[1]; T* out[1];
  const double* sums; const float *gamma, *beta; float slope, eps, momentum; long long M, count_mult; int C;
  float *mean, *invstd, *running_mean, *running_var; long long* num_batches;
  // Every thread derives (mean, invstd) of its 8 channels before it streams: fp64 division / square root are
  // ~100-instruction sequences on a 64-lane pipe, 24 of them per thread cost ~10 us per launch (measured: 62.7 us for
  // this op against 51.2 us for the plain apply pass at M = 4 Mi, C = 16).  So: multiply by a host-computed 1/M and take
  // 1/sqrt from the fp32 seed plus one fp64 Newton step (relative error ~1e-13, far below the fp32 result's 6e-8).
  double invM;
  __device__ __forceinline__ void chan(int c, float& mf, float& rf, double& var) const {
    const double m = sums[c] * invM;
    var = sums[C + c] * invM - m * m;
    if (var < 0) var = 0;
    const double t = var + (double)eps;
    double y = (double)rsqrtf((float)t);
    y = y * (1.5 - 0.5 * t * y * y);
    y = y * (1.5 - 0.5 * t * y * y);      // (second step: the fp32 seed is only good to ~2^-22)
    mf = (float)m; rf = (float)y;
  }
  template <int V> struct P { float a[V], b[V]; };     // y = x*a + b
  template <int V> __device__ __forceinline__ void load(int c0, P<V>& p) const {
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float mf, rf; double var;
      chan(c0 + j, mf, rf, var);
      const float a = rf * gamma[c0 + j]; p.a[j] = a; p.b[j] = beta[c0 + j] - mf * a;
    }
  }
  template <int V> __device__ __forceinline__ void apply(const float* v, int j, const P<V>& p, float* o) const {
    o[0] = lrelu(v[0] * p.a[j] + p.b[j], slope);
  }
  __device__ void finalize(int) const {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      float mf, rf; double var;
      chan(c, mf, rf, var);
      mean[c] = mf; invstd[c] = rf;
      if (running_mean) {
        const double Mu = (double)M * (double)count_mult;
        const double unbiased = Mu > 1 ? var * Mu / (Mu - 1.0) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mf;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
      }
    }
    if (threadIdx.x == 0 && num_batches) *num_batches += 1;
  }
};
// {sum x, sum x^2} of x[M, C] into sums[2C] (fp64); flags bit 1: sums is already zero
extern "C" int ttg_bn_sums(const void* x, long long M, int C, double* sums, int flags, int dtype, void* stream) {
  TTG_REQUIRE(M > 0 && C > 0 && sums != nullptr, "bn_sums: bad arguments");
  TTG_DISPATCH(dtype, {
    StatsOp<T> r; r.in[0] = (const T*)x;
    return launch_chan_reduce<T>("bn_stats", r, M, C, sums, (cudaStream_t)stream, (flags & 2) != 0);
  });
  return TTG_OK;
}

// train-mode BatchNorm + LeakyReLU in (at most) two launches: statistics (skipped when `sums` = {sum x, sum x^2} was
// already produced by the conv / join kernel that wrote x) and one apply pass that also finalises the statistics.
// `count`: the pixel count the sums were taken over (synchronised BatchNorm: the sums of every rank, count = world * M);
// the apply pass walks the M local rows.
extern "C" int ttg_bn_act_fwd_stats_n(const void* x, void* y, long long M, int C, long long count, const double* sums,
                                      const float* gamma, const float* beta, float eps, float momentum, float slope,
                                      float* mean, float* invstd, float* running_mean, float* running_var,
                                      long long* num_batches, long long count_mult, void* workspace, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(M > 0 && C > 0 && count >= M && count_mult >= 1 && mean && invstd, "bn_act_fwd_stats: bad arguments");
  TTG_REQUIRE(sums != nullptr || (workspace != nullptr && count == M),
              "bn_act_fwd_stats: needs sums, or a workspace to reduce the local sums into (then count == M)");
  if (sums == nullptr) {
    int rc = ttg_bn_sums(x, M, C, (double*)workspace, 0, dtype, stream);
    if (rc) return rc;
    sums = (const double*)workspace;
  }
  TTG_DISPATCH(dtype, {
    BnActFwdStatsOp<T> op; op.in[0] = (const T*)x; op.out[0] = (T*)y;
    op.sums = sums; op.gamma = gamma; op.beta = beta; op.slope = slope; op.eps = eps; op.momentum = momentum;
    op.M = count; op.invM = 1.0 / (double)count; op.count_mult = count_mult; op.C = C; op.mean = mean; op.invstd = invstd;
    op.running_mean = running_mean; op.running_var = running_var; op.num_batches = num_batches;
    return launch_chan_map<T>("bn_act_fwd_stats", op, M * C, C, st);
  });
  return TTG_OK;
}
extern "C" int ttg_bn_act_fwd_stats(const void* x, void* y, long long M, int C, const double* sums, const float* gamma,
                                    const float* beta, float eps, float momentum, float slope, float* mean, float* invstd,
                                    float* running_mean, float* running_var, long long* num_batches, long long count_mult,
                                    void* workspace, int dtype, void* stream) {
  return ttg_bn_act_fwd_stats_n(x, y, M, C, M, sums, gamma, beta, eps, momentum, slope, mean, invstd, running_mean,
                                running_var, num_batches, count_mult, workspace, dtype, stream);
}

// ---------------------------------------------------------------- backward
// d = ga * lrelu'(y);  gx = gamma*invstd*(d - mean(d) - xhat*mean(d*xhat))
// per-channel cache shared by the backward ops: xhat = x*r - mr,  y = g*xhat + b
template <int V> struct BnChan { float r[V], mr[V], g[V], b[V]; };
template <int V> __device__ __forceinline__ void bn_chan_load(int c0, BnChan<V>& p, const float* mean, const float* invstd,
                                                              const float* gamma, const float* beta) {
#pragma unroll
  for (int j = 0; j < V; ++j) {
    p.r[j] = invstd[c0 + j]; p.mr[j] = mean[c0 + j] * invstd[c0 + j]; p.g[j] = gamma[c0 + j]; p.b[j] = beta[c0 + j];
  }
}
template <typename T> struct BnActBwdRedOp {
  static constexpr int NIN = 2, NACC = 2;
  const T* in[2];   // x, ga
  const float *mean, *invstd, *gamma, *beta; float slope;
  template <int V> using P = BnChan<V>;
  template <int V> __device__ __forceinline__ void load(int c0, P<V>& p) const { bn_chan_load<V>(c0, p, mean, invstd, gamma, beta); }
  template <int V> __device__ __forceinline__ void acc(const float* v, int j, const P<V>& p, float* a) const {
    float xh = v[0] * p.r[j] - p.mr[j];
    float d = v[1] * lrelu_mask(xh * p.g[j] + p.b[j], slope);
    a[0] += d; a[1] += d * xh;
  }
};
template <typename T> struct BnActBwdMapOp {
  static constexpr int NIN = 2, NOUT = 1;
  const T* in[2]; T* out[1];
  const float *mean, *invstd, *gamma, *beta; float slope; const double* sums; int C; float invM;
  float *ggamma, *gbeta; int acc;                      // parameter gradients (block 0), added to the buffers when acc
  double pscale;                                       // ... times pscale
  __device__ void finalize(int) const {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      // (accumulating: atomic, because the D(real) and D(fake) backward chains may run on two streams at once)
      const float b = (float)(sums[c] * pscale), g = (float)(sums[C + c] * pscale);
      if (gbeta) { if (acc) atomicAdd(&gbeta[c], b); else gbeta[c] = b; }
      if (ggamma) { if (acc) atomicAdd(&ggamma[c], g); else ggamma[c] = g; }
    }
  }
  template <int V> struct P { BnChan<V> c; float db[V], cc[V]; };
  template <int V> __device__ __forceinline__ void load(int c0, P<V>& p) const {
    bn_chan_load<V>(c0, p.c, mean, invstd, gamma, beta);
#pragma unroll
    for (int j = 0; j < V; ++j) { p.db[j] = (float)sums[c0 + j] * invM; p.cc[j] = (float)sums[C + c0 + j] * invM; }
  }
  template <int V> __device__ __forceinline__ void apply(const float* v, int j, const P<V>& p, float* o) const {
    float xh = v[0] * p.c.r[j] - p.c.mr[j];
    float d = v[1] * lrelu_mask(xh * p.c.g[j] + p.c.b[j], slope);
    o[0] = p.c.g[j] * p.c.r[j] * (d - p.db[j] - xh * p.cc[j]);
  }
};
// acc != 0: the parameter gradients are ADDED to ggamma / gbeta (the caller passes views of the flat .grad buffer, so
// autograd's AccumulateGrad add kernels disappear)
__global__ void bn_param_grads_kernel(const double* sums, int C, float* ggamma, float* gbeta, int acc, double pscale) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    const float b = (float)(sums[c] * pscale), g = (float)(sums[C + c] * pscale);
    if (gbeta) { if (acc) atomicAdd(&gbeta[c], b); else gbeta[c] = b; }
    if (ggamma) { if (acc) atomicAdd(&ggamma[c], g); else ggamma[c] = g; }
  }
}

// The backward as two entry points, so that the 2C sums can be all-reduced between them (synchronised BatchNorm).
// reduce: sums[2C] = {sum d, sum d*xhat} over the M local rows; flags bit 1: sums is already zero.
extern "C" int ttg_bn_act_bwd_reduce(const void* x, const void* ga, long long M, int C, const float* mean,
                                     const float* invstd, const float* gamma, const float* beta, float slope, double* sums,
                                     int flags, int dtype, void* stream) {
  TTG_REQUIRE(M > 0 && C > 0 && sums != nullptr, "bn_act_bwd_reduce: bad arguments");
  TTG_DISPATCH(dtype, {
    BnActBwdRedOp<T> r; r.in[0] = (const T*)x; r.in[1] = (const T*)ga;
    r.mean = mean; r.invstd = invstd; r.gamma = gamma; r.beta = beta; r.slope = slope;
    return launch_chan_reduce<T>("bn_act_bwd_reduce", r, M, C, sums, (cudaStream_t)stream, (flags & 2) != 0);
  });
  return TTG_OK;
}
// apply: gx over the M local rows from sums taken over `count` pixels; ggamma / gbeta = param_scale * sums (written, or
// added when accumulate bit 0 is set).  gx NULL: parameter gradients only.
extern "C" int ttg_bn_act_bwd_apply(const void* x, const void* ga, void* gx, long long M, int C, long long count,
                                    const double* sums, const float* mean, const float* invstd, const float* gamma,
                                    const float* beta, float slope, float* ggamma, float* gbeta, float param_scale,
                                    int accumulate, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  TTG_REQUIRE(M > 0 && C > 0 && count >= M && sums != nullptr, "bn_act_bwd_apply: bad arguments");
  if (gx) {
    TTG_DISPATCH(dtype, {
      BnActBwdMapOp<T> m; m.in[0] = (const T*)x; m.in[1] = (const T*)ga; m.out[0] = (T*)gx;
      m.mean = mean; m.invstd = invstd; m.gamma = gamma; m.beta = beta; m.slope = slope;
      m.sums = sums; m.C = C; m.invM = 1.f / (float)count;
      m.ggamma = ggamma; m.gbeta = gbeta; m.acc = accumulate & 1; m.pscale = (double)param_scale;
      return launch_chan_map<T>("bn_act_bwd_apply", m, M * C, C, st);
    });
  } else if (ggamma || gbeta) {                         // (with gx the apply pass writes them)
    bn_param_grads_kernel<<<(C + 127) / 128, 128, 0, st>>>(sums, C, ggamma, gbeta, accumulate & 1, (double)param_scale);
    TTG_CHECK_LAUNCH("bn_param_grads");
  }
  return TTG_OK;
}

extern "C" int ttg_bn_act_bwd_acc(const void* x, const void* ga, void* gx, long long M, int C, const float* mean,
                                  const float* invstd, const float* gamma, const float* beta, float slope, float* ggamma,
                                  float* gbeta, int accumulate, void* workspace, int dtype, void* stream) {
  int rc = ttg_bn_act_bwd_reduce(x, ga, M, C, mean, invstd, gamma, beta, slope, (double*)workspace, accumulate & 2, dtype,
                                 stream);
  if (rc) return rc;
  return ttg_bn_act_bwd_apply(x, ga, gx, M, C, M, (const double*)workspace, mean, invstd, gamma, beta, slope, ggamma,
                              gbeta, 1.f, accumulate & 1, dtype, stream);
}
extern "C" int ttg_bn_act_bwd(const void* x, const void* ga, void* gx, long long M, int C, const float* mean,
                              const float* invstd, const float* gamma, const float* beta, float slope, float* ggamma,
                              float* gbeta, void* workspace, int dtype, void* stream) {
  return ttg_bn_act_bwd_acc(x, ga, gx, M, C, mean, invstd, gamma, beta, slope, ggamma, gbeta, 0, workspace, dtype, stream);
}

// ---------------------------------------------------------------- backward of backward
// Given u = cotangent of gx (see DESIGN.md "BN double backward"):
//   g_ga = m * gamma*r * P(u)
//   g_x  = gamma*r^2 * [ xhat*(c*e - cov) - e*P(d) - c*P(u) ]
//   g_gamma = r * M * (cov - c*e)
// with P(v) = v - mean(v) - xhat*mean(v*xhat), c = mean(d*xhat), e = mean(u*xhat),
// cov = mean(u*d) - mean(u)*mean(d).
template <typename T> struct BnActBwd2RedOp {
  static constexpr int NIN = 3, NACC = 5;
  const T* in[3];   // x, ga, u
  const float *mean, *invstd, *gamma, *beta; float slope;
  template <int V> using P = BnChan<V>;
  template <int V> __device__ __forceinline__ void load(int c0, P<V>& p) const { bn_chan_load<V>(c0, p, mean, invstd, gamma, beta); }
  template <int V> __device__ __forceinline__ void acc(const float* v, int j, const P<V>& p, float* a) const {
    float xh = v[0] * p.r[j] - p.mr[j];
    float d = v[1] * lrelu_mask(xh * p.g[j] + p.b[j], slope);
    float u = v[2];
    a[0] += d; a[1] += d * xh; a[2] += u; a[3] += u * xh; a[4] += u * d;
  }
};
template <typename T> struct BnActBwd2MapOp {
  static constexpr int NIN = 3, NOUT = 2;
  const T* in[3]; T* out[2];   // out: g_ga, g_x
  const float *mean, *invstd, *gamma, *beta; float slope; const double* sums; int C; float invM;
  float* ggamma; long long M; int acc;                 // M: the pixel count of the sums
  double pscale;                                       // ggamma = pscale * g_gamma
  __device__ void finalize(int) const {
    if (!ggamma) return;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      const double iM = 1.0 / (double)M;
      const double db = sums[c] * iM, cc = sums[C + c] * iM, ub = sums[2 * C + c] * iM, e = sums[3 * C + c] * iM;
      const double cov = sums[4 * C + c] * iM - ub * db;
      const float v = (float)((double)invstd[c] * (double)M * (cov - cc * e) * pscale);
      if (acc) atomicAdd(&ggamma[c], v); else ggamma[c] = v;
    }
  }
  template <int V> struct P { BnChan<V> c; float db[V], cc[V], ub[V], e[V], k[V]; };   // k = cc*e - cov
  template <int V> __device__ __forceinline__ void load(int c0, P<V>& p) const {
    bn_chan_load<V>(c0, p.c, mean, invstd, gamma, beta);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float db = (float)sums[c0 + j] * invM, cc = (float)sums[C + c0 + j] * invM;
      float ub = (float)sums[2 * C + c0 + j] * invM, e = (float)sums[3 * C + c0 + j] * invM;
      float cov = (float)sums[4 * C + c0 + j] * invM - ub * db;
      p.db[j] = db; p.cc[j] = cc; p.ub[j] = ub; p.e[j] = e; p.k[j] = cc * e - cov;
    }
  }
  template <int V> __device__ __forceinline__ void apply(const float* v, int j, const P<V>& p, float* o) const {
    float r = p.c.r[j], g = p.c.g[j];
    float xh = v[0] * r - p.c.mr[j];
    float m = lrelu_mask(xh * g + p.c.b[j], slope);
    float d = v[1] * m, u = v[2];
    float Pd = d - p.db[j] - xh * p.cc[j], Pu = u - p.ub[j] - xh * p.e[j];
    o[0] = m * g * r * Pu;
    o[1] = g * r * r * (xh * p.k[j] - p.e[j] * Pd - p.cc[j] * Pu);
  }
};
__global__ void bn_bwd2_gamma_kernel(const double* sums, const float* invstd, long long M, int C, float* ggamma, int acc) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    double invM = 1.0 / (double)M;
    double db = sums[c] * invM, cc = sums[C + c] * invM, ub = sums[2 * C + c] * invM, e = sums[3 * C + c] * invM;
    double cov = sums[4 * C + c] * invM - ub * db;
    const float v = (float)((double)invstd[c] * (double)M * (cov - cc * e));
    if (acc) atomicAdd(&ggamma[c], v); else ggamma[c] = v;
  }
}

// The same split for the double backward: reduce -> sums[5C] over the M local rows (flags bit 1: already zero);
// apply -> g_ga, g_x over the M local rows from sums taken over `count` pixels, ggamma = param_scale * g_gamma.
extern "C" int ttg_bn_act_bwd2_reduce(const void* x, const void* ga, const void* u, long long M, int C, const float* mean,
                                      const float* invstd, const float* gamma, const float* beta, float slope,
                                      double* sums, int flags, int dtype, void* stream) {
  TTG_REQUIRE(M > 0 && C > 0 && sums != nullptr, "bn_act_bwd2_reduce: bad arguments");
  TTG_DISPATCH(dtype, {
    BnActBwd2RedOp<T> r; r.in[0] = (const T*)x; r.in[1] = (const T*)ga; r.in[2] = (const T*)u;
    r.mean = mean; r.invstd = invstd; r.gamma = gamma; r.beta = beta; r.slope = slope;
    return launch_chan_reduce<T>("bn_act_bwd2_reduce", r, M, C, sums, (cudaStream_t)stream, (flags & 2) != 0);
  });
  return TTG_OK;
}
extern "C" int ttg_bn_act_bwd2_apply(const void* x, const void* ga, const void* u, void* g_ga, void* g_x, long long M,
                                     int C, long long count, const double* sums, const float* mean, const float* invstd,
                                     const float* gamma, const float* beta, float slope, float* ggamma, float param_scale,
                                     int accumulate, int dtype, void* stream) {
  TTG_REQUIRE(M > 0 && C > 0 && count >= M && sums != nullptr, "bn_act_bwd2_apply: bad arguments");
  TTG_DISPATCH(dtype, {
    BnActBwd2MapOp<T> m; m.in[0] = (const T*)x; m.in[1] = (const T*)ga; m.in[2] = (const T*)u;
    m.out[0] = (T*)g_ga; m.out[1] = (T*)g_x;
    m.mean = mean; m.invstd = invstd; m.gamma = gamma; m.beta = beta; m.slope = slope;
    m.sums = sums; m.C = C; m.invM = 1.f / (float)count;
    m.ggamma = ggamma; m.M = count; m.acc = accumulate & 1; m.pscale = (double)param_scale;
    return launch_chan_map<T>("bn_act_bwd2_apply", m, M * C, C, (cudaStream_t)stream);
  });
  return TTG_OK;
}

extern "C" int ttg_bn_act_bwd2_acc(const void* x, const void* ga, const void* u, void* g_ga, void* g_x, long long M, int C,
                                   const float* mean, const float* invstd, const float* gamma, const float* beta,
                                   float slope, float* ggamma, int accumulate, void* workspace, int dtype, void* stream) {
  int rc = ttg_bn_act_bwd2_reduce(x, ga, u, M, C, mean, invstd, gamma, beta, slope, (double*)workspace, accumulate & 2,
                                  dtype, stream);
  if (rc) return rc;
  return ttg_bn_act_bwd2_apply(x, ga, u, g_ga, g_x, M, C, M, (const double*)workspace, mean, invstd, gamma, beta, slope,
                               ggamma, 1.f, accumulate & 1, dtype, stream);
}
extern "C" int ttg_bn_act_bwd2(const void* x, const void* ga, const void* u, void* g_ga, void* g_x, long long M, int C,
                               const float* mean, const float* invstd, const float* gamma, const float* beta,
                               float slope, float* ggamma, void* workspace, int dtype, void* stream) {
  return ttg_bn_act_bwd2_acc(x, ga, u, g_ga, g_x, M, C, mean, invstd, gamma, beta, slope, ggamma, 0, workspace, dtype, stream);
}

// ---------------------------------------------------------------- plain LeakyReLU (--norm id)
template <typename T> struct LreluOp : NoParams {     // y = lrelu(x)
  static constexpr int NIN = 1, NOUT = 1;
  const T* in[1]; T* out[1]; float slope;
  template <int V> __device__ __forceinline__ void apply(const float* v, int, const P<V>&, float* o) const { o[0] = lrelu(v[0], slope); }
};
template <typename T> struct LreluMaskMulOp : NoParams {   // out = g * lrelu'(x)
  static constexpr int NIN = 2, NOUT = 1;
  const T* in[2]; T* out[1]; float slope;
  template <int V> __device__ __forceinline__ void apply(const float* v, int, const P<V>&, float* o) const { o[0] = v[1] * lrelu_mask(v[0], slope); }
};
extern "C" int ttg_lrelu_fwd(const void* x, void* y, long long n, float slope, int dtype, void* stream) {
  TTG_DISPATCH(dtype, {
    LreluOp<T> op; op.in[0] = (const T*)x; op.out[0] = (T*)y; op.slope = slope;
    return launch_chan_map<T>("lrelu_fwd", op, n, (n % 8 == 0) ? 8 : 1, (cudaStream_t)stream);
  });
  return TTG_OK;
}
extern "C" int ttg_lrelu_bwd(const void* x, const void* g, void* gx, long long n, float slope, int dtype, void* stream) {
  TTG_DISPATCH(dtype, {
    LreluMaskMulOp<T> op; op.in[0] = (const T*)x; op.in[1] = (const T*)g; op.out[0] = (T*)gx; op.slope = slope;
    return launch_chan_map<T>("lrelu_bwd", op, n, (n % 8 == 0) ? 8 : 1, (cudaStream_t)stream);
  });
  return TTG_OK;
}

// ---------------------------------------------------------------- ELU / SELU (--activation elu|selu, trainers/cnn.py:41-45)
// f(x) = scale * (x > 0 ? x : alpha * (exp(x) - 1));  nn.ELU: alpha 1, scale 1;  nn.SELU: alpha 1.6732632..., scale 1.0507009...
// order 0: y = f(x);  order 1: out = g * f'(x);  order 2: out = g * u * f''(x)  (the x-cotangent of the order-1 op under R1)
template <typename T, int ORDER> struct EluOp : NoParams {
  static constexpr int NIN = ORDER + 1, NOUT = 1;
  const T* in[ORDER + 1]; T* out[1]; float alpha, scale;
  template <int V> __device__ __forceinline__ void apply(const float* v, int, const P<V>&, float* o) const {
    const float x = v[0];
    const float e = scale * alpha * __expf(fminf(x, 0.f));        // = f'(x) = f''(x) for x <= 0
    if constexpr (ORDER == 0) o[0] = x > 0.f ? scale * x : scale * alpha * expm1f(x);
    else if constexpr (ORDER == 1) o[0] = v[1] * (x > 0.f ? scale : e);
    else o[0] = x > 0.f ? 0.f : v[1] * v[2] * e;
  }
};
template <int ORDER>
static int elu_launch(const char* name, const void* x, const void* a, const void* b, void* out, long long n, float alpha,
                      float scale, int dtype, void* stream) {
  TTG_DISPATCH(dtype, {
    EluOp<T, ORDER> op; op.in[0] = (const T*)x;
    if constexpr (ORDER >= 1) op.in[1] = (const T*)a;
    if constexpr (ORDER >= 2) op.in[2] = (const T*)b;
    op.out[0] = (T*)out; op.alpha = alpha; op.scale = scale;
    return launch_chan_map<T>(name, op, n, (n % 8 == 0) ? 8 : 1, (cudaStream_t)stream);
  });
  return TTG_OK;
}
extern "C" int ttg_elu_fwd(const void* x, void* y, long long n, float alpha, float scale, int dtype, void* stream) {
  return elu_launch<0>("elu_fwd", x, nullptr, nullptr, y, n, alpha, scale, dtype, stream);
}
extern "C" int ttg_elu_bwd(const void* x, const void* g, void* gx, long long n, float alpha, float scale, int dtype, void* stream) {
  return elu_launch<1>("elu_bwd", x, g, nullptr, gx, n, alpha, scale, dtype, stream);
}
extern "C" int ttg_elu_bwd2(const void* x, const void* g, const void* u, void* out, long long n, float alpha, float scale,
                            int dtype, void* stream) {
  return elu_launch<2>("elu_bwd2", x, g, u, out, n, alpha, scale, dtype, stream);
}

// ---------------------------------------------------------------- per-channel sum (conv bias gradient)
template <typename T> struct SumOp : NoParams {
  static constexpr int NIN = 1, NACC = 1;
  const T* in[1];
  template <int V> __device__ __forceinline__ void acc(const float* v, int, const P<V>&, float* a) const { a[0] += v[0]; }
};
__global__ void d2f_kernel(const double* s, int n, float* o, int acc) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = (acc ? o[i] : 0.f) + (float)s[i];
}
extern "C" int ttg_channel_sum_acc(const void* x, long long M, int C, float* out, int accumulate, void* workspace, int dtype, void* stream);
extern "C" int ttg_channel_sum(const void* x, long long M, int C, float* out, void* workspace, int dtype, void* stream) {
  return ttg_channel_sum_acc(x, M, C, out, 0, workspace, dtype, stream);
}
extern "C" int ttg_channel_sum_acc(const void* x, long long M, int C, float* out, int accumulate, void* workspace, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  double* ws = (double*)workspace;
  TTG_DISPATCH(dtype, {
    SumOp<T> op; op.in[0] = (const T*)x;
    int rc = launch_chan_reduce<T>("channel_sum", op, M, C, ws, st, (accumulate & 2) != 0);
    if (rc) return rc;
  });
  d2f_kernel<<<(C + 127) / 128, 128, 0, st>>>(ws, C, out, accumulate & 1);
  TTG_CHECK_LAUNCH("channel_sum_finalize");
  return TTG_OK;
}
