// Generic NHWC channel-wise drivers: a per-channel reduction over rows and an
// element-wise map with per-channel parameters.  Both are pure HBM streams:
// 16-byte vector accesses, coalesced along the channel (fastest) dimension,
// grid sized in multiples of the SM count (grid-stride loops).
#pragma once
#include "common.cuh"
#include <type_traits>

// Vector width per (dtype, Op): 16-byte vectors unless the Op asks for 4-element bf16 vectors (`BF16_V = 4`).
// Measured on B200 (bn_act_bwd, M = 4 Mi, C = 16): 8 channels per thread (80 / 105 registers, 3 / 2 blocks per SM)
// 182 us; 4 channels per thread (60 / 63 registers, 4 blocks per SM) 203 us -> every op keeps 16-byte vectors.
template <class Op, class = void> struct OpBf16V { static constexpr int value = 8; };
template <class Op> struct OpBf16V<Op, std::void_t<decltype(Op::BF16_V)>> { static constexpr int value = Op::BF16_V; };
template <typename T, class Op> struct ChanV { static constexpr int value = Vec<T>::N; };
template <class Op> struct ChanV<bf16, Op> { static constexpr int value = OpBf16V<Op>::value; };

// Op concept for reductions:
//   static constexpr int NIN, NACC;   const T* in[NIN];
//   template <int V> struct P { ... };                       per-thread cache of per-channel parameters
//   template <int V> __device__ void load(int c0, P<V>&) const;   (channels c0..c0+V-1, loaded ONCE per thread)
//   template <int V> __device__ void acc(const float* v /*NIN*/, int j, const P<V>&, float* a /*NACC*/) const;
template <typename T, int V, class Op>
__global__ void __launch_bounds__(256) chan_reduce_kernel(Op op, long long M, int C, double* __restrict__ out) {
  // block-level accumulators in DOUBLE: the warps add their partial sums with shared-memory atomics in arrival order; in
  // fp32 that order changed the statistics in the 7th digit from run to run, enough to flip a LeakyReLU mask now and then
  // (a rare, box-dependent 1 % deviation of a small gradient tensor in the fp32 parity tests); in fp64 it cannot
  extern __shared__ double s_acc[];   // [NACC][C]
  for (int i = threadIdx.x; i < Op::NACC * C; i += blockDim.x) s_acc[i] = 0.0;
  __syncthreads();
  const int groups = C / V;
  const int rpi = blockDim.x / groups;           // rows per block iteration
  const int g = threadIdx.x % groups, rsub = threadIdx.x / groups;
  float a[Op::NACC][V];
#pragma unroll
  for (int k = 0; k < Op::NACC; ++k)
#pragma unroll
    for (int j = 0; j < V; ++j) a[k][j] = 0.f;
  if (rsub < rpi) {
    typename Op::template P<V> prm;
    op.template load<V>(g * V, prm);
    constexpr int U = 2;                           // rows in flight per thread (4 measured slower: registers)
    const long long rstep = (long long)gridDim.x * rpi;
    long long r0 = (long long)blockIdx.x * rpi + rsub;
    for (; r0 + (U - 1) * rstep < M; r0 += U * rstep) {
      float v[U][Op::NIN][V];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long base = (r0 + u * rstep) * C + (long long)g * V;
#pragma unroll
        for (int t = 0; t < Op::NIN; ++t) {
          if constexpr (V == 1) v[u][t][0] = to_f(op.in[t][base]);
          else { VecN<T, V> q; q.load(op.in[t] + base); q.unpack(v[u][t]); }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int j = 0; j < V; ++j) {
          float vin[Op::NIN], acc[Op::NACC];
#pragma unroll
          for (int t = 0; t < Op::NIN; ++t) vin[t] = v[u][t][j];
#pragma unroll
          for (int k = 0; k < Op::NACC; ++k) acc[k] = a[k][j];
          op.template acc<V>(vin, j, prm, acc);
#pragma unroll
          for (int k = 0; k < Op::NACC; ++k) a[k][j] = acc[k];
        }
    }
    for (; r0 < M; r0 += rstep) {
      const long long base = r0 * C + (long long)g * V;
      float v[Op::NIN][V];
#pragma unroll
      for (int t = 0; t < Op::NIN; ++t) {
        if constexpr (V == 1) v[t][0] = to_f(op.in[t][base]);
        else { VecN<T, V> q; q.load(op.in[t] + base); q.unpack(v[t]); }
      }
#pragma unroll
      for (int j = 0; j < V; ++j) {
        float vin[Op::NIN], acc[Op::NACC];
#pragma unroll
        for (int t = 0; t < Op::NIN; ++t) vin[t] = v[t][j];
#pragma unroll
        for (int k = 0; k < Op::NACC; ++k) acc[k] = a[k][j];
        op.template acc<V>(vin, j, prm, acc);
#pragma unroll
        for (int k = 0; k < Op::NACC; ++k) a[k][j] = acc[k];
      }
    }
  }
  // block reduction: lanes that own the same channel group are first combined with warp shuffles
  // (power-of-two group counts), then one shared-memory atomic per (warp, channel)
  const bool pow2 = (groups & (groups - 1)) == 0 && groups <= 32;
  if (pow2) {
#pragma unroll
    for (int k = 0; k < Op::NACC; ++k)
#pragma unroll
      for (int j = 0; j < V; ++j) {
        float t = a[k][j];
        for (int o = 16; o >= groups; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        a[k][j] = t;
      }
  }
  if (rsub < rpi && (!pow2 || (threadIdx.x & 31) < groups)) {
#pragma unroll
    for (int k = 0; k < Op::NACC; ++k)
#pragma unroll
      for (int j = 0; j < V; ++j) atomicAdd(&s_acc[k * C + g * V + j], (double)a[k][j]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < Op::NACC * C; i += blockDim.x) atomicAdd(&out[i], s_acc[i]);
}


// ====================================================================================================================
// Bulk-copy (TMA 1-D) pipelined variants for bf16 tensors.  The register-fed kernels above keep at most
// 2 x NIN 16-byte loads per thread in flight, and the per-channel coefficients cost them most of their occupancy
// (80-180 registers), so they stall at 45-60 % of HBM bandwidth.  Here one producer lane streams 8 KB chunks of every
// input tensor into a 4-stage shared-memory ring with cp.async.bulk (bytes in flight per SM no longer depend on
// registers or occupancy); the 8 consumer warps read the ring with LDS.128, apply the same Op, and write results
// with coalesced 16-byte stores.
// Requirements: bf16, 16-byte aligned, (C / 8) a power of two <= 32  ->  a thread always sees the same 8 channels.
#include "tc_common.cuh"
#define CB_STAGES 4
#define CB_UNITS 512                      // 16-byte units per tensor per stage (8 KB)
#define CB_THREADS 288                    // 8 consumer warps + 1 producer warp

template <class Op>
__device__ __forceinline__ void cb_producer(const Op& op, uint8_t* ring, uint64_t* full, uint64_t* empty, long long nvec,
                                            long long nchunks) {
  if (!elect_one()) return;
  int it = 0;
  for (long long c = blockIdx.x; c < nchunks; c += gridDim.x, ++it) {
    const int s = it % CB_STAGES;
    if (it >= CB_STAGES) mbar_wait(&empty[s], (uint32_t)((it / CB_STAGES) - 1) & 1u);
    const long long off = c * CB_UNITS;
    const uint32_t units = (uint32_t)min((long long)CB_UNITS, nvec - off);
    const uint32_t bytes = units * 16u;
    const uint32_t bar = smem_u32(&full[s]);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * Op::NIN) : "memory");
#pragma unroll
    for (int t = 0; t < Op::NIN; ++t) {
      const uint8_t* src = reinterpret_cast<const uint8_t*>(op.in[t]) + off * 16;
      const uint32_t dst = smem_u32(ring + ((size_t)s * Op::NIN + t) * CB_UNITS * 16);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
    }
  }
}

// Optional per-launch epilogue of a map op: `__device__ void finalize(int C) const`, run by block 0 (all its threads)
// before the streaming loop - per-channel outputs derived from already reduced sums (parameter gradients, saved
// BatchNorm statistics) ride along with the apply pass instead of costing one more tiny kernel launch each.
template <class Op, class = void> struct chan_has_finalize : std::false_type {};
template <class Op> struct chan_has_finalize<Op, std::void_t<decltype(&Op::finalize)>> : std::true_type {};

template <class Op>
__global__ void __launch_bounds__(CB_THREADS) chan_map_bulk_kernel(Op op, long long nvec, int C) {
  extern __shared__ __align__(128) uint8_t cb_smem[];
  uint8_t* ring = cb_smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)CB_STAGES * Op::NIN * CB_UNITS * 16);
  uint64_t* empty = full + CB_STAGES;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    for (int i = 0; i < CB_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 8); }
    mbar_fence_init();
  }
  __syncthreads();
  if constexpr (chan_has_finalize<Op>::value) { if (blockIdx.x == 0) op.finalize(C); }
  const long long nchunks = (nvec + CB_UNITS - 1) / CB_UNITS;
  if (warp == 8) { cb_producer(op, ring, full, empty, nvec, nchunks); return; }
  typename Op::template P<8> prm;
  op.template load<8>((tid % (C >> 3)) * 8, prm);
  int it = 0;
  for (long long c = blockIdx.x; c < nchunks; c += gridDim.x, ++it) {
    const int s = it % CB_STAGES;
    const long long off = c * CB_UNITS;
    const int units = (int)min((long long)CB_UNITS, nvec - off);
    mbar_wait(&full[s], (uint32_t)(it / CB_STAGES) & 1u);
#pragma unroll
    for (int k = 0; k < CB_UNITS / 256; ++k) {
      const int u = tid + 256 * k;
      if (u < units) {
        float v[Op::NIN][8], o[Op::NOUT][8];
#pragma unroll
        for (int t = 0; t < Op::NIN; ++t) {
          Vec<bf16> q;
          q.raw = *reinterpret_cast<const uint4*>(ring + (((size_t)s * Op::NIN + t) * CB_UNITS + u) * 16);
          q.unpack(v[t]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float vin[Op::NIN], vout[Op::NOUT];
#pragma unroll
          for (int t = 0; t < Op::NIN; ++t) vin[t] = v[t][j];
          op.template apply<8>(vin, j, prm, vout);
#pragma unroll
          for (int t = 0; t < Op::NOUT; ++t) o[t][j] = vout[t];
        }
#pragma unroll
        for (int t = 0; t < Op::NOUT; ++t) { Vec<bf16> q; q.pack(o[t]); q.store(op.out[t] + (off + u) * 8); }
      }
    }
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&empty[s]);
  }
}

template <class Op>
__global__ void __launch_bounds__(CB_THREADS) chan_reduce_bulk_kernel(Op op, long long nvec, int C, double* __restrict__ out) {
  extern __shared__ __align__(128) uint8_t cb_smem[];
  uint8_t* ring = cb_smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)CB_STAGES * Op::NIN * CB_UNITS * 16);
  uint64_t* empty = full + CB_STAGES;
  double* s_acc = reinterpret_cast<double*>(empty + CB_STAGES);        // [NACC][C] (double: see chan_reduce_kernel)
  const int tid = threadIdx.x, warp = tid >> 5;
  for (int i = tid; i < Op::NACC * C; i += blockDim.x) s_acc[i] = 0.0;
  if (tid == 0) {
    for (int i = 0; i < CB_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 8); }
    mbar_fence_init();
  }
  __syncthreads();
  const long long nchunks = (nvec + CB_UNITS - 1) / CB_UNITS;
  const int groups = C >> 3, g = tid % groups;
  if (warp == 8) {
    cb_producer(op, ring, full, empty, nvec, nchunks);
  } else {
    float a[Op::NACC][8];
#pragma unroll
    for (int k = 0; k < Op::NACC; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) a[k][j] = 0.f;
    typename Op::template P<8> prm;
    op.template load<8>(g * 8, prm);
    int it = 0;
    for (long long c = blockIdx.x; c < nchunks; c += gridDim.x, ++it) {
      const int s = it % CB_STAGES;
      const int units = (int)min((long long)CB_UNITS, nvec - c * CB_UNITS);
      mbar_wait(&full[s], (uint32_t)(it / CB_STAGES) & 1u);
#pragma unroll
      for (int k = 0; k < CB_UNITS / 256; ++k) {
        const int u = tid + 256 * k;
        if (u < units) {
          float v[Op::NIN][8];
#pragma unroll
          for (int t = 0; t < Op::NIN; ++t) {
            Vec<bf16> q;
            q.raw = *reinterpret_cast<const uint4*>(ring + (((size_t)s * Op::NIN + t) * CB_UNITS + u) * 16);
            q.unpack(v[t]);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float vin[Op::NIN], acc[Op::NACC];
#pragma unroll
            for (int t = 0; t < Op::NIN; ++t) vin[t] = v[t][j];
#pragma unroll
            for (int k2 = 0; k2 < Op::NACC; ++k2) acc[k2] = a[k2][j];
            op.template acc<8>(vin, j, prm, acc);
#pragma unroll
            for (int k2 = 0; k2 < Op::NACC; ++k2) a[k2][j] = acc[k2];
          }
        }
      }
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(&empty[s]);
    }
    // lanes that own the same channel group are combined with shuffles, then one shared atomic per (warp, channel)
#pragma unroll
    for (int k = 0; k < Op::NACC; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float t = a[k][j];
        for (int o = 16; o >= groups; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        a[k][j] = t;
      }
    if ((tid & 31) < groups) {
#pragma unroll
      for (int k = 0; k < Op::NACC; ++k)
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(&s_acc[k * C + g * 8 + j], (double)a[k][j]);
    }
  }
  __syncthreads();
  for (int i = tid; i < Op::NACC * C; i += blockDim.x) atomicAdd(&out[i], s_acc[i]);
}

template <typename T, class Op> static inline bool cb_ok(int C, const void* const* ptrs, int n, long long nelem) {
  if (!std::is_same<T, bf16>::value) return false;
  const int groups = C >> 3;
  if (C % 8 || groups < 1 || groups > 32 || (groups & (groups - 1)) || nelem % 8) return false;
  for (int i = 0; i < n; ++i)
    if (reinterpret_cast<uintptr_t>(ptrs[i]) & 15) return false;
  return nelem >= 8LL * CB_UNITS * 148;            // small tensors: the register kernels (less fixed cost)
}
template <class Kern> static inline int cb_grid(Kern kernel, long long nchunks, size_t smem, int* err) {
  static std::mutex mu;
  static std::unordered_map<const void*, size_t> done;
  {
    std::lock_guard<std::mutex> lock(mu);
    auto it = done.find((const void*)kernel);
    if (it == done.end() || it->second < smem) {
      if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { *err = 1; return 1; }
      done[(const void*)kernel] = smem;
    }
  }
  long long cap = (long long)ttg_num_sms() * ttg_blocks_per_sm((const void*)kernel, CB_THREADS, smem);
  long long b = nchunks < cap ? nchunks : cap;
  return (int)(b < 1 ? 1 : b);
}

template <typename T> static inline bool ttg_vec_ok(int C, const void* const* ptrs, int n, int vec = Vec<T>::N) {
  if (C % vec) return false;
  for (int i = 0; i < n; ++i)
    if (reinterpret_cast<uintptr_t>(ptrs[i]) & 15) return false;
  return true;
}


// ====================================================================================================================
// C == 3 (the RGB tensors at the discriminator's input / the generator's output, 25 MB each at the headline size): the
// generic fallback for channel counts that are not a multiple of the vector width moves ONE 2-byte element per thread
// and instruction (measured < 1 TB/s: bn_act_fwd 64 us, bn_act_bwd 82 us at M = 4 Mi).  Here a thread owns groups of
// three 16-byte vectors (24 bf16 = 8 pixels, or 12 fp32 = 4 pixels): the channel of element e of a group is e % 3, a
// compile-time pattern, so the three per-channel parameter sets live in registers and every access is a vector.
template <typename T, class Op>
__global__ void __launch_bounds__(256) chan_map_c3_kernel(Op op, long long ngroups) {
  constexpr int VN = Vec<T>::N, G = 3 * VN;
  typename Op::template P<1> prm[3];
  if constexpr (chan_has_finalize<Op>::value) { if (blockIdx.x == 0) op.finalize(3); }
#pragma unroll
  for (int c = 0; c < 3; ++c) op.template load<1>(c, prm[c]);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
    float v[Op::NIN][G], o[Op::NOUT][G];
#pragma unroll
    for (int t = 0; t < Op::NIN; ++t)
#pragma unroll
      for (int k = 0; k < 3; ++k) { VecN<T, VN> q; q.load(op.in[t] + g * G + k * VN); q.unpack(&v[t][k * VN]); }
#pragma unroll
    for (int e = 0; e < G; ++e) {
      float vin[Op::NIN], vout[Op::NOUT];
#pragma unroll
      for (int t = 0; t < Op::NIN; ++t) vin[t] = v[t][e];
      op.template apply<1>(vin, 0, prm[e % 3], vout);
#pragma unroll
      for (int t = 0; t < Op::NOUT; ++t) o[t][e] = vout[t];
    }
#pragma unroll
    for (int t = 0; t < Op::NOUT; ++t)
#pragma unroll
      for (int k = 0; k < 3; ++k) { VecN<T, VN> q; q.pack(&o[t][k * VN]); q.store(op.out[t] + g * G + k * VN); }
  }
}
template <typename T, class Op>
__global__ void __launch_bounds__(256) chan_reduce_c3_kernel(Op op, long long ngroups, double* __restrict__ out) {
  constexpr int VN = Vec<T>::N, G = 3 * VN;
  __shared__ double s_acc[Op::NACC * 3];
  if (threadIdx.x < Op::NACC * 3) s_acc[threadIdx.x] = 0.0;
  __syncthreads();
  typename Op::template P<1> prm[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) op.template load<1>(c, prm[c]);
  float a[3][Op::NACC];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int k = 0; k < Op::NACC; ++k) a[c][k] = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
    float v[Op::NIN][G];
#pragma unroll
    for (int t = 0; t < Op::NIN; ++t)
#pragma unroll
      for (int k = 0; k < 3; ++k) { VecN<T, VN> q; q.load(op.in[t] + g * G + k * VN); q.unpack(&v[t][k * VN]); }
#pragma unroll
    for (int e = 0; e < G; ++e) {
      float vin[Op::NIN];
#pragma unroll
      for (int t = 0; t < Op::NIN; ++t) vin[t] = v[t][e];
      op.template acc<1>(vin, 0, prm[e % 3], a[e % 3]);
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int k = 0; k < Op::NACC; ++k) {
      float t = a[c][k];
      for (int o = 16; o >= 1; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if ((threadIdx.x & 31) == 0) atomicAdd(&s_acc[k * 3 + c], (double)t);
    }
  __syncthreads();
  if (threadIdx.x < Op::NACC * 3) atomicAdd(&out[threadIdx.x], s_acc[threadIdx.x]);
}
template <typename T> static inline bool c3_ok(int C, const void* const* ptrs, int nptr, long long n) {
  if (C != 3 || n % (3 * Vec<T>::N)) return false;
  for (int i = 0; i < nptr; ++i)
    if (reinterpret_cast<uintptr_t>(ptrs[i]) & 15) return false;
  return true;
}

// out must hold NACC*C doubles; zeroed here unless the caller guarantees it already is (out_is_zero).
template <typename T, class Op>
static int launch_chan_reduce(const char* name, Op op, long long M, int C, double* out, cudaStream_t st, bool out_is_zero = false) {
  if (!out_is_zero) cudaMemsetAsync(out, 0, sizeof(double) * Op::NACC * C, st);
  const void* ptrs[Op::NIN];
  for (int i = 0; i < Op::NIN; ++i) ptrs[i] = op.in[i];
  if (c3_ok<T>(C, ptrs, Op::NIN, M * C)) {
    const long long ngroups = M * C / (3 * Vec<T>::N);
    chan_reduce_c3_kernel<T, Op><<<ttg_grid_occ(chan_reduce_c3_kernel<T, Op>, ngroups, 256 * 2), 256, 0, st>>>(op, ngroups, out);
    TTG_CHECK_LAUNCH(name);
    return TTG_OK;
  }
  if constexpr (std::is_same<T, bf16>::value) {
    if (cb_ok<T, Op>(C, ptrs, Op::NIN, M * C)) {
      const long long nvec = M * C / 8, nchunks = (nvec + CB_UNITS - 1) / CB_UNITS;
      const size_t bsmem = (size_t)CB_STAGES * Op::NIN * CB_UNITS * 16 + 2 * CB_STAGES * 8 + sizeof(double) * Op::NACC * C;
      int err = 0;
      const int grid = cb_grid(chan_reduce_bulk_kernel<Op>, nchunks, bsmem, &err);
      if (err) return ttg_set_error(TTG_ERR_CUDA, "%s: shared memory attribute", name);
      chan_reduce_bulk_kernel<Op><<<grid, CB_THREADS, bsmem, st>>>(op, nvec, C, out);
      TTG_CHECK_LAUNCH(name);
      return TTG_OK;
    }
  }
  size_t smem = sizeof(double) * Op::NACC * C;
  constexpr int VV = ChanV<T, Op>::value;
  if (ttg_vec_ok<T>(C, ptrs, Op::NIN, VV) && C / VV <= 256) {
    constexpr int V = VV;
    int rpi = 256 / (C / V);
    int grid = ttg_grid_occ(chan_reduce_kernel<T, V, Op>, M, rpi * 4, 256, smem);
    chan_reduce_kernel<T, V, Op><<<grid, 256, smem, st>>>(op, M, C, out);
  } else {
    if (C > 256) return ttg_set_error(TTG_ERR_UNSUPPORTED, "%s: C=%d needs C%%%d==0 and 16B alignment", name, C, Vec<T>::N);
    int rpi = 256 / C;
    int grid = ttg_grid_occ(chan_reduce_kernel<T, 1, Op>, M, rpi * 8, 256, smem);
    chan_reduce_kernel<T, 1, Op><<<grid, 256, smem, st>>>(op, M, C, out);
  }
  TTG_CHECK_LAUNCH(name);
  return TTG_OK;
}

// Op concept for maps:
//   static constexpr int NIN, NOUT;  const T* in[NIN];  T* out[NOUT];
//   template <int V> struct P;  load<V>(c0, P&);  apply<V>(const float* v, int j, const P<V>&, float* o)
// When the grid stride keeps every thread on the same channel group (`invariant`), the per-channel
// parameters are loaded once per thread instead of once per element.
// `reverse`: walk the tensor from its end.  A map pass that follows a reduction over the same tensors then starts
// with the part of them the reduction touched last, i.e. the part that is still resident in the 126 MB L2.
template <typename T, int V, class Op>
__global__ void __launch_bounds__(256) chan_map_kernel(Op op, long long nvec, int C, int invariant, int reverse) {
  constexpr int U = 2;                             // vectors in flight per thread
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  typename Op::template P<V> prm;
  const long long last = nvec - 1;
  if constexpr (chan_has_finalize<Op>::value) { if (blockIdx.x == 0) op.finalize(C); }
  if (invariant && i0 < nvec) op.template load<V>((int)(((reverse ? last - i0 : i0) * V) % C), prm);
  for (; i0 < nvec; i0 += U * stride) {
    float v[U][Op::NIN][V];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long ii = i0 + u * stride;
      const long long i = reverse ? last - ii : ii;
      if (ii < nvec) {
#pragma unroll
        for (int t = 0; t < Op::NIN; ++t) {
          if constexpr (V == 1) v[u][t][0] = to_f(op.in[t][i]);
          else { VecN<T, V> q; q.load(op.in[t] + i * V); q.unpack(v[u][t]); }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long ii = i0 + u * stride;
      const long long i = reverse ? last - ii : ii;
      if (ii < nvec) {
        const long long base = i * V;
        if (!invariant) op.template load<V>((int)(base % C), prm);
        float o[Op::NOUT][V];
#pragma unroll
        for (int j = 0; j < V; ++j) {
          float vin[Op::NIN], vout[Op::NOUT];
#pragma unroll
          for (int t = 0; t < Op::NIN; ++t) vin[t] = v[u][t][j];
          op.template apply<V>(vin, j, prm, vout);
#pragma unroll
          for (int t = 0; t < Op::NOUT; ++t) o[t][j] = vout[t];
        }
#pragma unroll
        for (int t = 0; t < Op::NOUT; ++t) {
          if constexpr (V == 1) op.out[t][base] = from_f<T>(o[t][0]);
          else { VecN<T, V> q; q.pack(o[t]); q.store(op.out[t] + base); }
        }
      }
    }
  }
}

template <typename T, class Op>
static int launch_chan_map(const char* name, Op op, long long n, int C, cudaStream_t st, int reverse = 0) {
  const void* ptrs[Op::NIN + Op::NOUT];
  for (int i = 0; i < Op::NIN; ++i) ptrs[i] = op.in[i];
  for (int i = 0; i < Op::NOUT; ++i) ptrs[Op::NIN + i] = op.out[i];
  if (n == 0) return TTG_OK;
  if (!reverse && c3_ok<T>(C, ptrs, Op::NIN + Op::NOUT, n)) {
    const long long ngroups = n / (3 * Vec<T>::N);
    chan_map_c3_kernel<T, Op><<<ttg_grid_occ(chan_map_c3_kernel<T, Op>, ngroups, 256 * 2), 256, 0, st>>>(op, ngroups);
    TTG_CHECK_LAUNCH(name);
    return TTG_OK;
  }
  if constexpr (std::is_same<T, bf16>::value) {
    if (!reverse && cb_ok<T, Op>(C, ptrs, Op::NIN + Op::NOUT, n)) {
      const long long nvec = n / 8, nchunks = (nvec + CB_UNITS - 1) / CB_UNITS;
      const size_t bsmem = (size_t)CB_STAGES * Op::NIN * CB_UNITS * 16 + 2 * CB_STAGES * 8;
      int err = 0;
      const int grid = cb_grid(chan_map_bulk_kernel<Op>, nchunks, bsmem, &err);
      if (err) return ttg_set_error(TTG_ERR_CUDA, "%s: shared memory attribute", name);
      chan_map_bulk_kernel<Op><<<grid, CB_THREADS, bsmem, st>>>(op, nvec, C);
      TTG_CHECK_LAUNCH(name);
      return TTG_OK;
    }
  }
  if (ttg_vec_ok<T>(C, ptrs, Op::NIN + Op::NOUT, ChanV<T, Op>::value)) {
    constexpr int V = ChanV<T, Op>::value;
    long long nvec = n / V;
    int grid = ttg_grid_occ(chan_map_kernel<T, V, Op>, nvec, 256 * 2);
    int inv = ((long long)grid * 256 * V) % C == 0;
    chan_map_kernel<T, V, Op><<<grid, 256, 0, st>>>(op, nvec, C, inv, reverse);
  } else {
    int grid = ttg_grid_occ(chan_map_kernel<T, 1, Op>, n, 256 * 4);
    int inv = ((long long)grid * 256) % C == 0;
    chan_map_kernel<T, 1, Op><<<grid, 256, 0, st>>>(op, n, C, inv, reverse);
  }
  TTG_CHECK_LAUNCH(name);
  return TTG_OK;
}
