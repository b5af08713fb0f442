// HBM-bound passes between the convolutions: BatchNorm (train/eval) fused with the
// nonlinearity, the GateLayer2d product, bilinear x2 upsampling, pad/crop windows,
// Dropout2d mask generation.  NHWC activations (fp32 or bf16), fp32 math.
// Replaces the ATen elementwise / cuDNN BatchNorm kernels launched by lib/nn.py:50-99,121-126,
// boilr Interpolate (models/lvae.py:144) and boilr pad/crop (models/lvae.py:176,185).
#include "common.cuh"

// V-wide (4 or 8 element) typed vector IO: 16-byte transactions for bf16 when V = 8
template <typename T, int V> __device__ __forceinline__ void ldv(const T* p, float* f);
template <> __device__ __forceinline__ void ldv<float, 4>(const float* p, float* f) {
  float4 v = *reinterpret_cast<const float4*>(p);
  f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
}
template <> __device__ __forceinline__ void ldv<__nv_bfloat16, 4>(const __nv_bfloat16* p, float* f) {
  float4 v = ld4<__nv_bfloat16>(p);
  f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
}
template <> __device__ __forceinline__ void ldv<__nv_bfloat16, 8>(const __nv_bfloat16* p, float* f) {
  uint4 u = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float2 t = __bfloat1622float2(h[j]);
    f[2 * j] = t.x; f[2 * j + 1] = t.y;
  }
}
template <typename T, int V> __device__ __forceinline__ void stv(T* p, const float* f);
template <> __device__ __forceinline__ void stv<float, 4>(float* p, const float* f) {
  *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
}
template <> __device__ __forceinline__ void stv<__nv_bfloat16, 4>(__nv_bfloat16* p, const float* f) {
  st4<__nv_bfloat16>(p, make_float4(f[0], f[1], f[2], f[3]));
}
template <> __device__ __forceinline__ void stv<__nv_bfloat16, 8>(__nv_bfloat16* p, const float* f) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
  *reinterpret_cast<uint4*>(p) = u;
}

// Raw (unconverted) vector loads: a kernel issues them BEFORE its prologue (statistics tables, barriers) and converts
// after it, so the first global round trip overlaps the prologue; inside the loop the next iteration's loads are in
// flight while the current one computes.
template <typename T, int V> struct RawV;
template <> struct RawV<float, 4> { float4 v; };
template <> struct RawV<__nv_bfloat16, 4> { uint2 v; };
template <> struct RawV<__nv_bfloat16, 8> { uint4 v; };
template <typename T, int V> __device__ __forceinline__ RawV<T, V> ldraw(const T* p) {
  RawV<T, V> r;
  r.v = *reinterpret_cast<const decltype(r.v)*>(p);
  return r;
}
__device__ __forceinline__ void unraw(const RawV<float, 4>& r, float* f) { f[0] = r.v.x; f[1] = r.v.y; f[2] = r.v.z; f[3] = r.v.w; }
__device__ __forceinline__ void unraw(const RawV<__nv_bfloat16, 4>& r, float* f) {
  f[0] = __uint_as_float(r.v.x << 16); f[1] = __uint_as_float(r.v.x & 0xFFFF0000u);
  f[2] = __uint_as_float(r.v.y << 16); f[3] = __uint_as_float(r.v.y & 0xFFFF0000u);
}
__device__ __forceinline__ void unraw(const RawV<__nv_bfloat16, 8>& r, float* f) {
  const uint32_t w[4] = {r.v.x, r.v.y, r.v.z, r.v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) { f[2 * j] = __uint_as_float(w[j] << 16); f[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u); }
}
template <typename T> __device__ __forceinline__ float round_to(float v);
template <> __device__ __forceinline__ float round_to<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_to<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16(v)); }

// Per-channel accumulators are striped BN_STRIPES ways ([stripe][2][C] doubles): producers add into stripe
// (blockIdx.x % BN_STRIPES), consumers sum the stripes.
constexpr int BN_STRIPES = 8;
__device__ __forceinline__ double acc_sum(const double* acc, int idx, int C) {
  // pairwise tree: three dependent FP64 additions instead of eight (each costs ~40 cycles of latency on this part, and the
  // sum sits on the critical path of every BatchNorm-apply launch)
  double v[BN_STRIPES];
#pragma unroll
  for (int k = 0; k < BN_STRIPES; ++k) v[k] = acc[k * 2 * C + idx];
  return ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
}
__device__ __forceinline__ void acc_clear(double* acc, int idx, int C) {
#pragma unroll
  for (int k = 0; k < BN_STRIPES; ++k) acc[k * 2 * C + idx] = 0.0;
}

// =========================================================================================
// BatchNorm2d statistics: per-channel sum / sum of squares over (B,H,W), accumulated in
// double (fp32 partials per thread, double atomics per block).
// =========================================================================================
template <typename T, int V>
__global__ void bn_stats_kernel(const T* __restrict__ x, double* __restrict__ acc, long long P, int C) {
  pdl_wait();
  pdl_launch();
  // thread -> channel group (threadIdx.x % CV), row lane (threadIdx.x / CV)
  extern __shared__ float sm[];  // [2][blockDim.x*V]
  const int CV = C / V;
  const int cq = threadIdx.x % CV, rl = threadIdx.x / CV, rpb = blockDim.x / CV;
  float s[V], ss[V];
#pragma unroll
  for (int j = 0; j < V; ++j) s[j] = ss[j] = 0.f;
  for (long long r = (long long)blockIdx.x * rpb + rl; r < P; r += (long long)gridDim.x * rpb) {
    float v[V];
    ldv<T, V>(x + r * C + cq * V, v);
#pragma unroll
    for (int j = 0; j < V; ++j) { s[j] += v[j]; ss[j] += v[j] * v[j]; }
  }
  float* s_s = sm;
  float* s_ss = sm + blockDim.x * V;
#pragma unroll
  for (int j = 0; j < V; ++j) { s_s[threadIdx.x * V + j] = s[j]; s_ss[threadIdx.x * V + j] = ss[j]; }
  __syncthreads();
  // threads 0..C-1 reduce over row lanes
  if (threadIdx.x < C) {
    int c = threadIdx.x, q = c / V, e = c % V;
    double a = 0.0, b = 0.0;
    for (int r = 0; r < rpb; ++r) {
      a += (double)s_s[(r * CV + q) * V + e];
      b += (double)s_ss[(r * CV + q) * V + e];
    }
    double* accs = acc + (blockIdx.x & (BN_STRIPES - 1)) * 2 * C;   // striped accumulators: 8x less atomic contention
    atomicAdd(accs + c, a);
    atomicAdd(accs + C + c, b);
  }
}

// finalize: mean / rstd for this batch, update running stats (momentum), clear the accumulators.
__global__ void bn_finalize_kernel(double* acc, float* save_mean, float* save_rstd, float* running_mean,
                                   float* running_var, long long* num_batches_tracked, long long P, int C,
                                   float momentum, float eps) {
  pdl_wait();
  pdl_launch();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    double mean = acc_sum(acc, c, C) / (double)P;
    double var = acc_sum(acc, C + c, C) / (double)P - mean * mean;
    if (var < 0.0) var = 0.0;
    save_mean[c] = (float)mean;
    save_rstd[c] = (float)(1.0 / sqrt(var + (double)eps));
    if (running_mean) {
      double unb = P > 1 ? var * (double)P / (double)(P - 1) : var;
      running_mean[c] = (float)((1.0 - momentum) * (double)running_mean[c] + momentum * mean);
      running_var[c] = (float)((1.0 - momentum) * (double)running_var[c] + momentum * unb);
    }
    acc_clear(acc, c, C);
    acc_clear(acc, C + c, C);
  }
  if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;
}

// eval-mode: mean/rstd from running stats
__global__ void bn_eval_prepare_kernel(const float* running_mean, const float* running_var, float* save_mean,
                                       float* save_rstd, int C, float eps) {
  pdl_wait();
  pdl_launch();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    save_mean[c] = running_mean[c];
    save_rstd[c] = 1.0f / sqrtf(running_var[c] + eps);
  }
}

// y = act(((x - mean) * rstd) * gamma + beta); with mean == null this is a plain activation pass
template <typename TI, typename TO>
__global__ void bn_act_fwd_kernel(const TI* __restrict__ x, TO* __restrict__ y, const float* __restrict__ mean,
                                  const float* __restrict__ rstd, const float* __restrict__ gamma,
                                  const float* __restrict__ beta, long long nquads, int C, int act) {
  pdl_wait();
  pdl_launch();
  const int CV = C >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nquads; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % CV) * 4;
    float4 v = ld4<TI>(x + i * 4);
    float o[4] = {v.x, v.y, v.z, v.w};
    if (mean) {
      float4 m = *reinterpret_cast<const float4*>(mean + c), r = *reinterpret_cast<const float4*>(rstd + c);
      float4 g = *reinterpret_cast<const float4*>(gamma + c), b = *reinterpret_cast<const float4*>(beta + c);
      o[0] = (o[0] - m.x) * r.x * g.x + b.x;
      o[1] = (o[1] - m.y) * r.y * g.y + b.y;
      o[2] = (o[2] - m.z) * r.z * g.z + b.z;
      o[3] = (o[3] - m.w) * r.w * g.w + b.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = act_fwd_t<sizeof(TO) == 2>(o[j], act);
    st4<TO>(y + i * 4, make_float4(o[0], o[1], o[2], o[3]));
  }
}

// backward pass 1: g = dy * act'(pre); accumulate sum(g), sum(g*xhat) per channel (double)
template <typename T, int V>
__global__ void bn_act_bwd_reduce_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                         double* __restrict__ acc, long long P, int C, int act) {
  pdl_wait();
  pdl_launch();
  extern __shared__ float sm[];
  const int CV = C / V;
  const int cq = threadIdx.x % CV, rl = threadIdx.x / CV, rpb = blockDim.x / CV;
  const int c = cq * V;
  float mm[V], rr[V], gg[V], bb[V], s1[V], s2[V];
#pragma unroll
  for (int j = 0; j < V; ++j) {
    mm[j] = mean[c + j]; rr[j] = rstd[c + j]; gg[j] = gamma[c + j]; bb[j] = beta[c + j];
    s1[j] = s2[j] = 0.f;
  }
  for (long long row = (long long)blockIdx.x * rpb + rl; row < P; row += (long long)gridDim.x * rpb) {
    float xs[V], ds[V];
    ldv<T, V>(x + row * C + c, xs);
    ldv<T, V>(dy + row * C + c, ds);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float xh = (xs[j] - mm[j]) * rr[j];
      float gpre = ds[j] * act_bwd_t<sizeof(T) == 2>(xh * gg[j] + bb[j], act);
      s1[j] += gpre;
      s2[j] += gpre * xh;
    }
  }
  float* a1 = sm;
  float* a2 = sm + blockDim.x * V;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    a1[threadIdx.x * V + j] = s1[j];
    a2[threadIdx.x * V + j] = s2[j];
  }
  __syncthreads();
  if (threadIdx.x < C) {
    int cc = threadIdx.x, q = cc / V, e = cc % V;
    double u = 0.0, v = 0.0;
    for (int rrw = 0; rrw < rpb; ++rrw) {
      u += (double)a1[(rrw * CV + q) * V + e];
      v += (double)a2[(rrw * CV + q) * V + e];
    }
    double* accs = acc + (blockIdx.x & (BN_STRIPES - 1)) * 2 * C;
    atomicAdd(accs + cc, u);
    atomicAdd(accs + C + cc, v);
  }
}

// backward pass 2: dx = gamma*rstd*(g - sum_g/P - xhat*sum_gx/P) (train) or gamma*rstd*g (eval);
// block 0 also emits dgamma (+=) / dbeta (+=) and clears the accumulators via a second tiny kernel.
template <typename T>
__global__ void bn_act_bwd_apply_kernel(const T* __restrict__ dy, const T* __restrict__ x, T* __restrict__ dx,
                                        const float* __restrict__ mean, const float* __restrict__ rstd,
                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                        const double* __restrict__ acc, long long nquads, long long P, int C,
                                        int act, int training) {
  pdl_wait();
  pdl_launch();
  const int CV = C >> 2;
  const double invP = 1.0 / (double)P;
  // The per-channel constants (16 striped double loads + 6 dependent FP64 additions per channel) are re-derived only when the
  // thread's channel quad changes: with a grid stride that is a multiple of C / 4 (every C / 4 that divides 256) that is once
  // per thread, not once per element (68 -> ~10 us for the stem block's (256,16,16,64) tensor).
  int c_cur = -1;
  float mj[4], rj[4], gj[4], bj[4], m1[4], m2[4];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nquads; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % CV) * 4;
    float4 xv = ld4<T>(x + i * 4), dv = ld4<T>(dy + i * 4);
    if (c != c_cur) {
      c_cur = c;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        mj[j] = mean[c + j]; rj[j] = rstd[c + j]; gj[j] = gamma[c + j]; bj[j] = beta[c + j];
        m1[j] = m2[j] = 0.f;
        if (training) {
          m1[j] = (float)(acc_sum(acc, c + j, C) * invP);
          m2[j] = (float)(acc_sum(acc, C + c + j, C) * invP);
        }
      }
    }
    float xs[4] = {xv.x, xv.y, xv.z, xv.w}, ds[4] = {dv.x, dv.y, dv.z, dv.w}, o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float xh = (xs[j] - mj[j]) * rj[j];
      float gpre = ds[j] * act_bwd_t<sizeof(T) == 2>(xh * gj[j] + bj[j], act);
      if (training) o[j] = gj[j] * rj[j] * (gpre - m1[j] - xh * m2[j]);
      else o[j] = gj[j] * rj[j] * gpre;
    }
    st4<T>(dx + i * 4, make_float4(o[0], o[1], o[2], o[3]));
  }
}

__global__ void bn_bwd_params_kernel(double* acc, float* dgamma, float* dbeta, int C) {
  pdl_wait();
  pdl_launch();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    if (dbeta) dbeta[c] += (float)acc_sum(acc, c, C);
    if (dgamma) dgamma[c] += (float)acc_sum(acc, C + c, C);
    acc_clear(acc, c, C);
    acc_clear(acc, C + c, C);
  }
}

// plain activation backward (no BatchNorm): dx = dy * act'(x)
template <typename T>
__global__ void act_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ x, T* __restrict__ dx, long long nquads, int act) {
  pdl_wait();
  pdl_launch();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nquads; i += (long long)gridDim.x * blockDim.x) {
    float4 xv = ld4<T>(x + i * 4), dv = ld4<T>(dy + i * 4);
    constexpr bool F = sizeof(T) == 2;
    st4<T>(dx + i * 4, make_float4(dv.x * act_bwd_t<F>(xv.x, act), dv.y * act_bwd_t<F>(xv.y, act), dv.z * act_bwd_t<F>(xv.z, act),
                                   dv.w * act_bwd_t<F>(xv.w, act)));
  }
}

static inline int ew_grid(long long n, int threads) {
  long long g = (n + threads - 1) / threads;
  long long cap = 8LL * lvae_num_sms();
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

static bool bn_c_ok(int C) { return C >= 4 && C % 4 == 0 && C <= 256; }
static int bn_threads(int C) { return (256 / (C / 4)) * (C / 4); }
// 8-wide bf16 path: 16-byte transactions; needs C % 8 == 0 and 256 % (C/8) == 0 (C = 64: 8 threads per pixel)
static bool use_v8(int dtype, int C) { return dtype == 1 && C % 8 == 0 && C >= 8 && 256 % (C / 8) == 0 && C <= 256; }

static int launch_bn_stats(const void* x, double* acc, long long P, int C, int dtype, cudaStream_t stream) {
  if (use_v8(dtype, C)) {
    int threads = 256, rpb = threads / (C / 8);
    int grid = (int)min((long long)4 * lvae_num_sms(), (P + rpb - 1) / rpb);
    lvae_launch(bn_stats_kernel<__nv_bfloat16, 8>, grid, threads, (size_t)threads * 8 * 2 * sizeof(float), stream, (const __nv_bfloat16*)x, acc, P, C);
    return 0;
  }
  int threads = bn_threads(C), rpb = threads / (C / 4);
  int grid = (int)min((long long)4 * lvae_num_sms(), (P + rpb - 1) / rpb);
  size_t smem = (size_t)threads * 4 * 2 * sizeof(float);
  if (dtype == 0) lvae_launch(bn_stats_kernel<float, 4>, grid, threads, smem, stream, (const float*)x, acc, P, C);
  else lvae_launch(bn_stats_kernel<__nv_bfloat16, 4>, grid, threads, smem, stream, (const __nv_bfloat16*)x, acc, P, C);
  return 0;
}

static int launch_bwd_reduce(const void* dy, const void* x, const float* mean, const float* rstd, const float* gamma,
                             const float* beta, double* acc, long long P, int C, int act, int dtype, cudaStream_t stream) {
  if (use_v8(dtype, C)) {
    int threads = 256, rpb = threads / (C / 8);
    int grid = (int)min((long long)4 * lvae_num_sms(), (P + rpb - 1) / rpb);
    lvae_launch(bn_act_bwd_reduce_kernel<__nv_bfloat16, 8>, grid, threads, (size_t)threads * 8 * 2 * sizeof(float), stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, mean, rstd, gamma, beta, acc, P, C, act);
    return 0;
  }
  int threads = bn_threads(C), rpb = threads / (C / 4);
  int grid = (int)min((long long)4 * lvae_num_sms(), (P + rpb - 1) / rpb);
  size_t smem = (size_t)threads * 4 * 2 * sizeof(float);
  if (dtype == 0)
    lvae_launch(bn_act_bwd_reduce_kernel<float, 4>, grid, threads, smem, stream, (const float*)dy, (const float*)x, mean, rstd, gamma, beta, acc, P, C, act);
  else
    lvae_launch(bn_act_bwd_reduce_kernel<__nv_bfloat16, 4>, grid, threads, smem, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, mean, rstd, gamma, beta, acc, P, C, act);
  return 0;
}

LVAE_API int lvae_bn_stats(const void* x, double* acc, long long P, int C, int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(x && acc && P > 0, "bn_stats: bad args");
  LVAE_REQUIRE(bn_c_ok(C), "bn_stats: channels must be a multiple of 4 and <= 256 (got %d)", C);
  launch_bn_stats(x, acc, P, C, dtype, stream);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_stats");
  return LVAE_OK;
}

LVAE_API int lvae_bn_finalize(double* acc, float* save_mean, float* save_rstd, float* running_mean,
                              float* running_var, long long* num_batches_tracked, long long P, int C,
                              float momentum, float eps, cudaStream_t stream) {
  LVAE_REQUIRE(acc && save_mean && save_rstd, "bn_finalize: bad args");
  lvae_launch(bn_finalize_kernel, cdiv(C, 128), 128, 0, stream, acc, save_mean, save_rstd, running_mean, running_var,
                                                       num_batches_tracked, P, C, momentum, eps);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_finalize");
  return LVAE_OK;
}

LVAE_API int lvae_bn_eval_prepare(const float* running_mean, const float* running_var, float* save_mean,
                                  float* save_rstd, int C, float eps, cudaStream_t stream) {
  LVAE_REQUIRE(running_mean && running_var && save_mean && save_rstd, "bn_eval_prepare: bad args");
  lvae_launch(bn_eval_prepare_kernel, cdiv(C, 128), 128, 0, stream, running_mean, running_var, save_mean, save_rstd, C, eps);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_eval_prepare");
  return LVAE_OK;
}

// dtype_in / dtype_out: 0 f32, 1 bf16 (the bf16 conv path stores bf16 activations)
LVAE_API int lvae_bn_act_fwd(const void* x, void* y, const float* mean, const float* rstd, const float* gamma,
                             const float* beta, long long P, int C, int act, int dtype_in, int dtype_out,
                             cudaStream_t stream) {
  LVAE_REQUIRE(x && y && P > 0 && C % 4 == 0, "bn_act_fwd: bad args (C must be a multiple of 4)");
  long long nq = P * (C / 4);
  int g = ew_grid(nq, 256);
  if (dtype_in == 0 && dtype_out == 0)
    lvae_launch(bn_act_fwd_kernel<float, float>, g, 256, 0, stream, (const float*)x, (float*)y, mean, rstd, gamma, beta, nq, C, act);
  else if (dtype_in == 0 && dtype_out == 1)
    lvae_launch(bn_act_fwd_kernel<float, __nv_bfloat16>, g, 256, 0, stream, (const float*)x, (__nv_bfloat16*)y, mean, rstd, gamma, beta, nq, C, act);
  else if (dtype_in == 1 && dtype_out == 1)
    lvae_launch(bn_act_fwd_kernel<__nv_bfloat16, __nv_bfloat16>, g, 256, 0, stream, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, mean, rstd, gamma, beta, nq, C, act);
  else
    lvae_launch(bn_act_fwd_kernel<__nv_bfloat16, float>, g, 256, 0, stream, (const __nv_bfloat16*)x, (float*)y, mean, rstd, gamma, beta, nq, C, act);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_act_fwd");
  return LVAE_OK;
}

LVAE_API int lvae_bn_act_bwd(const void* dy, const void* x, void* dx, const float* mean, const float* rstd,
                             const float* gamma, const float* beta, double* acc, float* dgamma, float* dbeta,
                             long long P, int C, int act, int training, int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(dy && x && dx && P > 0, "bn_act_bwd: bad args");
  long long nq = P * (C / 4);
  if (!mean) {  // plain activation
    LVAE_REQUIRE(C % 4 == 0, "act_bwd: C must be a multiple of 4");
    int g = ew_grid(nq, 256);
    if (dtype == 0) lvae_launch(act_bwd_kernel<float>, g, 256, 0, stream, (const float*)dy, (const float*)x, (float*)dx, nq, act);
    else lvae_launch(act_bwd_kernel<__nv_bfloat16>, g, 256, 0, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (__nv_bfloat16*)dx, nq, act);
    LVAE_COUNT_LAUNCH();
    LVAE_CHECK_LAUNCH("act_bwd");
    return LVAE_OK;
  }
  LVAE_REQUIRE(bn_c_ok(C) && acc, "bn_act_bwd: channels must be a multiple of 4, <= 256, and acc non-null");
  launch_bwd_reduce(dy, x, mean, rstd, gamma, beta, acc, P, C, act, dtype, stream);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_act_bwd_reduce");
  int g = ew_grid(nq, 256);
  if (dtype == 0)
    lvae_launch(bn_act_bwd_apply_kernel<float>, g, 256, 0, stream, (const float*)dy, (const float*)x, (float*)dx, mean, rstd, gamma, beta, acc, nq, P, C, act, training);
  else
    lvae_launch(bn_act_bwd_apply_kernel<__nv_bfloat16>, g, 256, 0, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (__nv_bfloat16*)dx, mean, rstd, gamma, beta, acc, nq, P, C, act, training);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_act_bwd_apply");
  lvae_launch(bn_bwd_params_kernel, cdiv(C, 128), 128, 0, stream, acc, dgamma, dbeta, C);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_bwd_params");
  return LVAE_OK;
}

// =========================================================================================
// GateLayer2d (lib/nn.py:121-126) + residual (lib/nn.py:99): h is (P, 2C); out = act(h[:, :C]) * sigmoid(h[:, C:]) + res
// =========================================================================================
template <typename T>
__global__ void gate_fwd_kernel(const T* __restrict__ h, const T* __restrict__ res, T* __restrict__ out,
                                long long nquads, int C, int act) {
  pdl_wait();
  pdl_launch();
  const int CV = C >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nquads; i += (long long)gridDim.x * blockDim.x) {
    long long row = i / CV;
    int c = (int)(i - row * CV) * 4;
    float4 a = ld4<T>(h + row * 2 * C + c), g = ld4<T>(h + row * 2 * C + C + c);
    constexpr bool F = sizeof(T) == 2;
    float4 o = make_float4(act_fwd_t<F>(a.x, act) * sigmoid_t<F>(g.x), act_fwd_t<F>(a.y, act) * sigmoid_t<F>(g.y),
                           act_fwd_t<F>(a.z, act) * sigmoid_t<F>(g.z), act_fwd_t<F>(a.w, act) * sigmoid_t<F>(g.w));
    if (res) {
      float4 r = ld4<T>(res + i * 4);
      o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    }
    st4<T>(out + i * 4, o);
  }
}

// ACT >= 0: activation known at compile time (the launchers pick ACT_ELU, the model default); -1: runtime switch, which the
// compiler turns into one jump table per element inside the unrolled loops
template <typename T, int V, int ACT = -1>
__global__ void gate_bwd_kernel(const T* __restrict__ dout, const T* __restrict__ h, T* __restrict__ dh,
                                long long nvec, int C, int act_rt) {
  pdl_wait();
  pdl_launch();
  const int act = ACT >= 0 ? ACT : act_rt;
  const unsigned CV = (unsigned)(C / V);
  // 32-bit index arithmetic (lvae_gate_bwd checks that the element count fits): a 64-bit i / CV per iteration is ~100 instructions
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < (unsigned)nvec; i += gridDim.x * blockDim.x) {
    const unsigned row = i / CV;
    const int c = (int)(i - row * CV) * V;
    float av[V], gv[V], dv[V], da[V], dg[V];
    ldv<T, V>(h + (size_t)row * 2 * C + c, av);
    ldv<T, V>(h + (size_t)row * 2 * C + C + c, gv);
    ldv<T, V>(dout + (size_t)i * V, dv);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float s = sigmoid_t<sizeof(T) == 2>(gv[j]);
      da[j] = dv[j] * s * act_bwd_t<sizeof(T) == 2>(av[j], act);
      dg[j] = dv[j] * act_fwd_t<sizeof(T) == 2>(av[j], act) * s * (1.f - s);
    }
    stv<T, V>(dh + (size_t)row * 2 * C + c, da);
    stv<T, V>(dh + (size_t)row * 2 * C + C + c, dg);
  }
}

LVAE_API int lvae_gate_fwd(const void* h, const void* res, void* out, long long P, int C, int act, int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(h && out && P > 0 && C % 4 == 0, "gate_fwd: bad args");
  long long nq = P * (C / 4);
  int g = ew_grid(nq, 256);
  if (dtype == 0) lvae_launch(gate_fwd_kernel<float>, g, 256, 0, stream, (const float*)h, (const float*)res, (float*)out, nq, C, act);
  else lvae_launch(gate_fwd_kernel<__nv_bfloat16>, g, 256, 0, stream, (const __nv_bfloat16*)h, (const __nv_bfloat16*)res, (__nv_bfloat16*)out, nq, C, act);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("gate_fwd");
  return LVAE_OK;
}

LVAE_API int lvae_gate_bwd(const void* dout, const void* h, void* dh, long long P, int C, int act, int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(dout && h && dh && P > 0 && C % 4 == 0, "gate_bwd: bad args");
  LVAE_REQUIRE(P * (long long)C < (1LL << 32), "gate_bwd: more than 2^32 elements");
  if (dtype == 1 && C % 8 == 0) {
    long long nv = P * (C / 8);
    if (act == ACT_ELU) lvae_launch(gate_bwd_kernel<__nv_bfloat16, 8, ACT_ELU>, ew_grid(nv, 256), 256, 0, stream, (const __nv_bfloat16*)dout, (const __nv_bfloat16*)h, (__nv_bfloat16*)dh, nv, C, act);
    else lvae_launch(gate_bwd_kernel<__nv_bfloat16, 8>, ew_grid(nv, 256), 256, 0, stream, (const __nv_bfloat16*)dout, (const __nv_bfloat16*)h, (__nv_bfloat16*)dh, nv, C, act);
  } else {
    long long nq = P * (C / 4);
    int g = ew_grid(nq, 256);
    if (dtype == 0) lvae_launch(gate_bwd_kernel<float, 4>, g, 256, 0, stream, (const float*)dout, (const float*)h, (float*)dh, nq, C, act);
    else lvae_launch(gate_bwd_kernel<__nv_bfloat16, 4>, g, 256, 0, stream, (const __nv_bfloat16*)dout, (const __nv_bfloat16*)h, (__nv_bfloat16*)dh, nq, C, act);
  }
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("gate_bwd");
  return LVAE_OK;
}

// =========================================================================================
// Bilinear x2 upsampling, align_corners=False (boilr Interpolate(scale=2), models/lvae.py:144)
// =========================================================================================
__device__ __forceinline__ void up2_src(int o, int n_in, int& i0, int& i1, float& l) {
  float s = (o + 0.5f) * 0.5f - 0.5f;
  if (s < 0.f) s = 0.f;
  i0 = (int)s;
  i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
  l = s - (float)i0;
}

template <typename T>
__global__ void upsample2x_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int B, int H, int W, int C) {
  pdl_wait();
  pdl_launch();
  const int CV = C >> 2;
  long long total = (long long)B * 2 * H * 2 * W * CV;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % CV) * 4;
    long long p = i / CV;
    int ox = (int)(p % (2 * W));
    long long q = p / (2 * W);
    int oy = (int)(q % (2 * H));
    int b = (int)(q / (2 * H));
    int y0, y1, x0, x1;
    float ly, lx;
    up2_src(oy, H, y0, y1, ly);
    up2_src(ox, W, x0, x1, lx);
    const T* base = x + (long long)b * H * W * C + c;
    float4 v00 = ld4<T>(base + ((long long)y0 * W + x0) * C), v01 = ld4<T>(base + ((long long)y0 * W + x1) * C);
    float4 v10 = ld4<T>(base + ((long long)y1 * W + x0) * C), v11 = ld4<T>(base + ((long long)y1 * W + x1) * C);
    float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    float4 o = make_float4(w00 * v00.x + w01 * v01.x + w10 * v10.x + w11 * v11.x,
                           w00 * v00.y + w01 * v01.y + w10 * v10.y + w11 * v11.y,
                           w00 * v00.z + w01 * v01.z + w10 * v10.z + w11 * v11.z,
                           w00 * v00.w + w01 * v01.w + w10 * v10.w + w11 * v11.w);
    st4<T>(y + i * 4, o);
  }
}

// x / d and x % d for a divisor that is a power of two in every model configuration (channel vectors per pixel, image sides):
// sh >= 0 selects the shift / mask form; three runtime divisions per 16-byte output made the kernels below instruction-bound
// (59 us for the (1000,16,16,64) -> (1000,32,32,64) tensor of the IW evaluator, 2.8 TB/s).
__device__ __forceinline__ void divmod_u(unsigned x, unsigned d, int sh, unsigned& q, unsigned& r) {
  if (sh >= 0) { q = x >> sh; r = x & (d - 1u); }
  else { q = x / d; r = x - q * d; }
}
static inline int pow2_shift(unsigned d) {
  if (d == 0 || (d & (d - 1u))) return -1;
  int s = 0;
  while ((1u << s) < d) ++s;
  return s;
}

// bf16, C % 8 == 0: 16-byte transactions and 32-bit index arithmetic (the 4-channel kernel above spends most of its time in
// 64-bit divisions: 135 us for the (1000,16,16,64) -> (1000,32,32,64) tensor of the IW evaluator, 1.2 TB/s)
__global__ void upsample2x_fwd_bf16x8_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int H, int W,
                                             int C, int sh_cv, int sh_w, int sh_h) {
  pdl_wait();
  pdl_launch();
  const unsigned CV = (unsigned)C >> 3, W2 = 2u * W, H2 = 2u * H;
  const unsigned total = (unsigned)B * H2 * W2 * CV;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    unsigned cv, p, ox, q, oy, b;
    divmod_u(i, CV, sh_cv, p, cv);
    divmod_u(p, W2, sh_w, q, ox);
    divmod_u(q, H2, sh_h, b, oy);
    int y0, y1, x0, x1;
    float ly, lx;
    up2_src((int)oy, H, y0, y1, ly);
    up2_src((int)ox, W, x0, x1, lx);
    const __nv_bfloat16* base = x + ((size_t)b * H * W) * C + cv * 8;
    const uint4 r00 = __ldg(reinterpret_cast<const uint4*>(base + (size_t)(y0 * W + x0) * C));
    const uint4 r01 = __ldg(reinterpret_cast<const uint4*>(base + (size_t)(y0 * W + x1) * C));
    const uint4 r10 = __ldg(reinterpret_cast<const uint4*>(base + (size_t)(y1 * W + x0) * C));
    const uint4 r11 = __ldg(reinterpret_cast<const uint4*>(base + (size_t)(y1 * W + x1) * C));
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    const uint32_t* a = reinterpret_cast<const uint32_t*>(&r00);
    const uint32_t* bq = reinterpret_cast<const uint32_t*>(&r01);
    const uint32_t* c = reinterpret_cast<const uint32_t*>(&r10);
    const uint32_t* d = reinterpret_cast<const uint32_t*>(&r11);
    uint4 o;
    uint32_t* op = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float lo = w00 * __uint_as_float(a[j] << 16) + w01 * __uint_as_float(bq[j] << 16) + w10 * __uint_as_float(c[j] << 16) +
                       w11 * __uint_as_float(d[j] << 16);
      const float hi = w00 * __uint_as_float(a[j] & 0xFFFF0000u) + w01 * __uint_as_float(bq[j] & 0xFFFF0000u) +
                       w10 * __uint_as_float(c[j] & 0xFFFF0000u) + w11 * __uint_as_float(d[j] & 0xFFFF0000u);
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(lo, hi);
      op[j] = *reinterpret_cast<const uint32_t*>(&h2);
    }
    *reinterpret_cast<uint4*>(y + (size_t)i * 8) = o;
  }
}

// backward as a gather: every input pixel collects from the <= 3x3 output pixels that read it
template <typename T>
__global__ void upsample2x_bwd_kernel(const T* __restrict__ dy, T* __restrict__ dx, int B, int H, int W, int C) {
  pdl_wait();
  pdl_launch();
  const int CV = C >> 2;
  long long total = (long long)B * H * W * CV;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % CV) * 4;
    long long p = i / CV;
    int ix = (int)(p % W);
    long long q = p / W;
    int iy = (int)(q % H);
    int b = (int)(q / H);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int oy = max(0, 2 * iy - 2); oy <= min(2 * H - 1, 2 * iy + 2); ++oy) {
      int y0, y1;
      float ly;
      up2_src(oy, H, y0, y1, ly);
      float wy = (y0 == iy ? 1.f - ly : 0.f) + (y1 == iy ? ly : 0.f);
      if (wy == 0.f) continue;
      for (int ox = max(0, 2 * ix - 2); ox <= min(2 * W - 1, 2 * ix + 2); ++ox) {
        int x0, x1;
        float lx;
        up2_src(ox, W, x0, x1, lx);
        float wx = (x0 == ix ? 1.f - lx : 0.f) + (x1 == ix ? lx : 0.f);
        if (wx == 0.f) continue;
        float4 d = ld4<T>(dy + (((long long)b * 2 * H + oy) * 2 * W + ox) * C + c);
        float w = wy * wx;
        acc.x += w * d.x; acc.y += w * d.y; acc.z += w * d.z; acc.w += w * d.w;
      }
    }
    st4<T>(dx + i * 4, acc);
  }
}

// bf16, C % 8 == 0: the closed form of the same gather.  Along one axis input i collects
//   0.25 dy[2i-1] + 0.75 dy[2i] + 0.75 dy[2i+1] + 0.25 dy[2i+2],
// and the clamped borders fold the missing tap's weight onto its neighbour (i = 0: 1.0 dy[0]; i = n-1: 1.0 dy[2n-1]).
// All 16 loads of a thread are unconditional (clamped coordinates) and issued before the first use, the taps are added in
// the order of the generic kernel (so the result is the same to the bit), 16-byte transactions, 32-bit index arithmetic:
// the generic kernel evaluates up2_src for 25 candidate taps per element and takes 64 us for the (256,32,32,64) gradient.
__global__ void __launch_bounds__(256) upsample2x_bwd_bf16x8_kernel(const __nv_bfloat16* __restrict__ dy, __nv_bfloat16* __restrict__ dx,
                                                                    int B, int H, int W, int C, int sh_cv, int sh_w, int sh_h) {
  pdl_wait();
  pdl_launch();
  const unsigned CV = (unsigned)C >> 3, W2 = 2u * W, H2 = 2u * H;
  const unsigned total = (unsigned)B * H * W * CV;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    unsigned cv, p, uix, q, uiy, b;
    divmod_u(i, CV, sh_cv, p, cv);
    divmod_u(p, (unsigned)W, sh_w, q, uix);
    divmod_u(q, (unsigned)H, sh_h, b, uiy);
    const int ix = (int)uix, iy = (int)uiy;
    float wy[4], wx[4];
    int oy[4], ox[4];
    bool vy[4], vx[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int o_y = 2 * iy - 1 + t, o_x = 2 * ix - 1 + t;
      vy[t] = o_y >= 0 && o_y < (int)H2;
      vx[t] = o_x >= 0 && o_x < (int)W2;
      oy[t] = min(max(o_y, 0), (int)H2 - 1);
      ox[t] = min(max(o_x, 0), (int)W2 - 1);
    }
    wy[0] = 0.25f; wy[1] = iy > 0 ? 0.75f : 1.f; wy[2] = iy < H - 1 ? 0.75f : 1.f; wy[3] = 0.25f;
    wx[0] = 0.25f; wx[1] = ix > 0 ? 0.75f : 1.f; wx[2] = ix < W - 1 ? 0.75f : 1.f; wx[3] = 0.25f;
    const __nv_bfloat16* base = dy + ((size_t)b * H2 * W2) * C + cv * 8;
    uint4 r[4][4];
#pragma unroll
    for (int ty = 0; ty < 4; ++ty)
#pragma unroll
      for (int tx = 0; tx < 4; ++tx)
        r[ty][tx] = __ldg(reinterpret_cast<const uint4*>(base + (size_t)((unsigned)oy[ty] * W2 + (unsigned)ox[tx]) * C));
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
    for (int ty = 0; ty < 4; ++ty)
#pragma unroll
      for (int tx = 0; tx < 4; ++tx)
        if (vy[ty] && vx[tx]) {
          const float w = wy[ty] * wx[tx];
          const uint32_t* u = reinterpret_cast<const uint32_t*>(&r[ty][tx]);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc[2 * j] = fmaf(w, __uint_as_float(u[j] << 16), acc[2 * j]);
            acc[2 * j + 1] = fmaf(w, __uint_as_float(u[j] & 0xFFFF0000u), acc[2 * j + 1]);
          }
        }
    uint4 o;
    uint32_t* op = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(acc[2 * j], acc[2 * j + 1]);
      op[j] = *reinterpret_cast<const uint32_t*>(&h2);
    }
    *reinterpret_cast<uint4*>(dx + (size_t)i * 8) = o;
  }
}

LVAE_API int lvae_upsample2x_fwd(const void* x, void* y, int B, int H, int W, int C, int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(x && y && C % 4 == 0, "upsample2x_fwd: bad args");
  long long n = (long long)B * 4 * H * W * (C / 4);
  if (dtype == 0) lvae_launch(upsample2x_fwd_kernel<float>, ew_grid(n, 256), 256, 0, stream, (const float*)x, (float*)y, B, H, W, C);
  else if (C % 8 == 0 && n / 2 < (1LL << 31)) {
    lvae_launch(upsample2x_fwd_bf16x8_kernel, ew_grid(n / 2, 256), 256, 0, stream, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, B, H, W, C,
                pow2_shift((unsigned)C >> 3), pow2_shift(2u * W), pow2_shift(2u * H));
  } else lvae_launch(upsample2x_fwd_kernel<__nv_bfloat16>, ew_grid(n, 256), 256, 0, stream, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, B, H, W, C);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("upsample2x_fwd");
  return LVAE_OK;
}

LVAE_API int lvae_upsample2x_bwd(const void* dy, void* dx, int B, int H, int W, int C, int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(dy && dx && C % 4 == 0, "upsample2x_bwd: bad args");
  long long n = (long long)B * H * W * (C / 4);
  if (dtype == 0) lvae_launch(upsample2x_bwd_kernel<float>, ew_grid(n, 256), 256, 0, stream, (const float*)dy, (float*)dx, B, H, W, C);
  else if (C % 8 == 0 && n * 2 < (1LL << 31))      // n * 2 = output pixels x (C / 8) of the larger tensor, the kernel's widest 32-bit index
    lvae_launch(upsample2x_bwd_bf16x8_kernel, ew_grid(n / 2, 256), 256, 0, stream, (const __nv_bfloat16*)dy, (__nv_bfloat16*)dx, B, H, W, C,
                pow2_shift((unsigned)C >> 3), pow2_shift((unsigned)W), pow2_shift((unsigned)H));
  else lvae_launch(upsample2x_bwd_kernel<__nv_bfloat16>, ew_grid(n, 256), 256, 0, stream, (const __nv_bfloat16*)dy, (__nv_bfloat16*)dx, B, H, W, C);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("upsample2x_bwd");
  return LVAE_OK;
}

// =========================================================================================
// Window copy between layouts: dst[b, y+dy0, x+dx0, c] = src[b, y+sy0, x+sx0, c] for a (h,w) window.
// Used for boilr pad_img_tensor (NCHW image -> zero-padded NHWC) and crop_img_tensor (and their
// backward).  src_nchw / dst_nchw select the physical layout of either side.
// =========================================================================================
template <typename TS, typename TD>
__global__ void copy_window_kernel(const TS* __restrict__ src, TD* __restrict__ dst, int B, int C, int Hs, int Ws,
                                   int Hd, int Wd, int sy0, int sx0, int dy0, int dx0, int h, int w,
                                   int src_nchw, int dst_nchw) {
  pdl_wait();
  pdl_launch();
  long long total = (long long)B * h * w * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long p = i / C;
    int x = (int)(p % w);
    long long q = p / w;
    int y = (int)(q % h);
    int b = (int)(q / h);
    long long si = src_nchw ? (((long long)b * C + c) * Hs + (y + sy0)) * Ws + (x + sx0)
                            : (((long long)b * Hs + (y + sy0)) * Ws + (x + sx0)) * C + c;
    long long di = dst_nchw ? (((long long)b * C + c) * Hd + (y + dy0)) * Wd + (x + dx0)
                            : (((long long)b * Hd + (y + dy0)) * Wd + (x + dx0)) * C + c;
    st1<TD>(dst + di, ld1<TS>(src + si));
  }
}

// both sides NHWC, same element type, rows of C channels a multiple of 16 bytes: 16-byte copies, 32-bit index arithmetic
// (the crop of the IW evaluator's (1000,32,32,64) bf16 tensor to 28x28 took 288 us with one element per thread)
__global__ void copy_window_vec_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, unsigned B, unsigned CV, unsigned Hs,
                                       unsigned Ws, unsigned Hd, unsigned Wd, unsigned sy0, unsigned sx0, unsigned dy0, unsigned dx0,
                                       unsigned h, unsigned w) {
  pdl_wait();
  pdl_launch();
  const unsigned total = B * h * w * CV;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const unsigned cv = i % CV, p = i / CV;
    const unsigned x = p % w, q = p / w;
    const unsigned y = q % h, b = q / h;
    dst[(((size_t)b * Hd + (y + dy0)) * Wd + (x + dx0)) * CV + cv] = __ldg(src + (((size_t)b * Hs + (y + sy0)) * Ws + (x + sx0)) * CV + cv);
  }
}

LVAE_API int lvae_copy_window(const void* src, void* dst, int B, int C, int Hs, int Ws, int Hd, int Wd, int sy0,
                              int sx0, int dy0, int dx0, int h, int w, int src_nchw, int dst_nchw,
                              int src_dtype, int dst_dtype, cudaStream_t stream) {
  LVAE_REQUIRE(src && dst && B > 0 && C > 0 && h > 0 && w > 0, "copy_window: bad args");
  LVAE_REQUIRE(sy0 >= 0 && sx0 >= 0 && sy0 + h <= Hs && sx0 + w <= Ws && dy0 >= 0 && dx0 >= 0 && dy0 + h <= Hd && dx0 + w <= Wd,
               "copy_window: window out of range");
  long long n = (long long)B * h * w * C;
  const int esz = src_dtype == 0 ? 4 : 2;
  if (!src_nchw && !dst_nchw && src_dtype == dst_dtype && (C * esz) % 16 == 0 && n * esz / 16 < (1LL << 31)) {
    const unsigned CV = (unsigned)(C * esz / 16);
    lvae_launch(copy_window_vec_kernel, ew_grid(n * esz / 16, 256), 256, 0, stream, (const uint4*)src, (uint4*)dst, (unsigned)B, CV,
                (unsigned)Hs, (unsigned)Ws, (unsigned)Hd, (unsigned)Wd, (unsigned)sy0, (unsigned)sx0, (unsigned)dy0, (unsigned)dx0,
                (unsigned)h, (unsigned)w);
    LVAE_COUNT_LAUNCH();
    LVAE_CHECK_LAUNCH("copy_window");
    return LVAE_OK;
  }
  int g = ew_grid(n, 256);
#define CW(TS, TD) lvae_launch(copy_window_kernel<TS, TD>, g, 256, 0, stream, (const TS*)src, (TD*)dst, B, C, Hs, Ws, Hd, Wd, sy0, sx0, dy0, dx0, h, w, src_nchw, dst_nchw)
  if (src_dtype == 0 && dst_dtype == 0) CW(float, float);
  else if (src_dtype == 0 && dst_dtype == 1) CW(float, __nv_bfloat16);
  else if (src_dtype == 1 && dst_dtype == 0) CW(__nv_bfloat16, float);
  else CW(__nv_bfloat16, __nv_bfloat16);
#undef CW
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("copy_window");
  return LVAE_OK;
}

// =========================================================================================
// Dropout2d keep masks for every dropout site of one step in ONE launch:
// masks[i] = (u_i >= p) / (1-p), i over (site, sample, channel).  RNG state lives on the device.
// =========================================================================================
__global__ void dropout_masks_kernel(float* masks, long long n, float p, const PhiloxState* st, unsigned long long stream_id) {
  pdl_wait();
  pdl_launch();
  PhiloxState s = *st;
  float inv = 1.f / (1.f - p);
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q * 4 < n; q += (long long)gridDim.x * blockDim.x) {
    float4 u = philox_uniform4(s, stream_id, (unsigned long long)q);
    float v[4] = {u.x, u.y, u.z, u.w};
    for (int j = 0; j < 4 && q * 4 + j < n; ++j) masks[q * 4 + j] = v[j] > p ? inv : 0.f;
  }
}

LVAE_API int lvae_dropout_masks(float* masks, long long n, float p, const void* rng_state, unsigned long long stream_id,
                                cudaStream_t stream) {
  LVAE_REQUIRE(masks && n > 0 && p >= 0.f && p < 1.f && rng_state, "dropout_masks: bad args");
  lvae_launch(dropout_masks_kernel, ew_grid((n + 3) / 4, 256), 256, 0, stream, masks, n, p, (const PhiloxState*)rng_state, stream_id);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("dropout_masks");
  return LVAE_OK;
}

__global__ void rng_advance_kernel(PhiloxState* st, unsigned long long inc) {
  pdl_wait();
  pdl_launch(); st->offset += inc; }

// rng_state: device uint64[2] = {seed, offset}; advance once per step (graph-replay safe)
LVAE_API int lvae_rng_advance(void* rng_state, unsigned long long inc, cudaStream_t stream) {
  LVAE_REQUIRE(rng_state, "rng_advance: null state");
  lvae_launch(rng_advance_kernel, 1, 1, 0, stream, (PhiloxState*)rng_state, inc);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("rng_advance");
  return LVAE_OK;
}

// out[i] (+)= sum_b x[b, i]  (top-layer prior gradient: the prior is a batch-1 parameter, lvae_layers.py:131-136)
// A CTA owns 32 consecutive i; its eight warps split the batch (b = warp, warp + 8, ...: coalesced 128-byte rows, independent
// loads) and meet in shared memory in a fixed order.  One thread per i walking the whole batch (256 dependent iterations in a
// single CTA for the 2x2x64 prior) took 15-30 us on the main chain of the backward pass.
__global__ void __launch_bounds__(256) sum_batch_kernel(const float* __restrict__ x, float* __restrict__ out, int B, long long n,
                                                        int accumulate) {
  pdl_wait();
  pdl_launch();
  __shared__ float part[8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (long long i0 = (long long)blockIdx.x * 32; i0 < n; i0 += (long long)gridDim.x * 32) {
    const long long i = i0 + lane;
    float s = 0.f;
    if (i < n)
      for (int b = warp; b < B; b += 8) s += x[(long long)b * n + i];
    part[warp][lane] = s;
    __syncthreads();
    if (warp == 0 && i < n) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += part[w][lane];
      out[i] = accumulate ? out[i] + t : t;
    }
    __syncthreads();
  }
}

LVAE_API int lvae_sum_batch(const float* x, float* out, int B, long long n, int accumulate, cudaStream_t stream) {
  LVAE_REQUIRE(x && out && B > 0 && n > 0, "sum_batch: bad args");
  lvae_launch(sum_batch_kernel, ew_grid((n + 31) / 32, 1), 256, 0, stream, x, out, B, n, accumulate);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("sum_batch");
  return LVAE_OK;
}

// y[b,hw,c] = x[b,hw,c] * scale[b,c]   (Dropout2d mask applied to a gradient before the bf16 tensor-core dgrad,
// whose TMA-fed operands never pass through registers)
template <typename T>
__global__ void channel_scale_kernel(const T* __restrict__ x, const float* __restrict__ scale, T* __restrict__ y,
                                     long long nquads, int hw, int C) {
  pdl_wait();
  pdl_launch();
  const int CV = C >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nquads; i += (long long)gridDim.x * blockDim.x) {
    long long row = i / CV;
    int c = (int)(i - row * CV) * 4;
    long long b = row / hw;
    float4 v = ld4<T>(x + i * 4);
    float4 s = *reinterpret_cast<const float4*>(scale + b * C + c);
    st4<T>(y + i * 4, make_float4(v.x * s.x, v.y * s.y, v.z * s.z, v.w * s.w));
  }
}

LVAE_API int lvae_channel_scale(const void* x, const float* scale, void* y, int B, int HW, int C, int dtype_in,
                                cudaStream_t stream) {
  LVAE_REQUIRE(x && scale && y && C % 4 == 0, "channel_scale: bad args");
  long long nq = (long long)B * HW * (C / 4);
  if (dtype_in == 0) lvae_launch(channel_scale_kernel<float>, ew_grid(nq, 256), 256, 0, stream, (const float*)x, scale, (float*)y, nq, HW, C);
  else lvae_launch(channel_scale_kernel<__nv_bfloat16>, ew_grid(nq, 256), 256, 0, stream, (const __nv_bfloat16*)x, scale, (__nv_bfloat16*)y, nq, HW, C);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("channel_scale");
  return LVAE_OK;
}

// =========================================================================================
// Fused variants used by the block-level schedule (no finalize / params / mask kernels):
//   bn_act_fwd2: mean / rstd derived in-kernel from the statistics accumulator (train) or the running
//                statistics (eval); block 0 also writes the saved statistics and updates the running ones.
//   bn_act_bwd2: apply pass that also emits dgamma / dbeta, an optional Dropout2d mask on dx
//                (post_scale, the mask of the conv that produced x) and an optional residual add.
// The accumulators are NOT cleared here: the model zeroes its whole BatchNorm scratch arena once per forward.
// =========================================================================================
template <typename TI, typename TO, int V, int ACT = -1>
__global__ void bn_act_fwd2_kernel(const TI* __restrict__ x, TO* __restrict__ y, const double* __restrict__ acc,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* __restrict__ save, float* running_mean, float* running_var,
                                   long long* nbt, long long nvec, long long P, int C, int act_rt, int training,
                                   float momentum, float eps) {
  pdl_wait();
  pdl_launch();
  const int act = ACT >= 0 ? ACT : act_rt;
  __shared__ __align__(16) float s_scale[256], s_shift[256];       // y = act(x * scale + shift), C <= 256
  const int CV = C / V;
  const long long stride = (long long)gridDim.x * blockDim.x;      // multiple of CV by construction
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool has = i < nvec;
  RawV<TI, V> rx;
  if (has) rx = ldraw<TI, V>(x + i * V);                           // in flight during the statistics prologue
  // one thread per channel derives the statistics (the only double-precision math in the kernel; the reciprocal of P is
  // taken while the accumulator loads are in flight -- two double divisions behind them cost ~0.4 us per launch)
  // block 0 also updates the running statistics: their old values are requested now, not behind the statistics (a second,
  // dependent global round trip in the one block every launch has to wait for)
  float rm_old = 0.f, rv_old = 0.f;
  const bool upd = blockIdx.x == 0 && training && running_mean && (int)threadIdx.x < C;
  if (upd) { rm_old = running_mean[threadIdx.x]; rv_old = running_var[threadIdx.x]; }
  const double invP = 1.0 / (double)P;
  // FP64 issues at a fraction of the FP32 rate here, and the 2 x 7 stripe additions per channel were one dependent chain in two
  // warps (~0.9 us per launch, profiles/bench_bn_prologue.py): one thread per (statistic, channel) sums the stripes -- four
  // warps, one per scheduler for C = 64 -- and hands the two means over through shared memory
  __shared__ double s_m[2][256];
  if (training) {
    for (int k = threadIdx.x; k < 2 * C; k += blockDim.x) s_m[k >= C ? 1 : 0][k >= C ? k - C : k] = acc_sum(acc, k, C) * invP;
    __syncthreads();
  }
  for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
    float mean, rstd;
    if (training) {
      double m = s_m[0][ch];
      double var = s_m[1][ch] - m * m;
      if (var < 0.0) var = 0.0;
      mean = (float)m;
      rstd = rsqrtf((float)var + eps);
      if (blockIdx.x == 0 && running_mean) {
        double unb = P > 1 ? var * (double)P / (double)(P - 1) : var;
        const float ro = ch == (int)threadIdx.x ? rm_old : running_mean[ch], vo = ch == (int)threadIdx.x ? rv_old : running_var[ch];
        running_mean[ch] = (float)((1.0 - momentum) * (double)ro + momentum * m);
        running_var[ch] = (float)((1.0 - momentum) * (double)vo + momentum * unb);
      }
    } else {
      mean = running_mean[ch];
      rstd = rsqrtf(running_var[ch] + eps);
    }
    if (blockIdx.x == 0) {
      save[ch] = mean;
      save[C + ch] = rstd;
    }
    float sc = rstd * gamma[ch];
    s_scale[ch] = sc;
    s_shift[ch] = beta[ch] - mean * sc;
  }
  // (a reduction, not load-add-store: thread 0 would wait a global round trip in front of the barrier below)
  if (blockIdx.x == 0 && threadIdx.x == 0 && training && nbt) atomicAdd(reinterpret_cast<unsigned long long*>(nbt), 1ULL);
  __syncthreads();
  const int c = (int)(i % CV) * V;
  float sc[V], sh[V];
#pragma unroll
  for (int j = 0; j < V; ++j) { sc[j] = s_scale[c + j]; sh[j] = s_shift[c + j]; }
  while (has) {
    float v[V];
    unraw(rx, v);
    const long long inext = i + stride;
    const bool hn = inext < nvec;
    if (hn) rx = ldraw<TI, V>(x + inext * V);
#pragma unroll
    for (int j = 0; j < V; ++j) v[j] = act_fwd_t<sizeof(TO) == 2>(v[j] * sc[j] + sh[j], act);
    stv<TO, V>(y + i * V, v);
    i = inext;
    has = hn;
  }
}

// GATE: the gate backward of the residual block that PRODUCED x (the next block of the backward pass) rides in the same pass --
// dx of this BatchNorm (+ residual gradient) is exactly that block's output gradient: dh = gate'(dx, gh) is written next to dx,
// one launch and one re-read of dx less per pair of adjacent blocks (ops.GatedBlockFn hands the pending apply over).
template <typename T, int V, int ACT = -1, bool GATE = false>
__global__ void __launch_bounds__(256, GATE ? 2 : 3) bn_act_bwd2_kernel(const T* __restrict__ dy, const T* __restrict__ x, T* __restrict__ dx,
                                   const float* __restrict__ save, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, const double* __restrict__ acc,
                                   float* dgamma, float* dbeta, const float* __restrict__ post_scale,
                                   const T* __restrict__ add, long long nvec, long long P, int hw, int C, int act_rt,
                                   int training, const T* __restrict__ gh = nullptr, T* __restrict__ gdh = nullptr,
                                   int gate_act_rt = 0) {
  pdl_wait();
  pdl_launch();
  const int act = ACT >= 0 ? ACT : act_rt;
  const int gact = ACT >= 0 ? ACT : gate_act_rt;          // (the ELU instantiation serves blocks whose gate is ELU as well)
  // per-channel constants live in shared memory (two float4 per channel), not in 6 x V registers per thread
  __shared__ __align__(16) float s_t[6][256];                     // mean, rstd, gamma, beta, m1, m2 (SoA: conflict-free V-wide reads)
  const int CV = C / V;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c = (int)(i % CV) * V;
  bool has = i < nvec;
  RawV<T, V> rx, rd, ra, rha, rhg;
  if (has) {                                                       // in flight during the prologue
    rx = ldraw<T, V>(x + i * V);
    rd = ldraw<T, V>(dy + i * V);
    if (add) ra = ldraw<T, V>(add + i * V);
    if (GATE) {
      const size_t hrow = (size_t)((unsigned)i / (unsigned)CV) * 2 * C + c;
      rha = ldraw<T, V>(gh + hrow);
      rhg = ldraw<T, V>(gh + hrow + C);
    }
  }
  const double invP = 1.0 / (double)P;
  for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
    const double a1 = acc_sum(acc, ch, C), a2 = acc_sum(acc, C + ch, C);
    const float mean = save[ch], rstd = save[C + ch], gm = gamma[ch];
    s_t[0][ch] = mean; s_t[1][ch] = rstd; s_t[2][ch] = gm; s_t[3][ch] = beta[ch];
    s_t[4][ch] = training ? (float)(a1 * invP) : 0.f;
    s_t[5][ch] = training ? (float)(a2 * invP) : 0.f;
    if (blockIdx.x == 0) {
      // fire-and-forget reductions (RED): a load-add-store here is a dependent global round trip in the one block every
      // launch waits for; nothing else touches these gradient entries concurrently
      if (dbeta) atomicAdd(dbeta + ch, (float)a1);
      if (dgamma) atomicAdd(dgamma + ch, (float)a2);
    }
  }
  __syncthreads();
  while (has) {
    float xs[V], ds[V], av[V], o[V], ha[V], hg[V];
    unraw(rx, xs);
    unraw(rd, ds);
    if (add) unraw(ra, av);
    if (GATE) { unraw(rha, ha); unraw(rhg, hg); }
    const long long inext = i + stride;
    const bool hn = inext < nvec;
    if (hn) {
      rx = ldraw<T, V>(x + inext * V);
      rd = ldraw<T, V>(dy + inext * V);
      if (add) ra = ldraw<T, V>(add + inext * V);
      if (GATE) {
        const size_t hrow = (size_t)((unsigned)inext / (unsigned)CV) * 2 * C + c;
        rha = ldraw<T, V>(gh + hrow);
        rhg = ldraw<T, V>(gh + hrow + C);
      }
    }
    int cc = c;
    asm volatile("" : "+r"(cc));                                  // keep the table reads inside the loop (not hoisted into 6 x V registers)
#pragma unroll
    for (int q = 0; q < V / 4; ++q) {                              // four channels at a time: 6 LDS.128, 24 live constants
      float tb[6][4];
#pragma unroll
      for (int k = 0; k < 6; ++k) *reinterpret_cast<float4*>(&tb[k][0]) = *reinterpret_cast<const float4*>(&s_t[k][cc + 4 * q]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 4 * q + e;
        const float xh = (xs[j] - tb[0][e]) * tb[1][e];
        const float gpre = ds[j] * act_bwd_t<sizeof(T) == 2>(fmaf(xh, tb[2][e], tb[3][e]), act);
        o[j] = tb[2][e] * tb[1][e] * (gpre - tb[4][e] - xh * tb[5][e]);
      }
    }
    if (post_scale) {
      const unsigned bidx = ((unsigned)i / (unsigned)CV) / (unsigned)hw;      // vector, pixel and image indices fit 32 bits (checked by the launcher)
      const float* ps = post_scale + (size_t)bidx * C + c;
#pragma unroll
      for (int j = 0; j < V; ++j) o[j] *= ps[j];
    }
    if (add) {
#pragma unroll
      for (int j = 0; j < V; ++j) o[j] += av[j];
    }
    stv<T, V>(dx + i * V, o);
    if (GATE) {
      // same arithmetic as gate_bwd_kernel on dx AS STORED (rounded to T): bit-identical to the two-launch route
      float da[V], dg[V];
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float dv = round_to<T>(o[j]);
        const float sg = sigmoid_t<sizeof(T) == 2>(hg[j]);
        da[j] = dv * sg * act_bwd_t<sizeof(T) == 2>(ha[j], gact);
        dg[j] = dv * act_fwd_t<sizeof(T) == 2>(ha[j], gact) * sg * (1.f - sg);
      }
      const size_t hrow = (size_t)((unsigned)i / (unsigned)CV) * 2 * C + c;
      stv<T, V>(gdh + hrow, da);
      stv<T, V>(gdh + hrow + C, dg);
    }
    i = inext;
    has = hn;
  }
}

// grid whose total thread count is a multiple of C/4, so that every thread keeps the same channel quad
// Grid of the BatchNorm apply kernels: every CTA re-derives the per-channel table in double precision (FP64 issue rate is
// 1/64 of FP32 on this part), so fewer, longer-running CTAs win: cap at BN_CTAS_PER_SM CTAs per SM.
constexpr int BN_CTAS_PER_SM = 4;
static inline int bn_grid_cap() { return BN_CTAS_PER_SM * lvae_num_sms(); }
// resident CTAs per SM of a kernel at 256 threads (a grid of 4 CTAs per SM for a kernel that fits 3 runs as 1.33 waves)
template <typename K> static inline int resident_ctas(K kernel) {
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 256, 0) != cudaSuccess || occ < 1) occ = 1;
  return occ;
}
static inline int ew_grid_aligned(long long n, int threads, int CV, int max_resident = 1 << 20) {
  int g = ew_grid(n, threads);
  if (g > bn_grid_cap()) g = bn_grid_cap();
  if (g > max_resident * lvae_num_sms()) g = max_resident * lvae_num_sms();
  while (((long long)g * threads) % CV != 0) ++g;
  return g;
}

LVAE_API int lvae_bn_act_fwd2(const void* x, void* y, const double* acc, const float* gamma, const float* beta,
                              float* save, float* running_mean, float* running_var, long long* nbt, long long P, int C,
                              int act, int training, float momentum, float eps, int dtype_in, int dtype_out,
                              cudaStream_t stream) {
  LVAE_REQUIRE(x && y && gamma && beta && save && P > 0 && bn_c_ok(C), "bn_act_fwd2: bad args");
  LVAE_REQUIRE(training ? acc != nullptr : (running_mean && running_var), "bn_act_fwd2: statistics source missing");
  if (dtype_in == 1 && dtype_out == 1 && use_v8(1, C)) {
    long long nv = P * (C / 8);
    int g = ew_grid_aligned(nv, 256, C / 8);
    if (act == ACT_ELU)
      lvae_launch(bn_act_fwd2_kernel<__nv_bfloat16, __nv_bfloat16, 8, ACT_ELU>, g, 256, 0, stream, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, acc, gamma,
          beta, save, running_mean, running_var, nbt, nv, P, C, act, training, momentum, eps);
    else
      lvae_launch(bn_act_fwd2_kernel<__nv_bfloat16, __nv_bfloat16, 8>, g, 256, 0, stream, (const __nv_bfloat16*)x, (__nv_bfloat16*)y, acc, gamma,
          beta, save, running_mean, running_var, nbt, nv, P, C, act, training, momentum, eps);
  } else {
    long long nq = P * (C / 4);
    int g = ew_grid_aligned(nq, 256, C / 4);
#define FW2(TI, TO) lvae_launch(bn_act_fwd2_kernel<TI, TO, 4>, g, 256, 0, stream, (const TI*)x, (TO*)y, acc, gamma, beta, save, running_mean, running_var, nbt, nq, P, C, act, training, momentum, eps)
    if (dtype_in == 0 && dtype_out == 0) FW2(float, float);
    else if (dtype_in == 0 && dtype_out == 1) FW2(float, __nv_bfloat16);
    else if (dtype_in == 1 && dtype_out == 1) FW2(__nv_bfloat16, __nv_bfloat16);
    else FW2(__nv_bfloat16, float);
#undef FW2
  }
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_act_fwd2");
  return LVAE_OK;
}

// reduce pass (shared with lvae_bn_act_bwd) + fused apply
LVAE_API int lvae_bn_act_bwd2(const void* dy, const void* x, void* dx, const float* save, const float* gamma,
                              const float* beta, double* acc, float* dgamma, float* dbeta, const float* post_scale,
                              const void* add, long long P, int hw, int C, int act, int training, int dtype,
                              int skip_reduce, cudaStream_t stream) {
  LVAE_REQUIRE(dy && x && dx && save && gamma && beta && acc && P > 0 && bn_c_ok(C), "bn_act_bwd2: bad args");
  LVAE_REQUIRE(P * (long long)C < (1LL << 32), "bn_act_bwd2: more than 2^32 elements");
  long long nq = P * (C / 4);
  if (!skip_reduce) {            // the producer of dy (tcgen05 dgrad epilogue) may already have accumulated the sums
    launch_bwd_reduce(dy, x, save, save + C, gamma, beta, acc, P, C, act, dtype, stream);
    LVAE_COUNT_LAUNCH();
    LVAE_CHECK_LAUNCH("bn_act_bwd_reduce");
  }
  if (use_v8(dtype, C)) {
    long long nv = P * (C / 8);
    static const int occ_elu = resident_ctas(bn_act_bwd2_kernel<__nv_bfloat16, 8, ACT_ELU>);
    static const int occ_any = resident_ctas(bn_act_bwd2_kernel<__nv_bfloat16, 8>);
    int g = ew_grid_aligned(nv, 256, C / 8, act == ACT_ELU ? occ_elu : occ_any);
    if (act == ACT_ELU)
      lvae_launch(bn_act_bwd2_kernel<__nv_bfloat16, 8, ACT_ELU>, g, 256, 0, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (__nv_bfloat16*)dx, save,
          gamma, beta, acc, dgamma, dbeta, post_scale, (const __nv_bfloat16*)add, nv, P, hw, C, act, training,
          (const __nv_bfloat16*)nullptr, (__nv_bfloat16*)nullptr, 0);
    else
      lvae_launch(bn_act_bwd2_kernel<__nv_bfloat16, 8>, g, 256, 0, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (__nv_bfloat16*)dx, save,
          gamma, beta, acc, dgamma, dbeta, post_scale, (const __nv_bfloat16*)add, nv, P, hw, C, act, training,
          (const __nv_bfloat16*)nullptr, (__nv_bfloat16*)nullptr, 0);
  } else {
    int g = ew_grid_aligned(nq, 256, C / 4);
    if (dtype == 0)
      lvae_launch(bn_act_bwd2_kernel<float, 4>, g, 256, 0, stream, (const float*)dy, (const float*)x, (float*)dx, save, gamma, beta, acc, dgamma, dbeta, post_scale, (const float*)add, nq, P, hw, C, act, training, (const float*)nullptr, (float*)nullptr, 0);
    else
      lvae_launch(bn_act_bwd2_kernel<__nv_bfloat16, 4>, g, 256, 0, stream, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (__nv_bfloat16*)dx, save, gamma, beta, acc, dgamma, dbeta, post_scale, (const __nv_bfloat16*)add, nq, P, hw, C, act, training, (const __nv_bfloat16*)nullptr, (__nv_bfloat16*)nullptr, 0);
  }
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_act_bwd2");
  return LVAE_OK;
}

// BatchNorm-backward apply of one residual block (dx = BN'(dy, x) + add) and the gate backward of the block that produced x
// (dh = gate'(dx, gh), gh / dh: (P, 2C)) in one pass.  bf16, C % 8 == 0, C <= 256; the statistics sums are already in acc.
LVAE_API int lvae_bn_act_bwd2_gate(const void* dy, const void* x, void* dx, const float* save, const float* gamma,
                                   const float* beta, double* acc, float* dgamma, float* dbeta, const float* post_scale,
                                   const void* add, const void* gate_h, void* gate_dh, long long P, int hw, int C, int act,
                                   int gate_act, int training, cudaStream_t stream) {
  LVAE_REQUIRE(dy && x && dx && save && gamma && beta && acc && gate_h && gate_dh && P > 0 && bn_c_ok(C) && C % 8 == 0,
               "bn_act_bwd2_gate: bad args");
  LVAE_REQUIRE(P * (long long)C < (1LL << 32), "bn_act_bwd2_gate: more than 2^32 elements");
  typedef __nv_bfloat16 bf;
  const long long nv = P * (C / 8);
  if (act == ACT_ELU && gate_act == ACT_ELU) {
    static const int occ = resident_ctas(bn_act_bwd2_kernel<bf, 8, ACT_ELU, true>);
    const int g = ew_grid_aligned(nv, 256, C / 8, occ);
    lvae_launch(bn_act_bwd2_kernel<bf, 8, ACT_ELU, true>, g, 256, 0, stream, (const bf*)dy, (const bf*)x, (bf*)dx, save, gamma, beta,
                acc, dgamma, dbeta, post_scale, (const bf*)add, nv, P, hw, C, act, training, (const bf*)gate_h, (bf*)gate_dh, gate_act);
  } else {
    static const int occ = resident_ctas(bn_act_bwd2_kernel<bf, 8, -1, true>);
    const int g = ew_grid_aligned(nv, 256, C / 8, occ);
    lvae_launch(bn_act_bwd2_kernel<bf, 8, -1, true>, g, 256, 0, stream, (const bf*)dy, (const bf*)x, (bf*)dx, save, gamma, beta,
                acc, dgamma, dbeta, post_scale, (const bf*)add, nv, P, hw, C, act, training, (const bf*)gate_h, (bf*)gate_dh, gate_act);
  }
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("bn_act_bwd2_gate");
  return LVAE_OK;
}

template <typename T> __device__ __forceinline__ float4 round_as(float4 v);
template <> __device__ __forceinline__ float4 round_as<float>(float4 v) { return v; }
template <> __device__ __forceinline__ float4 round_as<__nv_bfloat16>(float4 v) {
  return make_float4(__bfloat162float(__float2bfloat16(v.x)), __bfloat162float(__float2bfloat16(v.y)),
                     __bfloat162float(__float2bfloat16(v.z)), __bfloat162float(__float2bfloat16(v.w)));
}

// gate forward that also accumulates the per-channel sum / sum of squares of its OUTPUT (the next
// residual block's first BatchNorm then needs no statistics pass of its own)
template <typename T, int V>
__global__ void gate_fwd_stats_kernel(const T* __restrict__ h, const T* __restrict__ res, T* __restrict__ out,
                                      double* __restrict__ acc, long long nvec, int C, int act) {
  pdl_wait();
  pdl_launch();
  extern __shared__ float sm[];
  const int CV = C / V;
  const long long stride = (long long)gridDim.x * blockDim.x;      // multiple of CV (256 % CV == 0)
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int cq = (int)(i % CV);
  float s[V], ss[V];
#pragma unroll
  for (int j = 0; j < V; ++j) s[j] = ss[j] = 0.f;
  for (; i < nvec; i += stride) {
    long long row = i / CV;
    int c = cq * V;
    float a[V], g[V], o[V];
    ldv<T, V>(h + row * 2 * C + c, a);
    ldv<T, V>(h + row * 2 * C + C + c, g);
#pragma unroll
    for (int j = 0; j < V; ++j) o[j] = act_fwd_t<sizeof(T) == 2>(a[j], act) * sigmoid_t<sizeof(T) == 2>(g[j]);
    if (res) {
      float r[V];
      ldv<T, V>(res + i * V, r);
#pragma unroll
      for (int j = 0; j < V; ++j) o[j] += r[j];
    }
    stv<T, V>(out + i * V, o);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float q = round_to<T>(o[j]);           // statistics of the value as stored (bf16-rounded on the bf16 path)
      s[j] += q;
      ss[j] += q * q;
    }
  }
  float* s_s = sm;
  float* s_ss = sm + blockDim.x * V;
#pragma unroll
  for (int j = 0; j < V; ++j) { s_s[threadIdx.x * V + j] = s[j]; s_ss[threadIdx.x * V + j] = ss[j]; }
  __syncthreads();
  if (threadIdx.x < C) {
    // blockDim % CV == 0, so thread t of any block owns channel group t % CV
    int cch = threadIdx.x, q = cch / V, e = cch % V;
    double a = 0.0, b = 0.0;
    for (int t = q; t < blockDim.x; t += CV) {
      a += (double)s_s[t * V + e];
      b += (double)s_ss[t * V + e];
    }
    double* accs = acc + (blockIdx.x & (BN_STRIPES - 1)) * 2 * C;
    atomicAdd(accs + cch, a);
    atomicAdd(accs + C + cch, b);
  }
}

LVAE_API int lvae_gate_fwd_stats(const void* h, const void* res, void* out, double* acc, long long P, int C, int act,
                                 int dtype, cudaStream_t stream) {
  LVAE_REQUIRE(h && out && acc && P > 0 && bn_c_ok(C) && 256 % (C / 4) == 0, "gate_fwd_stats: bad args");
  const int V = use_v8(dtype, C) ? 8 : 4;
  long long nv = P * (C / V);
  long long cap = 4LL * lvae_num_sms();
  long long want = (nv + 255) / 256;
  int g = (int)(want < cap ? (want > 0 ? want : 1) : cap);
  size_t smem = (size_t)256 * V * 2 * sizeof(float);
  if (V == 8) lvae_launch(gate_fwd_stats_kernel<__nv_bfloat16, 8>, g, 256, smem, stream, (const __nv_bfloat16*)h, (const __nv_bfloat16*)res, (__nv_bfloat16*)out, acc, nv, C, act);
  else if (dtype == 0) lvae_launch(gate_fwd_stats_kernel<float, 4>, g, 256, smem, stream, (const float*)h, (const float*)res, (float*)out, acc, nv, C, act);
  else lvae_launch(gate_fwd_stats_kernel<__nv_bfloat16, 4>, g, 256, smem, stream, (const __nv_bfloat16*)h, (const __nv_bfloat16*)res, (__nv_bfloat16*)out, acc, nv, C, act);
  LVAE_COUNT_LAUNCH();
  LVAE_CHECK_LAUNCH("gate_fwd_stats");
  return LVAE_OK;
}
