// HBM-bound backward kernels: GroupNorm(+SiLU) backward (two passes), per-(sample, channel)
// column sums (bias / time-embedding gradients), attention softmax backward, the tiny linear
// layers' backward, the loss gradient and a bf16 accumulate.  Channels-last bf16 activations,
// fp32 accumulation.  Reference semantics: autograd of the modules cited in include/mri_b200.h.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/mri_b200.h"
#include "common.h"

namespace mri {

__device__ __forceinline__ void unpack8b(const uint4& v, float (&f)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    f[2 * j] = __uint_as_float(w[j] << 16);
    f[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint4 pack8b(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
    w[j] = *reinterpret_cast<uint32_t*>(&h2);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// ---- packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2 issue two fp32 lanes per
// instruction).  The GroupNorm backward passes are co-limited by instruction issue (SiLU' costs
// ~20 scalar instructions per element against 4-6 bytes of HBM traffic), so the per-element
// math runs on channel PAIRS, and the sigmoid is 0.5 * tanh.approx(u / 2) + 0.5 (one MUFU
// instead of ex2 + rcp; relative error 2^-11, below the bf16 resolution of everything stored).
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float2 bf2_to_f2(uint32_t w) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t f2_to_bf2(float2 v) {
  __nv_bfloat162 h2 = __floats2bfloat162_rn(v.x, v.y);
  return *reinterpret_cast<uint32_t*>(&h2);
}
// du = d * silu'(u), u = xh * sc + sh
__device__ __forceinline__ float2 silu_bwd2(float2 d, float2 xh, float2 sc, float2 sh) {
  const float2 u = __ffma2_rn(xh, sc, sh);
  const float2 hu = __fmul2_rn(u, make_float2(0.5f, 0.5f));
  const float2 th = make_float2(tanh_approx(hu.x), tanh_approx(hu.y));
  const float2 sg = __ffma2_rn(th, make_float2(0.5f, 0.5f), make_float2(0.5f, 0.5f));
  const float2 t = __ffma2_rn(th, make_float2(-0.5f, -0.5f), make_float2(0.5f, 0.5f));  // 1 - sg
  const float2 w = __ffma2_rn(u, t, make_float2(1.0f, 1.0f));
  return __fmul2_rn(d, __fmul2_rn(sg, w));
}

struct GnCoef {
  float mean, rstd;
};
__device__ __forceinline__ GnCoef gn_coef(const double* stats, int sample, int stats_ld, int g,
                                          int comb, int cpg, int64_t spatial, float eps) {
  const double* st = stats + ((size_t)sample * stats_ld + g * comb) * 2;
  double s = 0.0, ss = 0.0;
  for (int j = 0; j < comb; ++j) {
    s += __ldg(st + 2 * j);
    ss += __ldg(st + 2 * j + 1);
  }
  const double inv_cnt = 1.0 / ((double)cpg * (double)spatial);
  const double mean = s * inv_cnt;
  double var = ss * inv_cnt - mean * mean;
  var = var < 0.0 ? 0.0 : var;
  GnCoef c;
  c.mean = (float)mean;
  c.rstd = rsqrtf((float)var + eps);
  return c;
}

// ---------------------------------------------------------------------------------------
// Pass A.  Per (sample, channel): S0 = sum dy, S1 = sum du, S2 = sum du * xhat, where
// u = xhat*gamma+beta, du = dy * silu'(u) (or dy when !silu).  With x == nullptr only S0 is
// produced (plain column sum).  grid (chunks, samples); thread = fixed 8-channel vector.
// sums: fp64 [3][samples][C] (fp64 atomics: the result does not depend on arrival order)
// ---------------------------------------------------------------------------------------
// kFine: groups of 4 channels (GroupNorm(8, 32) of the VAE's full-resolution level,
// ddpm_3d_ldm/vae.py:8): the two halves of a thread's 8-channel vector belong to different groups.
template <bool kSilu, bool kHasX, bool kFine>
__global__ void __launch_bounds__(256)
gn_bwd_reduce_kernel(const uint4* __restrict__ x, const uint4* __restrict__ dy,
                     const double* __restrict__ stats, const float* __restrict__ gamma,
                     const float* __restrict__ beta, double* __restrict__ sums, int samples,
                     int64_t spatial, int C, int groups, int stats_ld, int stats_cpg, float eps,
                     int rows_per_block) {
  extern __shared__ float part[];  // [rows_step][3][C]
  const int vec_per_row = C >> 3;
  const int sample = blockIdx.y;
  const int cv = threadIdx.x % vec_per_row;
  const int rsub = threadIdx.x / vec_per_row;
  const int rows_step = blockDim.x / vec_per_row;
  const int c = cv * 8;

  float2 sc[4], sh[4];
  constexpr int NH = kFine ? 2 : 1;
  float2 rs2[NH], nmr2[NH];  // xh = x * rstd - mean * rstd
#pragma unroll
  for (int h = 0; h < NH; ++h) {
    rs2[h] = make_float2(1.f, 1.f);
    nmr2[h] = make_float2(0.f, 0.f);
  }
  if (kHasX) {
    const int cpg = C / groups;
#pragma unroll
    for (int h = 0; h < NH; ++h) {
      const GnCoef k = gn_coef(stats, sample, stats_ld, (c + 4 * h) / cpg, cpg / stats_cpg, cpg,
                               spatial, eps);
      rs2[h] = make_float2(k.rstd, k.rstd);
      nmr2[h] = make_float2(-k.mean * k.rstd, -k.mean * k.rstd);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      sc[j] = make_float2(__ldg(gamma + c + 2 * j), __ldg(gamma + c + 2 * j + 1));
      sh[j] = make_float2(__ldg(beta + c + 2 * j), __ldg(beta + c + 2 * j + 1));
    }
  }
  float2 a0[4], a1[4], a2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) a0[j] = a1[j] = a2[j] = make_float2(0.f, 0.f);
  auto accum = [&](const uint4& dq, const uint4& xq) {
    const uint32_t dw[4] = {dq.x, dq.y, dq.z, dq.w};
    const uint32_t xw[4] = {xq.x, xq.y, xq.z, xq.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 d = bf2_to_f2(dw[j]);
      a0[j] = __fadd2_rn(a0[j], d);
      if (kHasX) {
        const int h = kFine ? (j >> 1) : 0;
        const float2 xh = __ffma2_rn(bf2_to_f2(xw[j]), rs2[h], nmr2[h]);
        const float2 du = kSilu ? silu_bwd2(d, xh, sc[j], sh[j]) : d;
        a1[j] = __fadd2_rn(a1[j], du);
        a2[j] = __ffma2_rn(du, xh, a2[j]);
      }
    }
  };
  // this block's rows [r0, r1) of the sample; thread rows r0 + rsub + k * rows_step
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = (int64_t)r0 + rows_per_block > spatial ? (int)spatial : r0 + rows_per_block;
  const uint4* dp = dy + (size_t)sample * spatial * vec_per_row + cv;
  const uint4* xp = kHasX ? x + (size_t)sample * spatial * vec_per_row + cv : dp;
  constexpr int U = 4;  // independent 16-byte loads in flight per thread and tensor
  const int stepv = rows_step * vec_per_row;
  int r = r0 + rsub;
  for (; r + (U - 1) * rows_step < r1; r += U * rows_step) {  // whole batches: no predicates
    uint4 dv[U], xv[U];
    const int o = r * vec_per_row;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      dv[u] = __ldg(dp + o + u * stepv);
      if (kHasX) xv[u] = __ldg(xp + o + u * stepv);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) accum(dv[u], kHasX ? xv[u] : dv[u]);
  }
  for (; r < r1; r += rows_step) {  // ragged end of the sample's last block
    const uint4 dq = __ldg(dp + r * vec_per_row);
    const uint4 xq = kHasX ? __ldg(xp + r * vec_per_row) : dq;
    accum(dq, xq);
  }
  float s0[8], s1[8], s2[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    s0[2 * j] = a0[j].x; s0[2 * j + 1] = a0[j].y;
    s1[2 * j] = a1[j].x; s1[2 * j + 1] = a1[j].y;
    s2[2 * j] = a2[j].x; s2[2 * j + 1] = a2[j].y;
  }
  // block reduction without shared-memory atomics: every thread parks its 24 fp32 partial sums,
  // then one thread per (quantity, channel) folds the rows_step partials in fp64 and issues the
  // block's single fp64 atomic for that address
  const int nq = kHasX ? 3 : 1;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    part[(size_t)(rsub * 3 + 0) * C + c + j] = s0[j];
    if (kHasX) {
      part[(size_t)(rsub * 3 + 1) * C + c + j] = s1[j];
      part[(size_t)(rsub * 3 + 2) * C + c + j] = s2[j];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nq * C; i += blockDim.x) {
    const int qi = i / C, ci = i - qi * C;
    double acc = 0.0;
    for (int r = 0; r < rows_step; ++r) acc += (double)part[(size_t)(r * 3 + qi) * C + ci];
    atomicAdd(sums + ((size_t)qi * samples + sample) * C + ci, acc);
  }
}

// ---------------------------------------------------------------------------------------
// Pass B.  dx = rstd * (gamma*du - m1 - xhat*m2) (+ add), with per (sample, group)
// m1 = mean(gamma*du), m2 = mean(gamma*du*xhat) from the pass-A sums.
// ---------------------------------------------------------------------------------------
template <bool kSilu, bool kFine>
__global__ void __launch_bounds__(256)
gn_bwd_apply_kernel(const uint4* __restrict__ x, const uint4* __restrict__ dy,
                    const uint4* __restrict__ add, uint4* __restrict__ dx,
                    const double* __restrict__ stats, const float* __restrict__ gamma,
                    const float* __restrict__ beta, const double* __restrict__ sums, int samples,
                    int64_t spatial, int C, int groups, int stats_ld, int stats_cpg, float eps,
                    int rows_per_block, double* __restrict__ colsum) {
  extern __shared__ float cpart[];  // [rows_step][C], only when colsum != nullptr
  __shared__ double gmean[2][64];   // per group: mean(gamma*du), mean(gamma*du*xhat)
  const int vec_per_row = C >> 3;
  const int sample = blockIdx.y;
  const int cv = threadIdx.x % vec_per_row;
  const int rsub = threadIdx.x / vec_per_row;
  const int rows_step = blockDim.x / vec_per_row;
  const int c = cv * 8;
  const int cpg = C / groups;
  constexpr int NH = kFine ? 2 : 1;   // kFine: cpg == 4, the vector's halves are two groups
  float csum[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) csum[j] = 0.f;
  GnCoef k[NH];
#pragma unroll
  for (int h = 0; h < NH; ++h)
    k[h] = gn_coef(stats, sample, stats_ld, (c + 4 * h) / cpg, cpg / stats_cpg, cpg, spatial, eps);
  {  // one warp per group folds the pass-A sums (every thread used to walk cpg channels itself)
    const double* S1 = sums + ((size_t)1 * samples + sample) * C;
    const double* S2 = sums + ((size_t)2 * samples + sample) * C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    const bool full = (blockDim.x & 31) == 0 || warp < nwarps - 1;  // partial last warp sits out
    if (full) {
      for (int gg = warp; gg < groups; gg += ((blockDim.x & 31) == 0 ? nwarps : nwarps - 1)) {
        double a1 = 0.0, a2 = 0.0;
        for (int j = gg * cpg + lane; j < (gg + 1) * cpg; j += 32) {
          const double gm = (double)__ldg(gamma + j);
          a1 += gm * __ldg(S1 + j);
          a2 += gm * __ldg(S2 + j);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          a1 += __shfl_xor_sync(0xffffffffu, a1, o);
          a2 += __shfl_xor_sync(0xffffffffu, a2, o);
        }
        if (lane == 0) {
          const double inv_cnt = 1.0 / ((double)cpg * (double)spatial);
          gmean[0][gg] = a1 * inv_cnt;
          gmean[1][gg] = a2 * inv_cnt;
        }
      }
    }
    __syncthreads();
  }
  // dx = (gamma * rstd) * du - rstd * m1 - (rstd * m2) * xh, on channel pairs
  float2 sc[4], sh[4], grs[4];
  float2 rs2[NH], nmr2[NH], nrm1[NH], nrm2[NH];
#pragma unroll
  for (int h = 0; h < NH; ++h) {
    const int g = (c + 4 * h) / cpg;
    const float m1 = (float)gmean[0][g];
    const float m2 = (float)gmean[1][g];
    rs2[h] = make_float2(k[h].rstd, k[h].rstd);
    nmr2[h] = make_float2(-k[h].mean * k[h].rstd, -k[h].mean * k[h].rstd);
    nrm1[h] = make_float2(-k[h].rstd * m1, -k[h].rstd * m1);
    nrm2[h] = make_float2(-k[h].rstd * m2, -k[h].rstd * m2);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int h = kFine ? (j >> 1) : 0;
    sc[j] = make_float2(__ldg(gamma + c + 2 * j), __ldg(gamma + c + 2 * j + 1));
    sh[j] = make_float2(__ldg(beta + c + 2 * j), __ldg(beta + c + 2 * j + 1));
    grs[j] = make_float2(sc[j].x * k[h].rstd, sc[j].y * k[h].rstd);
  }
  float2 cs2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) cs2[j] = make_float2(0.f, 0.f);
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block;
  if (r1 > spatial) r1 = spatial;
  const size_t base = (size_t)sample * spatial * vec_per_row + cv;
  constexpr int U = 4;  // independent 16-byte loads in flight per thread
  for (int64_t r = r0 + rsub; r < r1; r += (int64_t)rows_step * U) {
    uint4 xv[U], dv[U], av[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t ru = r + (int64_t)u * rows_step;
      if (ru < r1) {
        xv[u] = __ldg(x + base + ru * vec_per_row);
        dv[u] = __ldg(dy + base + ru * vec_per_row);
        if (add != nullptr) av[u] = __ldg(add + base + ru * vec_per_row);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t ru = r + (int64_t)u * rows_step;
      if (ru >= r1) continue;
      const uint32_t xw[4] = {xv[u].x, xv[u].y, xv[u].z, xv[u].w};
      const uint32_t dw[4] = {dv[u].x, dv[u].y, dv[u].z, dv[u].w};
      const uint32_t aw[4] = {av[u].x, av[u].y, av[u].z, av[u].w};
      uint32_t ow[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int h = kFine ? (j >> 1) : 0;
        const float2 d = bf2_to_f2(dw[j]);
        const float2 xh = __ffma2_rn(bf2_to_f2(xw[j]), rs2[h], nmr2[h]);
        const float2 du = kSilu ? silu_bwd2(d, xh, sc[j], sh[j]) : d;
        float2 o = __ffma2_rn(du, grs[j], nrm1[h]);
        o = __ffma2_rn(xh, nrm2[h], o);
        if (add != nullptr) o = __fadd2_rn(o, bf2_to_f2(aw[j]));
        ow[j] = f2_to_bf2(o);
        if (colsum != nullptr)  // column sums of the bf16 values a later pass would read
          cs2[j] = __fadd2_rn(cs2[j], bf2_to_f2(ow[j]));
      }
      dx[base + ru * vec_per_row] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    csum[2 * j] = cs2[j].x;
    csum[2 * j + 1] = cs2[j].y;
  }
  if (colsum != nullptr) {
#pragma unroll
    for (int j = 0; j < 8; ++j) cpart[(size_t)rsub * C + c + j] = csum[j];
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
      double acc = 0.0;
      for (int r = 0; r < rows_step; ++r) acc += (double)cpart[(size_t)r * C + i];
      atomicAdd(colsum + (size_t)sample * C + i, acc);
    }
  }
}

// out = a + b (bf16, 8 per thread)
__global__ void __launch_bounds__(256)
add_bf16_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out,
                int64_t nvec) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec;
       i += (int64_t)gridDim.x * blockDim.x) {
    float x[8], y[8];
    unpack8b(__ldg(a + i), x);
    unpack8b(__ldg(b + i), y);
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] += y[j];
    out[i] = pack8b(x);
  }
}

// dS = scale * P * (dP - sum_j dP_j P_j), one warp per row (fp32 dP, bf16 P -> bf16 dS)
template <int kPerLane>
__global__ void __launch_bounds__(256)
softmax_bwd_kernel(const __nv_bfloat16* __restrict__ P, const float* __restrict__ dP,
                   __nv_bfloat16* __restrict__ dS, int64_t rows, int cols, int ld_p, int ld_dp,
                   float scale) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const __nv_bfloat16* p = P + row * ld_p;
  const float* dp = dP + row * ld_dp;
  __nv_bfloat16* ds = dS + row * ld_p;
  float pv[kPerLane], dv[kPerLane];
  float dot = 0.f;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    const int c = lane + 32 * j;
    pv[j] = c < cols ? __bfloat162float(p[c]) : 0.f;
    dv[j] = c < cols ? __ldg(dp + c) : 0.f;
    dot = fmaf(pv[j], dv[j], dot);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) {
    const int c = lane + 32 * j;
    if (c < ld_p) ds[c] = __float2bfloat16(c < cols ? scale * pv[j] * (dv[j] - dot) : 0.f);
  }
}

// ---- tiny fp32 linear layers ------------------------------------------------------------
// dX[b, i] = sum_o dZ[b, o] W[o, i].  grid (i tiles, o chunks of 64, b): every block adds its
// partial sum with one fp32 atomic per element (dX is zeroed first) -- the concatenated block
// projections have out_f ~ 3.5-5 k, which one thread per (b, i) would walk serially.
__global__ void __launch_bounds__(256)
linear_bwd_input_kernel(const float* __restrict__ dZ, const float* __restrict__ W,
                        float* __restrict__ dX, int batch, int in_f, int out_f) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.z;
  const int o0 = blockIdx.y * 64;
  const int o1 = o0 + 64 < out_f ? o0 + 64 : out_f;
  if (i >= in_f) return;
  float acc = 0.f;
#pragma unroll 4
  for (int o = o0; o < o1; ++o)
    acc = fmaf(__ldg(dZ + (size_t)b * out_f + o), __ldg(W + (size_t)o * in_f + i), acc);
  atomicAdd(dX + (size_t)b * in_f + i, acc);
}
// dW[o, i] = sum_b dZ[b, o] X[b, i];  db[o] = sum_b dZ[b, o]   (overwrite)
__global__ void linear_bwd_weight_kernel(const float* __restrict__ dZ, const float* __restrict__ X,
                                         float* __restrict__ dW, float* __restrict__ db, int batch,
                                         int in_f, int out_f) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)out_f * in_f) return;
  const int o = (int)(idx / in_f), i = (int)(idx % in_f);
  float acc = 0.f, bs = 0.f;
  for (int b = 0; b < batch; ++b) {
    const float dz = __ldg(dZ + (size_t)b * out_f + o);
    acc = fmaf(dz, __ldg(X + (size_t)b * in_f + i), acc);
    bs += dz;
  }
  dW[idx] = acc;
  if (i == 0 && db != nullptr) db[o] = bs;
}
// SiLU forward / backward on small fp32 tensors (time-embedding MLP)
__global__ void silu_kernel(const float* __restrict__ z, float* __restrict__ y, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const float v = z[i];
    y[i] = v / (1.0f + expf(-v));
  }
}
__global__ void silu_bwd_kernel(const float* __restrict__ z, const float* __restrict__ dy,
                                float* __restrict__ dz, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const float v = z[i];
    const float sg = 1.0f / (1.0f + expf(-v));
    dz[i] = dy[i] * sg * (1.0f + v * (1.0f - sg));
  }
}

// d pred = upstream * 2 w_b / (B * P) * (pred - noise), w_b = min(snr, gamma)/snr (1 if gamma<=0)
__global__ void __launch_bounds__(256)
loss_bwd_kernel(const float* __restrict__ pred, const float* __restrict__ noise,
                const int64_t* __restrict__ t, const float* __restrict__ snr, float gamma,
                const float* __restrict__ upstream, float* __restrict__ dpred, int samples,
                int64_t per_sample) {
  const int sample = blockIdx.y;
  float w = 1.0f;
  if (gamma > 0.f) {
    const float s = snr[t[sample]];
    w = fminf(s, gamma) / s;
  }
  const float coef = upstream[0] * 2.0f * w / ((float)samples * (float)per_sample);
  const size_t base = (size_t)sample * per_sample;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < per_sample;
       j += (int64_t)gridDim.x * blockDim.x)
    dpred[base + j] = coef * (pred[base + j] - noise[base + j]);
}

// Multi-tensor Adam (torch.optim.Adam semantics: L2 weight decay added to the gradient, bias
// corrections, eps outside the square root of the corrected second moment), one launch for all
// parameters.  grad_scale / found_inf follow torch.amp.GradScaler's fused-optimizer protocol.
__global__ void __launch_bounds__(256)
adam_kernel(const MriAdamSeg* __restrict__ segs, int n_segs, float lr, float beta1, float beta2,
            float omb1, float omb2, float eps, float weight_decay, const float* __restrict__ step_dev,
            const float* __restrict__ grad_scale, const float* __restrict__ found_inf) {
  if (found_inf != nullptr && *found_inf != 0.f) return;  // skipped step (inf / nan gradients)
  // the step counter lives on the device (it must not advance on a skipped step, and the host
  // never learns about skips): bias corrections for step + 1
  const double stp = (double)*step_dev + 1.0;
  const float bc1 = (float)(1.0 - pow((double)beta1, stp));
  const float bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, stp));
  int lo = 0, hi = n_segs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (segs[mid].block0 <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const MriAdamSeg sg = segs[lo];
  const float inv_scale = grad_scale != nullptr ? 1.0f / *grad_scale : 1.0f;
  const float step_size = lr / bc1;
  auto update = [&](float& p, float g, float& m, float& v) {
    g *= inv_scale;
    if (weight_decay != 0.f) g = fmaf(weight_decay, p, g);
    m = m + omb1 * (g - m);               // exp_avg.lerp_(grad, 1 - beta1)
    v = fmaf(omb2 * g, g, beta2 * v);      // exp_avg_sq.mul_(beta2).addcmul_(g, g, value = 1 - beta2)
    const float denom = sqrtf(v) / bc2_sqrt + eps;
    p -= step_size * (m / denom);
  };
  const int64_t b0 = ((int64_t)blockIdx.x - sg.block0) * 1024;
  const bool vec = ((reinterpret_cast<uintptr_t>(sg.p) | reinterpret_cast<uintptr_t>(sg.g) |
                     reinterpret_cast<uintptr_t>(sg.m) | reinterpret_cast<uintptr_t>(sg.v)) & 15u) == 0 &&
                   b0 + 1024 <= sg.n;
  if (vec) {  // whole 1024-element block, 16-byte aligned streams: one float4 per thread and stream
    const int64_t i = b0 + (int64_t)threadIdx.x * 4;
    float4 p4 = *reinterpret_cast<const float4*>(sg.p + i);
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(sg.g + i));
    float4 m4 = *reinterpret_cast<const float4*>(sg.m + i);
    float4 v4 = *reinterpret_cast<const float4*>(sg.v + i);
    update(p4.x, g4.x, m4.x, v4.x);
    update(p4.y, g4.y, m4.y, v4.y);
    update(p4.z, g4.z, m4.z, v4.z);
    update(p4.w, g4.w, m4.w, v4.w);
    *reinterpret_cast<float4*>(sg.p + i) = p4;
    *reinterpret_cast<float4*>(sg.m + i) = m4;
    *reinterpret_cast<float4*>(sg.v + i) = v4;
    return;
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t i = b0 + threadIdx.x + (int64_t)u * 256;
    if (i >= sg.n) break;
    float p = sg.p[i], m = sg.m[i], v = sg.v[i];
    update(p, sg.g[i], m, v);
    sg.p[i] = p;
    sg.m[i] = m;
    sg.v[i] = v;
  }
}

__global__ void adam_advance_kernel(float* step_dev, const float* found_inf) {
  if (found_inf == nullptr || *found_inf == 0.f) *step_dev += 1.f;
}

// ATen's lerp (aten/src/ATen/native/Lerp.h) in fp32 opmath: the |w| < 0.5 branch and the other one
// are written as ATen writes them, so nvcc contracts them to the same FMAs as ATen's CUDA build.
__device__ __forceinline__ float ema_lerp(float e, float p, float w) {
  return fabsf(w) < 0.5f ? e + w * (p - e) : p - (p - e) * (1.0f - w);
}

// Multi-tensor EMA of the weights (see mri_ema_update): e <- lerp(e, p, 1 - d) for every segment,
// with d from the device-resident update counter.
__global__ void __launch_bounds__(256)
ema_update_kernel(const MriEmaSeg* __restrict__ segs, int n_segs, double decay, int warmup,
                  const int64_t* __restrict__ count_dev, const float* __restrict__ found_inf) {
  if (found_inf != nullptr && *found_inf != 0.f) return;  // skipped step: the average stays too
  const int64_t k = *count_dev + 1;
  const double d = !warmup ? decay : k <= 1 ? 0.0 : fmin(decay, (double)k / (9.0 + (double)k));
  const float w = (float)(1.0 - d);
  int lo = 0, hi = n_segs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (segs[mid].block0 <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const MriEmaSeg sg = segs[lo];
  const int64_t b0 = ((int64_t)blockIdx.x - sg.block0) * 1024;
  const bool vec = ((reinterpret_cast<uintptr_t>(sg.e) | reinterpret_cast<uintptr_t>(sg.p)) & 15u) == 0 &&
                   b0 + 1024 <= sg.n;
  if (vec) {  // whole 1024-element block, 16-byte aligned streams: one float4 per thread and stream
    const int64_t i = b0 + (int64_t)threadIdx.x * 4;
    float4 e4 = *reinterpret_cast<const float4*>(sg.e + i);
    const float4 p4 = __ldg(reinterpret_cast<const float4*>(sg.p + i));
    e4.x = ema_lerp(e4.x, p4.x, w);
    e4.y = ema_lerp(e4.y, p4.y, w);
    e4.z = ema_lerp(e4.z, p4.z, w);
    e4.w = ema_lerp(e4.w, p4.w, w);
    *reinterpret_cast<float4*>(sg.e + i) = e4;
    return;
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t i = b0 + threadIdx.x + (int64_t)u * 256;
    if (i >= sg.n) break;
    sg.e[i] = ema_lerp(sg.e[i], __ldg(sg.p + i), w);
  }
}

__global__ void ema_advance_kernel(int64_t* count_dev, const float* found_inf) {
  if (found_inf == nullptr || *found_inf == 0.f) *count_dev += 1;
}

// One launch finalises every parameter gradient of a backward segment (see MriFinalSeg).
__global__ void __launch_bounds__(256)
grad_finalize_kernel(const MriFinalSeg* __restrict__ segs, int n_segs) {
  int lo = 0, hi = n_segs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (segs[mid].block0 <= (int64_t)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const MriFinalSeg sg = segs[lo];
  const int64_t i0 = ((int64_t)blockIdx.x - sg.block0) * 2048 + threadIdx.x;
  if (sg.idx != nullptr) {
    const float* src = reinterpret_cast<const float*>(sg.src);
    int32_t e[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int64_t i = i0 + (int64_t)u * 256;
      e[u] = i < sg.n ? __ldg(sg.idx + i) : -1;
    }
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = e[u] >= 0 ? __ldg(src + e[u]) : 0.f;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int64_t i = i0 + (int64_t)u * 256;
      if (i < sg.n) sg.dst[i] = v[u];
    }
  } else {
    const double* src = reinterpret_cast<const double*>(sg.src);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int64_t i = i0 + (int64_t)u * 256;
      if (i >= sg.n) break;
      double acc = 0.0;
      for (int b = 0; b < sg.batch; ++b) acc += __ldg(src + (size_t)b * sg.ld + i);
      sg.dst[i] = (float)acc;
    }
  }
}

static inline int rows_per_block_for(int samples, int64_t spatial, int rows_step, dim3* grid,
                                     int blocks_per_sm = 2) {
  static const int env_bps = [] {
    const char* e = getenv("MRI_GN_BLOCKS_PER_SM");  // tuning probe (tools/gn_probe.py)
    return e != nullptr ? atoi(e) : 0;
  }();
  if (env_bps > 0) blocks_per_sm = env_bps;
  // chunks per sample rounded DOWN: the grid must fit ONE resident wave -- rounding up gives
  // e.g. 320 blocks on 296 slots at batch 64 (or 32), whose 24 stragglers run as a second wave
  int64_t want_blocks = (148 * blocks_per_sm) / samples;
  if (want_blocks < 1) want_blocks = 1;
  int64_t rows_per = (spatial + want_blocks - 1) / want_blocks;
  const int64_t quantum = (int64_t)rows_step * 4;
  rows_per = (rows_per + quantum - 1) / quantum * quantum;
  *grid = dim3((unsigned)((spatial + rows_per - 1) / rows_per), (unsigned)samples);
  return (int)rows_per;
}

}  // namespace mri

using namespace mri;

extern "C" int mri_adam_step(const MriAdamSeg* segs_dev, int n_segs, int64_t total_blocks, float lr,
                             float beta1, float beta2, float eps, float weight_decay, float* step_dev,
                             const float* grad_scale, const float* found_inf, void* stream) {
  if (n_segs < 1 || total_blocks < 1) return 0;
  if (step_dev == nullptr) return set_error(-2, "mri_adam_step: step counter missing");
  if (total_blocks > 0x7fffffffLL) return set_error(-2, "mri_adam_step: too many blocks");
  adam_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)stream>>>(
      segs_dev, n_segs, lr, beta1, beta2, (float)(1.0 - (double)beta1), (float)(1.0 - (double)beta2), eps,
      weight_decay, step_dev, grad_scale, found_inf);
  int rc = check_launch("adam_kernel");
  if (rc != 0) return rc;
  adam_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_dev, found_inf);
  return check_launch("adam_advance_kernel");
}

extern "C" int mri_ema_update(const MriEmaSeg* segs_dev, int n_segs, int64_t total_blocks, double decay,
                              int warmup, int64_t* count_dev, const float* found_inf, void* stream) {
  if (count_dev == nullptr) return set_error(-2, "mri_ema_update: update counter missing");
  if (!(decay >= 0.0 && decay < 1.0)) return set_error(-2, "mri_ema_update: decay outside [0, 1)");
  if (n_segs < 1 || total_blocks < 1) return 0;
  if (total_blocks > 0x7fffffffLL) return set_error(-2, "mri_ema_update: too many blocks");
  ema_update_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)stream>>>(
      segs_dev, n_segs, decay, warmup, count_dev, found_inf);
  int rc = check_launch("ema_update_kernel");
  if (rc != 0) return rc;
  ema_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(count_dev, found_inf);
  return check_launch("ema_advance_kernel");
}

extern "C" int mri_grad_finalize(const MriFinalSeg* segs_dev, int n_segs, int64_t total_blocks,
                                 void* stream) {
  if (n_segs < 1 || total_blocks < 1) return 0;
  if (total_blocks > 0x7fffffffLL) return set_error(-2, "mri_grad_finalize: too many blocks");
  grad_finalize_kernel<<<(unsigned)total_blocks, 256, 0, (cudaStream_t)stream>>>(segs_dev, n_segs);
  return check_launch("grad_finalize_kernel");
}

extern "C" int mri_gn_bwd_reduce(const void* x, const void* dy, const double* stats,
                                 const float* gamma, const float* beta, double* sums, int samples,
                                 int64_t spatial, int C, int groups, int stats_ld, int stats_cpg,
                                 float eps, int silu, void* stream) {
  if (C % 8 != 0 || C / 8 > 256) return set_error(-2, "mri_gn_bwd_reduce: bad C");
  if (x != nullptr && (groups < 1 || C % groups != 0 || (C / groups) % stats_cpg != 0))
    return set_error(-2, "mri_gn_bwd_reduce: bad group configuration");
  const int vpr = C / 8;
  const int threads = (256 / vpr) * vpr;
  dim3 grid;
  const int rpb = rows_per_block_for(samples, spatial, threads / vpr, &grid);
  const size_t smem = (size_t)threads * 24 * sizeof(float);  // [rows_step][3][C]
  const uint4* xp = reinterpret_cast<const uint4*>(x);
  const uint4* dp = reinterpret_cast<const uint4*>(dy);
  if (spatial * vpr > 0x7fffffffLL) return set_error(-2, "mri_gn_bwd_reduce: sample too large");
  cudaStream_t st = (cudaStream_t)stream;
#define MRI_GN_RED(S, X, F)                                                                     \
  gn_bwd_reduce_kernel<S, X, F><<<grid, threads, smem, st>>>(xp, dp, stats, gamma, beta, sums,  \
                                                             samples, spatial, C, groups,       \
                                                             stats_ld, stats_cpg, eps, rpb)
  const bool fine = x != nullptr && C / groups == 4;
  if (x != nullptr && (C / groups) % 8 != 0 && !fine)
    return set_error(-2, "mri_gn_bwd_reduce: channels per group must be 4 or a multiple of 8");
  if (x == nullptr) MRI_GN_RED(false, false, false);
  else if (silu && fine) MRI_GN_RED(true, true, true);
  else if (silu) MRI_GN_RED(true, true, false);
  else if (fine) MRI_GN_RED(false, true, true);
  else MRI_GN_RED(false, true, false);
#undef MRI_GN_RED
  return check_launch("gn_bwd_reduce_kernel");
}

extern "C" int mri_gn_bwd_apply(const void* x, const void* dy, const void* add, void* dx,
                                const double* stats, const float* gamma, const float* beta,
                                const double* sums, int samples, int64_t spatial, int C, int groups,
                                int stats_ld, int stats_cpg, float eps, int silu, double* colsum,
                                void* stream) {
  if (C % 8 != 0 || C / 8 > 256 || groups < 1 || C % groups != 0 || (C / groups) % stats_cpg != 0)
    return set_error(-2, "mri_gn_bwd_apply: bad channel / group configuration");
  const int vpr = C / 8;
  const int threads = (256 / vpr) * vpr;
  dim3 grid;
  const int rpb = rows_per_block_for(samples, spatial, threads / vpr, &grid);
  const uint4* xp = reinterpret_cast<const uint4*>(x);
  const uint4* dp = reinterpret_cast<const uint4*>(dy);
  const uint4* ap = reinterpret_cast<const uint4*>(add);
  uint4* op = reinterpret_cast<uint4*>(dx);
  if (groups > 64) return set_error(-2, "mri_gn_bwd_apply: more than 64 groups");
  const size_t csm = colsum != nullptr ? (size_t)threads * 8 * sizeof(float) : 0;
  const bool fine = C / groups == 4;
  if ((C / groups) % 8 != 0 && !fine)
    return set_error(-2, "mri_gn_bwd_apply: channels per group must be 4 or a multiple of 8");
#define MRI_GN_APP(S, F)                                                                          \
  gn_bwd_apply_kernel<S, F><<<grid, threads, csm, (cudaStream_t)stream>>>(                        \
      xp, dp, ap, op, stats, gamma, beta, sums, samples, spatial, C, groups, stats_ld, stats_cpg, \
      eps, rpb, colsum)
  if (silu && fine) MRI_GN_APP(true, true);
  else if (silu) MRI_GN_APP(true, false);
  else if (fine) MRI_GN_APP(false, true);
  else MRI_GN_APP(false, false);
#undef MRI_GN_APP
  return check_launch("gn_bwd_apply_kernel");
}

extern "C" int mri_add_bf16(const void* a, const void* b, void* out, int64_t n, void* stream) {
  if (n % 8 != 0) return set_error(-2, "mri_add_bf16: n must be a multiple of 8");
  const int64_t nvec = n / 8;
  int64_t blocks = (nvec + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  add_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b),
      reinterpret_cast<uint4*>(out), nvec);
  return check_launch("add_bf16_kernel");
}

extern "C" int mri_softmax_bwd(const void* P, const float* dP, void* dS, int64_t rows, int cols,
                               int ld_p, int ld_dp, float scale, void* stream) {
  if (rows < 1 || cols < 1 || ld_p < cols || ld_dp < cols || ld_p > 2048)
    return set_error(-2, "mri_softmax_bwd: bad shape");
  const unsigned grid = (unsigned)((rows + 7) / 8);
  const __nv_bfloat16* Pp = reinterpret_cast<const __nv_bfloat16*>(P);
  __nv_bfloat16* Sp = reinterpret_cast<__nv_bfloat16*>(dS);
  cudaStream_t st = (cudaStream_t)stream;
  const int per_lane = (ld_p + 31) / 32;
  if (per_lane <= 8) softmax_bwd_kernel<8><<<grid, 256, 0, st>>>(Pp, dP, Sp, rows, cols, ld_p, ld_dp, scale);
  else if (per_lane <= 40) softmax_bwd_kernel<40><<<grid, 256, 0, st>>>(Pp, dP, Sp, rows, cols, ld_p, ld_dp, scale);
  else softmax_bwd_kernel<64><<<grid, 256, 0, st>>>(Pp, dP, Sp, rows, cols, ld_p, ld_dp, scale);
  return check_launch("softmax_bwd_kernel");
}

extern "C" int mri_linear_bwd(const float* dZ, const float* X, const float* W, float* dX, float* dW,
                              float* db, int batch, int in_f, int out_f, void* stream) {
  if (batch < 1 || in_f < 1 || out_f < 1) return set_error(-2, "mri_linear_bwd: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  if (dX != nullptr) {
    cudaError_t e = cudaMemsetAsync(dX, 0, (size_t)batch * in_f * sizeof(float), st);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaMemsetAsync(dX)");
    const dim3 grid((in_f + 255) / 256, (out_f + 63) / 64, batch);
    linear_bwd_input_kernel<<<grid, 256, 0, st>>>(dZ, W, dX, batch, in_f, out_f);
    int rc = check_launch("linear_bwd_input_kernel");
    if (rc) return rc;
  }
  if (dW != nullptr) {
    const int64_t n = (int64_t)out_f * in_f;
    linear_bwd_weight_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dZ, X, dW, db, batch, in_f,
                                                                         out_f);
    return check_launch("linear_bwd_weight_kernel");
  }
  return 0;
}

extern "C" int mri_silu(const float* z, float* y, int64_t n, void* stream) {
  silu_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(z, y, n);
  return check_launch("silu_kernel");
}
extern "C" int mri_silu_bwd(const float* z, const float* dy, float* dz, int64_t n, void* stream) {
  silu_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(z, dy, dz, n);
  return check_launch("silu_bwd_kernel");
}

extern "C" int mri_minsnr_loss_bwd(const float* pred, const float* noise, const int64_t* t,
                                   const float* snr, float gamma, const float* upstream,
                                   float* dpred, int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_minsnr_loss_bwd: empty input");
  int64_t bx = (per_sample + 255) / 256;
  int64_t cap = (148 * 8 + samples - 1) / samples;
  if (bx > cap) bx = cap;
  loss_bwd_kernel<<<dim3((unsigned)bx, (unsigned)samples), 256, 0, (cudaStream_t)stream>>>(
      pred, noise, t, snr, gamma, upstream, dpred, samples, per_sample);
  return check_launch("loss_bwd_kernel");
}
