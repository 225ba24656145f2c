// DDPM / DDIM / DPM-Solver++(2M) arithmetic as single fused passes.  fp32, written with explicit
// round-to-nearest intrinsics (never contracted into FMAs) in the reference's exact association
// order, so the result is bit-identical to eager torch on the same inputs.
// Reference call sites: see include/mri_b200.h.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/mri_b200.h"
#include "common.h"

namespace mri {

// ------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller with ATen's element mapping, so that the draws are bit-identical to
// torch.randn / randn_like on the same device for the same (seed, offset):
//   ATen launches G = min(#SM * (maxThreadsPerSM / 256), ceil(numel / 256)) blocks of 256 threads;
//   thread j (subsequence j) makes one curand_normal4 call per grid-stride iteration `it`
//   (Philox counter offset / 4 + it) and component ii of that call goes to element
//   e = it * 4 * Tt + ii * Tt + j with Tt = 256 * G; the generator offset advances by
//   4 * ceil(numel / (4 * Tt))  (ATen/native/cuda/DistributionTemplates.h: calc_execution_policy,
//   distribution_elementwise_grid_stride_kernel, normal_and_transform; curand_normal.h:
//   _curand_box_muller).  Here one thread owns FOUR consecutive subsequences, so that for each
//   component it holds four consecutive elements: 16-byte loads and stores.
// ------------------------------------------------------------------------------------------
// block `ctr` of subsequence `sub` of the generator seeded with `seed`
__device__ __forceinline__ uint4 philox4x32_10(uint64_t seed, uint64_t ctr, uint64_t sub) {
  uint4 c = make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)sub, (uint32_t)(sub >> 32));
  uint2 k = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    if (i < 9) {
      k.x += 0x9E3779B9u;
      k.y += 0xBB67AE85u;
    }
  }
  return c;
}

// two standard normals from two 32-bit draws: the operations (and their roundings) of
// _curand_box_muller followed by ATen's `rand * std + mean` with std = 1, mean = 0
__device__ __forceinline__ float2 box_muller(uint32_t x, uint32_t y) {
  const float kInv = 2.3283064e-10f;
  const float kInv2Pi = 2.3283064e-10f * 6.2831855f;
  const float u = fmaf((float)x, kInv, kInv / 2);
  const float v = fmaf((float)y, kInv2Pi, kInv2Pi / 2);
  const float s = sqrtf(-2.0f * logf(u));
  float sn, cs;
  __sincosf(v, &sn, &cs);
  return make_float2(fmaf(sn * s, 1.0f, 0.0f), fmaf(cs * s, 1.0f, 0.0f));
}

struct AtenGrid {
  long long Tt;     // threads of ATen's launch
  int n_iter;       // grid-stride iterations = curand_normal4 calls per thread
};

static int g_sm_count = 0, g_threads_per_sm = 0;
static int device_props() {
  if (g_sm_count != 0) return 0;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess)
    e = cudaDeviceGetAttribute(&g_threads_per_sm, cudaDevAttrMaxThreadsPerMultiProcessor, dev);
  if (e != cudaSuccess) {
    g_sm_count = 0;
    return set_cuda_error(e, "cudaDeviceGetAttribute(SM count / threads per SM)");
  }
  return 0;
}

static AtenGrid aten_grid(long long numel) {
  long long grid = (numel + 255) / 256;
  const long long cap = (long long)g_sm_count * (g_threads_per_sm / 256);
  if (grid > cap) grid = cap;
  AtenGrid g;
  g.Tt = grid * 256;
  g.n_iter = (int)((numel - 1) / (g.Tt * 4) + 1);
  return g;
}

// z[m][ii]: component ii of subsequence j0 + m at counter c
__device__ __forceinline__ void draw16(uint64_t seed, uint64_t c, uint64_t j0, float (&z)[4][4]) {
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const uint4 r = philox4x32_10(seed, c, j0 + (uint64_t)m);
    const float2 a = box_muller(r.x, r.y), b = box_muller(r.z, r.w);
    z[m][0] = a.x;
    z[m][1] = a.y;
    z[m][2] = b.x;
    z[m][3] = b.y;
  }
}

// z of element idx of a draw at counter ctr0 with ATen's launch of Tt threads: component ii of
// call `it` of subsequence j
__device__ __forceinline__ float normal_at(uint64_t seed, uint64_t ctr0, long long idx, long long Tt) {
  const long long it = idx / (4 * Tt);
  const long long rem = idx - it * 4 * Tt;
  const int ii = (int)(rem / Tt);
  const long long j = rem - (long long)ii * Tt;
  const uint4 r = philox4x32_10(seed, ctr0 + (uint64_t)it, (uint64_t)j);
  const float2 bm = ii < 2 ? box_muller(r.x, r.y) : box_muller(r.z, r.w);
  return (ii & 1) ? bm.y : bm.x;
}

// The element loop shared by the kernels below.  MODE_RNG: z comes from Philox (ATen mapping);
// otherwise from `noise` (may be null when F ignores z).  F(e, z) handles ONE element; the
// loop hands it four consecutive elements at a time, so the compiler keeps 16-byte accesses where
// F's loads / stores are expressed through the Vec4 helpers.  ctr_skip: Philox counters skipped
// past the generator offset (a later draw of the same size: its offset increment / 4).
template <bool RNG, class F4, class F1>
__device__ __forceinline__ void element_loop(long long numel, long long Tt, int n_iter,
                                             const uint64_t* rng, const float* noise, F4 f4, F1 f1,
                                             uint64_t ctr_skip = 0) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long j0 = 4 * k;
  if (j0 >= Tt) return;
  uint64_t seed = 0, ctr0 = 0;
  if (RNG) {
    seed = rng[0];
    ctr0 = (rng[1] >> 2) + ctr_skip;
  }
  const bool n_al = (reinterpret_cast<uintptr_t>(noise) & 15) == 0;
  for (int it = 0; it < n_iter; ++it) {
    const long long base = (long long)it * 4 * Tt + j0;
    if (base >= numel) break;
    float z[4][4];
    if (RNG) draw16(seed, ctr0 + (uint64_t)it, (uint64_t)j0, z);
#pragma unroll
    for (int ii = 0; ii < 4; ++ii) {
      const long long e0 = base + (long long)ii * Tt;
      if (e0 >= numel) break;
      float zz[4] = {0.f, 0.f, 0.f, 0.f};
      const bool full = e0 + 3 < numel;
      if (RNG) {
#pragma unroll
        for (int m = 0; m < 4; ++m) zz[m] = z[m][ii];
      } else if (noise != nullptr) {
        if (full && n_al) {
          const float4 v = *reinterpret_cast<const float4*>(noise + e0);
          zz[0] = v.x; zz[1] = v.y; zz[2] = v.z; zz[3] = v.w;
        } else {
#pragma unroll
          for (int m = 0; m < 4; ++m)
            if (e0 + m < numel) zz[m] = noise[e0 + m];
        }
      }
      if (full) {
        f4(e0, zz);
      } else {
#pragma unroll
        for (int m = 0; m < 4; ++m)
          if (e0 + m < numel) f1(e0 + m, zz[m]);
      }
    }
  }
}

__device__ __forceinline__ bool aligned16(const void* p) {
  return (reinterpret_cast<uintptr_t>(p) & 15) == 0;
}
__device__ __forceinline__ void load4(const float* p, bool al, float (&v)[4]) {
  if (al) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m) v[m] = p[m];
  }
}
__device__ __forceinline__ void store4(float* p, bool al, const float (&v)[4]) {
  if (al) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m) p[m] = v[m];
  }
}

template <bool RNG>
__global__ void __launch_bounds__(256)
randn_kernel(float* out, long long numel, long long Tt, int n_iter, const uint64_t* rng) {
  const bool al = aligned16(out);
  element_loop<RNG>(numel, Tt, n_iter, rng, nullptr,
      [&](long long e0, const float (&z)[4]) { store4(out + e0, al, z); },
      [&](long long e, float z) { out[e] = z; });
}

// The forward-noising coefficients (a, b) of out = a * x + b * z at per-sample timestep t:
//   q_sample:     x_0 -> x_t,      (sqrt_ac[t], sqrt_1mac[t])
//   RePaint undo: x_l -> x_{l+1},  (sqrt(alphas[l + 1]), sqrt(betas[l + 1])), l >= -1
struct QSampleCoef {
  const float *sqrt_ac, *sqrt_1mac;
  __device__ __forceinline__ float2 operator()(int64_t t) const {
    return make_float2(__ldg(sqrt_ac + t), __ldg(sqrt_1mac + t));
  }
};
struct UndoCoef {
  const float *alphas, *betas;
  __device__ __forceinline__ float2 operator()(int64_t l) const {
    return make_float2(__fsqrt_rn(__ldg(alphas + l + 1)), __fsqrt_rn(__ldg(betas + l + 1)));
  }
};

// out = a * x0 + b * z with (a, b) = coef(t[n]) ; z optionally written out (the loss needs it).
// x0 / out may alias (no __restrict__).
template <class Coef, bool RNG>
__global__ void __launch_bounds__(256)
q_sample_kernel(const Coef coef, const float* x0, const float* noise, const uint64_t* rng,
                uint64_t ctr_skip, const int64_t* t, float* out, float* noise_out,
                long long per_sample, long long numel, long long Tt, int n_iter) {
  const bool al = aligned16(x0) && aligned16(out) && (noise_out == nullptr || aligned16(noise_out));
  auto one = [&](long long e, float z) {
    const float2 c = coef(t[e / per_sample]);
    out[e] = __fadd_rn(__fmul_rn(c.x, x0[e]), __fmul_rn(c.y, z));
    if (noise_out != nullptr) noise_out[e] = z;
  };
  element_loop<RNG>(numel, Tt, n_iter, rng, noise,
      [&](long long e0, const float (&z)[4]) {
        const long long n = e0 / per_sample;
        if ((e0 + 3) / per_sample != n) {
#pragma unroll
          for (int m = 0; m < 4; ++m) one(e0 + m, z[m]);
          return;
        }
        const float2 c = coef(t[n]);
        float xv[4], o[4];
        load4(x0 + e0, al, xv);
#pragma unroll
        for (int m = 0; m < 4; ++m) o[m] = __fadd_rn(__fmul_rn(c.x, xv[m]), __fmul_rn(c.y, z[m]));
        store4(out + e0, al, o);
        if (noise_out != nullptr) store4(noise_out + e0, al, z);
      },
      one, ctr_skip);
}

// ------------------------------------------------------------------------------------------
// The reverse-step updates, each defined once and shared by step_kernel and
// tap_gather_step_kernel: coef(n) fetches sample n's coefficients, apply(c, x, eps, z, x0p) returns
// one element's new state.  fp32 in the reference's association order:
//   DDPM:  out = c1*(x - q*eps) + w*z,  q = beta[t]/sqrt_1mac[t], c1 = sqrt_recip_alphas[t],
//          w = (t != 0)*sqrt(post_var[t])
//   DDIM (eta = 0):  x0 = (x - sqrt(1-a_t)*eps)/max(sqrt(a_t), 1e-8),
//          out = sqrt(a_p)*x0 + sqrt(1-a_p)*eps,  a_t / a_p = alphas_cumprod[t] / [t_prev]
//   DPM-Solver++(2M), row k = (s, r, A, B, C) of schedules.dpmpp_2m_table:
//          x0 = (x - s*eps)*r,  out = (A*x + B*x0) + C*(x0 - x0_prev),  x0_prev <- x0
// kNoise: the update takes z.  kX0Prev: it keeps the x0_prev state (x0p: that state in, this
// step's x0 out); the C term is skipped when C == 0, and the callers then do not read x0_prev at
// all (second(c) false: it may hold anything there, NaN included).  kPerSample: the coefficients
// depend on the sample (DPM-Solver++'s row does not, and step_kernel fetches it once).
// ------------------------------------------------------------------------------------------
struct DdpmUpdate {
  static constexpr bool kNoise = true, kX0Prev = false, kPerSample = true;
  struct Coef { float q, c1, w; };
  const int64_t* t;
  const float *betas, *sqrt_1mac, *sqrt_recip_alphas, *post_var;
  __device__ __forceinline__ Coef coef(long long n) const {
    const int64_t ts = t[n];
    return Coef{__fdiv_rn(__ldg(betas + ts), __ldg(sqrt_1mac + ts)), __ldg(sqrt_recip_alphas + ts),
                __fmul_rn(ts != 0 ? 1.0f : 0.0f, __fsqrt_rn(__ldg(post_var + ts)))};
  }
  __device__ __forceinline__ static float apply(const Coef& c, float x, float e, float z, float&) {
    return __fadd_rn(__fmul_rn(c.c1, __fsub_rn(x, __fmul_rn(c.q, e))), __fmul_rn(c.w, z));
  }
};

struct DdimUpdate {
  static constexpr bool kNoise = false, kX0Prev = false, kPerSample = true;
  struct Coef { float s1m_t, denom, sqrt_a_p, s1m_p; };
  const int64_t *t, *t_prev;
  const float* alphas_cumprod;
  __device__ __forceinline__ Coef coef(long long n) const {
    const float a_t = __ldg(alphas_cumprod + t[n]);
    const float a_p = __ldg(alphas_cumprod + t_prev[n]);
    return Coef{__fsqrt_rn(__fsub_rn(1.0f, a_t)), fmaxf(__fsqrt_rn(a_t), 1e-8f), __fsqrt_rn(a_p),
                __fsqrt_rn(__fsub_rn(1.0f, a_p))};
  }
  __device__ __forceinline__ static float apply(const Coef& c, float x, float e, float, float&) {
    const float x0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(c.s1m_t, e)), c.denom);
    return __fadd_rn(__fmul_rn(c.sqrt_a_p, x0), __fmul_rn(c.s1m_p, e));
  }
};

struct DpmppUpdate {
  static constexpr bool kNoise = false, kX0Prev = true, kPerSample = false;
  struct Coef { float s, r, A, B, C; };
  const float* table;   // [rows][5]
  const int64_t* k;     // device row index; null: row 0
  __device__ __forceinline__ Coef coef(long long) const {
    const float* c = table + 5 * (k != nullptr ? *k : 0);
    return Coef{c[0], c[1], c[2], c[3], c[4]};
  }
  __device__ __forceinline__ static bool second(const Coef& c) { return c.C != 0.f; }
  __device__ __forceinline__ static float apply(const Coef& c, float x, float e, float, float& x0p) {
    const float x0 = __fmul_rn(__fsub_rn(x, __fmul_rn(c.s, e)), c.r);
    const float o = __fadd_rn(__fmul_rn(c.A, x), __fmul_rn(c.B, x0));
    const float out = second(c) ? __fadd_rn(o, __fmul_rn(c.C, __fsub_rn(x0, x0p))) : o;
    x0p = x0;
    return out;
  }
};

// eps of NC[D]HW element (sample n, in-sample index j): fp32 in x's layout (ldc = 0) or the bf16
// channels-last UNet output [n][spatial][ldc]
__device__ __forceinline__ float load_eps(const void* eps, int ldc, long long spatial,
                                          long long per_sample, long long n, long long j) {
  if (ldc == 0) return reinterpret_cast<const float*>(eps)[n * per_sample + j];
  const long long c = j / spatial;
  const long long s = j - c * spatial;
  return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(eps)[(n * spatial + s) * ldc + c]);
}
// the same for elements j .. j + 3, which lie in one channel; al: the fp32 eps is 16-byte aligned
__device__ __forceinline__ void load_eps4(const void* eps, int ldc, long long spatial,
                                          long long per_sample, long long n, long long j, bool al,
                                          float (&v)[4]) {
  if (ldc == 0) {
    load4(reinterpret_cast<const float*>(eps) + n * per_sample + j, al, v);
    return;
  }
  const long long c = j / spatial;
  const long long s = j - c * spatial;
  const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(eps) + (n * spatial + s) * ldc + c;
#pragma unroll
  for (int m = 0; m < 4; ++m) v[m] = __bfloat162float(p[(long long)m * ldc]);
}

// One reverse step of update U over the fp32 NC[D]HW state; x / out may alias (the sampler updates
// its state in place).  z: Philox (RNG), else `noise`, null for updates without z; x0_prev: the
// kX0Prev state in x's layout, null otherwise.
template <class U, bool RNG>
__global__ void __launch_bounds__(256)
step_kernel(const U u, const float* x, const void* eps, int ldc, int channels, const float* noise,
            const uint64_t* rng, float* x0_prev, float* out, long long per_sample, long long numel,
            long long Tt, int n_iter) {
  const long long spatial = per_sample / (channels > 0 ? channels : 1);
  const bool al = aligned16(x) && aligned16(out) && aligned16(x0_prev);
  const bool eps_al = ldc == 0 && aligned16(eps);
  const typename U::Coef c_all = U::kPerSample ? typename U::Coef{} : u.coef(0);   // same for all n
  auto coef = [&](long long n) { return U::kPerSample ? u.coef(n) : c_all; };
  auto one = [&](long long e, float z) {
    const long long n = e / per_sample;
    const float ev = load_eps(eps, ldc, spatial, per_sample, n, e - n * per_sample);
    const typename U::Coef c = coef(n);
    float p = 0.f;
    if constexpr (U::kX0Prev) {
      if (U::second(c)) p = x0_prev[e];
    }
    out[e] = U::apply(c, x[e], ev, z, p);
    if constexpr (U::kX0Prev) x0_prev[e] = p;
  };
  element_loop<RNG>(numel, Tt, n_iter, rng, noise,
      [&](long long e0, const float (&z)[4]) {
        const long long n = e0 / per_sample;
        const long long j = e0 - n * per_sample;
        // four elements inside one sample and, for the channels-last eps, inside one channel
        if (j + 3 >= per_sample || (ldc != 0 && (j % spatial) + 3 >= spatial)) {
#pragma unroll
          for (int m = 0; m < 4; ++m) one(e0 + m, z[m]);
          return;
        }
        const typename U::Coef c = coef(n);
        float xv[4], ev[4], pv[4] = {0.f, 0.f, 0.f, 0.f}, o[4];
        load4(x + e0, al, xv);
        if constexpr (U::kX0Prev) {
          if (U::second(c)) load4(x0_prev + e0, al, pv);
        }
        load_eps4(eps, ldc, spatial, per_sample, n, j, eps_al, ev);
#pragma unroll
        for (int m = 0; m < 4; ++m) o[m] = U::apply(c, xv[m], ev[m], z[m], pv[m]);
        store4(out + e0, al, o);
        if constexpr (U::kX0Prev) store4(x0_prev + e0, al, pv);
      },
      one);
}

// k += 1, then t[b] = ts[min(k, rows - 1)] for b < n.  One block: every thread reads the old k
// before thread 0 writes the new one, for any n.
__global__ void __launch_bounds__(256)
step_table_advance_kernel(int64_t* t, int n, int64_t* k, const int64_t* ts, int rows) {
  const int64_t kn = *k + 1;
  __syncthreads();
  if (threadIdx.x == 0) *k = kn;
  const int64_t v = ts[kn < rows ? kn : rows - 1];
  for (int b = threadIdx.x; b < n; b += blockDim.x) t[b] = v;
}

// Inpainting by replacement, in place: x <- where(mask, x, kn) with, per sample, tau = t + t_delta
// and kn = known (tau < 0) or sqrt_ac[tau]*known + sqrt_1mac[tau]*z (q_sample_kernel's operations).
// Select, never blend: values of known where mask != 0 and of x where mask == 0 never reach the
// output, NaN included (the 16-byte path still loads all four of both); a four-element group with
// every mask byte set is not touched.
template <bool RNG>
__global__ void __launch_bounds__(256)
inpaint_merge_kernel(float* x, const float* known, const uint8_t* mask, const float* noise,
                     const uint64_t* rng, uint64_t ctr_skip, const int64_t* t, long long t_delta,
                     const float* sqrt_ac, const float* sqrt_1mac, long long per_sample,
                     long long numel, long long Tt, int n_iter) {
  const bool al = aligned16(x) && aligned16(known) && (reinterpret_cast<uintptr_t>(mask) & 3) == 0;
  auto kn = [&](long long tau, float k0, float z) {
    return tau < 0 ? k0 : __fadd_rn(__fmul_rn(__ldg(sqrt_ac + tau), k0), __fmul_rn(__ldg(sqrt_1mac + tau), z));
  };
  auto one = [&](long long e, float z) {
    if (mask[e] != 0) return;
    x[e] = kn(t[e / per_sample] + t_delta, known[e], z);
  };
  element_loop<RNG>(numel, Tt, n_iter, rng, noise,
      [&](long long e0, const float (&z)[4]) {
        const long long n = e0 / per_sample;
        if (!al || (e0 + 3) / per_sample != n) {
#pragma unroll
          for (int m = 0; m < 4; ++m) one(e0 + m, z[m]);
          return;
        }
        const uchar4 mk = *reinterpret_cast<const uchar4*>(mask + e0);
        const bool keep[4] = {mk.x != 0, mk.y != 0, mk.z != 0, mk.w != 0};
        if (keep[0] && keep[1] && keep[2] && keep[3]) return;
        const long long tau = t[n] + t_delta;
        float xv[4], kv[4];
        load4(x + e0, true, xv);
        load4(known + e0, true, kv);
#pragma unroll
        for (int m = 0; m < 4; ++m) xv[m] = keep[m] ? xv[m] : kn(tau, kv[m], z[m]);
        store4(x + e0, true, xv);
      },
      one, ctr_skip);
}

// ------------------------------------------------------------------------------------------
// Thin output convolution finished INSIDE the reverse step.  The k^d convolution with 1..4 output
// channels (out_conv) is computed as one GEMM over all taps, Y[q][tap * cout + co] = W[tap][co] . a[q]
// (the activation is read once); this kernel sums the shifted taps -- eps[q][co] = bias[co] +
// sum_tap Y[q + off(tap)][tap][co], in the same order and with the same bf16 rounding of the result
// as mri_tap_gather -- and applies the DDPM (noise drawn in-kernel, ATen mapping), DDIM or
// DPM-Solver++(2M) update to the fp32 NC[D]HW sampler state in place, so the predicted noise never
// goes to HBM.
// One CTA = a tile of (TD x TH x TW) output positions; the Y rows of the tile plus a one-voxel halo
// are staged in shared memory (odd word pitch: conflict-free), one thread per output position.
// ------------------------------------------------------------------------------------------
struct FusedStepArgs {
  const __nv_bfloat16* y;
  const float* bias;
  float* x;
  __nv_bfloat16* eps_out;   // optional bf16 [positions][ldo]
  const uint64_t* rng;      // DDPM
  float* x0_prev;           // DPM-Solver++
  DdpmUpdate ddpm;
  DdimUpdate ddim;
  DpmppUpdate dpmpp;
  int samples, D, H, W, ndim, cout, ldy, ldo, mode;  // 0: DDPM, 1: DDIM, 2: eps only, 3: DPM-Solver++
  int TD, TH, TW, pitch_w;  // tile and shared-memory row pitch in 32-bit words
  long long Tt;             // ATen launch geometry of a randn over the whole state
};

// update U of the cout state elements of one output position (channel co at idx0 + co * spatial,
// bf16-rounded eps e[co]); every load is issued before the first draw, whose latency it overlaps
template <class U>
__device__ __forceinline__ void fused_update(const U& u, const FusedStepArgs& a, int n, long long idx0,
                                             long long spatial, const float (&e)[4]) {
  const typename U::Coef c = u.coef(n);
  float xv[4], p[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int co = 0; co < 4; ++co) {
    if (co >= a.cout) break;
    xv[co] = a.x[idx0 + co * spatial];
    if constexpr (U::kX0Prev) {
      if (U::second(c)) p[co] = a.x0_prev[idx0 + co * spatial];
    }
  }
  uint64_t seed = 0, ctr0 = 0;
  if constexpr (U::kNoise) {
    seed = a.rng[0];
    ctr0 = a.rng[1] >> 2;
  }
#pragma unroll
  for (int co = 0; co < 4; ++co) {
    if (co >= a.cout) break;
    const long long idx = idx0 + (long long)co * spatial;
    const float z = U::kNoise ? normal_at(seed, ctr0, idx, a.Tt) : 0.f;
    a.x[idx] = U::apply(c, xv[co], e[co], z, p[co]);
    if constexpr (U::kX0Prev) a.x0_prev[idx] = p[co];
  }
}

template <int CH>   // 16-byte chunks per Y row that hold the tap products (0: run-time value)
__global__ void __launch_bounds__(256)
tap_gather_step_kernel(const FusedStepArgs a) {
  extern __shared__ uint32_t ysm[];
  const int hd = a.ndim == 3 ? 1 : 0;             // halo along depth only for 3-D filters
  const int RD = a.TD + 2 * hd, RH = a.TH + 2, RW = a.TW + 2;
  const int rows = RD * RH * RW;
  const int taps = a.ndim == 3 ? 27 : 9;
  const int row_elems = taps * a.cout;            // bf16 per Y row that matter
  const int row_words = (row_elems + 1) >> 1;
  const int chunks = CH > 0 ? CH : (row_words + 3) >> 2;
  // tile origin
  const int tiles_w = (a.W + a.TW - 1) / a.TW, tiles_h = (a.H + a.TH - 1) / a.TH;
  const int tiles_d = (a.D + a.TD - 1) / a.TD;
  int tix = (int)blockIdx.x;
  const int tw0 = (tix % tiles_w) * a.TW;
  tix /= tiles_w;
  const int th0 = (tix % tiles_h) * a.TH;
  tix /= tiles_h;
  const int td0 = (tix % tiles_d) * a.TD;
  const int n = tix / tiles_d;
  const long long spatial = (long long)a.D * a.H * a.W;
  const uint4* yn = reinterpret_cast<const uint4*>(a.y + (size_t)n * spatial * a.ldy);
  const int ldq = a.ldy >> 3;                     // Y row pitch in 16-byte units (ldy % 8 == 0)

  // ---- stage the halo tile -----------------------------------------------------------------------
  // (1) per halo row: its offset in Y (16-byte units) or -1 outside the tensor
  int* row_off = reinterpret_cast<int*>(ysm + (size_t)rows * a.pitch_w);
  for (int r = threadIdx.x; r < rows; r += 256) {
    int rr = r;
    const int w = tw0 + rr % RW - 1;
    rr /= RW;
    const int h = th0 + rr % RH - 1;
    const int d = td0 + rr / RH - hd;
    const bool ok = (unsigned)w < (unsigned)a.W && (unsigned)h < (unsigned)a.H && (unsigned)d < (unsigned)a.D;
    row_off[r] = ok ? (int)((((long long)d * a.H + h) * a.W + w) * ldq) : -1;
  }
  __syncthreads();
  // (2) 16-byte loads, four in flight per thread, scattered into rows of odd word pitch
  const int total = rows * chunks;
  for (int base = 0; base < total; base += 256 * 4) {
    uint4 v[4];
    int dst[4], jw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + u * 256 + (int)threadIdx.x;
      v[u] = make_uint4(0u, 0u, 0u, 0u);
      dst[u] = -1;
      jw[u] = 0;
      if (i < total) {
        const int r = i / chunks;
        const int j = i - r * chunks;
        const int off = row_off[r];
        if (off >= 0) v[u] = __ldg(yn + off + j);
        dst[u] = r * a.pitch_w + 4 * j;
        jw[u] = 4 * j;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (dst[u] >= 0) {
        const uint32_t w4[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (jw[u] + k < row_words) ysm[dst[u] + k] = w4[k];
      }
    }
  }
  __syncthreads();

  // ---- one output position per thread -------------------------------------------------------------
  int q = threadIdx.x;
  const int lw = q % a.TW;
  q /= a.TW;
  const int lh = q % a.TH;
  const int ld_ = q / a.TH;
  const int w0 = tw0 + lw, h0 = th0 + lh, d0 = td0 + ld_;
  if (ld_ >= a.TD || w0 >= a.W || h0 >= a.H || d0 >= a.D) return;
  float acc[4];
#pragma unroll
  for (int co = 0; co < 4; ++co) acc[co] = (co < a.cout && a.bias != nullptr) ? __ldg(a.bias + co) : 0.f;
  const __nv_bfloat16* ys = reinterpret_cast<const __nv_bfloat16*>(ysm);
  int tap = 0;
  const int kd_n = a.ndim == 3 ? 3 : 1;
  for (int kd = 0; kd < kd_n; ++kd)
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw, ++tap) {
        const int r = ((ld_ + kd) * RH + lh + kh) * RW + lw + kw;
        const __nv_bfloat16* row = ys + (size_t)r * a.pitch_w * 2 + tap * a.cout;
#pragma unroll
        for (int co = 0; co < 4; ++co)
          if (co < a.cout) acc[co] += __bfloat162float(row[co]);   // halo rows outside the tensor are 0
      }
  const long long s = ((long long)d0 * a.H + h0) * a.W + w0;
  float e[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int co = 0; co < 4; ++co) {
    if (co >= a.cout) break;
    const __nv_bfloat16 eb = __float2bfloat16_rn(acc[co]);
    if (a.eps_out != nullptr) a.eps_out[((size_t)n * spatial + s) * a.ldo + co] = eb;
    e[co] = __bfloat162float(eb);
  }
  const long long idx0 = (long long)n * a.cout * spatial + s;   // NC[D]HW element of channel 0
  if (a.mode == 0) fused_update(a.ddpm, a, n, idx0, spatial, e);
  else if (a.mode == 1) fused_update(a.ddim, a, n, idx0, spatial, e);
  else if (a.mode == 3) fused_update(a.dpmpp, a, n, idx0, spatial, e);
}

// one thread: t -= 1 for every sample (and t_prev), generator offset += rng_inc -- the bookkeeping
// between two replays of the captured reverse step
__global__ void step_advance_kernel(int64_t* t, int64_t* t_prev, int n, int64_t delta,
                                    uint64_t* rng, uint64_t rng_inc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    t[i] += delta;
    if (t_prev != nullptr) {  // strided DDIM: the last step lands on t_prev = 0
      const int64_t v = t_prev[i] + delta;
      t_prev[i] = v < 0 ? 0 : v;
    }
  }
  if (i == 0 && rng != nullptr) rng[1] += rng_inc;
}

// per-sample sum of squared differences; grid (blocks, samples)
__global__ void __launch_bounds__(256)
sqdiff_kernel(const float* __restrict__ pred, const float* __restrict__ noise,
              float* __restrict__ acc, int64_t per_sample) {
  const int sample = blockIdx.y;
  const size_t base = (size_t)sample * per_sample;
  float s = 0.f;
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < per_sample;
       j += (int64_t)gridDim.x * blockDim.x) {
    const float d = pred[base + j] - noise[base + j];
    s = fmaf(d, d, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ float part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += part[i];
    atomicAdd(acc + sample, tot);
  }
}

__global__ void loss_finalize_kernel(float* __restrict__ per_sample_acc, const int64_t* __restrict__ t,
                                     const float* __restrict__ snr, float gamma,
                                     float* __restrict__ loss_out, int samples, int64_t per_sample) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float tot = 0.f;
  for (int b = 0; b < samples; ++b) {
    const float mse = per_sample_acc[b] / (float)per_sample;
    float w = 1.0f;
    if (gamma > 0.f) {
      const float s = snr[t[b]];
      w = fminf(s, gamma) / s;
    }
    per_sample_acc[b] = mse;
    tot += w * mse;
  }
  loss_out[0] = tot / (float)samples;
}

__global__ void add_i64_kernel(int64_t* t, int n, int64_t delta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) t[i] += delta;
}

__global__ void rng_seed_kernel(uint64_t* rng, uint64_t seed, uint64_t offset) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    rng[0] = seed;
    rng[1] = offset;
  }
}

static inline dim3 ew_grid(int samples, int64_t per_sample) {
  int64_t bx = (per_sample + 255) / 256;
  int64_t cap = (148 * 8 + samples - 1) / samples;
  if (cap < 1) cap = 1;
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  return dim3((unsigned)bx, (unsigned)samples);
}

}  // namespace mri

using namespace mri;

static inline unsigned my_blocks(const AtenGrid& g) { return (unsigned)((g.Tt / 4 + 255) / 256); }

static int check_rng_args(const char* who, long long numel) {
  if (numel < 1) return set_error(-2, who);
  return device_props();
}

extern "C" int mri_randn_offset_increment(int64_t numel, uint64_t* increment_out) {
  if (numel < 1 || increment_out == nullptr)
    return set_error(-2, "mri_randn_offset_increment: empty tensor / null output");
  int rc = device_props();
  if (rc) return rc;
  *increment_out = 4ull * (uint64_t)aten_grid(numel).n_iter;
  return 0;
}

extern "C" int mri_randn(float* out, int64_t numel, const uint64_t* rng, void* stream) {
  int rc = check_rng_args("mri_randn: empty tensor", numel);
  if (rc) return rc;
  if (rng == nullptr) return set_error(-2, "mri_randn: null generator state");
  const AtenGrid g = aten_grid(numel);
  randn_kernel<true><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(out, numel, g.Tt, g.n_iter, rng);
  return check_launch("randn_kernel");
}

// q_sample_kernel<Coef> over samples * per_sample elements; z from Philox (rng_skip past the
// generator offset) when rng is set, else from `noise`
template <class Coef>
static int noise_launch(const char* who, const Coef& coef, const float* x0, const float* noise,
                        const uint64_t* rng, uint64_t rng_skip, const int64_t* t, float* out,
                        float* noise_out, int samples, int64_t per_sample, void* stream) {
  const long long numel = (long long)samples * per_sample;
  int rc = device_props();
  if (rc) return rc;
  const AtenGrid g = aten_grid(numel);
  if (rng != nullptr)
    q_sample_kernel<Coef, true><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(
        coef, x0, nullptr, rng, rng_skip / 4, t, out, noise_out, per_sample, numel, g.Tt, g.n_iter);
  else
    q_sample_kernel<Coef, false><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(
        coef, x0, noise, nullptr, 0, t, out, noise_out, per_sample, numel, g.Tt, g.n_iter);
  return check_launch(who);
}

static int q_sample_impl(const float* x0, const float* noise, const uint64_t* rng, const int64_t* t,
                         const float* sqrt_ac, const float* sqrt_1mac, float* out, float* noise_out,
                         int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_q_sample: empty input");
  return noise_launch("q_sample_kernel", QSampleCoef{sqrt_ac, sqrt_1mac}, x0, noise, rng, 0, t, out,
                      noise_out, samples, per_sample, stream);
}

extern "C" int mri_q_sample(const float* x0, const float* noise, const int64_t* t,
                            const float* sqrt_ac, const float* sqrt_1mac, float* out, int samples,
                            int64_t per_sample, void* stream) {
  if (noise == nullptr) return set_error(-2, "mri_q_sample: null noise");
  return q_sample_impl(x0, noise, nullptr, t, sqrt_ac, sqrt_1mac, out, nullptr, samples, per_sample,
                       stream);
}

extern "C" int mri_q_sample_rng(const float* x0, const uint64_t* rng, const int64_t* t,
                                const float* sqrt_ac, const float* sqrt_1mac, float* out,
                                float* noise_out, int samples, int64_t per_sample, void* stream) {
  if (rng == nullptr) return set_error(-2, "mri_q_sample_rng: null generator state");
  return q_sample_impl(x0, nullptr, rng, t, sqrt_ac, sqrt_1mac, out, noise_out, samples, per_sample,
                       stream);
}

// step_kernel<U> over samples * per_sample elements; z from Philox when rng is set (only DDPM
// takes z, so only DdpmUpdate is instantiated with RNG)
template <class U>
static int step_launch(const char* who, const U& u, const float* x, const void* eps, int ldc,
                       int channels, const float* noise, const uint64_t* rng, float* x0_prev,
                       float* out, int samples, int64_t per_sample, void* stream) {
  const long long numel = (long long)samples * per_sample;
  int rc = device_props();
  if (rc) return rc;
  const AtenGrid g = aten_grid(numel);
  if (rng != nullptr)
    step_kernel<U, U::kNoise><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(
        u, x, eps, ldc, channels, nullptr, rng, x0_prev, out, per_sample, numel, g.Tt, g.n_iter);
  else
    step_kernel<U, false><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(
        u, x, eps, ldc, channels, noise, nullptr, x0_prev, out, per_sample, numel, g.Tt, g.n_iter);
  return check_launch(who);
}

static int ddpm_step_impl(const float* x, const void* eps, int ldc, int channels, const float* noise,
                          const uint64_t* rng, const int64_t* t, const float* betas,
                          const float* sqrt_1mac, const float* sqrt_recip_alphas,
                          const float* post_var, float* out, int samples, int64_t per_sample,
                          void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_ddpm_step: empty input");
  if (ldc != 0 && (channels < 1 || per_sample % channels != 0))
    return set_error(-2, "mri_ddpm_step: per_sample must be channels * spatial");
  return step_launch("mri_ddpm_step", DdpmUpdate{t, betas, sqrt_1mac, sqrt_recip_alphas, post_var},
                     x, eps, ldc, channels, noise, rng, nullptr, out, samples, per_sample, stream);
}

extern "C" int mri_ddpm_step(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                             const float* noise, const int64_t* t, const float* betas,
                             const float* sqrt_1mac, const float* sqrt_recip_alphas,
                             const float* post_var, float* out, int samples, int64_t per_sample,
                             void* stream) {
  if (noise == nullptr) return set_error(-2, "mri_ddpm_step: null noise");
  return ddpm_step_impl(x, eps, eps_nhwc_ldc, channels, noise, nullptr, t, betas, sqrt_1mac,
                        sqrt_recip_alphas, post_var, out, samples, per_sample, stream);
}

extern "C" int mri_ddpm_step_rng(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                                 const uint64_t* rng, const int64_t* t, const float* betas,
                                 const float* sqrt_1mac, const float* sqrt_recip_alphas,
                                 const float* post_var, float* out, int samples, int64_t per_sample,
                                 void* stream) {
  if (rng == nullptr) return set_error(-2, "mri_ddpm_step_rng: null generator state");
  return ddpm_step_impl(x, eps, eps_nhwc_ldc, channels, nullptr, rng, t, betas, sqrt_1mac,
                        sqrt_recip_alphas, post_var, out, samples, per_sample, stream);
}

extern "C" int mri_ddim_step(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                             const int64_t* t, const int64_t* t_prev, const float* alphas_cumprod,
                             float* out, int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_ddim_step: empty input");
  if (eps_nhwc_ldc != 0 && (channels < 1 || per_sample % channels != 0))
    return set_error(-2, "mri_ddim_step: per_sample must be channels * spatial");
  return step_launch("mri_ddim_step", DdimUpdate{t, t_prev, alphas_cumprod}, x, eps, eps_nhwc_ldc,
                     channels, nullptr, nullptr, nullptr, out, samples, per_sample, stream);
}

extern "C" int mri_dpmpp_step(const float* x, const void* eps, int eps_nhwc_ldc, int channels,
                              float* x0_prev, const float* coef, const int64_t* k, float* out,
                              int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_dpmpp_step: empty input");
  if (x == nullptr || eps == nullptr || x0_prev == nullptr || coef == nullptr || out == nullptr)
    return set_error(-2, "mri_dpmpp_step: null x / eps / x0_prev / coef / out");
  if (eps_nhwc_ldc != 0 && (channels < 1 || per_sample % channels != 0 || eps_nhwc_ldc < channels))
    return set_error(-2, "mri_dpmpp_step: per_sample must be channels * spatial, ldc >= channels");
  return step_launch("mri_dpmpp_step", DpmppUpdate{coef, k}, x, eps, eps_nhwc_ldc, channels, nullptr,
                     nullptr, x0_prev, out, samples, per_sample, stream);
}

extern "C" int mri_step_table_advance(int64_t* t, int n, int64_t* k, const int64_t* ts, int rows,
                                      void* stream) {
  if (n < 1) return 0;
  if (t == nullptr || k == nullptr || ts == nullptr || rows < 1)
    return set_error(-2, "mri_step_table_advance: null t / k / ts or rows < 1");
  step_table_advance_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(t, n, k, ts, rows);
  return check_launch("step_table_advance_kernel");
}

extern "C" int mri_inpaint_merge(float* x, const float* known, const uint8_t* mask,
                                 const float* noise, const uint64_t* rng, uint64_t rng_skip,
                                 const int64_t* t, int64_t t_delta, const float* sqrt_ac,
                                 const float* sqrt_1mac, int samples, int64_t per_sample,
                                 void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_inpaint_merge: empty input");
  if (x == nullptr || known == nullptr || mask == nullptr || t == nullptr || sqrt_ac == nullptr ||
      sqrt_1mac == nullptr)
    return set_error(-2, "mri_inpaint_merge: null x / known / mask / t / schedule table");
  if ((noise == nullptr) == (rng == nullptr))
    return set_error(-2, "mri_inpaint_merge: exactly one of noise / rng");
  if (rng_skip % 4 != 0) return set_error(-2, "mri_inpaint_merge: rng_skip must be a multiple of 4");
  const long long numel = (long long)samples * per_sample;
  int rc = device_props();
  if (rc) return rc;
  const AtenGrid g = aten_grid(numel);
  if (rng != nullptr)
    inpaint_merge_kernel<true><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(
        x, known, mask, nullptr, rng, rng_skip / 4, t, t_delta, sqrt_ac, sqrt_1mac, per_sample, numel,
        g.Tt, g.n_iter);
  else
    inpaint_merge_kernel<false><<<my_blocks(g), 256, 0, (cudaStream_t)stream>>>(
        x, known, mask, noise, nullptr, 0, t, t_delta, sqrt_ac, sqrt_1mac, per_sample, numel, g.Tt,
        g.n_iter);
  return check_launch("inpaint_merge_kernel");
}

extern "C" int mri_repaint_undo(float* x, const float* noise, const uint64_t* rng, uint64_t rng_skip,
                                const int64_t* t, const float* alphas, const float* betas,
                                int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_repaint_undo: empty input");
  if (x == nullptr || t == nullptr || alphas == nullptr || betas == nullptr)
    return set_error(-2, "mri_repaint_undo: null x / t / schedule table");
  if ((noise == nullptr) == (rng == nullptr))
    return set_error(-2, "mri_repaint_undo: exactly one of noise / rng");
  if (rng_skip % 4 != 0) return set_error(-2, "mri_repaint_undo: rng_skip must be a multiple of 4");
  return noise_launch("q_sample_kernel<UndoCoef>", UndoCoef{alphas, betas}, x, noise, rng, rng_skip, t, x,
                      nullptr, samples, per_sample, stream);
}

extern "C" int mri_rng_seed(uint64_t* rng, uint64_t seed, uint64_t offset, void* stream) {
  if (rng == nullptr) return set_error(-2, "mri_rng_seed: null state");
  if (offset % 4 != 0) return set_error(-2, "mri_rng_seed: philox offset must be a multiple of 4");
  rng_seed_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rng, seed, offset);
  return check_launch("rng_seed_kernel");
}

extern "C" int mri_step_advance(int64_t* t, int64_t* t_prev, int n, int64_t delta, uint64_t* rng,
                                uint64_t rng_increment, void* stream) {
  if (n < 1) return 0;
  step_advance_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(t, t_prev, n, delta, rng,
                                                                        rng_increment);
  return check_launch("step_advance_kernel");
}

extern "C" int mri_minsnr_loss(const float* pred, const float* noise, const int64_t* t,
                               const float* snr, float gamma, float* per_sample_out,
                               float* loss_out, int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_minsnr_loss: empty input");
  cudaError_t e = cudaMemsetAsync(per_sample_out, 0, sizeof(float) * samples, (cudaStream_t)stream);
  if (e != cudaSuccess) return set_cuda_error(e, "cudaMemsetAsync(per_sample_out)");
  sqdiff_kernel<<<ew_grid(samples, per_sample), 256, 0, (cudaStream_t)stream>>>(
      pred, noise, per_sample_out, per_sample);
  int rc = check_launch("sqdiff_kernel");
  if (rc) return rc;
  loss_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(per_sample_out, t, snr, gamma, loss_out,
                                                          samples, per_sample);
  return check_launch("loss_finalize_kernel");
}

extern "C" int mri_add_i64(int64_t* t, int n, int64_t delta, void* stream) {
  if (n < 1) return 0;
  add_i64_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(t, n, delta);
  return check_launch("add_i64_kernel");
}

extern "C" int mri_tap_gather_step(const void* y, const float* bias, int samples, int D, int H, int W,
                                   int ndim, int cout, int ldy, float* x, void* eps_out, int ldo,
                                   int mode, const uint64_t* rng, const int64_t* t,
                                   const int64_t* t_prev, const float* betas, const float* sqrt_1mac,
                                   const float* sqrt_recip_alphas, const float* post_var,
                                   const float* alphas_cumprod, float* x0_prev, const float* coef,
                                   const int64_t* k, void* stream) {
  if (ndim != 2 && ndim != 3) return set_error(-2, "mri_tap_gather_step: ndim must be 2 or 3");
  if (cout < 1 || cout > 4) return set_error(-2, "mri_tap_gather_step: 1..4 output channels");
  const int taps = ndim == 3 ? 27 : 9;
  if (ldy % 2 != 0 || taps * cout > ldy) return set_error(-2, "mri_tap_gather_step: bad Y row layout");
  if (samples < 1 || D < 1 || H < 1 || W < 1) return set_error(-2, "mri_tap_gather_step: empty input");
  if (ndim == 2 && D != 1) return set_error(-2, "mri_tap_gather_step: 2-D problems have D = 1");
  if (mode < 0 || mode > 3)
    return set_error(-2, "mri_tap_gather_step: mode 0 (DDPM) / 1 (DDIM) / 2 (eps only) / 3 (DPM-Solver++)");
  if (mode == 3 && (x0_prev == nullptr || coef == nullptr || x == nullptr))
    return set_error(-2, "mri_tap_gather_step: DPM-Solver++ mode needs x, x0_prev and coef");
  if (mode == 0 && (rng == nullptr || t == nullptr || betas == nullptr || sqrt_1mac == nullptr ||
                    sqrt_recip_alphas == nullptr || post_var == nullptr || x == nullptr))
    return set_error(-2, "mri_tap_gather_step: DDPM mode needs x, rng, t and the four schedule tables");
  if (mode == 1 && (t == nullptr || t_prev == nullptr || alphas_cumprod == nullptr || x == nullptr))
    return set_error(-2, "mri_tap_gather_step: DDIM mode needs x, t, t_prev and alphas_cumprod");
  if (mode == 2 && eps_out == nullptr) return set_error(-2, "mri_tap_gather_step: eps-only mode needs eps_out");
  if (eps_out != nullptr && ldo < cout) return set_error(-2, "mri_tap_gather_step: ldo < cout");
  int rc = device_props();
  if (rc) return rc;
  FusedStepArgs a;
  a.y = reinterpret_cast<const __nv_bfloat16*>(y);
  a.bias = bias;
  a.x = x;
  a.eps_out = reinterpret_cast<__nv_bfloat16*>(eps_out);
  a.rng = rng;
  a.x0_prev = x0_prev;
  a.ddpm = DdpmUpdate{t, betas, sqrt_1mac, sqrt_recip_alphas, post_var};
  a.ddim = DdimUpdate{t, t_prev, alphas_cumprod};
  a.dpmpp = DpmppUpdate{coef, k};
  a.samples = samples; a.D = D; a.H = H; a.W = W; a.ndim = ndim; a.cout = cout; a.ldy = ldy; a.ldo = ldo;
  a.mode = mode;
  a.TD = ndim == 3 ? 4 : 1;
  a.TH = ndim == 3 ? 8 : 16;
  a.TW = ndim == 3 ? 8 : 16;
  const int row_words = (taps * cout + 1) / 2;
  a.pitch_w = row_words | 1;                         // odd pitch: consecutive rows hit different banks
  const long long numel = (long long)samples * cout * D * H * W;
  a.Tt = aten_grid(numel).Tt;
  const int rows = (a.TD + (ndim == 3 ? 2 : 0)) * (a.TH + 2) * (a.TW + 2);
  const int smem = rows * a.pitch_w * 4 + rows * 4;   // staged rows + the row-offset table
  if (ldy % 8 != 0) return set_error(-2, "mri_tap_gather_step: ldy must be a multiple of 8");
  if ((long long)D * H * W * (ldy / 8) > 0x7fffffffLL)
    return set_error(-2, "mri_tap_gather_step: sample too large for 32-bit row offsets");
  const long long tiles = (long long)samples * ((D + a.TD - 1) / a.TD) * ((H + a.TH - 1) / a.TH) *
                          ((W + a.TW - 1) / a.TW);
  if (tiles > 0x7fffffffLL) return set_error(-2, "mri_tap_gather_step: too many tiles");
  const int chunks = (row_words + 3) / 4;
  void (*kern)(const FusedStepArgs) = chunks == 11 ? tap_gather_step_kernel<11>
                                      : chunks == 5 ? tap_gather_step_kernel<5>
                                      : chunks == 2 ? tap_gather_step_kernel<2>
                                                    : tap_gather_step_kernel<0>;
  static int configured[4] = {0, 0, 0, 0};   // per instantiation (not re-done inside a graph capture)
  const int slot = chunks == 11 ? 0 : chunks == 5 ? 1 : chunks == 2 ? 2 : 3;
  if (smem > configured[slot]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(tap_gather_step_kernel)");
    configured[slot] = smem;
  }
  kern<<<(unsigned)tiles, 256, smem, (cudaStream_t)stream>>>(a);
  return check_launch("tap_gather_step_kernel");
}
