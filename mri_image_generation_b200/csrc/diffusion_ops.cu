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
// k-space data consistency (mri_kspace_merge): per sample, tau = t[n] + t_delta and
//   x <- x - P(x - s1m[tau] z) + (tau < 0 ? x_zf : sac[tau] x_zf)    (no z term at tau < 0)
// with P u = Re F^-1(M . F u), F the orthonormal 2-D DFT of each (H, W) plane and M the
// Hermitian-symmetric mask.  Because M is Hermitian, M . F u of a real u is Hermitian, so only
// the half spectrum k < Wh = W/2 + 1 is formed.  Three passes over a complex [plane][H][Wh] work
// buffer, each a direct fp32 summation (FMA) against a twiddle table in shared memory with the
// exact index (j k) mod N:
//   A  u = x - s1m z per row, forward row DFT (real -> half spectrum)        kKsRows rows a block
//   B  forward column DFT, times M, inverse column DFT                      kKsCols columns a block
//   C  inverse row DFT (half spectrum -> real), P u / (H W), the update       kKsRows rows a block
// ------------------------------------------------------------------------------------------
constexpr int kKsMaxN = 512;      // H, W limit: pass B keeps two H x kKsCols complex tiles
constexpr int kKsRows = 16;       // rows per block of passes A and C
constexpr int kKsCols = 16;       // columns per block of pass B (128-byte rows of the tile)
constexpr int kKsThreadsA = 128, kKsThreadsB = 256, kKsThreadsC = 256;

struct KspaceArgs {
  float* x;
  const float* zf;
  const uint8_t* mask;
  const float* noise;
  const uint64_t* rng;
  uint64_t ctr_skip;
  const int64_t* t;
  long long t_delta;
  const float* sqrt_ac;
  const float* sqrt_1mac;
  float2* work;
  int channels, H, W, Wh;
  long long Tt;     // ATen's launch for a draw of the whole x (normal_at)
};

// The twiddle table takes an even number of float2 entries, so the arrays after it, read with
// 16-byte loads, stay 16-byte aligned for odd H and W.
__host__ __device__ __forceinline__ int ks_tw_len(int n) { return (n + 1) & ~1; }
static int ks_smem_a(int W) { return ks_tw_len(W) * 8 + W * kKsRows * 4; }
static int ks_smem_b(int H) { return ks_tw_len(H) * 8 + 2 * H * kKsCols * 8 + H * 4; }
static int ks_smem_c(int W) { return ks_tw_len(W) * 8 + (W / 2 + 1) * kKsRows * 8; }

// tw[j] = exp(-2 pi i j / n), j < n: fp64 sincospi, rounded once to fp32
__device__ __forceinline__ void ks_twiddles(float2* tw, int n) {
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    double s, c;
    sincospi(2.0 * j / n, &s, &c);
    tw[j] = make_float2((float)c, (float)-s);
  }
}

// The four DFT sums the 2-D and 3-D passes share, each in one fixed FMA order.
// Bin k of the forward real DFT of kKsRows rows held as u[W][kKsRows].
__device__ __forceinline__ void ks_row_fwd(const float2* tw, const float* u, int W, int k,
                                           float (&re)[kKsRows], float (&im)[kKsRows]) {
#pragma unroll
  for (int r = 0; r < kKsRows; ++r) re[r] = im[r] = 0.f;
  int idx = 0;
  for (int w = 0; w < W; ++w) {
    const float2 c = tw[idx];
    const float4* up = reinterpret_cast<const float4*>(u + w * kKsRows);
#pragma unroll
    for (int q = 0; q < kKsRows / 4; ++q) {
      const float4 v = up[q];
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        re[4 * q + m] = fmaf(vv[m], c.x, re[4 * q + m]);
        im[4 * q + m] = fmaf(vv[m], c.y, im[4 * q + m]);
      }
    }
    idx += k;
    if (idx >= W) idx -= W;
  }
}

// Sample w of Re(inverse DFT) of kKsRows half spectra held as us[Wh][kKsRows] (bins other than 0
// and W/2 already doubled), unscaled.
__device__ __forceinline__ void ks_row_inv(const float2* tw, const float2* us, int W, int Wh, int w,
                                           float (&acc)[kKsRows]) {
#pragma unroll
  for (int r = 0; r < kKsRows; ++r) acc[r] = 0.f;
  int idx = 0;
  for (int k = 0; k < Wh; ++k) {
    const float2 c = tw[idx];          // Re(v exp(+i theta)) = v.x cos - v.y sin = v.x c.x + v.y c.y
    const float4* vp = reinterpret_cast<const float4*>(us + k * kKsRows);
#pragma unroll
    for (int q = 0; q < kKsRows / 2; ++q) {
      const float4 v = vp[q];
      acc[2 * q] = fmaf(v.y, c.y, fmaf(v.x, c.x, acc[2 * q]));
      acc[2 * q + 1] = fmaf(v.w, c.y, fmaf(v.z, c.x, acc[2 * q + 1]));
    }
    idx += w;
    if (idx >= W) idx -= W;
  }
}

// Bin m of the forward DFT of length N of kKsCols complex columns held as U[N][kKsCols]; thread m
// sums over n, so the U loads are warp broadcasts.
__device__ __forceinline__ void ks_col_fwd(const float2* tw, const float2* U, int N, int m,
                                           float (&re)[kKsCols], float (&im)[kKsCols]) {
#pragma unroll
  for (int j = 0; j < kKsCols; ++j) re[j] = im[j] = 0.f;
  int idx = 0;
  for (int h = 0; h < N; ++h) {
    const float2 c = tw[idx];
    const float4* up = reinterpret_cast<const float4*>(U + h * kKsCols);
#pragma unroll
    for (int q = 0; q < kKsCols / 2; ++q) {
      const float4 v = up[q];
      re[2 * q] = fmaf(-v.y, c.y, fmaf(v.x, c.x, re[2 * q]));
      im[2 * q] = fmaf(v.y, c.x, fmaf(v.x, c.y, im[2 * q]));
      re[2 * q + 1] = fmaf(-v.w, c.y, fmaf(v.z, c.x, re[2 * q + 1]));
      im[2 * q + 1] = fmaf(v.w, c.x, fmaf(v.z, c.y, im[2 * q + 1]));
    }
    idx += m;
    if (idx >= N) idx -= N;
  }
}

// Sample h of the inverse DFT (unscaled) of V[N][kKsCols]: exp(+2 pi i h m / N) = conj(tw); rows
// of V with live[m] == 0 add nothing
__device__ __forceinline__ void ks_col_inv(const float2* tw, const float2* V, const int* live, int N,
                                           int h, float (&re)[kKsCols], float (&im)[kKsCols]) {
#pragma unroll
  for (int j = 0; j < kKsCols; ++j) re[j] = im[j] = 0.f;
  int idx = 0;
  for (int m = 0; m < N; ++m) {
    if (live[m]) {
      const float2 c = tw[idx];
      const float4* vp = reinterpret_cast<const float4*>(V + m * kKsCols);
#pragma unroll
      for (int q = 0; q < kKsCols / 2; ++q) {
        const float4 v = vp[q];
        re[2 * q] = fmaf(v.y, c.y, fmaf(v.x, c.x, re[2 * q]));
        im[2 * q] = fmaf(-v.x, c.y, fmaf(v.y, c.x, im[2 * q]));
        re[2 * q + 1] = fmaf(v.w, c.y, fmaf(v.z, c.x, re[2 * q + 1]));
        im[2 * q + 1] = fmaf(-v.z, c.y, fmaf(v.w, c.x, im[2 * q + 1]));
      }
    }
    idx += h;
    if (idx >= N) idx -= N;
  }
}

template <bool RNG>
__global__ void __launch_bounds__(kKsThreadsA) kspace_rows_fwd_kernel(const KspaceArgs a) {
  extern __shared__ float4 ks_smem[];
  float2* tw = reinterpret_cast<float2*>(ks_smem);
  float* u = reinterpret_cast<float*>(tw + ks_tw_len(a.W));    // [W][kKsRows]
  const int nrb = (a.H + kKsRows - 1) / kKsRows;
  const long long plane = blockIdx.x / nrb;
  const int h0 = (int)(blockIdx.x % nrb) * kKsRows;
  const long long tau = a.t[plane / a.channels] + a.t_delta;
  ks_twiddles(tw, a.W);
  uint64_t seed = 0, ctr0 = 0;
  if (RNG) {
    seed = a.rng[0];
    ctr0 = (a.rng[1] >> 2) + a.ctr_skip;
  }
  const float s = tau < 0 ? 0.f : __ldg(a.sqrt_1mac + tau);
  for (int i = threadIdx.x; i < kKsRows * a.W; i += blockDim.x) {
    const int r = i / a.W, w = i - r * a.W;
    float v = 0.f;
    if (h0 + r < a.H) {
      const long long e = (plane * a.H + h0 + r) * a.W + w;
      v = a.x[e];
      if (tau >= 0) v = __fsub_rn(v, __fmul_rn(s, RNG ? normal_at(seed, ctr0, e, a.Tt) : a.noise[e]));
    }
    u[w * kKsRows + r] = v;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < a.Wh; k += blockDim.x) {
    float re[kKsRows], im[kKsRows];
    ks_row_fwd(tw, u, a.W, k, re, im);
#pragma unroll
    for (int r = 0; r < kKsRows; ++r)
      if (h0 + r < a.H) a.work[(plane * a.H + h0 + r) * a.Wh + k] = make_float2(re[r], im[r]);
  }
}

// The column passes over a complex work buffer of half spectra: `line` indexes the 1-D transforms
// of length N, element n of column c of line l at work[(l / inner) * outer + (l % inner) * inner_ld
// + n * ld + c], its mask byte likewise with the m_* strides.
struct KsColGeom {
  float2* work;
  const uint8_t* mask;
  int N, Wh, inner;
  long long outer, inner_ld, ld;
  long long m_outer, m_inner_ld, m_ld;
};

// kKsCols columns of one line a block.  kMode 0: forward DFT; 1: forward DFT, times M, inverse DFT;
// 2: inverse DFT.  In place: the block reads its whole tile before it writes.
template <int kMode>
__global__ void __launch_bounds__(kKsThreadsB) kspace_cols_kernel(const KsColGeom g) {
  extern __shared__ float4 ks_smem[];
  const int N = g.N;
  float2* tw = reinterpret_cast<float2*>(ks_smem);
  float2* U = tw + ks_tw_len(N);       // [N][kKsCols]: the input spectra
  float2* V = U + N * kKsCols;         // [N][kKsCols]: what the inverse reads
  int* live = reinterpret_cast<int*>(V + N * kKsCols);   // row m of V has a measured sample
  const int nct = (g.Wh + kKsCols - 1) / kKsCols;
  const long long line = blockIdx.x / nct;
  const int c0 = (int)(blockIdx.x % nct) * kKsCols;
  float2* base = g.work + (line / g.inner) * g.outer + (line % g.inner) * g.inner_ld + c0;
  ks_twiddles(tw, N);
  float2* in = kMode == 2 ? V : U;
  for (int i = threadIdx.x; i < N * kKsCols; i += blockDim.x) {
    const int n = i / kKsCols, c = i % kKsCols;
    in[i] = c0 + c < g.Wh ? base[n * g.ld + c] : make_float2(0.f, 0.f);
  }
  if (kMode == 2)
    for (int m = threadIdx.x; m < N; m += blockDim.x) live[m] = 1;
  __syncthreads();
  if (kMode != 2) {
    const uint8_t* mbase = g.mask + (line / g.inner) * g.m_outer + (line % g.inner) * g.m_inner_ld + c0;
    for (int m = threadIdx.x; m < N; m += blockDim.x) {
      float re[kKsCols], im[kKsCols];
      ks_col_fwd(tw, U, N, m, re, im);
      if (kMode == 0) {
#pragma unroll
        for (int j = 0; j < kKsCols; ++j)
          if (c0 + j < g.Wh) base[m * g.ld + j] = make_float2(re[j], im[j]);
        continue;
      }
      const uint8_t* mrow = mbase + m * g.m_ld;
      int any = 0;
#pragma unroll
      for (int j = 0; j < kKsCols; ++j) {
        const bool keep = c0 + j < g.Wh && mrow[j] != 0;
        any |= keep;
        V[m * kKsCols + j] = keep ? make_float2(re[j], im[j]) : make_float2(0.f, 0.f);
      }
      live[m] = any;
    }
    if (kMode == 0) return;
    __syncthreads();
  }
  for (int h = threadIdx.x; h < N; h += blockDim.x) {
    float re[kKsCols], im[kKsCols];
    ks_col_inv(tw, V, live, N, h, re, im);
    float2* out = base + h * g.ld;
#pragma unroll
    for (int j = 0; j < kKsCols; ++j)
      if (c0 + j < g.Wh) out[j] = make_float2(re[j], im[j]);
  }
}

// the half spectra of kKsRows rows starting at row h0 of `plane` into us[Wh][kKsRows], bins other
// than 0 and W/2 doubled: Re of the full inverse sum counts them twice (their mirror)
__device__ __forceinline__ void ks_load_half_rows(float2* us, const float2* work, long long plane, int rows,
                                                  int h0, int W, int Wh) {
  for (int i = threadIdx.x; i < kKsRows * Wh; i += blockDim.x) {
    const int r = i / Wh, k = i - r * Wh;
    float2 v = make_float2(0.f, 0.f);
    if (h0 + r < rows) {
      v = work[(plane * rows + h0 + r) * Wh + k];
      if (k != 0 && 2 * k != W) v = make_float2(2.f * v.x, 2.f * v.y);
    }
    us[k * kKsRows + r] = v;
  }
}

__global__ void __launch_bounds__(kKsThreadsC) kspace_rows_inv_kernel(const KspaceArgs a) {
  extern __shared__ float4 ks_smem[];
  float2* tw = reinterpret_cast<float2*>(ks_smem);
  float2* us = tw + ks_tw_len(a.W);                 // [Wh][kKsRows]
  const int nrb = (a.H + kKsRows - 1) / kKsRows;
  const long long plane = blockIdx.x / nrb;
  const int h0 = (int)(blockIdx.x % nrb) * kKsRows;
  const long long tau = a.t[plane / a.channels] + a.t_delta;
  ks_twiddles(tw, a.W);
  ks_load_half_rows(us, a.work, plane, a.H, h0, a.W, a.Wh);
  __syncthreads();
  const float scale = (float)(1.0 / ((double)a.H * a.W));
  const float sac = tau < 0 ? 1.f : __ldg(a.sqrt_ac + tau);
  for (int w = threadIdx.x; w < a.W; w += blockDim.x) {
    float acc[kKsRows];
    ks_row_inv(tw, us, a.W, a.Wh, w, acc);
#pragma unroll
    for (int r = 0; r < kKsRows; ++r) {
      if (h0 + r >= a.H) break;
      const long long e = (plane * a.H + h0 + r) * a.W + w;
      const float add = tau < 0 ? a.zf[e] : __fmul_rn(sac, a.zf[e]);
      a.x[e] = __fadd_rn(__fsub_rn(a.x[e], __fmul_rn(acc[r], scale)), add);
    }
  }
}

// ------------------------------------------------------------------------------------------
// Measurement-guided sampling of the 3-D latent model (mri_dc_project3d, mri_dc_mask,
// mri_guided_x0, mri_guided_eps).  The data terms write g = P u - x_zf and the per-sample
// ||g||^2; the sums of squares are fp64, per block in a fixed tree order, then per sample over
// the blocks in index order (dc_norm_kernel): no atomics, so a replay is bit-reproducible.
// ------------------------------------------------------------------------------------------
constexpr int kDcMaskBlocks = 128;     // blocks per sample of the image-mask term

// the fp64 sum of v over the block in a fixed order; valid in thread 0
__device__ __forceinline__ double block_sum_fixed(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
  return s;
}

// gg[n] = sum of partial[n * per][0 .. per), in order per thread, then a fixed tree
__global__ void __launch_bounds__(256) dc_norm_kernel(const double* partial, int per, float* gg) {
  __shared__ double red[8];
  const double* p = partial + (long long)blockIdx.x * per;
  double v = 0.0;
  for (int i = threadIdx.x; i < per; i += blockDim.x) v += p[i];
  const double s = block_sum_fixed(v, red);
  if (threadIdx.x == 0) gg[blockIdx.x] = (float)s;
}

struct Dc3Args {
  const float* u;
  const float* zf;
  float* g;
  float2* work;
  double* partial;     // one per block of the inverse row pass
  int rows, W, Wh;     // rows = D * H per plane
};

// forward real row DFT of u, rows of all planes: work[plane][D][H][Wh]
__global__ void __launch_bounds__(kKsThreadsA) dc3_rows_fwd_kernel(const Dc3Args a) {
  extern __shared__ float4 ks_smem[];
  float2* tw = reinterpret_cast<float2*>(ks_smem);
  float* u = reinterpret_cast<float*>(tw + ks_tw_len(a.W));    // [W][kKsRows]
  const int nrb = (a.rows + kKsRows - 1) / kKsRows;
  const long long plane = blockIdx.x / nrb;
  const int h0 = (int)(blockIdx.x % nrb) * kKsRows;
  ks_twiddles(tw, a.W);
  for (int i = threadIdx.x; i < kKsRows * a.W; i += blockDim.x) {
    const int r = i / a.W, w = i - r * a.W;
    u[w * kKsRows + r] = h0 + r < a.rows ? a.u[(plane * a.rows + h0 + r) * a.W + w] : 0.f;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < a.Wh; k += blockDim.x) {
    float re[kKsRows], im[kKsRows];
    ks_row_fwd(tw, u, a.W, k, re, im);
#pragma unroll
    for (int r = 0; r < kKsRows; ++r)
      if (h0 + r < a.rows) a.work[(plane * a.rows + h0 + r) * a.Wh + k] = make_float2(re[r], im[r]);
  }
}

// inverse real row DFT, g = P u - x_zf, and this block's sum of g^2
__global__ void __launch_bounds__(kKsThreadsC) dc3_rows_inv_kernel(const Dc3Args a, float scale) {
  extern __shared__ float4 ks_smem[];
  __shared__ double red[kKsThreadsC / 32];
  float2* tw = reinterpret_cast<float2*>(ks_smem);
  float2* us = tw + ks_tw_len(a.W);                 // [Wh][kKsRows]
  const int nrb = (a.rows + kKsRows - 1) / kKsRows;
  const long long plane = blockIdx.x / nrb;
  const int h0 = (int)(blockIdx.x % nrb) * kKsRows;
  ks_twiddles(tw, a.W);
  ks_load_half_rows(us, a.work, plane, a.rows, h0, a.W, a.Wh);
  __syncthreads();
  double ss = 0.0;
  for (int w = threadIdx.x; w < a.W; w += blockDim.x) {
    float acc[kKsRows];
    ks_row_inv(tw, us, a.W, a.Wh, w, acc);
#pragma unroll
    for (int r = 0; r < kKsRows; ++r) {
      if (h0 + r >= a.rows) break;
      const long long e = (plane * a.rows + h0 + r) * a.W + w;
      const float gv = __fsub_rn(__fmul_rn(acc[r], scale), a.zf[e]);
      a.g[e] = gv;
      ss += (double)gv * gv;
    }
  }
  const double s = block_sum_fixed(ss, red);
  if (threadIdx.x == 0) a.partial[blockIdx.x] = s;
}

// g = mask ? 0 : u - known (select: known is not read where mask != 0), grid (kDcMaskBlocks, samples)
__global__ void __launch_bounds__(256)
dc_mask_kernel(const float* u, const float* known, const uint8_t* mask, float* g, double* partial,
               long long per_sample) {
  __shared__ double red[8];
  const long long off = (long long)blockIdx.y * per_sample;
  double ss = 0.0;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < per_sample;
       j += (long long)gridDim.x * blockDim.x) {
    const long long e = off + j;
    const float gv = mask[e] != 0 ? 0.f : __fsub_rn(u[e], known[e]);
    g[e] = gv;
    ss += (double)gv * gv;
  }
  const double s = block_sum_fixed(ss, red);
  if (threadIdx.x == 0) partial[(long long)blockIdx.y * gridDim.x + blockIdx.x] = s;
}

// out = (z - s1m[t] eps) / sac[t] * inv_s per element (step 2 of the guided step)
__global__ void __launch_bounds__(256)
guided_x0_kernel(const float* z, const void* eps, int ldc, int channels, const int64_t* t,
                 const float* sqrt_ac, const float* sqrt_1mac, const float* inv_s, float* out,
                 long long per_sample, long long numel) {
  const long long spatial = per_sample / (channels > 0 ? channels : 1);
  const float is = *inv_s;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < numel;
       e += (long long)gridDim.x * blockDim.x) {
    const long long n = e / per_sample;
    const int64_t ts = t[n];
    const float ev = load_eps(eps, ldc, spatial, per_sample, n, e - n * per_sample);
    const float x0 = __fdiv_rn(__fsub_rn(z[e], __fmul_rn(__ldg(sqrt_1mac + ts), ev)), __ldg(sqrt_ac + ts));
    out[e] = __fmul_rn(x0, is);
  }
}

// eps' = eps - (sac[t] / s1m[t]) * delta, delta = -(lam / sqrt(gg[n])) * (dz * inv_s); eps' = eps
// where that coefficient is 0 (lam = 0 or ||g|| = 0)
__global__ void __launch_bounds__(256)
guided_eps_kernel(const void* eps, int ldc, int channels, const float* dz, const float* gg,
                  const float* lam, const float* inv_s, const int64_t* t, const float* sqrt_ac,
                  const float* sqrt_1mac, float* out, long long per_sample, long long numel) {
  const long long spatial = per_sample / (channels > 0 ? channels : 1);
  const float l = *lam, is = *inv_s;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < numel;
       e += (long long)gridDim.x * blockDim.x) {
    const long long n = e / per_sample;
    const int64_t ts = t[n];
    const float ev = load_eps(eps, ldc, spatial, per_sample, n, e - n * per_sample);
    const float q = gg[n];
    const float coef = q > 0.f ? __fdiv_rn(l, __fsqrt_rn(q)) : 0.f;
    if (coef == 0.f) {
      out[e] = ev;
      continue;
    }
    const float delta = __fmul_rn(-coef, __fmul_rn(dz[e], is));
    const float r = __fdiv_rn(__ldg(sqrt_ac + ts), __ldg(sqrt_1mac + ts));
    out[e] = __fsub_rn(ev, __fmul_rn(r, delta));
  }
}

// ------------------------------------------------------------------------------------------
// Terms of the variational bound on -log p(x0) for one evaluation step at per-sample timestep
// t[n], given x0, x_t = q_sample(x0, t, z), z and the predicted eps:
//   acc[n][t][0] += sum (eps - z)^2                      (L_t = lambda_t times this for t >= 1)
//   t = 0:  acc[n][0][1] += sum -log p(x0 | x_t),  mean mu = DdpmUpdate::apply at t = 0 (w = 0),
//           log-scale ls = 0.5 * post_log_var[0];  prior[n] += sum x0^2 (prior optional)
// Per-element arithmetic is fp32; thread and block partials are fp64, one atomicAdd per block,
// sample and quantity (order-insensitive to about 1e-16, as the GroupNorm statistics).
// kDecDiscrete: improved-diffusion's discretized_gaussian_log_likelihood (data in [-1, 1], bins
// +-1/255, edges at +-0.999, tanh CDF, logs clamped at 1e-12); otherwise the Gaussian density.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float approx_std_normal_cdf(float x) {
  const float k = 0.7978845608028654f;   // sqrt(2 / pi)
  return 0.5f * (1.0f + tanhf(k * (x + 0.044715f * (x * x * x))));
}

template <bool kDecDiscrete>
__device__ __forceinline__ float decoder_nll(float x0, float mu, float ls, float inv_std) {
  const float c = x0 - mu;
  if constexpr (kDecDiscrete) {
    const float cdf_plus = approx_std_normal_cdf(inv_std * (c + 1.0f / 255.0f));
    const float cdf_min = approx_std_normal_cdf(inv_std * (c - 1.0f / 255.0f));
    const float lp = x0 < -0.999f ? logf(fmaxf(cdf_plus, 1e-12f))
                     : x0 > 0.999f ? logf(fmaxf(1.0f - cdf_min, 1e-12f))
                                   : logf(fmaxf(cdf_plus - cdf_min, 1e-12f));
    return -lp;
  } else {
    const float y = c * inv_std;
    return 0.5f * (y * y) + ls + 0.91893853320467274f;   // + 0.5 log(2 pi)
  }
}

// grid (blocks, samples): block (b, n) strides over sample n only
template <bool kDecDiscrete>
__global__ void __launch_bounds__(256)
vb_terms_kernel(const DdpmUpdate u, const float* x0, const float* xt, const void* eps, int ldc,
                int channels, const float* z, const float* post_log_var, double* acc, double* prior,
                int T, long long per_sample) {
  const int n = blockIdx.y;
  const int64_t ts = u.t[n];
  if (ts < 0 || ts >= T) return;   // uniform over the block
  const bool dec = ts == 0;
  const long long spatial = per_sample / (channels > 0 ? channels : 1);
  const long long base = (long long)n * per_sample;
  DdpmUpdate::Coef c{0.f, 0.f, 0.f};
  float ls = 0.f, inv_std = 0.f;
  if (dec) {
    c = u.coef(n);
    ls = 0.5f * __ldg(post_log_var);
    inv_std = expf(-ls);
  }
  double s_mse = 0.0, s_dec = 0.0, s_x2 = 0.0;
  auto one = [&](long long j, float e, float zz) {
    const float d = e - zz;
    s_mse += (double)(d * d);
    if (dec) {
      const float x = x0[base + j];
      float unused;
      const float mu = DdpmUpdate::apply(c, xt[base + j], e, 0.f, unused);
      s_dec += (double)decoder_nll<kDecDiscrete>(x, mu, ls, inv_std);
      s_x2 += (double)(x * x);
    }
  };
  const long long step = 4LL * gridDim.x * blockDim.x;
  for (long long j = 4LL * ((long long)blockIdx.x * blockDim.x + threadIdx.x); j < per_sample; j += step) {
    // four elements inside the sample and, for the channels-last eps, inside one channel
    if (j + 3 >= per_sample || (ldc != 0 && (j % spatial) + 3 >= spatial)) {
      for (int m = 0; m < 4 && j + m < per_sample; ++m)
        one(j + m, load_eps(eps, ldc, spatial, per_sample, n, j + m), z[base + j + m]);
      continue;
    }
    float zv[4], ev[4];
    load4(z + base + j, aligned16(z + base + j), zv);
    load_eps4(eps, ldc, spatial, per_sample, n, j,
              ldc == 0 && aligned16(reinterpret_cast<const float*>(eps) + base + j), ev);
    if (!dec) {
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const float d = ev[m] - zv[m];
        s_mse += (double)(d * d);
      }
      continue;
    }
    float xv[4], tv[4];
    load4(x0 + base + j, aligned16(x0 + base + j), xv);
    load4(xt + base + j, aligned16(xt + base + j), tv);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const float d = ev[m] - zv[m];
      s_mse += (double)(d * d);
      float unused;
      const float mu = DdpmUpdate::apply(c, tv[m], ev[m], 0.f, unused);
      s_dec += (double)decoder_nll<kDecDiscrete>(xv[m], mu, ls, inv_std);
      s_x2 += (double)(xv[m] * xv[m]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s_mse += __shfl_xor_sync(0xffffffffu, s_mse, o);
    s_dec += __shfl_xor_sync(0xffffffffu, s_dec, o);
    s_x2 += __shfl_xor_sync(0xffffffffu, s_x2, o);
  }
  __shared__ double part[3][8];
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    part[0][w] = s_mse;
    part[1][w] = s_dec;
    part[2][w] = s_x2;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double tot[3] = {0.0, 0.0, 0.0};
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i)
#pragma unroll
    for (int q = 0; q < 3; ++q) tot[q] += part[q][i];
  double* a = acc + ((long long)n * T + ts) * 2;
  atomicAdd(a, tot[0]);
  if (dec) {
    atomicAdd(a + 1, tot[1]);
    if (prior != nullptr) atomicAdd(prior + n, tot[2]);
  }
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

// the column kernels' shared memory, once at the largest size (not re-done inside a graph capture)
static int ks_configure() {
  static bool configured = false;
  if (configured) return 0;
  void (*kerns[3])(const KsColGeom) = {kspace_cols_kernel<0>, kspace_cols_kernel<1>, kspace_cols_kernel<2>};
  for (auto k : kerns) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, ks_smem_b(kKsMaxN));
    if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(kspace_cols_kernel)");
  }
  configured = true;
  return 0;
}

static int kspace_dims(const char* who, int samples, int channels, int H, int W) {
  if (samples < 1 || channels < 1 || H < 1 || W < 1) return set_error(-2, who);
  if (H > kKsMaxN || W > kKsMaxN) return set_error(-2, "mri_kspace_merge: H and W must be at most 512");
  if ((long long)samples * channels * ((H + kKsRows - 1) / kKsRows) > 0x7fffffffLL)
    return set_error(-2, "mri_kspace_merge: too many planes");
  return 0;
}

extern "C" int mri_kspace_work_bytes(int samples, int channels, int H, int W, size_t* bytes_out) {
  int rc = kspace_dims("mri_kspace_work_bytes: empty input", samples, channels, H, W);
  if (rc) return rc;
  if (bytes_out == nullptr) return set_error(-2, "mri_kspace_work_bytes: null output");
  *bytes_out = (size_t)samples * channels * H * (W / 2 + 1) * sizeof(float2);
  return 0;
}

extern "C" int mri_kspace_merge(float* x, const float* x_zf, const uint8_t* kmask, const float* noise,
                                const uint64_t* rng, uint64_t rng_skip, const int64_t* t,
                                int64_t t_delta, const float* sqrt_ac, const float* sqrt_1mac,
                                void* work, size_t work_bytes, int samples, int channels, int H, int W,
                                void* stream) {
  size_t need = 0;
  int rc = mri_kspace_work_bytes(samples, channels, H, W, &need);
  if (rc) return rc;
  if (x == nullptr || x_zf == nullptr || kmask == nullptr || t == nullptr || sqrt_ac == nullptr ||
      sqrt_1mac == nullptr || work == nullptr)
    return set_error(-2, "mri_kspace_merge: null x / x_zf / kmask / t / schedule table / work");
  if ((noise == nullptr) == (rng == nullptr))
    return set_error(-2, "mri_kspace_merge: exactly one of noise / rng");
  if (rng_skip % 4 != 0) return set_error(-2, "mri_kspace_merge: rng_skip must be a multiple of 4");
  if (work_bytes < need || (reinterpret_cast<uintptr_t>(work) & 7) != 0)
    return set_error(-2, "mri_kspace_merge: work smaller than mri_kspace_work_bytes or not 8-byte aligned");
  rc = device_props();
  if (rc) return rc;
  rc = ks_configure();
  if (rc) return rc;
  KspaceArgs a;
  a.x = x;
  a.zf = x_zf;
  a.mask = kmask;
  a.noise = noise;
  a.rng = rng;
  a.ctr_skip = rng_skip / 4;
  a.t = t;
  a.t_delta = t_delta;
  a.sqrt_ac = sqrt_ac;
  a.sqrt_1mac = sqrt_1mac;
  a.work = static_cast<float2*>(work);
  a.channels = channels; a.H = H; a.W = W; a.Wh = W / 2 + 1;
  const long long planes = (long long)samples * channels;
  a.Tt = aten_grid(planes * H * W).Tt;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned rows_grid = (unsigned)(planes * ((H + kKsRows - 1) / kKsRows));
  if (rng != nullptr)
    kspace_rows_fwd_kernel<true><<<rows_grid, kKsThreadsA, ks_smem_a(W), st>>>(a);
  else
    kspace_rows_fwd_kernel<false><<<rows_grid, kKsThreadsA, ks_smem_a(W), st>>>(a);
  rc = check_launch("kspace_rows_fwd_kernel");
  if (rc) return rc;
  KsColGeom g{a.work, kmask, H, a.Wh, 1, (long long)H * a.Wh, 0, a.Wh, (long long)H * W, 0, W};
  kspace_cols_kernel<1><<<(unsigned)(planes * ((a.Wh + kKsCols - 1) / kKsCols)), kKsThreadsB, ks_smem_b(H),
                          st>>>(g);
  rc = check_launch("kspace_cols_kernel");
  if (rc) return rc;
  kspace_rows_inv_kernel<<<rows_grid, kKsThreadsC, ks_smem_c(W), st>>>(a);
  return check_launch("kspace_rows_inv_kernel");
}

static int dc3_dims(int samples, int channels, int D, int H, int W) {
  if (samples < 1 || channels < 1 || D < 1 || H < 1 || W < 1)
    return set_error(-2, "mri_dc_project3d: empty input");
  if (D > kKsMaxN || H > kKsMaxN || W > kKsMaxN)
    return set_error(-2, "mri_dc_project3d: D, H and W must be at most 512");
  const long long planes = (long long)samples * channels;
  if (planes * ((D * H + kKsRows - 1) / kKsRows) > 0x7fffffffLL || planes * H * ((W / 2 + 1 + kKsCols - 1) / kKsCols) > 0x7fffffffLL ||
      planes * D * ((W / 2 + 1 + kKsCols - 1) / kKsCols) > 0x7fffffffLL)
    return set_error(-2, "mri_dc_project3d: too many rows");
  return 0;
}

// the complex half spectra, then the fp64 partial sums of the inverse row pass
static size_t dc3_spectrum_bytes(int samples, int channels, int D, int H, int W) {
  const size_t b = (size_t)samples * channels * D * H * (W / 2 + 1) * sizeof(float2);
  return (b + 255) & ~(size_t)255;
}

extern "C" int mri_kspace3d_work_bytes(int samples, int channels, int D, int H, int W, size_t* bytes_out) {
  int rc = dc3_dims(samples, channels, D, H, W);
  if (rc) return rc;
  if (bytes_out == nullptr) return set_error(-2, "mri_kspace3d_work_bytes: null output");
  const size_t nrb = (size_t)(D * H + kKsRows - 1) / kKsRows;
  *bytes_out = dc3_spectrum_bytes(samples, channels, D, H, W) + (size_t)samples * channels * nrb * sizeof(double);
  return 0;
}

extern "C" int mri_dc_project3d(const float* u, const float* x_zf, const uint8_t* kmask, float* g,
                                float* gg, void* work, size_t work_bytes, int samples, int channels,
                                int D, int H, int W, void* stream) {
  size_t need = 0;
  int rc = mri_kspace3d_work_bytes(samples, channels, D, H, W, &need);
  if (rc) return rc;
  if (u == nullptr || x_zf == nullptr || kmask == nullptr || g == nullptr || gg == nullptr || work == nullptr)
    return set_error(-2, "mri_dc_project3d: null u / x_zf / kmask / g / gg / work");
  if (work_bytes < need || (reinterpret_cast<uintptr_t>(work) & 7) != 0)
    return set_error(-2, "mri_dc_project3d: work smaller than mri_kspace3d_work_bytes or not 8-byte aligned");
  rc = ks_configure();
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long planes = (long long)samples * channels;
  const int Wh = W / 2 + 1, nct = (Wh + kKsCols - 1) / kKsCols;
  const int rows = D * H, nrb = (rows + kKsRows - 1) / kKsRows;
  Dc3Args a;
  a.u = u;
  a.zf = x_zf;
  a.g = g;
  a.work = static_cast<float2*>(work);
  a.partial = reinterpret_cast<double*>(static_cast<char*>(work) + dc3_spectrum_bytes(samples, channels, D, H, W));
  a.rows = rows; a.W = W; a.Wh = Wh;
  const long long vol = (long long)D * H * Wh, slab = (long long)H * Wh;
  const long long mvol = (long long)D * H * W, mslab = (long long)H * W;
  dc3_rows_fwd_kernel<<<(unsigned)(planes * nrb), kKsThreadsA, ks_smem_a(W), st>>>(a);
  rc = check_launch("dc3_rows_fwd_kernel");
  if (rc) return rc;
  // forward along H: line (plane, d)
  const KsColGeom gh{a.work, nullptr, H, Wh, 1, slab, 0, Wh, 0, 0, 0};
  kspace_cols_kernel<0><<<(unsigned)(planes * D * nct), kKsThreadsB, ks_smem_b(H), st>>>(gh);
  rc = check_launch("kspace_cols_kernel<0>");
  if (rc) return rc;
  // forward along D, times M, inverse along D: line (plane, h)
  const KsColGeom gd{a.work, kmask, D, Wh, H, vol, Wh, slab, mvol, W, mslab};
  kspace_cols_kernel<1><<<(unsigned)(planes * H * nct), kKsThreadsB, ks_smem_b(D), st>>>(gd);
  rc = check_launch("kspace_cols_kernel<1>");
  if (rc) return rc;
  kspace_cols_kernel<2><<<(unsigned)(planes * D * nct), kKsThreadsB, ks_smem_b(H), st>>>(gh);
  rc = check_launch("kspace_cols_kernel<2>");
  if (rc) return rc;
  const float scale = (float)(1.0 / ((double)D * H * W));
  dc3_rows_inv_kernel<<<(unsigned)(planes * nrb), kKsThreadsC, ks_smem_c(W), st>>>(a, scale);
  rc = check_launch("dc3_rows_inv_kernel");
  if (rc) return rc;
  dc_norm_kernel<<<(unsigned)samples, 256, 0, st>>>(a.partial, (int)(channels * nrb), gg);
  return check_launch("dc_norm_kernel");
}

extern "C" int mri_dc_mask(const float* u, const float* known, const uint8_t* mask, float* g, float* gg,
                           void* work, size_t work_bytes, int samples, int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1) return set_error(-2, "mri_dc_mask: empty input");
  if (samples > 65535) return set_error(-2, "mri_dc_mask: at most 65535 samples");
  if (u == nullptr || known == nullptr || mask == nullptr || g == nullptr || gg == nullptr || work == nullptr)
    return set_error(-2, "mri_dc_mask: null u / known / mask / g / gg / work");
  if (work_bytes < (size_t)samples * kDcMaskBlocks * sizeof(double) || (reinterpret_cast<uintptr_t>(work) & 7) != 0)
    return set_error(-2, "mri_dc_mask: work smaller than 1024 bytes per sample or not 8-byte aligned");
  double* partial = static_cast<double*>(work);
  cudaStream_t st = (cudaStream_t)stream;
  dc_mask_kernel<<<dim3(kDcMaskBlocks, (unsigned)samples), 256, 0, st>>>(u, known, mask, g, partial, per_sample);
  int rc = check_launch("dc_mask_kernel");
  if (rc) return rc;
  dc_norm_kernel<<<(unsigned)samples, 256, 0, st>>>(partial, kDcMaskBlocks, gg);
  return check_launch("dc_norm_kernel");
}

static int guided_dims(const char* who, const void* eps, int ldc, int channels, int samples,
                       int64_t per_sample) {
  if (samples < 1 || per_sample < 1) return set_error(-2, who);
  if (eps == nullptr) return set_error(-2, who);
  if (ldc != 0 && (channels < 1 || per_sample % channels != 0 || ldc < channels)) return set_error(-2, who);
  return device_props();
}

extern "C" int mri_guided_x0(const float* z, const void* eps, int eps_nhwc_ldc, int channels,
                             const int64_t* t, const float* sqrt_ac, const float* sqrt_1mac,
                             const float* inv_s, float* out, int samples, int64_t per_sample,
                             void* stream) {
  int rc = guided_dims("mri_guided_x0: empty input, null eps or per_sample not channels * spatial, ldc >= channels",
                       eps, eps_nhwc_ldc, channels, samples, per_sample);
  if (rc) return rc;
  if (z == nullptr || t == nullptr || sqrt_ac == nullptr || sqrt_1mac == nullptr || inv_s == nullptr || out == nullptr)
    return set_error(-2, "mri_guided_x0: null z / t / schedule table / inv_s / out");
  const long long numel = (long long)samples * per_sample;
  guided_x0_kernel<<<my_blocks(aten_grid(numel)), 256, 0, (cudaStream_t)stream>>>(
      z, eps, eps_nhwc_ldc, channels, t, sqrt_ac, sqrt_1mac, inv_s, out, per_sample, numel);
  return check_launch("guided_x0_kernel");
}

extern "C" int mri_guided_eps(const void* eps, int eps_nhwc_ldc, int channels, const float* dz,
                              const float* gg, const float* lam, const float* inv_s, const int64_t* t,
                              const float* sqrt_ac, const float* sqrt_1mac, float* out, int samples,
                              int64_t per_sample, void* stream) {
  int rc = guided_dims("mri_guided_eps: empty input, null eps or per_sample not channels * spatial, ldc >= channels",
                       eps, eps_nhwc_ldc, channels, samples, per_sample);
  if (rc) return rc;
  if (dz == nullptr || gg == nullptr || lam == nullptr || inv_s == nullptr || t == nullptr ||
      sqrt_ac == nullptr || sqrt_1mac == nullptr || out == nullptr)
    return set_error(-2, "mri_guided_eps: null dz / gg / lam / inv_s / t / schedule table / out");
  const long long numel = (long long)samples * per_sample;
  guided_eps_kernel<<<my_blocks(aten_grid(numel)), 256, 0, (cudaStream_t)stream>>>(
      eps, eps_nhwc_ldc, channels, dz, gg, lam, inv_s, t, sqrt_ac, sqrt_1mac, out, per_sample, numel);
  return check_launch("guided_eps_kernel");
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

extern "C" int mri_vb_terms(const float* x0, const float* x_t, const void* eps, int eps_nhwc_ldc,
                            int channels, const float* z, const int64_t* t, const float* betas,
                            const float* sqrt_1mac, const float* sqrt_recip_alphas,
                            const float* post_var, const float* post_log_var, int decoder,
                            double* acc, double* prior, int timesteps, int samples,
                            int64_t per_sample, void* stream) {
  if (samples < 1 || per_sample < 1 || timesteps < 1) return set_error(-2, "mri_vb_terms: empty input");
  if (samples > 65535) return set_error(-2, "mri_vb_terms: at most 65535 samples");
  if (x0 == nullptr || x_t == nullptr || eps == nullptr || z == nullptr || t == nullptr ||
      betas == nullptr || sqrt_1mac == nullptr || sqrt_recip_alphas == nullptr ||
      post_var == nullptr || post_log_var == nullptr || acc == nullptr)
    return set_error(-2, "mri_vb_terms: null input / schedule table / acc");
  if (eps_nhwc_ldc != 0 && (channels < 1 || per_sample % channels != 0 || eps_nhwc_ldc < channels))
    return set_error(-2, "mri_vb_terms: per_sample must be channels * spatial, ldc >= channels");
  if (decoder != 0 && decoder != 1)
    return set_error(-2, "mri_vb_terms: decoder 0 (discretized) / 1 (Gaussian)");
  long long bx = (per_sample + 4 * 256 - 1) / (4 * 256);
  const long long cap = (148 * 8 + samples - 1) / samples;
  if (bx > cap) bx = cap;
  const dim3 grid((unsigned)bx, (unsigned)samples);
  const DdpmUpdate u{t, betas, sqrt_1mac, sqrt_recip_alphas, post_var};
  if (decoder == 0)
    vb_terms_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(
        u, x0, x_t, eps, eps_nhwc_ldc, channels, z, post_log_var, acc, prior, timesteps, per_sample);
  else
    vb_terms_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(
        u, x0, x_t, eps, eps_nhwc_ldc, channels, z, post_log_var, acc, prior, timesteps, per_sample);
  return check_launch("vb_terms_kernel");
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
