// Fused spatial self-attention of the bottleneck (AttentionBlock3D, ddpm_3d_ldm/unet_attention.py:
// 37-56), inference path: O = softmax(Q K^T / sqrt(d)) V per (sample, head) without the logits or
// the probabilities ever touching HBM.
//
// One CTA per (sample, head, tile of 128 queries), 192 threads:
//   warp 0     TMA producer: Q once, then K_j and V^T_j tiles (128 keys) through two-deep rings
//   warp 1     TMEM allocator + tcgen05.mma issuer (one elected thread):
//              S_j = Q K_j^T (M = 128 queries, N = 128 keys, K = d) into one of two S buffers, so
//              that S_{j+1} is computed while the softmax warps work on S_j;
//              O  += P_j V_j (M = 128, N = d, K = 128 keys), accumulating in TMEM
//   warps 2-5  softmax: thread = query row (TMEM lane).  Online softmax with a LAZY reference
//              maximum: the row keeps exponentiating against m_ref until the running maximum
//              exceeds it by more than 2^8 (in the exp2 domain); only then are l and the O
//              accumulator in TMEM rescaled (tcgen05.ld / st) -- with identical arithmetic up to
//              rounding, since any reference works as long as l and O use the same one.
//              P_j goes to shared memory as the bf16 K-major (128B-swizzled) A operand of the
//              second MMA; at the end O / l is written to the token-major output.
// Operand layouts: Q, K rows come straight from the qkv GEMM's token-major output [B][n][3C]
// (d contiguous = K-major for both operands of S); V^T comes from the kvT GEMM's output
// [B][rows][npad] (keys contiguous = K-major B operand of P V).  Precondition: V^T columns
// [n, npad) must be finite -- the masked keys meet P = 0 there, and 0 * NaN is NaN.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/mri_b200.h"
#include "common.h"
#include "ptx.cuh"

namespace mri {

constexpr int kAttnThreads = 192;
constexpr int kTile = 128;                    // queries per CTA, keys per step
constexpr int kSlab = kTile * 128;            // 128 rows x 64 bf16

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* map, uint32_t bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int D>
__host__ __device__ constexpr int attn_smem_bytes() {
  // Q (D/64 slabs) + K ring (2 x D/64 slabs) + V^T ring (2 x 2 slabs of D rows) + P (2 slabs)
  return (D / 64) * kSlab + 2 * (D / 64) * kSlab + 2 * 2 * D * 128 + 2 * kSlab + 1024;
}

template <int D>
__global__ void __launch_bounds__(kAttnThreads, 1)
attn_flash_kernel(const __grid_constant__ MriAttnArgs p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[16];
  __shared__ uint32_t tmem_holder;
  constexpr int DS = D / 64;                  // 64-channel slabs of a Q / K tile
  constexpr uint32_t kQBytes = DS * kSlab;
  constexpr uint32_t kKBytes = DS * kSlab;
  constexpr uint32_t kVBytes = 2 * D * 128;   // two 64-key slabs of D rows

  const int warp = uniform((int)(threadIdx.x >> 5));
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_smem = smem_base;
  const uint32_t k_smem = q_smem + kQBytes;             // + stage * kKBytes
  const uint32_t v_smem = k_smem + 2 * kKBytes;         // + stage * kVBytes
  const uint32_t p_smem = v_smem + 2 * kVBytes;

  const uint32_t bar0 = smem_u32(bars);
  const uint32_t q_full = bar0;
  auto k_full = [&](int s) { return bar0 + 8u * (1 + s); };
  auto k_empty = [&](int s) { return bar0 + 8u * (3 + s); };
  auto v_full = [&](int s) { return bar0 + 8u * (5 + s); };
  auto v_empty = [&](int s) { return bar0 + 8u * (7 + s); };
  auto s_full = [&](int s) { return bar0 + 8u * (9 + s); };
  auto s_empty = [&](int s) { return bar0 + 8u * (11 + s); };
  const uint32_t p_full = bar0 + 8u * 13;
  const uint32_t pv_done = bar0 + 8u * 14;

  // work item
  const int q_tiles = (p.n + kTile - 1) / kTile;
  int w = (int)blockIdx.x;
  const int qt = w % q_tiles;
  w /= q_tiles;
  const int head = w % p.heads;
  const int b = w / p.heads;
  const int q0 = qt * kTile;
  const int T = (p.n + kTile - 1) / kTile;    // key tiles

  if (warp == 0 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(k_full(s), 1);
      mbar_init(k_empty(s), 1);
      mbar_init(v_full(s), 1);
      mbar_init(v_empty(s), 1);
      mbar_init(s_full(s), 1);
      mbar_init(s_empty(s), 4);   // one arrive per softmax warp
    }
    mbar_init(p_full, 4);
    mbar_init(pv_done, 1);
    mbar_fence_init();
    tma_prefetch_desc(p.qk_map);
    tma_prefetch_desc(p.vt_map);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(&tmem_holder), 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_holder;
  const uint32_t tm_s0 = tmem_base;           // S buffers: columns [0,128) and [128,256)
  const uint32_t tm_o = tmem_base + 256u;     // O accumulator: columns [256, 256 + D)

  if (warp == 0) {
    // ================================ TMA producer ==================================
    if (elect_one_sync()) {
      mbar_arrive_expect_tx(q_full, kQBytes);
#pragma unroll
      for (int s = 0; s < DS; ++s)
        tma_load_3d(q_smem + s * kSlab, p.qk_map, q_full, head * D + s * 64, q0, b);
      for (int j = 0; j < T; ++j) {
        const int st = j & 1;
        const uint32_t par = (uint32_t)((j >> 1) & 1);
        mbar_wait(k_empty(st), par ^ 1u);
        mbar_arrive_expect_tx(k_full(st), kKBytes);
#pragma unroll
        for (int s = 0; s < DS; ++s)
          tma_load_3d(k_smem + st * kKBytes + s * kSlab, p.qk_map, k_full(st),
                      p.k_col0 + head * D + s * 64, j * kTile, b);
        mbar_wait(v_empty(st), par ^ 1u);
        mbar_arrive_expect_tx(v_full(st), kVBytes);
#pragma unroll
        for (int s = 0; s < 2; ++s)
          tma_load_3d(v_smem + st * kVBytes + s * (D * 128), p.vt_map, v_full(st),
                      j * kTile + s * 64, p.v_row0 + head * D, b);
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ====================================
    if (elect_one_sync()) {
      const uint32_t idesc_s = umma_idesc_bf16(kTile, kTile);
      const uint32_t idesc_o = umma_idesc_bf16(kTile, (uint32_t)D);
      auto issue_s = [&](int j) {
        const int st = j & 1;
        const uint32_t par = (uint32_t)((j >> 1) & 1);
        mbar_wait(k_full(st), par);
        mbar_wait(s_empty(st), par ^ 1u);
        tc_fence_after();
#pragma unroll
        for (int s = 0; s < DS; ++s) {
          const uint64_t a_desc = umma_desc_k_sw128(q_smem + s * kSlab, 1024);
          const uint64_t b_desc = umma_desc_k_sw128(k_smem + st * kKBytes + s * kSlab, 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tm_s0 + (uint32_t)(st * kTile), a_desc + 2u * k, b_desc + 2u * k, idesc_s,
                      (s != 0 || k != 0) ? 1u : 0u);
        }
        umma_commit(k_empty(st));
        umma_commit(s_full(st));
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < T; ++j) {
        if (j + 1 < T) issue_s(j + 1);
        const int st = j & 1;
        mbar_wait(v_full(st), (uint32_t)((j >> 1) & 1));
        mbar_wait(p_full, (uint32_t)(j & 1));
        tc_fence_after();
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const uint64_t a_desc = umma_desc_k_sw128(p_smem + s * kSlab, 1024);
          const uint64_t b_desc = umma_desc_k_sw128(v_smem + st * kVBytes + s * (D * 128), 1024);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tm_o, a_desc + 2u * k, b_desc + 2u * k, idesc_o,
                      (j != 0 || s != 0 || k != 0) ? 1u : 0u);
        }
        umma_commit(v_empty(st));
        umma_commit(pv_done);
      }
    }
  } else {
    // ================================ softmax warps =================================
    const int q = warp & 3;                   // TMEM lane quadrant
    const int row = q * 32 + lane;            // query row of this thread inside the tile
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float c = p.scale * 1.4426950408889634f;   // logits * log2(e)
    float m_ref = -INFINITY;                  // reference maximum (raw logits, before scaling)
    float l = 0.f;                            // sum of exp2((s - m_ref) * c)
    const uint32_t p_row = p_smem + (uint32_t)row * 128u;
    const uint32_t xr = (uint32_t)(row & 7);

    for (int j = 0; j < T; ++j) {
      const int st = j & 1;
      mbar_wait(s_full(st), (uint32_t)((j >> 1) & 1));
      tc_fence_after();
      uint32_t sv[4][32];
#pragma unroll
      for (int g = 0; g < 4; ++g)
        tmem_ld32(tm_s0 + lane_addr + (uint32_t)(st * kTile + g * 32), sv[g]);
      tmem_ld_wait();
      // the S buffer is in registers: the MMA warp may overwrite it with S_{j+2}
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty(st));

      const int nvalid = p.n - j * kTile;     // keys of this tile that exist (>= 1)
      float m_new = m_ref;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float s = __uint_as_float(sv[g][i]);
          if (g * 32 + i >= nvalid) s = -INFINITY;
          sv[g][i] = __float_as_uint(s);
          m_new = fmaxf(m_new, s);
        }
      }
      // lazy rescale: keep m_ref unless the maximum grew by more than 2^8 in the exp2 domain
      const bool grow = (m_new - m_ref) * c > 8.0f;   // also true on the first tile (m_ref = -inf)
      float alpha = 1.0f;
      if (grow) {
        alpha = (m_ref == -INFINITY) ? 0.0f : ex2((m_ref - m_new) * c);
        m_ref = m_new;
      }
      // everything below needs P V_{j-1} finished: it reads P and accumulates into O
      if (j > 0) mbar_wait(pv_done, (uint32_t)((j - 1) & 1));
      if (j > 0 && __any_sync(0xffffffffu, grow)) {
        tc_fence_after();
        l *= alpha;
#pragma unroll
        for (int g = 0; g < D / 32; ++g) {
          uint32_t ov[32];
          tmem_ld32(tm_o + lane_addr + (uint32_t)(g * 32), ov);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) ov[i] = __float_as_uint(__uint_as_float(ov[i]) * alpha);
          asm volatile(
              "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
              "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
              "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(
                  tm_o + lane_addr + (uint32_t)(g * 32)),
              "r"(ov[0]), "r"(ov[1]), "r"(ov[2]), "r"(ov[3]), "r"(ov[4]), "r"(ov[5]), "r"(ov[6]),
              "r"(ov[7]), "r"(ov[8]), "r"(ov[9]), "r"(ov[10]), "r"(ov[11]), "r"(ov[12]), "r"(ov[13]),
              "r"(ov[14]), "r"(ov[15]), "r"(ov[16]), "r"(ov[17]), "r"(ov[18]), "r"(ov[19]),
              "r"(ov[20]), "r"(ov[21]), "r"(ov[22]), "r"(ov[23]), "r"(ov[24]), "r"(ov[25]),
              "r"(ov[26]), "r"(ov[27]), "r"(ov[28]), "r"(ov[29]), "r"(ov[30]), "r"(ov[31])
              : "memory");
        }
        tmem_st_wait();
      } else if (j == 0) {
        l = 0.f;
      }
      // P_j = exp2((s - m_ref) * c): bf16, K-major rows of 64 keys (128 B), 16-byte units XOR-swizzled
      const float mc = m_ref * c;
      float lsum = 0.f;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {       // 8 keys = one 16-byte unit
          uint32_t wv[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float p0 = ex2(fmaf(__uint_as_float(sv[g][u * 8 + 2 * e]), c, -mc));
            const float p1 = ex2(fmaf(__uint_as_float(sv[g][u * 8 + 2 * e + 1]), c, -mc));
            // the row sum uses the bf16-rounded values: exactly what the second MMA multiplies
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(p0, p1);
            wv[e] = *reinterpret_cast<const uint32_t*>(&h2);
            lsum += __low2float(h2) + __high2float(h2);
          }
          const int key8 = g * 4 + u;         // 16-byte unit index along the 128 keys
          const uint32_t slab = (uint32_t)(key8 >> 3);
          const uint32_t unit = (uint32_t)(key8 & 7) ^ xr;
          asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(p_row + slab * kSlab + (unit << 4)),
                       "r"(wv[0]), "r"(wv[1]), "r"(wv[2]), "r"(wv[3])
                       : "memory");
        }
      }
      l += lsum;
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }
    // ---- O / l -> token-major bf16 output ------------------------------------------------------
    mbar_wait(pv_done, (uint32_t)((T - 1) & 1));
    tc_fence_after();
    const float inv_l = 1.0f / l;
    const int qrow = q0 + row;
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) +
                         ((size_t)b * p.n + (size_t)(qrow < p.n ? qrow : 0)) * p.ld_out + head * D;
#pragma unroll
    for (int g = 0; g < D / 32; ++g) {
      uint32_t ov[32];
      tmem_ld32(tm_o + lane_addr + (uint32_t)(g * 32), ov);
      tmem_ld_wait();
      if (qrow < p.n) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint32_t wv[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(ov[u * 8 + 2 * e]) * inv_l,
                                                            __uint_as_float(ov[u * 8 + 2 * e + 1]) * inv_l);
            wv[e] = *reinterpret_cast<const uint32_t*>(&h2);
          }
          *reinterpret_cast<uint4*>(dst + g * 32 + u * 8) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace mri

using namespace mri;

extern "C" int mri_attn_flash_supported(int d) { return (d == 64 || d == 128) ? 1 : 0; }

extern "C" int mri_attn_flash_launch(const MriAttnArgs* a, void* stream) {
  if (a == nullptr || a->qk_map == nullptr || a->vt_map == nullptr || a->out == nullptr)
    return set_error(-1, "mri_attn_flash_launch: null argument");
  if (a->batch < 1 || a->heads < 1 || a->n < 1) return set_error(-2, "mri_attn_flash_launch: empty problem");
  if (a->C != a->heads * a->d) return set_error(-2, "mri_attn_flash_launch: C must be heads * d");
  if (a->ld_out % 8 != 0 || a->ld_out < a->C)
    return set_error(-2, "mri_attn_flash_launch: output rows must hold C channels, 16-byte aligned");
  const int q_tiles = (a->n + kTile - 1) / kTile;
  const long long grid = (long long)q_tiles * a->heads * a->batch;
  if (grid > 0x7fffffffLL) return set_error(-2, "mri_attn_flash_launch: grid too large");
  cudaStream_t st = (cudaStream_t)stream;
  if (a->d == 128) {
    static int configured = 0;
    const int smem = attn_smem_bytes<128>();
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(attn_flash_kernel<128>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(attn_flash_kernel<128>)");
      configured = 1;
    }
    attn_flash_kernel<128><<<(unsigned)grid, kAttnThreads, smem, st>>>(*a);
  } else if (a->d == 64) {
    static int configured = 0;
    const int smem = attn_smem_bytes<64>();
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(attn_flash_kernel<64>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(attn_flash_kernel<64>)");
      configured = 1;
    }
    attn_flash_kernel<64><<<(unsigned)grid, kAttnThreads, smem, st>>>(*a);
  } else {
    return set_error(-2, "mri_attn_flash_launch: head dimension must be 64 or 128");
  }
  return check_launch("attn_flash_kernel");
}
