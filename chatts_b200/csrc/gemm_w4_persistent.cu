// chatts_b200 -- W4A16 GEMM for prefill-sized steps (T > 32) of GPTQ-Int4 checkpoints (README.md:52,262-263):
//     out[T, N] = epilogue(x[T, K] * W[N, K]^T),  W[n][k] = scale[n][k / g] * (q[n][k] - zp[n][k / g])
// It reads the SAME fragment-major 4-bit copy the decode kernel streams (csrc/gemm_w4_mma.cu, weights.py:repack_w4_mma), so a model
// keeps one 4-bit copy for every step size and no dense projection weights at all (ChatTSForCausalLM(..., w4_only=True)).
//
// Structure: the persistent tcgen05 GEMM of gemm_tcgen05.cu (gemm_tn_persistent_kernel) with the weight operand built in shared memory:
//   warp 0      producer (one lane): per 64-K block one cp.async.bulk of the tile's 4 KB of codes (features [0, 128) of a 256-feature chunk
//               are its first 4 KB, so a 128-row MMA tile is one contiguous half-chunk), one of its 512 B of {scale | magic + zp}, and the
//               [256 tokens x 64 K] token tile by TMA (128B swizzle), all onto the stage's `full` barrier
//   warps 6..13 dequantisers: warp w owns m-tile w - 6 (16 rows) of the tile; a lane reads ONE 16-byte word quadruple of codes (its 4 k16
//               steps), converts every pair with the magic-number trick of gemm_w4.cu -- (128 + code) - (128 + zp) is exact, x scale is
//               ONE rounding, i.e. the value dequantize_w4 / dequantize_gptq(scale_dtype = dtype) stores -- and writes 32-bit pairs into
//               the SWIZZLE_128B K-major A tile of the stage (conflict-free: the 8 rows a store instruction touches have 8 different
//               swizzle phases), then arrives on the stage's `ready` barrier
//   warp 1      TMEM allocator + tcgen05.mma issuer: 4 x (M = 128, N = 256, K = 16) per 64-K block into one of two 256-column accumulators
//   warps 2..5  epilogue (warp w reads TMEM lanes 32 (w % 4) ..): NONE (+bias), RESIDUAL (+bias, residual may alias out), SWIGLU_IL (the
//               interleaved gate/up tile: 64 gate rows then the 64 matching up rows -> 64 outputs), PARTIAL_F32 (fp32 [split, t, n])
// Work unit = (128-feature tile, 256-token tile, K split); units are walked in the L2-grouped order of the dense persistent kernel, the
// accumulator is double-buffered, so the epilogue of one unit overlaps the mainloop of the next.
//
// Results are BIT-IDENTICAL to cts_gemm on the dequantised weight: the same 16-bit operand values, the same 64-wide K blocks in the same
// order, the same K = 16 MMAs into an fp32 TMEM accumulator, cts_gemm's K partition of the splits and cts_gemm's epilogue arithmetic.
//
// Amortisation: one dequantised A stage feeds N = 256 tokens (as many as one of the two TMEM accumulators holds).  Per 64-K block a stage
// moves 4.5 KB of codes + 16 KB of A written by the dequantisers + 32 KB of tokens, and the MMA reads 48 KB -- about 10 % more shared
// memory traffic than the dense GEMM's 48 KB in / 48 KB out, for 128 x 256 x 64 MACs (DESIGN.md §4.4 has the measurement).
#include <type_traits>

#include "common.cuh"
#ifndef CTS_DYN_SMEM
#define CTS_DYN_SMEM(name) extern __shared__ __align__(128) uint8_t name[]
#endif
#include "tensormap.cuh"

namespace {

constexpr int kBM = 128, kBK = 64, kUmmaK = 16, kBN = 256;
constexpr int kStages = 4;
constexpr int kEpiWarps = 4, kDqWarps = 8;
constexpr int kThreads = (2 + kEpiWarps + kDqWarps) * 32;
constexpr int kABytes = kBM * kBK * 2;                  // 16 KB dequantised weight tile (MMA operand A)
constexpr int kXBytes = kBN * kBK * 2;                  // 32 KB token tile (operand B)
constexpr int kQBytes = kBM * kBK / 2;                  // 4 KB of codes: half of a fragment-major chunk
constexpr int kSzBytes = kBM * 4;                       // {scale | magic + zp} of the tile's 128 rows for the block's group
constexpr int kStageBytes = kABytes + kXBytes + kQBytes + 1024;   // the scale slot padded to 1 KB: every stage stays 1 KB aligned
constexpr int kChunkBytes = 2 * kQBytes;                // one fragment-major chunk: 256 features x 64 K
constexpr int kSzChunk = 2 * kSzBytes;                  // one szp row: 256 features
constexpr int kXchBytes = 16 * 64 * 2;                  // SWIGLU_IL: 16 tokens x 64 up rows handed to the gate warps

struct W4pParams {
  long long n, k, t, out_ld;
  int kb_total, split_k, group_size, n_groups, tiles_m, tiles_n, group_m, epilogue;
  const uint8_t* qw;
  const uint8_t* szp;
  const void* bias;
  const void* residual;
  void* out;
};

template <typename T> struct Magic4;
template <> struct Magic4<__nv_bfloat16> {
  static constexpr uint32_t kOr = 0x43004300u;          // bf16 128.0 in both halves: 128 + code
  static __device__ __forceinline__ uint32_t cvt(uint32_t codes, uint32_t b2, uint32_t s2) {
    const uint32_t y = codes | kOr;
    __nv_bfloat162 d = __hsub2(*reinterpret_cast<const __nv_bfloat162*>(&y), *reinterpret_cast<const __nv_bfloat162*>(&b2));   // exact small ints
    __nv_bfloat162 w = __hmul2(d, *reinterpret_cast<const __nv_bfloat162*>(&s2));                                              // one rounding
    return *reinterpret_cast<uint32_t*>(&w);
  }
};
template <> struct Magic4<__half> {
  static constexpr uint32_t kOr = 0x64006400u;          // fp16 1024.0: 1024 + code
  static __device__ __forceinline__ uint32_t cvt(uint32_t codes, uint32_t b2, uint32_t s2) {
    const uint32_t y = codes | kOr;
    __half2 d = __hsub2(*reinterpret_cast<const __half2*>(&y), *reinterpret_cast<const __half2*>(&b2));
    __half2 w = __hmul2(d, *reinterpret_cast<const __half2*>(&s2));
    return *reinterpret_cast<uint32_t*>(&w);
  }
};

// unit u -> (feature tile, token tile, split, K blocks [kb0, kb1)); tiles in the L2-grouped order of gemm_tn_persistent_kernel
__device__ __forceinline__ void w4p_unit(const W4pParams& p, int u, int& mb, int& nb, int& split, int& kb0, int& kb1) {
  const int tiles = p.tiles_m * p.tiles_n;
  const int tile = u % tiles;
  split = u / tiles;
  const int per_group = p.group_m * p.tiles_n;
  const int g = tile / per_group, r = tile - g * per_group;
  const int gm_here = min(p.group_m, p.tiles_m - g * p.group_m);
  nb = r / gm_here;
  mb = g * p.group_m + (r - nb * gm_here);
  kb0 = (int)(((long long)p.kb_total * split) / p.split_k);          // cts_gemm's partition (gemm_tcgen05.cu)
  kb1 = (int)(((long long)p.kb_total * (split + 1)) / p.split_k);
}

template <typename T>
__global__ void __launch_bounds__(kThreads, 1)
gemm_w4_prefill_kernel(const __grid_constant__ CUtensorMap tm_x, const W4pParams p) {
  CTS_DYN_SMEM(smem_raw);
  __shared__ uint64_t full_bar[kStages], ready_bar[kStages], empty_bar[kStages], tmem_full[2], tmem_empty[2];
  __shared__ uint32_t tmem_slot;
  constexpr bool kIsBf16 = std::is_same<T, __nv_bfloat16>::value;
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  T* xch = reinterpret_cast<T*>(smem + (size_t)kStages * kStageBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int units = p.tiles_m * p.tiles_n * p.split_k;

  pdl_trigger();
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_x);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&ready_bar[s], kDqWarps);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], kEpiWarps); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(&tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ------------------------------ producer: codes + scales by bulk copy, tokens by TMA ------------------------------
    if (lane == 0) {
      pdl_wait();
      uint32_t it = 0;
      for (int u = blockIdx.x; u < units; u += gridDim.x) {
        int mb, nb, split, kb0, kb1;
        w4p_unit(p, u, mb, nb, split, kb0, kb1);
        const uint8_t* qt = p.qw + (size_t)(mb >> 1) * p.kb_total * kChunkBytes + (size_t)(mb & 1) * kQBytes;
        const uint8_t* zt = p.szp + (size_t)(mb >> 1) * p.n_groups * kSzChunk + (size_t)(mb & 1) * kSzBytes;
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = (int)(it % kStages);
          mbar_wait(&empty_bar[s], ((it / kStages) & 1u) ^ 1u);
          mbar_expect_tx(&full_bar[s], (uint32_t)(kXBytes + kQBytes + kSzBytes));
          uint8_t* st = smem + (size_t)s * kStageBytes;
          bulk_load_1d(st + kABytes + kXBytes, qt + (size_t)kb * kChunkBytes, (uint32_t)kQBytes, &full_bar[s]);
          bulk_load_1d(st + kABytes + kXBytes + kQBytes, zt + (size_t)((kb * kBK) / p.group_size) * kSzChunk, (uint32_t)kSzBytes, &full_bar[s]);
          tma_load_2d(st + kABytes, &tm_x, &full_bar[s], kb * kBK, nb * kBN, CTS_L2_EVICT_NORMAL);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer ------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(kIsBf16 ? 1 : 0, kBN, kBM);
      uint32_t it = 0, lt = 0;
      for (int u = blockIdx.x; u < units; u += gridDim.x, ++lt) {
        int mb, nb, split, kb0, kb1;
        w4p_unit(p, u, mb, nb, split, kb0, kb1);
        const uint32_t buf = lt & 1u;
        mbar_wait(&tmem_empty[buf], ((lt >> 1) & 1u) ^ 1u);           // the epilogue has drained this accumulator
        tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = (int)(it % kStages);
          const uint32_t ph = (it / kStages) & 1u;
          mbar_wait(&full_bar[s], ph);                                 // token tile landed
          mbar_wait(&ready_bar[s], ph);                                // weight tile dequantised
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + (size_t)s * kStageBytes);
          const uint64_t a_desc = umma_desc_k_sw128(a_addr), b_desc = umma_desc_k_sw128(a_addr + kABytes);
#pragma unroll
          for (int kk = 0; kk < kBK / kUmmaK; ++kk) {
            const uint64_t adv = (uint64_t)(kk * ((kUmmaK * 2) >> 4));
            umma_f16(tmem_base + buf * kBN, a_desc + adv, b_desc + adv, idesc, (kb > kb0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tmem_full[buf]);
      }
    }
  } else if (warp >= 2 + kEpiWarps) {
    // ------------------------------ dequantisers: codes -> the swizzled K-major A tile ------------------------------
    const int wq = warp - 2 - kEpiWarps;                               // m-tile of the 128-row tile: rows 16 wq .. 16 wq + 15
    const int g = lane >> 2, tq = lane & 3;
    const int r0 = wq * 16 + g;                                        // fragment rows g / g + 8; both have swizzle phase g
    uint32_t it = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      int mb, nb, split, kb0, kb1;
      w4p_unit(p, u, mb, nb, split, kb0, kb1);
      for (int kb = kb0; kb < kb1; ++kb, ++it) {
        const int s = (int)(it % kStages);
        mbar_wait(&full_bar[s], (it / kStages) & 1u);
        uint8_t* st = smem + (size_t)s * kStageBytes;
        const uint4 wv = *reinterpret_cast<const uint4*>(st + kABytes + kXBytes + (wq * 32 + lane) * 16);
        const uint32_t z0 = *reinterpret_cast<const uint32_t*>(st + kABytes + kXBytes + kQBytes + r0 * 4);
        const uint32_t z1 = *reinterpret_cast<const uint32_t*>(st + kABytes + kXBytes + kQBytes + (r0 + 8) * 4);
        const uint32_t s2lo = (z0 & 0xFFFFu) * 0x00010001u, s2hi = (z1 & 0xFFFFu) * 0x00010001u;   // scale in both halves
        const uint32_t b2lo = (z0 >> 16) * 0x00010001u, b2hi = (z1 >> 16) * 0x00010001u;           // magic + zp in both halves
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint32_t w = ks == 0 ? wv.x : ks == 1 ? wv.y : ks == 2 ? wv.z : wv.w;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            // (w >> 4j) & 0x000F000F = codes at k = 16 ks + 8 (j / 2) + 2 tq + {0, 1} of row r0 + 8 (j % 2): 16-byte chunk 2 ks + j / 2
            const int hi = j & 1;
            const uint32_t v = Magic4<T>::cvt((w >> (4 * j)) & 0x000F000Fu, hi ? b2hi : b2lo, hi ? s2hi : s2lo);
            const int r = r0 + 8 * hi;
            *reinterpret_cast<uint32_t*>(st + r * 128 + (((2 * ks + (j >> 1)) ^ g) << 4) + 4 * tq) = v;
          }
        }
        fence_proxy_async_smem();                                      // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(&ready_bar[s]);
      }
    }
  } else {
    // ------------------------------ epilogue warps ------------------------------
    pdl_wait();                                                        // residual / out belong to the predecessor until now
    const int q = warp & 3;
    const int ft = q * 32 + lane;                                      // row of the weight tile == TMEM lane
    const int epi = p.epilogue;
    uint32_t lt = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x, ++lt) {
      int mb, nb, split, kb0, kb1;
      w4p_unit(p, u, mb, nb, split, kb0, kb1);
      const long long f0 = (long long)mb * kBM, t0 = (long long)nb * kBN;
      const long long f = f0 + ft;
      const bool f_ok = f < p.n;
      const uint32_t buf = lt & 1u;
      float bias = 0.f;
      if (p.bias != nullptr && f_ok) bias = DT<T>::to_f(reinterpret_cast<const T*>(p.bias)[f]);
      mbar_wait(&tmem_full[buf], (lt >> 1) & 1u);
      tc_fence_after();
      const uint32_t lane_addr = tmem_base + buf * kBN + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < kBN; c += 16) {
        if (t0 + c >= p.t) break;                                      // CTA-uniform
        uint32_t v[16];
        tmem_ld_32x32b_x16(lane_addr + (uint32_t)c, v);
        tmem_ld_wait();
        if (epi == CTS_EPI_PARTIAL_F32) {
          float* dst = reinterpret_cast<float*>(p.out) + (long long)split * p.t * p.n;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const long long t = t0 + c + j;
            if (t < p.t && f_ok) dst[t * p.n + f] = __uint_as_float(v[j]);
          }
        } else if (epi == CTS_EPI_SWIGLU_IL) {
          if (ft >= 64) {                                              // "up" rows: hand dtype(u) to the gate warps
#pragma unroll
            for (int j = 0; j < 16; ++j) xch[j * 64 + (ft - 64)] = DT<T>::from_f(__uint_as_float(v[j]));
          }
          named_bar_sync(1, kEpiWarps * 32);
          if (ft < 64) {
            T* o = reinterpret_cast<T*>(p.out);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const long long t = t0 + c + j;
              if (t >= p.t) continue;
              const float gv = rnd<T>(__uint_as_float(v[j]));
              const float uv = DT<T>::to_f(xch[j * 64 + ft]);
              o[t * p.out_ld + f0 / 2 + ft] = DT<T>::from_f(rnd<T>(silu_f(gv)) * uv);
            }
          }
          named_bar_sync(1, kEpiWarps * 32);                           // the exchange buffer is rewritten by the next chunk
        } else {
          T* o = reinterpret_cast<T*>(p.out);
          const T* res = reinterpret_cast<const T*>(p.residual);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const long long t = t0 + c + j;
            if (t >= p.t || !f_ok) continue;
            float r = __uint_as_float(v[j]) + bias;
            if (epi == CTS_EPI_RESIDUAL) r = rnd<T>(r) + DT<T>::to_f(res[t * p.out_ld + f]);   // read before the write: res may alias out
            o[t * p.out_ld + f] = DT<T>::from_f(r);
          }
        }
      }
      tc_fence_before();                                               // last TMEM read of this accumulator: hand it back to the MMA warp
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem_base);
}

template <typename T>
int launch_w4p(cts_ctx* ctx, const cts_gemm_w4p_args* a, cudaStream_t stream) {
  CUtensorMap tm_x;
  int rc = cts_make_tmap_2d(ctx, &tm_x, a->x, a->t, a->k, a->x_ld, kBN, a->dtype == CTS_BF16);
  if (rc) return rc;
  W4pParams p;
  p.n = a->n; p.k = a->k; p.t = a->t; p.out_ld = a->out_ld;
  p.kb_total = (int)(a->k / kBK);
  p.split_k = a->split_k; p.group_size = a->group_size; p.n_groups = (int)(a->k / a->group_size);
  p.tiles_m = (int)cdiv_ll(a->n, kBM); p.tiles_n = (int)cdiv_ll(a->t, kBN);
  p.epilogue = a->epilogue;
  p.qw = (const uint8_t*)a->qw; p.szp = (const uint8_t*)a->szp;
  p.bias = a->bias; p.residual = a->residual; p.out = a->out;
  {
    // feature tiles per L2 group: the group's codes (128 rows x K / 2 bytes per tile) within ~48 MB, balanced over the groups -- DRAM then
    // sees the weights once and the tokens once per group, as in the dense persistent GEMM
    long long gmax = (48LL << 20) / ((long long)kBM * a->k / 2);
    if (gmax < 1) gmax = 1;
    const long long groups = cdiv_ll(p.tiles_m, gmax);
    p.group_m = (int)cdiv_ll(p.tiles_m, groups);
  }
  const size_t smem = (size_t)kStages * kStageBytes + kXchBytes + 1024;
  auto kern = gemm_w4_prefill_kernel<T>;
  CTS_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long units = (long long)p.tiles_m * p.tiles_n * p.split_k;
  const unsigned grid = (unsigned)(units < ctx->sm_count ? units : ctx->sm_count);
  CTS_CUDA(ctx, launch_pdl(kern, dim3(grid), dim3(kThreads), smem, stream, 1, tm_x, p));
  return CTS_OK;
}

}  // namespace

extern "C" int cts_gemm_w4_prefill(cts_ctx* ctx, const cts_gemm_w4p_args* a, void* stream) {
  if (!ctx) return CTS_ERR_BAD_ARG;
  CTS_CHECK_ARG(ctx, a != nullptr && a->qw && a->szp && a->x && a->out, "null pointer");
  CTS_CHECK_ARG(ctx, a->n > 0 && a->k > 0 && a->t > 0, "n, k, t must be positive");
  CTS_CHECK_ARG(ctx, a->dtype == CTS_BF16 || a->dtype == CTS_F16, "dtype must be CTS_BF16 or CTS_F16");
  CTS_CHECK_ARG(ctx, a->k % 128 == 0, "k must be a multiple of 128");
  CTS_CHECK_ARG(ctx, a->group_size >= 64 && a->k % a->group_size == 0 && (a->group_size == 64 || a->group_size % 128 == 0),
                "group_size must be 64 or a multiple of 128, and divide k");
  CTS_CHECK_ARG(ctx, a->epilogue == CTS_EPI_NONE || a->epilogue == CTS_EPI_RESIDUAL || a->epilogue == CTS_EPI_SWIGLU_IL ||
                         a->epilogue == CTS_EPI_PARTIAL_F32,
                "epilogue must be CTS_EPI_NONE, CTS_EPI_RESIDUAL, CTS_EPI_SWIGLU_IL or CTS_EPI_PARTIAL_F32");
  CTS_CHECK_ARG(ctx, a->split_k >= 1 && a->split_k <= a->k / kBK, "split_k must be in [1, k / 64]");
  CTS_CHECK_ARG(ctx, a->split_k == 1 || a->epilogue == CTS_EPI_PARTIAL_F32, "split_k > 1 needs CTS_EPI_PARTIAL_F32");
  CTS_CHECK_ARG(ctx, a->bias == nullptr || a->epilogue == CTS_EPI_NONE || a->epilogue == CTS_EPI_RESIDUAL,
                "bias is applied by CTS_EPI_NONE and CTS_EPI_RESIDUAL only");
  CTS_CHECK_ARG(ctx, a->epilogue != CTS_EPI_RESIDUAL || a->residual != nullptr, "CTS_EPI_RESIDUAL needs residual");
  CTS_CHECK_ARG(ctx, a->x_ld >= a->k && a->x_ld % 8 == 0 && ((uintptr_t)a->x & 15) == 0, "x_ld must be >= k and x rows 16-byte aligned");
  CTS_CHECK_ARG(ctx, (((uintptr_t)a->qw | (uintptr_t)a->szp) & 15) == 0, "qw / szp must be 16-byte aligned");
  CTS_CHECK_ARG(ctx, a->epilogue == CTS_EPI_PARTIAL_F32 || a->out_ld >= (a->epilogue == CTS_EPI_SWIGLU_IL ? a->n / 2 : a->n),
                "out_ld smaller than the output width");
  CTS_CHECK_ARG(ctx, a->epilogue != CTS_EPI_SWIGLU_IL || (a->n % 128 == 0 && a->t > 128),
                "CTS_EPI_SWIGLU_IL needs n % 128 == 0 and t > 128 (small t: CTS_EPI_PARTIAL_F32 + cts_reduce_swiglu)");
  CTS_CHECK_ARG(ctx, cdiv_ll(a->n, kBM) * cdiv_ll(a->t, kBN) * a->split_k < (1LL << 31) && a->k / kBK < (1LL << 24), "problem too large");
  cudaStream_t st = (cudaStream_t)stream;
  return a->dtype == CTS_BF16 ? launch_w4p<__nv_bfloat16>(ctx, a, st) : launch_w4p<__half>(ctx, a, st);
}
