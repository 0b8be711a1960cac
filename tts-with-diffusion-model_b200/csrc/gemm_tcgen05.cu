// out = epilogue(A[M,K] · W[N,K]^T): the linear layers of the denoiser (SURVEY.md §8a rows A1,
// F1, H1; reference base.py:110,129,209-214,355).
//
// Persistent, warp-specialised sm_100a kernel:
//   warp 0 lane 0 : TMA producer   (cp.async.bulk.tensor 2D, SWIZZLE_128B, 4-stage ring)
//   warp 1 lane 0 : MMA issuer     (tcgen05.mma cta_group::1 kind::f16, 128x256x16, fp32 in TMEM)
//   warps 2..9    : epilogue       (tcgen05.ld -> bias / GELU -> swizzled smem -> TMA store, or
//                                   TMA reduce-add into the fp32 residual stream)
// TMEM holds two 128x256 fp32 accumulators (512 columns) so the epilogue of tile i overlaps the
// MMAs of tile i+1.  Both operands are K-major (nn.Linear stores W as (N, K)), so no transposes.
// Output never leaves the SM through per-thread stores: each epilogue warp writes 32 rows x 128 B
// into its own SWIZZLE_128B staging tile and one lane hands it to the TMA engine, which clips the
// M / N tails and, for BIAS_RESIDUAL, performs out += tile at L2 (no read of the residual by SMs).
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

#ifndef VB200_GEMM_BIAS_PREFETCH
#define VB200_GEMM_BIAS_PREFETCH 1
#endif
#ifndef VB200_GEMM_EARLY_LOAD
#define VB200_GEMM_EARLY_LOAD 1
#endif

namespace vb200 {

namespace gemm {
constexpr int BM = 128, BK = 64;   // BN (256, or 128 for small problems) is a kernel template parameter
constexpr int A_BYTES = BM * BK * 2;            // 16 KB
// CTAS = 1: one CTA per 128x256 tile, stage = A 16 KB + W 32 KB, 4 stages.
// CTAS = 2: a CTA pair (cluster of 2, cta_group::2) per 256x256 tile; each CTA stages its own 128
//           rows of A and HALF of the W tile (128 rows), 32 KB per stage, 6 stages.  The pair's
//           tensor cores read both halves, which halves every SM's shared-memory operand traffic —
//           measured necessary: a lone CTA sustains 163 cycles per 128x256x16 MMA against 128 nominal.
// CTAS = 1, BN = 128: narrow tiles for problems with fewer 128x256 tiles than SMs (one utterance
//           at a time: M ~ 1000) — twice the CTAs, 32 KB stages, 6 stages.
template <int CTAS, int BN> struct Cfg {
  static constexpr int B_ROWS = BN / CTAS;
  static constexpr int B_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (4 * 48 * 1024) / STAGE_BYTES;   // 4 x 48 KB, 4 x 40 KB (BN = 192), 6 x 32 KB, 8 x 24 KB
};
constexpr int EPI_WARPS = 8;
constexpr int THREADS = (2 + EPI_WARPS) * 32;   // 320
constexpr int EPI_TILE_BYTES = 32 * 128;        // 32 rows x 128 B per epilogue warp
constexpr int SMEM_BYTES = 4 * 48 * 1024 + EPI_WARPS * EPI_TILE_BYTES + 1024 /*align slack*/ +
                           256 /*barriers*/;     // 4 x 48 KB == 6 x 32 KB
constexpr uint32_t TMEM_COLS = 512;
}  // namespace gemm

// gelu(x) = 0.5 x (1 + erf(x / sqrt 2)) = x * (x > 0 ? 1 - q : q),  q(z) = 0.5 erfc(z),  z = |x| / sqrt 2.
// log2 q(z) is smooth: a degree-6 minimax polynomial on [0, 6] gives |gelu error| < 4.5e-5 for all x
// (beyond z = 6, i.e. |x| > 8.5, q < 1e-17); one MUFU (ex2) per element.
// Two elements at once with packed f32x2 arithmetic (FFMA2: half the issue slots of the polynomial),
// written as gelu(x) = x * (0.5 + copysign(0.5 - q, x)).  With a scalar form (12 instructions per
// element) the epilogue of the FFN1 GEMM (K = 1024) took longer than the tile's MMAs (tensor pipe
// 86 % active).
__device__ __forceinline__ void gelu_erf_fast2(float& x0, float& x1) {
  const float z0 = fminf(fabsf(x0) * 0.70710678118654752f, 6.0f);
  const float z1 = fminf(fabsf(x1) * 0.70710678118654752f, 6.0f);
  const uint64_t z = pack2(z0, z1);
  uint64_t p = ffma2(z, pack2(9.22344479e-05f, 9.22344479e-05f), pack2(-2.20238999e-03f, -2.20238999e-03f));
  p = ffma2(z, p, pack2(2.23510694e-02f, 2.23510694e-02f));
  p = ffma2(z, p, pack2(-1.29628107e-01f, -1.29628107e-01f));
  p = ffma2(z, p, pack2(-9.38564420e-01f, -9.38564420e-01f));
  p = ffma2(z, p, pack2(-1.62045550e+00f, -1.62045550e+00f));
  p = ffma2(z, p, pack2(-1.00044155e+00f, -1.00044155e+00f));
  float p0, p1, q0, q1, h0, h1;
  unpack2(p, p0, p1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(q0) : "f"(p0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(q1) : "f"(p1));
  unpack2(ffma2(pack2(q0, q1), pack2(-1.0f, -1.0f), pack2(0.5f, 0.5f)), h0, h1);   // 0.5 - q >= 0
  h0 = __uint_as_float(__float_as_uint(h0) | (__float_as_uint(x0) & 0x80000000u));
  h1 = __uint_as_float(__float_as_uint(h1) | (__float_as_uint(x1) & 0x80000000u));
  const uint64_t s = fadd2(pack2(h0, h1), pack2(0.5f, 0.5f));
  unpack2(ffma2(pack2(x0, x1), s, 0ull), x0, x1);
}

template <int EPI, typename OutT, int CTAS, int BN>
__global__ void __launch_bounds__(gemm::THREADS, 1) gemm_tcgen05_kernel(
    const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
    const __grid_constant__ CUtensorMap tm_out, const float* __restrict__ bias, int M, int N, int K,
    uint32_t a_is_f16) {
  using namespace gemm;
  using C = Cfg<CTAS, BN>;
  constexpr int STAGES = C::STAGES, STAGE_BYTES = C::STAGE_BYTES, B_ROWS = C::B_ROWS;
  constexpr int HALF_COLS = BN / 2;            // accumulator columns per epilogue warp
  const uint32_t cta_rank = CTAS == 2 ? cluster_ctarank() : 0;       // 0 = leader of the pair
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = ((raw_addr + 1023u) & ~1023u) - raw_addr;
  uint8_t* smem = smem_raw + pad;                      // 1024-byte aligned (SWIZZLE_128B atoms)
  uint8_t* epi_smem = smem + STAGES * STAGE_BYTES;     // EPI_WARPS x 4 KB, each 1024-aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem + EPI_WARPS * EPI_TILE_BYTES);
  uint64_t* full = bars;                 // [STAGES]  TMA -> MMA
  uint64_t* empty = bars + STAGES;       // [STAGES]  MMA -> TMA
  uint64_t* acc_full = bars + 2 * STAGES;   // [2]     MMA -> epilogue
  uint64_t* acc_empty = acc_full + 2;       // [2]     epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  // a "tile" is BM * CTAS rows; the CTAs of a pair take consecutive 128-row halves of it
  const int num_m = (M + BM * CTAS - 1) / (BM * CTAS), num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + BK - 1) / BK;
  const int tile0 = blockIdx.x / CTAS, tile_stride = gridDim.x / CTAS;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    tma_prefetch_desc(&tm_out);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], EPI_WARPS * CTAS); }
    fence_barrier_init();
#if VB200_GEMM_EARLY_LOAD
    // single-CTA kernels: the first ring's worth of loads of this CTA's first tile goes out before
    // the block-wide sync below (TMEM allocation): the first TMA round trip is on the critical path
    // of the one-wave launches of a single utterance
    if (CTAS == 1 && tile0 < num_tiles) {
      // With programmatic dependent launch (VB200_PDL & 4 / 8) this CTA may be resident while the previous
      // kernel still runs: the WEIGHT halves of the first ring (static data) go out at once, the activation
      // halves once the previous kernel has completed.
      pdl_launch_dependents();
      const int m_row = (tile0 / num_n) * BM, n_row = (tile0 % num_n) * BN;
      const int n_pre = num_kb < STAGES ? num_kb : STAGES;
      for (int kb = 0; kb < n_pre; ++kb) {
        mbar_arrive_expect_tx(&full[kb], STAGE_BYTES);
        tma_load_2d(smem + kb * STAGE_BYTES + A_BYTES, &tm_b, &full[kb], kb * BK, n_row);
      }
      pdl_wait();                                   // A is an earlier kernel's output
      for (int kb = 0; kb < n_pre; ++kb) tma_load_2d(smem + kb * STAGE_BYTES, &tm_a, &full[kb], kb * BK, m_row);
    }
#endif
  }
  if (warp == 1) {
    if (CTAS == 2) { tmem_alloc_pair(tmem_slot, TMEM_COLS); tmem_relinquish_pair(); }
    else { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  }
  tc_fence_before();
  if (CTAS == 2) cluster_sync_all(); else __syncthreads();   // barriers of both CTAs initialised
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: the prologue above (barriers, TMEM, tensor-map prefetch) overlapped the previous kernel's
  // tail; A, the residual stream and `out` may only be touched from here on.
  pdl_launch_dependents();
  pdl_wait();

  // Both control warps run their loops warp-uniformly (all lanes compute the same addresses, one
  // elected lane executes the TMA / MMA / commit instructions): issuing from a divergent
  // `if (lane == 0)` region makes the compiler wrap every tcgen05.mma in an elect / R2UR loop.
  if (warp == 0) {
    {
      // ------------------------------------------------------------ TMA producer
      const bool leader = elect_one();
      int stage = 0; uint32_t phase = 0;
      int kb0 = 0;
#if VB200_GEMM_EARLY_LOAD
      if (CTAS == 1) {                              // the prologue already requested these k-blocks
        kb0 = num_kb < STAGES ? num_kb : STAGES;
        if (kb0 == STAGES) phase = 1; else stage = kb0;
      }
#endif
      for (int tile = tile0; tile < num_tiles; tile += tile_stride) {
        const int m_blk = tile / num_n, n_blk = tile % num_n;
        const int m_row = (m_blk * CTAS + cta_rank) * BM, n_row = n_blk * BN + cta_rank * B_ROWS;
        for (int kb = kb0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          if (leader) {
            if (CTAS == 2) {
              // both CTAs' bytes are counted on the leader CTA's barrier
              if (cta_rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * STAGE_BYTES);
              tma_load_2d_pair(sa, &tm_a, &full[stage], kb * BK, m_row);
              tma_load_2d_pair(sa + A_BYTES, &tm_b, &full[stage], kb * BK, n_row);
            } else {
              mbar_arrive_expect_tx(&full[stage], STAGE_BYTES);
              tma_load_2d(sa, &tm_a, &full[stage], kb * BK, m_row);
              tma_load_2d(sa + A_BYTES, &tm_b, &full[stage], kb * BK, n_row);
            }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        kb0 = 0;
      }
    }
  } else if (warp == 1) {
    if (cta_rank == 0) {
      // ------------------------------------------------------------ MMA issuer (leader CTA of a pair)
      const bool leader = elect_one();
      // A (activations) and B (weights) are both bf16 or both fp16 (run-time)
      const uint32_t idesc = umma_idesc_bf16(BM * CTAS, BN, false, false) & ~(a_is_f16 ? kIdescBf16 : 0u);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int tile = tile0; tile < num_tiles; tile += tile_stride, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&acc_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint64_t da = umma_desc_kmajor_sw128(sa);
          const uint64_t db = umma_desc_kmajor_sw128(sa + A_BYTES);
          if (leader) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) { // +32 bytes (>>4 = 2) per UMMA_K inside the swizzle atom
              if (CTAS == 2) umma_ss_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
              else umma_ss(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            }
            if (CTAS == 2) umma_commit_pair(&empty[stage]);   // frees the slot in both CTAs
            else umma_commit(&empty[stage]);    // frees the smem slot once these MMAs retire
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (leader) {                           // accumulator complete -> epilogue (of both CTAs)
          if (CTAS == 2) umma_commit_pair(&acc_full[as]); else umma_commit(&acc_full[as]);
        }
        __syncwarp();
      }
    }
  } else {
    // -------------------------------------------------------------- epilogue warps
    const int e = warp - 2;
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int half = e >> 2;                   // which half of the BN accumulator columns
    uint8_t* stage_tile = epi_smem + e * EPI_TILE_BYTES;
    uint8_t* my_row = stage_tile + lane * 128;
    const int sw = lane & 7;                   // SWIZZLE_128B: 16-byte chunk index ^= row % 8
    constexpr bool kWide = sizeof(OutT) == 4;  // fp32: 32 columns per 128-byte row, else 64
    constexpr int CHUNK_COLS = kWide ? 32 : 64;
    // columns of the tile handled by this half of the epilogue warps: BN / 2 each, except BN = 192 (not a
    // multiple of 2 x 64): 128 + 64
    constexpr int HALF0_COLS = BN == 192 ? 128 : HALF_COLS;
    const int col_base = half * HALF0_COLS;
    const int n_chunks = (half == 0 ? HALF0_COLS : BN - HALF0_COLS) / CHUNK_COLS;
    const bool epi_leader = elect_one();       // the lane that owns this warp's bulk-store group
    int it = 0;
    for (int tile = tile0; tile < num_tiles; tile += tile_stride, ++it) {
      const int m_blk = tile / num_n, n_blk = tile % num_n;
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      if (EPI != VB200_EPI_NONE && VB200_GEMM_BIAS_PREFETCH) {
        // this warp's slice of the bias into L1 while the accumulator is still being computed: in a one-tile
        // launch (one utterance) the first __ldg below is otherwise an exposed L2 round trip per GEMM
        const int nb0 = n_blk * BN + col_base + lane * 32;
        if (lane * 32 < n_chunks * CHUNK_COLS && nb0 < N) prefetch_l1(bias + nb0);
      }
      mbar_wait(&acc_full[as], aphase);
      tc_fence_after();
      const int row0 = (m_blk * CTAS + cta_rank) * BM + quad * 32;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN + col_base;
#pragma unroll 1
      for (int c = 0; c < n_chunks; ++c) {
        const int n0 = n_blk * BN + col_base + c * CHUNK_COLS;
        if (epi_leader) tma_store_wait_read();  // previous store has finished reading the staging tile
        __syncwarp();
#pragma unroll
        for (int sub = 0; sub < CHUNK_COLS / 32; ++sub) {
          uint32_t r[32];
          tmem_ld_32x32(t_row + c * CHUNK_COLS + sub * 32, r);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
          const int nb = n0 + sub * 32;
          if (EPI != VB200_EPI_NONE) {
            if (nb + 32 <= N) {
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + nb + i));
                unpack2(fadd2(pack2(v[i], v[i + 1]), pack2(b4.x, b4.y)), v[i], v[i + 1]);
                unpack2(fadd2(pack2(v[i + 2], v[i + 3]), pack2(b4.z, b4.w)), v[i + 2], v[i + 3]);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) if (nb + i < N) v[i] += __ldg(bias + nb + i);
            }
          }
          if (EPI == VB200_EPI_BIAS_GELU) {
#pragma unroll
            for (int i = 0; i < 32; i += 2) gelu_erf_fast2(v[i], v[i + 1]);
          }
          if (kWide) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<float4*>(my_row + ((q ^ sw) << 4)) =
                  make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          } else {
            constexpr bool is_bf16 = std::is_same<OutT, __nv_bfloat16>::value;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              uint4 p;
              if (is_bf16) {
                p.x = pack_bf16x2(v[8 * q], v[8 * q + 1]); p.y = pack_bf16x2(v[8 * q + 2], v[8 * q + 3]);
                p.z = pack_bf16x2(v[8 * q + 4], v[8 * q + 5]); p.w = pack_bf16x2(v[8 * q + 6], v[8 * q + 7]);
              } else {
                p.x = pack_f16x2(v[8 * q], v[8 * q + 1]); p.y = pack_f16x2(v[8 * q + 2], v[8 * q + 3]);
                p.z = pack_f16x2(v[8 * q + 4], v[8 * q + 5]); p.w = pack_f16x2(v[8 * q + 6], v[8 * q + 7]);
              }
              *reinterpret_cast<uint4*>(my_row + (((sub * 4 + q) ^ sw) << 4)) = p;
            }
          }
        }
        fence_proxy_async_smem();              // generic-proxy smem writes -> visible to the TMA engine
        __syncwarp();
        if (epi_leader && row0 < M && n0 < N) {
          if (EPI == VB200_EPI_BIAS_RESIDUAL) tma_reduce_add_2d(&tm_out, stage_tile, n0, row0);
          else tma_store_2d(&tm_out, stage_tile, n0, row0);
          tma_store_commit();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {                                // one arrival per epilogue warp, on the leader's barrier
        if (CTAS == 2 && cta_rank != 0) mbar_arrive_remote(&acc_empty[as], 0);
        else mbar_arrive(&acc_empty[as]);
      }
    }
    if (epi_leader) tma_store_wait_all();
  }

  tc_fence_before();
  if (CTAS == 2) cluster_sync_all(); else __syncthreads();   // nobody leaves while the peer still uses it
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    if (CTAS == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS); else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------- host side
template <int EPI, typename OutT>
static int launch_gemm(void* out, vb200_dtype dt, const void* A, vb200_dtype a_dt, const void* W, const float* bias,
                       int M, int N, int K, cudaStream_t st) {
  const uint32_t a_f16 = a_dt == VB200_F16 ? 1u : 0u;
  using namespace gemm;
  PdlTag pdl_tag(EPI == VB200_EPI_BIAS_RESIDUAL ? 8 : 4);
  // Four tilings, picked by estimated cycles = waves x k-steps x cycles per MMA (tools/mma_bench.cu):
  //   CTA pair 256x256 (~135 cycles per k-step, half as many schedulable units, + ~5 000 cycles per
  //   launch: cluster scheduling, pair TMEM allocation, two cluster-wide syncs — measured with
  //   tools/gemm_small_probe.py, it only matters for one or two utterances at a time),
  //   one CTA 128x256 (~163), one CTA 128x128 (~99, twice the tiles),
  //   one CTA 128x64 (~75; fp32 outputs only: the two residual GEMMs) when even the 128-wide tiling
  //   leaves SMs idle (one utterance: 72 tiles) — twice the CTAs each pull 3/4 of the operand bytes,
  //   and a single-wave launch is bound by how fast an SM ingests operands from L2 (~60 B/clk).
  constexpr int BN = 256;
  const int sms = num_sms(), mt = (M + BM - 1) / BM, nn = (N + BN - 1) / BN;
  const long ksteps = static_cast<long>((K + BK - 1) / BK) * (BK / 16);
  auto waves = [](long tiles, long units) { return (tiles + units - 1) / units; };
  const long t_wide = waves(static_cast<long>(mt) * nn, sms) * ksteps * 163;
  const long t_pair = waves(static_cast<long>((M + 2 * BM - 1) / (2 * BM)) * nn, sms / 2) * ksteps * 135 + 5000;
  const long t_narrow = N > 128 ? waves(static_cast<long>(mt) * ((N + 127) / 128), sms) * ksteps * 99 : (1l << 60);
  const long t_n64 = (sizeof(OutT) == 4 && N > 64) ? waves(static_cast<long>(mt) * ((N + 63) / 64), sms) * ksteps * 75
                                                   : (1l << 60);
  // one CTA 128x192 (~130): only as a ONE-wave launch of a bf16 / fp16 output whose N it divides — QKV of one
  // utterance: 9 x 16 = 144 tiles on 148 SMs, 640 KB of operands per CTA, against 108 tiles of 768 KB
  const long tiles_192 = static_cast<long>(mt) * (N / 192);
  const long t_n192 = (sizeof(OutT) == 2 && N % 192 == 0 && tiles_192 <= sms) ? ksteps * 130 : (1l << 60);
  int ctas = t_pair <= t_wide ? 2 : 1;
  bool narrow = false, narrow64 = false, n192 = false;
  long best = ctas == 2 ? t_pair : t_wide;
  if (t_narrow < best) { ctas = 1; narrow = true; best = t_narrow; }
  if (t_n64 < best) { ctas = 1; narrow = false; narrow64 = true; best = t_n64; }
  if (t_n192 < best) { ctas = 1; narrow = false; narrow64 = false; n192 = true; best = t_n192; }
  // VB200_GEMM_TILE=pair|wide|narrow|n64|n192 forces a tiling (A/B measurements, tools/gemm_small_probe.py, and
  // the per-tiling tests); where the forced tiling cannot apply, the 128x256 one runs instead
  static int tile_forced = -1;
  if (tile_forced < 0) {
    const char* e = getenv("VB200_GEMM_TILE");
    tile_forced = !e ? 0 : e[0] == 'p' ? 1 : e[0] == 'w' ? 2 : (e[0] == 'n' && e[1] == 'a') ? 3
                : (e[0] == 'n' && e[1] == '6') ? 4 : (e[0] == 'n' && e[1] == '1') ? 5 : 0;
  }
  if (tile_forced) {
    ctas = tile_forced == 1 ? 2 : 1;
    narrow = tile_forced == 3 && N > 128;
    narrow64 = tile_forced == 4 && sizeof(OutT) == 4 && N > 64;
    n192 = tile_forced == 5 && sizeof(OutT) == 2 && N % 192 == 0;
  }
  const int bn = n192 ? 192 : narrow64 ? 64 : (narrow ? 128 : BN);
  CUtensorMap ta, tb, tout;
  int rc = cached_tmap(&ta, a_dt, A, K, M, static_cast<uint64_t>(K) * 2, BK, BM);
  if (rc != VB200_OK) return rc;
  rc = cached_tmap(&tb, a_dt, W, K, N, static_cast<uint64_t>(K) * 2, BK, bn / ctas);
  if (rc != VB200_OK) return rc;
  const int esz = sizeof(OutT);   // store box: 32 rows x 128 bytes
  rc = cached_tmap(&tout, dt, out, N, M, static_cast<uint64_t>(N) * esz, 128 / esz, 32);
  if (rc != VB200_OK) return rc;
  const int tiles = ((M + BM * ctas - 1) / (BM * ctas)) * ((N + bn - 1) / bn);
  const int groups = num_sms() / ctas;
  const int grid = (tiles < groups ? tiles : groups) * ctas;
  if (n192) {
    if constexpr (sizeof(OutT) == 2) {
      auto kern = gemm_tcgen05_kernel<EPI, OutT, 1, 192>;
      VB_CONFIGURE_SMEM(kern, SMEM_BYTES);
      VB_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 1, ta, tb, tout, bias, M, N, K, a_f16));
    }
  } else if (narrow64) {
    if constexpr (sizeof(OutT) == 4) {
      auto kern = gemm_tcgen05_kernel<EPI, OutT, 1, 64>;
      VB_CONFIGURE_SMEM(kern, SMEM_BYTES);
      VB_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 1, ta, tb, tout, bias, M, N, K, a_f16));
    }
  } else if (narrow) {
    auto kern = gemm_tcgen05_kernel<EPI, OutT, 1, 128>;
    VB_CONFIGURE_SMEM(kern, SMEM_BYTES);
    VB_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 1, ta, tb, tout, bias, M, N, K, a_f16));
  } else if (ctas == 1) {
    auto kern = gemm_tcgen05_kernel<EPI, OutT, 1, 256>;
    VB_CONFIGURE_SMEM(kern, SMEM_BYTES);
    VB_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 1, ta, tb, tout, bias, M, N, K, a_f16));
  } else {
    auto kern = gemm_tcgen05_kernel<EPI, OutT, 2, 256>;
    VB_CONFIGURE_SMEM(kern, SMEM_BYTES);
    VB_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 2, ta, tb, tout, bias, M, N, K, a_f16));
  }
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

template <int EPI>
static int launch_gemm_dtype(void* out, vb200_dtype dt, const void* A, vb200_dtype a_dt, const void* W,
                             const float* bias, int M, int N, int K, cudaStream_t st) {
  switch (dt) {
    case VB200_F32: return launch_gemm<EPI, float>(out, dt, A, a_dt, W, bias, M, N, K, st);
    case VB200_BF16: return launch_gemm<EPI, __nv_bfloat16>(out, dt, A, a_dt, W, bias, M, N, K, st);
    case VB200_F16: return launch_gemm<EPI, __half>(out, dt, A, a_dt, W, bias, M, N, K, st);
  }
  set_error("gemm: unknown out dtype %d", static_cast<int>(dt));
  return VB200_ERR_INVALID;
}

}  // namespace vb200

using namespace vb200;

extern "C" int vb200_gemm_bf16(void* out, vb200_dtype out_dtype, const void* A, vb200_dtype a_dtype, const void* W,
                               const float* bias, const float* residual, int32_t M, int32_t N,
                               int32_t K, vb200_epilogue epi, vb200_stream_t stream) {
  VB_REQUIRE(M >= 0 && N > 0 && K > 0, "gemm: bad sizes M=%d N=%d K=%d", M, N, K);
  VB_REQUIRE(a_dtype == VB200_BF16 || a_dtype == VB200_F16, "gemm: A and W must be bf16 or f16");
  if (M == 0) return VB200_OK;                    // nothing to do (empty tensors carry null pointers)
  VB_REQUIRE(out && A && W, "gemm: null pointer");
  VB_REQUIRE(K % 8 == 0, "gemm: K=%d must be a multiple of 8 (TMA row stride is 16-byte granular)", K);
  VB_REQUIRE(N % 8 == 0, "gemm: N=%d must be a multiple of 8 (16-byte vector stores)", N);
  VB_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "gemm: out must be 16-byte aligned");
  VB_REQUIRE(epi == VB200_EPI_NONE || bias, "gemm: epilogue %d needs bias", static_cast<int>(epi));
  VB_REQUIRE(epi == VB200_EPI_NONE || (reinterpret_cast<uintptr_t>(bias) & 15) == 0,
             "gemm: bias must be 16-byte aligned (the epilogue reads it as float4)");
  VB_REQUIRE(epi != VB200_EPI_BIAS_RESIDUAL || (residual && out_dtype == VB200_F32),
             "gemm: BIAS_RESIDUAL needs residual and fp32 output");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (epi) {
    case VB200_EPI_NONE: return launch_gemm_dtype<VB200_EPI_NONE>(out, out_dtype, A, a_dtype, W, bias, M, N, K, st);
    case VB200_EPI_BIAS: return launch_gemm_dtype<VB200_EPI_BIAS>(out, out_dtype, A, a_dtype, W, bias, M, N, K, st);
    case VB200_EPI_BIAS_GELU: return launch_gemm_dtype<VB200_EPI_BIAS_GELU>(out, out_dtype, A, a_dtype, W, bias, M, N, K, st);
    case VB200_EPI_BIAS_RESIDUAL:
      // out (+)= acc + bias is a TMA reduce-add into `out`; a distinct residual is copied in first
      if (residual != static_cast<const float*>(out))
        VB_CHECK_CUDA(cudaMemcpyAsync(out, residual, static_cast<size_t>(M) * N * sizeof(float),
                                      cudaMemcpyDeviceToDevice, st));
      return launch_gemm<VB200_EPI_BIAS_RESIDUAL, float>(out, out_dtype, A, a_dtype, W, bias, M, N, K, st);
  }
  set_error("gemm: unknown epilogue %d", static_cast<int>(epi));
  return VB200_ERR_INVALID;
}
