// Classifier GEMM with the D3PM reverse step as its EPILOGUE (SURVEY.md §8a rows H1 + P; reference
// base.py:355,440 followed by ar_discrete.py:347-375,401-420): logits never leave the SM.
//
// A token's posterior needs the softmax normaliser over all K classes of its level, i.e. over
// K / 256 accumulator tiles, before anything can be drawn from it by inverse CDF — which is why the
// unfused kernel (d3pm.cu) wants the finished logits.  The way around it is to decompose the
// posterior instead of normalising it: its total weight is  cA + K cst + dx + dm  (posterior.cuh),
// so the draw is a MIXTURE:
//     with probability  cA / total     a class from softmax(logits),
//                       K cst / total  a uniform class,
//                       dx / total     x_t,          dm / total   the absorbing class m.
// Only dx, dm need Z (known once the last tile has passed), and a draw from softmax(logits) can be
// made STREAMING, tile by tile, with weighted reservoir sampling under the online-softmax
// rescaling: after a chunk of 32 classes with mass s (relative to the running max) the running
// mass is W <- W r + s and the chunk takes over as the candidate with probability s / W; the class
// inside the winning chunk is picked by inverse CDF over its 32 weights.  Every step is an exact
// conditional draw, so the result is distributed exactly as the reference's Gumbel-max sample —
// from 6 Philox calls per token instead of K uniforms.
//
// Structure: the CTA-pair tcgen05 GEMM of gemm_tcgen05.cu (TMA ring, one MMA-issuing lane,
// double-buffered TMEM accumulators), walking WORK ITEMS (256-row block, level) = K / 256
// consecutive column tiles, so that each epilogue thread (one accumulator row, half of the 256
// columns of a tile) carries its token's streaming state in registers across the tiles of the
// item; the two threads of a row merge at the end of the item and one of them writes the code.
#include "posterior.cuh"

namespace vb200 {

namespace hs {
constexpr int BM = 128, BN = 256, BK = 64, STAGES = 5;
constexpr int A_BYTES = BM * BK * 2;            // 16 KB
constexpr int B_ROWS = BN / 2;                  // each CTA of the pair stages half of the W tile
constexpr int STAGE_BYTES = A_BYTES + B_ROWS * BK * 2;   // 32 KB
constexpr int EPI_WARPS = 8;
constexpr int THREADS = (2 + EPI_WARPS) * 32;   // 320
constexpr int ROW_BYTES = 128;                  // staging: 32 fp32 weights of the current chunk per thread
constexpr int XCHG_WORDS = 12;                  // per row: what half 1 hands to half 0 at the end of a token
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_WARPS * 32 * ROW_BYTES + BM * XCHG_WORDS * 4 +
                           1024 /*align slack*/ + 256 /*barriers*/;
constexpr uint32_t TMEM_COLS = 512;
constexpr int MODE_CE = 100;                    // epilogue = cross-entropy against target classes (no sampling)
}  // namespace hs

__device__ __forceinline__ void hs_bar_sync(int id, int n_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}

// per-token streaming state of one thread (one accumulator row, one half of each tile's columns)
struct HsState {
  float m, Z;            // running max of the logits seen (natural log units) and mass relative to it
  float e_x, m_x;        // weight of class x_t as first seen, and the max it was relative to
  float e_m, m_m;        // same for the absorbing class
  float best;            // largest logit seen (greedy / t == 0), and its class
  int best_j;
  int win_col;           // first class of the candidate chunk
};

template <int NOISE>
__global__ void __launch_bounds__(hs::THREADS, 1) head_sample_kernel(
    const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
    int32_t* __restrict__ x_out, float* __restrict__ loss_out, const float* __restrict__ bias,
    const int32_t* __restrict__ x_t_all,
    const int32_t* __restrict__ row_utt, const int32_t* __restrict__ t_utt, const int32_t* __restrict__ utt,
    const float* __restrict__ table, int n_rows, int n_levels, int K, int Kd, int S, int transition,
    uint32_t seed_lo, uint32_t seed_hi, uint32_t a_is_f16, const int32_t* __restrict__ known) {
  using namespace hs;
  const uint32_t cta_rank = cluster_ctarank();          // 0 = leader of the pair
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint8_t* row_smem = smem + STAGES * STAGE_BYTES;                       // [EPI_WARPS][32 rows][128 B]
  float* xchg = reinterpret_cast<float*>(row_smem + EPI_WARPS * 32 * ROW_BYTES);   // [128 rows][XCHG_WORDS]
  uint64_t* bars = reinterpret_cast<uint64_t*>(xchg + BM * XCHG_WORDS);
  uint64_t* full = bars;                 // [STAGES]  TMA -> MMA
  uint64_t* empty = bars + STAGES;       // [STAGES]  MMA -> TMA
  uint64_t* acc_full = bars + 2 * STAGES;   // [2]     MMA -> epilogue
  uint64_t* acc_empty = acc_full + 2;       // [2]     epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int tpl = K / BN;                               // column tiles per level
  const int num_m = (n_rows + 2 * BM - 1) / (2 * BM);
  const int num_items = num_m * n_levels;               // item = (256-row block, level), level fastest
  const int num_kb = (Kd + BK - 1) / BK;
  const int item0 = blockIdx.x / 2, item_stride = gridDim.x / 2;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], EPI_WARPS * 2); }
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc_pair(tmem_slot, TMEM_COLS); tmem_relinquish_pair(); }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    const bool leader = elect_one();
    int stage = 0; uint32_t phase = 0;
    for (int item = item0; item < num_items; item += item_stride) {
      const int m_blk = item / n_levels, level = item - m_blk * n_levels;
      const int m_row = (m_blk * 2 + cta_rank) * BM;
      for (int q = 0; q < tpl; ++q) {
        const int n_row = (level * tpl + q) * BN + cta_rank * B_ROWS;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          if (leader) {
            if (cta_rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * STAGE_BYTES);
            tma_load_2d_pair(sa, &tm_a, &full[stage], kb * BK, m_row);
            tma_load_2d_pair(sa + A_BYTES, &tm_b, &full[stage], kb * BK, n_row);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (cta_rank == 0) {
      // ------------------------------------------------------------ MMA issuer (leader CTA of the pair)
      const bool leader = elect_one();
      const uint32_t idesc = umma_idesc_bf16(BM * 2, BN, false, false) & ~(a_is_f16 ? kIdescBf16 : 0u);   // rows and weights: both bf16 or both fp16
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int item = item0; item < num_items; item += item_stride) {
        for (int q = 0; q < tpl; ++q, ++it) {
          const int as = it & 1;
          mbar_wait(&acc_empty[as], ((it >> 1) & 1) ^ 1);
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
              for (int k = 0; k < BK / 16; ++k) umma_ss_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
              umma_commit_pair(&empty[stage]);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          if (leader) umma_commit_pair(&acc_full[as]);
          __syncwarp();
        }
      }
    }
  } else {
    // -------------------------------------------------------------- epilogue warps: the reverse step
    const int e = warp - 2;
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int half = e >> 2;                   // columns [half*128, half*128+128) of every tile
    const int r_cta = quad * 32 + lane;        // accumulator row inside this CTA
    uint8_t* my_row = row_smem + (e * 32 + lane) * ROW_BYTES;
    const int sw = lane & 7;                   // 16-byte chunk index ^= row % 8: conflict-free 128-bit stores
    float* my_x = xchg + r_cta * XCHG_WORDS;
    const int m_abs = transition == VB200_ABSORBING ? K / 2 : -1;
    const Philox ph{seed_lo, seed_hi};
    int it = 0;
    for (int item = item0; item < num_items; item += item_stride) {
      const int m_blk = item / n_levels, level = item - m_blk * n_levels;
      const int grow = (m_blk * 2 + cta_rank) * BM + r_cta;      // response row of this thread
      const bool valid = grow < n_rows;
      // ---- token identity and noise key
      int x_t = 0, t = 1;
      uint32_t key1 = 0, gid = 0;
      int b = 0;
      int kn = -1;                                 // x0 of the token when it is given, else -1
      if (valid) {
        x_t = x_t_all[static_cast<size_t>(grow) * n_levels + level];     // MODE_CE: the target class
        if (known) kn = known[static_cast<size_t>(grow) * n_levels + level];
        if (NOISE != MODE_CE) {
          b = row_utt[grow];
          t = clamp_timestep(t_utt[b], S);
          const TokenKey key = token_key(utt, b, grow, level, n_levels);
          key1 = key.tok;
          gid = key.gid;
        }
      }
      const bool need_arg = NOISE == VB200_NOISE_GREEDY || (NOISE != MODE_CE && t == 0);
      HsState st{-INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f, -INFINITY, 0x7fffffff, 0};
      float win[32];                            // weights of the candidate chunk (local memory: written rarely)
#pragma unroll
      for (int i = 0; i < 32; ++i) win[i] = 0.f;
      const float* bias_l = bias + static_cast<size_t>(level) * K;

      for (int q = 0; q < tpl; ++q, ++it) {
        const int as = it & 1;
        mbar_wait(&acc_full[as], (it >> 1) & 1);
        tc_fence_after();
        const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BN + half * 128;
        // four reservoir decisions per tile from one Philox call (stream 1 + half, counter = tile)
        uint4 rnd = make_uint4(0, 0, 0, 0);
        if (NOISE == VB200_NOISE_PHILOX) rnd = ph(0xC0DF0000u + (half << 8) + q, key1, gid, t);
        const uint32_t rw[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int col0 = q * BN + half * 128 + c * 32;         // first class of this chunk
          uint32_t r[32];
          tmem_ld_32x32(t_row + c * 32, r);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias_l + col0 + i));
            unpack2(fadd2(pack2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), pack2(b4.x, b4.y)), v[i], v[i + 1]);
            unpack2(fadd2(pack2(__uint_as_float(r[i + 2]), __uint_as_float(r[i + 3])), pack2(b4.z, b4.w)), v[i + 2], v[i + 3]);
          }
          float m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3];
#pragma unroll
          for (int i = 4; i < 32; i += 4) {
            m0 = fmaxf(m0, v[i]); m1 = fmaxf(m1, v[i + 1]); m2 = fmaxf(m2, v[i + 2]); m3 = fmaxf(m3, v[i + 3]);
          }
          const float cmax = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
          if (__any_sync(0xffffffffu, need_arg && cmax > st.best)) {     // greedy / t == 0 only
            if (need_arg && cmax > st.best) {
              st.best = cmax;
#pragma unroll
              for (int i = 31; i >= 0; --i) if (v[i] == cmax) st.best_j = col0 + i;   // lowest index wins
            }
          }
          if (NOISE == MODE_CE) {                       // the target's raw logit, through this thread's staging row
#pragma unroll
            for (int k = 0; k < 8; ++k)
              *reinterpret_cast<float4*>(my_row + ((k ^ sw) << 4)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
            const int dxt = x_t - col0;
            if (dxt >= 0 && dxt < 32)
              st.e_x = *reinterpret_cast<const float*>(my_row + (((dxt >> 2) ^ sw) << 4) + (dxt & 3) * 4);
          }
          const float m_new = fmaxf(st.m, cmax);
          st.Z *= exp2f_fast((st.m - m_new) * kLog2e);            // 0 on the first chunk (m = -inf)
          st.m = m_new;
          const float mneg = -m_new * kLog2e;
          const uint64_t l2e2 = pack2(kLog2e, kLog2e), mneg2 = pack2(mneg, mneg);
          uint64_t acc = 0ull;
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float x0, x1;
            unpack2(ffma2(pack2(v[i], v[i + 1]), l2e2, mneg2), x0, x1);
            v[i] = exp2f_fast(x0);
            v[i + 1] = exp2f_fast(x1);
            acc = fadd2(acc, pack2(v[i], v[i + 1]));
          }
          float a0, a1;
          unpack2(acc, a0, a1);
          const float s_c = a0 + a1;
          st.Z += s_c;
          if (NOISE != MODE_CE) {
            // the chunk's weights go to this thread's staging row: class x_t is read back from it
#pragma unroll
            for (int k = 0; k < 8; ++k)
              *reinterpret_cast<float4*>(my_row + ((k ^ sw) << 4)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
            const int dxt = x_t - col0;
            if (dxt >= 0 && dxt < 32) {
              st.e_x = *reinterpret_cast<const float*>(my_row + (((dxt >> 2) ^ sw) << 4) + (dxt & 3) * 4);
              st.m_x = m_new;
            }
            if (col0 == (m_abs & ~31)) { st.e_m = v[0]; st.m_m = m_new; }   // K/2 is a multiple of 128
          }
          // weighted reservoir: this chunk becomes the candidate with probability s_c / Z
          if (NOISE == VB200_NOISE_PHILOX) {
            if (u01(rw[c]) * st.Z < s_c) {
              st.win_col = col0;
#pragma unroll
              for (int i = 0; i < 32; ++i) win[i] = v[i];
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {                                // accumulator drained: one arrival per epilogue warp
          if (cta_rank != 0) mbar_arrive_remote(&acc_empty[as], 0);
          else mbar_arrive(&acc_empty[as]);
        }
      }

      // ---- end of the token: class inside this half's candidate chunk, then merge the two halves
      uint4 fin = make_uint4(0, 0, 0, 0);
      int cand = st.win_col;
      if (NOISE == VB200_NOISE_PHILOX) {
        fin = ph(0xC0DF0000u + (half << 8) + 0xff, key1, gid, t);
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) tot += win[i];
        const float target = u01(fin.x) * tot;
        float run = 0.f;
        int idx = 0;
#pragma unroll
        for (int i = 0; i < 31; ++i) {                  // prefix sums are monotone: count those <= target
          run += win[i];
          idx += target >= run ? 1 : 0;
        }
        cand = st.win_col + idx;
      }
      if (half == 1) {
        my_x[0] = st.m; my_x[1] = st.Z; my_x[2] = st.e_x; my_x[3] = st.m_x; my_x[4] = st.e_m; my_x[5] = st.m_m;
        my_x[6] = st.best; my_x[7] = __int_as_float(st.best_j); my_x[8] = __int_as_float(cand);
      }
      hs_bar_sync(1 + quad, 64);
      if (half == 0) {
        const float m_b = my_x[0], Z_b = my_x[1];
        const float m_f = fmaxf(st.m, m_b);
        const float Za = st.Z * exp2f_fast((st.m - m_f) * kLog2e), Zb = Z_b * exp2f_fast((m_b - m_f) * kLog2e);
        const float Z = Za + Zb, invZ = 1.0f / Z;
        // class x_t / m: whichever half saw it (weights were relative to the max at that time)
        const float e_x = st.e_x * exp2f_fast((st.m_x - m_f) * kLog2e) + my_x[2] * exp2f_fast((my_x[3] - m_f) * kLog2e);
        const float e_m = st.e_m * exp2f_fast((st.m_m - m_f) * kLog2e) + my_x[4] * exp2f_fast((my_x[5] - m_f) * kLog2e);
        float best = st.best;
        int best_j = st.best_j;
        {
          const float b1 = my_x[6];
          const int j1 = __float_as_int(my_x[7]);
          if (b1 > best || (b1 == best && j1 < best_j)) { best = b1; best_j = j1; }   // lowest index wins ties
        }
        const int cand_b = __float_as_int(my_x[8]);
        int pick = 0;
        if (NOISE == MODE_CE) {
          // -log softmax(logits)[target] = max + ln Z - logit[target]; exactly one half saw the target
          if (valid) loss_out[static_cast<size_t>(grow) * n_levels + level] = m_f + __logf(Z) - (st.e_x + my_x[2]);
        } else if (kn >= 0) {                            // x0 given: O(1) law of posterior.cuh, logits unused
          pick = known_pick(post_scalars(table, t, x_t, K, transition), kn, t, K, NOISE == VB200_NOISE_GREEDY,
                            u01(fin.y), u01(fin.z));
        } else if (t == 0) {
          pick = best_j;                                 // raw logits, no noise (ar_discrete.py:407,413)
        } else {
          const PostScalars ps = post_scalars(table, t, x_t, K, transition);
          const float cA = ps.cA(), cst = ps.cst();
          const float coef = cA * invZ;
          const PostSpecial w = post_special(ps, e_x, e_m, invZ, coef, cst);
          if (NOISE == VB200_NOISE_GREEDY) {
            pick = post_greedy(ps, w, fmaf(exp2f_fast((best - m_f) * kLog2e), coef, cst), best_j);
          } else {
            const float w_uni = static_cast<float>(K) * cst;
            const float target = u01(fin.y) * (cA + w_uni + w.dx + w.dm);
            if (target < w.dx) pick = x_t;
            else if (target < w.dx + w.dm) pick = m_abs;
            else if (target < w.dx + w.dm + w_uni) pick = min(static_cast<int>(u01(fin.z) * K), K - 1);
            else pick = (u01(fin.w) * Z < Zb) ? cand_b : cand;     // softmax(logits): merge the two candidates
          }
        }
        if (NOISE != MODE_CE && valid) x_out[static_cast<size_t>(grow) * n_levels + level] = pick;
      }
      hs_bar_sync(1 + quad, 64);                        // half 1 may overwrite its exchange words again
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, TMEM_COLS);
  }
}

template <int NOISE>
static int launch_head_sample(int32_t* x_out, float* loss_out, const void* head_in, const void* W, const float* bias,
                              const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
                              const int32_t* utt, const float* table, int n_rows, int d, int n_levels,
                              int K, int S, int tr, uint64_t seed, int in_f16, const int32_t* known, cudaStream_t st) {
  using namespace hs;
  CUtensorMap ta, tb;
  int rc = cached_tmap(&ta, in_f16 ? VB200_F16 : VB200_BF16, head_in, d, n_rows, static_cast<uint64_t>(d) * 2, BK, BM);
  if (rc != VB200_OK) return rc;
  rc = cached_tmap(&tb, in_f16 ? VB200_F16 : VB200_BF16, W, d, static_cast<uint64_t>(n_levels) * K, static_cast<uint64_t>(d) * 2, BK, B_ROWS);
  if (rc != VB200_OK) return rc;
  const int items = ((n_rows + 2 * BM - 1) / (2 * BM)) * n_levels;
  const int groups = num_sms() / 2;
  const int grid = (items < groups ? items : groups) * 2;
  auto kern = head_sample_kernel<NOISE>;
  VB_CONFIGURE_SMEM(kern, SMEM_BYTES);
  PdlTag pdl_tag(32);
  VB_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(THREADS), SMEM_BYTES, st, 2, ta, tb, x_out, loss_out, bias, x_t, row_utt,
                           t_utt, utt, table, n_rows, n_levels, K, d, S, tr, static_cast<uint32_t>(seed),
                           static_cast<uint32_t>(seed >> 32), static_cast<uint32_t>(in_f16 ? 1 : 0), known));
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

int head_sample_fused(int32_t* x_out, const void* head_in, const void* W, const float* bias,
                      const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt, const int32_t* utt,
                      const float* table, int n_rows, int d, int n_levels, int K, int S, int tr, int noise,
                      uint64_t seed, int in_f16, const int32_t* known, cudaStream_t st) {
  if (noise == VB200_NOISE_GREEDY)
    return launch_head_sample<VB200_NOISE_GREEDY>(x_out, nullptr, head_in, W, bias, x_t, row_utt, t_utt, utt, table, n_rows,
                                                  d, n_levels, K, S, tr, seed, in_f16, known, st);
  return launch_head_sample<VB200_NOISE_PHILOX>(x_out, nullptr, head_in, W, bias, x_t, row_utt, t_utt, utt, table, n_rows, d,
                                                n_levels, K, S, tr, seed, in_f16, known, st);
}


// classifier GEMM with per-token cross-entropy as its epilogue: loss[r, l] = -log softmax(logits[r, l, :])[target[r, l]]
int head_ce_fused(float* loss_out, const void* head_in, const void* W, const float* bias, const int32_t* targets,
                  int n_rows, int d, int n_levels, int K, int in_f16, cudaStream_t st) {
  return launch_head_sample<hs::MODE_CE>(nullptr, loss_out, head_in, W, bias, targets, nullptr, nullptr, nullptr,
                                         nullptr, n_rows, d, n_levels, K, 1, VB200_UNIFORM, 0, in_f16, nullptr, st);
}

}  // namespace vb200

extern "C" int vb200_head_fused(int32_t d, int32_t K, vb200_noise noise) {
  return K % 256 == 0 && K >= 256 && K <= 4096 && d % 8 == 0 && noise != VB200_NOISE_UNIFORMS;
}
