// D3PM forward noising (row Q) and closed-form reverse step (row P), SURVEY.md §8(a).
// One warp per token, O(K) work, fp32 in registers; the reference's dense (K,K) fp16 matmuls
// (ar_discrete.py:337-345,377-400) collapse to a handful of per-timestep scalars.
#include "posterior.cuh"

namespace vb200 {

constexpr float kTiny = 1.17549435e-38f; // torch.finfo(float32).tiny, ar_discrete.py:414,485

// Gumbel noise exactly as the reference forms it, evaluated through double so that each fp32
// log is correctly rounded (the CPU reference's SLEEF logf is <= 1 ulp; agreeing with the
// correctly rounded value is the closest a different libm can get).
__device__ __forceinline__ float gumbel_exact(float u) {
  u = fminf(fmaxf(u, kTiny), 1.0f);
  const float inner = static_cast<float>(log(static_cast<double>(u)));
  return -static_cast<float>(log(static_cast<double>(-inner)));
}
__device__ __forceinline__ float gumbel_fast(float u) {
  u = fmaxf(u, kTiny);
  return -__logf(-__logf(u));
}

struct Best {
  float v;
  int j;
};
__device__ __forceinline__ void best_update(Best& b, float v, int j) {
  if (v > b.v || (v == b.v && j < b.j)) { b.v = v; b.j = j; }
}
__device__ __forceinline__ Best warp_best(Best b) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float v = __shfl_xor_sync(0xffffffffu, b.v, o);
    const int j = __shfl_xor_sync(0xffffffffu, b.j, o);
    best_update(b, v, j);
  }
  return b;
}

// ---------------------------------------------------------------- Q: q_sample
// DENSE: row x0 of the caller's own fp16 table log(Qbar_t + eps) (S, K, K) replaces the per-timestep
// scalars — for the uniform transition, whose K-term fp16 chain product is not rank-structured to the
// last bit (which entry rounds up depends on the summation order of the GEMM that built the table).
template <bool DENSE>
__global__ void __launch_bounds__(256) q_sample_kernel(
    int32_t* __restrict__ x_out, const int32_t* __restrict__ x0, const int32_t* __restrict__ t_tok,
    const int32_t* __restrict__ mask, const float* __restrict__ uniforms,
    const float* __restrict__ table, const __half* __restrict__ log_qbar, int n_tok, int K, int S,
    int transition) {
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  for (int tok = blockIdx.x * warps_per_block + (threadIdx.x >> 5); tok < n_tok;
       tok += gridDim.x * warps_per_block) {
    const int x = x0[tok];
    int t = t_tok[tok];
    t = min(max(t, 0), S - 1);
    const int m = K / 2;
    const bool absorbing = transition == VB200_ABSORBING;
    float l_keep = 0.f, l_off = 0.f, l_abs = 0.f, l_both = 0.f;
    const __half* row = nullptr;
    if (DENSE) {
      row = log_qbar + (static_cast<size_t>(t) * K + min(max(x, 0), K - 1)) * K;
    } else {
      const float* tab = table + static_cast<size_t>(t) * VB200_TAB_STRIDE;
      l_keep = tab[VB200_TAB_LOG_KEEP]; l_off = tab[VB200_TAB_LOG_OFF];
      l_abs = tab[VB200_TAB_LOG_ABSORB]; l_both = tab[VB200_TAB_LOG_BOTH];
    }
    const float* u = uniforms + static_cast<size_t>(tok) * K;
    Best best{-INFINITY, 0x7fffffff};
    for (int j = lane; j < K; j += 32) {
      float lg;
      if (DENSE) {
        lg = __half2float(row[j]);
      } else if (absorbing) {
        if (x == m) lg = (j == m) ? l_both : l_off;           // row m of Qbar: [0 .. 1 .. 0]
        else lg = (j == x) ? l_keep : ((j == m) ? l_abs : l_off);
      } else {
        lg = (j == x) ? l_keep : l_off;
      }
      best_update(best, lg + gumbel_exact(__ldg(u + j)), j);
    }
    best = warp_best(best);
    if (lane == 0) x_out[tok] = best.j * (mask ? mask[tok] : 1);
  }
}

// q_sample with in-kernel noise: the same categorical law as above — weights exp(fp16 log(Qbar_t[x0, j]
// + eps)), read from the table — drawn in O(1) from one Philox uniform per token instead of an
// argmax over K Gumbel variates: only the classes x0 and m carry their own weight, all others share
// one (the eps leak), so the CDF has three pieces.  For training forwards (ar_discrete.py:651-653),
// where the reference draws K uniforms per token on the CPU and ships them to the device.
__global__ void __launch_bounds__(256) q_sample_philox_kernel(
    int32_t* __restrict__ x_out, const int32_t* __restrict__ x0, const int32_t* __restrict__ t_tok,
    const int32_t* __restrict__ mask, const float* __restrict__ table, int n_tok, int K, int S,
    int transition, uint32_t seed_lo, uint32_t seed_hi) {
  pdl_launch_dependents();
  pdl_wait();
  const Philox ph{seed_lo, seed_hi};
  for (int tok = blockIdx.x * blockDim.x + threadIdx.x; tok < n_tok; tok += gridDim.x * blockDim.x) {
    const int x = x0[tok];
    const int t = min(max(t_tok[tok], 0), S - 1);
    const float* tab = table + static_cast<size_t>(t) * VB200_TAB_STRIDE;
    const bool absorbing = transition == VB200_ABSORBING;
    const int m = absorbing ? K / 2 : -1;
    const float w_off = __expf(tab[VB200_TAB_LOG_OFF]);
    float w_self, w_m = 0.f;
    int n_other;
    if (absorbing && x == m) { w_self = __expf(tab[VB200_TAB_LOG_BOTH]); n_other = K - 1; }
    else if (absorbing) { w_self = __expf(tab[VB200_TAB_LOG_KEEP]); w_m = __expf(tab[VB200_TAB_LOG_ABSORB]); n_other = K - 2; }
    else { w_self = __expf(tab[VB200_TAB_LOG_KEEP]); n_other = K - 1; }
    const uint4 r = ph(0x0D3B0000u, static_cast<uint32_t>(tok), 0u, static_cast<uint32_t>(t));
    const float target = u01(r.x) * (w_self + w_m + n_other * w_off);
    int pick;
    if (target < w_self) {
      pick = x;
    } else if (target < w_self + w_m) {
      pick = m;
    } else {                                              // one of the other classes, uniformly
      int j = min(static_cast<int>(u01(r.y) * n_other), n_other - 1);
      const int lo = (w_m > 0.f) ? min(x, m) : x, hi = (w_m > 0.f) ? max(x, m) : -1;
      if (j >= lo) ++j;                                   // skip x (and m), in ascending order
      if (hi >= 0 && j >= hi) ++j;
      pick = j;
    }
    x_out[tok] = pick * (mask ? mask[tok] : 1);
  }
}

// ---------------------------------------------------------------- P: posterior + sample
template <typename T>
__device__ __forceinline__ float load_logit(const T* p, int j);
template <>
__device__ __forceinline__ float load_logit<float>(const float* p, int j) { return __ldg(p + j); }
template <>
__device__ __forceinline__ float load_logit<__nv_bfloat16>(const __nv_bfloat16* p, int j) {
  return __bfloat162float(p[j]);
}
template <>
__device__ __forceinline__ float load_logit<__half>(const __half* p, int j) {
  return __half2float(p[j]);
}

// Loads 8 consecutive logits (16-byte aligned for 2-byte types) into fp32.
template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&v)[8]);
template <>
__device__ __forceinline__ void load8<float>(const float* p, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <>
__device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
template <>
__device__ __forceinline__ void load8<__half>(const __half* p, float (&v)[8]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}

// log w_j; raw (t == 0): the posterior logits are the raw logits (ar_discrete.py:374,407)
__device__ __forceinline__ float post_logit(const PostScalars& s, bool raw, float logit, float p, int j) {
  if (raw) return logit;
  const float f1 = (j == s.x_t) ? s.f1_self : s.f1_oth;
  const bool is_m = (j == s.m);
  const float a = is_m ? s.a_m : s.a_gen, c = is_m ? s.c_m : s.c_gen;
  const float f2 = fmaf(p, a - c, c);
  return logf(f1) + logf(f2 + kEps);
}

// One warp's reverse step of a token whose x0 = k is given.  With supplied uniforms the code is the Gumbel-arg max
// of its K posterior logits (the reference's noise convention); Philox and greedy take the O(1) form of
// posterior.cuh, with the Philox counter posterior_fast_kernel uses, so the two kernels draw the same code.
// post_out gets the logits of the ids form of q_posterior_logits (0 at t == 0, as the reference's
// torch.where(t == 0, x_start_logits=False, ...) gives).
template <int NOISE>
__device__ __forceinline__ void known_token(int32_t* __restrict__ x_out, float* __restrict__ post_out,
                                            const float* __restrict__ uniforms, const float* __restrict__ table,
                                            const int32_t* __restrict__ utt, int tok, int b, int row, int level,
                                            int n_levels, int t, int x_t, int k, int K, int transition,
                                            uint32_t seed_lo, uint32_t seed_hi, int lane) {
  const PostScalars ps = post_scalars(table, t, x_t, K, transition);
  const bool raw = t == 0;
  if (post_out || NOISE == VB200_NOISE_UNIFORMS) {
    float* prow = post_out ? post_out + static_cast<size_t>(tok) * K : nullptr;
    const float* urow = NOISE == VB200_NOISE_UNIFORMS ? uniforms + static_cast<size_t>(tok) * K : nullptr;
    Best best{-INFINITY, 0x7fffffff};
    for (int j = lane; j < K; j += 32) {
      const float pl = raw ? 0.f : known_logit(ps, k, j);
      if (prow) prow[j] = pl;
      best_update(best, (NOISE == VB200_NOISE_UNIFORMS && !raw) ? pl + gumbel_exact(__ldg(urow + j)) : pl, j);
    }
    best = warp_best(best);
    if (NOISE == VB200_NOISE_UNIFORMS && !raw) {
      if (lane == 0) x_out[tok] = best.j;
      return;
    }
  }
  uint4 r = make_uint4(0, 0, 0, 0);
  if (NOISE == VB200_NOISE_PHILOX) {
    const TokenKey key = token_key(utt, b, row, level, n_levels);
    r = Philox{seed_lo, seed_hi}(0xC0DEu, key.tok, key.gid, t);
  }
  const int pick = known_pick(ps, k, t, K, NOISE == VB200_NOISE_GREEDY, u01(r.x), u01(r.y));
  if (lane == 0) x_out[tok] = pick;
}

template <typename T, int NOISE>
__global__ void __launch_bounds__(256) posterior_sample_kernel(
    int32_t* __restrict__ x_out, float* __restrict__ post_out, const T* __restrict__ logits,
    int64_t ld_logits, const int32_t* __restrict__ x_t_all, const int32_t* __restrict__ row_utt,
    const int32_t* __restrict__ t_utt, const int32_t* __restrict__ utt,
    const float* __restrict__ table, int n_rows, int n_levels, int K, int S, int transition,
    const float* __restrict__ uniforms, uint32_t seed_lo, uint32_t seed_hi, const int32_t* __restrict__ known,
    float inv_temp) {
  pdl_launch_dependents();
  pdl_wait();                                   // everything below reads / writes activations
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tok = n_rows * n_levels;
  const bool vec = (K % 8 == 0) && (ld_logits % 8 == 0) &&
                   ((reinterpret_cast<uintptr_t>(logits) & 15) == 0);
  for (int tok = blockIdx.x * warps_per_block + (threadIdx.x >> 5); tok < n_tok;
       tok += gridDim.x * warps_per_block) {
    const int row = tok / n_levels, level = tok - row * n_levels;
    const int b = row_utt[row];
    const int t = clamp_timestep(t_utt[b], S);
    const bool raw = t == 0;   // raw logits and no noise (nonzero_mask, ar_discrete.py:412-419)
    const int kn = known ? known[tok] : -1;
    if (kn >= 0) {             // x0 given: its law never reads the logits (posterior.cuh, known_pick)
      known_token<NOISE>(x_out, post_out, uniforms, table, utt, tok, b, row, level, n_levels, t, x_t_all[tok], kn, K,
                         transition, seed_lo, seed_hi, lane);
      continue;
    }
    const T* lrow = logits + static_cast<size_t>(row) * ld_logits + static_cast<size_t>(level) * K;

    // pass 1: row max; pass 2: sum exp (the row is 2-4 KB and stays in L1 between passes).  p̂(x0) is
    // softmax(logits * inv_temp); the raw logits are what t == 0 returns (x * 1.0f is exact: tau = 1 is unscaled).
    float mx = -INFINITY;
    if (vec) {
      for (int j0 = lane * 8; j0 < K; j0 += 256) {
        float v[8]; load8<T>(lrow + j0, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) mx = fmaxf(mx, v[i] * inv_temp);
      }
    } else {
      for (int j = lane; j < K; j += 32) mx = fmaxf(mx, load_logit<T>(lrow, j) * inv_temp);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    if (vec) {
      for (int j0 = lane * 8; j0 < K; j0 += 256) {
        float v[8]; load8<T>(lrow + j0, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) sum += __expf(v[i] * inv_temp - mx);
      }
    } else {
      for (int j = lane; j < K; j += 32) sum += __expf(load_logit<T>(lrow, j) * inv_temp - mx);
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    const PostScalars ps = post_scalars(table, t, x_t_all[tok], K, transition);

    // Philox key: (seed) ; counter: (j/4, frame*n_levels+level, global utterance id, t)
    const TokenKey key = NOISE == VB200_NOISE_PHILOX ? token_key(utt, b, row, level, n_levels) : TokenKey{0, 0};
    const Philox ph{seed_lo, seed_hi};
    const float* urow = (NOISE == VB200_NOISE_UNIFORMS) ? uniforms + static_cast<size_t>(tok) * K : nullptr;
    float* prow = post_out ? post_out + static_cast<size_t>(tok) * K : nullptr;

    Best best{-INFINITY, 0x7fffffff};
    if (vec) {
      for (int j0 = lane * 8; j0 < K; j0 += 256) {
        float v[8]; load8<T>(lrow + j0, v);
        float g[8];
        if (NOISE == VB200_NOISE_PHILOX) {
          const uint4 r0 = ph(j0 >> 2, key.tok, key.gid, t);
          const uint4 r1 = ph((j0 >> 2) + 1, key.tok, key.gid, t);
          const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
          for (int i = 0; i < 8; ++i) g[i] = gumbel_fast(u01(rr[i]));
        } else if (NOISE == VB200_NOISE_UNIFORMS) {
#pragma unroll
          for (int i = 0; i < 8; ++i) g[i] = gumbel_exact(__ldg(urow + j0 + i));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int j = j0 + i;
          const float pl = post_logit(ps, raw, v[i], __expf(v[i] * inv_temp - mx) * inv, j);
          if (prow) prow[j] = pl;
          const float sc = (NOISE != VB200_NOISE_GREEDY && !raw) ? pl + g[i] : pl;
          best_update(best, sc, j);
        }
      }
    } else {
      for (int j = lane; j < K; j += 32) {
        const float l = load_logit<T>(lrow, j);
        const float pl = post_logit(ps, raw, l, __expf(l * inv_temp - mx) * inv, j);
        if (prow) prow[j] = pl;
        float sc = pl;
        if (NOISE == VB200_NOISE_PHILOX && !raw) {
          const uint4 r = ph(j >> 2, key.tok, key.gid, t);
          const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
          sc += gumbel_fast(u01(rr[j & 3]));
        } else if (NOISE == VB200_NOISE_UNIFORMS && !raw) {
          sc += gumbel_exact(__ldg(urow + j));
        }
        best_update(best, sc, j);
      }
    }
    best = warp_best(best);
    if (lane == 0) x_out[tok] = best.j;
  }
}


// 8 logits as one 16-byte word (2-byte types) or two (fp32), and their unpacking to fp32.
template <typename T> struct Raw8 { uint4 a; };
template <> struct Raw8<float> { uint4 a, b; };
template <typename T>
__device__ __forceinline__ Raw8<T> load_raw8(const T* p) {
  Raw8<T> r;
  r.a = __ldcs(reinterpret_cast<const uint4*>(p));
  return r;
}
template <>
__device__ __forceinline__ Raw8<float> load_raw8<float>(const float* p) {
  Raw8<float> r;
  r.a = __ldcs(reinterpret_cast<const uint4*>(p));
  r.b = __ldcs(reinterpret_cast<const uint4*>(p) + 1);
  return r;
}
__device__ __forceinline__ void unpack8(const Raw8<__half>& r, float* v) {
  const uint32_t w[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ void unpack8(const Raw8<__nv_bfloat16>& r, float* v) {
  const uint32_t w[4] = {r.a.x, r.a.y, r.a.z, r.a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ void unpack8(const Raw8<float>& r, float* v) {
  v[0] = __uint_as_float(r.a.x); v[1] = __uint_as_float(r.a.y); v[2] = __uint_as_float(r.a.z); v[3] = __uint_as_float(r.a.w);
  v[4] = __uint_as_float(r.b.x); v[5] = __uint_as_float(r.b.y); v[6] = __uint_as_float(r.b.z); v[7] = __uint_as_float(r.b.w);
}

// raw (unconverted) single logit, so that a prefetch never waits on the load it has just issued
template <typename T> struct Raw1 { T v; };
template <typename T>
__device__ __forceinline__ Raw1<T> load_raw1(const T* p, int j) { return Raw1<T>{p[j]}; }
__device__ __forceinline__ float cvt1(Raw1<float> r) { return r.v; }
__device__ __forceinline__ float cvt1(Raw1<__half> r) { return __half2float(r.v); }
__device__ __forceinline__ float cvt1(Raw1<__nv_bfloat16> r) { return __bfloat162float(r.v); }

// ---------------------------------------------------------------- P, production form
// Register-resident O(K) reverse step for K = 256*KC (<= 1024): one warp per token, the K logits
// are read from HBM exactly once (16-byte loads), softmax statistics stay in registers, and the
// token is drawn by inverse CDF from ONE Philox uniform — an exact categorical sample, equal in
// distribution to the reference's Gumbel-max over K uniforms (ar_discrete.py:402-419) at 1/K of
// the random numbers and no per-class logarithm.  The total weight is closed form (posterior.cuh);
// the per-class weights are only walked when the draw lands in the generic part.
//
// A warp walks its tokens in batches of 32.  Everything about a token that is not its logits —
// timestep, x_t, the table-derived scalars, the Philox draw — is produced LANE-PARALLEL at the
// head of the batch (lane k prepares the batch's k-th token) and handed out with shuffles, so no
// token waits on the utterance -> timestep -> table chain of dependent loads and the ten Philox
// rounds cost 1/32 of a token each.  The logits of token k+1 (packed, unconverted) are in flight
// while token k is reduced.
// KNOWN: `known` (x0 given for some tokens) is read; a template flag, so that without it the kernel is the
// register-tight loop it was (a runtime branch costs spills at KC = 4).
// inv_temp = 1/tau: p̂(x0) = softmax(logits / tau).  A logit only enters an exponent exp2((l - max) * log2 e), so
// 1/tau is folded into that factor and the max and arg max (greedy, t == 0) stay on the raw logits.  tau = 1
// multiplies by exactly 1.0f: the unscaled arithmetic bit for bit.
template <typename T, int KC, int NOISE, bool KNOWN>
__global__ void __launch_bounds__(256, 3) posterior_fast_kernel(
    int32_t* __restrict__ x_out, const T* __restrict__ logits, int64_t ld_logits,
    const int32_t* __restrict__ x_t_all, const int32_t* __restrict__ row_utt,
    const int32_t* __restrict__ t_utt, const int32_t* __restrict__ utt,
    const float* __restrict__ table, int n_rows, int n_levels, int S, int transition,
    uint32_t seed_lo, uint32_t seed_hi, const int32_t* __restrict__ known, float inv_temp) {
  constexpr int K = KC * 256;
  pdl_launch_dependents();
  pdl_wait();                                   // everything below reads / writes activations
  constexpr int NR = KC * 8;                  // logits per lane
  constexpr unsigned kFull = 0xffffffffu;
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tok = n_rows * n_levels;
  const int stride = gridDim.x * warps_per_block;
  const int w0 = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
  const int m_abs = transition == VB200_ABSORBING ? K / 2 : -1;
  const int m_probe = K / 2;                  // column read for the absorbing class (unused otherwise)

  Raw8<T> nxt[KC];
  Raw1<T> nxt_lx{}, nxt_lm{};
  auto prefetch = [&](int tk, int xt) {
    const int rw = tk / n_levels, lv = tk - rw * n_levels;
    const T* lr = logits + static_cast<size_t>(rw) * ld_logits + static_cast<size_t>(lv) * K;
#pragma unroll
    for (int c = 0; c < KC; ++c) nxt[c] = load_raw8<T>(lr + c * 256 + lane * 8);
    nxt_lx = load_raw1<T>(lr, xt);
    nxt_lm = load_raw1<T>(lr, m_probe);
  };

#pragma unroll 1
  for (int base = w0; base < n_tok; base += 32 * stride) {
    // ---- lane-parallel: everything but the logits of token `mine`
    const int mine = base + lane * stride;
    int my_t = 0;
    uint32_t my_rnd = 0;
    int my_known = -1;                        // the code of a token whose x0 is given, drawn here in O(1)
    PostScalars my{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0, m_abs};
    if (mine < n_tok) {
      const int row = mine / n_levels, level = mine - row * n_levels;
      const int b = row_utt[row];
      my_t = clamp_timestep(t_utt[b], S);
      my = post_scalars(table, my_t, x_t_all[mine], K, transition);
      uint4 r = make_uint4(0, 0, 0, 0);
      if (NOISE == VB200_NOISE_PHILOX) {
        const TokenKey key = token_key(utt, b, row, level, n_levels);
        const Philox ph{seed_lo, seed_hi};
        r = ph(0xC0DEu, key.tok, key.gid, my_t);
        my_rnd = r.x;
      }
      if (KNOWN) {
        const int kn = known[mine];
        if (kn >= 0) my_known = known_pick(my, kn, my_t, K, NOISE == VB200_NOISE_GREEDY, u01(r.x), u01(r.y));
      }
    }
    // x_t of the next batch's first token, so that the last prefetch of this batch has its column
    const int nb = base + 32 * stride;
    const int nb_xt = nb < n_tok ? x_t_all[nb] : 0;
    if (base == w0) prefetch(base, __shfl_sync(kFull, my.x_t, 0));

#pragma unroll 1
    for (int k = 0; k < 32; ++k) {
      const int tok = base + k * stride;
      if (tok >= n_tok) break;
      const int t = __shfl_sync(kFull, my_t, k);
      const int x_t = __shfl_sync(kFull, my.x_t, k);
      // lane owns classes j = c*256 + lane*8 + i  (c < KC, i < 8) in registers v[c*8 + i]
      float v[NR];
#pragma unroll
      for (int c = 0; c < KC; ++c) unpack8(nxt[c], v + c * 8);
      const float l_x = cvt1(nxt_lx), l_m = cvt1(nxt_lm);
      if (tok + stride < n_tok) {
        const int xt_next = __shfl_sync(kFull, my.x_t, (k + 1) & 31);
        prefetch(tok + stride, k == 31 ? nb_xt : xt_next);
      }
      if (KNOWN) {
        const int kp = __shfl_sync(kFull, my_known, k);
        if (kp >= 0) {
          if (lane == 0) x_out[tok] = kp;
          continue;
        }
      }
      // Row max; the arg max (lowest index wins ties) is only needed for greedy decoding and for
      // t == 0 (raw logits, no noise, ar_discrete.py:407,413), so the sampling path pays for a plain max.
      Best top{-INFINITY, 0x7fffffff};
      if (NOISE == VB200_NOISE_GREEDY || t == 0) {
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          const int j = (r >> 3) * 256 + lane * 8 + (r & 7);
          if (v[r] > top.v) { top.v = v[r]; top.j = j; }   // ascending j inside a lane
        }
        top = warp_best(top);
      } else {
        float m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3];
#pragma unroll
        for (int r = 4; r < NR; r += 4) {
          m0 = fmaxf(m0, v[r]); m1 = fmaxf(m1, v[r + 1]); m2 = fmaxf(m2, v[r + 2]); m3 = fmaxf(m3, v[r + 3]);
        }
        top.v = warp_max(fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)));
      }
      if (t == 0) {
        if (lane == 0) x_out[tok] = top.j;
        continue;
      }
      const float l2e = kLog2e * inv_temp;
      const float mx_l2 = -top.v * l2e;
      const uint64_t l2e2 = pack2(l2e, l2e), mxl2 = pack2(mx_l2, mx_l2);
      float part[KC];                                       // per-lane partial sums of e_j, one per 8-chunk
      float lane_sum = 0.f;
#pragma unroll
      for (int c = 0; c < KC; ++c) {
        uint64_t acc = 0ull;
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
          float x0, x1;
          unpack2(ffma2(pack2(v[c * 8 + i], v[c * 8 + i + 1]), l2e2, mxl2), x0, x1);
          const float e0 = exp2f_fast(x0), e1 = exp2f_fast(x1);
          v[c * 8 + i] = e0;
          v[c * 8 + i + 1] = e1;
          acc = fadd2(acc, pack2(e0, e1));
        }
        float a0, a1;
        unpack2(acc, a0, a1);
        part[c] = a0 + a1;
        lane_sum += part[c];
      }
      // inclusive warp scan of the lane sums (class order of the CDF = lane-major, any fixed order works)
      float incl = lane_sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float n = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += n;
      }
      const float e_x = exp2f_fast(fmaf(l_x, l2e, mx_l2));
      const float e_m = exp2f_fast(fmaf(l_m, l2e, mx_l2));
      const float Z = __shfl_sync(kFull, incl, 31);
      const float invZ = 1.0f / Z;

      // token k's scalars, from the lane that prepared them
      const PostScalars ps{__shfl_sync(kFull, my.f1_self, k), __shfl_sync(kFull, my.f1_oth, k),
                           __shfl_sync(kFull, my.a_gen, k),   __shfl_sync(kFull, my.c_gen, k),
                           __shfl_sync(kFull, my.a_m, k),     __shfl_sync(kFull, my.c_m, k), x_t, m_abs};
      const float coef = ps.cA() * invZ;                    // generic class: w_j = coef * e_j + cst
      const float cst = ps.cst();
      const PostSpecial w = post_special(ps, e_x, e_m, invZ, coef, cst);
      int pick;
      if (NOISE == VB200_NOISE_GREEDY) {
        pick = post_greedy(ps, w, fmaf(exp2f_fast(fmaf(top.v, l2e, mx_l2)), coef, cst), top.j);
      } else {
        const uint32_t rnd = __shfl_sync(kFull, my_rnd, k);
        const float w_generic = fmaf(coef, Z, static_cast<float>(K) * cst);
        float target = u01(rnd) * (w_generic + w.dx + w.dm);
        if (target < w.dx) {
          pick = x_t;
        } else if (target < w.dx + w.dm) {
          pick = m_abs;
        } else {
          target -= w.dx + w.dm;
          // lane-level CDF of the generic weights: lane sum = coef * sum(e) + NR * cst
          const float w_incl = fmaf(coef, incl, static_cast<float>((lane + 1) * NR) * cst);
          const unsigned ball = __ballot_sync(kFull, target < w_incl);
          const int src = ball ? __ffs(ball) - 1 : 31;      // rounding at the top end -> last lane
          // every lane walks its own 32 classes (branch-free, no divergence); the owner's answer is kept
          float run = w_incl - fmaf(coef, lane_sum, static_cast<float>(NR) * cst);   // weight before this lane
          int c_sel = 0;
          {
            float cum = run;
#pragma unroll
            for (int c = 0; c < KC - 1; ++c) {               // which 8-class chunk
              cum += fmaf(coef, part[c], 8.0f * cst);
              const bool past = target >= cum;
              c_sel += past ? 1 : 0;
              run = past ? cum : run;
            }
          }
          float e8[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            e8[i] = v[i];
#pragma unroll
            for (int c = 1; c < KC; ++c) e8[i] = c_sel == c ? v[c * 8 + i] : e8[i];
          }
          int i_sel = 0;                                     // prefix sums are monotone: count those <= target
#pragma unroll
          for (int i = 0; i < 7; ++i) {                      // rounding at the top end -> last class
            run += fmaf(coef, e8[i], cst);
            i_sel += target >= run ? 1 : 0;
          }
          pick = __shfl_sync(kFull, c_sel * 256 + lane * 8 + i_sel, src);
        }
      }
      if (lane == 0) x_out[tok] = pick;
    }
  }
}

template <typename T>
static int launch_posterior(int32_t* x_out, float* post_out, const void* logits, int64_t ld,
                            const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
                            const int32_t* utt, const float* table, int n_rows, int n_levels,
                            int K, int S, int tr, int noise, const float* uniforms,
                            uint64_t seed, const int32_t* known, float inv_temp, cudaStream_t st) {
  const int n_tok = n_rows * n_levels;
  const int wpb = 8;
  int grid = (n_tok + wpb - 1) / wpb;
  const int cap = num_sms() * 8 * 4;
  if (grid > cap) grid = cap;
  const uint32_t lo = static_cast<uint32_t>(seed), hi = static_cast<uint32_t>(seed >> 32);
  cudaError_t launch_rc = cudaSuccess;
  // production form: register-resident, single read of the logits (see posterior_fast_kernel)
  const bool aligned = (ld % 8 == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0);
  if (!post_out && aligned && noise != VB200_NOISE_UNIFORMS && K % 256 == 0 && K <= 1024) {
    const T* lg = static_cast<const T*>(logits);
#define VB_LAUNCH_F(KC, NZ)                                                                                  \
  launch_rc = known ? launch_pdl(posterior_fast_kernel<T, KC, NZ, true>, dim3(grid), dim3(wpb * 32), 0, st, 1, x_out, \
                                 lg, static_cast<int64_t>(ld), x_t, row_utt, t_utt, utt, table, n_rows, n_levels, S, \
                                 tr, lo, hi, known, inv_temp)                                                        \
                    : launch_pdl(posterior_fast_kernel<T, KC, NZ, false>, dim3(grid), dim3(wpb * 32), 0, st, 1, x_out, \
                                 lg, static_cast<int64_t>(ld), x_t, row_utt, t_utt, utt, table, n_rows, n_levels, S, \
                                 tr, lo, hi, known, inv_temp)
#define VB_LAUNCH_FK(NZ)                                              \
  switch (K / 256) {                                                  \
    case 1: VB_LAUNCH_F(1, NZ); break;                                \
    case 2: VB_LAUNCH_F(2, NZ); break;                                \
    case 3: VB_LAUNCH_F(3, NZ); break;                                \
    default: VB_LAUNCH_F(4, NZ); break;                               \
  }
    if (noise == VB200_NOISE_GREEDY) { VB_LAUNCH_FK(VB200_NOISE_GREEDY) } else { VB_LAUNCH_FK(VB200_NOISE_PHILOX) }
#undef VB_LAUNCH_FK
#undef VB_LAUNCH_F
    VB_CHECK_CUDA(launch_rc);
    VB_CHECK_CUDA(cudaGetLastError());
    return VB200_OK;
  }
#define VB_LAUNCH_P(NZ)                                                                        \
  launch_rc = launch_pdl(posterior_sample_kernel<T, NZ>, dim3(grid), dim3(wpb * 32), 0, st, 1, x_out, post_out,  \
                         static_cast<const T*>(logits), static_cast<int64_t>(ld), x_t, row_utt, t_utt, utt, table, \
                         n_rows, n_levels, K, S, tr, uniforms, lo, hi, known, inv_temp)
  if (noise == VB200_NOISE_PHILOX) VB_LAUNCH_P(VB200_NOISE_PHILOX);
  else if (noise == VB200_NOISE_UNIFORMS) VB_LAUNCH_P(VB200_NOISE_UNIFORMS);
  else VB_LAUNCH_P(VB200_NOISE_GREEDY);
#undef VB_LAUNCH_P
  VB_CHECK_CUDA(launch_rc);
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

// ---------------------------------------------------------------- plain categorical draw (NAR levels)
// One class per row from softmax(logits / tau), for the K the fused classifier head does not take: one warp per
// row, lane i owns the contiguous classes [i*per, (i+1)*per), and the code is the inverse CDF of one Philox uniform
// (the warp scan of the lane sums finds the lane, the lane walks its classes), as posterior_fast_kernel draws.
// Greedy: the arg max of the raw logits, lowest class wins ties.  The code goes to x_out[row * ld_out + col]; the
// Philox counter (CAT_STREAM_1, frame * 8 + level, global utterance id, 0) is used by no D3PM draw.
constexpr uint32_t CAT_STREAM_1 = 0xCA710000u;
template <typename T, int NOISE>
__global__ void __launch_bounds__(256) categorical_kernel(
    int32_t* __restrict__ x_out, int64_t ld_out, int col, const T* __restrict__ logits, int64_t ld_logits,
    const int32_t* __restrict__ row_utt, const int32_t* __restrict__ utt, int n_rows, int K, float inv_temp,
    uint32_t seed_lo, uint32_t seed_hi) {
  pdl_launch_dependents();
  pdl_wait();                                   // everything below reads / writes activations
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int per = (K + 31) / 32;
  const int j0 = min(lane * per, K), j1 = min(j0 + per, K);
  for (int row = blockIdx.x * warps_per_block + (threadIdx.x >> 5); row < n_rows;
       row += gridDim.x * warps_per_block) {
    const T* lrow = logits + static_cast<size_t>(row) * ld_logits;
    int pick;
    if (NOISE == VB200_NOISE_GREEDY) {
      Best best{-INFINITY, 0x7fffffff};
      for (int j = j0; j < j1; ++j) best_update(best, load_logit<T>(lrow, j), j);
      pick = warp_best(best).j;
    } else {
      float mx = -INFINITY;
      for (int j = j0; j < j1; ++j) mx = fmaxf(mx, load_logit<T>(lrow, j) * inv_temp);
      mx = warp_max(mx);
      float lane_sum = 0.f;
      for (int j = j0; j < j1; ++j) lane_sum += __expf(load_logit<T>(lrow, j) * inv_temp - mx);
      float incl = lane_sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      const float Z = __shfl_sync(0xffffffffu, incl, 31);
      const TokenKey key = token_key(utt, row_utt[row], row, col, static_cast<int>(ld_out));
      const uint4 r = Philox{seed_lo, seed_hi}(CAT_STREAM_1, key.tok, key.gid, 0u);
      const float target = u01(r.x) * Z;
      const unsigned ball = __ballot_sync(0xffffffffu, target < incl && j1 > j0);
      const int last = (K - 1) / per;                // last lane that owns a class: rounding at the top end
      const int src = ball ? __ffs(ball) - 1 : last;
      float run = incl - lane_sum;                   // mass before this lane's classes
      int idx = j0;
      for (int j = j0; j + 1 < j1; ++j) {            // prefix sums are monotone: count those <= target
        run += __expf(load_logit<T>(lrow, j) * inv_temp - mx);
        idx += target >= run ? 1 : 0;
      }
      pick = __shfl_sync(0xffffffffu, idx, src);
    }
    if (lane == 0) x_out[static_cast<size_t>(row) * ld_out + col] = pick;
  }
}

int categorical_from_logits(int32_t* x_out, int64_t ld_out, int col, const void* logits, vb200_dtype logits_dtype,
                            int64_t ld_logits, const int32_t* row_utt, const int32_t* utt, int n_rows, int K,
                            int noise, uint64_t seed, float inv_temp, cudaStream_t st) {
  const int wpb = 8;
  int grid = (n_rows + wpb - 1) / wpb;
  const int cap = num_sms() * 8 * 4;
  if (grid > cap) grid = cap;
  const uint32_t lo = static_cast<uint32_t>(seed), hi = static_cast<uint32_t>(seed >> 32);
  cudaError_t rc = cudaSuccess;
#define VB_LAUNCH_C(T)                                                                                               \
  rc = noise == VB200_NOISE_GREEDY                                                                                   \
           ? launch_pdl(categorical_kernel<T, VB200_NOISE_GREEDY>, dim3(grid), dim3(wpb * 32), 0, st, 1, x_out, ld_out, \
                        col, static_cast<const T*>(logits), ld_logits, row_utt, utt, n_rows, K, inv_temp, lo, hi)     \
           : launch_pdl(categorical_kernel<T, VB200_NOISE_PHILOX>, dim3(grid), dim3(wpb * 32), 0, st, 1, x_out, ld_out, \
                        col, static_cast<const T*>(logits), ld_logits, row_utt, utt, n_rows, K, inv_temp, lo, hi)
  switch (logits_dtype) {
    case VB200_F32: VB_LAUNCH_C(float); break;
    case VB200_BF16: VB_LAUNCH_C(__nv_bfloat16); break;
    case VB200_F16: VB_LAUNCH_C(__half); break;
    default:
      set_error("categorical: unknown logits dtype %d", static_cast<int>(logits_dtype));
      return VB200_ERR_INVALID;
  }
#undef VB_LAUNCH_C
  VB_CHECK_CUDA(rc);
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

__global__ void step_timesteps_kernel(int32_t* t_utt, int B, int delta) {
  pdl_launch_dependents();
  pdl_wait();                                   // everything below reads / writes activations
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) t_utt[i] += delta;
}

// t_utt[b] = next_t[t_utt[b]]: the successor of each utterance's timestep in the loop's schedule
__global__ void step_timesteps_to_kernel(int32_t* t_utt, int B, const int32_t* __restrict__ next_t, int S) {
  pdl_launch_dependents();
  pdl_wait();                                   // everything below reads / writes activations
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) t_utt[i] = next_t[clamp_timestep(t_utt[i], S)];
}

}  // namespace vb200

using namespace vb200;

extern "C" int vb200_q_sample(int32_t* x_out, const int32_t* x0, const int32_t* t_tok,
                              const int32_t* mask, const float* uniforms, const float* table,
                              int32_t n_tok, int32_t K, int32_t S, vb200_transition tr,
                              vb200_stream_t stream) {
  if (n_tok == 0) return VB200_OK;
  VB_REQUIRE(x_out && x0 && t_tok && uniforms && table, "q_sample: null pointer");
  VB_REQUIRE(n_tok >= 0 && K >= 2 && S >= 1, "q_sample: bad sizes n_tok=%d K=%d S=%d", n_tok, K, S);
  if (n_tok == 0) return VB200_OK;
  const int wpb = 8;
  int grid = (n_tok + wpb - 1) / wpb;
  const int cap = num_sms() * 32;
  if (grid > cap) grid = cap;
  q_sample_kernel<false><<<grid, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      x_out, x0, t_tok, mask, uniforms, table, nullptr, n_tok, K, S, static_cast<int>(tr));
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

extern "C" int vb200_q_sample_dense(int32_t* x_out, const int32_t* x0, const int32_t* t_tok,
                                    const int32_t* mask, const float* uniforms, const void* log_qbar_f16,
                                    int32_t n_tok, int32_t K, int32_t S, vb200_stream_t stream) {
  if (n_tok == 0) return VB200_OK;
  VB_REQUIRE(x_out && x0 && t_tok && uniforms && log_qbar_f16, "q_sample_dense: null pointer");
  VB_REQUIRE(n_tok >= 0 && K >= 2 && S >= 1, "q_sample_dense: bad sizes n_tok=%d K=%d S=%d", n_tok, K, S);
  const int wpb = 8;
  int grid = (n_tok + wpb - 1) / wpb;
  const int cap = num_sms() * 32;
  if (grid > cap) grid = cap;
  q_sample_kernel<true><<<grid, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      x_out, x0, t_tok, mask, uniforms, nullptr, static_cast<const __half*>(log_qbar_f16), n_tok, K, S,
      VB200_UNIFORM);
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

extern "C" int vb200_q_sample_philox(int32_t* x_out, const int32_t* x0, const int32_t* t_tok,
                                     const int32_t* mask, const float* table, int32_t n_tok, int32_t K,
                                     int32_t S, vb200_transition tr, uint64_t seed, vb200_stream_t stream) {
  if (n_tok == 0) return VB200_OK;
  VB_REQUIRE(x_out && x0 && t_tok && table, "q_sample_philox: null pointer");
  VB_REQUIRE(n_tok >= 0 && K >= 4 && S >= 1, "q_sample_philox: bad sizes n_tok=%d K=%d S=%d", n_tok, K, S);
  int grid = (n_tok + 255) / 256;
  const int cap = num_sms() * 8;
  if (grid > cap) grid = cap;
  VB_CHECK_CUDA(launch_pdl(q_sample_philox_kernel, dim3(grid), dim3(256), 0, static_cast<cudaStream_t>(stream), 1,
                           x_out, x0, t_tok, mask, table, n_tok, K, S, static_cast<int>(tr),
                           static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

extern "C" int vb200_posterior_sample_from_logits_temp(
    int32_t* x_out, float* post_out, const void* logits, vb200_dtype logits_dtype,
    int64_t ld_logits, const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
    const int32_t* utt, const float* table, int32_t n_rows, int32_t n_levels, int32_t K,
    int32_t S, vb200_transition tr, vb200_noise noise, const float* uniforms, uint64_t seed,
    const int32_t* known, float temperature, vb200_stream_t stream) {
  VB_REQUIRE(valid_temperature(temperature), "posterior: temperature must be finite and > 0, got %g",
             static_cast<double>(temperature));
  const float inv_temp = 1.0f / temperature;
  if (n_rows == 0) return VB200_OK;
  VB_REQUIRE(x_out && logits && x_t && row_utt && t_utt && table, "posterior: null pointer");
  VB_REQUIRE(n_rows >= 0 && n_levels >= 1 && K >= 2 && S >= 1, "posterior: bad sizes");
  VB_REQUIRE(ld_logits >= static_cast<int64_t>(n_levels) * K, "posterior: ld_logits too small");
  VB_REQUIRE(noise != VB200_NOISE_UNIFORMS || uniforms, "posterior: uniforms required");
  VB_REQUIRE(noise != VB200_NOISE_PHILOX || utt, "posterior: utt records required for Philox");
  if (n_rows == 0) return VB200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (logits_dtype) {
    case VB200_F32:
      return launch_posterior<float>(x_out, post_out, logits, ld_logits, x_t, row_utt, t_utt, utt,
                                     table, n_rows, n_levels, K, S, tr, noise, uniforms, seed, known, inv_temp, st);
    case VB200_BF16:
      return launch_posterior<__nv_bfloat16>(x_out, post_out, logits, ld_logits, x_t, row_utt,
                                             t_utt, utt, table, n_rows, n_levels, K, S, tr, noise,
                                             uniforms, seed, known, inv_temp, st);
    case VB200_F16:
      return launch_posterior<__half>(x_out, post_out, logits, ld_logits, x_t, row_utt, t_utt,
                                      utt, table, n_rows, n_levels, K, S, tr, noise, uniforms,
                                      seed, known, inv_temp, st);
  }
  set_error("posterior: unknown logits dtype %d", static_cast<int>(logits_dtype));
  return VB200_ERR_INVALID;
}

extern "C" int vb200_posterior_sample_from_logits_known(
    int32_t* x_out, float* post_out, const void* logits, vb200_dtype logits_dtype,
    int64_t ld_logits, const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
    const int32_t* utt, const float* table, int32_t n_rows, int32_t n_levels, int32_t K,
    int32_t S, vb200_transition tr, vb200_noise noise, const float* uniforms, uint64_t seed,
    const int32_t* known, vb200_stream_t stream) {
  return vb200_posterior_sample_from_logits_temp(x_out, post_out, logits, logits_dtype, ld_logits, x_t, row_utt,
                                                 t_utt, utt, table, n_rows, n_levels, K, S, tr, noise, uniforms,
                                                 seed, known, 1.0f, stream);
}

extern "C" int vb200_posterior_sample_from_logits(
    int32_t* x_out, float* post_out, const void* logits, vb200_dtype logits_dtype,
    int64_t ld_logits, const int32_t* x_t, const int32_t* row_utt, const int32_t* t_utt,
    const int32_t* utt, const float* table, int32_t n_rows, int32_t n_levels, int32_t K,
    int32_t S, vb200_transition tr, vb200_noise noise, const float* uniforms, uint64_t seed,
    vb200_stream_t stream) {
  return vb200_posterior_sample_from_logits_known(x_out, post_out, logits, logits_dtype, ld_logits, x_t, row_utt,
                                                  t_utt, utt, table, n_rows, n_levels, K, S, tr, noise, uniforms,
                                                  seed, nullptr, stream);
}

extern "C" int vb200_step_timesteps(int32_t* t_utt, int32_t B, int32_t delta,
                                    vb200_stream_t stream) {
  VB_REQUIRE(t_utt && B >= 0, "step_timesteps: bad arguments");
  if (B == 0) return VB200_OK;
  VB_CHECK_CUDA(launch_pdl(step_timesteps_kernel, dim3((B + 127) / 128), dim3(128), 0,
                           static_cast<cudaStream_t>(stream), 1, t_utt, B, delta));
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}

extern "C" int vb200_step_timesteps_to(int32_t* t_utt, int32_t B, const int32_t* next_t, int32_t S,
                                       vb200_stream_t stream) {
  VB_REQUIRE(t_utt && next_t && B >= 0 && S >= 1, "step_timesteps_to: bad arguments");
  if (B == 0) return VB200_OK;
  VB_CHECK_CUDA(launch_pdl(step_timesteps_to_kernel, dim3((B + 127) / 128), dim3(128), 0,
                           static_cast<cudaStream_t>(stream), 1, t_utt, B, next_t, S));
  VB_CHECK_CUDA(cudaGetLastError());
  return VB200_OK;
}
