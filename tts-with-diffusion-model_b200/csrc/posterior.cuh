// The D3PM reverse step q(x_{t-1} | x_t, p̂(x_0)) in closed form (ar_discrete.py:347-375), written once for
// the three kernels that draw from it: posterior_sample_kernel and posterior_fast_kernel (d3pm.cu) and
// head_sample_kernel, the classifier GEMM's epilogue (head_sample_tcgen05.cu).
//
// With e_j = exp(l_j - max), Z = sum e_j, p_j = e_j / Z the unnormalised posterior weight is
//   w_j = (f1_j + eps) (f2_j + eps),  f1_j = Q_t[j, x_t],  f2_j + eps = p_j (a_j - c_j) + c_j + eps,
// a_j = Qbar_{t-1}[j, j], c_j = Qbar_{t-1}[i, j] (i != j).  Every class except x_t (and the absorbing class m)
// shares f1 / a / c, so a generic class weighs  w_j = coef e_j + cst  with coef = cA / Z, and
//   sum_j w_j = cA + K cst + dx + dm,
// where dx, dm >= 0 are what x_t and m weigh beyond the generic formula (DESIGN.md).
#pragma once
#include "common.cuh"

namespace vb200 {

constexpr float kLog2e = 1.4426950408889634f;

// a token's timestep, clamped into the table as the reference indexes it
__device__ __forceinline__ int clamp_timestep(int t, int S) { return min(max(t, 0), S - 1); }

// Per-token scalars of the reverse step (at t == 0 the reference takes the raw logits and none of this applies).
struct PostScalars {
  float f1_self, f1_oth;   // Q_t[x_t, x_t] + eps, Q_t[j, x_t] + eps for j != x_t
  float a_gen, c_gen;      // a, c of a generic class
  float a_m, c_m;          // a, c of the absorbing class (the generic pair for the uniform transition)
  int x_t, m;              // m = K / 2 for the absorbing transition, -1 for the uniform one
  __device__ __forceinline__ bool at_m() const { return m >= 0 && x_t == m; }
  __device__ __forceinline__ bool has_m() const { return m >= 0 && x_t != m; }   // m is a special class
  __device__ __forceinline__ float cA() const { return (a_gen - c_gen) * f1_oth; }
  __device__ __forceinline__ float cst() const { return (c_gen + kEps) * f1_oth; }
};

// t: clamped timestep.  The only reader of the Q_t / Qbar_{t-1} entries of the scalar table.  A schedule table
// (d3pm.schedule_table) holds Q_{t|s} and Qbar_s in those places for a step that jumps from t to s, so the same
// reads give the jump posterior q(x_s | x_t, x̂0).
__device__ __forceinline__ PostScalars post_scalars(const float* __restrict__ table, int t, int x_t, int K,
                                                    int transition) {
  const float* one = table + static_cast<size_t>(t) * VB200_TAB_STRIDE;
  const float* cum = table + static_cast<size_t>(max(t - 1, 0)) * VB200_TAB_STRIDE;
  const bool absorbing = transition == VB200_ABSORBING;
  PostScalars s;
  s.x_t = x_t;
  s.m = absorbing ? K / 2 : -1;
  const bool at_m = s.at_m();
  s.f1_self = (at_m ? one[VB200_TAB_ONE_BOTH] : one[VB200_TAB_ONE_KEEP]) + kEps;
  s.f1_oth = (at_m ? one[VB200_TAB_ONE_ABSORB] : one[VB200_TAB_ONE_OFF]) + kEps;
  s.a_gen = cum[VB200_TAB_CUM_KEEP];
  s.c_gen = cum[VB200_TAB_CUM_OFF];
  s.a_m = absorbing ? cum[VB200_TAB_CUM_BOTH] : s.a_gen;
  s.c_m = absorbing ? cum[VB200_TAB_CUM_ABSORB] : s.c_gen;
  return s;
}

// Weights of the special classes and their excess over the generic formula coef * e + cst.
struct PostSpecial { float w_x, dx, w_m, dm; };
// e_x, e_m: exp(l - max) of classes x_t and m; coef = cA / Z; cst = PostScalars::cst()
__device__ __forceinline__ PostSpecial post_special(const PostScalars& s, float e_x, float e_m, float invZ, float coef,
                                                    float cst) {
  const bool at_m = s.at_m(), has_m = s.has_m();
  PostSpecial w;
  w.w_x = s.f1_self * fmaf(e_x * invZ, at_m ? s.a_m - s.c_m : s.a_gen - s.c_gen, (at_m ? s.c_m : s.c_gen) + kEps);
  w.dx = fmaxf(w.w_x - fmaf(e_x, coef, cst), 0.f);
  w.w_m = has_m ? s.f1_oth * fmaf(e_m * invZ, s.a_m - s.c_m, s.c_m + kEps) : 0.f;
  w.dm = has_m ? fmaxf(w.w_m - fmaf(e_m, coef, cst), 0.f) : 0.f;
  return w;
}

// Greedy decoding, the arg max of the weights: generic weights are monotone in the logit and the special classes
// only gain, so the candidates are the top generic class (weight top_w, class top_j), x_t and m.  The lowest
// class wins ties.
__device__ __forceinline__ int post_greedy(const PostScalars& s, const PostSpecial& w, float top_w, int top_j) {
  float best_w = top_w;
  int pick = top_j;
  if (top_j == s.x_t) best_w = w.w_x;
  else if (top_j == s.m) best_w = w.w_m;
  if (w.w_x > best_w || (w.w_x == best_w && s.x_t < pick)) { best_w = w.w_x; pick = s.x_t; }
  if (s.has_m() && (w.w_m > best_w || (w.w_m == best_w && s.m < pick))) pick = s.m;
  return pick;
}

// A token whose x0 is given (generate_audio(known_list=...)): the reverse step draws from q(x_s | x_t, x0 = k),
//   w_j = (Q_{t|s}[j, x_t] + eps) (Qbar_s[k, j] + eps),
// the ids form of ar_discrete.py:347-375.  Row k of Qbar_s is CUM_BOTH / CUM_KEEP at j = k (k = m or not),
// CUM_ABSORB at j = m != k and CUM_OFF elsewhere, so at most three classes {x_t, k, m} weigh something of their
// own and the K - n others share one weight: the law is drawn in O(1) without reading a logit.
// f1 = Q_{t|s}[j, x_t] + eps and f2 = Qbar_s[k, j] of class j
__device__ __forceinline__ float2 known_factors(const PostScalars& s, int k, int j) {
  return make_float2(j == s.x_t ? s.f1_self : s.f1_oth,
                     j == k ? (j == s.m ? s.a_m : s.a_gen) : (j == s.m ? s.c_m : s.c_gen));
}
__device__ __forceinline__ float known_weight(const PostScalars& s, int k, int j) {
  const float2 f = known_factors(s, k, j);
  return f.x * (f.y + kEps);
}

// The special classes of a known token in ascending order, padded with kNone (n of them are classes), their
// weights (0 for padding) and the weight every other class shares.  Fixed indices only: it stays in registers.
constexpr int kNone = 0x7fffffff;
struct KnownLaw {
  int c[3], n;
  float w[3], w_gen;
};
__device__ __forceinline__ KnownLaw known_law(const PostScalars& s, int k) {
  KnownLaw l;
  const int c1 = k != s.x_t ? k : kNone;
  const int c2 = (s.m >= 0 && s.m != s.x_t && s.m != k) ? s.m : kNone;
  const int lo = min(s.x_t, c1), hi = max(s.x_t, c1);
  l.c[0] = min(lo, c2);
  l.c[1] = max(lo, min(hi, c2));
  l.c[2] = max(hi, c2);
  l.n = 1 + (c1 != kNone ? 1 : 0) + (c2 != kNone ? 1 : 0);
#pragma unroll
  for (int i = 0; i < 3; ++i) l.w[i] = l.c[i] != kNone ? known_weight(s, k, l.c[i]) : 0.f;
  l.w_gen = s.f1_oth * (s.c_gen + kEps);
  return l;
}

// The reverse step of a known token k.  greedy: the arg max of w, lowest class winning ties (the generic
// candidate is the lowest class that is not special).  Otherwise a draw from u0 (which group: a special class
// or the generic ones) and u1 (which generic class, uniformly, special classes skipped).  t == 0 returns k.
__device__ __forceinline__ int known_pick(const PostScalars& s, int k, int t, int K, bool greedy, float u0, float u1) {
  if (t == 0) return k;
  const KnownLaw l = known_law(s, k);
  const int n_gen = K - l.n;
  if (greedy) {
    int g0 = 0;                                          // lowest generic class
#pragma unroll
    for (int i = 0; i < 3; ++i) g0 += g0 == l.c[i] ? 1 : 0;
    float best_w = n_gen > 0 ? l.w_gen : -1.f;
    int pick = n_gen > 0 ? g0 : kNone;
#pragma unroll
    for (int i = 0; i < 3; ++i)
      if (l.c[i] != kNone && (l.w[i] > best_w || (l.w[i] == best_w && l.c[i] < pick))) { best_w = l.w[i]; pick = l.c[i]; }
    return pick;
  }
  float target = u0 * (l.w[0] + l.w[1] + l.w[2] + static_cast<float>(n_gen) * l.w_gen);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    if (l.c[i] != kNone && target < l.w[i]) return l.c[i];
    target -= l.w[i];
  }
  if (n_gen <= 0) return l.n == 3 ? l.c[2] : (l.n == 2 ? l.c[1] : l.c[0]);   // rounding at the top end, K == n
  int j = min(static_cast<int>(u1 * static_cast<float>(n_gen)), n_gen - 1);
#pragma unroll
  for (int i = 0; i < 3; ++i) j += j >= l.c[i] ? 1 : 0;  // skip the special classes, ascending
  return j;
}

// log w_j of a known token: the posterior logits of the ids form (post_out, Gumbel-max with supplied uniforms)
__device__ __forceinline__ float known_logit(const PostScalars& s, int k, int j) {
  const float2 f = known_factors(s, k, j);
  return logf(f.x) + logf(f.y + kEps);
}

// Philox counter words of a token's draws: (frame * n_levels + level, global utterance id), which do not depend on
// how the batch is packed or sharded.  b: the token's utterance, row: its packed response row.
struct TokenKey { uint32_t tok, gid; };
__device__ __forceinline__ TokenKey token_key(const int32_t* __restrict__ utt, int b, int row, int level,
                                              int n_levels) {
  const int32_t* ur = utt + static_cast<size_t>(b) * VB200_U_STRIDE;
  return TokenKey{static_cast<uint32_t>(row - ur[VB200_U_RESP0]) * n_levels + level,
                  static_cast<uint32_t>(ur[VB200_U_GID])};
}

}  // namespace vb200
