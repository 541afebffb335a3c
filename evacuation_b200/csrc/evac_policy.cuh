// Fused forward of the RPO transformer-embedding actor-critic -- the consumer of the step kernel in the rollout loop
// of BASELINE config 5 (SURVEY section 8 row f1).  Reference (paths relative to /root/reference/src/agents):
//   networks/rpo_transformer_agent_network.py:36-75    MultiHeadAttention  (set attention: d_model is the batch-of-heads
//                                                       axis, num_heads the contracted axis, scale = sqrt(d_model))
//   networks/rpo_transformer_agent_network.py:78-131   TransformerBlock    (attn -> dropout -> [resid] -> LayerNorm ->
//                                                       Linear, Dropout, ReLU, Linear -> dropout -> [resid] -> LayerNorm)
//   networks/rpo_transformer_agent_network.py:133-163  RPOTransformerEmbedding
//   networks/rpo_linear_agent_network.py:19-61         RPOLinearNetwork    (critic / actor_mean MLPs, Normal sampling)
//   rpo_agent.py:24-33                                 NormalizeObservation + clip, NormalizeReward + clip (gymnasium)
//
// Two kernels, float32 throughout (nothing here is a large dense contraction: K = 3 / 6 / 96 / 372):
//   evac_policy_embed_kernel<D, H, TRAIN>   one WARP per environment, lane L owns observation rows L and L + 32
//       (S = N + 2 <= 64 rows of D values).  Both transformer blocks run out of registers; the only shared-memory
//       traffic is the (k, v) tile of ONE pseudo-head d at a time (2 * H * 64 floats per warp) and the packed
//       weights (broadcast LDS.128, ~8 KB per block, loaded once per CTA).  Scores, the softmax shift, the
//       probability-weighted value sums, the projections and the feed-forward all run on packed f32x2 instructions:
//       the attention packs two keys (j, j + 1) per instruction, the projections / feed-forward pack two output
//       features.  Softmax uses the Cauchy-Schwarz bound |q| max_j |k_j| as its shift (no max pass; a row whose
//       bound is so loose that the sum underflows is redone with the exact maximum).  Optional prologue: the per-env
//       NormalizeObservation update + clip.  Optional dropout (training mode, like the reference's rollouts which never
//       call .eval()): counter-hash Bernoulli masks keyed by (seed, offset, env, block, row, element).
//   evac_policy_heads_kernel<NH>            32 environments per CTA: X tile [32, S*D] in shared memory, the first
//       layers of critic and actor as ONE [S*D] x [2*NH] register-tiled product (weights streamed from L2, coalesced),
//       tanh, the two NH x NH layers, the output layers, then Normal sampling (Philox4x32 Box-Muller), log-probability,
//       entropy and the clipped action (ClipAction).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "evac_policy_ops.cuh"
#include "philox.cuh"

namespace evacp {

constexpr int PW_WARPS = 4;  // environments (warps) per CTA of the embedding kernel
constexpr int PW_MINB = 4;   // resident CTAs per SM the embedding kernel's register allocation is sized for
constexpr int PW_MAX_S = 64;  // rows per environment handled by one warp

__host__ __device__ constexpr int round_up(int a, int b) { return (a + b - 1) / b * b; }

// Packed (shared-memory) layout of ONE transformer block, in floats; every section starts on a float4 boundary.
template <int D, int H>
struct EmbLayout {
  static constexpr int QP = round_up(3 * H, 4);  // outputs [q(H) | k(H) | v(H)] of one (d, c) weight column, padded
  static constexpr int DP = round_up(D, 4);
  static constexpr int QKV_W = 0;                     // [(d * D + c) * QP + t]   t = h | H + h | 2H + h
  static constexpr int QKV_B = QKV_W + D * D * QP;    // [d * QP + t]
  static constexpr int WD = QKV_B + D * QP;           // [(d * H + h) * DP + c] = dense.weight[c][d * H + h]
  static constexpr int BD = WD + D * H * DP;
  static constexpr int LN1G = BD + DP, LN1B = LN1G + DP;
  static constexpr int B2 = LN1B + DP;
  static constexpr int LN2G = B2 + DP, LN2B = LN2G + DP;
  static constexpr int FF = LN2B + DP;                // groups of 4 hidden features: [b1(4) | W1[c](4) x D | W2[c](4) x D]
  static constexpr int GS = 4 + 8 * D;
  __host__ __device__ static constexpr int stride(int F4) { return FF + (F4 / 4) * GS; }  // F4 = d_ff rounded up to 4
};

struct PArgs {
  int E, S, F4, NB;
  int use_resid;
  float ln_eps, qscale;          // qscale = log2(e) / sqrt(D)
  float drop_scale;              // 1 / (1 - p)
  uint32_t drop_thresh;          // round(p * 65536): a 16-bit word below it drops the element
  uint32_t seed_lo, seed_hi;
  unsigned long long offset;     // + *offset_dev when set (a device counter survives CUDA-graph replay)
  const unsigned long long* offset_dev;
  long long env_offset;
  const float* obs;              // [E, S*D] (raw when the normaliser pointers are set, else already normalised)
  float* emb;                    // [E, S*D] out
  float* norm_mean;              // optional fused NormalizeObservation: [E, S*D] running mean / variance (in place)
  float* norm_var;
  const double* norm_count;      // device scalar: samples seen so far (the caller advances it)
  float* obs_norm;               // optional [E, S*D] out: the normalised, clipped observation (rollout storage)
  float norm_eps, norm_clip;
  const float* w;                // NB packed blocks (EmbLayout), device
  int wstride;
};

__device__ __forceinline__ float2 splat(float v) { return make_float2(v, v); }
__device__ __forceinline__ float2 lo(const float4& v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ float2 hi(const float4& v) { return make_float2(v.z, v.w); }
__device__ __forceinline__ float ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

__host__ __device__ __forceinline__ uint32_t fmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}
// Dropout stream (host-callable, so that the tests can pin their restatement of it to this code).  An element is dropped when
// its 16-bit word is below round(p * 65536).
// base key of one forward call: (seed, stream offset, global env index)
__host__ __device__ __forceinline__ uint32_t drop_base_key(uint32_t seed_lo, uint32_t seed_hi, unsigned long long off, uint32_t env_g) {
  return fmix32(seed_lo ^ fmix32(env_g * 0x9E3779B1u + (uint32_t)off) ^ (seed_hi * 0x85EBCA77u) ^ ((uint32_t)(off >> 32) * 0xC2B2AE3Du));
}
// key of the (block, row) stream
__host__ __device__ __forceinline__ uint32_t drop_row_key(uint32_t base, int blk, int row) {
  return fmix32(base ^ ((uint32_t)(blk * PW_MAX_S + row) * 0x27D4EB2Fu));
}
// 16-bit word k of the (env, block, row) stream: k = c for the attention output, k = 8 + c for the block output
__host__ __device__ __forceinline__ uint32_t drop_word(uint32_t row_key, uint32_t k) {
  const uint32_t t = fmix32(row_key + (k >> 1) * 0x9E3779B9u);
  return (k & 1u) ? (t >> 16) : (t & 0xFFFFu);
}
// feed-forward group g (hidden features 4g .. 4g + 3): feature 4g + 2i + j reads 16-bit half j of word i, word 0 = drop_ff_word and
// word 1 = drop_ff_mix of it (a cheap second mix: multiply + xor-shift)
__host__ __device__ __forceinline__ uint32_t drop_ff_word(uint32_t row_key, uint32_t g) { return fmix32(row_key + (8u + g) * 0x9E3779B9u); }
// the second mix of the words of a lane's two rows at once: one call keeps the kernel's instruction order and register allocation
__host__ __device__ __forceinline__ uint2 drop_ff_mix(uint32_t ta, uint32_t tb) {
  uint32_t a = ta * 0x9E3779B1u, b = tb * 0x9E3779B1u;
  a ^= a >> 15; b ^= b >> 15;
  return make_uint2(a, b);
}
// half j of word w dropped, compared in place against th16 = threshold << 16 (the lower half shifted up, the upper half as it is)
__host__ __device__ __forceinline__ bool drop_ff_dropped(uint32_t w, int j, uint32_t th16) { return (j ? w : w << 16) < th16; }
__device__ __forceinline__ float drop_mask(uint32_t row_key, uint32_t k, const PArgs& a) {
  return drop_word(row_key, k) < a.drop_thresh ? 0.f : a.drop_scale;
}

template <int D>
__device__ __forceinline__ void load_row(const float* __restrict__ p, float (&x)[D]) {
  if constexpr (D % 2 == 0) {
#pragma unroll
    for (int c = 0; c < D; c += 2) { const float2 v = *reinterpret_cast<const float2*>(p + c); x[c] = v.x; x[c + 1] = v.y; }
  } else {
#pragma unroll
    for (int c = 0; c < D; ++c) x[c] = p[c];
  }
}
template <int D>
__device__ __forceinline__ void store_row(float* __restrict__ p, const float (&x)[D]) {
  if constexpr (D % 2 == 0) {
#pragma unroll
    for (int c = 0; c < D; c += 2) *reinterpret_cast<float2*>(p + c) = make_float2(x[c], x[c + 1]);
  } else {
#pragma unroll
    for (int c = 0; c < D; ++c) p[c] = x[c];
  }
}

// nn.LayerNorm over the D values of one row (biased variance, eps inside the square root)
template <int D>
__device__ __forceinline__ void layer_norm(float (&x)[D], const float* __restrict__ g, const float* __restrict__ b, float eps) {
  float mu = 0.f;
#pragma unroll
  for (int c = 0; c < D; ++c) mu += x[c];
  mu *= (1.f / D);
  float var = 0.f;
#pragma unroll
  for (int c = 0; c < D; ++c) { x[c] -= mu; var = fmaf(x[c], x[c], var); }
  const float r = rsqrtf(var * (1.f / D) + eps);
#pragma unroll
  for (int c = 0; c < D; ++c) x[c] = fmaf(x[c] * r, g[c], b[c]);
}

// exact-maximum softmax row (slow path of the attention; also the restatement the fast path must agree with)
template <int H>
__device__ __noinline__ void attn_row_exact(const float* __restrict__ ks, const float* __restrict__ vs, int S, const float (&q)[H],
                                            float (&out)[H]) {
  float m = -INFINITY;
  for (int j = 0; j < S; ++j) {
    float s = 0.f;
#pragma unroll
    for (int h = 0; h < H; ++h) s = fmaf(q[h], ks[h * PW_MAX_S + j], s);
    m = fmaxf(m, s);
  }
  float l = 0.f, acc[H];
#pragma unroll
  for (int h = 0; h < H; ++h) acc[h] = 0.f;
  for (int j = 0; j < S; ++j) {
    float s = -m;
#pragma unroll
    for (int h = 0; h < H; ++h) s = fmaf(q[h], ks[h * PW_MAX_S + j], s);
    const float p = exp2f(s);
    l += p;
#pragma unroll
    for (int h = 0; h < H; ++h) acc[h] = fmaf(p, vs[h * PW_MAX_S + j], acc[h]);
  }
#pragma unroll
  for (int h = 0; h < H; ++h) out[h] = acc[h] / l;
}

// four keys j .. j+3 against the two query rows (a, b) of this lane.  Scores are packed over key PAIRS (query as the
// scalar-broadcast operand); the probabilities, the normaliser and the probability-weighted value sums are packed over the
// two ROWS: acc[h] = (row a, row b) += (p_a, p_b) * v_j[h] with the value as the 32-bit broadcast operand and (p_a, p_b)
// shared by the H consecutive instructions of a key -- the FMA pipe's full-rate operand forms (DESIGN.md 3.1: three distinct
// 64-bit sources run at 61 %), and the sums run over the keys in index order.
template <int H, bool TAIL>
__device__ __forceinline__ void attn_group(const float* __restrict__ ks, const float* __restrict__ vs, int j, int nvalid,
                                           const float2 (&qa)[H], const float2 (&qb)[H], float2 nma, float2 nmb,
                                           float2& l, float2 (&acc)[H]) {
  float4 k4[H], v4[H];
#pragma unroll
  for (int h = 0; h < H; ++h) {
    k4[h] = *reinterpret_cast<const float4*>(ks + h * PW_MAX_S + j);
    v4[h] = *reinterpret_cast<const float4*>(vs + h * PW_MAX_S + j);
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    float2 sa = nma, sb = nmb;
#pragma unroll
    for (int h = 0; h < H; ++h) {
      const float2 kk = half ? hi(k4[h]) : lo(k4[h]);
      sa = __ffma2_rn(qa[h], kk, sa);
      sb = __ffma2_rn(qb[h], kk, sb);
    }
    float2 p0 = make_float2(ex2(sa.x), ex2(sb.x)), p1 = make_float2(ex2(sa.y), ex2(sb.y));  // key 2 half, key 2 half + 1: (row a, row b)
    if (TAIL) {
      if (2 * half >= nvalid) p0 = make_float2(0.f, 0.f);
      if (2 * half + 1 >= nvalid) p1 = make_float2(0.f, 0.f);
    }
    l = __fadd2_rn(l, p0);
    l = __fadd2_rn(l, p1);
#pragma unroll
    for (int h = 0; h < H; ++h) acc[h] = __ffma2_rn(p0, splat(half ? v4[h].z : v4[h].x), acc[h]);
#pragma unroll
    for (int h = 0; h < H; ++h) acc[h] = __ffma2_rn(p1, splat(half ? v4[h].w : v4[h].y), acc[h]);
  }
}

// FROZEN: evaluation with the normaliser's statistics read-only (EvacPolicyIO.norm_frozen); instantiated with TRAIN = false only
template <int D, int H, bool TRAIN, bool FROZEN = false>
__global__ void __launch_bounds__(PW_WARPS * 32, PW_MINB) evac_policy_embed_kernel(const __grid_constant__ PArgs a) {
  static_assert(!(TRAIN && FROZEN), "evaluation runs without dropout");
  using L = EmbLayout<D, H>;
  extern __shared__ float4 smem4[];
  float* wsm = reinterpret_cast<float*>(smem4);
  {  // packed weights: once per CTA
    const int n4 = a.NB * a.wstride / 4;
    const float4* __restrict__ src = reinterpret_cast<const float4*>(a.w);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) smem4[i] = src[i];
    if (TRAIN) {
      // dropout of the hidden layer: relu(m s h) W2 = relu(m h) (s W2) for s = 1 / (1 - p) > 0 -- the scale is folded into the
      // staged copy of W2, the mask only zeroes
      __syncthreads();
      const int groups = a.F4 >> 2;
      for (int i = threadIdx.x; i < a.NB * groups * 4 * D; i += blockDim.x) {
        const int b = i / (groups * 4 * D), r = i - b * (groups * 4 * D), g = r / (4 * D), t = r - g * (4 * D);
        wsm[b * a.wstride + L::FF + g * L::GS + 4 + 4 * D + t] *= a.drop_scale;
      }
    }
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * PW_WARPS + warp;
  if (e >= a.E) return;
  float* ks = wsm + a.NB * a.wstride + warp * (2 * H * PW_MAX_S);
  float* vs = ks + H * PW_MAX_S;
  const int S = a.S;
  const int ra = lane, rb = lane + 32;
  const bool va = ra < S, vb = rb < S;
  const size_t row0 = (size_t)e * S * D;

  // ---------------- load the two rows (+ fused NormalizeObservation: gymnasium RunningMeanStd, one sample per step)
  float xa[D], xb[D];
#pragma unroll
  for (int c = 0; c < D; ++c) xa[c] = xb[c] = 0.f;
  if (va) load_row<D>(a.obs + row0 + ra * D, xa);
  if (vb) load_row<D>(a.obs + row0 + rb * D, xb);
  if (FROZEN && a.norm_mean != nullptr) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k == 0 ? va : vb) {
        float (&x)[D] = k == 0 ? xa : xb;
        const size_t off = row0 + (k == 0 ? ra : rb) * D;
        float mean[D], var[D];
        load_row<D>(a.norm_mean + off, mean);
        load_row<D>(a.norm_var + off, var);
#pragma unroll
        for (int c = 0; c < D; ++c) x[c] = norm_frozen(x[c], mean[c], var[c], a.norm_eps, a.norm_clip);
        if (a.obs_norm != nullptr) store_row<D>(a.obs_norm + off, x);
      }
    }
  } else if (a.norm_mean != nullptr) {
    const double cnt = *a.norm_count, tot = cnt + 1.0;
    const float w_new = (float)(1.0 / tot), w_old = (float)(cnt / tot);
    const float w_mix = __fmul_rn(w_old, w_new);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k == 0 ? va : vb) {
        float (&x)[D] = k == 0 ? xa : xb;
        const size_t off = row0 + (k == 0 ? ra : rb) * D;
        float mean[D], var[D];
        load_row<D>(a.norm_mean + off, mean);
        load_row<D>(a.norm_var + off, var);
#pragma unroll
        for (int c = 0; c < D; ++c) {
          const float delta = __fsub_rn(x[c], mean[c]);
          mean[c] = __fadd_rn(mean[c], __fmul_rn(delta, w_new));
          var[c] = __fadd_rn(__fmul_rn(var[c], w_old), __fmul_rn(__fmul_rn(delta, delta), w_mix));
          const float z = __fmul_rn(__fsub_rn(x[c], mean[c]), rsqrtf(__fadd_rn(var[c], a.norm_eps)));
          x[c] = min_nan(max_nan(z, -a.norm_clip), a.norm_clip);
        }
        store_row<D>(a.norm_mean + off, mean);
        store_row<D>(a.norm_var + off, var);
        if (a.obs_norm != nullptr) store_row<D>(a.obs_norm + off, x);
      }
    }
  }

  const uint32_t env_g = (uint32_t)(a.env_offset + e);
  uint32_t drop_base = 0;
  if (TRAIN) {
    const unsigned long long off = a.offset + (a.offset_dev ? *a.offset_dev : 0ull);
    drop_base = drop_base_key(a.seed_lo, a.seed_hi, off, env_g);
  }
  for (int blk = 0; blk < a.NB; ++blk) {
    const float* __restrict__ W = wsm + blk * a.wstride;
    uint32_t key_a = 0, key_b = 0;
    if (TRAIN) {
      key_a = drop_row_key(drop_base, blk, ra);
      key_b = drop_row_key(drop_base, blk, rb);
    }
    // ---------------- set attention [rpo_transformer_agent_network.py:57-75]
    float ya[D], yb[D];
#pragma unroll
    for (int c = 0; c < D; ++c) ya[c] = yb[c] = W[L::BD + c];
    float2 xsa[D], xsb[D];
#pragma unroll
    for (int c = 0; c < D; ++c) { xsa[c] = splat(xa[c]); xsb[c] = splat(xb[c]); }
#pragma unroll 1
    for (int d = 0; d < D; ++d) {
      // q, k, v of pseudo-head d: output feature h * D + d of Wq / Wk / Wv (split_heads views [.., H, D] and permutes)
      float2 pa[L::QP / 2], pb[L::QP / 2];
      {
        const float4* __restrict__ bq = reinterpret_cast<const float4*>(W + L::QKV_B + d * L::QP);
#pragma unroll
        for (int t = 0; t < L::QP / 4; ++t) {
          const float4 b = bq[t];
          pa[2 * t] = pb[2 * t] = lo(b);
          pa[2 * t + 1] = pb[2 * t + 1] = hi(b);
        }
      }
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const float4* __restrict__ wq = reinterpret_cast<const float4*>(W + L::QKV_W + (d * D + c) * L::QP);
#pragma unroll
        for (int t = 0; t < L::QP / 4; ++t) {
          const float4 w = wq[t];
          pa[2 * t] = __ffma2_rn(xsa[c], lo(w), pa[2 * t]);
          pa[2 * t + 1] = __ffma2_rn(xsa[c], hi(w), pa[2 * t + 1]);
          pb[2 * t] = __ffma2_rn(xsb[c], lo(w), pb[2 * t]);
          pb[2 * t + 1] = __ffma2_rn(xsb[c], hi(w), pb[2 * t + 1]);
        }
      }
      auto flat = [](const float2* p, int t) { return (t & 1) ? p[t >> 1].y : p[t >> 1].x; };
      float qa[H], qb[H];
      float kn_a = 0.f, kn_b = 0.f, qn_a = 0.f, qn_b = 0.f;
#pragma unroll
      for (int h = 0; h < H; ++h) {
        qa[h] = flat(pa, h) * a.qscale;
        qb[h] = flat(pb, h) * a.qscale;
        const float ka = flat(pa, H + h), kb = flat(pb, H + h);
        ks[h * PW_MAX_S + ra] = ka;
        ks[h * PW_MAX_S + rb] = kb;
        vs[h * PW_MAX_S + ra] = flat(pa, 2 * H + h);
        vs[h * PW_MAX_S + rb] = flat(pb, 2 * H + h);
        kn_a = fmaf(ka, ka, kn_a); kn_b = fmaf(kb, kb, kn_b);
        qn_a = fmaf(qa[h], qa[h], qn_a); qn_b = fmaf(qb[h], qb[h], qn_b);
      }
      // softmax shift: q.k_j <= |q| max_j |k_j|   (non-negative floats order like their bit patterns -> one REDUX)
      const float kn = fmaxf(va ? kn_a : 0.f, vb ? kn_b : 0.f);
      const float kmax = sqrtf(__uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(kn))));
      const float2 nma = splat(-sqrtf(qn_a) * kmax), nmb = splat(-sqrtf(qn_b) * kmax);
      float2 qa2[H], qb2[H], acc[H];   // acc[h] = (row a, row b)
#pragma unroll
      for (int h = 0; h < H; ++h) { qa2[h] = splat(qa[h]); qb2[h] = splat(qb[h]); acc[h] = make_float2(0.f, 0.f); }
      float2 l = make_float2(0.f, 0.f);
      __syncwarp();
      int j = 0;
#pragma unroll 2
      for (; j + 4 <= S; j += 4) attn_group<H, false>(ks, vs, j, 4, qa2, qb2, nma, nmb, l, acc);
      if (j < S) attn_group<H, true>(ks, vs, j, S - j, qa2, qb2, nma, nmb, l, acc);
      float oa[H], ob[H];
      const float sum_a = l.x, sum_b = l.y;
      {
        const float ia = 1.f / sum_a, ib = 1.f / sum_b;
#pragma unroll
        for (int h = 0; h < H; ++h) { oa[h] = acc[h].x * ia; ob[h] = acc[h].y * ib; }
      }
      // a bound so loose that every term underflowed (or a non-finite input): redo the row with the exact maximum
      const bool bad_a = va && !(sum_a >= 1e-30f && sum_a <= 3e38f), bad_b = vb && !(sum_b >= 1e-30f && sum_b <= 3e38f);
      if (__any_sync(0xffffffffu, bad_a || bad_b)) {
        if (bad_a) attn_row_exact<H>(ks, vs, S, qa, oa);
        if (bad_b) attn_row_exact<H>(ks, vs, S, qb, ob);
      }
      // dense: y[c] += out[d][h] * dense.weight[c][d * H + h]   (flatten(-2, -1) of [.., D, H])
#pragma unroll
      for (int h = 0; h < H; ++h) {
        const float* __restrict__ wd = W + L::WD + (d * H + h) * L::DP;
#pragma unroll
        for (int c = 0; c < D; ++c) { ya[c] = fmaf(oa[h], wd[c], ya[c]); yb[c] = fmaf(ob[h], wd[c], yb[c]); }
      }
      __syncwarp();  // the (k, v) tile is rewritten by the next pseudo-head
    }
    if (TRAIN) {
#pragma unroll
      for (int c = 0; c < D; ++c) { ya[c] *= drop_mask(key_a, c, a); yb[c] *= drop_mask(key_b, c, a); }
    }
#pragma unroll
    for (int c = 0; c < D; ++c) { xa[c] = a.use_resid ? xa[c] + ya[c] : ya[c]; xb[c] = a.use_resid ? xb[c] + yb[c] : yb[c]; }
    layer_norm<D>(xa, W + L::LN1G, W + L::LN1B, a.ln_eps);
    layer_norm<D>(xb, W + L::LN1G, W + L::LN1B, a.ln_eps);

    // ---------------- feed-forward: Linear(D, F) -> Dropout -> ReLU -> Linear(F, D), four hidden features per group
    float2 fa[D], fb[D];
#pragma unroll
    for (int c = 0; c < D; ++c) { xsa[c] = splat(xa[c]); xsb[c] = splat(xb[c]); fa[c] = fb[c] = make_float2(0.f, 0.f); }
    const int groups = a.F4 >> 2;
#pragma unroll 1
    for (int g = 0; g < groups; ++g) {
      const float4* __restrict__ G = reinterpret_cast<const float4*>(W + L::FF + g * L::GS);
      const float4 b1 = G[0];
      float2 h01a = lo(b1), h23a = hi(b1), h01b = lo(b1), h23b = hi(b1);
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const float4 w = G[1 + c];
        h01a = __ffma2_rn(xsa[c], lo(w), h01a); h23a = __ffma2_rn(xsa[c], hi(w), h23a);
        h01b = __ffma2_rn(xsb[c], lo(w), h01b); h23b = __ffma2_rn(xsb[c], hi(w), h23b);
      }
      if (TRAIN) {
        // four 16-bit words per row (drop_ff_word, drop_ff_mix); a dropped element is zeroed (the 1 / (1 - p) scale sits in the
        // staged W2, see above)
        const uint32_t ta = drop_ff_word(key_a, g), tb = drop_ff_word(key_b, g);
        const uint2 t2 = drop_ff_mix(ta, tb);
        const uint32_t ta2 = t2.x, tb2 = t2.y;
        const uint32_t th = a.drop_thresh << 16;
        if (drop_ff_dropped(ta, 0, th)) h01a.x = 0.f;
        if (drop_ff_dropped(ta, 1, th)) h01a.y = 0.f;
        if (drop_ff_dropped(ta2, 0, th)) h23a.x = 0.f;
        if (drop_ff_dropped(ta2, 1, th)) h23a.y = 0.f;
        if (drop_ff_dropped(tb, 0, th)) h01b.x = 0.f;
        if (drop_ff_dropped(tb, 1, th)) h01b.y = 0.f;
        if (drop_ff_dropped(tb2, 0, th)) h23b.x = 0.f;
        if (drop_ff_dropped(tb2, 1, th)) h23b.y = 0.f;
      }
      h01a.x = max_nan(h01a.x, 0.f); h01a.y = max_nan(h01a.y, 0.f); h23a.x = max_nan(h23a.x, 0.f); h23a.y = max_nan(h23a.y, 0.f);
      h01b.x = max_nan(h01b.x, 0.f); h01b.y = max_nan(h01b.y, 0.f); h23b.x = max_nan(h23b.x, 0.f); h23b.y = max_nan(h23b.y, 0.f);
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const float4 w = G[1 + D + c];
        fa[c] = __ffma2_rn(h01a, lo(w), fa[c]); fa[c] = __ffma2_rn(h23a, hi(w), fa[c]);
        fb[c] = __ffma2_rn(h01b, lo(w), fb[c]); fb[c] = __ffma2_rn(h23b, hi(w), fb[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < D; ++c) {
      float za = W[L::B2 + c] + (fa[c].x + fa[c].y), zb = W[L::B2 + c] + (fb[c].x + fb[c].y);
      if (TRAIN) { za *= drop_mask(key_a, 8 + c, a); zb *= drop_mask(key_b, 8 + c, a); }
      xa[c] = a.use_resid ? xa[c] + za : za;
      xb[c] = a.use_resid ? xb[c] + zb : zb;
    }
    layer_norm<D>(xa, W + L::LN2G, W + L::LN2B, a.ln_eps);
    layer_norm<D>(xb, W + L::LN2G, W + L::LN2B, a.ln_eps);
  }
  if (va) store_row<D>(a.emb + row0 + ra * D, xa);
  if (vb) store_row<D>(a.emb + row0 + rb * D, xb);
}

// ------------------------------------------------------------------------------------------------------------------
// critic / actor heads + sampling
//
// CTA = 32 environments x 128 hidden columns = one warp pair per split-K group (4 groups) (columns [0, 64) critic, [64, 128) actor; a head narrower than 64
// is zero-padded).  Layer 1 is a register-tiled [32 x K] x [K x 128] product: K in chunks of 16, the weight chunk
// [16][128] and the embedding chunk [32][16] double-buffered in shared memory with cp.async, every thread an
// 8-environment x 8-column tile (columns 4c..4c+3 of BOTH heads, so that the 16 lanes of a half-warp read one contiguous
// 256-byte weight row segment; the two half-warps take different environments) = 64 accumulators, 256 FFMA per 16
// LDS.128.  The K dimension is additionally split over HD_KS warp pairs (each takes one k-quad of every chunk; partial
// tiles are summed through shared memory) so that 8192 environments put ~14 warps on every SM instead of ~3.5.
// Layer 2 (two NH x NH products) reuses the tile shape and the split with the weights staged once per CTA.
constexpr int HD_TM = 32;        // environments per CTA
constexpr int HD_KS = 4;         // split-K groups: warp pair g accumulates the k with (k / 4) % 4 == g, then the groups are summed
constexpr int HD_THREADS = 64 * HD_KS;
constexpr int HD_COLS = 128;     // [critic hidden (64) | actor hidden (64)]
constexpr int HD_HS = 64;        // column stride between the two heads
constexpr int HD_KC = 16;        // K chunk
static_assert(HD_KC == 4 * HD_KS, "one k-quad of every chunk per split-K group");
constexpr int HD_XS = HD_KC + 4; // padded row of the embedding chunk
constexpr int HD_STAGES = 4;     // cp.async ring: chunks are requested three iterations ahead (L2 latency >> one chunk of math)
constexpr int HD_H1S = HD_COLS + 4;
constexpr int HD_H2S = HD_COLS + 1;
constexpr size_t HD_SMEM_FLOATS = HD_STAGES * HD_KC * HD_COLS + HD_STAGES * HD_TM * HD_XS + HD_HS * HD_COLS + HD_TM * HD_H1S + HD_TM * HD_H2S + HD_TM * 4;

__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// acc[i][c] += x[i] . w[c] over four consecutive k: x = 8 float4 (one per environment), w rows from shared memory
__device__ __forceinline__ void heads_tile_fma(float (&acc)[8][8], const float4 (&x)[8], const float* __restrict__ wrow, int cq) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 wa = *reinterpret_cast<const float4*>(wrow + q * HD_COLS + 4 * cq);
    const float4 wb = *reinterpret_cast<const float4*>(wrow + q * HD_COLS + HD_HS + 4 * cq);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float xv = q == 0 ? x[i].x : q == 1 ? x[i].y : q == 2 ? x[i].z : x[i].w;
      acc[i][0] = fmaf(xv, wa.x, acc[i][0]); acc[i][1] = fmaf(xv, wa.y, acc[i][1]);
      acc[i][2] = fmaf(xv, wa.z, acc[i][2]); acc[i][3] = fmaf(xv, wa.w, acc[i][3]);
      acc[i][4] = fmaf(xv, wb.x, acc[i][4]); acc[i][5] = fmaf(xv, wb.y, acc[i][5]);
      acc[i][6] = fmaf(xv, wb.z, acc[i][6]); acc[i][7] = fmaf(xv, wb.w, acc[i][7]);
    }
  }
}

// NORM: the linear policy's NormalizeObservation (NArgs) on every X element as it is loaded.  One CTA owns its 32 rows and every
// column, and each k-chunk is loaded once, so each (env, k) statistic is read and written by exactly one thread of the grid.  The
// X chunks then travel through registers (load, update, normalise, st.shared) instead of cp.async; the weight chunks keep the ring.
// FROZEN (with NORM): the statistics are only read (evaluation, EvacPolicyIO.norm_frozen); obs_norm is the one store.
template <bool NORM, bool FROZEN = false>
__global__ void __launch_bounds__(HD_THREADS, 2) evac_policy_heads_kernel(const __grid_constant__ HArgs a, const __grid_constant__ NArgs n) {
  static_assert(NORM || !FROZEN, "FROZEN is a mode of the fused normaliser");
  extern __shared__ float4 smem4[];
  float* wc = reinterpret_cast<float*>(smem4);        // [HD_STAGES][HD_KC][HD_COLS]
  float* xc = wc + HD_STAGES * HD_KC * HD_COLS;       // [HD_STAGES][HD_TM][HD_XS]
  float* w2s = xc + HD_STAGES * HD_TM * HD_XS;        // [HD_HS][HD_COLS]
  float* h1 = w2s + HD_HS * HD_COLS;                  // [HD_TM][HD_H1S]   (float4 reads along k)
  float* h2 = h1 + HD_TM * HD_H1S;                    // [HD_TM][HD_H2S]   (scalar reads, env varies across lanes)
  float* o3 = h2 + HD_TM * HD_H2S;                    // [HD_TM][4]: value, mean...
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kg = warp >> 1;                            // split-K group of this warp pair
  const int t64 = tid & 63;                            // position inside the 64-thread tile grid
  const int e0 = blockIdx.x * HD_TM;
  const int ne = min(HD_TM, a.E - e0);
  const int cq = lane & 15;                            // column quad: columns 4cq..4cq+3 and 64+4cq..64+4cq+3
  const int eb = (warp & 1) * 16 + (lane >> 4) * 8;    // first of this thread's 8 environments
  float* red = wc;                                     // [64][65] split-K exchange, aliases the chunk buffers once they are drained
  // sum the partial tiles of the split-K groups into group 0 (sequential rounds through one 16.6 KB buffer)
  auto reduce_groups = [&](float (&t)[8][8]) {
    __syncthreads();
    for (int g = 1; g < HD_KS; ++g) {
      if (kg == g) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < 8; ++c) red[(i * 8 + c) * 65 + t64] = t[i][c];
      }
      __syncthreads();
      if (kg == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < 8; ++c) t[i][c] += red[(i * 8 + c) * 65 + t64];
      }
      __syncthreads();
    }
  };
  const bool x_vec = (a.K & 3) == 0;                   // rows of the embedding are 16-byte aligned

  auto load_chunk = [&](int c, int buf) {
    const int k0 = c * HD_KC;
    float* wd = wc + buf * HD_KC * HD_COLS;
    const float* ws = a.w1t + (size_t)k0 * HD_COLS;    // 16 x 128 floats, contiguous (rows >= K are zero)
#pragma unroll
    for (int i = 0; i < HD_KC * HD_COLS / 4 / HD_THREADS; ++i) {
      const int v = i * HD_THREADS + tid;
      cp_async16(wd + 4 * v, ws + 4 * v, 16);
    }
    float* xd = xc + buf * HD_TM * HD_XS;
    if constexpr (FROZEN) {
      for (int v = tid; v < HD_TM * HD_KC; v += HD_THREADS) {
        const int r = v / HD_KC, kk = v - r * HD_KC, k = k0 + kk;
        float z = 0.f;
        if (r < ne && k < a.K) {
          const size_t i = (size_t)(e0 + r) * a.K + k;
          z = norm_frozen(a.emb[i], n.mean[i], n.var[i], n.eps, n.clip);
          if (n.obs_norm != nullptr) n.obs_norm[i] = z;
        }
        xd[r * HD_XS + kk] = z;
      }
    } else if constexpr (NORM) {
      const NormWeights nw = norm_weights(n);
      for (int v = tid; v < HD_TM * HD_KC; v += HD_THREADS) {
        const int r = v / HD_KC, kk = v - r * HD_KC, k = k0 + kk;
        float z = 0.f;
        if (r < ne && k < a.K) {
          const size_t i = (size_t)(e0 + r) * a.K + k;
          float mean = n.mean[i], var = n.var[i];
          z = norm_update(a.emb[i], mean, var, nw, n);
          n.mean[i] = mean; n.var[i] = var;
          if (n.obs_norm != nullptr) n.obs_norm[i] = z;
        }
        xd[r * HD_XS + kk] = z;
      }
    } else if (x_vec) {
      for (int v = tid; v < HD_TM * HD_KC / 4; v += HD_THREADS) {
        const int r = v >> 2, kq = (v & 3) * 4;
        const int k = k0 + kq;
        const int bytes = (r < ne && k < a.K) ? 16 : 0;   // K % 4 == 0: a float4 is entirely inside or outside the row
        cp_async16(xd + r * HD_XS + kq, a.emb + (size_t)(e0 + min(r, ne - 1)) * a.K + min(k, a.K - 4), bytes);
      }
    } else {
      for (int v = tid; v < HD_TM * HD_KC; v += HD_THREADS) {
        const int r = v / HD_KC, kk = v - r * HD_KC, k = k0 + kk;
        xd[r * HD_XS + kk] = (r < ne && k < a.K) ? a.emb[(size_t)(e0 + r) * a.K + k] : 0.f;
      }
    }
    cp_async_commit();
  };

  float acc[8][8];
  // ---- layer 1
  {
    float4 ba = make_float4(0.f, 0.f, 0.f, 0.f), bb = ba;
    if (kg == 0) { ba = *reinterpret_cast<const float4*>(a.b1 + 4 * cq); bb = *reinterpret_cast<const float4*>(a.b1 + HD_HS + 4 * cq); }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      acc[i][0] = ba.x; acc[i][1] = ba.y; acc[i][2] = ba.z; acc[i][3] = ba.w;
      acc[i][4] = bb.x; acc[i][5] = bb.y; acc[i][6] = bb.z; acc[i][7] = bb.w;
    }
    const int chunks = a.K16 / HD_KC;
    // the layer-2 weights ride along in the first group
    for (int v = tid; v < HD_HS * HD_COLS / 4; v += HD_THREADS) cp_async16(w2s + 4 * v, a.w2t + 4 * v, 16);
#pragma unroll
    for (int c = 0; c < HD_STAGES - 1; ++c) {
      if (c < chunks) load_chunk(c, c); else cp_async_commit();   // group index == chunk index, always
    }
    for (int c = 0; c < chunks; ++c) {
      cp_async_wait<HD_STAGES - 2>();   // all but the newest HD_STAGES - 2 groups have landed -> chunk c is here
      __syncthreads();                  // ... for every thread, and every warp is done with chunk c - 1, whose buffer is refilled now
      if (c + HD_STAGES - 1 < chunks) load_chunk(c + HD_STAGES - 1, (c + HD_STAGES - 1) % HD_STAGES); else cp_async_commit();
      const float* wb_ = wc + (c % HD_STAGES) * HD_KC * HD_COLS;
      const float* xb_ = xc + (c % HD_STAGES) * HD_TM * HD_XS + eb * HD_XS;
      {
        const int kk = 4 * kg;  // HD_KC == 4 * HD_KS: one k-quad of every chunk per group
        float4 x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = *reinterpret_cast<const float4*>(xb_ + i * HD_XS + kk);
        heads_tile_fma(acc, x, wb_ + kk * HD_COLS, cq);
      }
    }
    reduce_groups(acc);
    if (kg == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        *reinterpret_cast<float4*>(h1 + (eb + i) * HD_H1S + 4 * cq) = make_float4(tanhf(acc[i][0]), tanhf(acc[i][1]), tanhf(acc[i][2]), tanhf(acc[i][3]));
        *reinterpret_cast<float4*>(h1 + (eb + i) * HD_H1S + HD_HS + 4 * cq) = make_float4(tanhf(acc[i][4]), tanhf(acc[i][5]), tanhf(acc[i][6]), tanhf(acc[i][7]));
      }
    }
  }
  __syncthreads();
  // ---- layer 2: columns 4cq.. of the critic read h1[.., 0:64), columns 64+4cq.. of the actor read h1[.., 64:128)
  {
    float4 ba = make_float4(0.f, 0.f, 0.f, 0.f), bb = ba;
    if (kg == 0) { ba = *reinterpret_cast<const float4*>(a.b2 + 4 * cq); bb = *reinterpret_cast<const float4*>(a.b2 + HD_HS + 4 * cq); }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      acc[i][0] = ba.x; acc[i][1] = ba.y; acc[i][2] = ba.z; acc[i][3] = ba.w;
      acc[i][4] = bb.x; acc[i][5] = bb.y; acc[i][6] = bb.z; acc[i][7] = bb.w;
    }
#pragma unroll 2
    for (int k = kg * (HD_HS / HD_KS); k < (kg + 1) * (HD_HS / HD_KS); k += 4) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 wa = *reinterpret_cast<const float4*>(w2s + (k + q) * HD_COLS + 4 * cq);
        const float4 wb = *reinterpret_cast<const float4*>(w2s + (k + q) * HD_COLS + HD_HS + 4 * cq);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float xc_ = h1[(eb + i) * HD_H1S + k + q], xa_ = h1[(eb + i) * HD_H1S + HD_HS + k + q];
          acc[i][0] = fmaf(xc_, wa.x, acc[i][0]); acc[i][1] = fmaf(xc_, wa.y, acc[i][1]);
          acc[i][2] = fmaf(xc_, wa.z, acc[i][2]); acc[i][3] = fmaf(xc_, wa.w, acc[i][3]);
          acc[i][4] = fmaf(xa_, wb.x, acc[i][4]); acc[i][5] = fmaf(xa_, wb.y, acc[i][5]);
          acc[i][6] = fmaf(xa_, wb.z, acc[i][6]); acc[i][7] = fmaf(xa_, wb.w, acc[i][7]);
        }
      }
    }
    reduce_groups(acc);
    if (kg == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          h2[(eb + i) * HD_H2S + 4 * cq + c] = tanhf(acc[i][c]);
          h2[(eb + i) * HD_H2S + HD_HS + 4 * cq + c] = tanhf(acc[i][4 + c]);
        }
      }
    }
  }
  __syncthreads();
  // ---- layer 3: value (row 0 of w3, critic hidden) and the action mean (rows 1..A, actor hidden)
  const int R = 1 + a.A;
  for (int t = tid; t < HD_TM * R; t += HD_THREADS) {
    const int r = t % R, el = t / R;
    const float* __restrict__ hp = h2 + el * HD_H2S + (r == 0 ? 0 : HD_HS);
    const float* __restrict__ w = a.w3 + r * HD_HS;
    float s = a.b3[r];
    for (int k = 0; k < a.NH; ++k) s = fmaf(hp[k], w[k], s);
    o3[el * 4 + r] = s;   // A <= 3 (checked on the host)
  }
  __syncthreads();
  // ---- Normal(mean, exp(logstd)): sample / log-probability / entropy
  if (tid < ne) heads_finish(a, e0 + tid, o3 + tid * 4, true, true);
}

// ------------------------------------------------------------------------------------------------------------------
// NormalizeReward(gamma) + clip [rpo_agent.py:31-32; gymnasium NormalizeReward.step]: per-env discounted return,
// RunningMeanStd of it (one sample per step), reward / sqrt(var + eps), clip.
struct RArgs {
  int E;
  const float* reward;
  const uint8_t* terminated;
  const uint8_t* truncated;   // optional, with done_out
  float* done_out;            // optional [E]: float(terminated | truncated) = next_done of rpo_agent.py:194
  float* returns;
  float* ret_mean;
  float* ret_var;
  const double* count;
  float* out;
  float gamma, eps, clip;
};

__global__ void evac_normalize_reward_kernel(const RArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E) return;
  const double cnt = *a.count, tot = cnt + 1.0;
  const float w_new = (float)(1.0 / tot), w_old = (float)(cnt / tot), w_mix = __fmul_rn(w_old, w_new);
  const float r = a.reward[e];
  const float keep = a.terminated[e] ? 0.f : 1.f;
  const float ret = __fadd_rn(__fmul_rn(a.returns[e], __fmul_rn(a.gamma, keep)), r);
  a.returns[e] = ret;
  float mean = a.ret_mean[e], var = a.ret_var[e];
  const float delta = __fsub_rn(ret, mean);
  mean = __fadd_rn(mean, __fmul_rn(delta, w_new));
  var = __fadd_rn(__fmul_rn(var, w_old), __fmul_rn(__fmul_rn(delta, delta), w_mix));
  a.ret_mean[e] = mean; a.ret_var[e] = var;
  const float z = __fmul_rn(r, rsqrtf(__fadd_rn(var, a.eps)));
  a.out[e] = min_nan(max_nan(z, -a.clip), a.clip);
  if (a.done_out != nullptr) a.done_out[e] = (a.terminated[e] | (a.truncated ? a.truncated[e] : (uint8_t)0)) ? 1.f : 0.f;
}

}  // namespace evacp
