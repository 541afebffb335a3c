// Per-environment arithmetic of the RPO policy heads and of gymnasium's NormalizeObservation, shared by the heads kernels
// (evac_policy.cuh) and the one-warp policy rollout (evac_warp.cuh, evac_rollout_policy).  No kernel is defined here, so that
// both translation units of the library can include it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "philox.cuh"

namespace evacp {

// NaN-propagating max / min (torch.relu / torch.clamp keep NaN; fmaxf / fminf would drop it)
__device__ __forceinline__ float max_nan(float a, float b) { float r; asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ float min_nan(float a, float b) { float r; asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r; }

struct HArgs {
  int E, K, K16, NH, A;          // K = S * D inputs, K16 = K rounded up to the chunk
  const float* emb;              // [E, K]
  const float* w1t;              // [K16, 128]  column o < 64: critic.0.weight[o], 64 <= o: actor_mean.0.weight[o - 64] (zero padded)
  const float* b1;               // [128]
  const float* w2t;              // [64, 128]   row k, column o: (critic|actor).2.weight[o % 64][k] of o's own head (zero padded)
  const float* b2;               // [128]
  const float* w3;               // [(1 + A), 64]: critic.4.weight, actor_mean.4.weight rows (zero padded)
  const float* b3;               // [1 + A]
  const float* logstd;           // [A]
  const float* given_action;     // optional [E, A]: evaluate this action instead of sampling (rpo_alpha perturbation excluded)
  float* mean;                   // [E, A] out (may be NULL)
  float* value;                  // [E] out
  float* action;                 // [E, A] out: sampled (or given) action
  float* action_clipped;         // [E, A] out: clip(action, -1, 1)  (ClipAction, rpo_agent.py:27) (may be NULL)
  float* logprob;                // [E] out (may be NULL)
  float* entropy;                // [E] out (may be NULL)
  int sample;                    // 0: action = mean
  uint32_t seed_lo, seed_hi;
  unsigned long long offset;
  const unsigned long long* offset_dev;
  long long env_offset;
};

// Normal draws of the heads (host-callable, like the dropout stream): the Philox4x32-10 words of (seed, stream offset, global env)
__host__ __device__ __forceinline__ evac::Philox4 normal_words(uint32_t seed_lo, uint32_t seed_hi, unsigned long long off, uint32_t env_g) {
  return evac::philox4x32_10(env_g, (uint32_t)off, (uint32_t)(off >> 32), 0x504F4C49u, seed_lo, seed_hi);
}
// component c (< 3) of the standard Normal draw: Box-Muller on two 24-bit uniforms in (0, 1); words (0, 1) -> components 0 (cos)
// and 1 (sin), words (2, 3) -> component 2 (cos)
__host__ __device__ __forceinline__ float normal_draw(const uint32_t (&words)[4], int c) {
  const int p = (c >> 1) * 2;
  const float u1 = ((float)(words[p] >> 8) + 0.5f) * 5.9604644775390625e-08f;
  const float u2 = ((float)(words[p + 1] >> 8) + 0.5f) * 5.9604644775390625e-08f;
  const float rad = sqrtf(-2.f * logf(u1));
  float sn, cs;
  sincosf(6.28318530717958647692f * u2, &sn, &cs);
  return rad * ((c & 1) ? sn : cs);
}

// value + Normal(mean, exp(logstd)): sample / log-probability / entropy of environment e [rpo_linear_agent_network.py:47-61];
// o = {value, mean[0], mean[1], mean[2]}.  `critic` / `actor` select which half is written (the tensor-core kernel splits the
// two heads over two CTAs for small batches).
__device__ __forceinline__ void heads_finish(const HArgs& a, int e, const float* o, bool critic, bool actor) {
  if (critic && a.value) a.value[e] = o[0];
  if (!actor) return;
  const uint32_t env_g = (uint32_t)(a.env_offset + e);
  float lp = 0.f, ent = 0.f;
  const unsigned long long off = a.offset + (a.offset_dev ? *a.offset_dev : 0ull);
  const evac::Philox4 r = normal_words(a.seed_lo, a.seed_hi, off, env_g);
  const uint32_t words[4] = {r.x, r.y, r.z, r.w};
  for (int c = 0; c < a.A; ++c) {
    const float mu = o[1 + c];
    const float ls = a.logstd[c], sd = expf(ls);
    float act = mu;
    if (a.given_action != nullptr) act = a.given_action[(size_t)e * a.A + c];
    else if (a.sample) act = fmaf(sd, normal_draw(words, c), mu);
    const float z = (act - mu) / sd;
    lp += -0.5f * z * z - ls - 0.918938533204672741780f;
    ent += 0.5f + 0.918938533204672741780f + ls;
    if (a.mean) a.mean[(size_t)e * a.A + c] = mu;
    if (a.action) a.action[(size_t)e * a.A + c] = act;
    if (a.action_clipped) a.action_clipped[(size_t)e * a.A + c] = min_nan(max_nan(act, -1.f), 1.f);
  }
  if (a.logprob) a.logprob[e] = lp;
  if (a.entropy) a.entropy[e] = ent;
}

// NormalizeObservation + clip of the linear policy (num_blocks = 0), fused into the heads' load of X; with blocks it runs in the
// embedding kernel's prologue instead.  Same fields and meaning as the PArgs norm_* fields.
struct NArgs {
  float* mean;                   // [E, K] running mean / variance (in place)
  float* var;
  const double* count;           // device scalar: samples seen so far (the caller advances it)
  float* obs_norm;               // optional [E, K] out
  float eps, clip;
};

// The per-call weights of one RunningMeanStd sample (gymnasium; op for op VectorNormalizer._update).
struct NormWeights {
  float w_new, w_old, w_mix;
};
__device__ __forceinline__ NormWeights norm_weights(const NArgs& n) {
  const double cnt = *n.count, tot = cnt + 1.0;
  NormWeights w;
  w.w_new = (float)(1.0 / tot); w.w_old = (float)(cnt / tot);
  w.w_mix = __fmul_rn(w.w_old, w.w_new);
  return w;
}
// one (env, k) element: update its statistics in place, return the normalised, clipped value
__device__ __forceinline__ float norm_update(float x, float& mean, float& var, const NormWeights& w, const NArgs& n) {
  const float delta = __fsub_rn(x, mean);
  mean = __fadd_rn(mean, __fmul_rn(delta, w.w_new));
  var = __fadd_rn(__fmul_rn(var, w.w_old), __fmul_rn(__fmul_rn(delta, delta), w.w_mix));
  const float z = __fmul_rn(__fsub_rn(x, mean), rsqrtf(__fadd_rn(var, n.eps)));
  return min_nan(max_nan(z, -n.clip), n.clip);
}
// one (env, k) element against frozen statistics (evaluation, EvacPolicyIO.norm_frozen): the normalised, clipped value, op for
// op norm_update's last two lines; nothing is written
__device__ __forceinline__ float norm_frozen(float x, float mean, float var, float eps, float clip) {
  const float z = __fmul_rn(__fsub_rn(x, mean), rsqrtf(__fadd_rn(var, eps)));
  return min_nan(max_nan(z, -clip), clip);
}

}  // namespace evacp

// Internal to the library (not exported through include/evac_b200.h): the heads' view of a policy for evac_rollout_policy
// (evac_abi.cu) -- K, NH, A and the weights where evac_policy_load_weights put them, in the CUDA-core heads layout -- plus its
// num_blocks and device.  Fails with EVAC_ERR_INVALID before the weights are loaded.
typedef struct EvacPolicy EvacPolicy;
__attribute__((visibility("hidden"))) int evac_policy_heads_view_(const EvacPolicy* p, evacp::HArgs* h, int* num_blocks, int* device);
