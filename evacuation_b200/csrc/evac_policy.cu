// C ABI of the fused RPO policy forward (the transformer embedding + heads, or, with num_blocks = 0, the linear network on the
// observation) and the reward normaliser (include/evac_b200.h, "rollout-loop glue").  Host side: weight repacking + launch plumbing; the arithmetic lives in evac_policy.cuh.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/evac_b200.h"
#include "evac_policy.cuh"
#include "evac_policy_tc.cuh"

using namespace evacp;

int evac_set_error_(int code, const char* msg);  // evac_abi.cu

static int pfail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return evac_set_error_(code, buf);
}

#define PCK(call)                                                                                  \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return pfail(EVAC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// widest observation the linear policy (num_blocks = 0) takes: every flattened observation at N <= 64 (Dict rel + ohe: 388) fits
// with room; the heads' K loops have no structural limit, the cap bounds the weight upload and the per-CTA K loop
constexpr int PL_MAX_K = 4096;

struct EvacPolicy {
  EvacPolicyConfig cfg;
  int device = 0;
  int S = 0, D = 0, H = 0, F = 0, F4 = 0, NB = 0, NH = 0, A = 0, K = 0, K16 = 0;
  int wstride = 0;
  float* d_emb_w = nullptr;   // NB packed blocks
  float *d_w1t = nullptr, *d_b1 = nullptr, *d_w2t = nullptr, *d_b2 = nullptr, *d_w3 = nullptr, *d_b3 = nullptr, *d_logstd = nullptr;
  float* d_scratch = nullptr;  // embedding scratch [scratch_envs, K]
  int scratch_envs = 0;
  // layer 1 of the heads on the tensor cores (evac_policy_tc.cuh): split + swizzled weight tiles for both column tilings, H1 scratch
  float *d_w1tc64 = nullptr, *d_w1tc128 = nullptr, *d_w2tc = nullptr;
  int tc_chunks = 0;
  bool use_tc = false;
  bool tc_cols128 = false;  // EVAC_POLICY_TC=128: 128-column tiles at every batch size (measurement hook)
  bool loaded = false;
  int64_t launches = 0;
  size_t embed_smem = 0, heads_smem = 0;
};

template <int D, int H>
static int stride_of(int F4) { return EmbLayout<D, H>::stride(F4); }

// (D, H) dispatch table
#define EVAC_POLICY_SHAPES(X) X(6, 1) X(6, 2) X(6, 3) X(6, 4) X(3, 1) X(3, 2) X(3, 3) X(3, 4) X(2, 1) X(2, 2) X(2, 3) X(2, 4)

static int block_stride(int D, int H, int F4) {
#define X(d, h) if (D == d && H == h) return stride_of<d, h>(F4);
  EVAC_POLICY_SHAPES(X)
#undef X
  return -1;
}

template <int D, int H>
static void pack_block(const float* src, float* dst, int F, int F4) {
  using L = EmbLayout<D, H>;
  const float* Wq = src; const float* bq = Wq + H * D * D;
  const float* Wk = bq + H * D; const float* bk = Wk + H * D * D;
  const float* Wv = bk + H * D; const float* bv = Wv + H * D * D;
  const float* Wd = bv + H * D; const float* bd = Wd + D * H * D;
  const float* W1 = bd + D; const float* b1 = W1 + F * D;
  const float* W2 = b1 + F; const float* b2 = W2 + D * F;
  const float* g1 = b2 + D; const float* be1 = g1 + D; const float* g2 = be1 + D; const float* be2 = g2 + D;
  const float* Wqkv[3] = {Wq, Wk, Wv};
  const float* bqkv[3] = {bq, bk, bv};
  for (int d = 0; d < D; ++d)
    for (int m = 0; m < 3; ++m)
      for (int h = 0; h < H; ++h) {
        const int o = h * D + d;  // split_heads: view(.., H, D)
        for (int c = 0; c < D; ++c) dst[L::QKV_W + (d * D + c) * L::QP + m * H + h] = Wqkv[m][o * D + c];
        dst[L::QKV_B + d * L::QP + m * H + h] = bqkv[m][o];
      }
  for (int d = 0; d < D; ++d)
    for (int h = 0; h < H; ++h)
      for (int c = 0; c < D; ++c) dst[L::WD + (d * H + h) * L::DP + c] = Wd[c * (D * H) + d * H + h];  // flatten(-2,-1) of [.., D, H]
  for (int c = 0; c < D; ++c) {
    dst[L::BD + c] = bd[c]; dst[L::LN1G + c] = g1[c]; dst[L::LN1B + c] = be1[c];
    dst[L::B2 + c] = b2[c]; dst[L::LN2G + c] = g2[c]; dst[L::LN2B + c] = be2[c];
  }
  for (int f = 0; f < F; ++f) {
    float* G = dst + L::FF + (f >> 2) * L::GS;
    const int t = f & 3;
    G[t] = b1[f];
    for (int c = 0; c < D; ++c) { G[4 + 4 * c + t] = W1[f * D + c]; G[4 + 4 * D + 4 * c + t] = W2[c * F + f]; }
  }
  (void)F4;
}

// frozen: evaluation with the normaliser's statistics read-only (never together with train)
template <int D, int H>
static int launch_embed(EvacPolicy* p, const PArgs& a, bool train, bool frozen, cudaStream_t st) {
  auto k_eval = evac_policy_embed_kernel<D, H, false>;
  auto k_train = evac_policy_embed_kernel<D, H, true>;
  auto k_frozen = evac_policy_embed_kernel<D, H, false, true>;
  static thread_local size_t attr_set[16] = {0};
  if (p->embed_smem > 48 * 1024 && attr_set[p->device & 15] < p->embed_smem) {
    PCK(cudaFuncSetAttribute(k_eval, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->embed_smem));
    PCK(cudaFuncSetAttribute(k_train, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->embed_smem));
    PCK(cudaFuncSetAttribute(k_frozen, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->embed_smem));
    attr_set[p->device & 15] = p->embed_smem;
  }
  const int grid = (a.E + PW_WARPS - 1) / PW_WARPS;
  if (train) k_train<<<grid, PW_WARPS * 32, p->embed_smem, st>>>(a);
  else if (frozen) k_frozen<<<grid, PW_WARPS * 32, p->embed_smem, st>>>(a);
  else k_eval<<<grid, PW_WARPS * 32, p->embed_smem, st>>>(a);
  PCK(cudaGetLastError());
  p->launches++;
  return EVAC_OK;
}

// the heads kernel on X = the embedding, or the observation of the linear policy (+ its fused normaliser when n.mean is set: updated,
// or read-only when frozen)
static int launch_heads(EvacPolicy* p, const EvacPolicyIO* io, const float* x, const NArgs& n, bool frozen, cudaStream_t st) {
  const bool norm = n.mean != nullptr;
  HArgs h;
  memset(&h, 0, sizeof(h));
  h.E = io->num_envs; h.K = p->K; h.K16 = p->K16; h.NH = p->NH; h.A = p->A;
  h.emb = x; h.w1t = p->d_w1t; h.b1 = p->d_b1; h.w2t = p->d_w2t; h.b2 = p->d_b2; h.w3 = p->d_w3; h.b3 = p->d_b3; h.logstd = p->d_logstd;
  h.given_action = io->given_action;
  h.mean = io->mean; h.value = io->value; h.action = io->action; h.action_clipped = io->action_clipped; h.logprob = io->logprob; h.entropy = io->entropy;
  h.sample = io->sample;
  h.seed_lo = (uint32_t)io->seed; h.seed_hi = (uint32_t)(io->seed >> 32);
  h.offset = io->offset; h.offset_dev = reinterpret_cast<const unsigned long long*>(io->offset_device); h.env_offset = io->env_index_offset;
  if (p->use_tc) {
    // the heads on the tensor cores; 64-column tiles (critic and actor in separate CTAs) while 128-column tiles would not fill the SMs
    TCArgs t;
    t.h = h; t.chunks = p->tc_chunks; t.w2tc = p->d_w2tc;
    const int gx = (h.E + TC_M - 1) / TC_M;
    // shapes: 64 columns x 4 stages (critic and actor in separate CTAs) while 128-column tiles would not fill the SMs, 128 columns
    // x 3 stages beyond (X is read once).  Measured per 8192 / 20 000 / 65 536 envs: 20.3 / 49.3 / 121.5 us (64x4), 29.7 / 50.4 /
    // 105.0 us (128x3); 64 columns x 2 stages with two CTAs per SM: 24.6 / 53.6 / 113.1 us.
    // The fused normaliser's update always takes the 128-column tiles: one CTA per row tile updates the statistics (DESIGN.md
    // section 7).  Frozen, it writes nothing two CTAs share and takes the normaliser-free rule (DESIGN.md section 7.3).
    auto k64 = evac_policy_heads_tc_kernel<64, 4, 2, 1>;
    auto k128 = evac_policy_heads_tc_kernel<128, 3, 2, 1>;
    auto k128n = evac_policy_heads_tc_kernel<128, 3, 2, 1, true>;
    auto k64f = evac_policy_heads_tc_kernel<64, 4, 2, 1, true, true>;
    auto k128f = evac_policy_heads_tc_kernel<128, 3, 2, 1, true, true>;
    using S64 = TCShape<64, 4, 2>; using S128 = TCShape<128, 3, 2>;
    static thread_local bool tc_attr[16] = {false};
    if (!tc_attr[p->device & 15]) {
      PCK(cudaFuncSetAttribute(k64, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S64::SMEM_BYTES));
      PCK(cudaFuncSetAttribute(k128, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S128::SMEM_BYTES));
      PCK(cudaFuncSetAttribute(k128n, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S128::SMEM_BYTES));
      PCK(cudaFuncSetAttribute(k64f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S64::SMEM_BYTES));
      PCK(cudaFuncSetAttribute(k128f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S128::SMEM_BYTES));
      tc_attr[p->device & 15] = true;
    }
    if (norm && !frozen) { t.w1tc = p->d_w1tc128; k128n<<<dim3(gx, 1), TC_THREADS, S128::SMEM_BYTES, st>>>(t, n); }
    else if (gx < 2 * 148 && !p->tc_cols128) {
      t.w1tc = p->d_w1tc64;
      if (norm) k64f<<<dim3(gx, 2), TC_THREADS, S64::SMEM_BYTES, st>>>(t, n);
      else k64<<<dim3(gx, 2), TC_THREADS, S64::SMEM_BYTES, st>>>(t, n);
    } else {
      t.w1tc = p->d_w1tc128;
      if (norm) k128f<<<dim3(gx, 1), TC_THREADS, S128::SMEM_BYTES, st>>>(t, n);
      else k128<<<dim3(gx, 1), TC_THREADS, S128::SMEM_BYTES, st>>>(t, n);
    }
    PCK(cudaGetLastError());
    p->launches++;
    return EVAC_OK;
  }
  static thread_local size_t hattr[16] = {0};
  if (p->heads_smem > 48 * 1024 && hattr[p->device & 15] < p->heads_smem) {
    PCK(cudaFuncSetAttribute(evac_policy_heads_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->heads_smem));
    PCK(cudaFuncSetAttribute(evac_policy_heads_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->heads_smem));
    PCK(cudaFuncSetAttribute(evac_policy_heads_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->heads_smem));
    hattr[p->device & 15] = p->heads_smem;
  }
  if (norm && frozen) evac_policy_heads_kernel<true, true><<<(h.E + HD_TM - 1) / HD_TM, HD_THREADS, p->heads_smem, st>>>(h, n);
  else if (norm) evac_policy_heads_kernel<true><<<(h.E + HD_TM - 1) / HD_TM, HD_THREADS, p->heads_smem, st>>>(h, n);
  else evac_policy_heads_kernel<false><<<(h.E + HD_TM - 1) / HD_TM, HD_THREADS, p->heads_smem, st>>>(h, n);
  PCK(cudaGetLastError());
  p->launches++;
  return EVAC_OK;
}

int evac_policy_heads_view_(const EvacPolicy* p, HArgs* h, int* num_blocks, int* device) {
  if (!p) return pfail(EVAC_ERR_INVALID, "policy is NULL");
  if (!p->loaded) return pfail(EVAC_ERR_INVALID, "evac_policy_load_weights has not been called");
  memset(h, 0, sizeof(*h));
  h->K = p->K; h->K16 = p->K16; h->NH = p->NH; h->A = p->A;
  h->w1t = p->d_w1t; h->b1 = p->d_b1; h->w2t = p->d_w2t; h->b2 = p->d_b2; h->w3 = p->d_w3; h->b3 = p->d_b3; h->logstd = p->d_logstd;
  *num_blocks = p->NB;
  *device = p->device;
  return EVAC_OK;
}

extern "C" {

int evac_policy_default_config(EvacPolicyConfig* cfg, int32_t number_of_pedestrians, int32_t d_model) {
  if (!cfg) return pfail(EVAC_ERR_INVALID, "cfg is NULL");
  memset(cfg, 0, sizeof(*cfg));
  cfg->abi_version = EVAC_ABI_VERSION;
  cfg->seq_len = number_of_pedestrians + 2;
  cfg->d_model = d_model;
  cfg->num_heads = 3;          // rpo_transformer_agent_network.py:22
  cfg->dim_feedforward = 96;   // :25
  cfg->num_blocks = 2;         // :20
  cfg->use_resid = 0;          // :31
  cfg->dropout = 0.1f;         // :28
  cfg->layer_norm_eps = 1e-5f;
  cfg->num_hidden = 64;        // rpo_linear_agent_network.py:12
  cfg->action_dim = 2;
  return EVAC_OK;
}

int evac_policy_default_linear_config(EvacPolicyConfig* cfg, int32_t obs_dim) {
  if (!cfg) return pfail(EVAC_ERR_INVALID, "cfg is NULL");
  memset(cfg, 0, sizeof(*cfg));
  cfg->abi_version = EVAC_ABI_VERSION;
  cfg->seq_len = 1;            // K = seq_len * d_model = obs_dim
  cfg->d_model = obs_dim;
  cfg->num_blocks = 0;         // RPOLinearNetwork directly on the observation
  cfg->num_hidden = 64;        // rpo_linear_agent_network.py:12
  cfg->action_dim = 2;
  return EVAC_OK;
}

int evac_policy_create(const EvacPolicyConfig* cfg, int32_t device, EvacPolicy** out) {
  if (!cfg || !out) return pfail(EVAC_ERR_INVALID, "cfg / out is NULL");
  if (cfg->abi_version != EVAC_ABI_VERSION) return pfail(EVAC_ERR_INVALID, "EvacPolicyConfig.abi_version %d != %d", cfg->abi_version, EVAC_ABI_VERSION);
  const bool linear = cfg->num_blocks == 0;
  if (!linear && (cfg->seq_len < 1 || cfg->seq_len > PW_MAX_S))
    return pfail(EVAC_ERR_UNSUPPORTED, "fused policy: seq_len (number_of_pedestrians + 2) must be 1..%d, got %d", PW_MAX_S, cfg->seq_len);
  if (cfg->num_blocks < 0 || cfg->num_blocks > 8 || (!linear && cfg->dim_feedforward < 1)) return pfail(EVAC_ERR_INVALID, "bad dim_feedforward / num_blocks");
  // the linear network's K: from 1 (rows that are not a multiple of 4 floats take the heads' scalar loads) to PL_MAX_K
  const int64_t K_lin = (int64_t)cfg->seq_len * cfg->d_model;
  if (linear && (cfg->seq_len < 1 || cfg->d_model < 1 || K_lin > PL_MAX_K))
    return pfail(EVAC_ERR_UNSUPPORTED, "fused linear policy: seq_len * d_model (the observation width) must be 1..%d, got %lld", PL_MAX_K, (long long)K_lin);
  if (cfg->num_hidden < 4 || cfg->num_hidden > 64 || cfg->num_hidden % 4) return pfail(EVAC_ERR_UNSUPPORTED, "fused policy: num_hidden must be a multiple of 4 in 4..64, got %d", cfg->num_hidden);
  if (cfg->action_dim < 1 || cfg->action_dim > 3) return pfail(EVAC_ERR_UNSUPPORTED, "fused policy: action_dim must be 1..3");
  if (!(cfg->dropout >= 0.f && cfg->dropout < 1.f)) return pfail(EVAC_ERR_INVALID, "dropout must be in [0, 1)");
  const int F4 = round_up(cfg->dim_feedforward, 4);
  const int ws = linear ? 0 : block_stride(cfg->d_model, cfg->num_heads, F4);
  if (ws < 0) return pfail(EVAC_ERR_UNSUPPORTED, "fused policy: (d_model, num_heads) = (%d, %d) is not instantiated", cfg->d_model, cfg->num_heads);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return pfail(EVAC_ERR_NO_DEVICE, "no CUDA device (evacuation_b200 has no CPU fallback)");
  if (device < 0 || device >= ndev) return pfail(EVAC_ERR_INVALID, "device %d out of range", device);
  PCK(cudaSetDevice(device));
  EvacPolicy* p = new (std::nothrow) EvacPolicy();
  if (!p) return pfail(EVAC_ERR_INVALID, "out of host memory");
  p->cfg = *cfg; p->device = device;
  p->S = cfg->seq_len; p->D = cfg->d_model; p->H = cfg->num_heads; p->F = cfg->dim_feedforward; p->F4 = F4; p->NB = cfg->num_blocks;
  p->NH = cfg->num_hidden; p->A = cfg->action_dim; p->K = p->S * p->D; p->K16 = round_up(p->K, HD_KC);
  p->wstride = ws;
  p->embed_smem = linear ? 0 : ((size_t)p->NB * ws + (size_t)PW_WARPS * 2 * p->H * PW_MAX_S) * sizeof(float);
  p->heads_smem = HD_SMEM_FLOATS * sizeof(float);
  if (p->embed_smem > 200 * 1024 || p->heads_smem > 200 * 1024) { delete p; return pfail(EVAC_ERR_UNSUPPORTED, "fused policy: shape needs too much shared memory"); }
  cudaError_t e = cudaSuccess;
  auto alloc = [&](float** q, size_t n) { if (e == cudaSuccess) { e = cudaMalloc(q, n * sizeof(float)); if (e == cudaSuccess) e = cudaMemset(*q, 0, n * sizeof(float)); } };
  if (!linear) alloc(&p->d_emb_w, (size_t)p->NB * ws);
  alloc(&p->d_w1t, (size_t)p->K16 * HD_COLS); alloc(&p->d_b1, HD_COLS);
  alloc(&p->d_w2t, (size_t)HD_HS * HD_COLS); alloc(&p->d_b2, HD_COLS);
  alloc(&p->d_w3, (size_t)(1 + p->A) * HD_HS); alloc(&p->d_b3, 4); alloc(&p->d_logstd, 4);
  // the tensor-core kernel reads float4 rows (K % 4 == 0); otherwise layer 1 of the heads runs on the CUDA cores.
  // EVAC_POLICY_TC=0 is a test hook: it selects the CUDA-core heads so that tests can compare the two kernels bit for bit.
  const char* tc_env = getenv("EVAC_POLICY_TC");
  p->use_tc = (p->K % 4 == 0) && !(tc_env && tc_env[0] == '0');
  // EVAC_POLICY_TC=128 is a measurement hook: the tensor-core heads take the 128-column tiles at every batch size, so that the
  // two tilings can be timed at the same size (tools/policy_eval.py)
  p->tc_cols128 = tc_env && strcmp(tc_env, "128") == 0;
  p->tc_chunks = (p->K + TC_KC - 1) / TC_KC;
  if (p->use_tc) {
    alloc(&p->d_w1tc64, (size_t)p->tc_chunks * 2 * TC_COLS * TC_KC);
    alloc(&p->d_w1tc128, (size_t)p->tc_chunks * 2 * TC_COLS * TC_KC);
    alloc(&p->d_w2tc, (size_t)2 * TC_W2_HEAD_BYTES / 4);
  }
  if (e != cudaSuccess) { evac_policy_destroy(p); return pfail(EVAC_ERR_CUDA, "cudaMalloc failed: %s", cudaGetErrorString(e)); }
  *out = p;
  return EVAC_OK;
}

int evac_policy_destroy(EvacPolicy* p) {
  if (!p) return EVAC_OK;
  cudaSetDevice(p->device);
  float* bufs[] = {p->d_emb_w, p->d_w1t, p->d_b1, p->d_w2t, p->d_b2, p->d_w3, p->d_b3, p->d_logstd, p->d_scratch, p->d_w1tc64, p->d_w1tc128, p->d_w2tc};
  for (float* b : bufs) if (b) cudaFree(b);
  delete p;
  return EVAC_OK;
}

int64_t evac_policy_num_weights(const EvacPolicy* p) {
  if (!p) return -1;
  const int64_t D = p->D, H = p->H, F = p->F, NH = p->NH, A = p->A, K = p->K;
  const int64_t block = 3 * (H * D * D + H * D) + (D * H * D + D) + (F * D + F) + (D * F + D) + 4 * D;
  const int64_t heads = 2 * (NH * K + NH + NH * NH + NH) + (NH + 1) + (A * NH + A) + A;
  return p->NB * block + heads;
}

int evac_policy_load_weights(EvacPolicy* p, const float* w, int64_t count) {
  if (!p || !w) return pfail(EVAC_ERR_INVALID, "policy / weights is NULL");
  if (count != evac_policy_num_weights(p)) return pfail(EVAC_ERR_INVALID, "expected %lld weights, got %lld", (long long)evac_policy_num_weights(p), (long long)count);
  PCK(cudaSetDevice(p->device));
  const int D = p->D, H = p->H, F = p->F, NH = p->NH, A = p->A, K = p->K;
  const int64_t block = 3 * (H * D * D + H * D) + (D * H * D + D) + (F * D + F) + (D * F + D) + 4 * D;
  std::vector<float> emb((size_t)p->NB * p->wstride, 0.f);
  for (int b = 0; b < p->NB; ++b) {
#define X(d, h) if (D == d && H == h) pack_block<d, h>(w + b * block, emb.data() + (size_t)b * p->wstride, F, p->F4);
    EVAC_POLICY_SHAPES(X)
#undef X
  }
  const float* c0w = w + p->NB * block; const float* c0b = c0w + (size_t)NH * K;
  const float* c2w = c0b + NH; const float* c2b = c2w + NH * NH;
  const float* c4w = c2b + NH; const float* c4b = c4w + NH;
  const float* a0w = c4b + 1; const float* a0b = a0w + (size_t)NH * K;
  const float* a2w = a0b + NH; const float* a2b = a2w + NH * NH;
  const float* a4w = a2b + NH; const float* a4b = a4w + A * NH;
  const float* lsd = a4b + A;
  // heads: critic columns [0, 64), actor columns [64, 128), everything zero padded
  std::vector<float> w1t((size_t)p->K16 * HD_COLS, 0.f), b1(HD_COLS, 0.f), w2t((size_t)HD_HS * HD_COLS, 0.f), b2(HD_COLS, 0.f),
      w3((size_t)(1 + A) * HD_HS, 0.f), b3(4, 0.f), ls(4, 0.f);
  for (int o = 0; o < NH; ++o) {
    for (int k = 0; k < K; ++k) { w1t[(size_t)k * HD_COLS + o] = c0w[(size_t)o * K + k]; w1t[(size_t)k * HD_COLS + HD_HS + o] = a0w[(size_t)o * K + k]; }
    b1[o] = c0b[o]; b1[HD_HS + o] = a0b[o];
    for (int k = 0; k < NH; ++k) { w2t[(size_t)k * HD_COLS + o] = c2w[o * NH + k]; w2t[(size_t)k * HD_COLS + HD_HS + o] = a2w[o * NH + k]; }
    b2[o] = c2b[o]; b2[HD_HS + o] = a2b[o];
  }
  for (int k = 0; k < NH; ++k) w3[k] = c4w[k];
  for (int r = 0; r < A; ++r) for (int k = 0; k < NH; ++k) w3[(size_t)(1 + r) * HD_HS + k] = a4w[r * NH + k];
  b3[0] = c4b[0];
  for (int r = 0; r < A; ++r) { b3[1 + r] = a4b[r]; ls[r] = lsd[r]; }
  PCK(cudaDeviceSynchronize());
  if (!emb.empty()) PCK(cudaMemcpy(p->d_emb_w, emb.data(), emb.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_w1t, w1t.data(), w1t.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_b1, b1.data(), b1.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_w2t, w2t.data(), w2t.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_b2, b2.data(), b2.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_w3, w3.data(), w3.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_b3, b3.data(), b3.size() * sizeof(float), cudaMemcpyHostToDevice));
  PCK(cudaMemcpy(p->d_logstd, ls.data(), ls.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (p->use_tc) {
    // per 32-k chunk and column tile: [hi tile | lo tile], NT rows (columns of W1) x 32 k, K-major SWIZZLE_128B (tc_swizzle)
    for (int NT : {64, 128}) {
      const int ny = TC_COLS / NT;
      std::vector<float> t((size_t)p->tc_chunks * 2 * TC_COLS * TC_KC, 0.f);
      for (int c = 0; c < p->tc_chunks; ++c)
        for (int y = 0; y < ny; ++y) {
          float* hi = t.data() + ((size_t)c * ny + y) * (2 * NT * TC_KC);
          float* lo = hi + NT * TC_KC;
          for (int n = 0; n < NT; ++n)
            for (int kk = 0; kk < TC_KC; ++kk) {
              const int k = c * TC_KC + kk;
              const float v = k < K ? w1t[(size_t)k * HD_COLS + y * NT + n] : 0.f;
              const float h = tc_hi(v);
              const size_t off = tc_swizzle(n, kk >> 2) / 4 + (kk & 3);
              hi[off] = h; lo[off] = v - h;
            }
        }
      PCK(cudaMemcpy(NT == 64 ? p->d_w1tc64 : p->d_w1tc128, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
  }
  if (p->use_tc) {
    // layer 2, per head: [k-chunk (2)][hi tile | lo tile], 64 rows (output columns of the head) x 32 k
    std::vector<float> t((size_t)2 * TC_W2_HEAD_BYTES / 4, 0.f);
    for (int hd = 0; hd < 2; ++hd)
      for (int c = 0; c < HD_HS / TC_KC; ++c) {
        float* hi = t.data() + (size_t)hd * (TC_W2_HEAD_BYTES / 4) + (size_t)c * (2 * HD_HS * TC_KC);
        float* lo = hi + HD_HS * TC_KC;
        for (int n = 0; n < HD_HS; ++n)
          for (int kk = 0; kk < TC_KC; ++kk) {
            const float v = w2t[(size_t)(c * TC_KC + kk) * HD_COLS + hd * HD_HS + n];
            const float hv = tc_hi(v);
            const size_t off = tc_swizzle(n, kk >> 2) / 4 + (kk & 3);
            hi[off] = hv; lo[off] = v - hv;
          }
      }
    PCK(cudaMemcpy(p->d_w2tc, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  p->loaded = true;
  return EVAC_OK;
}

int evac_policy_reserve(EvacPolicy* p, int32_t max_envs) {
  if (!p || max_envs < 1) return pfail(EVAC_ERR_INVALID, "bad arguments");
  if (max_envs <= p->scratch_envs || p->NB == 0) return EVAC_OK;   // the linear policy has no embedding scratch
  PCK(cudaSetDevice(p->device));
  if (p->d_scratch) { PCK(cudaDeviceSynchronize()); PCK(cudaFree(p->d_scratch)); p->d_scratch = nullptr; p->scratch_envs = 0; }
  PCK(cudaMalloc(&p->d_scratch, (size_t)max_envs * p->K * sizeof(float)));
  p->scratch_envs = max_envs;
  return EVAC_OK;
}

int evac_policy_forward(EvacPolicy* p, const EvacPolicyIO* io, void* stream) {
  if (!p || !io) return pfail(EVAC_ERR_INVALID, "policy / io is NULL");
  if (!p->loaded) return pfail(EVAC_ERR_INVALID, "evac_policy_load_weights has not been called");
  if (io->num_envs < 1 || !io->obs) return pfail(EVAC_ERR_INVALID, "num_envs < 1 or obs is NULL");
  if ((io->norm_mean != nullptr) != (io->norm_var != nullptr) || (io->norm_mean && !io->norm_count))
    return pfail(EVAC_ERR_INVALID, "norm_mean, norm_var and norm_count must be given together");
  if (io->norm_frozen && io->training && p->NB > 0)
    return pfail(EVAC_ERR_UNSUPPORTED, "norm_frozen (evaluation) runs the transformer without dropout: set training = 0");
  const bool frozen = io->norm_frozen != 0 && io->norm_mean != nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  PCK(cudaSetDevice(p->device));
  if (p->NB == 0) {
    // the linear policy: no embedding kernel; the heads read the observation, with the NormalizeObservation update fused into
    // their X load, and always run (so that the normaliser does even without head outputs)
    if (io->embedding) return pfail(EVAC_ERR_INVALID, "the linear policy (num_blocks = 0) has no embedding output");
    if ((p->K & 3) == 0 && ((reinterpret_cast<uintptr_t>(io->obs) | reinterpret_cast<uintptr_t>(io->norm_mean) | reinterpret_cast<uintptr_t>(io->norm_var) |
                             reinterpret_cast<uintptr_t>(io->obs_norm)) & 15u) != 0)
      return pfail(EVAC_ERR_INVALID, "obs, norm_mean, norm_var and obs_norm must be 16-byte aligned");
    NArgs n{io->norm_mean, io->norm_var, io->norm_count, io->obs_norm, io->norm_eps, io->norm_clip};
    return launch_heads(p, io, io->obs, n, frozen, st);
  }
  const bool heads = io->mean || io->value || io->action || io->action_clipped || io->logprob || io->entropy;
  float* emb = io->embedding;
  if (!emb && p->scratch_envs < io->num_envs) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    PCK(cudaStreamIsCapturing(st, &cs));
    if (cs != cudaStreamCaptureStatusNone) return pfail(EVAC_ERR_INVALID, "call evac_policy_reserve(%d) before capturing a forward without an embedding buffer", io->num_envs);
    const int rc = evac_policy_reserve(p, io->num_envs);
    if (rc) return rc;
  }
  if (!emb) emb = p->d_scratch;
  if ((p->K & 3) == 0 && (reinterpret_cast<uintptr_t>(emb) & 15u) != 0)  // the heads read the rows with 16-byte requests
    return pfail(EVAC_ERR_INVALID, "embedding buffer must be 16-byte aligned");
  const bool train = io->training != 0 && p->cfg.dropout > 0.f;
  PArgs a;
  memset(&a, 0, sizeof(a));
  a.E = io->num_envs; a.S = p->S; a.F4 = p->F4; a.NB = p->NB; a.use_resid = p->cfg.use_resid;
  a.ln_eps = p->cfg.layer_norm_eps;
  a.qscale = (float)(1.4426950408889634 / sqrt((double)p->D));
  a.drop_scale = 1.f / (1.f - p->cfg.dropout);
  a.drop_thresh = (uint32_t)lrint((double)p->cfg.dropout * 65536.0);
  a.seed_lo = (uint32_t)io->seed; a.seed_hi = (uint32_t)(io->seed >> 32);
  a.offset = io->offset; a.offset_dev = reinterpret_cast<const unsigned long long*>(io->offset_device);
  a.env_offset = io->env_index_offset;
  a.obs = io->obs; a.emb = emb;
  a.norm_mean = io->norm_mean; a.norm_var = io->norm_var; a.norm_count = io->norm_count; a.obs_norm = io->obs_norm;
  a.norm_eps = io->norm_eps; a.norm_clip = io->norm_clip;
  a.w = p->d_emb_w; a.wstride = p->wstride;
  int rc = EVAC_ERR_UNSUPPORTED;
#define X(d, h) if (p->D == d && p->H == h) rc = launch_embed<d, h>(p, a, train, frozen, st);
  EVAC_POLICY_SHAPES(X)
#undef X
  if (rc) return rc;
  if (!heads) return EVAC_OK;
  return launch_heads(p, io, emb, NArgs{}, false, st);
}

int64_t evac_policy_launch_count(const EvacPolicy* p) { return p ? p->launches : -1; }

int evac_normalize_reward(int32_t num_envs, const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns,
                          float* ret_mean, float* ret_var, const double* count, float* out, float* done_out, float gamma, float eps,
                          float clip, void* stream) {
  if (num_envs < 1 || !reward || !terminated || !returns || !ret_mean || !ret_var || !count || !out) return pfail(EVAC_ERR_INVALID, "evac_normalize_reward: NULL argument");
  RArgs a{num_envs, reward, terminated, truncated, done_out, returns, ret_mean, ret_var, count, out, gamma, eps, clip};
  evac_normalize_reward_kernel<<<(num_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(a);
  PCK(cudaGetLastError());
  return EVAC_OK;
}

}  // extern "C"
