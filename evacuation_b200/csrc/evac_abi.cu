// C ABI of the B200-native evacuation environment (see include/evac_b200.h for the contract and the
// reference interfaces each entry point replaces).  Host side: handle + launch plumbing only; all
// arithmetic lives in evac_kernels.cuh.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "../../include/evac_b200.h"
#include "evac_kernels.cuh"
#include "evac_warp.cuh"

using namespace evac;

// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// other translation units of this library (evac_policy.cu) report through the same thread-local message
int evac_set_error_(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return fail(EVAC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct EvacHandle {
  EvacConfig cfg;
  int E, N, device, obs_dim, prec;
  uint64_t seed;
  long long env_offset;
  // device state
  void* pos = nullptr;
  void* dir = nullptr;
  uint8_t* status = nullptr;
  float2* agent_pos = nullptr;
  float2* agent_dir = nullptr;
  int* now = nullptr;
  int* episode = nullptr;
  long long* overall = nullptr;
  double* acc = nullptr;
  float* ep_stats = nullptr;
  uint8_t* ep_finished = nullptr;
  double* totals = nullptr;
  int* agent_state = nullptr;
  unsigned char* blocks = nullptr;  // EnvBlock layout (N <= 64 float32, one-warp kernel): replaces every array above
  // staging for the *_host entry points
  cudaStream_t stream = nullptr;
  float *h_actions = nullptr, *h_noise = nullptr, *h_obs = nullptr, *h_reward = nullptr;
  const void* pin_key[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // evac_step_host: caller pointers of the last call ...
  bool pin_val[7] = {false, false, false, false, false, false, false};                        // ... and whether each was page-locked
  uint8_t *h_term = nullptr, *h_trunc = nullptr;
  float *d_actions = nullptr, *d_noise = nullptr, *d_obs = nullptr, *d_reward = nullptr;
  uint8_t *d_term = nullptr, *d_trunc = nullptr, *d_status = nullptr, *h_status = nullptr;
  int64_t launches = 0;
  int threads = 0, ppt = 0;
  int num_sms = 0;
  int cells_x = 0, cells_y = 0, cell_reach = 1;  // > 0: cell-list neighbour search (fp32; N <= 64: the sparse pass's cell masks)
  int cell_pair_walk = 1;        // paired walk of the sorted slots (0: one slot per thread)
  int cluster = 1;               // > 1: one environment per thread-block cluster of this many 1024 x 4 CTAs (N > 4096, evac_cluster.cuh)
  // per-environment parameters (evac_set_env_params): the caller's records and their device conversion ([E] EnvParamRec<real>,
  // allocated by the first call and kept); per_env selects the PE kernel instances
  EvacEnvParams* env_params = nullptr;
  void* d_params = nullptr;
  bool per_env = false;
};

// smallest double b such that sqrt(v) >= t for every v >= b  <=>  (v < b) == (sqrt(v) < t)
static double sq_boundary(double t) {
  double v = t * t;
  while (v > 0 && sqrt(nextafter(v, 0.0)) >= t) v = nextafter(v, 0.0);
  while (sqrt(v) < t) v = nextafter(v, INFINITY);
  return v;
}
static float round_up_f32(double b) {
  float f = (float)b;
  if ((double)f < b) f = nextafterf(f, INFINITY);
  return f;
}
template <typename real> static real thr2_of(double t);
template <> float thr2_of<float>(double t) { return round_up_f32(sq_boundary(t)); }
template <> double thr2_of<double>(double t) { return sq_boundary(t); }

static int compute_obs_dim(const EvacConfig& c) {
  const int n = c.number_of_pedestrians;
  if (c.positions == EVAC_POS_GRAV) return 6;
  const int sc = c.statuses == EVAC_STAT_OHE ? 4 : (c.statuses == EVAC_STAT_CAT ? 1 : 0);
  if (c.obs_type == EVAC_OBS_BOX) return (n + 2) * (2 + sc);
  return 4 + 2 * n + sc * n;
}

// Cell grid of the one-warp kernel's sparse pass: edge >= (1 + 1e-4) x vision radius (two pedestrians closer than the radius
// sit in the same or in adjacent cells, float32 rounding of the cell index included), 1 .. WCELLS cells per axis.
static void warp_cell_grid(const EvacConfig& c, int* gx, int* gy) {
  const double edge = c.to_pedestrian * (1.0 + 1e-4);
  *gx = (int)fmax(1.0, fmin((double)WCELLS, floor(2.0 * c.width / edge)));
  *gy = (int)fmax(1.0, fmin((double)WCELLS, floor(2.0 * c.height / edge)));
}

// GravityEncoding: alpha + 2 when it is a small integer (ipow by squaring in the kernels), else 0 (pow)
static int alpha_plus2_int_of(double alpha) {
  const double ap2 = alpha + 2.0;
  return (ap2 == floor(ap2) && ap2 >= 1.0 && ap2 <= 64.0) ? (int)ap2 : 0;
}

// one EvacEnvParams record as the kernels read it: the same conversions make_args applies to the EvacConfig fields
template <typename real>
static EnvParamRec<real> env_param_rec(const EvacEnvParams& p) {
  EnvParamRec<real> r;
  memset(&r, 0, sizeof(r));
  r.one_minus_enslaving = (real)(1.0 - p.enslaving_degree);
  r.alpha = (real)p.alpha;
  r.init_reward = (real)p.init_reward_each_step;
  r.intrinsic_coef = (real)p.intrinsic_reward_coef;
  r.noise_coef = (float)(real)p.noise_coef;
  r.enslaving_f = (float)p.enslaving_degree;
  r.max_timesteps = p.max_timesteps;
  r.bits = alpha_plus2_int_of(p.alpha) | (p.is_new_exiting_reward != 0) << 8 | (p.is_new_followers_reward != 0) << 9 |
           (p.is_termination_agent_wall_collision != 0) << 10;
  return r;
}

template <typename real>
static KArgs<real> make_args(const EvacHandle* h) {
  const EvacConfig& c = h->cfg;
  KArgs<real> a;
  memset(&a, 0, sizeof(a));
  a.E = h->E; a.N = h->N; a.obs_dim = h->obs_dim;
  a.width = (real)c.width; a.height = (real)c.height; a.step_size = (real)c.step_size; a.noise_coef = (real)c.noise_coef;
  a.enslaving = (real)c.enslaving_degree; a.one_minus_enslaving = (real)(1.0 - c.enslaving_degree);
  a.width_f = (float)c.width; a.height_f = (float)c.height; a.step_size_f = (float)c.step_size;
  a.eps_f = (float)c.eps; a.enslaving_f = (float)c.enslaving_degree;
  a.thr2_ped = thr2_of<real>(c.to_pedestrian); a.thr2_leader = thr2_of<real>(c.to_leader);
  a.thr2_exit = thr2_of<real>(c.to_exit); a.thr2_escape = thr2_of<real>(c.to_escape);
  a.cells_x = h->cells_x; a.cells_y = h->cells_y; a.cell_reach = h->cell_reach; a.cell_pair_walk = h->cell_pair_walk;
  a.cell_force = h->blocks != nullptr && c.neighbor_search == EVAC_SEARCH_CELLS;  // one-warp kernel, "cells"
  a.cell_inv_x = a.cells_x > 0 ? (float)(a.cells_x / (2.0 * c.width)) : 0.f;
  a.cell_inv_y = a.cells_y > 0 ? (float)(a.cells_y / (2.0 * c.height)) : 0.f;
  a.exit_reward = c.is_new_exiting_reward; a.follow_reward = c.is_new_followers_reward;
  a.term_wall = c.is_termination_agent_wall_collision;
  a.init_reward = (real)c.init_reward_each_step; a.intrinsic_coef = (real)c.intrinsic_reward_coef;
  a.max_timesteps = c.max_timesteps;
  a.inv_200n = (real)(1.0 / (200.0 * h->N)); a.inv_n = (real)(1.0 / h->N);
  a.positions = c.positions; a.statuses = c.statuses; a.obs_type = c.obs_type;
  a.alpha = (real)c.alpha; a.eps = (real)c.eps;
  a.alpha_plus2_int = alpha_plus2_int_of(c.alpha);
  a.auto_reset = c.auto_reset;
  a.pos = reinterpret_cast<typename vec2<real>::type*>(h->pos);
  a.dir = reinterpret_cast<typename vec2<real>::type*>(h->dir);
  a.status = h->status; a.agent_pos = h->agent_pos; a.agent_dir = h->agent_dir;
  a.now = h->now; a.episode = h->episode; a.overall = h->overall; a.acc = h->acc;
  a.ep_stats = h->ep_stats; a.ep_finished = h->ep_finished; a.totals = h->totals;
  a.agent_state = h->agent_state;
  a.blocks = h->blocks;
  {  // baseline_wacuum_cleaner.py:17-28 (float64 expressions, compared against float32 positions -> rounded to float32)
    const double half_reach = c.to_leader / 2.0;
    a.wac_top = (float)(c.height - half_reach + c.step_size); a.wac_right = (float)(c.width - half_reach + c.step_size);
    a.wac_left = (float)(-c.width + half_reach - c.step_size); a.wac_bottom = (float)(-c.height + half_reach - c.step_size);
  }
  a.seed = h->seed; a.env_offset = h->env_offset;
  a.num_steps = 1; a.agent_kind = AGENT_TABLE;
  return a;
}

// the kernels' last argument: the handle's per-env records (read by the PE instances only)
template <typename real>
static const EnvParamRec<real>* params_of(const EvacHandle* h) {
  return h->per_env ? static_cast<const EnvParamRec<real>*>(h->d_params) : nullptr;
}

// ------------------------------------------------------------------------------------------
template <typename real, int THREADS, int PPT, bool PE>
static int launch_step_pe(EvacHandle* h, const KArgs<real>& a, cudaStream_t st) {
  size_t smem = Tile<real>::bytes(THREADS * PPT);                                           // source tile
  if (a.cells_x > 0) smem += CellSmem::bytes(THREADS * PPT, a.cells_x * a.cells_y);         // + cell list
  static thread_local size_t attr_set[16] = {0};
  auto kern = evac_step_kernel<real, THREADS, PPT, 1, PE>;
  if (smem > 48 * 1024 && attr_set[h->device & 15] < smem) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // the whole unified L1 / shared-memory array as shared memory
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    attr_set[h->device & 15] = smem;
  }
  kern<<<a.E, THREADS, smem, st>>>(a, params_of<real>(h));
  CK(cudaGetLastError());
  h->launches++;
  return EVAC_OK;
}
template <typename real, int THREADS, int PPT>
static int launch_step_t(EvacHandle* h, const KArgs<real>& a, cudaStream_t st) {
  return h->per_env ? launch_step_pe<real, THREADS, PPT, true>(h, a, st) : launch_step_pe<real, THREADS, PPT, false>(h, a, st);
}

// One environment per cluster of CL CTAs (crowds above one SM's shared memory): grid = E x CL, cluster dimension as a
// launch attribute.
template <int CL, bool PE>
static int launch_cluster_pe(EvacHandle* h, const KArgs<float>& a, cudaStream_t st) {
  constexpr int THREADS = 1024, PPT = 4;
  const int C = a.cells_x * a.cells_y;
  const size_t smem = Tile<float>::bytes(THREADS * PPT) + CellSmem::bytes(THREADS * PPT, C) + ClusterSmem::bytes(C);
  static thread_local size_t attr_set[16] = {0};
  auto kern = evac_step_kernel<float, THREADS, PPT, CL, PE>;
  if (attr_set[h->device & 15] < smem) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[h->device & 15] = smem;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)a.E * CL);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  CK(cudaLaunchKernelEx(&cfg, kern, a, params_of<float>(h)));
  h->launches++;
  return EVAC_OK;
}
template <int CL>
static int launch_cluster_t(EvacHandle* h, const KArgs<float>& a, cudaStream_t st) {
  return h->per_env ? launch_cluster_pe<CL, true>(h, a, st) : launch_cluster_pe<CL, false>(h, a, st);
}

static void pick_shape(int n, int* threads, int* ppt) {
  if (n <= 64) { *threads = 32; *ppt = 2; }
  else if (n <= 128) { *threads = 128; *ppt = 1; }
  else if (n <= 256) { *threads = 256; *ppt = 1; }
  else if (n <= 512) { *threads = 256; *ppt = 2; }
  else if (n <= 1024) { *threads = 512; *ppt = 2; }
  else if (n <= 2048) { *threads = 512; *ppt = 4; }
  else if (n <= 4096) { *threads = 1024; *ppt = 4; }  // one CTA per SM
  else { *threads = 1024; *ppt = 8; }  // up to 8192: the sorted tile (16 B per pedestrian) + cell list still fit one SM's shared memory
}

// N <= 64, float32: the dedicated one-warp kernel (evac_warp.cuh), observation encoding resolved at compile time.  One
// environment per CTA: measured on B200 at 4096 envs with 1 / 2 / 4 / 8 environments per CTA, 14.0 / 14.4 / 14.4 / 14.9 us.
template <bool PE>
static void launch_warp_pe(const KArgs<float>& a, const EnvParamRec<float>* params, cudaStream_t st) {
  if (a.positions == POS_REL && a.statuses == STAT_OHE && a.obs_type == OBS_BOX) evac_warp_kernel<WMODE_REL_OHE_BOX, PE><<<a.E, 32, 0, st>>>(a, params);
  else if (a.positions == POS_GRAV) evac_warp_kernel<WMODE_GRAV, PE><<<a.E, 32, 0, st>>>(a, params);
  else evac_warp_kernel<WMODE_GENERIC, PE><<<a.E, 32, 0, st>>>(a, params);
}
static int launch_warp(EvacHandle* h, const KArgs<float>& a, cudaStream_t st) {
  if (h->per_env) launch_warp_pe<true>(a, params_of<float>(h), st);
  else launch_warp_pe<false>(a, nullptr, st);
  CK(cudaGetLastError());
  h->launches++;
  return EVAC_OK;
}

template <typename real>
static int launch_step(EvacHandle* h, const KArgs<real>& a, cudaStream_t st) {
  if constexpr (std::is_same<real, float>::value) {
    if (h->threads == 32) return launch_warp(h, a, st);
    switch (h->cluster) {
      case 2: return launch_cluster_t<2>(h, a, st);
      case 4: return launch_cluster_t<4>(h, a, st);
      case 8: return launch_cluster_t<8>(h, a, st);
    }
  }
  switch (h->threads * 16 + h->ppt) {
    case 32 * 16 + 2:
      if constexpr (std::is_same<real, double>::value) return launch_step_t<real, 32, 2>(h, a, st);
      break;  // float32: evac_warp_kernel
    case 128 * 16 + 1: return launch_step_t<real, 128, 1>(h, a, st);
    case 256 * 16 + 1: return launch_step_t<real, 256, 1>(h, a, st);
    case 256 * 16 + 2: return launch_step_t<real, 256, 2>(h, a, st);
    case 512 * 16 + 2: return launch_step_t<real, 512, 2>(h, a, st);
    case 512 * 16 + 4: return launch_step_t<real, 512, 4>(h, a, st);
    case 1024 * 16 + 4: return launch_step_t<real, 1024, 4>(h, a, st);
    case 1024 * 16 + 8:
      if constexpr (std::is_same<real, float>::value) return launch_step_t<real, 1024, 8>(h, a, st);
      break;  // fp64 parity mode: 32 B per tile slot, N <= 4096
  }
  return fail(EVAC_ERR_INVALID, "no kernel shape for N=%d", h->N);
}

// f(make_args<real>(h)) with real = the handle's precision
template <typename F>
static int with_args(const EvacHandle* h, F&& f) { return h->prec == EVAC_PREC_F64 ? f(make_args<double>(h)) : f(make_args<float>(h)); }

static int launch_aux(EvacHandle* h, int flags, const uint8_t* mask, float* obs, cudaStream_t st) {
  return with_args(h, [&](const auto& a) -> int {
    using real = decltype(a.width);  // the handle's precision
    if (h->per_env) evac_aux_kernel<real, true><<<h->E, 128, 0, st>>>(a, flags, mask, obs, params_of<real>(h));
    else evac_aux_kernel<real, false><<<h->E, 128, 0, st>>>(a, flags, mask, obs, nullptr);
    CK(cudaGetLastError());
    h->launches++;
    return EVAC_OK;
  });
}

static int set_device(const EvacHandle* h) {
  CK(cudaSetDevice(h->device));
  return EVAC_OK;
}

// ------------------------------------------------------------------------------------------
extern "C" {

int32_t evac_abi_version(void) { return EVAC_ABI_VERSION; }
// content hash of csrc/ + include/ at build time (evacuation_b200/build.py); the marker is also greppable in the binary
#ifndef EVAC_BUILD_ID
#define EVAC_BUILD_ID "unversioned-build"
#endif
static const char g_build_id[] = "EVAC_BUILD_ID=" EVAC_BUILD_ID;
const char* evac_build_id(void) { return g_build_id + 14; }
const char* evac_last_error(void) { return g_err; }

int evac_default_config(EvacConfig* c) {
  if (!c) return fail(EVAC_ERR_INVALID, "cfg is NULL");
  memset(c, 0, sizeof(*c));
  c->abi_version = EVAC_ABI_VERSION;
  c->number_of_pedestrians = 10;  // config.py:11
  c->width = 1.0; c->height = 1.0; c->step_size = 0.01; c->noise_coef = 0.2; c->eps = 1e-8;
  c->enslaving_degree = 1.0;
  c->is_new_exiting_reward = 0; c->is_new_followers_reward = 1; c->intrinsic_reward_coef = 0.0;
  c->is_termination_agent_wall_collision = 0; c->init_reward_each_step = -1.0; c->max_timesteps = 2000;
  c->positions = EVAC_POS_ABS; c->statuses = EVAC_STAT_NO; c->obs_type = EVAC_OBS_DICT; c->alpha = 3.0;
  c->to_leader = 0.2; c->to_pedestrian = 0.1; c->to_exit = 0.4; c->to_escape = 0.01;  // constants.py:35-38
  c->auto_reset = 0; c->precision = EVAC_PREC_F32; c->neighbor_search = EVAC_SEARCH_AUTO;
  return EVAC_OK;
}

int evac_create(const EvacConfig* cfg, int32_t num_envs, int32_t device, uint64_t seed, int64_t env_index_offset,
                EvacHandle** out) {
  if (!cfg || !out) return fail(EVAC_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (cfg->abi_version != EVAC_ABI_VERSION) return fail(EVAC_ERR_INVALID, "EvacConfig.abi_version %d != %d", cfg->abi_version, EVAC_ABI_VERSION);
  if (num_envs < 1) return fail(EVAC_ERR_INVALID, "num_envs must be >= 1");
  if (cfg->number_of_pedestrians < 1 || cfg->number_of_pedestrians > 32768)
    return fail(EVAC_ERR_INVALID, "number_of_pedestrians=%d outside the supported range 1..32768", cfg->number_of_pedestrians);
  if (cfg->number_of_pedestrians > 8192 && cfg->neighbor_search == EVAC_SEARCH_BRUTE)
    return fail(EVAC_ERR_INVALID, "number_of_pedestrians=%d: the all-pairs search keeps one environment in one SM's shared memory (1..8192); "
                                  "larger crowds run the clustered cell list", cfg->number_of_pedestrians);
  if (cfg->number_of_pedestrians > 4096 && cfg->precision == EVAC_PREC_F64)
    return fail(EVAC_ERR_INVALID, "number_of_pedestrians=%d: the fp64 parity mode supports 1..4096 (32 B per shared-memory tile slot)", cfg->number_of_pedestrians);
  if (cfg->positions < 0 || cfg->positions > 2 || cfg->statuses < 0 || cfg->statuses > 2 || cfg->obs_type < 0 || cfg->obs_type > 1)
    return fail(EVAC_ERR_INVALID, "invalid observation mode");  // ValueError in the reference (wrappers.py:45,75)
  if (cfg->positions == EVAC_POS_GRAV && cfg->obs_type == EVAC_OBS_BOX)
    return fail(EVAC_ERR_UNSUPPORTED, "positions='grav' with type='Box' is NotImplementedError in the reference (wrappers/config.py:80-81)");
  if (cfg->precision != EVAC_PREC_F32 && cfg->precision != EVAC_PREC_F64) return fail(EVAC_ERR_INVALID, "invalid precision");
  if (cfg->neighbor_search < EVAC_SEARCH_AUTO || cfg->neighbor_search > EVAC_SEARCH_CELLS) return fail(EVAC_ERR_INVALID, "invalid neighbor_search");
  if (!(cfg->to_leader > 0 && cfg->to_pedestrian > 0 && cfg->to_exit > 0 && cfg->to_escape > 0))
    return fail(EVAC_ERR_INVALID, "switch distances must be positive");
  if (cfg->max_timesteps < 1 || cfg->max_timesteps > (1 << 21)) return fail(EVAC_ERR_INVALID, "max_timesteps must be in 1 .. 2^21 (the step index is a 21-bit field of the Philox counter)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(EVAC_ERR_NO_DEVICE, "no CUDA device available; this library has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return fail(EVAC_ERR_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(EVAC_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);

  EvacHandle* h = new (std::nothrow) EvacHandle();
  if (!h) return fail(EVAC_ERR_INVALID, "out of host memory");
  h->cfg = *cfg; h->E = num_envs; h->N = cfg->number_of_pedestrians; h->device = device;
  h->obs_dim = compute_obs_dim(*cfg); h->prec = cfg->precision; h->seed = seed; h->env_offset = env_index_offset;
  h->num_sms = prop.multiProcessorCount;
  pick_shape(h->N, &h->threads, &h->ppt);
  if (h->N > 64 && h->prec == EVAC_PREC_F32 && cfg->neighbor_search != EVAC_SEARCH_BRUTE) {
    // above the 8192 pedestrians one SM's shared memory holds: a cluster of 4 / 8 CTAs (1024 threads x 4 pedestrians) per
    // environment.  EVAC_CLUSTER = 1 | 2 | 4 | 8 overrides the choice where the crowd fits: a test hook, so that tests can
    // check cluster-size invariance and compare clusters with the oracle.  Measured on B200 (10 steps after 32): 128 x 8192
    // one 1024 x 8 CTA 226 us, cluster of 2 263 us; 256 x 4096 one CTA 161 us, cluster of 2 288 us -> clusters only where
    // one CTA cannot hold the crowd.
    int want = h->N <= 8192 ? 1 : (h->N <= 16384 ? 4 : 8);
    const char* cl = getenv("EVAC_CLUSTER");  // test hook (see above)
    if (cl) {
      const int v = atoi(cl);
      if ((v == 2 || v == 4 || v == 8) && v * 4096 >= h->N) want = v;
      if (v == 1 && h->N <= 8192) want = 1;
    }
    h->cluster = want;
    if (h->cluster > 1) { h->threads = 1024; h->ppt = 4; }
  }
  if (h->N > 64 && h->threads > 32 && h->prec == EVAC_PREC_F32 && cfg->neighbor_search != EVAC_SEARCH_BRUTE) {
    // cell edge >= (1 + 1e-4) x vision radius: two pedestrians closer than the radius always sit in the same or
    // in adjacent cells, float32 rounding of the cell index included; at most 64 x 64 cells
    // reach 2 (default when the grid fits): half-size cells, 5 x 5 block -> 1.44x fewer candidates in 5 row segments
    // (measured 10-17 % faster than the 3 x 3 block of full-size cells at 256 x 4096)
    int reach = 2;
    double edge = cfg->to_pedestrian * (1.0 + 1e-4) / reach;
    if (2.0 * cfg->width / edge > 64.0 || 2.0 * cfg->height / edge > 64.0) { reach = 1; edge = cfg->to_pedestrian * (1.0 + 1e-4); }
    int gx = (int)fmin(64.0, floor(2.0 * cfg->width / edge)), gy = (int)fmin(64.0, floor(2.0 * cfg->height / edge));
    {  // the sorted tile + cell list of one environment live in ONE SM's shared memory: coarsen the grid (larger cells stay
       // valid) until they fit -- only reached above 4096 pedestrians with a grid near the 64 x 64 cap
      const size_t budget = (size_t)prop.sharedMemPerBlockOptin - 4096 /* static */, slots = (size_t)h->threads * h->ppt;
      while (gx * gy > 16 && Tile<float>::bytes((int)slots) + CellSmem::bytes((int)slots, gx * gy) > budget) { gx = (gx * 7 + 7) / 8; gy = (gy * 7 + 7) / 8; }
      // clustered pass: the per-warp group counts [32 warps][cells] alias one CTA's tile slice -> at most 2048 cells
      while (h->cluster > 1 && gx * gy > 2048) { gx = (gx * 7 + 7) / 8; gy = (gy * 7 + 7) / 8; }
    }
    if (gx >= 1 && gy >= 1 && (cfg->neighbor_search == EVAC_SEARCH_CELLS || gx * gy >= 16 || h->cluster > 1)) { h->cells_x = gx; h->cells_y = gy; h->cell_reach = reach; }
    // paired walk (two adjacent sorted slots per thread share one window): pays when neighbouring slots usually share a cell.
    // Measured on B200, 20 steps after 0 / 64 / 300 warm-up steps: 256 x 4096 (2.7 per cell) 144 / 177 / 271 -> 129 / 167 / 265 us,
    // 1024 x 1000 109 -> 107 us, 2048 x 256 (0.17 per cell) 58 -> 63 us  => on from half a pedestrian per cell
    h->cell_pair_walk = 2 * h->N >= gx * gy;
    // EVAC_CELL_PAIR_WALK=0 | 1 is a test hook: tests compare the paired walk with the one-slot walk bit for bit
    { const char* pw = getenv("EVAC_CELL_PAIR_WALK"); if (pw) h->cell_pair_walk = atoi(pw) != 0; }
    // Walks measured on B200 and not kept (256 x 4096, 20 steps after 0 / 64 / 300 warm-up steps):
    //  * chunks of the paired walk drawn from a shared counter instead of equal static shares: 109.2 / 147.5 / 246.1 us static vs
    //    111.7 / 146.3 / 247.3 us dynamic -- the flocked regime is bound by the total number of candidate pairs, not by the
    //    balance between the warps of a CTA;
    //  * a grouped walk (four lanes share one window of 8 consecutive sorted slots, a quarter of the shared-memory wavefronts for
    //    ~25 % more candidates): 109.8 / 147.8 / 246.1 us paired vs 118.1 / 153.4 / 247.9 us grouped (128 x 8192: 226.9 vs 234.6;
    //    1024 x 1000: 85.1 vs 89.9) -- the walk is not bound by shared-memory bandwidth either: what it costs is the number of
    //    evaluated candidate pairs times the trip-count divergence inside a warp.
  } else if (h->threads == 32 && h->prec == EVAC_PREC_F32 && cfg->neighbor_search != EVAC_SEARCH_BRUTE) {
    // one-warp kernel: the cell masks of the sparse pass.  "cells" pins the kernel to it (whenever exact), "auto" chooses per
    // warp and step (KArgs::cell_force); evac_num_cells reports the grid only where it is pinned
    warp_cell_grid(*cfg, &h->cells_x, &h->cells_y);
  }
  const size_t en = (size_t)h->E * h->N, es = h->prec == EVAC_PREC_F64 ? 16 : 8;
#define ALLOC(ptr, bytes)                                                      \
  do {                                                                         \
    cudaError_t _e = cudaMalloc((void**)&(ptr), (bytes));                      \
    if (_e != cudaSuccess) { evac_destroy(h); return fail(EVAC_ERR_CUDA, "cudaMalloc(%zu) failed: %s", (size_t)(bytes), cudaGetErrorString(_e)); } \
    cudaMemset((ptr), 0, (bytes));                                             \
  } while (0)
  if (h->threads == 32 && h->prec == EVAC_PREC_F32) {
    // the one-warp kernel family keeps the whole state of an environment in one packed 1152-byte block (EnvBlock)
    ALLOC(h->blocks, (size_t)h->E * BLK_BYTES);
  } else {
    ALLOC(h->pos, en * es); ALLOC(h->dir, en * es); ALLOC(h->status, en);
    ALLOC(h->agent_pos, (size_t)h->E * sizeof(float2)); ALLOC(h->agent_dir, (size_t)h->E * sizeof(float2));
    ALLOC(h->now, (size_t)h->E * sizeof(int)); ALLOC(h->episode, (size_t)h->E * sizeof(int));
    ALLOC(h->overall, (size_t)h->E * sizeof(long long)); ALLOC(h->acc, (size_t)h->E * 3 * sizeof(double));
    ALLOC(h->agent_state, (size_t)h->E * sizeof(int));
  }
  ALLOC(h->ep_stats, (size_t)h->E * EVAC_NUM_EPISODE_STATS * sizeof(float)); ALLOC(h->ep_finished, (size_t)h->E);
  ALLOC(h->totals, (1 + EVAC_NUM_EPISODE_STATS) * sizeof(double));
#undef ALLOC
  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CK(cudaDeviceSynchronize());
  *out = h;
  return EVAC_OK;
}

int evac_destroy(EvacHandle* h) {
  if (!h) return EVAC_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  void* dptrs[] = {h->pos, h->dir, h->status, h->agent_pos, h->agent_dir, h->now, h->episode, h->overall, h->acc,
                   h->ep_stats, h->ep_finished, h->totals, h->agent_state, h->blocks, h->d_actions, h->d_noise, h->d_obs /* one block: obs | reward | flags */,
                   h->d_params};
  for (void* p : dptrs) if (p) cudaFree(p);
  void* hptrs[] = {h->h_actions, h->h_noise, h->h_obs /* one block */};
  for (void* p : hptrs) if (p) cudaFreeHost(p);
  if (h->stream) cudaStreamDestroy(h->stream);
  free(h->env_params);
  delete h;
  return EVAC_OK;
}

int32_t evac_obs_dim(const EvacHandle* h) { return h ? h->obs_dim : -1; }
int32_t evac_num_cells(const EvacHandle* h) {
  if (!h) return -1;
  return h->threads == 32 && h->cfg.neighbor_search == EVAC_SEARCH_AUTO ? 0 : h->cells_x * h->cells_y;
}
int32_t evac_num_envs(const EvacHandle* h) { return h ? h->E : -1; }
int32_t evac_state_elem_size(const EvacHandle* h) { return h ? (h->prec == EVAC_PREC_F64 ? 8 : 4) : -1; }
int64_t evac_launch_count(const EvacHandle* h) { return h ? h->launches : -1; }

int evac_reset(EvacHandle* h, const uint8_t* reset_mask, float* obs, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const int flags = AUX_RESET | (obs ? AUX_OBS : 0);
  return launch_aux(h, flags, reset_mask, obs, st);
}

int evac_observe(EvacHandle* h, float* obs, void* stream) {
  if (!h || !obs) return fail(EVAC_ERR_INVALID, "NULL argument");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  return launch_aux(h, AUX_OBS, nullptr, obs, st);
}

int evac_set_state(EvacHandle* h, const void* positions, const void* directions, const uint8_t* statuses,
                   const float* agent_position, const float* agent_direction, const int32_t* now, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t en = (size_t)h->E * h->N, es = h->prec == EVAC_PREC_F64 ? 16 : 8;
  if (h->blocks) {
    StateIO io = {(float2*)positions, (float2*)directions, (uint8_t*)statuses, (float2*)agent_position, (float2*)agent_direction, (int*)now, nullptr, nullptr};
    evac_block_io_kernel<true><<<h->E, 64, 0, st>>>(h->blocks, h->E, h->N, io);
    CK(cudaGetLastError());
    h->launches++;
    if (!statuses && (positions || agent_position)) return launch_aux(h, AUX_STATUS, nullptr, nullptr, st);
    return EVAC_OK;
  }
  if (positions) CK(cudaMemcpyAsync(h->pos, positions, en * es, cudaMemcpyDeviceToDevice, st));
  if (directions) CK(cudaMemcpyAsync(h->dir, directions, en * es, cudaMemcpyDeviceToDevice, st));
  if (agent_position) CK(cudaMemcpyAsync(h->agent_pos, agent_position, (size_t)h->E * 8, cudaMemcpyDeviceToDevice, st));
  if (agent_direction) CK(cudaMemcpyAsync(h->agent_dir, agent_direction, (size_t)h->E * 8, cudaMemcpyDeviceToDevice, st));
  if (now) CK(cudaMemcpyAsync(h->now, now, (size_t)h->E * 4, cudaMemcpyDeviceToDevice, st));
  if (agent_position) CK(cudaMemsetAsync(h->agent_state, 0, (size_t)h->E * sizeof(int), st));  // a moved agent restarts its script
  if (statuses) {
    CK(cudaMemcpyAsync(h->status, statuses, en, cudaMemcpyDeviceToDevice, st));
  } else if (positions || agent_position) {  // pedestrians.py:21-26: statuses follow from the positions
    return launch_aux(h, AUX_STATUS, nullptr, nullptr, st);
  }
  return EVAC_OK;
}

int evac_get_state(EvacHandle* h, void* positions, void* directions, uint8_t* statuses, float* agent_position,
                   float* agent_direction, int32_t* now, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t en = (size_t)h->E * h->N, es = h->prec == EVAC_PREC_F64 ? 16 : 8;
  if (h->blocks) {
    StateIO io = {(float2*)positions, (float2*)directions, statuses, (float2*)agent_position, (float2*)agent_direction, now, nullptr, nullptr};
    evac_block_io_kernel<false><<<h->E, 64, 0, st>>>(h->blocks, h->E, h->N, io);
    CK(cudaGetLastError());
    h->launches++;
    return EVAC_OK;
  }
  if (positions) CK(cudaMemcpyAsync(positions, h->pos, en * es, cudaMemcpyDeviceToDevice, st));
  if (directions) CK(cudaMemcpyAsync(directions, h->dir, en * es, cudaMemcpyDeviceToDevice, st));
  if (statuses) CK(cudaMemcpyAsync(statuses, h->status, en, cudaMemcpyDeviceToDevice, st));
  if (agent_position) CK(cudaMemcpyAsync(agent_position, h->agent_pos, (size_t)h->E * 8, cudaMemcpyDeviceToDevice, st));
  if (agent_direction) CK(cudaMemcpyAsync(agent_direction, h->agent_dir, (size_t)h->E * 8, cudaMemcpyDeviceToDevice, st));
  if (now) CK(cudaMemcpyAsync(now, h->now, (size_t)h->E * 4, cudaMemcpyDeviceToDevice, st));
  return EVAC_OK;
}

static int rollout_impl(EvacHandle* h, int32_t num_steps, int32_t agent_kind, const float* actions, const float* noise, float* obs,
                        int32_t obs_every_step, float* reward_sum, uint8_t* terminated, uint8_t* truncated, uint16_t* status_counts,
                        uint8_t* status_out, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (num_steps < 1) return fail(EVAC_ERR_INVALID, "num_steps must be >= 1");
  if (agent_kind < EVAC_AGENT_TABLE || agent_kind > EVAC_AGENT_WACUUM) return fail(EVAC_ERR_INVALID, "invalid agent_kind");
  if (agent_kind == EVAC_AGENT_TABLE && !actions) return fail(EVAC_ERR_INVALID, "actions is NULL");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  return with_args(h, [&](auto a) -> int {
    a.actions = (const float2*)actions; a.noise = noise; a.obs = obs; a.obs_every_step = obs_every_step;
    a.reward = reward_sum; a.terminated = terminated; a.truncated = truncated; a.num_steps = num_steps; a.agent_kind = agent_kind;
    a.status_counts = status_counts; a.status_out = status_out;
    return launch_step(h, a, st);
  });
}

int evac_rollout(EvacHandle* h, int32_t num_steps, int32_t agent_kind, const float* actions, const float* noise, float* obs,
                 int32_t obs_every_step, float* reward_sum, uint8_t* terminated, uint8_t* truncated, uint16_t* status_counts,
                 void* stream) {
  return rollout_impl(h, num_steps, agent_kind, actions, noise, obs, obs_every_step, reward_sum, terminated, truncated, status_counts, nullptr, stream);
}

int evac_step(EvacHandle* h, const float* actions, const float* noise, float* obs, float* reward, uint8_t* terminated,
              uint8_t* truncated, void* stream) {
  if (!actions) return fail(EVAC_ERR_INVALID, "actions is NULL");
  return evac_rollout(h, 1, EVAC_AGENT_TABLE, actions, noise, obs, 0, reward, terminated, truncated, nullptr, stream);
}

int evac_rollout_policy(EvacHandle* h, const EvacPolicy* p, int32_t num_steps, const EvacPolicyRolloutIO* io, void* stream) {
  if (!h || !p || !io) return fail(EVAC_ERR_INVALID, "evac_rollout_policy: handle / policy / io is NULL");
  if (num_steps < 1) return fail(EVAC_ERR_INVALID, "num_steps must be >= 1");
  if (h->blocks == nullptr)
    return fail(EVAC_ERR_UNSUPPORTED, "evac_rollout_policy runs in the one-warp step kernel: float32 and N <= 64 (N = %d, %s)", h->N,
                h->prec == EVAC_PREC_F64 ? "float64" : "float32");
  if (h->cfg.positions != EVAC_POS_GRAV) return fail(EVAC_ERR_UNSUPPORTED, "evac_rollout_policy needs positions = grav (obs_dim 6)");
  evacp::HArgs ha;
  int nb = 0, pdev = 0;
  if (int r = evac_policy_heads_view_(p, &ha, &nb, &pdev)) return r;
  if (nb != 0 || ha.K != 6 || ha.A != 2)
    return fail(EVAC_ERR_UNSUPPORTED, "evac_rollout_policy takes the linear policy (num_blocks = 0) with K = 6 and action_dim 2, got "
                "num_blocks %d, K %d, action_dim %d", nb, ha.K, ha.A);
  if (pdev != h->device) return fail(EVAC_ERR_INVALID, "policy on device %d, environments on device %d", pdev, h->device);
  if (!io->obs || !io->next_done) return fail(EVAC_ERR_INVALID, "obs and next_done are required");
  if ((io->norm_mean != nullptr) != (io->norm_var != nullptr) || (io->norm_mean && !io->norm_count))
    return fail(EVAC_ERR_INVALID, "norm_mean, norm_var and norm_count must be given together");
  const bool rn = io->returns != nullptr;
  if (rn != (io->ret_mean != nullptr) || rn != (io->ret_var != nullptr) || rn != (io->ret_count != nullptr))
    return fail(EVAC_ERR_INVALID, "returns, ret_mean, ret_var and ret_count must be given together");
  if (io->reward_norm && !rn) return fail(EVAC_ERR_INVALID, "reward_norm needs the reward normaliser (returns, ret_mean, ret_var, ret_count)");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  KArgs<float> a = make_args<float>(h);
  a.obs = io->obs; a.obs_every_step = 0; a.num_steps = num_steps;
  a.reward = io->reward_sum; a.terminated = io->terminated; a.truncated = io->truncated; a.status_counts = io->status_counts;
  WPolArgs w;
  memset(&w, 0, sizeof(w));
  w.h = ha;
  w.h.E = h->E;
  w.h.value = io->value; w.h.action = io->action; w.h.logprob = io->logprob;
  w.h.sample = io->sample;
  w.h.seed_lo = (uint32_t)io->seed; w.h.seed_hi = (uint32_t)(io->seed >> 32);
  w.h.offset = io->offset; w.h.offset_dev = reinterpret_cast<const unsigned long long*>(io->offset_device);
  w.h.env_offset = io->env_index_offset;
  w.n.mean = io->norm_mean; w.n.var = io->norm_var; w.n.count = io->norm_count; w.n.obs_norm = io->obs_norm;
  w.n.eps = io->norm_eps; w.n.clip = io->norm_clip;
  w.norm_update = io->norm_update != 0;
  w.next_done = io->next_done; w.dones = io->dones;
  w.returns = io->returns; w.ret_mean = io->ret_mean; w.ret_var = io->ret_var; w.ret_count = io->ret_count;
  w.reward_norm = io->reward_norm;
  w.gamma = io->gamma; w.ret_eps = io->eps; w.ret_clip = io->clip;
  if (h->per_env) evac_warp_policy_kernel<true><<<a.E, 32, 0, st>>>(a, params_of<float>(h), w);
  else evac_warp_policy_kernel<false><<<a.E, 32, 0, st>>>(a, nullptr, w);
  CK(cudaGetLastError());
  h->launches++;
  double* oc = io->norm_mean && io->norm_update ? io->norm_count : nullptr;
  unsigned long long* off = reinterpret_cast<unsigned long long*>(io->offset_device);
  if (oc || io->ret_count || off) {
    evac_policy_counters_kernel<<<1, 1, 0, st>>>(oc, io->ret_count, off, num_steps);
    CK(cudaGetLastError());
    h->launches++;
  }
  return EVAC_OK;
}

static bool is_pinned(const void* p) {
  if (!p) return false;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return attr.type == cudaMemoryTypeHost;
}

int evac_step_host(EvacHandle* h, const float* actions, const float* noise, float* obs, float* reward, uint8_t* terminated,
                   uint8_t* truncated, uint8_t* statuses) {
  if (!h || !actions) return fail(EVAC_ERR_INVALID, "NULL argument");
  if (int r = set_device(h)) return r;
  const size_t E = h->E, N = h->N, D = h->obs_dim;
  if (!h->h_actions) {
    CK(cudaMallocHost((void**)&h->h_actions, E * 8)); CK(cudaMalloc((void**)&h->d_actions, E * 8));
    // outputs live in ONE device block and ONE pinned block, [obs | reward | terminated | truncated | statuses], so a caller
    // whose (page-locked) result arrays are laid out the same way gets them with a single D2H copy
    const size_t out_bytes = E * D * 4 + E * 4 + 2 * E + E * N;
    unsigned char *hb = nullptr, *db = nullptr;
    CK(cudaMallocHost((void**)&hb, out_bytes)); CK(cudaMalloc((void**)&db, out_bytes));
    h->h_obs = (float*)hb; h->h_reward = (float*)(hb + E * D * 4); h->h_term = hb + E * D * 4 + E * 4; h->h_trunc = h->h_term + E; h->h_status = h->h_trunc + E;
    h->d_obs = (float*)db; h->d_reward = (float*)(db + E * D * 4); h->d_term = db + E * D * 4 + E * 4; h->d_trunc = h->d_term + E; h->d_status = h->d_trunc + E;
  }
  if (noise && !h->h_noise) { CK(cudaMallocHost((void**)&h->h_noise, E * N * 4)); CK(cudaMalloc((void**)&h->d_noise, E * N * 4)); }
  cudaStream_t st = h->stream;
  // Page-locked caller buffers are used directly (zero staging copies); pageable ones go through the
  // handle's pinned staging buffers.
  // (a caller that re-uses its buffers -- the Python host face does -- pays the attribute queries once)
  const void* ptrs[7] = {actions, noise, obs, reward, terminated, truncated, statuses};
  for (int i = 0; i < 7; ++i)
    if (ptrs[i] != h->pin_key[i]) { h->pin_key[i] = ptrs[i]; h->pin_val[i] = is_pinned(ptrs[i]); }
  const bool pa = h->pin_val[0], pn = h->pin_val[1], po = h->pin_val[2], pr = h->pin_val[3], pt = h->pin_val[4], pu = h->pin_val[5], ps = h->pin_val[6];
  // Small batches (the reference-shaped single environment above all; up to kZeroCopyMaxBytes of inputs + results = ~680 envs x
  // 60): when every caller buffer is page-locked the kernel reads the actions / noise from and writes its results into HOST memory
  // directly (unified addressing: a page-locked host pointer is a device pointer) -- one launch + one synchronise instead of copy,
  // launch, copy, synchronise; a few KB over PCIe cost less than the latency of two copy operations.  Measured per step with /
  // without: 21 / 27 us (1 env), 24 / 28 (32), 27 / 32 (128), 40 / 45 (512); beyond, the copy engine wins (2048 envs: 124 / 95 us,
  // 4096: 401 / 145 -- the strided observation stores over PCIe).
  {
    constexpr size_t kZeroCopyMaxBytes = (size_t)1 << 20;
    const size_t bytes = E * (D * 4 + 14 + N * 5);
    if (bytes <= kZeroCopyMaxBytes && pa && (!noise || pn) && (!obs || po) && (!reward || pr) && (!terminated || pt) && (!truncated || pu) &&
        (!statuses || ps)) {
      if (int r = rollout_impl(h, 1, EVAC_AGENT_TABLE, actions, noise, obs, 0, reward ? reward : h->d_reward, terminated ? terminated : h->d_term,
                               truncated ? truncated : h->d_trunc, nullptr, statuses, st)) return r;
      CK(cudaStreamSynchronize(st));
      return EVAC_OK;
    }
  }
  // large batches: the results go through the copy engine; page-locked ACTIONS (8 bytes per environment) are still read by the kernel
  // straight from host memory -- one copy operation less in front of the launch (measured 86.5 vs 91.1 us at 2048 envs, 142.8 vs
  // 143.0 at 4096)
  const float* act_dev = actions;
  if (!pa) {
    memcpy(h->h_actions, actions, E * 8);
    CK(cudaMemcpyAsync(h->d_actions, h->h_actions, E * 8, cudaMemcpyHostToDevice, st));
    act_dev = h->d_actions;
  }
  if (noise) {
    if (!pn) memcpy(h->h_noise, noise, E * N * 4);
    CK(cudaMemcpyAsync(h->d_noise, pn ? noise : h->h_noise, E * N * 4, cudaMemcpyHostToDevice, st));
  }
  if (int r = rollout_impl(h, 1, EVAC_AGENT_TABLE, act_dev, noise ? h->d_noise : nullptr, obs ? h->d_obs : nullptr, 0, h->d_reward, h->d_term,
                           h->d_trunc, nullptr, statuses ? h->d_status : nullptr, st)) return r;
  const size_t head_bytes = E * D * 4 + E * 4 + 2 * E;
  const bool packed = reward == obs + E * D && terminated == (uint8_t*)(reward + E) && truncated == terminated + E &&
                      (!statuses || statuses == truncated + E);
  const bool packed_pinned = po && pr && pt && pu && (!statuses || ps) && obs && packed;
  const bool all_pageable = !po && !pr && !pt && !pu && !ps && obs && reward && terminated && truncated;
  if (packed_pinned || all_pageable) {
    CK(cudaMemcpyAsync(packed_pinned ? (void*)obs : (void*)h->h_obs, h->d_obs, head_bytes + (statuses ? E * N : 0), cudaMemcpyDeviceToHost, st));
  } else {
    if (obs) CK(cudaMemcpyAsync(po ? obs : h->h_obs, h->d_obs, E * D * 4, cudaMemcpyDeviceToHost, st));
    if (reward) CK(cudaMemcpyAsync(pr ? reward : h->h_reward, h->d_reward, E * 4, cudaMemcpyDeviceToHost, st));
    if (terminated) CK(cudaMemcpyAsync(pt ? terminated : h->h_term, h->d_term, E, cudaMemcpyDeviceToHost, st));
    if (truncated) CK(cudaMemcpyAsync(pu ? truncated : h->h_trunc, h->d_trunc, E, cudaMemcpyDeviceToHost, st));
    if (statuses) CK(cudaMemcpyAsync(ps ? statuses : h->h_status, h->d_status, E * N, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  if (obs && !po) memcpy(obs, h->h_obs, E * D * 4);
  if (reward && !pr) memcpy(reward, h->h_reward, E * 4);
  if (terminated && !pt) memcpy(terminated, h->h_term, E);
  if (truncated && !pu) memcpy(truncated, h->h_trunc, E);
  if (statuses && !ps) memcpy(statuses, h->h_status, E * N);
  return EVAC_OK;
}

int evac_get_accumulators(EvacHandle* h, double* acc, int64_t* overall_timesteps, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  if (h->blocks) {
    StateIO io = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, acc, (long long*)overall_timesteps};
    evac_block_io_kernel<false><<<h->E, 64, 0, st>>>(h->blocks, h->E, h->N, io);
    CK(cudaGetLastError());
    h->launches++;
    return EVAC_OK;
  }
  if (acc) CK(cudaMemcpyAsync(acc, h->acc, (size_t)h->E * 3 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (overall_timesteps) CK(cudaMemcpyAsync(overall_timesteps, h->overall, (size_t)h->E * sizeof(long long), cudaMemcpyDeviceToDevice, st));
  return EVAC_OK;
}

// ---- checkpoint / resume: the COMPLETE device state of a handle as one flat byte image
struct StateRegion { void* ptr; size_t bytes; };
static int state_regions(EvacHandle* h, StateRegion* r) {
  const size_t E = h->E, en = (size_t)h->E * h->N, es = h->prec == EVAC_PREC_F64 ? 16 : 8;
  int n = 0;
  if (h->blocks) {
    r[n++] = {h->blocks, E * BLK_BYTES};
  } else {
    r[n++] = {h->pos, en * es}; r[n++] = {h->dir, en * es}; r[n++] = {h->status, en};
    r[n++] = {h->agent_pos, E * 8}; r[n++] = {h->agent_dir, E * 8}; r[n++] = {h->now, E * 4}; r[n++] = {h->episode, E * 4};
    r[n++] = {h->overall, E * 8}; r[n++] = {h->acc, E * 24}; r[n++] = {h->agent_state, E * 4};
  }
  r[n++] = {h->ep_stats, E * EVAC_NUM_EPISODE_STATS * 4}; r[n++] = {h->ep_finished, E};
  r[n++] = {h->totals, (1 + EVAC_NUM_EPISODE_STATS) * 8};
  return n;
}

int64_t evac_state_bytes(EvacHandle* h) {
  if (!h) return -1;
  StateRegion r[16];
  const int n = state_regions(h, r);
  size_t total = 0;
  for (int i = 0; i < n; ++i) total += (r[i].bytes + 15) & ~(size_t)15;
  return (int64_t)total;
}

static int state_copy(EvacHandle* h, unsigned char* image, bool save, cudaStream_t st) {
  StateRegion r[16];
  const int n = state_regions(h, r);
  size_t off = 0;
  for (int i = 0; i < n; ++i) {
    if (save) CK(cudaMemcpyAsync(image + off, r[i].ptr, r[i].bytes, cudaMemcpyDeviceToDevice, st));
    else CK(cudaMemcpyAsync(r[i].ptr, image + off, r[i].bytes, cudaMemcpyDeviceToDevice, st));
    off += (r[i].bytes + 15) & ~(size_t)15;
  }
  return EVAC_OK;
}

int evac_save_state(EvacHandle* h, void* image, void* stream) {
  if (!h || !image) return fail(EVAC_ERR_INVALID, "NULL argument");
  if (int r = set_device(h)) return r;
  return state_copy(h, (unsigned char*)image, true, (cudaStream_t)stream);
}

int evac_load_state(EvacHandle* h, const void* image, void* stream) {
  if (!h || !image) return fail(EVAC_ERR_INVALID, "NULL argument");
  if (int r = set_device(h)) return r;
  return state_copy(h, (unsigned char*)image, false, (cudaStream_t)stream);
}

int evac_set_env_params(EvacHandle* h, const EvacEnvParams* params, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (!params) { h->per_env = false; return EVAC_OK; }
  for (int e = 0; e < h->E; ++e)
    if (params[e].max_timesteps < 1 || params[e].max_timesteps > (1 << 21))
      return fail(EVAC_ERR_INVALID, "env %d: max_timesteps must be in 1 .. 2^21 (the step index is a 21-bit field of the Philox counter)", e);
  if (int r = set_device(h)) return r;
  const bool f64 = h->prec == EVAC_PREC_F64;
  const size_t rec = f64 ? sizeof(EnvParamRec<double>) : sizeof(EnvParamRec<float>), bytes = (size_t)h->E * rec;
  if (!h->env_params) {
    h->env_params = (EvacEnvParams*)malloc((size_t)h->E * sizeof(EvacEnvParams));
    if (!h->env_params) return fail(EVAC_ERR_INVALID, "out of host memory");
    CK(cudaMalloc(&h->d_params, bytes));
  }
  unsigned char* conv = (unsigned char*)malloc(bytes);
  if (!conv) return fail(EVAC_ERR_INVALID, "out of host memory");
  for (int e = 0; e < h->E; ++e) {
    if (f64) { const EnvParamRec<double> r = env_param_rec<double>(params[e]); memcpy(conv + e * rec, &r, rec); }
    else { const EnvParamRec<float> r = env_param_rec<float>(params[e]); memcpy(conv + e * rec, &r, rec); }
  }
  // pageable source: the copy is staged before cudaMemcpyAsync returns, so `conv` may be freed right after it
  const cudaError_t err = cudaMemcpyAsync(h->d_params, conv, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream);
  free(conv);
  if (err != cudaSuccess) return fail(EVAC_ERR_CUDA, "cudaMemcpyAsync(env params) failed: %s", cudaGetErrorString(err));
  memcpy(h->env_params, params, (size_t)h->E * sizeof(EvacEnvParams));
  h->per_env = true;
  return EVAC_OK;
}

int evac_get_env_params(const EvacHandle* h, EvacEnvParams* out) {
  if (!h || !out) return fail(EVAC_ERR_INVALID, "NULL argument");
  if (h->per_env) { memcpy(out, h->env_params, (size_t)h->E * sizeof(EvacEnvParams)); return EVAC_OK; }
  const EvacConfig& c = h->cfg;
  for (int e = 0; e < h->E; ++e) {
    EvacEnvParams& p = out[e];
    p.noise_coef = c.noise_coef; p.enslaving_degree = c.enslaving_degree; p.alpha = c.alpha;
    p.intrinsic_reward_coef = c.intrinsic_reward_coef; p.init_reward_each_step = c.init_reward_each_step;
    p.is_new_exiting_reward = c.is_new_exiting_reward; p.is_new_followers_reward = c.is_new_followers_reward;
    p.is_termination_agent_wall_collision = c.is_termination_agent_wall_collision; p.max_timesteps = c.max_timesteps;
  }
  return EVAC_OK;
}

int evac_episode_stats(EvacHandle* h, float* stats, uint8_t* finished, double* totals, void* stream) {
  if (!h) return fail(EVAC_ERR_INVALID, "NULL handle");
  if (int r = set_device(h)) return r;
  cudaStream_t st = (cudaStream_t)stream;
  if (stats) CK(cudaMemcpyAsync(stats, h->ep_stats, (size_t)h->E * EVAC_NUM_EPISODE_STATS * 4, cudaMemcpyDeviceToDevice, st));
  if (finished) {
    CK(cudaMemcpyAsync(finished, h->ep_finished, (size_t)h->E, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemsetAsync(h->ep_finished, 0, (size_t)h->E, st));
  }
  if (totals) CK(cudaMemcpyAsync(totals, h->totals, (1 + EVAC_NUM_EPISODE_STATS) * sizeof(double), cudaMemcpyDeviceToDevice, st));
  return EVAC_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// Measurement probes.
template <bool PACKED>
__global__ void __launch_bounds__(256) probe_fma_kernel(float* out, int iters, float seed_a, float seed_b) {
  // 8 independent chains per thread; PACKED uses fma.rn.f32x2 (2 FMAs per instruction)
  const float t = (float)threadIdx.x * 1e-3f;
  if (PACKED) {
    float2 c[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) c[k] = make_float2(t + k, t - k);
    const float2 a = make_float2(seed_a, seed_a), b = make_float2(seed_b, seed_b);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __ffma2_rn(c[k], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += c[k].x + c[k].y;
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  } else {
    float c[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) c[k] = t + k;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 16; ++k) c[k] = fmaf(c[k], seed_a, seed_b);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += c[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  }
}

// Standalone launch of the SAME pairwise_pass device function the fused step kernel uses (one environment per warp,
// THREADS x PPT = 32x2) and of narrower mappings: THREADS lanes per environment, WPC environments (each with its own tile) per
// CTA, UNR slot pairs per unrolled iteration.
template <int THREADS, int PPT, int UNR = 4, int WPC = 1, int MINB = 1>
__global__ void __launch_bounds__(THREADS * WPC, MINB) probe_pairwise_kernel(const float2* __restrict__ pos, const float2* __restrict__ unit,
                                                                             float2* __restrict__ out, int N, int reps, float thr2, int E) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int wic = threadIdx.x / THREADS;
  Tile<float> tile(smem_raw + (size_t)wic * Tile<float>::bytes(THREADS * PPT), THREADS * PPT);
  const int tid = threadIdx.x % THREADS, e = blockIdx.x * WPC + wic;
  if (e >= E) return;
  float xi[PPT], yi[PPT], sx[PPT], sy[PPT], accx[PPT], accy[PPT];
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    const int i = k * THREADS + tid;
    float2 p = make_float2(PARK, PARK), u = make_float2(0.f, 0.f);
    if (i < N) { p = pos[(size_t)e * N + i]; u = unit[(size_t)e * N + i]; }
    tile.put(i, p.x, p.y, u.x, u.y);
    xi[k] = p.x; yi[k] = p.y; accx[k] = accy[k] = 0.f;
  }
  if (THREADS == 32) __syncwarp(); else __syncthreads();
  for (int r = 0; r < reps; ++r) {
    pairwise_pass<PPT, UNR>(tile, N, xi, yi, thr2, sx, sy);
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      accx[k] += sx[k]; accy[k] += sy[k];
      xi[k] += 1e-9f * sx[k];  // data dependence between passes so they cannot be hoisted
    }
  }
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    const int i = k * THREADS + tid;
    if (i < N) out[(size_t)e * N + i] = make_float2(accx[k], accy[k]);
  }
}

// FMA-pipe micro-probes for the packed instruction mix of pairwise_pass (no shared memory, operands in registers):
//   MODE 2: FFMA2 with three distinct 64-bit register operands per instruction (register-file bandwidth check)
//   MODE 3: FADD2 with a scalar-broadcast operand, MODE 4: FMUL2, MODE 5: the pairwise mix (2 FADD2, FMUL2, FFMA2, 2 FSET, 2 FFMA2)
template <int MODE>
__global__ void __launch_bounds__(256) probe_mix_kernel(float* out, int iters, float seed_a, float seed_b) {
  const float t = (float)threadIdx.x * 1e-3f;
  float2 c[8], a[8], b[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { c[k] = make_float2(t + k, t - k); a[k] = make_float2(seed_a + 1e-7f * k + 1e-9f * t, seed_a - 1e-7f * k - 1e-9f * t); b[k] = make_float2(seed_b * (k + 1) + 1e-9f * t, seed_b * (k + 2) - 1e-9f * t); }
  if (MODE == 2) {
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __ffma2_rn(c[k], a[k], b[k]);
    }
  } else if (MODE == 3) {
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __fadd2_rn(c[k], make_float2(seed_b, seed_b));
    }
  } else if (MODE == 4) {
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __fmul2_rn(c[k], a[k]);
    }
  } else if (MODE == 6) {  // FFMA2 acc = a(64-bit) * s(32-bit broadcast) + acc
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __ffma2_rn(a[k], make_float2(b[k].x, b[k].x), c[k]);
    }
  } else if (MODE == 7) {  // FSETP + predicated FADD2 acc += a
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) if (b[k].x < c[k].y) c[k] = __fadd2_rn(c[k], a[k]);
    }
  } else if (MODE == 8) {  // FFMA2 acc = a * a + acc (two distinct 64-bit operands)
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __ffma2_rn(a[k], a[k], c[k]);
    }
  } else if (MODE == 9) {  // FFMA2 acc = a0 * b + acc (a0 shared by consecutive instructions: operand-reuse cache)
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __ffma2_rn(a[0], b[k], c[k]);
    }
  } else if (MODE == 10) {  // FFMA2 acc = a * b + acc, three distinct (accumulator form)
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) c[k] = __ffma2_rn(a[k], b[k], c[k]);
    }
  } else if (MODE == 11) {  // scalar FFMA acc = a * b + acc, three distinct 32-bit operands (16 chains)
    float* cs = reinterpret_cast<float*>(c); float* as = reinterpret_cast<float*>(a); float* bs = reinterpret_cast<float*>(b);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 16; ++k) cs[k] = fmaf(as[k], bs[k], cs[k]);
    }
  } else {
    // sources: a[k] = (x_j, x_j+1), b[k] = (y_j, y_j+1), c[k] = (ux_j, ux_j+1); uy = a[k] again (values are irrelevant)
    float2 nx[2] = {make_float2(-t, -t), make_float2(-t - 0.5f, -t - 0.5f)}, ny[2] = {make_float2(t, t), make_float2(t + 0.25f, t + 0.25f)};
    float2 ax[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)}, ay[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
    for (int i = 0; i < iters; ++i) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const float2 dx = __fadd2_rn(a[k], nx[q]);
          const float2 dy = __fadd2_rn(b[k], ny[q]);
          float2 d2 = __fmul2_rn(dx, dx);
          d2 = __ffma2_rn(dy, dy, d2);
          const float2 w = make_float2(d2.x < seed_a ? 1.f : 0.f, d2.y < seed_a ? 1.f : 0.f);
          ax[q] = __ffma2_rn(w, c[k], ax[q]);
          ay[q] = __ffma2_rn(w, a[k], ay[q]);
        }
      }
      nx[0].x += 1e-9f * ax[0].x; nx[1].y += 1e-9f * ay[1].y;  // data dependence between iterations
    }
    c[0] = __fadd2_rn(__fadd2_rn(ax[0], ax[1]), __fadd2_rn(ay[0], ay[1]));
  }
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) s += c[k].x + c[k].y;
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" {

int evac_probe_fma(int32_t device, int32_t packed, int32_t iters, float* ms, double* flops) {
  if (!ms || !flops) return fail(EVAC_ERR_INVALID, "NULL argument");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  float* out = nullptr;
  CK(cudaMalloc((void**)&out, (size_t)blocks * threads * 4));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  for (int rep = 0; rep < 2; ++rep) {
    CK(cudaEventRecord(e0));
    switch (packed) {  // 0 scalar FFMA, 1 FFMA2 (shared operands); 2-5: probe_mix_kernel modes
      case 0: probe_fma_kernel<false><<<blocks, threads>>>(out, iters, 1.0000001f, 1e-7f); break;
      case 1: probe_fma_kernel<true><<<blocks, threads>>>(out, iters, 1.0000001f, 1e-7f); break;
      case 2: probe_mix_kernel<2><<<blocks, threads>>>(out, iters, 1.0000001f, 1e-7f); break;
      case 3: probe_mix_kernel<3><<<blocks, threads>>>(out, iters, 1.0000001f, 1e-7f); break;
      case 4: probe_mix_kernel<4><<<blocks, threads>>>(out, iters, 1.0000001f, 1e-7f); break;
      case 6: probe_mix_kernel<6><<<blocks, threads>>>(out, iters, 1.0000001f, 1e-7f); break;
      case 7: probe_mix_kernel<7><<<blocks, threads>>>(out, iters, 1e-9f, 1e-7f); break;
      case 8: probe_mix_kernel<8><<<blocks, threads>>>(out, iters, 1e-9f, 1e-7f); break;
      case 9: probe_mix_kernel<9><<<blocks, threads>>>(out, iters, 1e-9f, 1e-7f); break;
      case 10: probe_mix_kernel<10><<<blocks, threads>>>(out, iters, 1e-9f, 1e-7f); break;
      case 11: probe_mix_kernel<11><<<blocks, threads>>>(out, iters, 1e-9f, 1e-7f); break;
      default: probe_mix_kernel<5><<<blocks, threads>>>(out, iters, 0.5f, 1e-7f); break;
    }
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
  }
  CK(cudaEventElapsedTime(ms, e0, e1));
  // FMA-pipe lane-operations x 2 (an FFMA counts 2 flops; FADD2 / FMUL2 lane-ops are counted the same way so that every mode
  // reads as FMA-pipe occupancy); mode 5 issues 96 packed FMA-pipe instructions (+ 32 FSET on the ALU pipe) per iteration
  *flops = (double)blocks * threads * (double)iters * (packed == 5 ? 96.0 * 2.0 : 16.0) * 2.0;
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  return EVAC_OK;
}

int evac_probe_pairwise(int32_t device, int32_t num_envs, int32_t n, int32_t reps, float* ms, double* pairs) {
  if (!ms || !pairs || n < 1 || n > 64 || num_envs < 1) return fail(EVAC_ERR_INVALID, "bad argument");
  CK(cudaSetDevice(device));
  const size_t en = (size_t)num_envs * n;
  float2 *pos = nullptr, *unit = nullptr, *out = nullptr;
  CK(cudaMalloc((void**)&pos, en * 8)); CK(cudaMalloc((void**)&unit, en * 8)); CK(cudaMalloc((void**)&out, en * 8));
  float2* hp = (float2*)malloc(en * 8);
  float2* hu = (float2*)malloc(en * 8);
  uint32_t s = 12345u;
  auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (float)(s >> 8) * (1.0f / 16777216.0f); };
  for (size_t i = 0; i < en; ++i) {
    hp[i] = make_float2(2.f * rnd() - 1.f, 2.f * rnd() - 1.f);
    const float th = 6.2831853f * rnd();
    hu[i] = make_float2(cosf(th), sinf(th));
  }
  CK(cudaMemcpy(pos, hp, en * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(unit, hu, en * 8, cudaMemcpyHostToDevice));
  free(hp); free(hu);
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  const float thr2 = round_up_f32(sq_boundary(0.1));
  const size_t tb = Tile<float>::bytes(64);
  // EVAC_PROBE_HALFWARP selects the mapping: unset, one environment per warp (32 x 2, the step kernel's); 2, 16 lanes x 4
  // pedestrians per environment, two environments per warp; 8, 8 lanes x 8 pedestrians, four environments per warp
  const char* hw = getenv("EVAC_PROBE_HALFWARP");
  const int mapping = hw ? atoi(hw) : 0;
  for (int rep = 0; rep < 2; ++rep) {
    CK(cudaEventRecord(e0));
    if (mapping == 2) probe_pairwise_kernel<16, 4, 2, 2, 16><<<(num_envs + 1) / 2, 32, 2 * tb>>>(pos, unit, out, n, reps, thr2, num_envs);
    // quarter warp x 8 pedestrians per environment, four environments per warp: one broadcast LDS.128 pair per 64 packed math
    // instructions (32 x 2: per 16) -- measured 50.9 % of the FFMA2 peak at 65 536 x 60 (32 x 2: 46.2 %, 16 x 4: 48.1 %); unroll 1 / 4,
    // 12 resident warps or eight environments per CTA: 46.4 / 48.3 / 50.1 / 50.2 %
    else if (mapping == 8) probe_pairwise_kernel<8, 8, 2, 4, 16><<<(num_envs + 3) / 4, 32, 4 * tb>>>(pos, unit, out, n, reps, thr2, num_envs);
    else probe_pairwise_kernel<32, 2><<<num_envs, 32, tb>>>(pos, unit, out, n, reps, thr2, num_envs);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
  }
  CK(cudaGetLastError());
  CK(cudaEventElapsedTime(ms, e0, e1));
  *pairs = (double)num_envs * (double)n * (double)n * (double)reps;
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(pos); cudaFree(unit); cudaFree(out);
  return EVAC_OK;
}

}  // extern "C"
