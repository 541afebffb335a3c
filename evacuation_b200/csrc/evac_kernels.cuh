// Fused evacuation step kernels for sm_100a (B200).
//
// One CTA per environment.  The CTA stages that environment's pedestrian positions and unit
// directions in shared memory, every thread owns PPT pedestrians in registers, and ONE kernel
// performs, per step (reference file:line in brackets, relative to the reference root):
//   agent step + wall test                         [src/env/env/area.py:182-210]
//   escaped / exiting preparation                  [area.py:79-90]
//   Vicsek neighbour alignment inside the vision radius, O(N^2) pairwise pass   [area.py:93-120]
//   additive angular noise (injected or Philox)    [area.py:124-133]
//   leader enslaving blend                         [area.py:138-142]
//   position integration + wall reflection         [area.py:144-152]
//   status transitions                             [src/env/env/statuses.py:29-48]
//   status / intrinsic rewards, termination        [src/env/env/reward.py:19-46, area.py:174-180, env.py:158-171]
//   observation encoding (abs/rel, no/ohe/cat, Dict/Box, gravity)   [src/env/wrappers/wrappers.py:8-96,
//                                                   src/env/wrappers/gravity_encoding.py:8-81]
//   optional same-step auto-reset                  [pedestrians.py:16-27 semantics, gymnasium vector env]
// and can iterate `num_steps` steps with the state resident in registers / shared memory.
//
// The pairwise pass uses Blackwell's packed FP32 pipe instructions (FADD2 / FMUL2 / FFMA2 via
// __fadd2_rn / __fmul2_rn / __ffma2_rn, sm_100+ only): two neighbours j are evaluated per
// instruction, the "is inside the vision radius" mask is folded into the data as a 0/1 float
// (one FSET per pair) so there is no predicated control flow, and non-moving (escaped / padding)
// slots are parked far away with a zero direction.  Nothing here is a dense contraction, so the
// tensor cores are not used (BASELINE.json north_star).
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <type_traits>

#include "philox.cuh"

namespace evac {

constexpr int ST_NONE = 0, ST_VISCEK = 1, ST_FOLLOWER = 2, ST_EXITING = 3, ST_ESCAPED = 4;
constexpr int POS_ABS = 0, POS_REL = 1, POS_GRAV = 2;
constexpr int STAT_NO = 0, STAT_OHE = 1, STAT_CAT = 2;
constexpr int OBS_DICT = 0, OBS_BOX = 1;
constexpr int AGENT_TABLE = 0, AGENT_RANDOM = 1, AGENT_ROTATING = 2, AGENT_WACUUM = 3;
constexpr int NUM_EPISODE_STATS = 9;
constexpr float PARK = 1.0e18f;  // parking coordinate of non-moving slots: (1e18)^2*2 < FLT_MAX

template <typename real> struct vec2;
template <> struct vec2<float> { using type = float2; };
template <> struct vec2<double> { using type = double2; };

// Everything a launch needs; passed by value as a __grid_constant__.
template <typename real>
struct KArgs {
  // ---- shapes
  int E, N, obs_dim;
  // ---- physics (EnvConfig)
  real width, height, step_size, noise_coef, enslaving, one_minus_enslaving;
  float width_f, height_f, step_size_f, eps_f, enslaving_f;  // the agent's arithmetic is float32 in the reference
  // thresholds on SQUARED distances, chosen on the host so that (d2 < thr2) == (sqrt(d2) < thr) exactly
  real thr2_ped, thr2_leader, thr2_exit, thr2_escape;
  // uniform cell grid of the neighbour search (float32): cells_x * cells_y cells of edge >= vision radius over
  // [-width,width] x [-height,height]; cells_x == 0 -> brute-force tiled pass.  N <= 64: the cell masks of the one-warp
  // kernel's sparse pass (evac_warp.cuh), taken per warp and step unless the all-pairs loop is cheaper or cell_force is set
  int cells_x, cells_y, cell_reach;  // neighbours within `cell_reach` cells (cell edge >= radius / cell_reach)
  int cell_pair_walk;                // cell_list_pass step 5: two adjacent sorted slots of one cell row per thread (shared window)
  int cell_force;                    // N <= 64: the sparse pass whenever it is exact (no cost comparison)
  float cell_inv_x, cell_inv_y;      // cells per unit length
  int exit_reward, follow_reward, term_wall;
  real init_reward, intrinsic_coef;
  int max_timesteps;
  real inv_200n, inv_n;  // 1/(200 N), 1/N  (float path only; the double path divides like the reference)
  // ---- observation (EnvWrappersConfig)
  int positions, statuses, obs_type;
  real alpha, eps;
  int alpha_plus2_int;  // alpha + 2 when it is a small integer, else 0 (=> pow)
  int auto_reset;
  // ---- persistent state (owned by the handle)
  typename vec2<real>::type* pos;  // [E,N]
  typename vec2<real>::type* dir;  // [E,N]
  uint8_t* status;                 // [E,N]
  float2* agent_pos;               // [E]
  float2* agent_dir;               // [E]
  int* now;                        // [E]
  int* episode;                    // [E]   episode index (Philox counter word)
  long long* overall;              // [E]   overall_timesteps
  double* acc;                     // [E,3] episode_reward, episode_intrinsic_reward, episode_status_reward
  float* ep_stats;                 // [E,9] last finished episode
  uint8_t* ep_finished;            // [E]
  double* totals;                  // [1+9]
  int* agent_state;                // [E]   WacuumCleaner state machine (phase | heading << 2 | steps-down << 8)
  // N <= 64 float32 handles (the one-warp kernel family) keep ALL of the above in one packed block per environment instead
  // (EnvBlock below; the pointers above are NULL then)
  unsigned char* blocks;           // [E, BLK_BYTES] or NULL
  // WacuumCleaner lane edges [baseline_wacuum_cleaner.py:17-28], compared in float32 like NumPy's weak-scalar promotion
  float wac_top, wac_right, wac_left, wac_bottom;
  // ---- per-call I/O
  const float2* actions;  // [steps,E] or NULL
  const float* noise;     // [steps,E,N] or NULL
  float* obs;             // [E,obs_dim] or [steps,E,obs_dim]
  int obs_every_step;
  float* reward;          // [E]  (sum over steps)
  uint8_t* terminated;    // [E]  (OR over steps)
  uint8_t* truncated;     // [E]
  uint16_t* status_counts;  // [steps,E,4] or NULL: escaped, exiting, following, viscek after every step (pedestrians.py:37-44)
  uint8_t* status_out;      // [E,N] or NULL: dense copy of the statuses after the launch (host face: part of the result block)
  int num_steps, agent_kind;
  uint64_t seed;
  long long env_offset;
};

// ------------------------------------------------------------------------------------------
// Per-environment parameters.  The host converts every EvacEnvParams record exactly as make_args converts the EvacConfig
// fields of the same name, so an environment of a per-env launch computes what a uniform handle built with its record's values
// computes, bit for bit.  One packed, 16-byte aligned record per environment: 32 bytes (float32: two LDG.128), 48 bytes
// (float64: three), loaded once per environment and launch.  The [E] records reach the kernels as their LAST argument, after
// KArgs and the aux kernel's own arguments, so that no argument of the uniform instances moves.
template <typename real>
struct __align__(16) EnvParamRec {
  real one_minus_enslaving, alpha, init_reward, intrinsic_coef;
  float noise_coef, enslaving_f;  // (float)(real)noise_coef, (float)enslaving_degree
  int max_timesteps;
  int bits;  // alpha_plus2_int | exit_reward << 8 | follow_reward << 9 | term_wall << 10
};
static_assert(sizeof(EnvParamRec<float>) == 32 && sizeof(EnvParamRec<double>) == 48, "EnvParamRec is packed");

// The view the step functions read their per-environment parameters from: the fields of KArgs with the same names.  The
// uniform instances pass KArgs itself (env_params<false>), so their code is the code without per-env parameters.
template <typename real>
struct EnvParams {
  real one_minus_enslaving, alpha, init_reward, intrinsic_coef;
  float noise_coef, enslaving_f;
  int max_timesteps, alpha_plus2_int, exit_reward, follow_reward, term_wall;
};

template <bool PE, typename real>
__device__ __forceinline__ std::conditional_t<PE, EnvParams<real>, const KArgs<real>&> env_params(const KArgs<real>& a,
                                                                                                 const EnvParamRec<real>* params, int e) {
  if constexpr (PE) {
    constexpr int V = sizeof(EnvParamRec<real>) / 16;
    union { uint4 v[V]; EnvParamRec<real> r; } u;
    const uint4* src = reinterpret_cast<const uint4*>(params + e);
#pragma unroll
    for (int k = 0; k < V; ++k) u.v[k] = __ldg(src + k);
    EnvParams<real> p;
    p.one_minus_enslaving = u.r.one_minus_enslaving; p.alpha = u.r.alpha;
    p.init_reward = u.r.init_reward; p.intrinsic_coef = u.r.intrinsic_coef;
    p.noise_coef = u.r.noise_coef; p.enslaving_f = u.r.enslaving_f; p.max_timesteps = u.r.max_timesteps;
    p.alpha_plus2_int = u.r.bits & 0xff;
    p.exit_reward = (u.r.bits >> 8) & 1; p.follow_reward = (u.r.bits >> 9) & 1; p.term_wall = (u.r.bits >> 10) & 1;
    return p;
  } else {
    return a;
  }
}

// ------------------------------------------------------------------------------------------
// EnvBlock: packed per-environment state of the one-warp kernel family (N <= 64, float32).  Everything a step reads and
// writes sits in ONE 1152-byte, 128-byte-aligned block, so the kernel forms one address per environment and every access
// is that address + an immediate (+ 16 * lane): two broadcast LDG.128 for the record, one LDG.128 per pedestrian
// ({px, py, dx, dy} interleaved), one LDG.U16 for the lane's two statuses -- and the mirror image for the write-back.
//   [   0,   64)  EnvRec
//   [  64,  128)  statuses: byte 2 l = pedestrian l, byte 2 l + 1 = pedestrian l + 32   (0 = padding slot)
//   [ 128, 1152)  float4 {px, py, dx, dy} of pedestrian i at 128 + 16 i, 64 slots (slots >= N stay zero)
struct __align__(16) EnvRec {
  float2 agent_pos, agent_dir;     //  0: float32 like the reference's agent
  int now, episode, agent_state, pad;  // 16: step in episode, episode index (Philox key word), WacuumCleaner state machine
  long long overall;               // 32: overall_timesteps
  double acc[3];                   // 40: episode_reward, episode_intrinsic_reward, episode_status_reward (env.py:168-170)
};
static_assert(sizeof(EnvRec) == 64, "EnvRec is one 64-byte record");
constexpr int BLK_STATUS = 64, BLK_PED = 128, BLK_SLOTS = 64, BLK_BYTES = BLK_PED + 16 * BLK_SLOTS;
__host__ __device__ __forceinline__ int blk_status_off(int i) { return BLK_STATUS + 2 * (i & 31) + (i >> 5); }

// Layout-independent state access for the kernels OFF the per-step path (reset / status / observe / get / set state).
template <typename real>
__device__ __forceinline__ void state_load_ped(const KArgs<real>& a, int e, int i, real& px, real& py, real& dx, real& dy, int& st) {
  if constexpr (std::is_same<real, float>::value) {
    if (a.blocks != nullptr) {
      const unsigned char* b = a.blocks + (size_t)e * BLK_BYTES;
      const float4 v = reinterpret_cast<const float4*>(b + BLK_PED)[i];
      px = v.x; py = v.y; dx = v.z; dy = v.w;
      st = b[blk_status_off(i)];
      return;
    }
  }
  const typename vec2<real>::type p = a.pos[(size_t)e * a.N + i], d = a.dir[(size_t)e * a.N + i];
  px = p.x; py = p.y; dx = d.x; dy = d.y;
  st = a.status[(size_t)e * a.N + i];
}
template <typename real>
__device__ __forceinline__ void state_store_ped(const KArgs<real>& a, int e, int i, real px, real py, real dx, real dy) {
  if constexpr (std::is_same<real, float>::value) {
    if (a.blocks != nullptr) {
      reinterpret_cast<float4*>(a.blocks + (size_t)e * BLK_BYTES + BLK_PED)[i] = make_float4(px, py, dx, dy);
      return;
    }
  }
  typename vec2<real>::type p, d;
  p.x = px; p.y = py; d.x = dx; d.y = dy;
  a.pos[(size_t)e * a.N + i] = p;
  a.dir[(size_t)e * a.N + i] = d;
}
template <typename real>
__device__ __forceinline__ void state_store_status(const KArgs<real>& a, int e, int i, int st) {
  if constexpr (std::is_same<real, float>::value) {
    if (a.blocks != nullptr) { a.blocks[(size_t)e * BLK_BYTES + blk_status_off(i)] = (uint8_t)st; return; }
  }
  a.status[(size_t)e * a.N + i] = (uint8_t)st;
}
template <typename real>
__device__ __forceinline__ EnvRec* state_rec(const KArgs<real>& a, int e) {
  if constexpr (std::is_same<real, float>::value) return a.blocks ? reinterpret_cast<EnvRec*>(a.blocks + (size_t)e * BLK_BYTES) : nullptr;
  else return nullptr;
}
template <typename real>
__device__ __forceinline__ float2 state_agent_pos(const KArgs<real>& a, int e) {
  const EnvRec* r = state_rec(a, e);
  return r ? r->agent_pos : a.agent_pos[e];
}
template <typename real>
__device__ __forceinline__ int state_episode(const KArgs<real>& a, int e) {
  const EnvRec* r = state_rec(a, e);
  return r ? r->episode : a.episode[e];
}
// thread 0 of a reset: agent at the origin, time and accumulators zeroed, next episode index (area.py:27-30,49-51; env.py:129-135)
template <typename real>
__device__ __forceinline__ void state_reset_rec(const KArgs<real>& a, int e, int episode) {
  if (EnvRec* r = state_rec(a, e)) {
    r->agent_pos = make_float2(0.f, 0.f); r->agent_dir = make_float2(0.f, 0.f);
    r->now = 0; r->episode = episode; r->agent_state = 0;
    r->acc[0] = r->acc[1] = r->acc[2] = 0.0;
    return;
  }
  a.agent_state[e] = 0;
  a.agent_pos[e] = make_float2(0.f, 0.f); a.agent_dir[e] = make_float2(0.f, 0.f);
  a.now[e] = 0; a.episode[e] = episode;
  a.acc[3 * (size_t)e] = a.acc[3 * (size_t)e + 1] = a.acc[3 * (size_t)e + 2] = 0.0;
}

// ------------------------------------------------------------------------------------------
// small math helpers, float / double overloads
__device__ __forceinline__ float rsqrt_(float x) { return rsqrtf(x); }
__device__ __forceinline__ double rsqrt_(double x) { return 1.0 / sqrt(x); }
__device__ __forceinline__ float sqrt_(float x) { return __fsqrt_rn(x); }
__device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
__device__ __forceinline__ float div_(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_(double a, double b) { return a / b; }
__device__ __forceinline__ float min_(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double min_(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ float max_(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double max_(double a, double b) { return fmax(a, b); }

// sqrt for quantities that only feed a 1e-5-tolerance output (intrinsic reward): MUFU.SQRT for float
__device__ __forceinline__ float sqrt_fast(float x) { float r; asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ double sqrt_fast(double x) { return sqrt(x); }

// 1/sqrt(x): float = MUFU.RSQ + one Newton step (rounding-limited, ~1 ulp); rsqrt(0) = inf and the
// Newton step turns it into NaN, so v * inv_norm(0) = NaN exactly like the reference's 0/0 (area.py:101).
__device__ __forceinline__ float inv_norm(float n2) {
  const float y = rsqrtf(n2);
  return y * fmaf(-0.5f * n2 * y, y, 1.5f);
}
__device__ __forceinline__ double inv_norm(double n2) { return 1.0 / sqrt(n2); }

// sin/cos of the angular noise.  |x| <= pi/4 (always true for noise_coef <= pi/2): Cephes single-precision
// minimax polynomials (<= 1 ulp on that interval); otherwise the library sincosf.
__device__ __forceinline__ void sincos_noise(float x, float& sn, float& cn) {
  if (fabsf(x) <= 0.785398163f) {
    const float z = x * x;
    sn = fmaf(fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f) * z, x, x);
    cn = fmaf(fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f) * z, z, fmaf(-0.5f, z, 1.0f));
  } else {
    sincosf(x, &sn, &cn);
  }
}

template <typename real>
__device__ __forceinline__ real ipow(real x, int n) {  // x^n, n >= 1, by squaring
  real r = (real)1;
  while (n) {
    if (n & 1) r *= x;
    x *= x;
    n >>= 1;
  }
  return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// status is a pure function of (pedestrian position, agent position)  [statuses.py:29-48]
template <typename real>
__device__ __forceinline__ int status_of(real px, real py, real apx, real apy, const KArgs<real>& a, real& d2_exit) {
  const real ax = apx - px, ay = apy - py;
  const real da2 = ax * ax + ay * ay;
  const real ex = (real)0 - px, ey = (real)-1 - py;  // exit = (0,-1)  [area.py:36-39]
  d2_exit = ex * ex + ey * ey;
  int s = ST_VISCEK;
  if (da2 < a.thr2_leader) s = ST_FOLLOWER;
  if (d2_exit < a.thr2_exit) s = ST_EXITING;
  if (d2_exit < a.thr2_escape) s = ST_ESCAPED;
  return s;
}

// ------------------------------------------------------------------------------------------
// Shared-memory tile of "source" records: for slot j the position (x,y) and unit direction (ux,uy).
//   float : two slots per float4 -> P2[j/2] = (x_j, x_j+1, y_j, y_j+1), U2[j/2] = (ux_j, ux_j+1, uy_j, uy_j+1)
//           so one LDS.128 feeds one packed (f32x2) operand pair.
//   double: four planar arrays.
template <typename real>
struct Tile;

template <>
struct Tile<float> {
  float4* P2;
  float4* U2;
  __device__ __forceinline__ Tile(unsigned char* base, int slots) {
    P2 = reinterpret_cast<float4*>(base);
    U2 = P2 + slots / 2 + 1;  // +1: spare look-ahead entry (pairwise_pass)
  }
  static __host__ __device__ constexpr size_t bytes(int slots) { return (size_t)slots * 16 + 32; }
  __device__ __forceinline__ void put(int j, float x, float y, float ux, float uy) const {
    float* p = reinterpret_cast<float*>(P2 + (j >> 1)) + (j & 1);
    float* u = reinterpret_cast<float*>(U2 + (j >> 1)) + (j & 1);
    p[0] = x;
    p[2] = y;
    u[0] = ux;
    u[2] = uy;
  }
};

// THE pair evaluation of every float32 neighbour search: one slot pair of the tile (p = P2 entry, u = U2 entry) against one
// pedestrian at (-nx, -ny) (splatted), adds the unit directions of the slots with d² < thr² to (ax, ay).  The host picks thr²
// (sq_boundary, evac_abi.cu) so that this strict < on this float32 expression equals sqrt(d²) < radius.  w * u with w = 0 and
// u = NaN gives NaN, like the reference's (intersection * efv_directions) product.
__device__ __forceinline__ void accumulate_pair(float4 p, float4 u, float2 nx, float2 ny, float thr2, float2& ax, float2& ay) {
  const float2 dx = __fadd2_rn(make_float2(p.x, p.y), nx);
  const float2 dy = __fadd2_rn(make_float2(p.z, p.w), ny);
  float2 d2 = __fmul2_rn(dx, dx);
  d2 = __ffma2_rn(dy, dy, d2);
  const float2 w = make_float2(d2.x < thr2 ? 1.f : 0.f, d2.y < thr2 ? 1.f : 0.f);
  ax = __ffma2_rn(w, make_float2(u.x, u.y), ax);
  ay = __ffma2_rn(w, make_float2(u.z, u.w), ay);
}

template <>
struct Tile<double> {
  double *X, *Y, *UX, *UY;
  __device__ __forceinline__ Tile(unsigned char* base, int slots) {
    X = reinterpret_cast<double*>(base);
    Y = X + slots;
    UX = Y + slots;
    UY = UX + slots;
  }
  static __host__ __device__ constexpr size_t bytes(int slots) { return (size_t)slots * 32; }
  __device__ __forceinline__ void put(int j, double x, double y, double ux, double uy) const {
    X[j] = x;
    Y[j] = y;
    UX[j] = ux;
    UY[j] = uy;
  }
};

// The pairwise neighbour-alignment pass [area.py:105-119]: for each of this thread's PPT pedestrians
// i, sum the unit directions of all slots j with |p_i - p_j|^2 < thr2 (self included).
// The fp64 pass (parity mode) also returns cnt[], the number of neighbours (area.py:108).
template <int PPT, int UNR = 4>  // @region pairwise
__device__ __forceinline__ void pairwise_pass(const Tile<float>& t, int nslots, const float (&xi)[PPT],
                                              const float (&yi)[PPT], float thr2, float (&sx)[PPT], float (&sy)[PPT]) {
  float2 ax[PPT], ay[PPT], nx[PPT], ny[PPT];
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    ax[k] = make_float2(0.f, 0.f);
    ay[k] = make_float2(0.f, 0.f);
    nx[k] = make_float2(-xi[k], -xi[k]);
    ny[k] = make_float2(-yi[k], -yi[k]);
  }
  const int n2 = (nslots + 1) >> 1;
  // software pipeline: the operands of iteration j+1 are loaded (broadcast LDS.128) while iteration j is
  // computed, so the ~30-cycle shared-memory latency is off the dependent chain.  The tile carries one
  // spare entry per array, so the look-ahead load of the last iteration stays inside the allocation.
  float4 p = t.P2[0], u = t.U2[0];
#pragma unroll(UNR)
  for (int j = 0; j < n2; ++j) {
    const float4 pn = t.P2[j + 1];
    const float4 un = t.U2[j + 1];
#pragma unroll
    for (int k = 0; k < PPT; ++k) accumulate_pair(p, u, nx[k], ny[k], thr2, ax[k], ay[k]);
    p = pn;
    u = un;
  }
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    sx[k] = ax[k].x + ax[k].y;
    sy[k] = ay[k].x + ay[k].y;
  }
}

template <int PPT>  // @region pairwise64
__device__ __forceinline__ void pairwise_pass(const Tile<double>& t, int nslots, const double (&xi)[PPT],
                                              const double (&yi)[PPT], double thr2, double (&sx)[PPT],
                                              double (&sy)[PPT], double (&cnt)[PPT]) {
#pragma unroll
  for (int k = 0; k < PPT; ++k) sx[k] = sy[k] = cnt[k] = 0.0;
  for (int j = 0; j < nslots; ++j) {
    const double x = t.X[j], y = t.Y[j], ux = t.UX[j], uy = t.UY[j];
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      const double dx = x - xi[k], dy = y - yi[k];
      const double w = (dx * dx + dy * dy < thr2) ? 1.0 : 0.0;
      sx[k] += w * ux;
      sy[k] += w * uy;
      cnt[k] += w;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Cell-list neighbour search for crowds larger than one warp tile (BASELINE config 4: 4096 pedestrians).
// [area.py:105-119 computes the full |fv| x |efv| distance matrix; only pairs closer than the vision
// radius contribute, so binning the sources into a uniform grid of cells with edge >= radius and scanning
// the 3x3 block of cells around each pedestrian evaluates the SAME predicate on a superset of the
// contributing pairs.]  All in shared memory, one CTA per environment:
//   1. histogram of the moving pedestrians over the cells (shared-memory atomics; the returned count is a
//      provisional, non-deterministic rank)                          2. exclusive scan -> cell_start[]
//   3. provisional scatter of pedestrian indices                     4. canonical rank = number of
//      lower-indexed pedestrians of the same cell -> the tile is sorted by (cell, index): the summation
//      order, hence every float32 result, is deterministic
//   5. threads walk the SORTED slots (neighbouring lanes sit in the same / adjacent cells: shared-memory
//      broadcasts, coherent trip counts), three contiguous slot ranges (one per cell row), packed f32x2
//      pair evaluation (accumulate_pair); result scattered to res[original index]
//   6. the owner threads read res[] back.
// Steps 1, 2, the paired walk of step 5 and step 6 are functions shared with the cluster pass (evac_cluster.cuh).
struct CellSmem {
  float2* res;           // [SLOTS]  (aliases `list` until step 5)
  uint16_t* list;        // [SLOTS]  provisional cell lists
  uint16_t* sorted_idx;  // [SLOTS]  original index | 0x8000 if VISCEK/FOLLOWER
  int* cell_start;       // [C + 1]
  int* warp_tot;         // [32]
  int* row_pairs;        // [cells_y + 1 <= 65, 68 reserved: 16-byte multiple]  paired walk: number of slot pairs in the cell rows below (exclusive scan)
  static __host__ __device__ constexpr size_t bytes(int slots, int cells) {
    return (size_t)slots * 8 + (size_t)slots * 2 + (((size_t)cells + 1 + 3) & ~(size_t)3) * 4 + (32 + 68) * 4;
  }
  __device__ __forceinline__ CellSmem(unsigned char* base, int slots, int cells) {
    res = reinterpret_cast<float2*>(base);
    list = reinterpret_cast<uint16_t*>(base);
    sorted_idx = reinterpret_cast<uint16_t*>(base + (size_t)slots * 8);
    cell_start = reinterpret_cast<int*>(base + (size_t)slots * 10);
    warp_tot = cell_start + ((cells + 1 + 3) & ~3);
    row_pairs = warp_tot + 32;
  }
};

template <typename A>
__device__ __forceinline__ int cell_of(float x, float y, const A& a, int& cx, int& cy) {
  cx = min(max((int)((x + a.width_f) * a.cell_inv_x), 0), a.cells_x - 1);  // (int)NaN == 0
  cy = min(max((int)((y + a.height_f) * a.cell_inv_y), 0), a.cells_y - 1);
  return cy * a.cells_x + cx;
}

// ---- Phases shared by cell_list_pass (one CTA) and cell_list_pass_cluster (evac_cluster.cuh).  Both sort the sources by
// (cell, pedestrian index), so every float32 sum has the same value in either.

// Step 1: the cell of every moving pedestrian and its rank among the moving pedestrians of that cell in pedestrian index
// order (pass k, warp, lane); the cell totals are added to count[] (zeroed by the caller).
//   * lanes of one warp that share a cell find each other with MATCH.ANY (rank among them = lower lanes),
//   * the leader records the group size in cnt[warp][cell] (uint8, [WARPS][C] bytes that alias the tile: the caller writes
//     the tile only afterwards) and adds it to the counter (integer atomics commute),
//   * after the barrier a source's rank is counter-after-this-pass minus the groups of the warps at or above its own.
// Returns whether one of this thread's sources has no direction.
template <int THREADS, int PPT, typename A>
__device__ __forceinline__ bool rank_in_cells(const Tile<float>& tile, int* count, const A& a, const float (&px)[PPT],
                                              const float (&py)[PPT], const float (&ux)[PPT], const float (&uy)[PPT],
                                              const bool (&efv)[PPT], int (&cell)[PPT], int (&rank)[PPT]) {
  constexpr int WARPS = THREADS / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = a.cells_x * a.cells_y;
  uint8_t* cnt = reinterpret_cast<uint8_t*>(tile.P2);
  const int n16 = (WARPS * C + 15) >> 4;
  const uint32_t lt_mask = (1u << lane) - 1u;
  bool nan_src = false;
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    for (int i = tid; i < n16; i += THREADS) reinterpret_cast<uint4*>(cnt)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    cell[k] = 0; rank[k] = 0;
    int lrank = 0;
    const uint32_t act = __ballot_sync(0xffffffffu, efv[k]);
    if (efv[k]) {
      int cx, cy;
      cell[k] = cell_of(px[k], py[k], a, cx, cy);
      nan_src |= (ux[k] != ux[k]) | (uy[k] != uy[k]);
      const uint32_t peers = __match_any_sync(act, cell[k]);
      lrank = __popc(peers & lt_mask);
      if (lrank == 0) {
        const int n = __popc(peers);
        cnt[warp * C + cell[k]] = (uint8_t)n;
        atomicAdd(&count[cell[k]], n);
      }
    }
    __syncthreads();
    if (efv[k]) {
      int above = 0;
      for (int w = warp; w < WARPS; ++w) above += cnt[w * C + cell[k]];
      rank[k] = count[cell[k]] - above + lrank;
    }
    __syncthreads();  // cnt is cleared and the counters move on in the next pass
  }
  return nan_src;
}

// Step 2: exclusive scan of the C + 1 counters cs.cell_start[] in place (entry C receives the total).  Returns the total,
// after a barrier.
template <int THREADS>
__device__ __forceinline__ int scan_cell_counts(const CellSmem& cs, int C) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (C + THREADS) / THREADS;  // ceil((C + 1) / THREADS)
  const int lo = min(tid * per, C + 1), hi = min(lo + per, C + 1);
  int sum = 0;
  for (int c = lo; c < hi; ++c) sum += cs.cell_start[c];
  int inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
  if (lane == 31) cs.warp_tot[warp] = inc;
  __syncthreads();
  int off = inc - sum;
  for (int w = 0; w < warp; ++w) off += cs.warp_tot[w];
  for (int c = lo; c < hi; ++c) { const int v = cs.cell_start[c]; cs.cell_start[c] = off; off += v; }
  __syncthreads();
  return cs.cell_start[C];
}

// Paired walk, by warp 0: slot pairs per cell row (a pair never straddles two rows), exclusive scan over the <= 64 rows ->
// cs.row_pairs[].
template <typename A>
__device__ __forceinline__ void scan_row_pairs(const CellSmem& cs, const A& a) {
  const int lane = threadIdx.x & 31;
  int cnt[2], inc = 0, run = 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = lane + 32 * k;
    cnt[k] = r < a.cells_y ? (cs.cell_start[(r + 1) * a.cells_x] - cs.cell_start[r * a.cells_x] + 1) >> 1 : 0;
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    inc = cnt[k];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
    const int r = lane + 32 * k;
    if (r <= a.cells_y) cs.row_pairs[r] = run + inc - cnt[k];
    run += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (lane == 0 && a.cells_y == 64) cs.row_pairs[64] = run;
}

// The sorted slots as the paired walk sees them in one CTA: sorted_idx[], the tile and res[] in this CTA's shared memory.
// run(j, je, end): the slot pairs [j, end) that p(q) / u(q) read from one base (here all of [j, je)).
// (The cluster pass has the same interface over the tile distributed across the cluster: ClusterSlots, evac_cluster.cuh.)
struct CtaSlots {
  const Tile<float>& tile;
  const CellSmem& cs;
  struct Run {
    const float4 *P, *U;
    __device__ __forceinline__ float4 p(int q) const { return P[q]; }
    __device__ __forceinline__ float4 u(int q) const { return U[q]; }
  };
  __device__ __forceinline__ int sorted_idx(int s) const { return cs.sorted_idx[s]; }
  __device__ __forceinline__ float4 p2(int pair) const { return tile.P2[pair]; }
  __device__ __forceinline__ Run run(int j, int je, int& end) const {
    end = je;
    return {tile.P2 + j, tile.U2 + j};
  }
  __device__ __forceinline__ void put_res(int i, float2 r) const { cs.res[i] = r; }
};

// Paired walk of slot pair t: the two adjacent sorted slots 2t', 2t' + 1 of ONE cell row (row_pairs[] numbering) sit in the
// same or in neighbouring cells, so one walk over the union of their windows serves both -- every loaded source pair is
// evaluated against two pedestrians (half the LDS per evaluated pair, like the 2-pedestrians-per-lane all-pairs pass).  A slot
// outside a pedestrian's own window fails the distance test and adds an exact zero, so the sums equal the one-slot walk bit
// for bit.  cs: this CTA's cell_start[] and row_pairs[]; Slots: where the sorted slots and the results live.
template <typename Slots, typename A>
__device__ __forceinline__ void walk_slot_pair(const Slots& slots, const CellSmem& cs, const A& a, int t) {
  int row = 0;
  {  // largest row with row_pairs[row] <= t
    int hi_r = a.cells_y;
    while (hi_r - row > 1) { const int mid = (row + hi_r) >> 1; if (cs.row_pairs[mid] <= t) row = mid; else hi_r = mid; }
  }
  const int row_end = cs.cell_start[(row + 1) * a.cells_x];
  const int s0 = cs.cell_start[row * a.cells_x] + 2 * (t - cs.row_pairs[row]);
  const bool two = s0 + 1 < row_end;
  const int id0 = slots.sorted_idx(s0), id1 = two ? slots.sorted_idx(s0 + 1) : 0;
  if (!((id0 | id1) & 0x8000)) return;
  const float4 p0 = slots.p2(s0 >> 1);
  const float x0 = (s0 & 1) ? p0.y : p0.x, y0 = (s0 & 1) ? p0.w : p0.z;
  float x1 = x0, y1 = y0;
  if (two) { const float4 p1 = slots.p2((s0 + 1) >> 1); x1 = ((s0 + 1) & 1) ? p1.y : p1.x; y1 = ((s0 + 1) & 1) ? p1.w : p1.z; }
  const int reach = a.cell_reach;
  int cxa, cxb, cy_;
  cell_of(x0, y0, a, cxa, cy_);
  cell_of(x1, y1, a, cxb, cy_);
  const int cx0 = max(min(cxa, cxb) - reach, 0), cx1 = min(max(cxa, cxb) + reach, a.cells_x - 1);
  const float2 nx0 = make_float2(-x0, -x0), ny0 = make_float2(-y0, -y0), nx1 = make_float2(-x1, -x1), ny1 = make_float2(-y1, -y1);
  const float thr2 = a.thr2_ped;
  float2 ax0 = make_float2(0.f, 0.f), ay0 = ax0, ax1 = ax0, ay1 = ax0;
  int done = 0;  // even slot index below which everything has been evaluated already
  for (int r = max(row - reach, 0); r <= min(row + reach, a.cells_y - 1); ++r) {
    const int lo = max(cs.cell_start[r * a.cells_x + cx0] & ~1, done);
    const int hi = (cs.cell_start[r * a.cells_x + cx1 + 1] + 1) & ~1;
    int j = lo >> 1;
    const int je = hi >> 1;
    while (j < je) {
      int end;
      const typename Slots::Run run = slots.run(j, je, end);
      // software pipeline: the next slot pair is in flight while this one is evaluated (the look-ahead of the last iteration
      // reads one entry past the run: at most the spare entry behind the tile or slice, allocated and never used)
      float4 p = run.p(0), u = run.u(0);
#pragma unroll 2
      for (int q = 0; q < end - j; ++q) {
        const float4 pn = run.p(q + 1), un = run.u(q + 1);
        accumulate_pair(p, u, nx0, ny0, thr2, ax0, ay0);
        accumulate_pair(p, u, nx1, ny1, thr2, ax1, ay1);
        p = pn;
        u = un;
      }
      j = end;
    }
    done = max(done, hi);
  }
  if (id0 & 0x8000) slots.put_res(id0 & 0x7fff, make_float2(ax0.x + ax0.y, ay0.x + ay0.y));
  if (id1 & 0x8000) slots.put_res(id1 & 0x7fff, make_float2(ax1.x + ax1.y, ay1.x + ay1.y));
}

// Last step: the owners read their results back from res[]; one source without a direction poisons EVERY sum in the
// reference (0 * NaN = NaN, area.py:101,118).
template <int THREADS, int PPT>
__device__ __forceinline__ void read_results(const CellSmem& cs, bool poisoned, const int (&st)[PPT], float (&sx)[PPT],
                                             float (&sy)[PPT]) {
  const float qnan = __int_as_float(0x7fc00000);
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    sx[k] = sy[k] = 0.f;
    const bool fv = (unsigned)(st[k] - ST_VISCEK) <= (unsigned)(ST_FOLLOWER - ST_VISCEK);
    if (fv) {
      const float2 r = cs.res[k * THREADS + threadIdx.x];
      sx[k] = poisoned ? qnan : r.x;
      sy[k] = poisoned ? qnan : r.y;
    }
  }
}

template <int THREADS, int PPT, typename A>
__device__ __forceinline__ void cell_list_pass(const Tile<float>& tile, const CellSmem& cs, const A& a, const float (&px)[PPT],
                                               const float (&py)[PPT], const float (&ux)[PPT], const float (&uy)[PPT],
                                               const bool (&efv)[PPT], const int (&st)[PPT], float (&sx)[PPT], float (&sy)[PPT]) {
  constexpr int WARPS = THREADS / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = a.cells_x * a.cells_y;
  // ---- 1. histogram + rank of every source inside its cell (rank_in_cells).  If its [WARPS][C] byte table does not fit in
  // the tile (more than 2048 cells at 32 warps) the ranks come from the arrival order of the atomics and are made canonical
  // by counting lower indices in the cell (step 4b).
  for (int c = tid; c <= C; c += THREADS) cs.cell_start[c] = 0;
  int cell[PPT], rank[PPT];
  bool nan_src = false;
  const bool fast_rank = (size_t)WARPS * C + 16 <= Tile<float>::bytes(THREADS * PPT);
  if (fast_rank) {
    nan_src = rank_in_cells<THREADS, PPT>(tile, cs.cell_start, a, px, py, ux, uy, efv, cell, rank);
  } else {
    __syncthreads();
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      cell[k] = 0; rank[k] = 0;
      if (efv[k]) {
        int cx, cy;
        cell[k] = cell_of(px[k], py[k], a, cx, cy);
        rank[k] = atomicAdd(&cs.cell_start[cell[k]], 1);
        nan_src |= (ux[k] != ux[k]) | (uy[k] != uy[k]);
      }
    }
  }
  const bool poisoned = __syncthreads_or(nan_src);
  // ---- 2. exclusive scan of the C + 1 counters
  const int n_src = scan_cell_counts<THREADS>(cs, C);
  // ---- 3. (arrival-order ranks only) provisional scatter, 4b. canonical rank = number of lower indices in the cell
  if (!fast_rank) {
#pragma unroll
    for (int k = 0; k < PPT; ++k)
      if (efv[k]) cs.list[cs.cell_start[cell[k]] + rank[k]] = (uint16_t)(k * THREADS + tid);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      if (efv[k]) {
        const int i = k * THREADS + tid;
        const int b = cs.cell_start[cell[k]], e = cs.cell_start[cell[k] + 1];
        int r = 0;
        for (int q = b; q < e; ++q) r += ((int)cs.list[q] < i);
        rank[k] = r;
      }
    }
  }
  // ---- 4. final scatter of the source records (tile / sorted_idx do not alias list)
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    if (efv[k]) {
      const int i = k * THREADS + tid;
      const int r = cs.cell_start[cell[k]] + rank[k];
      const bool fv = (unsigned)(st[k] - ST_VISCEK) <= (unsigned)(ST_FOLLOWER - ST_VISCEK);
      tile.put(r, px[k], py[k], ux[k], uy[k]);
      cs.sorted_idx[r] = (uint16_t)(i | (fv ? 0x8000 : 0));
    }
  }
  if (tid < 2) tile.put(n_src + tid, PARK, PARK, 0.f, 0.f);  // pad to an even count (the tile has 2 spare slots)
  if (a.cell_pair_walk && warp == 0) scan_row_pairs(cs, a);
  __syncthreads();  // list[] (aliased by res[]) is dead from here on
  // ---- 5. walk the sorted slots
  if (a.cell_pair_walk) {
    // chunks of 32 slot pairs are handed to the warps statically: warp w walks chunks w, w + WARPS, ...
    const int n_pairs = cs.row_pairs[a.cells_y];
#pragma unroll 1
    for (int chunk = warp; chunk * 32 < n_pairs; chunk += WARPS) {
      const int t = chunk * 32 + lane;
      if (t < n_pairs) walk_slot_pair(CtaSlots{tile, cs}, cs, a, t);
    }
  } else {
    const float thr2 = a.thr2_ped;
#pragma unroll 1
    for (int s = tid; s < n_src; s += THREADS) {
      const int id = cs.sorted_idx[s];
      if (!(id & 0x8000)) continue;
      const float4 pp = tile.P2[s >> 1];
      const float x = (s & 1) ? pp.y : pp.x, y = (s & 1) ? pp.w : pp.z;
      int cx, cy;
      cell_of(x, y, a, cx, cy);
      const int reach = a.cell_reach;
      const int cx0 = max(cx - reach, 0), cx1 = min(cx + reach, a.cells_x - 1);
      const float2 nx = make_float2(-x, -x), ny = make_float2(-y, -y);
      float2 ax = make_float2(0.f, 0.f), ay = make_float2(0.f, 0.f);
      int done = 0;  // even slot index below which everything has been evaluated already
      for (int row = max(cy - reach, 0); row <= min(cy + reach, a.cells_y - 1); ++row) {
        const int lo = max(cs.cell_start[row * a.cells_x + cx0] & ~1, done);
        const int hi = (cs.cell_start[row * a.cells_x + cx1 + 1] + 1) & ~1;
        int j = lo >> 1;
        const int je = hi >> 1;
        if (j < je) {
          // software pipeline as in walk_slot_pair
          float4 p = tile.P2[j], u = tile.U2[j];
#pragma unroll 2
          for (; j < je; ++j) {
            const float4 pn = tile.P2[j + 1], un = tile.U2[j + 1];
            accumulate_pair(p, u, nx, ny, thr2, ax, ay);
            p = pn;
            u = un;
          }
        }
        done = max(done, hi);
      }
      cs.res[id & 0x7fff] = make_float2(ax.x + ax.y, ay.x + ay.y);
    }
  }
  __syncthreads();
  // ---- 6. back to the owners
  read_results<THREADS, PPT>(cs, poisoned, st, sx, sy);
}

// A one-warp CTA only needs warp-level convergence + memory ordering, not a hardware barrier.  // @region helpers
template <int WARPS>
__device__ __forceinline__ void cta_sync() {
  if constexpr (WARPS == 1) __syncwarp(); else __syncthreads();
}

// ------------------------------------------------------------------------------------------
// CTA-wide reductions.  Warp level: REDUX (ints) / shuffles (floats); across warps: shared memory.
template <int WARPS>
struct RedScratch {
  int i[WARPS][4];
  double f[WARPS][4];
};

// ------------------------------------------------------------------------------------------
// Observation encoding of ONE pedestrian row + (thread 0) the agent / exit rows.
template <typename real>  // @region obs
__device__ __forceinline__ void store_ped_obs(float* __restrict__ row, int i, int N, real px, real py, int st,
                                              float apx, float apy, const KArgs<real>& a) {
  float x = (float)px, y = (float)py;
  if (a.positions == POS_REL) {  // wrappers.py:20-27, hypotenuse sqrt(2) in float32
    const real inv = (real)(1.0 / 1.41421353816986083984375);
    x = (float)((px - (real)apx) * inv);
    y = (float)((py - (real)apy) * inv);
  }
  const int s = 4 - st;  // wrappers.py:47-51: ESCAPED->0, EXITING->1, FOLLOWER->2, VISCEK->3
  if (a.obs_type == OBS_BOX) {
    if (a.statuses == STAT_OHE) {
      float2* r = reinterpret_cast<float2*>(row + (size_t)(i + 2) * 6);
      r[0] = make_float2(x, y);
      r[1] = make_float2(s == 0 ? 1.f : 0.f, s == 1 ? 1.f : 0.f);
      r[2] = make_float2(s == 2 ? 1.f : 0.f, s == 3 ? 1.f : 0.f);
    } else if (a.statuses == STAT_CAT) {
      float* r = row + (size_t)(i + 2) * 3;
      r[0] = x;
      r[1] = y;
      r[2] = 0.25f * (float)s;
    } else {
      *reinterpret_cast<float2*>(row + (size_t)(i + 2) * 2) = make_float2(x, y);
    }
  } else {  // Dict: [agent(2) | exit(2) | peds(2N) | statuses]
    // (scalar stores: the row stride 4+2N(+4N|+N) floats is not always a multiple of 8 bytes)
    row[4 + 2 * (size_t)i] = x;
    row[5 + 2 * (size_t)i] = y;
    float* sr = row + 4 + 2 * (size_t)N;
    if (a.statuses == STAT_OHE) {
      sr[4 * (size_t)i + 0] = s == 0 ? 1.f : 0.f;
      sr[4 * (size_t)i + 1] = s == 1 ? 1.f : 0.f;
      sr[4 * (size_t)i + 2] = s == 2 ? 1.f : 0.f;
      sr[4 * (size_t)i + 3] = s == 3 ? 1.f : 0.f;
    } else if (a.statuses == STAT_CAT) {
      sr[i] = 0.25f * (float)s;
    }
  }
}

template <typename real>
__device__ __forceinline__ void store_head_obs(float* __restrict__ row, float apx, float apy, const KArgs<real>& a) {
  float ex = 0.f, ey = -1.f;
  if (a.positions == POS_REL) {
    const float inv_hyp = (float)(1.0 / 1.41421353816986083984375);
    ex = (0.f - apx) * inv_hyp;
    ey = (-1.f - apy) * inv_hyp;
  }
  if (a.obs_type == OBS_BOX) {
    if (a.statuses == STAT_OHE) {  // wrappers.py:82-88: agent stat [0,0,0,0], exit stat [1,0,0,0]
      float2* r = reinterpret_cast<float2*>(row);
      r[0] = make_float2(apx, apy);
      r[1] = make_float2(0.f, 0.f);
      r[2] = make_float2(0.f, 0.f);
      r[3] = make_float2(ex, ey);
      r[4] = make_float2(1.f, 0.f);
      r[5] = make_float2(0.f, 0.f);
    } else if (a.statuses == STAT_CAT) {  // wrappers.py:89-91: agent 0, exit 1
      row[0] = apx; row[1] = apy; row[2] = 0.f;
      row[3] = ex;  row[4] = ey;  row[5] = 1.f;
    } else {
      row[0] = apx; row[1] = apy; row[2] = ex; row[3] = ey;
    }
  } else {
    row[0] = apx; row[1] = apy; row[2] = ex; row[3] = ey;
  }
}

// per-pedestrian term of grad_potential_pedestrians [gravity_encoding.py:8-25]; pp: the environment's parameters (env_params)
template <typename real, typename P>
__device__ __forceinline__ void grav_term(real px, real py, float apx, float apy, const KArgs<real>& a, const P& pp, real& gx, real& gy) {
  const real rx = (real)apx - px, ry = (real)apy - py;
  const real norm = sqrt_(rx * rx + ry * ry) + a.eps;
  const real p = pp.alpha_plus2_int ? ipow(norm, pp.alpha_plus2_int) : (real)pow((double)norm, (double)pp.alpha + 2.0);
  const real c = div_(-pp.alpha, p);
  gx = c * rx;
  gy = c * ry;
}

template <typename real, typename P>
__device__ __forceinline__ void store_grav_obs(float* __restrict__ row, float apx, float apy, real gpx, real gpy,
                                               int n_followers, const KArgs<real>& a, const P& pp) {
  // grad_potential_exit [gravity_encoding.py:28-38], float32 like the reference (agent, exit are float32)
  const float rx = apx - 0.f, ry = apy + 1.f;
  const float norm = __fsqrt_rn(rx * rx + ry * ry) + (float)a.eps;
  const float alpha = (float)pp.alpha;
  const float p = pp.alpha_plus2_int ? ipow(norm, pp.alpha_plus2_int) : powf(norm, alpha + 2.f);
  const float c = __fdiv_rn(-alpha, p);
  row[0] = apx;
  row[1] = apy;
  row[2] = c * rx * (float)n_followers;
  row[3] = c * ry * (float)n_followers;
  row[4] = (float)gpx;
  row[5] = (float)gpy;
}

// WacuumCleaner.act [baseline_wacuum_cleaner.py:31-80]: climb to the top wall, sweep in horizontal lanes (25 steps down
// between lanes), then walk to the exit.  state = phase (0 climb, 1 sweep, 2 exit) | heading-left << 2 | steps-down << 8.
template <typename A>
__device__ __forceinline__ void wacuum_act(float px, float py, int& state, const A& a, float& ax, float& ay) {
  int phase = state & 3, left = (state >> 2) & 1, down = state >> 8;
  ax = 0.f - px; ay = -1.f - py;  // task_2: exit_position - pos (float32)
  if (phase == 0) {
    if (py < a.wac_top) { ax = 0.f; ay = 1.f; }
    else { phase = 1; ax = 1.f; ay = 0.f; }
  } else if (phase == 1) {
    if (down > 0) {
      down -= 1;
      if (py > a.wac_bottom) { ax = 0.f; ay = -1.f; }
      else phase = 2;
    } else {
      const bool lane_open = left ? (px > a.wac_left) : (px < a.wac_right);
      if (lane_open) { ax = left ? -1.f : 1.f; ay = 0.f; }
      else { left ^= 1; down = 25; ax = 0.f; ay = -1.f; }
    }
  }
  state = phase | (left << 2) | (down << 8);
}

// fresh random layout of one pedestrian [pedestrians.py:17-20]  // @region reset
template <typename real>
__device__ __forceinline__ void random_layout(uint64_t seed, uint32_t env, uint32_t episode, uint32_t ped, real& px,
                                              real& py, real& dx, real& dy) {
  const Philox4 r = evac_random(seed, STREAM_RESET, env, episode, 0u, ped);
  px = (real)(2.f * u01(r.x) - 1.f);
  py = (real)(2.f * u01(r.y) - 1.f);
  real vx = (real)(2.f * u01(r.z) - 1.f), vy = (real)(2.f * u01(r.w) - 1.f);
  if (vx == (real)0 && vy == (real)0) vx = (real)1;
  const real n = sqrt_(vx * vx + vy * vy);
  dx = div_(vx, n);
  dy = div_(vy, n);
}

// ------------------------------------------------------------------------------------------
// The per-environment part of a step, shared by evac_warp_kernel and evac_step_kernel.  Each kernel keeps its own loads
// (placed where their latency hides) and reductions, and passes the loaded values and reduced counts in.

// RandomAgent: action_space.sample() ~ U[-1,1)^2 [random_agent.py:8-9]
__device__ __forceinline__ float2 random_action(uint64_t seed, uint32_t env, uint32_t episode, uint32_t now_prev) {
  const uint2 r = evac_agent_block(seed, env, episode, now_prev);
  return make_float2(2.f * u01(r.x) - 1.f, 2.f * u01(r.y) - 1.f);
}

// WacuumCleaner / RotatingAgent action; calls = the RotatingAgent's act() count including this call, which never restarts
// with an episode [rotating_agent.py:8-16].  (Table and random actions are selected by the caller, next to their loads.)
template <typename A>
__device__ __forceinline__ float2 scripted_action(const A& a, long long calls, float2 ap, int& wac_state) {
  if (a.agent_kind == AGENT_WACUUM) { float2 act; wacuum_act(ap.x, ap.y, wac_state, a, act.x, act.y); return act; }
  const double ph = 0.05 * (double)calls;  // float64 like the reference
  return make_float2((float)sin(ph), (float)cos(ph));
}

// Area.agent_step [area.py:182-210], IEEE float32 like the reference; p: the environment's parameters (env_params)
template <typename A, typename P>
__device__ __forceinline__ void agent_step(const A& a, const P& p, float2 act, float2& ap, float2& ad, float& r_agent, bool& term_agent) {
  const float nrm = __fadd_rn(__fsqrt_rn(__fadd_rn(__fmul_rn(act.x, act.x), __fmul_rn(act.y, act.y))), a.eps_f);
  const float ax = __fdiv_rn(act.x, nrm), ay = __fdiv_rn(act.y, nrm);
  ad.x = __fmul_rn(a.step_size_f, ax); ad.y = __fmul_rn(a.step_size_f, ay);
  const float ptx = __fadd_rn(ap.x, ad.x), pty = __fadd_rn(ap.y, ad.y);
  const bool collide = (ptx < -a.width_f) | (ptx > a.width_f) | (pty < -a.height_f) | (pty > a.height_f);
  r_agent = 0.f; term_agent = false;
  if (!collide) { ap.x = ptx; ap.y = pty; }
  else { r_agent = -5.f; term_agent = p.term_wall != 0; }
}

// rewards + termination [reward.py:19-46, area.py:174-180, env.py:158-171]; sd = sum of the distances to the exit
template <typename real, typename P>
__device__ __forceinline__ void step_reward(const KArgs<real>& a, const P& p, int N, int now, real sd, int K_exit, int K_fol, int N_esc,
                                            float r_agent, bool term_agent, real& intrinsic, real& r_status, real& reward, bool& terminated) {
  real tf;
  if constexpr (std::is_same<real, double>::value) { tf = (real)1 - (real)now / (real)(200 * N); intrinsic = (real)0 - sd / (real)N; }
  else { tf = (real)1 - (real)now * a.inv_200n; intrinsic = (real)0 - sd * a.inv_n; }
  real r_ped = p.init_reward;
  if (p.exit_reward) r_ped += ((real)15 + (real)10 * tf) * (real)K_exit;
  if (p.follow_reward) r_ped += ((real)10 + (real)5 * tf) * (real)K_fol;
  r_status = (real)r_agent + r_ped;
  reward = r_status + p.intrinsic_coef * intrinsic;
  terminated = term_agent || (N_esc == N);
}

// pedestrians.status_stats after step s, before a same-step reset [pedestrians.py:37-44]
template <typename real>
__device__ __forceinline__ void store_status_counts(const KArgs<real>& a, int s, int e, int N, int N_esc, int N_exi, int N_fol) {
  reinterpret_cast<ushort4*>(a.status_counts)[(size_t)s * a.E + e] =
      make_ushort4((unsigned short)N_esc, (unsigned short)N_exi, (unsigned short)N_fol, (unsigned short)(N - N_esc - N_exi - N_fol));
}

// a finished episode: the logging dict of env.py:115-125 from its final accumulators and overall_timesteps
template <typename real>
__device__ __forceinline__ void record_episode(const KArgs<real>& a, int e, double acc_i, double acc_s, double acc_r, int now, int N,
                                               int N_esc, int N_exi, int N_fol, long long overall) {
  float* es = a.ep_stats + (size_t)e * NUM_EPISODE_STATS;
  const float v[NUM_EPISODE_STATS] = {(float)acc_i, (float)acc_s, (float)acc_r, (float)now, (float)N_esc, (float)N_exi,
                                      (float)N_fol, (float)(N - N_esc - N_exi - N_fol), (float)overall};
#pragma unroll
  for (int t = 0; t < NUM_EPISODE_STATS; ++t) { es[t] = v[t]; atomicAdd(a.totals + 1 + t, (double)v[t]); }
  atomicAdd(a.totals, 1.0);
  a.ep_finished[e] = 1;
}

// pedestrian i of a new episode: random layout and its status with the agent at the origin; returns the status
template <typename real>
__device__ __forceinline__ int reset_pedestrian(const KArgs<real>& a, uint32_t env, uint32_t episode, uint32_t i, real& px, real& py,
                                                real& dx, real& dy) {
  random_layout<real>(a.seed, env, episode, i, px, py, dx, dy);
  real d2e;
  return status_of<real>(px, py, (real)0, (real)0, a, d2e);
}

// ------------------------------------------------------------------------------------------
// THE fused step kernel.  grid = one CTA per environment (grid-stride), THREADS threads,
// PPT pedestrians per thread (pedestrian i = k*THREADS + tid).  float32 N <= 64 runs evac_warp_kernel
// (evac_warp.cuh) instead; fp64 N <= 64 runs here as ONE WARP per environment (THREADS = 32, PPT = 2):
// no block barrier, reductions are pure REDUX / shuffles, and the moving pedestrians are compacted
// (ballot + popc) so the pairwise pass only visits them.
#include "evac_cluster.cuh"

// CL > 1: ONE environment per thread-block cluster of CL CTAs (evac_cluster.cuh) -- CTA r owns pedestrians
// [r * SLOTS, (r + 1) * SLOTS); float32 + cell list only; per-environment scalars are written by CTA 0.
// PE: per-environment parameters (every CTA loads its environment's EnvParamRec; env_params).
template <typename real, int THREADS, int PPT, int CL = 1, bool PE = false>  // @region load
__global__ void __launch_bounds__(THREADS, THREADS == 32 ? 32 : 1) evac_step_kernel(const __grid_constant__ KArgs<real> a,
                                                                                      const EnvParamRec<real>* __restrict__ params) {
  constexpr int WARPS = THREADS / 32;
  constexpr int SLOTS = THREADS * PPT;
  constexpr bool F64 = std::is_same<real, double>::value;
  constexpr bool COMPACT = (WARPS == 1);
  using real2 = typename vec2<real>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ RedScratch<WARPS> red_a, red_b;
  __shared__ double cl_slot[8];  // CL > 1: this CTA's partial sums, read by the other CTAs of the cluster
  int rank_cta = 0;
  if constexpr (CL > 1) rank_cta = (int)cg::this_cluster().block_rank();
  const int base_i = rank_cta * SLOTS;  // first pedestrian of this CTA
  Tile<real> tile(smem_raw, SLOTS);
  bool use_cells = false;  // CTA-uniform: cell-list neighbour search instead of the brute-force tiled pass
  if constexpr (!COMPACT && !F64) use_cells = a.cells_x > 0;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool lead = tid == 0 && rank_cta == 0;  // writes the per-environment scalars
  const int N = a.N;
  const uint32_t lt_mask = (1u << lane) - 1u;
  const float noise_c_cfg = (float)a.noise_coef;  // uniform instances: read here as before (in the loop it schedules differently)

  for (int e = blockIdx.x / CL; e < a.E; e += gridDim.x / CL) {
    decltype(auto) p = env_params<PE>(a, params, e);
    const float noise_c = PE ? (float)p.noise_coef : noise_c_cfg;
    // ---------------- load state (coalesced real2 per thread)
    real2* __restrict__ pos_e = a.pos + (size_t)e * N;
    real2* __restrict__ dir_e = a.dir + (size_t)e * N;
    uint8_t* __restrict__ st_e = a.status + (size_t)e * N;
    real px[PPT], py[PPT], dx[PPT], dy[PPT];
    int st[PPT];
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      const int i = base_i + k * THREADS + tid;
      px[k] = py[k] = dx[k] = dy[k] = (real)0;
      st[k] = ST_NONE;
      if (i < N) {
        const real2 p = pos_e[i];
        const real2 d = dir_e[i];
        px[k] = p.x; py[k] = p.y; dx[k] = d.x; dy[k] = d.y;
        st[k] = st_e[i];
      }
    }
    float2 ap = a.agent_pos[e], ad = a.agent_dir[e];
    int wac_state = (a.agent_kind == AGENT_WACUUM) ? a.agent_state[e] : 0;
    int now = a.now[e];
    int episode = a.episode[e];
    const long long overall_start = a.overall[e];
    int steps_total = 0;
    double acc_r = 0, acc_i = 0, acc_s = 0;
    const uint32_t env_g = (uint32_t)(a.env_offset + e);
    float reward_sum = 0.f;
    int any_term = 0, any_trunc = 0;
    bool acc_reset = false;
    const float* noise_e = a.noise ? a.noise + (size_t)e * N : nullptr;
    float* obs_e = a.obs ? a.obs + (size_t)e * a.obs_dim : nullptr;

    for (int s = 0; s < a.num_steps; ++s) {  // @region rng
      // ---------------- Time.step [area.py:53-59]
      const int now_prev = now;
      now += 1; steps_total += 1;
      const bool truncated = now >= p.max_timesteps;
      // ---------------- random streams of this step (Philox2x32-10, philox.cuh): the RandomAgent action is computed
      // redundantly by every thread; the noise words are drawn where used
      float2 action_r = make_float2(0.f, 0.f);
      if (a.agent_kind == AGENT_RANDOM) action_r = random_action(a.seed, env_g, (uint32_t)episode, (uint32_t)now_prev);
      // ---------------- escaped / exiting preparation + source records [area.py:79-101]  // @region prep
      bool any_fv = false;
      bool efv[PPT];
      real ux[PPT], uy[PPT];
#pragma unroll
      for (int k = 0; k < PPT; ++k) {
        const int so = st[k];
        if (so == ST_ESCAPED) { dx[k] = dy[k] = (real)0; px[k] = (real)0; py[k] = (real)-1; }
        real vx = dx[k], vy = dy[k];
        if (so == ST_EXITING) { vx = (real)0 - px[k]; vy = (real)-1 - py[k]; }
        efv[k] = (unsigned)(so - ST_VISCEK) <= (unsigned)(ST_EXITING - ST_VISCEK);
        any_fv |= (unsigned)(so - ST_VISCEK) <= (unsigned)(ST_FOLLOWER - ST_VISCEK);
        // u = v / |v| (a zero direction gives NaN exactly like area.py:101); exiting: dir = u * min(|v|, step_size)
        if constexpr (F64) {
          const real len = sqrt_(vx * vx + vy * vy);
          ux[k] = div_(vx, len); uy[k] = div_(vy, len);
          if (so == ST_EXITING) { const real sz = min_(len, a.step_size); dx[k] = ux[k] * sz; dy[k] = uy[k] * sz; }
        } else {
          const real n2 = vx * vx + vy * vy;
          const real inv = inv_norm(n2);
          ux[k] = vx * inv; uy[k] = vy * inv;
          if (so == ST_EXITING) { const real sc = min_(n2 * inv, a.step_size) * inv; dx[k] = vx * sc; dy[k] = vy * sc; }
        }
      }
      int n_src = N;  // number of source slots the pairwise pass visits  // @region compact
      if constexpr (COMPACT) {
        // one warp: rank the moving (exiting / following / viscek) pedestrians and store them densely
        int base = 0;
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
          const uint32_t m = __ballot_sync(0xffffffffu, efv[k]);
          if (efv[k]) tile.put(base + __popc(m & lt_mask), px[k], py[k], ux[k], uy[k]);
          base += __popc(m);
        }
        n_src = base;
        if (lane < 2) tile.put(base + lane, (real)PARK, (real)PARK, (real)0, (real)0);  // pad to an even count
      } else if (!use_cells) {
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
          const int i = k * THREADS + tid;
          if (efv[k]) tile.put(i, px[k], py[k], ux[k], uy[k]);
          else tile.put(i, (real)PARK, (real)PARK, (real)0, (real)0);
        }
      }
      cta_sync<WARPS>();
      // ---------------- action source + Area.agent_step [area.py:182-210]  // @region agent
      float2 act;
      if (a.agent_kind == AGENT_TABLE) act = a.actions[(size_t)s * a.E + e];
      else if (a.agent_kind == AGENT_RANDOM) act = action_r;
      else act = scripted_action(a, overall_start + steps_total, ap, wac_state);
      float r_agent; bool term_agent;
      agent_step(a, p, act, ap, ad, r_agent, term_agent);
      // ---------------- pairwise alignment [area.py:105-119]  // @region pairwise
      real sx[PPT], sy[PPT], cnt[PPT];  // cnt: number of neighbours, used by the fp64 update only
      if constexpr (!COMPACT && !F64) {
        if (use_cells) {
          const CellSmem cs(smem_raw + Tile<real>::bytes(SLOTS), SLOTS, a.cells_x * a.cells_y);
          if constexpr (CL > 1) {
            const ClusterSmem xs(smem_raw + Tile<real>::bytes(SLOTS) + CellSmem::bytes(SLOTS, a.cells_x * a.cells_y), a.cells_x * a.cells_y);
            cell_list_pass_cluster<THREADS, PPT, CL>(tile, cs, xs, a, px, py, ux, uy, efv, st, sx, sy);
          } else {
            cell_list_pass<THREADS, PPT>(tile, cs, a, px, py, ux, uy, efv, st, sx, sy);
          }
        }
      }
      if (!use_cells) {
        if (__any_sync(0xffffffffu, any_fv)) {
          if constexpr (F64) pairwise_pass<PPT>(tile, n_src, px, py, a.thr2_ped, sx, sy, cnt);
          else pairwise_pass<PPT>(tile, n_src, px, py, a.thr2_ped, sx, sy);
        } else {
#pragma unroll
          for (int k = 0; k < PPT; ++k) sx[k] = sy[k] = cnt[k] = (real)0;
        }
      }
      // ---------------- new directions, enslaving, integration, reflection, statuses  // @region update
      int k_exit = 0, k_fol = 0, n_esc = 0, n_exi = 0, n_fol = 0;
      real sum_dexit = (real)0;
      const real e_adx = (real)__fmul_rn(p.enslaving_f, ad.x), e_ady = (real)__fmul_rn(p.enslaving_f, ad.y);
#pragma unroll
      for (int k = 0; k < PPT; ++k) {
        const int i = base_i + k * THREADS + tid;
        const int so = st[k];
        const bool fv = (unsigned)(so - ST_VISCEK) <= (unsigned)(ST_FOLLOWER - ST_VISCEK);
        if (fv) {
          float nzf;
          if (noise_e) {
            nzf = noise_e[((size_t)s * a.E) * N + i];
          } else {
            const uint2 r = evac_noise_block(a.seed, env_g, (uint32_t)episode, (uint32_t)now_prev, evac_noise_block_of((uint32_t)i));
            nzf = (u01(evac_noise_word_of((uint32_t)i) ? r.y : r.x) - 0.5f) * noise_c;
          }
          if constexpr (F64) {  // literal transcription of area.py:108-133
            const double n = fmax(1.0, cnt[k]);
            const double th = atan2(sy[k] / n, sx[k] / n) + (double)nzf;
            dx[k] = cos(th) * a.step_size; dy[k] = sin(th) * a.step_size;
          } else {
            // cos/sin(atan2(my,mx) + nz) == unit(m) rotated by nz; atan2(0,0) = 0 -> unit = (1,0)
            const float m2 = sx[k] * sx[k] + sy[k] * sy[k];
            float cx = 1.f, cy = 0.f;
            if (m2 != 0.f) { const float inv = inv_norm(m2); cx = sx[k] * inv; cy = sy[k] * inv; }
            float sn, cn;
            sincos_noise(nzf, sn, cn);
            dx[k] = a.step_size * (cx * cn - cy * sn);
            dy[k] = a.step_size * (cx * sn + cy * cn);
          }
          if (so == ST_FOLLOWER) {  // area.py:138-142; e * agent.direction is float32 in the reference
            dx[k] = e_adx + p.one_minus_enslaving * dx[k];
            dy[k] = e_ady + p.one_minus_enslaving * dy[k];
          }
        }
        if (efv[k]) { px[k] += dx[k]; py[k] += dy[k]; }
        {  // wall reflection for ALL pedestrians [area.py:147-152]
          const real cx = min_(max_(px[k], -a.width), a.width);
          const real cy = min_(max_(py[k], -a.height), a.height);
          const real mx = px[k] - cx, my = py[k] - cy;
          px[k] -= (real)2 * mx; py[k] -= (real)2 * my;
          if (mx != (real)0) dx[k] = -dx[k];
          if (my != (real)0) dy[k] = -dy[k];
        }
        real d2e;
        int sn_ = status_of<real>(px[k], py[k], (real)ap.x, (real)ap.y, a, d2e);
        if (i >= N) { sn_ = ST_NONE; d2e = (real)0; }
        sum_dexit += sqrt_fast(d2e);
        k_exit += (fv && sn_ == ST_EXITING);
        k_fol += (so == ST_VISCEK && sn_ == ST_FOLLOWER);
        n_esc += (sn_ == ST_ESCAPED); n_exi += (sn_ == ST_EXITING); n_fol += (sn_ == ST_FOLLOWER);
        st[k] = sn_;
      }
      // ---------------- CTA reduction of counts + intrinsic distance sum  // @region reduce_reward
      int q0, q1, q2;
      double sd;
      {
        int p0 = k_exit | (k_fol << 16), p1 = n_esc | (n_exi << 16), p2 = n_fol;
        p0 = __reduce_add_sync(0xffffffffu, p0);
        p1 = __reduce_add_sync(0xffffffffu, p1);
        p2 = __reduce_add_sync(0xffffffffu, p2);
        const float sdw = warp_sum((float)sum_dexit);
        if constexpr (WARPS == 1) {
          q0 = p0; q1 = p1; q2 = p2; sd = (double)sdw;
        } else {
          if (lane == 0) { red_a.i[warp][0] = p0; red_a.i[warp][1] = p1; red_a.i[warp][2] = p2; red_a.f[warp][0] = (double)sdw; }
          cta_sync<WARPS>();
          q0 = q1 = q2 = 0; sd = 0;
#pragma unroll
          for (int w = 0; w < WARPS; ++w) { q0 += red_a.i[w][0]; q1 += red_a.i[w][1]; q2 += red_a.i[w][2]; sd += red_a.f[w][0]; }
        }
      }
      int K_exit = q0 & 0xffff, K_fol = q0 >> 16, N_esc = q1 & 0xffff, N_exi = q1 >> 16, N_fol = q2;
      if constexpr (CL > 1) {  // sums over the CTAs of the cluster, in rank order (same bits in every CTA)
        double v[6] = {(double)K_exit, (double)K_fol, (double)N_esc, (double)N_exi, (double)N_fol, sd};
        cluster_sum<CL, 6>(cl_slot, v);
        K_exit = (int)v[0]; K_fol = (int)v[1]; N_esc = (int)v[2]; N_exi = (int)v[3]; N_fol = (int)v[4]; sd = v[5];
      }
      if (a.status_counts != nullptr && lead) store_status_counts(a, s, e, N, N_esc, N_exi, N_fol);
      real intrinsic, r_status, reward; bool terminated;
      step_reward(a, p, N, now, (real)sd, K_exit, K_fol, N_esc, r_agent, term_agent, intrinsic, r_status, reward, terminated);
      reward_sum += (float)reward;
      any_term |= terminated; any_trunc |= truncated;
      acc_r += (double)reward; acc_i += (double)intrinsic; acc_s += (double)r_status;
      // ---------------- same-step auto-reset  // @region reset
      if (a.auto_reset && (terminated || truncated)) {
        if (lead) {
          if (!acc_reset) { acc_r += a.acc[3 * (size_t)e]; acc_i += a.acc[3 * (size_t)e + 1]; acc_s += a.acc[3 * (size_t)e + 2]; }
          record_episode(a, e, acc_i, acc_s, acc_r, now, N, N_esc, N_exi, N_fol, a.overall[e] + steps_total);
        }
        acc_r = acc_i = acc_s = 0; acc_reset = true;
        now = 0; episode += 1; wac_state = 0;
        ap = make_float2(0.f, 0.f); ad = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < PPT; ++k) {
          const int i = base_i + k * THREADS + tid;
          if (i < N) st[k] = reset_pedestrian<real>(a, env_g, (uint32_t)episode, (uint32_t)i, px[k], py[k], dx[k], dy[k]);
        }
      }
      // ---------------- observation  // @region obs
      if (obs_e != nullptr && (a.obs_every_step || s == a.num_steps - 1)) {
        float* row = obs_e + (a.obs_every_step ? (size_t)s * a.E * a.obs_dim : (size_t)0);
        if (a.positions == POS_GRAV) {
          real gx = (real)0, gy = (real)0;
          int nf = 0;
#pragma unroll
          for (int k = 0; k < PPT; ++k) {
            if (st[k] == ST_VISCEK) { real tx, ty; grav_term<real>(px[k], py[k], ap.x, ap.y, a, p, tx, ty); gx += tx; gy += ty; }
            nf += (st[k] == ST_FOLLOWER);
          }
          nf = __reduce_add_sync(0xffffffffu, nf);
          double wx = warp_sum((double)gx), wy = warp_sum((double)gy);
          if constexpr (WARPS > 1) {
            if (lane == 0) { red_b.i[warp][0] = nf; red_b.f[warp][0] = wx; red_b.f[warp][1] = wy; }
            cta_sync<WARPS>();
            nf = 0; wx = 0; wy = 0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) { nf += red_b.i[w][0]; wx += red_b.f[w][0]; wy += red_b.f[w][1]; }
          }
          if constexpr (CL > 1) {
            double v[3] = {(double)nf, wx, wy};
            cluster_sum<CL, 3>(cl_slot, v);
            nf = (int)v[0]; wx = v[1]; wy = v[2];
          }
          if (lead) store_grav_obs<real>(row, ap.x, ap.y, (real)wx, (real)wy, nf, a, p);
        } else {
          if (lead) store_head_obs<real>(row, ap.x, ap.y, a);
#pragma unroll
          for (int k = 0; k < PPT; ++k) {
            const int i = base_i + k * THREADS + tid;
            if (i < N) store_ped_obs<real>(row, i, N, px[k], py[k], st[k], ap.x, ap.y, a);
          }
        }
      }
    }  // steps

    // ---------------- write back  // @region writeback
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      const int i = base_i + k * THREADS + tid;
      if (i < N) {
        real2 p, d;
        p.x = px[k]; p.y = py[k]; d.x = dx[k]; d.y = dy[k];
        pos_e[i] = p;
        dir_e[i] = d;
        st_e[i] = (uint8_t)st[k];
        if (a.status_out != nullptr) a.status_out[(size_t)e * N + i] = (uint8_t)st[k];
      }
    }
    if (lead) {
      a.agent_pos[e] = ap; a.agent_dir[e] = ad;
      a.now[e] = now; a.episode[e] = episode; a.overall[e] += steps_total;
      if (a.agent_kind == AGENT_WACUUM) a.agent_state[e] = wac_state;
      if (acc_reset) { a.acc[3 * (size_t)e] = acc_r; a.acc[3 * (size_t)e + 1] = acc_i; a.acc[3 * (size_t)e + 2] = acc_s; }
      else { a.acc[3 * (size_t)e] += acc_r; a.acc[3 * (size_t)e + 1] += acc_i; a.acc[3 * (size_t)e + 2] += acc_s; }
      if (a.reward) a.reward[e] = reward_sum;
      if (a.terminated) a.terminated[e] = (uint8_t)any_term;
      if (a.truncated) a.truncated[e] = (uint8_t)any_trunc;
    }
    cta_sync<WARPS>();  // smem tile / scratch reuse by the next environment of this CTA
  }
}

// ------------------------------------------------------------------------------------------  // @region aux
// Auxiliary kernel (not on the per-step path): reset / recompute statuses / encode observations.
// One 128-thread CTA per environment, pedestrians strided over the threads.
enum { AUX_RESET = 1, AUX_STATUS = 2, AUX_OBS = 4 };

// PE: per-environment parameters (the gravity encoding's alpha).
template <typename real, bool PE = false>
__global__ void __launch_bounds__(128) evac_aux_kernel(const __grid_constant__ KArgs<real> a, int flags,
                                                       const uint8_t* __restrict__ mask, float* __restrict__ obs,
                                                       const EnvParamRec<real>* __restrict__ params) {
  __shared__ RedScratch<4> red;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = a.N;
  for (int e = blockIdx.x; e < a.E; e += gridDim.x) {
    const bool sel = (mask == nullptr) || (mask[e] != 0);
    const uint32_t env_g = (uint32_t)(a.env_offset + e);
    if ((flags & AUX_RESET) && sel) {
      __syncthreads();
      const int episode = state_episode(a, e) + 1;
      __syncthreads();
      for (int i = tid; i < N; i += 128) {
        real px, py, dx, dy, d2e;
        random_layout<real>(a.seed, env_g, (uint32_t)episode, (uint32_t)i, px, py, dx, dy);
        state_store_ped<real>(a, e, i, px, py, dx, dy);
        state_store_status<real>(a, e, i, status_of<real>(px, py, (real)0, (real)0, a, d2e));
      }
      if (tid == 0) state_reset_rec<real>(a, e, episode);
    }
    if ((flags & AUX_STATUS) && sel) {
      const float2 ap = state_agent_pos(a, e);
      for (int i = tid; i < N; i += 128) {
        real px, py, dx, dy, d2e;
        int st;
        state_load_ped<real>(a, e, i, px, py, dx, dy, st);
        state_store_status<real>(a, e, i, status_of<real>(px, py, (real)ap.x, (real)ap.y, a, d2e));
      }
    }
    if ((flags & AUX_OBS) && obs != nullptr) {
      __syncthreads();  // this CTA's own global writes above are visible to it after the barrier
      float2 ap = state_agent_pos(a, e);
      if ((flags & AUX_RESET) && sel) ap = make_float2(0.f, 0.f);
      float* row = obs + (size_t)e * a.obs_dim;
      if (a.positions == POS_GRAV) {
        decltype(auto) p = env_params<PE>(a, params, e);
        real gx = (real)0, gy = (real)0;
        int nf = 0;
        for (int i = tid; i < N; i += 128) {
          real px, py, dx, dy;
          int s;
          state_load_ped<real>(a, e, i, px, py, dx, dy, s);
          if (s == ST_VISCEK) { real tx, ty; grav_term<real>(px, py, ap.x, ap.y, a, p, tx, ty); gx += tx; gy += ty; }
          nf += (s == ST_FOLLOWER);
        }
        nf = __reduce_add_sync(0xffffffffu, nf);
        const double wx = warp_sum((double)gx), wy = warp_sum((double)gy);
        if (lane == 0) { red.i[warp][0] = nf; red.f[warp][0] = wx; red.f[warp][1] = wy; }
        __syncthreads();
        if (tid == 0) {
          int t = 0; double tx = 0, ty = 0;
          for (int w = 0; w < 4; ++w) { t += red.i[w][0]; tx += red.f[w][0]; ty += red.f[w][1]; }
          store_grav_obs<real>(row, ap.x, ap.y, (real)tx, (real)ty, t, a, p);
        }
      } else {
        if (tid == 0) store_head_obs<real>(row, ap.x, ap.y, a);
        for (int i = tid; i < N; i += 128) {
          real px, py, dx, dy;
          int s;
          state_load_ped<real>(a, e, i, px, py, dx, dy, s);
          store_ped_obs<real>(row, i, N, px, py, s, ap.x, ap.y, a);
        }
      }
    }
    __syncthreads();
  }
}

// get_state / set_state / get_accumulators of an EnvBlock handle (SoA handles use plain copies): one 64-thread CTA per
// environment; any array pointer may be NULL.  WRITE = set_state (API arrays -> blocks), else blocks -> API arrays.
struct StateIO {
  float2* positions;   // [E,N]
  float2* directions;  // [E,N]
  uint8_t* statuses;   // [E,N]
  float2* agent_position;
  float2* agent_direction;
  int* now;            // [E]
  double* acc;         // [E,3]   (read only)
  long long* overall;  // [E]     (read only)
};
template <bool WRITE>
__global__ void __launch_bounds__(64) evac_block_io_kernel(unsigned char* __restrict__ blocks, int E, int N, StateIO io) {
  const int e = blockIdx.x, i = threadIdx.x;
  if (e >= E) return;
  unsigned char* b = blocks + (size_t)e * BLK_BYTES;
  float4* ped = reinterpret_cast<float4*>(b + BLK_PED);
  EnvRec* rec = reinterpret_cast<EnvRec*>(b);
  if (i < N) {
    const size_t g = (size_t)e * N + i;
    if (WRITE) {
      float4 v = ped[i];
      if (io.positions) { const float2 p = io.positions[g]; v.x = p.x; v.y = p.y; }
      if (io.directions) { const float2 d = io.directions[g]; v.z = d.x; v.w = d.y; }
      if (io.positions || io.directions) ped[i] = v;
      if (io.statuses) b[blk_status_off(i)] = io.statuses[g];
    } else {
      const float4 v = ped[i];
      if (io.positions) io.positions[g] = make_float2(v.x, v.y);
      if (io.directions) io.directions[g] = make_float2(v.z, v.w);
      if (io.statuses) io.statuses[g] = b[blk_status_off(i)];
    }
  }
  if (i == 0) {
    if (WRITE) {
      if (io.agent_position) { rec->agent_pos = io.agent_position[e]; rec->agent_state = 0; }  // a moved agent restarts its script
      if (io.agent_direction) rec->agent_dir = io.agent_direction[e];
      if (io.now) rec->now = io.now[e];
    } else {
      if (io.agent_position) io.agent_position[e] = rec->agent_pos;
      if (io.agent_direction) io.agent_direction[e] = rec->agent_dir;
      if (io.now) io.now[e] = rec->now;
      if (io.acc) { io.acc[3 * (size_t)e] = rec->acc[0]; io.acc[3 * (size_t)e + 1] = rec->acc[1]; io.acc[3 * (size_t)e + 2] = rec->acc[2]; }
      if (io.overall) io.overall[e] = rec->overall;
    }
  }
}

}  // namespace evac
