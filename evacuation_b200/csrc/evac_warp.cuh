// One-warp-per-environment fused step kernel for N <= 64 pedestrians, float32 (the BASELINE headline
// shapes: 60 pedestrians).  Same semantics as evac_step_kernel (evac_kernels.cuh; reference file:line citations there and
// inline below), and the same code for the agent, rewards, episode record and reset (random_action, scripted_action,
// agent_step, step_reward, store_status_counts, record_episode, reset_pedestrian), but the pedestrian work is
// written as straight-line warp code:
//   * lane L owns pedestrians L and L + 32; every per-pedestrian quantity is kept as an (x, y) float2 so the
//     epilogue arithmetic runs on Blackwell's packed FP32 instructions (FADD2 / FMUL2 / FFMA2) exactly like the
//     pairwise pass -- one instruction per pedestrian instead of one per component;
//   * the observation encoding is a template parameter (no per-step mode branches), all loads of a step are
//     issued up front (incl. the read-modify-write words of lane 0), reductions are one REDUX + one shuffle tree;
//   * the angular noise is one Philox2x32-10 block per lane (two words = the lane's two pedestrians), no
//     shared-memory staging; no block barrier anywhere (one warp: __syncwarp only).
#pragma once
#include "evac_kernels.cuh"
#include "evac_policy_ops.cuh"

namespace evac {

enum { WMODE_GENERIC = 0, WMODE_REL_OHE_BOX = 1, WMODE_GRAV = 2 };

__device__ __forceinline__ float2 splat(float v) { return make_float2(v, v); }

// ---- Sparse neighbour pass from 2-D cell masks (N <= 64, a.cells_x > 0).
// A uniform grid of cells_x x cells_y cells (edge >= 1.0001 x vision radius, at most 32 per axis) over the area: every pair
// with d² < thr² sits in the 3 x 3 block of cells around the target, float32 rounding of the cell index included.  Per row
// and per column of the grid one 64-bit set of TILE SLOTS (.x = slots 0-31, .y = 32-63) of the moving sources in it; the
// candidates of a target in cell (r, c) are (rows r-1..r+1) & (columns c-1..c+1).  Entry 0 and entry cells + 1 of both
// arrays stay empty, so the three neighbouring entries of any cell are read without bounds tests.
constexpr int WCELLS = 32;
constexpr int WREC_PARK = 64;  // per-slot record of a parked source: what a lane with no candidate left reads

__device__ __forceinline__ uint2 or3(const uint2* m, int c) {
  const uint2 a = m[c], b = m[c + 1], d = m[c + 2];
  return make_uint2(a.x | b.x | d.x, a.y | b.y | d.y);
}

// Neighbour sums of ONE pedestrian at (x, y) over the slots of the candidate set m, walked in increasing slot order, T times
// (the warp's maximum: a lane whose set is empty reads the parked record, which fails the distance test and adds 0 * 0).
// Bit-identical to pairwise_pass<2, ..> (the all-pairs loop) when no source direction is NaN:
//   * the pair test is the same float32 expression as accumulate_pair, written with explicit round-to-nearest intrinsics so
//     that no contraction can differ from the packed form: dx = x_j + (-x), dy likewise, d² = fma(dy, dy, dx * dx) < thr²;
//   * the all-pairs loop keeps two chains per component, even slots in .x and odd slots in .y, each in increasing slot
//     order, and returns .x + .y: here the candidate goes into the chain of its slot's parity (w = 0 in the other one),
//     in increasing slot order too;
//   * the all-pairs loop also adds fma(0, u_j, acc) for every slot that fails the test, which is what the sparse walk skips.
//     That is an exact no-op: u_j is finite (no NaN source; a unit vector is finite or NaN), so 0 * u_j = ±0, and
//     acc + ±0 == acc unless acc is -0 -- which it never is: acc starts at +0, and a round-to-nearest sum is -0 only when
//     both terms are -0.  Slots outside the 3 x 3 block fail the test (the superset property above), so skipping them
//     and skipping the failing candidates both leave every chain's bits unchanged.
__device__ __forceinline__ void sparse_pass(const float4* rec, uint2 m, int T, float x, float y, float thr2, float& sx, float& sy) {
  const float nx = -x, ny = -y;
  float2 ax = make_float2(0.f, 0.f), ay = make_float2(0.f, 0.f);
  for (int t = 0; t < T; ++t) {
    // next slot, written as selects (no branch): the lowest bit of .x, else 32 + the lowest bit of .y, else the parked record
    const unsigned jy = 32u + min((unsigned)(__ffs(m.y) - 1), 32u);
    const unsigned j = m.x ? (unsigned)(__ffs(m.x) - 1) : jy;
    const unsigned y1 = m.y & (m.y - 1u);
    m.y = m.x ? m.y : y1;
    m.x &= m.x - 1u;
    const float4 r = rec[j];
    const float dx = __fadd_rn(r.x, nx), dy = __fadd_rn(r.y, ny);
    const float d2 = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));
    const float w = d2 < thr2 ? 1.f : 0.f;
    const float2 w2 = (j & 1) ? make_float2(0.f, w) : make_float2(w, 0.f);
    ax = __ffma2_rn(w2, splat(r.z), ax);
    ay = __ffma2_rn(w2, splat(r.w), ay);
  }
  sx = ax.x + ax.y;
  sy = ay.x + ay.y;
}

// Warp-maximum walk lengths against the all-pairs loop: the sparse pass is taken when
// SPARSE_COST_NUM * (T0 + T1) <= SPARSE_COST_DEN * (slot pairs of the all-pairs loop).  1 : 1 is an estimate from the SASS,
// NOT a measurement: one walk step (bit extraction, LDS.128, pair test, two FFMA2) is ~24 instructions in a two-step unrolled
// body, one slot pair of the all-pairs loop (two LDS.128, four pair evaluations) ~20; the walk step also waits on its own
// LDS.128 where the all-pairs loop loads one iteration ahead, so the true break-even may lie below 1 : 1.
constexpr int SPARSE_COST_NUM = 1, SPARSE_COST_DEN = 1;

// per-pedestrian working set of the warp kernel
struct WPed {
  float2 p, d;  // position, direction
  int st;       // status (ST_NONE for padding lanes)
};

// resident warps per SM the register allocation is sized for.  28 -> 70 registers per thread, no spills in the step loop, and
// still 29 warps per SM: the headline batch (4096 envs = 27.7 warps per SM) stays one wave.  Measured on B200 against 32
// (64 registers, 8 bytes spilled per step): 9.23 -> 8.90 us per 4096-env step, 5.11 -> 4.92 us in-rollout; 24 (76 registers,
// 26 warps per SM) pushes 4096 envs into a second wave: 9.81 us.
constexpr int WARP_MINB = 28;
constexpr int PAIR_UNROLL = 4;  // slot pairs per unrolled iteration of the pairwise loop
// ---- The linear RPO policy as the agent of the grav kernel (evac_rollout_policy): each step runs rpo_agent.py:180-203 --
// NormalizeObservation, the heads, Normal sampling, ClipAction, the step, NormalizeReward and next_done -- inside the step loop.
// The heads are the CUDA-core heads kernel's sums for K = 6 (evac_policy_heads_kernel<NORM>, the kernel K = 6 takes), in the same
// order: lane L owns hidden columns L and L + 32 of each head, the layer-1 and layer-2 outputs are exchanged through shared memory.
struct WPolArgs {
  evacp::HArgs h;      // weights (CUDA-core layout), NH, A = 2, sample, seed, offset, offset_dev, env_offset; value / action / logprob
                       // are the per-step bases [T, E, ..] (each may be NULL; value NULL skips the critic columns)
  evacp::NArgs n;      // NormalizeObservation (n.mean NULL: none); *n.count is read once per launch; n.obs_norm [T, E, 6] or NULL
  int norm_update;     // 0: the statistics are used frozen (evaluation)
  float* next_done;    // [E] in / out
  float* dones;        // [T, E]: next_done before each step (or NULL)
  float *returns, *ret_mean, *ret_var;  // NormalizeReward state [E] (returns NULL: no reward normaliser)
  const double* ret_count;
  float* reward_norm;  // [T, E] or NULL
  float gamma, ret_eps, ret_clip;
};
constexpr int WPOL_H1 = 16, WPOL_H2 = WPOL_H1 + 128, WPOL_SMEM = WPOL_H2 + 128;  // pol_sm layout (floats)
// resident warps per SM the policy instance is sized for (DESIGN.md section 7.2)
constexpr int WARP_POL_MINB = 16;

// Policy part of step s of environment e: returns the clipped action every lane applies.  sm[0..5] holds the raw observation.
// Lane k < 6 updates (or, frozen, reads) the statistics of value k; `cnt` is the normaliser's sample count before this step.
__device__ __forceinline__ float2 warp_policy_act(const WPolArgs& P, int E, int s, int e, int lane, float& mean, float& var, double cnt,
                                                  float done, float* sm) {
  const size_t se = (size_t)s * E + e;
  if (lane == 0 && P.dones != nullptr) P.dones[se] = done;
  // ---- NormalizeObservation + clip (op for op the heads kernel's NORM load)
  const float x = lane < 6 ? sm[lane] : 0.f;
  float z = x;
  if (P.n.mean != nullptr) {
    if (P.norm_update) {
      evacp::NArgs n = P.n;
      n.count = &cnt;
      z = evacp::norm_update(x, mean, var, evacp::norm_weights(n), n);
    } else {
      z = evacp::min_nan(evacp::max_nan(__fmul_rn(__fsub_rn(x, mean), rsqrtf(__fadd_rn(var, P.n.eps))), -P.n.clip), P.n.clip);
    }
  }
  if (lane < 6) {
    sm[8 + lane] = z;
    if (P.n.obs_norm != nullptr) P.n.obs_norm[se * 6 + lane] = z;
  }
  __syncwarp();
  const evacp::HArgs& h = P.h;
  const bool critic = h.value != nullptr;
  const float4 x03 = *reinterpret_cast<const float4*>(sm + 8);
  const float2 x45 = *reinterpret_cast<const float2*>(sm + 12);
  // ---- layer 1, column o = 32 j + lane (j = 0, 1 critic, 2, 3 actor).  The heads kernel sums four split-K chains over k = 4g .. 4g + 3
  // of the 16-wide chunk: chain 0 from b1 over k = 0..3, chain 1 from +0 over k = 4..7, chains 2 and 3 from +0 over k >= 8.  Every
  // term with k >= 6 is fma(+0, +0, acc) (the observation is zero-filled, the weight rows are zero padding) = acc + 0.f, and chains 2
  // and 3 are exactly +0, so they are written as the additions of +0 they are (acc + 0.f is not acc when acc is -0).
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (j < 2 && !critic) continue;
    const int o = 32 * j + lane;
    const float* w = h.w1t + o;
    float g0 = h.b1[o];
    g0 = fmaf(x03.x, w[0], g0); g0 = fmaf(x03.y, w[128], g0); g0 = fmaf(x03.z, w[256], g0); g0 = fmaf(x03.w, w[384], g0);
    float g1 = fmaf(x45.x, w[512], 0.f);
    g1 = fmaf(x45.y, w[640], g1);
    g1 = __fadd_rn(__fadd_rn(g1, 0.f), 0.f);                                   // k = 6, 7
    sm[WPOL_H1 + o] = tanhf(__fadd_rn(__fadd_rn(__fadd_rn(g0, g1), 0.f), 0.f));  // + chain 2 + chain 3
  }
  __syncwarp();
  // ---- layer 2: four chains over k in [16 g, 16 g + 16), chain 0 from b2, summed in order (the heads kernel's split-K groups)
  float c[4][4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int g = 0; g < 4; ++g) c[j][g] = (g == 0 && (j >= 2 || critic)) ? h.b2[32 * j + lane] : 0.f;
  const float* hc = sm + WPOL_H1;
  const float* ha = sm + WPOL_H1 + 64;
#pragma unroll 1
  for (int kk = 0; kk < 16; kk += 4) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int k = 16 * g + kk;
      const float4 va = *reinterpret_cast<const float4*>(ha + k);
      const float av[4] = {va.x, va.y, va.z, va.w};
      const float* wr = h.w2t + (size_t)k * 128 + lane;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        c[2][g] = fmaf(av[q], wr[q * 128 + 64], c[2][g]);
        c[3][g] = fmaf(av[q], wr[q * 128 + 96], c[3][g]);
      }
      if (critic) {
        const float4 vc = *reinterpret_cast<const float4*>(hc + k);
        const float cv[4] = {vc.x, vc.y, vc.z, vc.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          c[0][g] = fmaf(cv[q], wr[q * 128], c[0][g]);
          c[1][g] = fmaf(cv[q], wr[q * 128 + 32], c[1][g]);
        }
      }
    }
  }
  __syncwarp();  // h1 is read by every lane before h2 (its neighbour in sm) is written
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (j >= 2 || critic) sm[WPOL_H2 + 32 * j + lane] = tanhf(((c[j][0] + c[j][1]) + c[j][2]) + c[j][3]);
  __syncwarp();
  // ---- layer 3: row r = lane (0 value, 1..2 the action mean), one chain from b3[r] over k < NH
  float o3 = 0.f;
  if (lane < 3 && (lane > 0 || critic)) {
    const float* hp = sm + WPOL_H2 + (lane == 0 ? 0 : 64);
    const float* w = h.w3 + lane * 64;
    o3 = h.b3[lane];
    for (int k = 0; k < h.NH; ++k) o3 = fmaf(hp[k], w[k], o3);
  }
  const float m0 = __shfl_sync(0xffffffffu, o3, 1), m1 = __shfl_sync(0xffffffffu, o3, 2);
  // ---- Normal(mean, exp(logstd)) sample, log-probability, ClipAction: heads_finish of environment e, with the step's stream offset
  if (lane == 0) {
    evacp::HArgs f = h;
    f.A = 2;
    f.given_action = nullptr; f.mean = nullptr; f.entropy = nullptr;
    f.value = h.value ? h.value + se : nullptr;
    f.action = h.action ? h.action + se * 2 : nullptr;
    f.logprob = h.logprob ? h.logprob + se : nullptr;
    f.action_clipped = sm + 14;
    f.offset = h.offset + (unsigned long long)s;
    f.env_offset = h.env_offset + e;
    const float o[4] = {o3, m0, m1, 0.f};
    evacp::heads_finish(f, 0, o, true, true);
  }
  __syncwarp();
  return make_float2(sm[14], sm[15]);
}

// NormalizeReward + clip and next_done of one step (lane 0), op for op evac_normalize_reward_kernel on what evac_step writes: the
// reward 0.f + reward (its one-step sum), terminated and truncated.  Returns next_done.
__device__ __forceinline__ float warp_policy_reward(const WPolArgs& P, size_t se, float reward, bool terminated, bool truncated, float& ret,
                                                   float& mean, float& var, double cnt) {
  if (P.returns != nullptr) {
    evacp::NArgs n{};
    n.count = &cnt;
    const evacp::NormWeights w = evacp::norm_weights(n);  // the same weights the reward kernel forms from *count
    const float r = __fadd_rn(0.f, reward);
    const float keep = terminated ? 0.f : 1.f;
    ret = __fadd_rn(__fmul_rn(ret, __fmul_rn(P.gamma, keep)), r);
    const float delta = __fsub_rn(ret, mean);
    mean = __fadd_rn(mean, __fmul_rn(delta, w.w_new));
    var = __fadd_rn(__fmul_rn(var, w.w_old), __fmul_rn(__fmul_rn(delta, delta), w.w_mix));
    const float z = __fmul_rn(r, rsqrtf(__fadd_rn(var, P.ret_eps)));
    if (P.reward_norm != nullptr) P.reward_norm[se] = evacp::min_nan(evacp::max_nan(z, -P.ret_clip), P.ret_clip);
  }
  return (terminated || truncated) ? 1.f : 0.f;
}
// The step loop of one environment (one warp).  PE: per-environment parameters (the environment's EnvParamRec, loaded with the
// state; env_params).  POL: the action of every step comes from the linear policy (warp_policy_act, evac_rollout_policy).
template <int MODE, bool PE, bool POL>
__device__ __forceinline__ void warp_env_loop(const KArgs<float>& a, const EnvParamRec<float>* __restrict__ params,
                                              const WPolArgs* pol, const int lane) {  // @region wload
  // Tile<float> of 64 slots (+ the look-ahead entries) = 66 float4
  __shared__ __align__(16) float4 tile_smem[66];
  // sparse pass (a.cells_x > 0): {x, y, ux, uy} of every slot (+ the parked record) and the row / column slot masks
  __shared__ float4 rec[WREC_PARK + 1];
  __shared__ uint2 row_mask[WCELLS + 2], col_mask[WCELLS + 2];
  // POL: [raw observation (6) + 2 | normalised observation (6) + clipped action (2) | h1 (128) | h2 (128)]
  __shared__ __align__(16) float pol_sm[POL ? WPOL_SMEM : 1];
  const int e = blockIdx.x, N = a.N;
  if (e >= a.E) return;
  const Tile<float> tile(reinterpret_cast<unsigned char*>(tile_smem), 64);
  const bool cells = a.cells_x > 0;
  if (lane == 0) rec[WREC_PARK] = make_float4(PARK, PARK, 0.f, 0.f);
  const uint32_t lt_mask = (1u << lane) - 1u;
  const bool valid[2] = {lane < N, lane + 32 < N};
  const uint32_t env_g = (uint32_t)(a.env_offset + e);
  const float2 exit_p = make_float2(0.f, -1.f);  // area.py:36-39

  // ---------------- load state: everything this launch reads is requested before anything is used.  One address per
  // environment (EnvBlock, evac_kernels.cuh): the record as two broadcast LDG.128, one LDG.128 per pedestrian
  // ({px, py, dx, dy}), one LDG.U16 for the lane's two statuses; slots >= N hold zeros / status 0 and are never valid.
  unsigned char* const blk = a.blocks + (size_t)e * BLK_BYTES;
  float4* const ped_l = reinterpret_cast<float4*>(blk + BLK_PED) + lane;
  unsigned short* const st_l = reinterpret_cast<unsigned short*>(blk + BLK_STATUS) + lane;
  const float4 pd0 = ped_l[0], pd1 = ped_l[32];
  const unsigned st2 = *st_l;
  const float4 rec0 = *reinterpret_cast<const float4*>(blk);      // agent_pos, agent_dir
  const int4 rec1 = *reinterpret_cast<const int4*>(blk + 16);     // now, episode, agent_state
  // overall_timesteps (all lanes: the RotatingAgent's call counter) and, lane 0, the episode accumulators of env.py:168-170
  const longlong2 rec2 = *reinterpret_cast<const longlong2*>(blk + 32);
  long long overall = rec2.x;
  double acc_r = __longlong_as_double(rec2.y), acc_i = 0, acc_s = 0;
  if (lane == 0) {
    const double2 r3 = *reinterpret_cast<const double2*>(blk + 48);
    acc_i = r3.x; acc_s = r3.y;
  }
  WPed q[2];
  q[0].p = make_float2(pd0.x, pd0.y); q[0].d = make_float2(pd0.z, pd0.w); q[0].st = (int)(st2 & 0xffu);
  q[1].p = make_float2(pd1.x, pd1.y); q[1].d = make_float2(pd1.z, pd1.w); q[1].st = (int)(st2 >> 8);
  float2 ap = make_float2(rec0.x, rec0.y), ad = make_float2(rec0.z, rec0.w);
  int now = rec1.x, episode = rec1.y, wac_state = rec1.z;
  float reward_sum = 0.f;
  int any_term = 0, any_trunc = 0;
  decltype(auto) p = env_params<PE>(a, params, e);
  const float noise_c = p.noise_coef;
  const float* noise_e = a.noise ? a.noise + (size_t)e * N : nullptr;
  float* obs_e = a.obs ? a.obs + (size_t)e * a.obs_dim : nullptr;
  const float2 wall = make_float2(a.width, a.height);
  // POL: lane k < 6 keeps the running mean / variance of observation value k, lane 0 next_done and the NormalizeReward state
  [[maybe_unused]] float o_mean = 0.f, o_var = 0.f, done = 0.f, ret = 0.f, r_mean = 0.f, r_var = 0.f;
  [[maybe_unused]] double o_cnt = 0.0, r_cnt = 0.0;
  if constexpr (POL) {
    if (lane < 6) {
      pol_sm[lane] = obs_e[lane];
      if (pol->n.mean != nullptr) { o_mean = pol->n.mean[(size_t)e * 6 + lane]; o_var = pol->n.var[(size_t)e * 6 + lane]; }
    }
    if (pol->n.mean != nullptr) o_cnt = *pol->n.count;
    if (lane == 0) {
      done = pol->next_done[e];
      if (pol->returns != nullptr) { ret = pol->returns[e]; r_mean = pol->ret_mean[e]; r_var = pol->ret_var[e]; r_cnt = *pol->ret_count; }
    }
    __syncwarp();
  }

  for (int s = 0; s < a.num_steps; ++s) {  // @region wrng
    // ---------------- Time.step [area.py:53-59]
    const int now_prev = now;
    now += 1;
    const bool truncated = now >= p.max_timesteps;
    // the action is requested first so that its (cold) latency overlaps the preparation below
    float2 act_tbl = make_float2(0.f, 0.f);
    if constexpr (POL) act_tbl = warp_policy_act(*pol, a.E, s, e, lane, o_mean, o_var, o_cnt, done, pol_sm);
    else if (a.agent_kind == AGENT_TABLE) act_tbl = a.actions[(size_t)s * a.E + e];
    // ---------------- angular noise of this lane's two pedestrians [area.py:124]
    float nz[2];
    if (noise_e != nullptr) {
      const float* np_ = noise_e + (size_t)s * a.E * N;
      nz[0] = valid[0] ? np_[lane] : 0.f;
      nz[1] = valid[1] ? np_[lane + 32] : 0.f;
    } else {
      const uint2 r = evac_noise_block(a.seed, env_g, (uint32_t)episode, (uint32_t)now_prev, (uint32_t)lane);
      nz[0] = (u01(r.x) - 0.5f) * noise_c;
      nz[1] = (u01(r.y) - 0.5f) * noise_c;
    }
    // ---------------- escaped / exiting preparation + unit directions [area.py:79-101]  // @region wprep
    float2 u[2];
    bool efv[2], fv[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int so = q[k].st;
      if (so == ST_ESCAPED) { q[k].d = make_float2(0.f, 0.f); q[k].p = exit_p; }
      float2 v = q[k].d;
      if (so == ST_EXITING) v = __fadd2_rn(exit_p, make_float2(-q[k].p.x, -q[k].p.y));
      efv[k] = (unsigned)(so - ST_VISCEK) <= (unsigned)(ST_EXITING - ST_VISCEK);
      fv[k] = (unsigned)(so - ST_VISCEK) <= (unsigned)(ST_FOLLOWER - ST_VISCEK);
      // u = v / |v|; a zero direction gives NaN exactly like area.py:101
      const float2 sq = __fmul2_rn(v, v);
      const float n2 = sq.x + sq.y;
      const float inv = inv_norm(n2);
      u[k] = __fmul2_rn(v, splat(inv));
      if (so == ST_EXITING) q[k].d = __fmul2_rn(v, splat(fminf(n2 * inv, a.step_size) * inv));  // dir = u * min(|v|, step)
    }
    // ---------------- compact the moving pedestrians into the shared tile  // @region wcompact
    const uint32_t m0 = __ballot_sync(0xffffffffu, efv[0]), m1 = __ballot_sync(0xffffffffu, efv[1]);
    const int c0 = __popc(m0), slot[2] = {__popc(m0 & lt_mask), c0 + __popc(m1 & lt_mask)};
    const int n_src = c0 + __popc(m1);
#pragma unroll
    for (int k = 0; k < 2; ++k)
      if (efv[k]) tile.put(slot[k], q[k].p.x, q[k].p.y, u[k].x, u[k].y);
    if (lane < 2) tile.put(n_src + lane, PARK, PARK, 0.f, 0.f);  // pad to an even count
    // sparse pass: per-slot records and the row / column slot masks (atomicOr of slot bits: commutative, so the masks do
    // not depend on the order the atomics retire).  A source without a direction (NaN) poisons every sum in the reference
    // (0 * NaN in the all-pairs product), which only the all-pairs loop reproduces.  Each moving source is stored twice, in
    // the pair-packed tile above and in its per-slot record below, because which pass runs is known only after the masks
    // are built; a single layout serving both passes was not built or measured.
    bool sparse = false;
    uint2 cand[2] = {make_uint2(0u, 0u), make_uint2(0u, 0u)};
    int T[2] = {0, 0};
    if (cells) {
      row_mask[lane] = col_mask[lane] = make_uint2(0u, 0u);
      if (lane < 2) row_mask[WCELLS + lane] = col_mask[WCELLS + lane] = make_uint2(0u, 0u);
      int cx[2], cy[2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {  // entry 1 + cell index; (int)NaN == 0
        cx[k] = 1 + min(max((int)((q[k].p.x + a.width_f) * a.cell_inv_x), 0), a.cells_x - 1);
        cy[k] = 1 + min(max((int)((q[k].p.y + a.height_f) * a.cell_inv_y), 0), a.cells_y - 1);
        if (efv[k]) rec[slot[k]] = make_float4(q[k].p.x, q[k].p.y, u[k].x, u[k].y);
      }
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (efv[k]) {
          unsigned* r = slot[k] < 32 ? &row_mask[cy[k]].x : &row_mask[cy[k]].y;
          unsigned* c = slot[k] < 32 ? &col_mask[cx[k]].x : &col_mask[cx[k]].y;
          atomicOr(r, 1u << (slot[k] & 31));
          atomicOr(c, 1u << (slot[k] & 31));
        }
      }
      __syncwarp();
      int walk[2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (fv[k]) {
          const uint2 rm = or3(row_mask, cy[k] - 1), cm = or3(col_mask, cx[k] - 1);
          cand[k] = make_uint2(rm.x & cm.x, rm.y & cm.y);
        }
        walk[k] = __popc(cand[k].x) + __popc(cand[k].y);
      }
      T[0] = __reduce_max_sync(0xffffffffu, walk[0]);
      T[1] = __reduce_max_sync(0xffffffffu, walk[1]);
      const bool nan_src = (efv[0] && (u[0].x != u[0].x || u[0].y != u[0].y)) || (efv[1] && (u[1].x != u[1].x || u[1].y != u[1].y));
      sparse = !__any_sync(0xffffffffu, nan_src) &&
               (a.cell_force || SPARSE_COST_NUM * (T[0] + T[1]) <= SPARSE_COST_DEN * ((n_src + 1) >> 1));
    }
    __syncwarp();
    // ---------------- action source + Area.agent_step [area.py:182-210]  // @region wagent
    float2 act;
    if (POL || a.agent_kind == AGENT_TABLE) act = act_tbl;
    else if (a.agent_kind == AGENT_RANDOM) act = random_action(a.seed, env_g, (uint32_t)episode, (uint32_t)now_prev);
    else act = scripted_action(a, overall + 1, ap, wac_state);
    float r_agent; bool term_agent;
    agent_step(a, p, act, ap, ad, r_agent, term_agent);
    // ---------------- pairwise alignment [area.py:105-119]  // @region wpairwise
    float sx[2], sy[2];
    if (sparse) {
#pragma unroll
      for (int k = 0; k < 2; ++k) sparse_pass(rec, cand[k], T[k], q[k].p.x, q[k].p.y, a.thr2_ped, sx[k], sy[k]);
    } else {
      const float xi[2] = {q[0].p.x, q[1].p.x}, yi[2] = {q[0].p.y, q[1].p.y};
      if (__any_sync(0xffffffffu, fv[0] | fv[1])) pairwise_pass<2, PAIR_UNROLL>(tile, n_src, xi, yi, a.thr2_ped, sx, sy);
      else sx[0] = sx[1] = sy[0] = sy[1] = 0.f;
    }
    // ---------------- new headings, enslaving, integration, reflection, statuses  // @region wupdate
    const float2 e_ad = make_float2(__fmul_rn(p.enslaving_f, ad.x), __fmul_rn(p.enslaving_f, ad.y));  // float32 like area.py:140
    int counts = 0;  // k_exit | k_fol << 8 | n_esc << 16 | n_exi << 24   (each <= 64)
    float sum_dexit = 0.f;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int so = q[k].st;
      if (fv[k]) {
        // cos/sin(atan2(my, mx) + nz) == unit(m) rotated by nz; atan2(0, 0) = 0 -> unit = (1, 0)  [area.py:120-136]
        const float m2 = fmaf(sx[k], sx[k], sy[k] * sy[k]);
        float2 c = make_float2(1.f, 0.f);
        if (m2 != 0.f) c = __fmul2_rn(make_float2(sx[k], sy[k]), splat(inv_norm(m2)));
        float sn, cn;
        sincos_noise(nz[k], sn, cn);
        float2 nd = __fmul2_rn(splat(c.x), make_float2(cn, sn));
        nd = __ffma2_rn(make_float2(-c.y, c.y), make_float2(sn, cn), nd);
        nd = __fmul2_rn(nd, splat(a.step_size));
        if (so == ST_FOLLOWER) nd = __ffma2_rn(splat(p.one_minus_enslaving), nd, e_ad);  // area.py:138-142
        q[k].d = nd;
      }
      if (efv[k]) q[k].p = __fadd2_rn(q[k].p, q[k].d);
      {  // wall reflection for ALL pedestrians [area.py:147-152]
        const float2 cl = make_float2(fminf(fmaxf(q[k].p.x, -wall.x), wall.x), fminf(fmaxf(q[k].p.y, -wall.y), wall.y));
        const float2 miss = __fadd2_rn(q[k].p, make_float2(-cl.x, -cl.y));
        q[k].p = __ffma2_rn(splat(-2.f), miss, q[k].p);
        if (miss.x != 0.f) q[k].d.x = -q[k].d.x;
        if (miss.y != 0.f) q[k].d.y = -q[k].d.y;
      }
      // statuses: a pure function of (position, agent position) [statuses.py:29-48]
      const float2 da = __fadd2_rn(make_float2(ap.x, ap.y), make_float2(-q[k].p.x, -q[k].p.y));
      const float2 de = __fadd2_rn(exit_p, make_float2(-q[k].p.x, -q[k].p.y));
      const float da2 = fmaf(da.x, da.x, da.y * da.y), de2 = fmaf(de.x, de.x, de.y * de.y);
      int sn_ = ST_VISCEK;
      if (da2 < a.thr2_leader) sn_ = ST_FOLLOWER;
      if (de2 < a.thr2_exit) sn_ = ST_EXITING;
      if (de2 < a.thr2_escape) sn_ = ST_ESCAPED;
      if (valid[k]) {
        sum_dexit += sqrt_fast(de2);
        counts += (int)(fv[k] && sn_ == ST_EXITING) + ((int)(so == ST_VISCEK && sn_ == ST_FOLLOWER) << 8) +
                  ((int)(sn_ == ST_ESCAPED) << 16) + ((int)(sn_ == ST_EXITING) << 24);
        q[k].st = sn_;
      }
    }
    // ---------------- warp reduction, rewards, termination [reward.py:19-46, area.py:174-180, env.py:158-171]  // @region wreward
    counts = __reduce_add_sync(0xffffffffu, counts);
    const float sd = warp_sum(sum_dexit);
    const int K_exit = counts & 0xff, K_fol = (counts >> 8) & 0xff, N_esc = (counts >> 16) & 0xff, N_exi = (counts >> 24) & 0xff;
    if (a.status_counts != nullptr) {
      const int n_fol = __popc(__ballot_sync(0xffffffffu, q[0].st == ST_FOLLOWER)) + __popc(__ballot_sync(0xffffffffu, q[1].st == ST_FOLLOWER));
      if (lane == 0) store_status_counts(a, s, e, N, N_esc, N_exi, n_fol);
    }
    float intrinsic, r_status, reward; bool terminated;
    step_reward(a, p, N, now, sd, K_exit, K_fol, N_esc, r_agent, term_agent, intrinsic, r_status, reward, terminated);
    reward_sum += reward;
    any_term |= terminated; any_trunc |= truncated;
    acc_r += (double)reward; acc_i += (double)intrinsic; acc_s += (double)r_status;
    overall += 1;
    if constexpr (POL) {
      if (lane == 0) done = warp_policy_reward(*pol, (size_t)s * a.E + e, reward, terminated, truncated, ret, r_mean, r_var, r_cnt);
      o_cnt += 1.0; r_cnt += 1.0;  // the caller's per-step `count += 1.0`, in the same order
    }
    // ---------------- same-step auto-reset (gymnasium vector-env semantics)  // @region wreset
    if (a.auto_reset && (terminated || truncated)) {
      const int N_fol = __popc(__ballot_sync(0xffffffffu, q[0].st == ST_FOLLOWER)) + __popc(__ballot_sync(0xffffffffu, q[1].st == ST_FOLLOWER));
      if (lane == 0) record_episode(a, e, acc_i, acc_s, acc_r, now, N, N_esc, N_exi, N_fol, overall);
      acc_r = acc_i = acc_s = 0;
      now = 0; episode += 1; wac_state = 0;
      ap = make_float2(0.f, 0.f); ad = make_float2(0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 2; ++k)
        if (valid[k]) q[k].st = reset_pedestrian<float>(a, env_g, (uint32_t)episode, (uint32_t)(lane + 32 * k), q[k].p.x, q[k].p.y, q[k].d.x, q[k].d.y);
    }
    // ---------------- observation [wrappers.py:8-96, gravity_encoding.py:8-81]  // @region wobs
    if (obs_e != nullptr && (a.obs_every_step || s == a.num_steps - 1 || POL)) {
      float* row = obs_e + (a.obs_every_step ? (size_t)s * a.E * a.obs_dim : (size_t)0);
      if constexpr (POL) row = pol_sm;  // the next step's policy reads the 6 values from shared memory; obs gets the last step's
      if constexpr (MODE == WMODE_REL_OHE_BOX) {
        // rows = [agent; exit; pedestrians], cols = [x, y, ohe(4)]; relative positions / sqrt(2) (float32 hypotenuse).
        // Three float2 stores per pedestrian straight from registers (24-byte row stride: a warp's STG.64 touches 24 sectors for
        // 256 useful bytes, the sectors are completed in L2 by the neighbouring lanes' stores).  Measured on B200, same box,
        // 4096 x 60 per-step regime, against a row staged in shared memory and copied out with one 16-byte store per lane and
        // round: the load -> observe -> write-back skeleton gets faster (5.23 -> 4.82 us) but the FULL step slower (8.42 ->
        // 8.66 us: STS -> LDS -> STG adds a dependent shared-memory round trip to every warp's tail); the staged row sent as ONE
        // cp.async.bulk by lane 0: 8.76 vs 8.52 us -- also slower, so the direct stores stay.
        const float inv_hyp = (float)(1.0 / 1.41421353816986083984375);
        const float2 nap = make_float2(-ap.x, -ap.y);
        if (lane == 0) {
          const float2 ex = __fmul2_rn(__fadd2_rn(exit_p, nap), splat(inv_hyp));
          float2* r = reinterpret_cast<float2*>(row);
          r[0] = ap; r[1] = make_float2(0.f, 0.f); r[2] = make_float2(0.f, 0.f);
          r[3] = ex; r[4] = make_float2(1.f, 0.f); r[5] = make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          if (valid[k]) {
            float2* r = reinterpret_cast<float2*>(row + (lane + 32 * k + 2) * 6);
            const int st = q[k].st;
            r[0] = __fmul2_rn(__fadd2_rn(q[k].p, nap), splat(inv_hyp));
            r[1] = make_float2(st == ST_ESCAPED ? 1.f : 0.f, st == ST_EXITING ? 1.f : 0.f);
            r[2] = make_float2(st == ST_FOLLOWER ? 1.f : 0.f, st == ST_VISCEK ? 1.f : 0.f);
          }
        }
      } else if (MODE == WMODE_GRAV || a.positions == POS_GRAV) {
        // gravity encoding [gravity_encoding.py:8-38]: per VISCEK pedestrian -alpha / (|R| + eps)^(alpha + 2) * R, R = agent - p.
        // Straight-line and unconditional for both pedestrians of the lane (select, not branch); MUFU square root and
        // reciprocal (~2 ulp each against the parity bar of 2e-5 of the largest term); the two sums over the warp in double.
        float gx = 0.f, gy = 0.f;
        int nf = 0;
        const float alpha = (float)p.alpha, eps = (float)a.eps;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float2 R = __fadd2_rn(ap, make_float2(-q[k].p.x, -q[k].p.y));
          const float norm = sqrt_fast(fmaf(R.x, R.x, R.y * R.y)) + eps;
          const float n2 = norm * norm;
          float pw;
          switch (p.alpha_plus2_int) {  // alpha = 2 .. 5 (BASELINE config 3) without a loop
            case 4: pw = n2 * n2; break;
            case 5: pw = n2 * n2 * norm; break;
            case 6: pw = n2 * n2 * n2; break;
            case 7: pw = n2 * n2 * n2 * norm; break;
            default: pw = p.alpha_plus2_int ? ipow(norm, p.alpha_plus2_int) : powf(norm, alpha + 2.f);
          }
          const float c = __fdividef(-alpha, pw);
          const bool vk = q[k].st == ST_VISCEK;
          gx += vk ? c * R.x : 0.f;
          gy += vk ? c * R.y : 0.f;
          nf += (q[k].st == ST_FOLLOWER);
        }
        nf = __reduce_add_sync(0xffffffffu, nf);
        const double wx = warp_sum((double)gx), wy = warp_sum((double)gy);
        if (lane == 0) store_grav_obs<float>(row, ap.x, ap.y, (float)wx, (float)wy, nf, a, p);
      } else {
        if (lane == 0) store_head_obs<float>(row, ap.x, ap.y, a);
#pragma unroll
        for (int k = 0; k < 2; ++k)
          if (valid[k]) store_ped_obs<float>(row, lane + 32 * k, N, q[k].p.x, q[k].p.y, q[k].st, ap.x, ap.y, a);
      }
    }
    __syncwarp();  // the tile is rewritten by the next step
  }  // steps

  // ---------------- write back  // @region wwriteback
  ped_l[0] = make_float4(q[0].p.x, q[0].p.y, q[0].d.x, q[0].d.y);
  ped_l[32] = make_float4(q[1].p.x, q[1].p.y, q[1].d.x, q[1].d.y);
  *st_l = (unsigned short)(q[0].st | (q[1].st << 8));
  if (a.status_out != nullptr) {  // host face: dense [E,N] statuses travel in the result block
    uint8_t* so = a.status_out + (size_t)e * N + lane;
    if (valid[0]) so[0] = (uint8_t)q[0].st;
    if (valid[1]) so[32] = (uint8_t)q[1].st;
  }
  if (lane == 0) {
    *reinterpret_cast<float4*>(blk) = make_float4(ap.x, ap.y, ad.x, ad.y);
    *reinterpret_cast<int4*>(blk + 16) = make_int4(now, episode, wac_state, 0);
    *reinterpret_cast<longlong2*>(blk + 32) = make_longlong2(overall, __double_as_longlong(acc_r));
    *reinterpret_cast<double2*>(blk + 48) = make_double2(acc_i, acc_s);
    if (a.reward) a.reward[e] = reward_sum;
    if (a.terminated) a.terminated[e] = (uint8_t)any_term;
    if (a.truncated) a.truncated[e] = (uint8_t)any_trunc;
  }
  if constexpr (POL) {
    if (lane < 6) {
      obs_e[lane] = pol_sm[lane];
      if (pol->n.mean != nullptr && pol->norm_update) { pol->n.mean[(size_t)e * 6 + lane] = o_mean; pol->n.var[(size_t)e * 6 + lane] = o_var; }
    }
    if (lane == 0) {
      pol->next_done[e] = done;
      if (pol->returns != nullptr) { pol->returns[e] = ret; pol->ret_mean[e] = r_mean; pol->ret_var[e] = r_var; }
    }
  }
}

// One environment per one-warp CTA (launch_warp in evac_abi.cu); no block-level barrier anywhere.
template <int MODE, bool PE = false>
__global__ void __launch_bounds__(32, WARP_MINB) evac_warp_kernel(const __grid_constant__ KArgs<float> a,
                                                                  const EnvParamRec<float>* __restrict__ params) {
  // lane is read here: the kernel's launch bounds (32 threads) make threadIdx.x & 31 free only at the kernel's own level
  warp_env_loop<MODE, PE, false>(a, params, nullptr, threadIdx.x & 31);
}

// evac_rollout_policy: the gravity-encoding step loop with the linear policy as its agent (DESIGN.md section 7.2).
template <bool PE>
__global__ void __launch_bounds__(32, WARP_POL_MINB) evac_warp_policy_kernel(const __grid_constant__ KArgs<float> a,
                                                                             const EnvParamRec<float>* __restrict__ params,
                                                                             const __grid_constant__ WPolArgs pol) {
  warp_env_loop<WMODE_GRAV, PE, true>(a, params, &pol, threadIdx.x & 31);
}

// The counters the caller advances once per step (NormalizeObservation's and NormalizeReward's sample counts, the policy's stream
// offset), advanced by n steps AFTER the step kernel: every CTA of that kernel reads them at its start.  Sequential += 1.0, so the
// counts equal what n per-step `count += 1.0` give (1e-4 + n is not always that).
__global__ void evac_policy_counters_kernel(double* obs_count, double* ret_count, unsigned long long* offset, int n) {
  if (obs_count != nullptr) { double c = *obs_count; for (int i = 0; i < n; ++i) c += 1.0; *obs_count = c; }
  if (ret_count != nullptr) { double c = *ret_count; for (int i = 0; i < n; ++i) c += 1.0; *ret_count = c; }
  if (offset != nullptr) *offset += (unsigned long long)n;
}

}  // namespace evac
