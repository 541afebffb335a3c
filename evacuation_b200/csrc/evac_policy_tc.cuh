// The policy heads (critic | actor MLPs, Normal sampling) on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a only.
//
//   H1[E, 128] = tanh( X[E, K] * W1[K, 128] + b1 )        X = transformer embedding (K = S * D = 372 at the reference shape),
//   H2 = tanh( H1 * W2 + b2 ) per head (64 x 64)          W1 = [critic.0.weight^T | actor_mean.0.weight^T]
//   value / mean = H2 * W3 + b3, Normal(mean, exp(logstd)) sample / log-probability / entropy
//   [src/agents/networks/rpo_linear_agent_network.py:23-61 -- layer 1 is the one large dense contraction on the rollout path]
//
// One CTA = 128 environments x NT hidden columns: NT = 128 (both heads) for large batches, NT = 64 (blockIdx.y = 0: critic,
// 1: actor -- the heads share nothing after the embedding) for batches that would otherwise leave SMs idle.
//
// Layer 1: K in chunks of 32 (one 128-byte swizzle row of float32).  float32 fidelity from kind::tf32 MMAs (10-bit mantissa
// operands) by the 3xTF32 split:  x = xh + xl, w = wh + wl (xh / wh = the 10-mantissa-bit part, xl / wl = the float32
// remainder, of which the tensor core keeps the top 10 bits):
//   x w  ~=  xh wh + xl wh + xh wl          (error ~2^-21 per product; the xl wl term is below float32 resolution)
// accumulated in float32 in tensor memory.  Per chunk and CTA: 4 k-steps (UMMA_K = 8) x 2 = 8 tcgen05.mma -- xh x [wh | wl]
// (N = 2 NT: the hi and lo weight tiles are one B tile) and xl x wh (N = NT), M = 128 -- issued by ONE elected lane of a dedicated warp; operands in shared memory in the canonical K-major
// SWIZZLE_128B layout (8-row x 128-byte atoms, 16-byte chunk index XOR row-in-atom).  X arrives by cp.async straight into
// the swizzled hi tile, two chunks ahead (kind::tf32 ignores the low mantissa bits itself, so the raw value is xh), the eight
// producer warps only add the lo tile; the weight tiles are split and swizzled once on the host (evac_policy_load_weights)
// and arrive as ONE bulk copy per chunk (cp.async.bulk + mbarrier complete_tx).  Ring of STAGES stages: full[s] (256
// producer arrivals + the bulk copy's bytes) / empty[s] (tcgen05.commit).
//
// Layer 2 stays on chip: epilogue 1 (tcgen05.ld 32x32b: warp w reads TMEM lanes 32 (w % 4) .. = environments and column half
// w / 4; + bias, tanh) writes H1 -- split into hi / lo again -- as the A operand tiles of the second product into the drained
// ring, the layer-2 weight tiles (32 KB per head) arrive by one more bulk copy, 24 MMAs (N = 64) per head accumulate into
// further TMEM columns.  Epilogue 2: + bias, tanh, the (1 + A) x 64 output layer as per-thread dot products straight from the
// TMEM loads (column halves combined through shared memory), then the sampling tail shared with the CUDA-core kernel
// (heads_finish).  H1 / H2 never touch global memory.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

namespace evacp {

constexpr int TC_M = 128, TC_KC = 32;
constexpr int TC_COLS = 128;                                 // = HD_COLS
constexpr int TC_EW = 8;                                     // producer / epilogue warps: two per TMEM lane quarter (= two per scheduler)
constexpr int TC_ET = 32 * TC_EW;                            // ... threads
constexpr int TC_THREADS = TC_ET + 32;                       // + warp TC_EW: MMA issue + TMEM allocation
constexpr int TC_XTILE_BYTES = TC_M * TC_KC * 4;             // 16 KB: one A tile (128 rows x 128 bytes)
constexpr int TC_W2_HEAD_BYTES = 2 * 2 * HD_HS * TC_KC * 4;  // layer-2 weights of one head: 2 k-chunks x (hi | lo) x 64 rows x 128 bytes
// NT = hidden columns per CTA, ST = ring stages, AH = chunks of X in flight ahead of the one being finished (< ST)
template <int NT, int ST, int AH> struct TCShape {
  static constexpr int WTILE_BYTES = NT * TC_KC * 4;         // one W1 tile (NT rows x 128 bytes)
  static constexpr int STAGE_BYTES = 2 * TC_XTILE_BYTES + 2 * WTILE_BYTES;   // X hi | X lo | W hi | W lo
  static constexpr int STAGES = ST, AHEAD = AH;
  static_assert(AH >= 1 && AH < ST, "look-ahead must leave the stage being consumed alone");
  static constexpr int HEADS = NT / HD_HS;                   // heads handled by one CTA
  static constexpr int A2_BYTES = (NT / TC_KC) * 2 * TC_XTILE_BYTES;         // H1 as A operand: NT / 32 k-chunks x (hi | lo)
  static constexpr int W2_BYTES = HEADS * TC_W2_HEAD_BYTES;
  static_assert(A2_BYTES + W2_BYTES <= STAGES * STAGE_BYTES, "layer-2 operands reuse the drained ring");
  static constexpr int BAR_BYTES = 256;
  static constexpr int CONST_FLOATS = 2 * TC_COLS + 4 * HD_HS + 8 + 4 * TC_M;   // b1 | b2 | w3 | b3 | partial outputs of the upper column half
  static constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + 1024 /* alignment slack */ + BAR_BYTES + CONST_FLOATS * 4;
};

struct TCArgs {
  HArgs h;                 // shapes, biases, output layer, outputs, sampling (w1t / w2t unused here)
  int chunks;              // ceil(K / 32)
  const float* w1tc;       // [chunks][128 / NT][hi tile | lo tile], each tile NT (column) rows x 32 k, swizzled
  const float* w2tc;       // [head][k-chunk (2)][hi tile | lo tile], each tile 64 (column) rows x 32 k, swizzled
};

// byte offset of element (row r, 16-byte chunk c4) inside a K-major SWIZZLE_128B tile
__host__ __device__ __forceinline__ uint32_t tc_swizzle(int r, int c4) { return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c4 ^ (r & 7)) << 4)); }
// the nearest value with 13 zero low mantissa bits (exactly representable as TF32); the remainder x - tc_hi(x) then has at most
// 12 significant bits, of which the tensor core keeps 11
__host__ __device__ __forceinline__ float tc_hi(float x) {
#ifdef __CUDA_ARCH__
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
#else
  uint32_t u; memcpy(&u, &x, 4); u = (u + 0x1000u) & 0xFFFFE000u; float y; memcpy(&y, &u, 4); return y;
#endif
}

// the value as kind::tf32 reads it: the 13 low mantissa bits ignored
__device__ __forceinline__ float tc_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(tc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {  // raises the transaction count, no arrival
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(tc_smem_u32(bar)), "r"(parity) : "memory");
}
// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in [0,14), leading
// byte offset (unused for swizzled K-major layouts; 1) in [16,30), stride byte offset = 1024 B (next 8-row atom) >> 4 in
// [32,46), descriptor version 1 in [46,48), layout type SWIZZLE_128B = 2 in [61,64): low word = tc_desc_lo(address), high word constant
// instruction descriptor (cute::UMMA::InstrDescriptor), kind::tf32: D = F32 (1 << 4), A = B = TF32 (2 << 7, 2 << 10), both K-major,
// N >> 3 in [17,23), M >> 4 in [24,29)
template <int NT>
__host__ __device__ constexpr uint32_t tc_idesc() { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24); }

// low word of the descriptor above (start address | leading byte offset); the high word is the constant TC_DESC_HI
__device__ __forceinline__ uint32_t tc_desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
constexpr uint32_t TC_DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);

// one MMA: D[tmem] (+)= A[desc a] * B[desc b]; descriptors passed as their low words (advancing along K = + 2 per UMMA_K step)
template <bool ACC>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %4};\n\t"
      "mov.b64 db, {%2, %4};\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t}" ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(TC_DESC_HI), "r"(ACC ? 1u : 0u)
      : "memory");
}
// one elected lane of a converged warp (elect.sync): the compiler keeps the enclosed code on the uniform datapath
__device__ __forceinline__ bool tc_elect() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {  // implies tcgen05.fence::before_thread_sync
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tc_bulk_load(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc_smem_u32(dst_smem)), "l"(src),
               "r"(bytes), "r"(tc_smem_u32(bar))
               : "memory");
}
// 32 consecutive TMEM columns of this thread's lane (32x32b: warp w reads lanes 32 w .. 32 w + 31), complete on return
__device__ __forceinline__ void tc_tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, "
      "%29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
        "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
        "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// NORM: the linear policy's NormalizeObservation (NArgs) on X as the producers load it.  Only with NT = 128: one CTA then owns its
// rows and every column, so each (env, k) statistic is read and written by exactly one thread of the grid (with NT = 64 the critic
// and the actor CTA of a row tile would both read the statistics while one of them updates them).
// FROZEN (with NORM): the statistics are only read (evaluation, EvacPolicyIO.norm_frozen), so nothing is shared that a CTA writes
// and both tilings are valid; with NT = 64 the critic CTA (blockIdx.y = 0) alone stores obs_norm.
template <int NT, int ST, int AH, int MINB, bool NORM = false, bool FROZEN = false>
__global__ void __launch_bounds__(TC_THREADS, MINB) evac_policy_heads_tc_kernel(const __grid_constant__ TCArgs a, const __grid_constant__ NArgs n) {
  static_assert(NORM || !FROZEN, "FROZEN is a mode of the fused normaliser");
  static_assert(!NORM || FROZEN || NT == TC_COLS, "the fused normaliser's update needs one CTA per row tile");
  using SH = TCShape<NT, ST, AH>;
  constexpr int STAGES = SH::STAGES, HEADS = SH::HEADS, TC_AHEAD = SH::AHEAD;
  // TMEM columns: layer 1 [0, NT) = xh wh + xl wh, [NT, 2 NT) = xh wl (summed by epilogue 1); layer 2 from 2 NT; power of two
  constexpr int TMEM_COLS = NT == 64 ? 256 : 512;
  extern __shared__ uint8_t tc_smem_raw[];
  uint8_t* smem = tc_smem_raw + ((1024u - (tc_smem_u32(tc_smem_raw) & 1023u)) & 1023u);  // swizzle atoms: 1024-byte aligned (offset, so the pointer stays a shared-memory one)
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * SH::STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* accum = empty + STAGES;      // accum[0]: layer-1 accumulators complete, accum[1]: layer-2 accumulators complete
  uint64_t* full2 = accum + 2;           // layer-2 operands (H1 tiles + weight tiles) in place
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full2 + 1);
  float* cst = reinterpret_cast<float*>(smem + STAGES * SH::STAGE_BYTES + SH::BAR_BYTES);
  float* b1s = cst, *b2s = cst + TC_COLS, *w3s = cst + 2 * TC_COLS, *b3s = w3s + 4 * HD_HS, *opart = b3s + 8;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int e0 = blockIdx.x * TC_M;
  const int ny = TC_COLS / NT, y = blockIdx.y;   // NT = 64: y = 0 critic, y = 1 actor
  const HArgs& h = a.h;

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { tc_mbar_init(&full[s], TC_ET); tc_mbar_init(&empty[s], 1); }
    tc_mbar_init(&accum[0], 1); tc_mbar_init(&accum[1], 1); tc_mbar_init(full2, TC_ET);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == TC_EW) {  // 2 NT TMEM columns of float32 accumulators (layer 1 | layer 2), one warp allocates and later frees
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < TC_COLS; i += TC_THREADS) { b1s[i] = h.b1[i]; b2s[i] = h.b2[i]; }
  for (int i = tid; i < 4 * HD_HS; i += TC_THREADS) w3s[i] = i < (1 + h.A) * HD_HS ? h.w3[i] : 0.f;
  if (tid < 4) b3s[tid] = tid < 1 + h.A ? h.b3[tid] : 0.f;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;
  uint8_t* a2 = smem;                       // H1 operand tiles: k-chunk j at j * 32 KB (hi | lo)
  uint8_t* w2 = smem + SH::A2_BYTES;        // layer-2 weight tiles of this CTA's head(s)

  if (warp == TC_EW) {
    // ---- MMA issue: the whole warp follows the barriers, ONE elected lane issues (12 tcgen05.mma per chunk, stage handed back
    // through tcgen05.commit)
    constexpr uint32_t IDESC1 = tc_idesc<NT>(), IDESC1W = tc_idesc<2 * NT>(), IDESC2 = tc_idesc<HD_HS>();
    for (int c = 0; c < a.chunks; ++c) {
      const int s = c % STAGES;
      tc_mbar_wait(&full[s], (uint32_t)((c / STAGES) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (tc_elect()) {
        const uint32_t xh = tc_desc_lo(tc_smem_u32(smem + s * SH::STAGE_BYTES)), xl = xh + (TC_XTILE_BYTES >> 4);
        const uint32_t wh = xh + (2 * TC_XTILE_BYTES >> 4);   // [W hi | W lo]: 2 NT rows, the lo tile right behind the hi tile
        // per k-step TWO MMAs: xh x [wh | wl] (the hi and lo weight tiles are one 2 NT-row B tile: N = 2 NT) and xl x wh (N = NT)
        // -- the xh slice is read from shared memory once instead of twice (14 instead of 18 KB of operand reads per k-step)
        if (c == 0) tc_mma<false>(tmem, xh, wh, IDESC1W); else tc_mma<true>(tmem, xh, wh, IDESC1W);
        tc_mma<true>(tmem, xl, wh, IDESC1);
#pragma unroll
        for (int k = 1; k < TC_KC / 8; ++k) {  // UMMA_K = 8 float32 = 32 bytes along the swizzled row = + 2 in the descriptor
          tc_mma<true>(tmem, xh + 2 * k, wh + 2 * k, IDESC1W);
          tc_mma<true>(tmem, xl + 2 * k, wh + 2 * k, IDESC1);
        }
        tc_commit(&empty[s]);
        if (c == a.chunks - 1) tc_commit(&accum[0]);
      }
      __syncwarp();
    }
    // ---- layer 2: per head [128 x 64] x [64 x 64], operands written by epilogue 1 / the second bulk copy
    tc_mbar_wait(full2, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tc_elect()) {
#pragma unroll
      for (int hd = 0; hd < HEADS; ++hd) {
        const uint32_t d = tmem + (uint32_t)(2 * NT + hd * HD_HS);
#pragma unroll
        for (int c = 0; c < HD_HS / TC_KC; ++c) {
          const uint32_t xh = tc_desc_lo(tc_smem_u32(a2 + (hd * (HD_HS / TC_KC) + c) * 2 * TC_XTILE_BYTES)), xl = xh + (TC_XTILE_BYTES >> 4);
          const uint32_t wh = tc_desc_lo(tc_smem_u32(w2 + hd * TC_W2_HEAD_BYTES + c * (2 * HD_HS * TC_KC * 4))), wl = wh + (HD_HS * TC_KC * 4 >> 4);
#pragma unroll
          for (int k = 0; k < TC_KC / 8; ++k) {
            if (c == 0 && k == 0) tc_mma<false>(d, xh, wh, IDESC2); else tc_mma<true>(d, xh + 2 * k, wh + 2 * k, IDESC2);
            tc_mma<true>(d, xl + 2 * k, wh + 2 * k, IDESC2);
            tc_mma<true>(d, xh + 2 * k, wl + 2 * k, IDESC2);
          }
        }
      }
      tc_commit(&accum[1]);
    }
    __syncwarp();
  } else {
    // ---- producers.  X travels global -> shared as raw float32 straight into the swizzled "hi" tile (cp.async, 16 bytes per
    // request, TC_AHEAD chunks ahead): kind::tf32 ignores the 13 low mantissa bits of its operands, so the raw value IS
    // xh = trunc(x) to the tensor core; each thread then reads back the eight float4 it requested itself, writes
    // xl = x - trunc(x) into the "lo" tile and arrives.  The weight tiles of the same chunk ride on one bulk copy.
    const int kq = h.K >> 2;  // float4 per row of X
    auto request = [&](int c) {
      const int s = c % STAGES, use = c / STAGES;
      if (use > 0) tc_mbar_wait(&empty[s], (uint32_t)((use - 1) & 1));  // the MMAs that read this stage have completed
      uint8_t* st = smem + s * SH::STAGE_BYTES;
      if constexpr (!NORM) {   // with NORM the X tiles of chunk c are written when chunk c is finished (below)
#pragma unroll
        for (int i = 0; i < 1024 / TC_ET; ++i) {
          const int idx = i * TC_ET + tid, r = idx >> 3, c4 = idx & 7;
          const int e = e0 + r, q = c * 8 + c4;
          const bool in = e < h.E && q < kq;
          cp_async16(reinterpret_cast<float*>(st + tc_swizzle(r, c4)), h.emb + (in ? (size_t)e * h.K + 4 * q : (size_t)0), in ? 16 : 0);
        }
      }
      if (tid == 0) {
        tc_mbar_expect_tx(&full[s], 2 * SH::WTILE_BYTES);
        tc_bulk_load(st + 2 * TC_XTILE_BYTES, a.w1tc + ((size_t)c * ny + y) * (2 * SH::WTILE_BYTES / 4), 2 * SH::WTILE_BYTES, &full[s]);
      }
    };
#pragma unroll
    for (int c = 0; c < TC_AHEAD; ++c) {
      if (c < a.chunks) request(c);
      cp_async_commit();
    }
    for (int c = 0; c < a.chunks; ++c) {
      if (c + TC_AHEAD < a.chunks) request(c + TC_AHEAD);
      cp_async_commit();               // one group per iteration, empty or not: group index == chunk index
      cp_async_wait<TC_AHEAD>();       // this thread's requests of chunk c have landed
      uint8_t* st = smem + (c % STAGES) * SH::STAGE_BYTES;
      if constexpr (NORM) {
        // X through registers: the raw rows and their statistics in (all loads of the chunk issued before the first use),
        // update + normalise + clip, statistics and obs_norm out, then the normalised value as the hi tile (the tensor core
        // truncates it itself, as it does the cp.async'd raw value above) and its remainder as the lo tile.  FROZEN: no update, the
        // statistics are not stored
        NormWeights nw;
        if constexpr (!FROZEN) nw = norm_weights(n);
        float4 x[1024 / TC_ET], m[1024 / TC_ET], v[1024 / TC_ET];
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 1024 / TC_ET; ++i) {
          const int idx = i * TC_ET + tid, r = idx >> 3, c4 = idx & 7;
          const int e = e0 + r, q = c * 8 + c4;
          x[i] = m[i] = v[i] = zero;
          if (e < h.E && q < kq) {
            const size_t g = (size_t)e * h.K + 4 * q;
            x[i] = *reinterpret_cast<const float4*>(h.emb + g);
            m[i] = *reinterpret_cast<const float4*>(n.mean + g);
            v[i] = *reinterpret_cast<const float4*>(n.var + g);
          }
        }
#pragma unroll
        for (int i = 0; i < 1024 / TC_ET; ++i) {
          const int idx = i * TC_ET + tid, r = idx >> 3, c4 = idx & 7;
          const int e = e0 + r, q = c * 8 + c4;
          float4 z = zero;
          if (e < h.E && q < kq) {
            const size_t g = (size_t)e * h.K + 4 * q;
            if constexpr (FROZEN) {
              z.x = norm_frozen(x[i].x, m[i].x, v[i].x, n.eps, n.clip); z.y = norm_frozen(x[i].y, m[i].y, v[i].y, n.eps, n.clip);
              z.z = norm_frozen(x[i].z, m[i].z, v[i].z, n.eps, n.clip); z.w = norm_frozen(x[i].w, m[i].w, v[i].w, n.eps, n.clip);
              if (n.obs_norm != nullptr && y == 0) *reinterpret_cast<float4*>(n.obs_norm + g) = z;
            } else {
              z.x = norm_update(x[i].x, m[i].x, v[i].x, nw, n); z.y = norm_update(x[i].y, m[i].y, v[i].y, nw, n);
              z.z = norm_update(x[i].z, m[i].z, v[i].z, nw, n); z.w = norm_update(x[i].w, m[i].w, v[i].w, nw, n);
              *reinterpret_cast<float4*>(n.mean + g) = m[i];
              *reinterpret_cast<float4*>(n.var + g) = v[i];
              if (n.obs_norm != nullptr) *reinterpret_cast<float4*>(n.obs_norm + g) = z;
            }
          }
          const uint32_t off = tc_swizzle(r, c4);
          *reinterpret_cast<float4*>(st + off) = z;
          *reinterpret_cast<float4*>(st + TC_XTILE_BYTES + off) =
              make_float4(z.x - tc_trunc(z.x), z.y - tc_trunc(z.y), z.z - tc_trunc(z.z), z.w - tc_trunc(z.w));
        }
      } else {
#pragma unroll
        for (int i = 0; i < 1024 / TC_ET; ++i) {
          const int idx = i * TC_ET + tid, r = idx >> 3, c4 = idx & 7;
          const uint32_t off = tc_swizzle(r, c4);
          const float4 x = *reinterpret_cast<const float4*>(st + off);
          *reinterpret_cast<float4*>(st + TC_XTILE_BYTES + off) =
              make_float4(x.x - tc_trunc(x.x), x.y - tc_trunc(x.y), x.z - tc_trunc(x.z), x.w - tc_trunc(x.w));
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // cp.async / generic-proxy stores -> visible to the tensor core (async proxy)
      tc_mbar_arrive(&full[c % STAGES]);
    }
    // ---- epilogue 1: TMEM lane = environment (this thread's row), column = hidden unit -> H1 operand tiles of layer 2
    tc_mbar_wait(&accum[0], 0u);           // every layer-1 MMA has completed: accumulators final, the ring is free
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (tid == 0) {
      tc_mbar_expect_tx(full2, SH::W2_BYTES);
      tc_bulk_load(w2, a.w2tc + (size_t)(NT == 64 ? y : 0) * (TC_W2_HEAD_BYTES / 4), SH::W2_BYTES, full2);
    }
    // warp w: TMEM lane quarter w & 3 (the hardware's rule: a warp reads lanes 32 (w % 4) ..), column half w >> 2 of the CTA's NT
    const int row = (warp & 3) * 32 + lane, ch = warp >> 2;
    constexpr int CW = NT / (TC_EW / 4);                        // columns per warp
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
#pragma unroll 1
    for (int jj = 0; jj < CW / 32; ++jj) {
      const int j = ch * (CW / 32) + jj;                        // 32-column block = k-chunk of layer 2
      uint32_t v[32], v2[32];
      tc_tmem_ld32(trow + (uint32_t)(j * 32), v);
      tc_tmem_ld32(trow + (uint32_t)(NT + j * 32), v2);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(v2[i]));
      uint8_t* tile = a2 + j * 2 * TC_XTILE_BYTES;
      const float* bj = b1s + y * NT + j * 32;
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 t = make_float4(tanhf(__uint_as_float(v[i]) + bj[i]), tanhf(__uint_as_float(v[i + 1]) + bj[i + 1]),
                                     tanhf(__uint_as_float(v[i + 2]) + bj[i + 2]), tanhf(__uint_as_float(v[i + 3]) + bj[i + 3]));
        float4 hi, lo;
        hi.x = tc_hi(t.x); lo.x = t.x - hi.x;
        hi.y = tc_hi(t.y); lo.y = t.y - hi.y;
        hi.z = tc_hi(t.z); lo.z = t.z - hi.z;
        hi.w = tc_hi(t.w); lo.w = t.w - hi.w;
        const uint32_t off = tc_swizzle(row, i >> 2);
        *reinterpret_cast<float4*>(tile + off) = hi;
        *reinterpret_cast<float4*>(tile + TC_XTILE_BYTES + off) = lo;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_mbar_arrive(full2);
    // ---- epilogue 2: H2 = tanh(. + b2) and the output layer as dot products over the TMEM loads, then the sampling tail
    tc_mbar_wait(&accum[1], 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
    for (int jj = 0; jj < CW / 32; ++jj) {
      const int j = ch * (CW / 32) + jj;
      uint32_t v[32];
      tc_tmem_ld32(trow + (uint32_t)(2 * NT + j * 32), v);
      const int col0 = y * NT + j * 32;               // hidden column of v[0]: < 64 critic, >= 64 actor
      const float* bj = b2s + col0;
      if (col0 < HD_HS) {
        const float* w = w3s + col0;
#pragma unroll
        for (int i = 0; i < 32; ++i) o[0] = fmaf(tanhf(__uint_as_float(v[i]) + bj[i]), w[i], o[0]);
      } else {
        const float* w = w3s + HD_HS + (col0 - HD_HS);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float t = tanhf(__uint_as_float(v[i]) + bj[i]);
          o[1] = fmaf(t, w[i], o[1]); o[2] = fmaf(t, w[HD_HS + i], o[2]); o[3] = fmaf(t, w[2 * HD_HS + i], o[3]);
        }
      }
    }
    const int e = e0 + row;
    if constexpr (NT == 128) {   // column half 0 = the critic's 64 columns, half 1 = the actor's: every thread finishes one head
#pragma unroll
      for (int c = 0; c < 4; ++c) o[c] += b3s[c];
      if (e < h.E) heads_finish(h, e, o, ch == 0, ch == 1);
    } else {                     // the head's 64 columns are split over the two halves: the upper half hands its partial sums over
      if (ch == 1) *reinterpret_cast<float4*>(opart + 4 * row) = make_float4(o[0], o[1], o[2], o[3]);
      asm volatile("bar.sync 1, %0;" ::"n"(TC_ET) : "memory");
      if (ch == 0) {
        const float4 u = *reinterpret_cast<const float4*>(opart + 4 * row);
        o[0] = b3s[0] + (o[0] + u.x); o[1] = b3s[1] + (o[1] + u.y); o[2] = b3s[2] + (o[2] + u.z); o[3] = b3s[3] + (o[3] + u.w);
        if (e < h.E) heads_finish(h, e, o, y == 0, y == 1);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == TC_EW) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS) : "memory");
  }
}

}  // namespace evacp
