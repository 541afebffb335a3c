// Crowds larger than one SM's shared memory: ONE environment per thread-block CLUSTER of CL CTAs (CL = 2, 4, 8;
// 1024 threads x 4 pedestrians each -> up to 32 768 pedestrians), the cell-list neighbour search of
// evac_kernels.cuh::cell_list_pass distributed over the cluster through distributed shared memory (DSMEM).
// Included by evac_kernels.cuh (needs Tile, CellSmem and the phases shared with cell_list_pass).  [area.py:105-119; SURVEY 8 row f3]
//
//   CTA r owns pedestrians [r * SLOTS, (r + 1) * SLOTS) in registers (as in the one-CTA kernel) and the slice
//   [r * SLOTS, (r + 1) * SLOTS) of the SORTED source tile in its shared memory.
//   1. every CTA: histogram of its own moving pedestrians over the cells + rank inside (cell, CTA) (rank_in_cells)
//                                                                                                       -> cluster barrier
//   2. every CTA (redundantly): cell totals = sum of the CL histograms read through DSMEM, exclusive scan (scan_cell_counts)
//      -> cell_start[] (global slot numbering); below[c] = pedestrians of lower-ranked CTAs in c.
//      Global slot = cell_start[c] + below[c] + rank: the tile is sorted by (cell, pedestrian index) exactly like the
//      one-CTA pass, so every float32 sum has the same value as there.
//   3. scatter of the source records into the tile slice of the CTA that owns the slot (DSMEM stores) -> cluster barrier
//   4. paired walk (walk_slot_pair over ClusterSlots); the warps of the whole cluster draw chunks of slot pairs from one
//      counter, so a crowd that has collapsed into one corner is still walked by all CTAs; tile reads go to whichever CTA
//      owns the slot pair; the result goes to the CTA that owns the pedestrian                          -> cluster barrier
//   5. the owners read their results (read_results).
// (textually included inside namespace evac, after cell_list_pass; <cooperative_groups.h> comes from evac_kernels.cuh)
#pragma once
namespace cg = cooperative_groups;

// extra per-CTA arrays of the cluster pass, placed after CellSmem
struct ClusterSmem {
  int* hist;    // [C + 1] own moving pedestrians per cell (read by the other CTAs)
  int* below;   // [C + 1] moving pedestrians of the lower-ranked CTAs in each cell
  int* flags;   // [4]     [0] a source of this CTA has no direction (NaN poisoning)  [1] (CTA 0) next slot pair of the walk
  static __host__ __device__ constexpr size_t bytes(int cells) { return 2 * (((size_t)cells + 1 + 3) & ~(size_t)3) * 4 + 16; }
  __device__ __forceinline__ ClusterSmem(unsigned char* p, int cells) {
    hist = reinterpret_cast<int*>(p);
    below = hist + ((cells + 1 + 3) & ~3);
    flags = below + ((cells + 1 + 3) & ~3);
  }
};

// the CTA that owns global slot pair `pair` of the sorted tile, and the pair's index inside that CTA's slice
// (the last CTA also owns the tile's spare entries behind its slice)
template <int SLOTS, int CL>
__device__ __forceinline__ void owner_of_pair(int pair, int& owner, int& local) {
  owner = min(pair / (SLOTS / 2), CL - 1);
  local = pair - owner * (SLOTS / 2);
}

// shared::cluster addressing of the walk: one MAPA per segment, then LDS-like 128-bit loads from the owning CTA
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, int cta_rank) {
  uint32_t r;
  asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ float4 ld_cluster_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// The sorted tile distributed over the cluster, with the interface of CtaSlots (evac_kernels.cuh): slot pair -> owning CTA by
// owner_of_pair; a run is the part of [j, je) inside one CTA's slice, read with one MAPA and ld.shared::cluster; a result goes
// to the shared memory of the CTA that owns the pedestrian.
template <int SLOTS, int CL>
struct ClusterSlots {
  const Tile<float>& tile;
  const CellSmem& cs;
  struct Run {
    uint32_t pa, ua;
    __device__ __forceinline__ float4 p(int q) const { return ld_cluster_f4(pa + 16u * (uint32_t)q); }
    __device__ __forceinline__ float4 u(int q) const { return ld_cluster_f4(ua + 16u * (uint32_t)q); }
  };
  __device__ __forceinline__ int sorted_idx(int s) const {
    int owner, lp;
    owner_of_pair<SLOTS, CL>(s >> 1, owner, lp);
    return cg::this_cluster().map_shared_rank(cs.sorted_idx, owner)[s - owner * SLOTS];
  }
  __device__ __forceinline__ float4 p2(int pair) const {
    int owner, lp;
    owner_of_pair<SLOTS, CL>(pair, owner, lp);
    return *cg::this_cluster().map_shared_rank(tile.P2 + lp, owner);
  }
  __device__ __forceinline__ Run run(int j, int je, int& end) const {
    int owner, lp;
    owner_of_pair<SLOTS, CL>(j, owner, lp);
    end = owner == CL - 1 ? je : min(je, (owner + 1) * (SLOTS / 2));
    const uint32_t pa = mapa_u32(smem_u32(tile.P2 + lp), owner);
    return {pa, pa + (uint32_t)((SLOTS / 2 + 1) * sizeof(float4))};  // U2 = P2 + SLOTS / 2 + 1 in every CTA
  }
  __device__ __forceinline__ void put_res(int i, float2 r) const { cg::this_cluster().map_shared_rank(cs.res, i / SLOTS)[i % SLOTS] = r; }
};

template <int THREADS, int PPT, int CL, typename A>
__device__ __forceinline__ void cell_list_pass_cluster(const Tile<float>& tile, const CellSmem& cs, const ClusterSmem& xs, const A& a,
                                                       const float (&px)[PPT], const float (&py)[PPT], const float (&ux)[PPT],
                                                       const float (&uy)[PPT], const bool (&efv)[PPT], const int (&st)[PPT],
                                                       float (&sx)[PPT], float (&sy)[PPT]) {
  constexpr int SLOTS = THREADS * PPT;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank_cta = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int C = a.cells_x * a.cells_y;
  // ---- 1. own histogram + rank inside (cell, CTA); the [WARPS][C] byte table fits the tile slice (the host caps the grid at
  // 2048 cells), and nobody writes the slice before the cluster barrier
  for (int c = tid; c <= C; c += THREADS) xs.hist[c] = 0;
  if (tid == 0) { xs.flags[0] = 0; xs.flags[1] = 0; }
  int cell[PPT], rank[PPT];
  const bool nan_src = rank_in_cells<THREADS, PPT>(tile, xs.hist, a, px, py, ux, uy, efv, cell, rank);
  if (__syncthreads_or(nan_src) && tid == 0) xs.flags[0] = 1;
  cluster.sync();  // every histogram is final and nobody uses its tile slice as scratch any more
  // ---- 2. cell totals over the cluster, exclusive scan
  bool poisoned = false;
#pragma unroll
  for (int r = 0; r < CL; ++r) poisoned |= cluster.map_shared_rank(xs.flags, r)[0] != 0;
  for (int c = tid; c <= C; c += THREADS) {
    int tot = 0, below = 0;
    if (c < C) {
#pragma unroll
      for (int r = 0; r < CL; ++r) {
        const int v = cluster.map_shared_rank(xs.hist, r)[c];
        tot += v;
        if (r < rank_cta) below += v;
      }
    }
    cs.cell_start[c] = tot;
    xs.below[c] = below;
  }
  __syncthreads();
  const int n_src = scan_cell_counts<THREADS>(cs, C);
  // ---- 3. scatter into the slice of the CTA that owns the slot: global slot = cell start + pedestrians of the lower-ranked
  // CTAs in the cell + rank inside (cell, CTA)
  const int base_i = rank_cta * SLOTS;
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    if (efv[k]) {
      const int g = cs.cell_start[cell[k]] + xs.below[cell[k]] + rank[k];
      int owner, lp;
      owner_of_pair<SLOTS, CL>(g >> 1, owner, lp);
      const bool fv = (unsigned)(st[k] - ST_VISCEK) <= (unsigned)(ST_FOLLOWER - ST_VISCEK);
      float* p = cluster.map_shared_rank(reinterpret_cast<float*>(tile.P2 + lp) + (g & 1), owner);
      float* u = cluster.map_shared_rank(reinterpret_cast<float*>(tile.U2 + lp) + (g & 1), owner);
      p[0] = px[k]; p[2] = py[k]; u[0] = ux[k]; u[2] = uy[k];
      const int ls = g - owner * SLOTS;
      cluster.map_shared_rank(cs.sorted_idx, owner)[ls] = (uint16_t)((base_i + k * THREADS + tid) | (fv ? 0x8000 : 0));
    }
  }
  if (tid < 2) {  // pad to an even count
    const int g = n_src + tid;
    int owner, lp;
    owner_of_pair<SLOTS, CL>(g >> 1, owner, lp);
    if (owner == rank_cta) tile.put(2 * lp + (g & 1), PARK, PARK, 0.f, 0.f);
  }
  if (warp == 0) scan_row_pairs(cs, a);
  cluster.sync();  // the whole sorted tile is in place
  // ---- 4. paired walk.  The warps of the whole cluster draw chunks of 32 slot pairs from ONE counter (a DSMEM atomic on
  // CTA 0's shared memory): a walk costs as much as its cells are crowded, so equal shares of slot pairs would leave the
  // CTAs of a cluster waiting at the barrier for the one that drew the densest cells (ncu: `barrier` was the top stall).
  // The result of a pair does not depend on who walks it.
  const int n_pairs = cs.row_pairs[a.cells_y];
  int* const next_pair = cluster.map_shared_rank(xs.flags, 0) + 1;
#pragma unroll 1
  for (;;) {
    int tb = 0;
    if (lane == 0) tb = atomicAdd(next_pair, 32);
    tb = __shfl_sync(0xffffffffu, tb, 0);
    if (tb >= n_pairs) break;
    const int t = tb + lane;
    if (t < n_pairs) walk_slot_pair(ClusterSlots<SLOTS, CL>{tile, cs}, cs, a, t);
    __syncwarp();
  }
  cluster.sync();  // every result has reached its owner
  // ---- 5. back to the owners
  read_results<THREADS, PPT>(cs, poisoned, st, sx, sy);
}

// Sum of per-CTA partials over the cluster in rank order (every CTA gets the same bits).  `slot` is a [8]-double
// array in each CTA's shared memory; two cluster barriers fence the exchange.
template <int CL, int NV>
__device__ __forceinline__ void cluster_sum(double* slot, double (&v)[NV]) {
  cg::cluster_group cluster = cg::this_cluster();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 0; q < NV; ++q) slot[q] = v[q];
  }
  cluster.sync();
#pragma unroll
  for (int q = 0; q < NV; ++q) v[q] = 0.0;
#pragma unroll
  for (int r = 0; r < CL; ++r) {
    const double* s = cluster.map_shared_rank(slot, r);
#pragma unroll
    for (int q = 0; q < NV; ++q) v[q] += s[q];
  }
  cluster.sync();  // everyone has read before the slot is written again
}

