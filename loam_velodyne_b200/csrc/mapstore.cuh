// Persistent, incrementally maintained map (SURVEY.md §8f rank 1: "sweeps/s independent of M").
//
// mappool.cuh's first device-resident map re-derived everything from the flat pool every sweep: classify 1 M points,
// compact the visible cubes, sort them by cell for the search grid, and at the end of the sweep sort the visible cubes
// plus the new points by voxel -- four O(M) radix sorts per sweep for ~23 k new points.  Here the pool of each kind
// (corner / surface) is kept SORTED BY CELL across sweeps, with its cell table, so that
//   * the search grid of the scan-to-map loop simply exists when a sweep starts (no per-sweep build);
//   * "which cubes are in the field of view" is a lookup per probed cell (the cube of a 1 m cell is a function of the
//     cell: cube faces sit on integer coordinates, BasicLaserMapping.cpp:540-553);
//   * the end-of-sweep voxel filter only sorts the NEW points: a voxel that received points finds the map point it
//     already holds through the cell table, the centroid replaces it (pcl::VoxelGrid of "old centroid + new points",
//     which is what re-filtering the whole cube computes for that voxel, :580-588); untouched voxels are not touched;
//   * the updated pool is produced by one merge of two sorted sequences (pool minus replaced points, new centroids).
// Cell key = slot << 17 | cell-in-cube, slot = the cube's position in the 21 x 11 x 21 grid taken modulo the grid
// dimensions of its ABSOLUTE cube coordinates, so keys do not change when the grid rolls (:311-441 only changes the
// centre offsets); points of cubes that left the grid are dropped by the merge of the sweep in which the roll happened.
// A point is RAW until a voxel filter has seen it: seeded maps and points inserted into cubes outside the field of view
// stay unfiltered, exactly like the reference's cube clouds, until their cube is visible at the end of a sweep.
#pragma once

#include "clustersort.cuh"
#include "gridnn.cuh"
#include "mappool.cuh"

namespace loamb {

constexpr unsigned char ST_RAW = 1, ST_DEAD = 2;

__host__ __device__ __forceinline__ int floordiv_i(int v, int d) { return v >= 0 ? v / d : -((-v + d - 1) / d); }
__host__ __device__ __forceinline__ int pmod_i(int v, int d) {
  const int r = v % d;
  return r < 0 ? r + d : r;
}

struct CellAxis {
  int a;   // absolute cube coordinate
  int r;   // cell inside the cube, 0..49
  int pm;  // a modulo the grid dimension
};
__device__ __forceinline__ CellAxis cell_axis(int c, int dim) {
  CellAxis x;
  x.a = floordiv_i(c + 25, 50);
  x.r = c + 25 - 50 * x.a;
  x.pm = pmod_i(x.a, dim);
  return x;
}
__device__ __forceinline__ CellAxis axis_step(CellAxis x, int d, int dim) {  // d in {-1, 0, +1}
  x.r += d;
  if (x.r == 50) {
    x.r = 0; x.a++; x.pm = (x.pm + 1 == dim) ? 0 : x.pm + 1;
  } else if (x.r < 0) {
    x.r = 49; x.a--; x.pm = (x.pm == 0) ? dim - 1 : x.pm - 1;
  }
  return x;
}
__device__ __forceinline__ unsigned torus_key(const CellAxis& x, const CellAxis& y, const CellAxis& z) {
  const unsigned slot = (unsigned)(x.pm + CUBE_W * (y.pm + CUBE_H * z.pm));
  return (slot << 17) | (unsigned)((z.r * 50 + y.r) * 50 + x.r);
}
__device__ __forceinline__ unsigned torus_key_of(const float4& p) {
  return torus_key(cell_axis(store_cell(p.x), CUBE_W), cell_axis(store_cell(p.y), CUBE_H), cell_axis(store_cell(p.z), CUBE_D));
}

struct MapGridView {
  const uint4* table;   // {key + 1 (0 = empty), start, count, -}
  unsigned mask;
  const float4* pts;    // pool in cell order (w = intensity)
  const unsigned char* rank_of_cube;  // by grid index; < n_valid when the cube is in the field of view this sweep
  int cen_w, cen_h, cen_d, n_valid;
};

__device__ __forceinline__ bool store_probe(const MapGridView& g, unsigned key, unsigned& start, unsigned& count,
                                            unsigned* probes) {
  unsigned h = grid_hash(key) & g.mask;
  uint4 e = __ldg(&g.table[h]);
  if (probes) (*probes)++;
  while (e.x != 0u && e.x != key + 1u) {
    h = (h + 1) & g.mask;
    e = __ldg(&g.table[h]);
    if (probes) (*probes)++;
  }
  if (e.x != key + 1u) return false;
  start = e.y;
  count = e.z;
  return true;
}

// neighbour-cell lookup of the scan-to-map search (plugs into grid_knn5_group8)
struct MapCellLookup {
  MapGridView g;
  CellAxis ax, ay, az;
  int prune;  // see GridCellLookup
  __device__ __forceinline__ bool prepare(float qx, float qy, float qz) {
    ax = cell_axis((int)floorf(qx), CUBE_W);
    ay = cell_axis((int)floorf(qy), CUBE_H);
    az = cell_axis((int)floorf(qz), CUBE_D);
    return g.table != nullptr;
  }
  template <bool STATS>
  __device__ __forceinline__ void cell(int t, unsigned& start, unsigned& count, unsigned* stats) const {
    const CellAxis x = axis_step(ax, t % 3 - 1, CUBE_W), y = axis_step(ay, (t / 3) % 3 - 1, CUBE_H),
                   z = axis_step(az, t / 9 - 1, CUBE_D);
    const int ix = x.a + g.cen_w, iy = y.a + g.cen_h, iz = z.a + g.cen_d;
    if (ix < 0 || ix >= CUBE_W || iy < 0 || iy >= CUBE_H || iz < 0 || iz >= CUBE_D) return;
    if ((int)__ldg(&g.rank_of_cube[ix + CUBE_W * iy + CUBE_W * CUBE_H * iz]) >= g.n_valid) return;  // not in view
    store_probe(g, torus_key(x, y, z), start, count, STATS ? stats : nullptr);
  }
  __device__ __forceinline__ const float4* points() const { return g.pts; }
};

// ---------------------------------------------------------------------------------------------- (re)build from scratch
__global__ void store_key_kernel(const float4* __restrict__ p, int n, unsigned* __restrict__ keys, int* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = torus_key_of(p[i]);
  vals[i] = i;
}

__global__ void store_gather_kernel(const float4* __restrict__ p, const unsigned char* __restrict__ st,
                                    const int* __restrict__ order, int n, const int* __restrict__ n_dev,
                                    float4* __restrict__ p_out, unsigned char* __restrict__ st_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (n_dev) n = min(n, *n_dev);
  if (i >= n) return;
  const int o = order[i];
  p_out[i] = p[o];
  st_out[i] = st[o];
}

// per cube slot: [start, end) of its points in the sorted pool and the number of RAW points among them
__global__ void store_stats_kernel(const unsigned* __restrict__ keys, const unsigned char* __restrict__ st, int n,
                                   const int* __restrict__ n_dev, int* __restrict__ cube_start, int* __restrict__ cube_end,
                                   int* __restrict__ cube_raw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (n_dev) n = min(n, *n_dev);
  const bool in = i < n;
  const unsigned slot = in ? (keys[i] >> 17) : 0xffffffffu;
  if (in) {
    if (i == 0 || (keys[i - 1] >> 17) != slot) cube_start[slot] = i;
    if (i == n - 1 || (keys[i + 1] >> 17) != slot) cube_end[slot] = i + 1;
  }
  // warp-aggregated count of raw points (keys are sorted: a warp rarely spans more than one slot)
  const bool raw = in && (st[i] & ST_RAW);
  const unsigned peers = __match_any_sync(0xffffffffu, raw ? slot : 0xfffffffeu);
  if (raw && (peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0) atomicAdd(&cube_raw[slot], __popc(peers));
}

// begin of a sweep: points (and raw points) in the cubes of the field of view, pool size -> out[0..2]
__global__ void store_window_counts_kernel(const unsigned char* __restrict__ rank_of_cube, int n_valid, CubeGrid g,
                                           const int* __restrict__ cube_start, const int* __restrict__ cube_end,
                                           const int* __restrict__ cube_raw, int* __restrict__ out_from_map,
                                           int* __restrict__ out_raw_valid) {
  __shared__ int s_cnt[32], s_raw[32];
  int cnt = 0, raw = 0;
  for (int idx = threadIdx.x; idx < CUBE_NUM; idx += blockDim.x) {
    if ((int)rank_of_cube[idx] >= n_valid) continue;
    const int i = idx % CUBE_W, j = (idx / CUBE_W) % CUBE_H, k = idx / (CUBE_W * CUBE_H);
    const int slot = pmod_i(i - g.cen_w, CUBE_W) + CUBE_W * (pmod_i(j - g.cen_h, CUBE_H) + CUBE_H * pmod_i(k - g.cen_d, CUBE_D));
    cnt += cube_end[slot] - cube_start[slot];
    raw += cube_raw[slot];
  }
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    raw += __shfl_xor_sync(0xffffffffu, raw, o);
  }
  if ((threadIdx.x & 31) == 0) { s_cnt[threadIdx.x >> 5] = cnt; s_raw[threadIdx.x >> 5] = raw; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int c = 0, r = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { c += s_cnt[w]; r += s_raw[w]; }
    *out_from_map = c;
    *out_raw_valid = r;
  }
}

// ---------------------------------------------------------------------------------------------- end of a sweep
// filter key of a point that takes part in this sweep's voxel filter: rank << 24 | vz << 16 | vy << 8 | vx for the
// cubes in view, a unique key behind them for points of invisible cubes (KEEP) and of no cube at all (DROP)
__device__ __forceinline__ unsigned filter_key_of(const float4& q, int i, const CubeGrid& g,
                                                  const unsigned char* __restrict__ rank_of_cube, float inv_leaf) {
  int ci, cj, ck;
  const int cidx = cube_index(q, g, ci, cj, ck);
  const unsigned char cl = cidx < 0 ? CLS_DROP : rank_of_cube[cidx];
  if (cl >= CLS_KEEP) return ((unsigned)cl << 24) | ((unsigned)i & 0xffffffu);
  const float bx = 50.0f * (float)(ci - g.cen_w) - 25.5f;
  const float by = 50.0f * (float)(cj - g.cen_h) - 25.5f;
  const float bz = 50.0f * (float)(ck - g.cen_d) - 25.5f;
  const int vx = (int)floorf(q.x * inv_leaf) - (int)floorf(bx * inv_leaf);
  const int vy = (int)floorf(q.y * inv_leaf) - (int)floorf(by * inv_leaf);
  const int vz = (int)floorf(q.z * inv_leaf) - (int)floorf(bz * inv_leaf);
  return ((unsigned)cl << 24) | ((unsigned)(vz & 255) << 16) | ((unsigned)(vy & 255) << 8) | (unsigned)(vx & 255);
}

// S[0..n_ins) = pointAssociateToMap(stackDS) with the optimised pose (:536-577) + its filter key
__global__ void store_insert_kernel(const float4* __restrict__ stack_ds, int n, MapIterArgs a, CubeGrid g,
                                    const unsigned char* __restrict__ rank_of_cube, float inv_leaf,
                                    float4* __restrict__ s_pts, unsigned* __restrict__ keys, int* __restrict__ vals,
                                    ShardSpec sh) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 q = stack_ds[i];
  float x, y, z;
  associate_to_map(a, q, x, y, z);
  const float4 p = make_float4(x, y, z, q.w);
  s_pts[i] = p;
  // a sharded map only takes the points of the cells this rank stores (the others go to the rank that does)
  keys[i] = shard_stores(sh, store_cell(p.x)) ? filter_key_of(p, i, g, rank_of_cube, inv_leaf)
                                              : (((unsigned)CLS_DROP << 24) | ((unsigned)i & 0xffffffu));
  vals[i] = i;
}

// raw pool points of the cubes in view take part in the filter like new points (they leave the pool: DEAD):
// pass 1 flags + counts them, the scatter pass appends them behind the inserted points
__global__ void __launch_bounds__(SCAN_BS)
store_raw_select_count_kernel(const unsigned* __restrict__ keys, const unsigned char* __restrict__ st, int n,
                              const int* __restrict__ n_dev, const unsigned char* __restrict__ valid_by_slot,
                              unsigned* __restrict__ local_pos, unsigned* __restrict__ block_sums) {
  __shared__ unsigned ws[32];
  if (n_dev) n = min(n, *n_dev);
  const int i = blockIdx.x * SCAN_BS + threadIdx.x;
  const unsigned h = (i < n && (st[i] & ST_RAW) && !(st[i] & ST_DEAD) && valid_by_slot[keys[i] >> 17]) ? 1u : 0u;
  unsigned x = h;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned y = __shfl_up_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) >= o) x += y;
  }
  if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
  __syncthreads();
  if (threadIdx.x < 32) {
    unsigned w = ws[threadIdx.x];
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned y = __shfl_up_sync(0xffffffffu, w, o);
      if (threadIdx.x >= o) w += y;
    }
    ws[threadIdx.x] = w;
  }
  __syncthreads();
  const unsigned incl = x + ((threadIdx.x >> 5) ? ws[(threadIdx.x >> 5) - 1] : 0u);
  if (i < n) local_pos[i] = (incl - h) | (h << 31);
  if (threadIdx.x == SCAN_BS - 1) block_sums[blockIdx.x] = incl;
}

__global__ void store_raw_select_scatter_kernel(const float4* __restrict__ pool, unsigned char* __restrict__ st, int n,
                                                const int* __restrict__ n_dev, const unsigned* __restrict__ local_pos,
                                                const unsigned* __restrict__ block_off, int s_offset, int s_cap, CubeGrid g,
                                                const unsigned char* __restrict__ rank_of_cube, float inv_leaf,
                                                float4* __restrict__ s_pts, unsigned* __restrict__ keys,
                                                int* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (n_dev) n = min(n, *n_dev);
  if (i >= n) return;
  const unsigned pv = local_pos[i];
  if (!(pv >> 31)) return;
  const int d = s_offset + (int)((pv & 0x7fffffffu) + block_off[i / SCAN_BS]);
  if (d >= s_cap) return;  // cannot happen: the host sized S from the exact raw count of the window
  const float4 p = pool[i];
  st[i] |= ST_DEAD;
  s_pts[d] = p;
  keys[d] = filter_key_of(p, d, g, rank_of_cube, inv_leaf);
  vals[d] = d;
}

// Front of the end-of-sweep update in ONE cluster launch (S <= CS_MAX_N): [INSERT: store_insert_kernel's points and
// filter keys of the stack] -> stable sort by filter key (cluster_sort, radix_sort_pairs' four passes) -> voxel run
// heads.  It leaves what the multi-launch front (store_insert_kernel, radix_sort_pairs, voxel_head_kernel +
// radix_scan_kernel) leaves for store_voxel_merge_kernel: the sorted (key, index) pairs in place over keys / vals, and
// pos[i] = heads before i | head flag << 31, here as global ranks with block_off[0..nb] = 0.  Without INSERT the
// unsorted S is read from keys / vals (raw seed points joined it, store_raw_select_scatter_kernel).
template <bool INSERT>
__global__ void __cluster_dims__(CS_CL, 1, 1) __launch_bounds__(CS_THREADS)
store_front_cluster_kernel(const float4* __restrict__ stack_ds, int n, MapIterArgs a, CubeGrid g,
                           const unsigned char* __restrict__ rank_of_cube, float inv_leaf, ShardSpec sh,
                           float4* __restrict__ s_pts, unsigned* keys, int* vals, unsigned* __restrict__ pos,
                           unsigned* __restrict__ block_off) {
  extern __shared__ __align__(16) unsigned char cs_raw[];
  ClusterSortSmem& sm = *reinterpret_cast<ClusterSortSmem*>(cs_raw);
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned my = cluster.block_rank();
  const int per = (n + CS_CL - 1) / CS_CL;
  const int m_local = cs_local_count(n, per, my);
  const int g0 = (int)my * per;
  for (int i = threadIdx.x; i < m_local; i += CS_THREADS) {
    const int gi = g0 + i;
    if (INSERT) {
      const float4 q = stack_ds[gi];
      float x, y, z;
      associate_to_map(a, q, x, y, z);
      const float4 p = make_float4(x, y, z, q.w);
      s_pts[gi] = p;
      sm.keys[0][i] = shard_stores(sh, store_cell(p.x)) ? filter_key_of(p, gi, g, rank_of_cube, inv_leaf)
                                                        : (((unsigned)CLS_DROP << 24) | ((unsigned)gi & 0xffffffu));
      sm.vals[0][i] = gi;
    } else {
      sm.keys[0][i] = keys[gi];
      sm.vals[0][i] = vals[gi];
    }
  }
  if (my == 0)
    for (int b = threadIdx.x; b <= (n + SCAN_BS - 1) / SCAN_BS; b += CS_THREADS) block_off[b] = 0;
  __syncthreads();
  const int cur = cluster_sort(sm, n, per, 4);

  // heads before every element inside this CTA (block scan in rounds, as voxel_filter_cluster_kernel), kept in the
  // sort's spare value buffer with the head flag in bit 31 -> exchange the CTA totals -> global ranks
  auto key_at = [&](int gi) -> unsigned {
    const int r = gi / per;
    return cluster.map_shared_rank(&sm.keys[cur][0], r)[gi - r * per];
  };
  unsigned* rank_in_cta = reinterpret_cast<unsigned*>(&sm.vals[cur ^ 1][0]);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned carry = 0;
  for (int base = 0; base < m_local; base += CS_THREADS) {
    const int i = base + threadIdx.x;
    const bool head = i < m_local && (g0 + i == 0 || sm.keys[cur][i] != (i > 0 ? sm.keys[cur][i - 1] : key_at(g0 - 1)));
    const unsigned bal = __ballot_sync(0xffffffffu, head);
    if (lane == 0) sm.wsum[warp] = __popc(bal);
    __syncthreads();
    unsigned woff = 0, round_total = 0;
    for (int w = 0; w < CS_NW; w++) {
      const unsigned c = sm.wsum[w];
      if (w < warp) woff += c;
      round_total += c;
    }
    if (i < m_local) rank_in_cta[i] = (carry + woff + __popc(bal & ((1u << lane) - 1u))) | (head ? 1u << 31 : 0u);
    carry += round_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) sm.scal[0] = carry;
  cluster.sync();
  unsigned cta_base = 0;
  for (unsigned r = 0; r < my; r++) cta_base += cluster.map_shared_rank(&sm.scal[0], r)[0];
  for (int i = threadIdx.x; i < m_local; i += CS_THREADS) {
    keys[g0 + i] = sm.keys[cur][i];
    vals[g0 + i] = sm.vals[cur][i];
    pos[g0 + i] = rank_in_cta[i] + cta_base;
  }
  cluster.sync();  // nobody leaves while a neighbour may still read its shared memory
}

// One thread per voxel run of the sorted S.  Visible voxel: centroid over [the filtered map points already in that
// voxel (found through the cell table, marked DEAD), then the run's points in sorted order] -> one filtered point.
// Invisible cube: the (single) point goes to the map unfiltered.  Every emitted point also gets its cell key.
// n_runs_out (optional): the number of runs that are emitted (runs outside the grid, class 0xFF, sort last and are cut
// off), written by the last element below them -- what runs_below_kernel computes, without a launch of its own.
__global__ void store_voxel_merge_kernel(const float4* __restrict__ s_pts, const unsigned* __restrict__ s_keys,
                                         const int* __restrict__ s_vals, const unsigned* __restrict__ pos,
                                         const unsigned* __restrict__ block_off, int n_s, MapGridView pool,
                                         unsigned char* __restrict__ pool_state, float inv_leaf, float leaf,
                                         float4* __restrict__ e_pts, unsigned char* __restrict__ e_state,
                                         unsigned* __restrict__ e_keys, int* __restrict__ e_vals,
                                         int* __restrict__ n_runs_out = nullptr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_s) return;
  const unsigned pv = pos[i];
  if (n_runs_out) {
    constexpr unsigned CUT = (unsigned)CLS_DROP << 24;
    const unsigned ki = s_keys[i];
    if (ki < CUT && (i + 1 == n_s || s_keys[i + 1] >= CUT))
      *n_runs_out = (int)((pv & 0x7fffffffu) + block_off[i / SCAN_BS] + (pv >> 31));
    else if (i == 0 && ki >= CUT)
      *n_runs_out = 0;
  }
  if (!(pv >> 31)) return;
  const unsigned dst = (pv & 0x7fffffffu) + block_off[i / SCAN_BS];
  const unsigned k = s_keys[i];
  const unsigned cls = k >> 24;
  if (cls == CLS_DROP) return;
  const float4 q0 = s_pts[s_vals[i]];
  if (cls == CLS_KEEP) {
    e_pts[dst] = q0;
    e_state[dst] = ST_RAW;
    e_keys[dst] = torus_key_of(q0);
    e_vals[dst] = (int)dst;
    return;
  }
  const float fvx = floorf(q0.x * inv_leaf), fvy = floorf(q0.y * inv_leaf), fvz = floorf(q0.z * inv_leaf);
  const CellAxis qx = cell_axis(store_cell(q0.x), CUBE_W), qy = cell_axis(store_cell(q0.y), CUBE_H),
                 qz = cell_axis(store_cell(q0.z), CUBE_D);
  float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
  int cnt = 0;
  // cells the voxel can overlap (a margin covers the rounding of x * inv_leaf)
  const float mx = 1e-3f + 1e-6f * fabsf(fvx * leaf), my = 1e-3f + 1e-6f * fabsf(fvy * leaf), mz = 1e-3f + 1e-6f * fabsf(fvz * leaf);
  const int cx0 = (int)floorf(fvx * leaf - mx), cx1 = (int)floorf((fvx + 1.f) * leaf + mx);
  const int cy0 = (int)floorf(fvy * leaf - my), cy1 = (int)floorf((fvy + 1.f) * leaf + my);
  const int cz0 = (int)floorf(fvz * leaf - mz), cz1 = (int)floorf((fvz + 1.f) * leaf + mz);
  for (int cz = cz0; cz <= cz1; cz++) {
    const CellAxis z = cell_axis(cz, CUBE_D);
    if (z.a != qz.a) continue;
    for (int cy = cy0; cy <= cy1; cy++) {
      const CellAxis y = cell_axis(cy, CUBE_H);
      if (y.a != qy.a) continue;
      for (int cx = cx0; cx <= cx1; cx++) {
        const CellAxis x = cell_axis(cx, CUBE_W);
        if (x.a != qx.a) continue;  // pcl filters cube by cube: a voxel never merges across a cube face
        unsigned start = 0, count = 0;
        if (!store_probe(pool, torus_key(x, y, z), start, count, nullptr)) continue;
        // four points of the cell's run per step: the loads are issued together (the byte store below may alias anything
        // as far as the compiler knows, so a plain loop became one dependent load per point: 39 us for ~20 k voxels),
        // evaluated in order -- the summation order is unchanged
        for (unsigned j0 = start; j0 < start + count; j0 += 4) {
          unsigned char st4[4];
          float4 p4[4];
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const unsigned j = j0 + u;
            const bool in = j < start + count;
            st4[u] = in ? pool_state[j] : (unsigned char)ST_DEAD;
            p4[u] = in ? __ldg(&pool.pts[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int u = 0; u < 4; u++) {
            if (st4[u] & (ST_RAW | ST_DEAD)) continue;
            const float4 p = p4[u];
            if (floorf(p.x * inv_leaf) == fvx && floorf(p.y * inv_leaf) == fvy && floorf(p.z * inv_leaf) == fvz) {
              sx += p.x; sy += p.y; sz += p.z; si += p.w;
              cnt++;
              pool_state[j0 + u] = st4[u] | ST_DEAD;
            }
          }
        }
      }
    }
  }
  for (int u = i; u < n_s && s_keys[u] == k; u++) {
    const float4 q = s_pts[s_vals[u]];
    sx += q.x; sy += q.y; sz += q.z; si += q.w;
    cnt++;
  }
  const float fn = (float)cnt;
  const float4 c = make_float4(sx / fn, sy / fn, sz / fn, si / fn);
  e_pts[dst] = c;
  e_state[dst] = 0;
  e_keys[dst] = torus_key_of(c);
  e_vals[dst] = (int)dst;
}

// what store_index_kernel fills in: cleared by the pass before the merge instead of by memsets of their own
struct IndexClear {
  uint4* table = nullptr;
  unsigned table_n = 0;
  int* stats = nullptr;  // cube_stats, 3 x CUBE_NUM
  int* n_cells = nullptr;
};

// pool elements that survive the sweep: not replaced, and (after a roll of the grid) still inside it
template <bool CHECK_GRID>
__global__ void __launch_bounds__(SCAN_BS)
store_live_count_kernel(const float4* __restrict__ pts, const unsigned char* __restrict__ st, int n,
                        const int* __restrict__ n_dev, CubeGrid g, unsigned* __restrict__ local_pos,
                        unsigned* __restrict__ block_sums, IndexClear clr = IndexClear{}) {
  __shared__ unsigned ws[32];
  if (clr.table) {  // (the voxel merge, the last reader of the old table, ran before this kernel)
    const unsigned t = blockIdx.x * SCAN_BS + threadIdx.x, stride = gridDim.x * SCAN_BS;
    for (unsigned j = t; j < clr.table_n; j += stride) clr.table[j] = make_uint4(0u, 0u, 0u, 0u);
    for (unsigned j = t; j < 3u * CUBE_NUM; j += stride) clr.stats[j] = 0;
    if (t == 0) *clr.n_cells = 0;
  }
  if (n_dev) n = min(n, *n_dev);
  const int i = blockIdx.x * SCAN_BS + threadIdx.x;
  bool live = i < n && !(st[i] & ST_DEAD);
  if (CHECK_GRID && live) {
    int ci, cj, ck;
    live = cube_index(pts[i], g, ci, cj, ck) >= 0;
  }
  const unsigned h = live ? 1u : 0u;
  unsigned x = h;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned y = __shfl_up_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) >= o) x += y;
  }
  if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
  __syncthreads();
  if (threadIdx.x < 32) {
    unsigned w = ws[threadIdx.x];
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned y = __shfl_up_sync(0xffffffffu, w, o);
      if (threadIdx.x >= o) w += y;
    }
    ws[threadIdx.x] = w;
  }
  __syncthreads();
  const unsigned incl = x + ((threadIdx.x >> 5) ? ws[(threadIdx.x >> 5) - 1] : 0u);
  if (i < n) local_pos[i] = (incl - h) | (h << 31);
  if (threadIdx.x == SCAN_BS - 1) block_sums[blockIdx.x] = incl;
}

__device__ __forceinline__ int lower_bound_u32(const unsigned* __restrict__ a, int lo, int hi, unsigned key) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ int upper_bound_u32(const unsigned* __restrict__ a, int lo, int hi, unsigned key) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] <= key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// merge of two sequences sorted by cell key: live pool elements keep their relative order and precede the new points
// of the same cell.  Threads [0, np_bound) handle pool elements, threads [np_bound, np_bound + ne_bound) new points.
constexpr int MERGE_BS = 256;
__global__ void __launch_bounds__(MERGE_BS)
store_merge_kernel(const float4* __restrict__ p_pts, const unsigned* __restrict__ p_keys,
                   const unsigned char* __restrict__ p_state, const unsigned* __restrict__ live_pos,
                   const unsigned* __restrict__ live_boff, int np_bound, const int* __restrict__ np_dev,
                   const int* __restrict__ live_total_dev, const float4* __restrict__ e_pts,
                   const unsigned* __restrict__ e_keys, const int* __restrict__ e_order,
                   const unsigned char* __restrict__ e_state, int ne_bound, const int* __restrict__ ne_dev,
                   float4* __restrict__ o_pts, unsigned* __restrict__ o_keys, unsigned char* __restrict__ o_state,
                   int* __restrict__ n_out_dev) {
  const int np = min(np_bound, *np_dev), ne = min(ne_bound, *ne_dev), live_total = *live_total_dev;
  const int pool_blocks = (np_bound + MERGE_BS - 1) / MERGE_BS;
  if ((int)blockIdx.x < pool_blocks) {
    // the block's keys span [k_first, k_last]: search the new points once per block, then inside that window
    __shared__ int s_lo, s_hi;
    const int b0 = blockIdx.x * MERGE_BS;
    if (b0 >= np) return;
    if (threadIdx.x == 0) {
      const int b1 = min(b0 + MERGE_BS, np) - 1;
      s_lo = lower_bound_u32(e_keys, 0, ne, p_keys[b0]);
      s_hi = lower_bound_u32(e_keys, s_lo, ne, p_keys[b1]);
    }
    __syncthreads();
    const int i = b0 + threadIdx.x;
    if (i >= np) return;
    const unsigned pv = live_pos[i];
    if (!(pv >> 31)) return;
    const unsigned key = p_keys[i];
    const int lb = lower_bound_u32(e_keys, s_lo, s_hi, key);
    const int dst = (int)((pv & 0x7fffffffu) + live_boff[i / SCAN_BS]) + lb;
    o_pts[dst] = p_pts[i];
    o_keys[dst] = key;
    o_state[dst] = p_state[i];
  } else {
    const int j = ((int)blockIdx.x - pool_blocks) * MERGE_BS + threadIdx.x;
    if (j == 0) *n_out_dev = live_total + ne;
    if (j >= ne) return;
    const unsigned key = e_keys[j];
    const int ub = upper_bound_u32(p_keys, 0, np, key);
    const int live_before = ub < np ? (int)((live_pos[ub] & 0x7fffffffu) + live_boff[ub / SCAN_BS]) : live_total;
    const int dst = j + live_before;
    const int src = e_order[j];
    o_pts[dst] = e_pts[src];
    o_keys[dst] = key;
    o_state[dst] = e_state[src];
  }
}

// grid_insert_kernel and store_stats_kernel over the merged pool in one pass: cell table entries (linear probing),
// occupied cells -> *n_cells, per cube slot [start, end) and raw count.  Table, stats and *n_cells start zeroed.
__global__ void store_index_kernel(const unsigned* __restrict__ keys, const unsigned char* __restrict__ st, int n,
                                   const int* __restrict__ n_dev, uint4* __restrict__ table, unsigned mask,
                                   int* __restrict__ n_cells, int* __restrict__ cube_start, int* __restrict__ cube_end,
                                   int* __restrict__ cube_raw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (n_dev) n = min(n, *n_dev);
  const bool in = i < n;
  const unsigned k = in ? keys[i] : 0u;
  const unsigned slot = in ? (k >> 17) : 0xffffffffu;
  const bool head = in && (i == 0 || keys[i - 1] != k);
  if (in) {
    if (i == 0 || (keys[i - 1] >> 17) != slot) cube_start[slot] = i;
    if (i == n - 1 || (keys[i + 1] >> 17) != slot) cube_end[slot] = i + 1;
  }
  const bool raw = in && (st[i] & ST_RAW);
  const unsigned peers = __match_any_sync(0xffffffffu, raw ? slot : 0xfffffffeu);
  if (raw && (peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0) atomicAdd(&cube_raw[slot], __popc(peers));
  const int heads = __syncthreads_count(head ? 1 : 0);
  if (threadIdx.x == 0 && heads > 0) atomicAdd(n_cells, heads);
  if (!head) return;
  int cnt = 1;
  while (i + cnt < n && keys[i + cnt] == k) cnt++;
  unsigned h = grid_hash(k) & mask;
  for (unsigned tries = 0; tries <= mask; tries++) {  // bounded, as in grid_insert_kernel
    const unsigned prev = atomicCAS(&table[h].x, 0u, k + 1u);
    if (prev == 0u) {
      table[h].y = (unsigned)i;
      table[h].z = (unsigned)cnt;
      return;
    }
    h = (h + 1) & mask;
  }
}

// slot-indexed view of the window table: 1 when the cube that currently owns the slot is in the field of view
__global__ void store_valid_by_slot_kernel(const unsigned char* __restrict__ rank_of_cube, int n_valid, CubeGrid g,
                                           unsigned char* __restrict__ valid_by_slot) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= CUBE_NUM) return;
  const int i = idx % CUBE_W, j = (idx / CUBE_W) % CUBE_H, k = idx / (CUBE_W * CUBE_H);
  const int slot = pmod_i(i - g.cen_w, CUBE_W) + CUBE_W * (pmod_i(j - g.cen_h, CUBE_H) + CUBE_H * pmod_i(k - g.cen_d, CUBE_D));
  valid_by_slot[slot] = ((int)rank_of_cube[idx] < n_valid) ? 1 : 0;
}

}  // namespace loamb
