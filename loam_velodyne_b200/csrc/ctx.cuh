// Context, device-buffer management and launch bookkeeping for libloam_b200.so.
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cfloat>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/loam_b200.h"

namespace loamb {

// While a thread records an enqueue sequence by stream capture (run_captured, loam_b200.cu) the kernels it has "launched"
// have not run yet: a buffer that grows in the middle of the sequence must not be freed under them.  The recording thread
// points this at a list; buffers replaced during the recording are parked there and freed once the graph has executed.
inline thread_local std::vector<void*>* tl_deferred_free = nullptr;
inline void free_device_buffer(void* q) {
  if (tl_deferred_free) tl_deferred_free->push_back(q);
  else cudaFree(q);
}

// growable device allocation (never shrinks; geometric growth so steady-state sweeps allocate nothing)
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    size_t want = cap ? cap : 256;
    while (want < n) want = 2 * want + 256;  // a reallocation synchronises the device: keep them rare (180 GB of HBM)
    if (p) free_device_buffer(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc((void**)&p, want * sizeof(T));
    if (e == cudaSuccess) cap = want;
    return e;
  }
  // grow while preserving the first `keep` elements (stream-ordered device copy)
  cudaError_t reserve_keep(size_t n, size_t keep, cudaStream_t st) {
    if (n <= cap) return cudaSuccess;
    size_t want = cap ? cap : 256;
    while (want < n) want = 2 * want + 256;
    T* q = nullptr;
    cudaError_t e = cudaMalloc((void**)&q, want * sizeof(T));
    if (e != cudaSuccess) return e;
    if (p && keep) {
      e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) { cudaFree(q); return e; }
      cudaStreamSynchronize(st);
    }
    if (p) cudaFree(p);
    p = q;
    cap = want;
    return cudaSuccess;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

// pinned host staging buffer
template <typename T>
struct PinBuf {
  T* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    size_t want = cap ? cap : 256;
    while (want < n) want = want + want / 2 + 256;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMallocHost((void**)&p, want * sizeof(T));
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

// 64-byte BVH node: both child boxes + child links, one 64 B aligned read per visit.
// child < 0  ->  leaf, leaf id = ~child
struct __align__(16) BvhNode {
  float4 lo0;  // child0 min xyz, w = bit pattern of child0 link
  float4 hi0;  // child0 max xyz, w = bit pattern of child1 link
  float4 lo1;  // child1 min xyz
  float4 hi1;  // child1 max xyz
};

struct Tree {
  int m = 0;        // points
  int n_leaf = 0;   // leaves (LEAF_SIZE consecutive Morton-sorted points each)
  int root = 0;     // root link (>= 0 internal node, < 0 leaf)
  DevBuf<float4> pts;      // original order (xyz, intensity) when the tree owns its points
  const float4* ext_pts = nullptr;  // ... or a cloud slot's buffer (device-resident stage API)
  const float4* points() const { return ext_pts ? ext_pts : pts.p; }
  DevBuf<float4> sorted;   // Morton order (xyz, original index as int bits)
  DevBuf<BvhNode> nodes;   // n_leaf - 1 internal nodes
  DevBuf<uint32_t> leaf_key;
  DevBuf<int> parent;      // parent of internal node i / of leaf (stored at n_leaf-1+leaf)
  DevBuf<int> flags;
  DevBuf<float4> box_lo, box_hi;  // per-node total boxes during refit (internal then leaves)
};

struct FeatSlots { int cap_sharp = 0, cap_less = 0, cap_flat = 0; };
struct CubeGridHost { int cen_w = 10, cen_h = 5, cen_d = 10; };

struct GridMetaHost { int v[6]; };
struct Grid {            // uniform 1 m grid over a map cloud (gridnn.cuh)
  int m = 0;
  unsigned mask = 0;
  DevBuf<uint4> table;
  DevBuf<float4> sorted;
  DevBuf<GridMetaHost> meta;
};

// pre-instantiated CUDA graph of a device-resident Gauss-Newton loop: gate kernel -> WHILE { iteration kernels, step }
struct LoopGraph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  unsigned long long handle = 0;  // cudaGraphConditionalHandle of the WHILE node
  int cap_a = 0, cap_b = 0;       // query capacities (corner-like, surface-like) the kernel grids were sized for
  int variant = -1;               // which kernel instantiation the body holds
  const void* baked[4] = {nullptr, nullptr, nullptr, nullptr};  // device buffers whose addresses sit in the nodes
  long long builds = 0;
  void destroy() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    exec = nullptr;
    graph = nullptr;
    handle = 0;
  }
};

// A fixed sequence of enqueues (kernels, memsets, copies, fork / join events) that a stage issues every sweep with slightly
// different arguments.  Instead of submitting the calls one by one, the sequence is recorded by stream capture, the
// resident executable graph is updated in place (cudaGraphExecUpdate: same topology, new arguments) and launched with ONE
// submission.  tools/probes/capture_update.cu on B200, 30 small kernels per sequence: 40.7 -> 15.7 us of host time
// alone, 85.9 -> 37.8 us with three threads issuing concurrently (the streaming pipeline), and the kernels run back to
// back on the GPU (98 -> 55 us per sequence).  A changed topology (a branch taken for the first time) re-instantiates.
struct CapturedSeq {
  cudaGraphExec_t exec = nullptr;
  long long launches = 0, rebuilds = 0;
  std::vector<void*> parked;      // device buffers replaced while a sequence was being recorded ...
  cudaEvent_t parked_ev = nullptr;  // ... free once the launch that may still read them has finished
  void free_parked(bool wait) {
    if (parked.empty()) return;
    if (parked_ev) {
      if (wait) cudaEventSynchronize(parked_ev);
      else if (cudaEventQuery(parked_ev) != cudaSuccess) { cudaGetLastError(); return; }
    }
    for (void* q : parked) cudaFree(q);
    parked.clear();
  }
  void destroy() {
    free_parked(true);
    if (parked_ev) cudaEventDestroy(parked_ev);
    parked_ev = nullptr;
    if (exec) cudaGraphExecDestroy(exec);
    exec = nullptr;
  }
};

struct SortScratch {
  DevBuf<uint32_t> keys_a, keys_b;
  DevBuf<int> vals_a, vals_b;
  DevBuf<uint32_t> hist;
};

}  // namespace loamb

// One helper thread per context for work whose ISSUE time (tens of launches) would otherwise sit on the caller's critical
// path although nothing waits for its result: the end-of-sweep map update (28 launches, ~70 us of host time) is posted
// here and the caller returns at once; every later API call on the context first waits for the job (async_join).
struct AsyncWorker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<int()> job;
  bool has_job = false, busy = false, stop = false;
  int last_rc = 0;
};

struct loam_b200_ctx {
  int device = 0;
  int sm_count = 0;
  AsyncWorker* worker = nullptr;
  loam_b200_ctx* aux = nullptr;       // auxiliary context of the asynchronous surround cloud (stages.inc)
  bool surround_in_aux = false;
  bool cluster_ok = false;  // single-launch cluster kernels of clustersort.cuh usable (LOAM_B200_NO_CLUSTER=1 disables)
  cudaStream_t stream = nullptr;
  cudaStream_t main_stream = nullptr;  // == stream outside LaneScope; the copy other threads may read (never swapped)
  std::string last_error;
  long long launches = 0;

  // profiling
  bool prof_on = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double prof_ms[LOAM_B200_NUM_KERNEL_FAMILIES] = {0};
  long long prof_launches[LOAM_B200_NUM_KERNEL_FAMILIES] = {0};
  int prof_family = -1;
  long long prof_launches_at_begin = 0;

  // multi-GPU: query slice of this rank and the NCCL communicator (comm.inc)
  void* comm = nullptr;
  int shard_rank = 0, shard_world = 1;
  // multi-GPU, cube-sharded map (peer.inc): slab width in cells (0 = off), this rank's inbox (slots + flags + the
  // reduction counter, one allocation) and the peers' inboxes mapped through CUDA IPC
  int shard_slab = 0;
  unsigned* peer_inbox = nullptr;
  void* peer_mapped[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool peer_is_ipc[8] = {false, false, false, false, false, false, false, false};  // opened with cudaIpcOpenMemHandle
  bool peer_ready = false;

  // scan registration
  loamb::DevBuf<float4> reg_pts;
  loamb::DevBuf<int> reg_ring_start, reg_ring_end;
  loamb::DevBuf<int> reg_picks;        // per ring: sharp | less sharp | flat slots
  loamb::DevBuf<int> reg_counts;       // per ring: n_sharp, n_less_sharp, n_flat, n_less_flat_ds
  loamb::DevBuf<int8_t> reg_label;
  loamb::DevBuf<float4> reg_lessflat;  // per ring slots of voxel-filtered less-flat points
  loamb::PinBuf<unsigned char> stage;  // generic pinned staging
  loamb::PinBuf<unsigned char> stage2;

  // trees
  loamb::Tree tree[LOAM_B200_NUM_TREES];
  loamb::Grid grid[2];  // corner / surface surrounding map
  loamb::SortScratch sort;
  loamb::DevBuf<float> bbox;  // 6 floats (encoded) for the tree build
  loamb::DevBuf<float4> knn_q;
  loamb::DevBuf<int> knn_idx;
  loamb::DevBuf<float> knn_d2;

  // mapping
  loamb::DevBuf<float4> map_q;  // corner queries then surf queries (kernel-level API: loam_b200_map_set_queries)
  const float4* map_q_corner = nullptr;  // where the kernels read the queries: map_q, or the two down-sized stack clouds
  const float4* map_q_surf = nullptr;    // of the stage API (no copy)
  int map_nc = 0, map_ns = 0;
  loamb::DevBuf<float> partials;   // per-block partial normal equations
  loamb::DevBuf<float> result;     // 36 floats
  loamb::DevBuf<unsigned int> ticket;
  loamb::DevBuf<unsigned long long> walk_totals;
  loamb::DevBuf<float4> dbg_coeff;
  loamb::DevBuf<int8_t> dbg_sel;
  loamb::PinBuf<float> result_host;
  loamb::PinBuf<float> result_mailbox;   // mapped pinned memory the iteration kernels post their sums to (ResultMailbox)
  int result_seq = 0;
  loamb::PinBuf<int> int_mailbox;        // same for small integer results (stage counts); [511] = sequence
  int int_seq = 0;
  loamb::PinBuf<int> ring_table_host;
  loamb::DevBuf<float> bin_xyz;           // raw xyz of the ring-binning front end (frontend.cuh)
  loamb::DevBuf<unsigned char> lm_state;  // OdomLmState + MapLmState (lmstep.cuh): pose of the device-resident loops
  loamb::LoopGraph odom_loop, map_loop;   // their loop graphs (loam_b200_odom_solve / loam_b200_map_solve)
  loamb::CapturedSeq seq_features, seq_begin_sweep, seq_end_sweep, seq_rebuild;  // per-sweep enqueue sequences (run_captured)
  // While a stream records, cudaDeviceSynchronize() from ANY thread of the process fails (CUDA cannot wait for a recording
  // stream).  Sequences recorded inside a blocking API call are safe for single-threaded callers; the end-of-sweep update
  // runs on the helper thread while the caller is back in its own code, so it is only recorded when the caller opted in
  // (loam_b200_allow_async_capture: the streaming pipeline, whose users synchronise through loam_b200_pipeline_sync).
  bool async_capture_ok = false;
  // map_iterate_v2_kernel (persistent, warp-specialised, bulk-staged candidates): persistent grid per instantiation
  // [store / bounding-box lookup][stage API / device loop] for the candidate capacity in use, 0 = not yet queried
  int map_v2_grid[2][2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};
  bool map_v2_off = false;

  // odometry
  loamb::DevBuf<float4> od_q;  // sharp then flat
  int od_nsharp = 0, od_nflat = 0;
  loamb::DevBuf<int> od_ind;   // (n_sharp + n_flat) x 3 persisted correspondence indices
  bool od_last_set = false;
  bool od_rebuild_pending = false;
  int od_rebuild_lanes = 2;    // side lanes the pending rebuild runs on
  bool od_prepared = false;    // od_q already holds this sweep's queries (loam_b200_odom_adopt)
  loamb::DevBuf<int> od_ring_off[2];  // ring offset tables of the last corner / surface clouds (odometry_lm.cuh)

  // device-resident clouds of the stage API
  loamb::DevBuf<float4> cloud[LOAM_B200_NUM_CLOUDS];
  int cloud_n[LOAM_B200_NUM_CLOUDS] = {0};
  int reg_totals[4] = {0, 0, 0, 0};
  int reg_n_rings = 0, reg_n = 0;
  loamb::FeatSlots reg_slots;
  // map pools: class per point, cube tables, scratch
  loamb::DevBuf<unsigned char> pool_cls[2];
  loamb::DevBuf<unsigned char> rank_of_cube;
  // persistent cell-sorted map (mapstore.cuh): cloud[POOL_SLOT[k]] holds the points, these the parallel arrays;
  // the *_alt buffers receive the merged pool of a sweep and are swapped in
  struct MapStore {
    loamb::DevBuf<uint32_t> keys, keys_alt;
    loamb::DevBuf<unsigned char> state, state_alt;
    loamb::DevBuf<float4> pts_alt;
    loamb::DevBuf<uint4> table;
    unsigned mask = 0;
    loamb::DevBuf<int> cube_stats;   // [3][CUBE_NUM]: start, end, raw count per cube slot
    loamb::DevBuf<unsigned char> valid_by_slot;
    loamb::DevBuf<float4> s_pts, e_pts;            // this sweep's filter input / emitted points
    loamb::DevBuf<unsigned char> e_state;
    loamb::DevBuf<uint32_t> e_keys;                // cell keys of the emitted points (before sorting)
    loamb::DevBuf<int> e_vals;
    bool dirty = false;        // points were appended unsorted: rebuild before the next sweep
    bool check_grid = false;   // the next merge must drop points whose cube is outside the grid
    int n_raw_valid = 0;       // raw points in the cubes in view (exact, from begin_sweep's readback)
    int n_cells = -1;          // occupied cells of the current table (exact, same readback; -1 = not known)
    int n_slot = 0;            // which of the two device-side pool counters is current
    int last_cen[3] = {1 << 30, 0, 0};
  } store[2];
  bool map_use_store = false;      // scan-to-map search goes through the store (stage API) / through grid[] (kernel API)
  bool map_debug_from_map = false; // begin_sweep also materialises the from-map clouds (tests)
  bool split_map_update = false;   // every end-of-sweep update takes the multi-launch chain (LOAM_B200_SPLIT_MAP_UPDATE
                                   // at creation; the reference the single-cluster chain is tested against)
  loamb::DevBuf<float4> pool_tmp;
  loamb::DevBuf<unsigned char> pool_tmp_cls;
  loamb::DevBuf<unsigned> cmp_pos, cmp_bsum;
  loamb::DevBuf<int> dcount;          // device-side element counts (stage API keeps sizes on the GPU between kernels)
  loamb::PinBuf<int> hcount;          // their pinned host mirror (one readback per stage)
  loamb::PinBuf<unsigned char> cube_table_host;
  loamb::CubeGridHost map_grid;
  int map_n_valid = 0;
  float map_leaf[2] = {0.2f, 0.4f};
  // The end-of-sweep map update runs on its own stream (lane 3) so that the next sweep's hand-off and stack filters do not
  // queue behind it: it starts after ev_loop_done (the loop of its sweep, main stream), and whatever reads the map next
  // waits for ev_update first (async_join orders the main stream behind it; begin_sweep does so only after its filters).
  cudaEvent_t ev_loop_done = nullptr, ev_update = nullptr;
  bool update_pending = false;
  loamb::DevBuf<float4> stack_alt[2];            // the two down-sized stacks are double-buffered (the update of sweep k
  loamb::DevBuf<unsigned char> rank_of_cube_alt;  // still reads them / the cube table while sweep k + 1 writes its own)
  cudaEvent_t ev_xfer = nullptr;
  cudaEvent_t ev_table = nullptr;
  bool ev_table_pending = false;

  // extra lanes: independent pieces of a stage (corner / surface kind, stack filter / map grid) run concurrently on
  // their own stream with their own scratch; LaneScope swaps a lane's stream + scratch into the fields above
  struct Lane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    loamb::SortScratch sort;
    loamb::DevBuf<float> bbox;
    loamb::DevBuf<uint32_t> vox_key;
    loamb::DevBuf<unsigned> cmp_pos, cmp_bsum;
    loamb::DevBuf<float4> tmp_pts, tmp_pts2, pool_tmp;
  };
  static constexpr int NUM_LANES = 3;   // lanes 1..3 (lane 0 = the context's own stream and scratch)
  Lane lanes[NUM_LANES];
  cudaEvent_t ev_fork = nullptr;

  // generic scratch
  loamb::DevBuf<float4> tmp_pts;
  loamb::DevBuf<float4> tmp_pts2;
  loamb::DevBuf<uint32_t> vox_key;
  loamb::DevBuf<int> vox_val;
  loamb::DevBuf<int> vox_scalars;
};

namespace loamb {

inline int fail_cuda(loam_b200_ctx* c, cudaError_t e, const char* what, int line) {
  char buf[512];
  snprintf(buf, sizeof buf, "%s failed at line %d: %s", what, line, cudaGetErrorString(e));
  if (c) c->last_error = buf;
  cudaGetLastError();  // clear sticky-less error state
  return LOAM_B200_ERR_CUDA;
}

#define LB_CUDA(ctx, expr)                                                   \
  do {                                                                       \
    cudaError_t _e = (expr);                                                 \
    if (_e != cudaSuccess) return loamb::fail_cuda(ctx, _e, #expr, __LINE__); \
  } while (0)

extern std::atomic<long long> g_total_launches;

#define LB_LAUNCH_CHECK(ctx)                                                            \
  do {                                                                                  \
    (ctx)->launches++;                                                                  \
    loamb::g_total_launches.fetch_add(1, std::memory_order_relaxed);                                                      \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) return loamb::fail_cuda(ctx, _e, "kernel launch", __LINE__); \
  } while (0)

// Run the enclosed calls on lane `i` (1..NUM_LANES; 0 = the context's own stream): swaps stream + scratch buffers in,
// and back out on destruction.  Callers fork / join the lanes with lanes_fork / lanes_join.
struct LaneScope {
  loam_b200_ctx* c;
  loam_b200_ctx::Lane* l;
  LaneScope(loam_b200_ctx* ctx, int i) : c(ctx), l(i > 0 ? &ctx->lanes[i - 1] : nullptr) { swap(); }
  ~LaneScope() { swap(); }
  void swap() {
    if (!l) return;
    std::swap(c->stream, l->stream);
    std::swap(c->sort, l->sort);
    std::swap(c->bbox, l->bbox);
    std::swap(c->vox_key, l->vox_key);
    std::swap(c->cmp_pos, l->cmp_pos);
    std::swap(c->cmp_bsum, l->cmp_bsum);
    std::swap(c->tmp_pts, l->tmp_pts);
    std::swap(c->tmp_pts2, l->tmp_pts2);
    std::swap(c->pool_tmp, l->pool_tmp);
  }
};
// every lane starts after everything enqueued so far on the main stream ...
inline cudaError_t lanes_fork(loam_b200_ctx* c, int n_lanes) {
  cudaError_t e = cudaEventRecord(c->ev_fork, c->stream);
  for (int i = 0; i < n_lanes && e == cudaSuccess; i++) e = cudaStreamWaitEvent(c->lanes[i].stream, c->ev_fork, 0);
  return e;
}
// one particular lane (1-based) forked from / joined into the current stream
inline cudaError_t lane_fork_one(loam_b200_ctx* c, int lane) {
  cudaError_t e = cudaEventRecord(c->ev_fork, c->stream);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(c->lanes[lane - 1].stream, c->ev_fork, 0);
  return e;
}
inline cudaError_t lane_join_one(loam_b200_ctx* c, int lane) {
  cudaError_t e = cudaEventRecord(c->lanes[lane - 1].done, c->lanes[lane - 1].stream);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(c->stream, c->lanes[lane - 1].done, 0);
  return e;
}
// ... and the main stream continues after all of them
inline cudaError_t lanes_join(loam_b200_ctx* c, int n_lanes) {
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < n_lanes && e == cudaSuccess; i++) {
    e = cudaEventRecord(c->lanes[i].done, c->lanes[i].stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c->stream, c->lanes[i].done, 0);
  }
  return e;
}

// RAII-less profiling bracket: begin/end around a family's kernels on the ctx stream
inline void prof_begin(loam_b200_ctx* c, int family) {
  if (!c->prof_on) return;
  c->prof_family = family;
  c->prof_launches_at_begin = c->launches;
  cudaEventRecord(c->ev0, c->stream);
}
inline void prof_end(loam_b200_ctx* c) {
  if (!c->prof_on || c->prof_family < 0) return;
  cudaEventRecord(c->ev1, c->stream);
  cudaEventSynchronize(c->ev1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev0, c->ev1);
  c->prof_ms[c->prof_family] += ms;
  c->prof_launches[c->prof_family] += c->launches - c->prof_launches_at_begin;
  c->prof_family = -1;
}

}  // namespace loamb
