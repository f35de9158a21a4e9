// libloam_b200.so -- extern "C" entry points (include/loam_b200.h) over the sm_100a kernels.
// There is no CPU fallback anywhere in this file: without a CUDA device every compute entry point fails loudly.
#include <atomic>
#include <chrono>
#include <cmath>

#include "ctx.cuh"
#include "features.cuh"
#include "lbvh.cuh"
#include "mapping_lm.cuh"
#include "odometry_lm.cuh"
#include "voxel.cuh"
#include "mappool.cuh"
#include "clustersort.cuh"
#include "mapstore.cuh"
#include "frontend.cuh"

using namespace loamb;

namespace loamb {
std::atomic<long long> g_total_launches{0};  // helper threads launch too
}

// every entry point first waits for the context's helper thread (ctx.cuh: AsyncWorker) and reports its status
static int async_join(loam_b200_ctx* c, bool order = true);
#define CHECK_CTX(c)                      \
  if (!(c)) return LOAM_B200_ERR_ARG;     \
  {                                       \
    const int _rcj = async_join(c);       \
    if (_rcj) return _rcj;                \
  }
// ... without ordering the main stream behind a pending map update (entry points that do not read the map first)
#define CHECK_CTX_NO_ORDER(c)             \
  if (!(c)) return LOAM_B200_ERR_ARG;     \
  {                                       \
    const int _rcj = async_join(c, false);\
    if (_rcj) return _rcj;                \
  }

namespace {

inline int blocks_for(long long n, int bs) { return (int)((n + bs - 1) / bs); }

TreeView view_of(const Tree& t) {
  TreeView v;
  v.nodes = t.nodes.p;
  v.sorted = t.sorted.p;
  v.m = t.m;
  v.n_leaf = t.n_leaf;
  v.root = t.root;
  return v;
}

}  // namespace

namespace loamb {
// radix sort (keys, vals) of length m in ctx->sort (input in keys_a / vals_a); 8 bits per pass.  The sorted arrays are
// returned through keys_out / vals_out (buffer a after an even number of passes, b after an odd one).
template <int ITEMS>
static int radix_sort_launch(loam_b200_ctx* c, int m, int passes, const int* n_dev, unsigned*& ka, int*& va, unsigned*& kb,
                             int*& vb) {
  SortScratch& s = c->sort;
  const int n_tiles = blocks_for(m, RS_THREADS * ITEMS);
  LB_CUDA(c, s.hist.reserve((size_t)RS_HEADER + (size_t)passes * n_tiles * 256));
  unsigned* header = s.hist.p;
  unsigned* status = s.hist.p + RS_HEADER;
  LB_CUDA(c, cudaMemsetAsync(header, 0, RS_HEADER * sizeof(unsigned), c->stream));
  onesweep_hist_kernel<ITEMS><<<n_tiles, RS_THREADS, 0, c->stream>>>(ka, m, n_dev, passes, header, status, n_tiles);
  LB_LAUNCH_CHECK(c);
  for (int p = 0; p < passes; p++) {
    onesweep_pass_kernel<ITEMS><<<n_tiles, RS_THREADS, 0, c->stream>>>(
        ka, va, m, n_dev, 8 * p, header + p * 256, status + (size_t)p * n_tiles * 256, header + RS_MAX_PASSES * 256 + p,
        kb, vb);
    LB_LAUNCH_CHECK(c);
    std::swap(ka, kb);
    std::swap(va, vb);
  }
  return LOAM_B200_OK;
}

// LSD radix sort of (keys_a, vals_a) in c->sort, m = launch bound, live count = min(m, *n_dev) when n_dev is given
// (elements past it are left alone).  Sorted arrays are returned through the out params; callers that read buffer a
// directly get an even number of passes.
int radix_sort_pairs(loam_b200_ctx* c, int m, int key_bits, unsigned** keys_out, int** vals_out, const int* n_dev) {
  SortScratch& s = c->sort;
  unsigned *ka = s.keys_a.p, *kb = s.keys_b.p;
  int *va = s.vals_a.p, *vb = s.vals_b.p;
  int passes = std::min((key_bits + 7) / 8, RS_MAX_PASSES);
  if (!keys_out && (passes & 1)) passes++;
  if (cluster_path_ok(c, m)) {
    // small array: the whole sort is one cluster launch (clustersort.cuh), sorted in place
    cluster_sort_pairs_kernel<<<CS_CL, CS_THREADS, sizeof(ClusterSortSmem), c->stream>>>(ka, va, m, n_dev, passes, ka, va);
    LB_LAUNCH_CHECK(c);
  } else if (m > 0) {
    const int rc = rs_items_for(m) == 4 ? radix_sort_launch<4>(c, m, passes, n_dev, ka, va, kb, vb)
                                        : radix_sort_launch<16>(c, m, passes, n_dev, ka, va, kb, vb);
    if (rc) return rc;
  }
  if (keys_out) *keys_out = ka;
  if (vals_out) *vals_out = va;
  return LOAM_B200_OK;
}

bool cluster_path_ok(const loam_b200_ctx* c, int n) { return c->cluster_ok && n > 0 && n <= CS_MAX_N; }

int voxel_filter_cluster(loam_b200_ctx* c, const float4* d_in, int n, float leaf, const void* roundtrip, float4* d_tmp,
                         float4* d_out, int* d_count) {
  const float inv = 1.0f / leaf;
  if (roundtrip) {
    voxel_filter_cluster_kernel<true><<<CS_CL, CS_THREADS, sizeof(ClusterSortSmem), c->stream>>>(
        d_in, n, inv, *static_cast<const MapIterArgs*>(roundtrip), d_tmp, d_out, d_count);
  } else {
    voxel_filter_cluster_kernel<false><<<CS_CL, CS_THREADS, sizeof(ClusterSortSmem), c->stream>>>(
        d_in, n, inv, MapIterArgs{}, nullptr, d_out, d_count);
  }
  LB_LAUNCH_CHECK(c);
  return LOAM_B200_OK;
}

}  // namespace loamb

namespace {

GridView grid_view_of(const Grid& g) {
  GridView v;
  v.table = g.table.p;
  v.mask = g.mask;
  v.sorted = g.sorted.p;
  v.meta = reinterpret_cast<const GridMeta*>(g.meta.p);
  v.m = g.m;
  return v;
}

MapCellLookup store_lookup_of(const loam_b200_ctx* c, int kind) {
  const auto& st = c->store[kind];
  MapCellLookup lk;
  lk.g = MapGridView{st.table.p, st.mask, c->cloud[kind == 0 ? LOAM_B200_C_MAP_CORNER_POOL : LOAM_B200_C_MAP_SURF_POOL].p,
                     c->rank_of_cube.p, c->map_grid.cen_w, c->map_grid.cen_h, c->map_grid.cen_d, c->map_n_valid};
  lk.ax = lk.ay = lk.az = CellAxis{0, 0, 0};
  lk.prune = (long long)c->cloud_n[LOAM_B200_C_MAP_CORNER_POOL] + c->cloud_n[LOAM_B200_C_MAP_SURF_POOL] > 4000000 ? 1 : 0;
  return lk;
}

// 1 m uniform grid over d_pts: the search structure of the scan-to-map loop (gridnn.cuh).  m is the launch bound; when
// n_dev is given the live count is read on the device (no host round trip after the compaction that produced it).
int grid_build_device(loam_b200_ctx* c, Grid& g, const float4* d_pts, int m, const int* n_dev = nullptr) {
  g.m = m;
  if (m <= 0) return LOAM_B200_OK;
  SortScratch& s = c->sort;
  LB_CUDA(c, s.keys_a.reserve(m));
  LB_CUDA(c, s.keys_b.reserve(m));
  LB_CUDA(c, s.vals_a.reserve(m));
  LB_CUDA(c, s.vals_b.reserve(m));
  LB_CUDA(c, c->bbox.reserve(8));
  LB_CUDA(c, g.sorted.reserve(m));
  LB_CUDA(c, g.meta.reserve(1));
  size_t tsize = 1024;
  while (tsize < 2 * (size_t)m) tsize <<= 1;  // occupied cells <= points: load factor <= 0.5 (typically ~0.08), probes always end
  LB_CUDA(c, g.table.reserve(tsize));
  g.mask = (unsigned)(tsize - 1);
  LB_CUDA(c, cudaMemsetAsync(g.table.p, 0, tsize * sizeof(uint4), c->stream));
  unsigned* bb = reinterpret_cast<unsigned*>(c->bbox.p);
  GridMeta* meta = reinterpret_cast<GridMeta*>(g.meta.p);
  bbox_init_kernel<<<1, 32, 0, c->stream>>>(bb);
  LB_LAUNCH_CHECK(c);
  const int bbox_blocks = std::min(blocks_for(m, 256), c->sm_count * 2);
  bbox_kernel<<<bbox_blocks, 256, 0, c->stream>>>(d_pts, m, bb, n_dev);
  LB_LAUNCH_CHECK(c);
  grid_meta_kernel<<<1, 32, 0, c->stream>>>(bb, meta);
  LB_LAUNCH_CHECK(c);
  grid_key_kernel<<<blocks_for(m, 256), 256, 0, c->stream>>>(d_pts, m, meta, s.keys_a.p, s.vals_a.p, n_dev);
  LB_LAUNCH_CHECK(c);
  unsigned* keys = nullptr;
  int* vals = nullptr;
  int rc = radix_sort_pairs(c, m, 32, &keys, &vals, n_dev);  // keys < 1290^3 < 2^31: the top pass is usually a copy
  if (rc) return rc;
  gather_sorted_kernel<<<blocks_for(m, 256), 256, 0, c->stream>>>(d_pts, vals, m, g.sorted.p, n_dev);
  LB_LAUNCH_CHECK(c);
  grid_insert_kernel<<<blocks_for(m, 256), 256, 0, c->stream>>>(keys, m, g.table.p, g.mask, n_dev);
  LB_LAUNCH_CHECK(c);
  return LOAM_B200_OK;
}

// ring offset tables of the odometry's last-sweep clouds (odometry_lm.cuh: ring_offsets_kernel); both live in one buffer
int* ring_off_ptr(loam_b200_ctx* c, int kind) { return c->od_ring_off[0].p ? c->od_ring_off[0].p + kind * RING_OFF_WORDS : nullptr; }
int odom_ring_offsets(loam_b200_ctx* c, int kind, const float4* d_pts, int m) {
  LB_CUDA(c, c->od_ring_off[0].reserve(2 * RING_OFF_WORDS));
  LB_CUDA(c, cudaMemsetAsync(ring_off_ptr(c, kind), 0, RING_OFF_WORDS * sizeof(int), c->stream));
  if (m > 0) {
    ring_offsets_kernel<<<blocks_for(m, 256), 256, 0, c->stream>>>(d_pts, m, ring_off_ptr(c, kind));
    LB_LAUNCH_CHECK(c);
  }
  return LOAM_B200_OK;
}
// ... of both clouds: one memset + one launch
int odom_ring_offsets_pair(loam_b200_ctx* c, const float4* p0, int m0, const float4* p1, int m1) {
  LB_CUDA(c, c->od_ring_off[0].reserve(2 * RING_OFF_WORDS));
  LB_CUDA(c, cudaMemsetAsync(c->od_ring_off[0].p, 0, 2 * RING_OFF_WORDS * sizeof(int), c->stream));
  const int m = std::max(m0, m1);
  if (m > 0) {
    ring_offsets_kernel<<<dim3(blocks_for(m, 256), 2), 256, 0, c->stream>>>(p0, m0, ring_off_ptr(c, 0), p1, m1, ring_off_ptr(c, 1));
    LB_LAUNCH_CHECK(c);
  }
  return LOAM_B200_OK;
}

// buffers of a tree over m points (no scratch of the multi-launch build)
int tree_reserve(loam_b200_ctx* c, Tree& t, int m) {
  t.m = m;
  t.n_leaf = 0;
  t.root = 0;
  if (m <= 0) return LOAM_B200_OK;
  const int n_leaf = (m + LEAF_SIZE - 1) / LEAF_SIZE;
  t.n_leaf = n_leaf;
  LB_CUDA(c, t.sorted.reserve(m));
  LB_CUDA(c, t.nodes.reserve(n_leaf > 1 ? n_leaf - 1 : 1));
  LB_CUDA(c, t.leaf_key.reserve(n_leaf));
  LB_CUDA(c, t.parent.reserve(2 * (size_t)n_leaf));
  LB_CUDA(c, t.flags.reserve(n_leaf));
  LB_CUDA(c, t.box_lo.reserve(2 * (size_t)n_leaf));
  LB_CUDA(c, t.box_hi.reserve(2 * (size_t)n_leaf));
  return LOAM_B200_OK;
}
BvhBuildArgs bvh_args_of(const Tree& t) {
  return BvhBuildArgs{t.points(), t.m, t.n_leaf, t.sorted.p, t.leaf_key.p, t.nodes.p, t.parent.p, t.box_lo.p, t.box_hi.p, t.flags.p};
}

// both trees of the odometry stage in ONE launch (two clusters); false when a cloud needs the multi-launch path
int tree_build_pair_cluster(loam_b200_ctx* c, Tree& t0, int m0, Tree& t1, int m1, bool* done) {
  *done = false;
  if (!cluster_path_ok(c, m0) || !cluster_path_ok(c, m1)) return LOAM_B200_OK;
  int rc = tree_reserve(c, t0, m0);
  if (rc == LOAM_B200_OK) rc = tree_reserve(c, t1, m1);
  if (rc) return rc;
  bvh_build_cluster_kernel<<<2 * CS_CL, CS_THREADS, sizeof(ClusterSortSmem), c->stream>>>(bvh_args_of(t0), bvh_args_of(t1));
  LB_LAUNCH_CHECK(c);
  t0.root = t0.n_leaf == 1 ? ~0 : 0;
  t1.root = t1.n_leaf == 1 ? ~0 : 0;
  *done = true;
  return LOAM_B200_OK;
}

// build the BVH of tree t from t.pts (device, m points)
int tree_build_device(loam_b200_ctx* c, Tree& t, int m) {
  int rc0 = tree_reserve(c, t, m);
  if (rc0) return rc0;
  if (m <= 0) return LOAM_B200_OK;
  const int n_leaf = t.n_leaf;
  if (cluster_path_ok(c, m)) {
    BvhBuildArgs none{};
    bvh_build_cluster_kernel<<<CS_CL, CS_THREADS, sizeof(ClusterSortSmem), c->stream>>>(bvh_args_of(t), none);
    LB_LAUNCH_CHECK(c);
    t.root = n_leaf == 1 ? ~0 : 0;
    return LOAM_B200_OK;
  }
  SortScratch& s = c->sort;
  LB_CUDA(c, s.keys_a.reserve(m));
  LB_CUDA(c, s.keys_b.reserve(m));
  LB_CUDA(c, s.vals_a.reserve(m));
  LB_CUDA(c, s.vals_b.reserve(m));
  LB_CUDA(c, c->bbox.reserve(8));
  unsigned* bb = reinterpret_cast<unsigned*>(c->bbox.p);
  bbox_init_kernel<<<1, 32, 0, c->stream>>>(bb);
  LB_LAUNCH_CHECK(c);
  const int bbox_blocks = std::min(blocks_for(m, 256), c->sm_count * 2);
  bbox_kernel<<<bbox_blocks, 256, 0, c->stream>>>(t.points(), m, bb);
  LB_LAUNCH_CHECK(c);
  morton_kernel<<<blocks_for(m, 256), 256, 0, c->stream>>>(t.points(), m, bb, s.keys_a.p, s.vals_a.p);
  LB_LAUNCH_CHECK(c);
  int rc = radix_sort_pairs(c, m, 30);
  if (rc) return rc;
  gather_sorted_kernel<<<blocks_for(m, 256), 256, 0, c->stream>>>(t.points(), s.vals_a.p, m, t.sorted.p);
  LB_LAUNCH_CHECK(c);
  leaf_kernel<<<blocks_for(n_leaf, 256), 256, 0, c->stream>>>(t.sorted.p, s.keys_a.p, m, n_leaf, t.leaf_key.p,
                                                              t.box_lo.p, t.box_hi.p, t.flags.p);
  LB_LAUNCH_CHECK(c);
  if (n_leaf == 1) {
    t.root = ~0;
    return LOAM_B200_OK;
  }
  karras_kernel<<<blocks_for(n_leaf - 1, 256), 256, 0, c->stream>>>(t.leaf_key.p, n_leaf, t.nodes.p, t.parent.p);
  LB_LAUNCH_CHECK(c);
  refit_kernel<<<blocks_for(n_leaf, 256), 256, 0, c->stream>>>(n_leaf, t.nodes.p, t.parent.p, t.box_lo.p, t.box_hi.p,
                                                               t.flags.p);
  LB_LAUNCH_CHECK(c);
  t.root = 0;
  return LOAM_B200_OK;
}

int upload_points(loam_b200_ctx* c, DevBuf<float4>& dst, const float* src, int n) {
  if (n <= 0) return LOAM_B200_OK;
  LB_CUDA(c, dst.reserve(n));
  LB_CUDA(c, cudaMemcpyAsync(dst.p, src, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
  return LOAM_B200_OK;
}

void fill_map_args(const loam_b200_pose* p, MapIterArgs& a) { map_args_from(p->sin_, p->cos_, p->pos, a); }

void fill_odom_args(const loam_b200_odom_pose* p, OdomIterArgs& a) {
  odom_args_from(p->rot, p->sin_, p->cos_, p->pos, p->inv_scan_period, p->iter, a);
}

// BVHs of the last clouds are rebuilt asynchronously on lane 1 (+ lane 2 on the multi-launch path)
cudaError_t odom_join_rebuild(loam_b200_ctx* c) {
  if (!c->od_rebuild_pending) return cudaSuccess;
  const int lanes = c->od_rebuild_lanes;
  c->od_rebuild_pending = false;
  return lanes_join(c, lanes);
}

static void unpack_normal_eq(const float* r, loam_b200_normal_eq* out) {
  int k = 0;
  for (int i = 0; i < 6; i++)
    for (int j = i; j < 6; j++) {
      out->AtA[i * 6 + j] = r[k];
      out->AtA[j * 6 + i] = r[k];
      k++;
    }
  for (int i = 0; i < 6; i++) out->AtB[i] = r[21 + i];
  out->n_selected = std::isfinite(r[27]) ? (int)(r[27] + 0.5f) : 0;
  out->n_corner_selected = std::isfinite(r[28]) ? (int)(r[28] + 0.5f) : 0;
}

bool getenv_no_mailbox() {
  static const bool off = getenv("LOAM_B200_NO_MAILBOX") != nullptr;
  return off;
}

// mailbox of the next iteration kernel: mapped pinned memory + a fresh sequence number (mapping_lm.cuh: ResultMailbox)
ResultMailbox next_mailbox(loam_b200_ctx* c) {
  if (c->result_mailbox.reserve(64) != cudaSuccess) {
    cudaGetLastError();
    return ResultMailbox{nullptr, 0};
  }
  c->result_seq = c->result_seq == 0x7fffffff ? 1 : c->result_seq + 1;
  return ResultMailbox{c->result_mailbox.p, c->result_seq};
}

// wait for the kernel launched with next_mailbox() to post its sums; falls back to a stream synchronise (which also
// surfaces launch failures) when nothing arrives for a long time
int fetch_normal_eq_mailbox(loam_b200_ctx* c, loam_b200_normal_eq* out) {
  volatile int* seq = reinterpret_cast<volatile int*>(c->result_mailbox.p + 32);
  const auto t0 = std::chrono::steady_clock::now();
  long long spins = 0;
  while (*seq != c->result_seq) {
    if ((++spins & 0xfff) == 0 &&
        std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 2.0) {
      LB_CUDA(c, cudaStreamSynchronize(c->stream));  // error or a very long kernel: by now the post is visible
      if (*seq != c->result_seq) return LOAM_B200_ERR_CUDA;
      break;
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  float r[NEQ];
  for (int i = 0; i < NEQ; i++) r[i] = reinterpret_cast<volatile float*>(c->result_mailbox.p)[i];
  unpack_normal_eq(r, out);
  return LOAM_B200_OK;
}

int fetch_normal_eq(loam_b200_ctx* c, loam_b200_normal_eq* out) {
  LB_CUDA(c, c->result_host.reserve(NEQ));
  LB_CUDA(c, cudaMemcpyAsync(c->result_host.p, c->result.p, NEQ * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  unpack_normal_eq(c->result_host.p, out);
  return LOAM_B200_OK;
}

// Small integer results (stage counts) take the same route as the normal equations: one 32-thread kernel behind the
// producers copies them into mapped host memory and posts a sequence number; the host spins (no memcpy + synchronise).
__global__ void post_ints_kernel(const int* __restrict__ src, int n, int* host, int seq) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) host[i] = src[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    *reinterpret_cast<volatile int*>(host + 511) = seq;
  }
}

int fetch_ints(loam_b200_ctx* c, const int* d_src, int n, int* h_dst) {
  if (n > 500 || getenv_no_mailbox() || c->int_mailbox.reserve(512) != cudaSuccess) {
    cudaGetLastError();
    LB_CUDA(c, c->hcount.reserve(512));
    LB_CUDA(c, cudaMemcpyAsync(c->hcount.p, d_src, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LB_CUDA(c, cudaStreamSynchronize(c->stream));
    if (h_dst != c->hcount.p) memcpy(h_dst, c->hcount.p, (size_t)n * sizeof(int));
    return LOAM_B200_OK;
  }
  c->int_seq = c->int_seq == 0x7fffffff ? 1 : c->int_seq + 1;
  post_ints_kernel<<<1, 32, 0, c->stream>>>(d_src, n, c->int_mailbox.p, c->int_seq);
  LB_LAUNCH_CHECK(c);
  volatile int* seq = reinterpret_cast<volatile int*>(c->int_mailbox.p + 511);
  const auto t0 = std::chrono::steady_clock::now();
  long long spins = 0;
  while (*seq != c->int_seq) {
    if ((++spins & 0xfff) == 0 && std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 2.0) {
      LB_CUDA(c, cudaStreamSynchronize(c->stream));
      if (*seq != c->int_seq) return LOAM_B200_ERR_CUDA;
      break;
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  for (int i = 0; i < n; i++) h_dst[i] = reinterpret_cast<volatile int*>(c->int_mailbox.p)[i];
  return LOAM_B200_OK;
}

// Run `body` (enqueues on c->stream and its lanes only: no host synchronisation, no waits on events of other contexts)
// through capture + update + one launch (ctx.cuh: CapturedSeq).  LOAM_B200_NO_CAPTURE=1 or profiling: direct enqueues.
static thread_local bool tl_in_worker = false;

template <typename F>
int run_captured(loam_b200_ctx* c, CapturedSeq& cs, F body) {
  static const bool off = getenv("LOAM_B200_NO_CAPTURE") != nullptr;
  if (off || c->prof_on || (tl_in_worker && !c->async_capture_ok)) return body();
  cudaStream_t origin = c->stream;
  cs.free_parked(false);  // buffers replaced during an earlier recording whose launch has finished by now
  LB_CUDA(c, cudaStreamBeginCapture(origin, cudaStreamCaptureModeRelaxed));
  std::vector<void*> replaced;
  tl_deferred_free = &replaced;  // DevBuf::reserve parks replaced buffers instead of freeing them under recorded kernels
  const int rc = body();
  tl_deferred_free = nullptr;
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(origin, &g);
  if (!replaced.empty()) {  // (also on the failure path below: an earlier launch may still read them)
    if (!cs.parked.empty()) cs.free_parked(true);  // rare: two growth steps in a row
    cs.parked.swap(replaced);
    if (!cs.parked_ev) cudaEventCreateWithFlags(&cs.parked_ev, cudaEventDisableTiming);
  }
  if (rc != LOAM_B200_OK || e != cudaSuccess || !g) {
    if (g) cudaGraphDestroy(g);
    cudaGetLastError();
    if (rc != LOAM_B200_OK) return rc;
    return fail_cuda(c, e == cudaSuccess ? cudaErrorUnknown : e, "cudaStreamEndCapture", __LINE__);
  }
  bool updated = false;
  if (cs.exec) {
    cudaGraphExecUpdateResultInfo info;
    if (cudaGraphExecUpdate(cs.exec, g, &info) == cudaSuccess) {
      updated = true;
    } else {  // the sequence took a different branch: instantiate anew (the parked buffers stay parked)
      cudaGetLastError();
      cudaGraphExecDestroy(cs.exec);
      cs.exec = nullptr;
    }
  }
  if (!updated) {
    const cudaError_t ei = cudaGraphInstantiate(&cs.exec, g, 0);
    if (ei != cudaSuccess) {
      cudaGraphDestroy(g);
      cs.exec = nullptr;
      return fail_cuda(c, ei, "cudaGraphInstantiate", __LINE__);
    }
    cs.rebuilds++;
  }
  const cudaError_t el = cudaGraphLaunch(cs.exec, origin);
  cudaGraphDestroy(g);
  if (el != cudaSuccess) return fail_cuda(c, el, "cudaGraphLaunch", __LINE__);
  if (!cs.parked.empty()) {
    if (!cs.parked_ev) cudaEventCreateWithFlags(&cs.parked_ev, cudaEventDisableTiming);
    cudaEventRecord(cs.parked_ev, origin);
  }
  cs.launches++;
  return LOAM_B200_OK;
}

}  // namespace

#include "comm.inc"
#include "peer.inc"

// the main stream continues behind the map update that runs on the update stream
static int order_after_update(loam_b200_ctx* c) {
  if (!c->update_pending) return LOAM_B200_OK;
  c->update_pending = false;
  LB_CUDA(c, cudaStreamWaitEvent(c->main_stream, c->ev_update, 0));
  return LOAM_B200_OK;
}

static int async_join(loam_b200_ctx* c, bool order) {
  AsyncWorker* w = c->worker;
  if (tl_in_worker) return LOAM_B200_OK;
  int rc = LOAM_B200_OK;
  if (w) {
    std::unique_lock<std::mutex> lk(w->m);
    w->cv.wait(lk, [w] { return !w->busy && !w->has_job; });
    rc = w->last_rc;
    w->last_rc = LOAM_B200_OK;
  }
  if (rc == LOAM_B200_OK && order) rc = order_after_update(c);
  return rc;
}

static void async_worker_main(loam_b200_ctx* c) {
  cudaSetDevice(c->device);
  tl_in_worker = true;
  AsyncWorker* w = c->worker;
  for (;;) {
    std::function<int()> job;
    {
      std::unique_lock<std::mutex> lk(w->m);
      w->cv.wait(lk, [w] { return w->has_job || w->stop; });
      if (w->stop && !w->has_job) return;
      job = std::move(w->job);
      w->has_job = false;
      w->busy = true;
    }
    const int rc = job();
    {
      std::lock_guard<std::mutex> lk(w->m);
      w->busy = false;
      if (rc) w->last_rc = rc;
    }
    w->cv.notify_all();
  }
}

// post a job; the previous one has been joined by the caller's CHECK_CTX
static int async_post(loam_b200_ctx* c, std::function<int()> job) {
  if (!c->worker) {
    c->worker = new AsyncWorker();
    c->worker->th = std::thread(async_worker_main, c);
  }
  AsyncWorker* w = c->worker;
  {
    std::lock_guard<std::mutex> lk(w->m);
    w->job = std::move(job);
    w->has_job = true;
  }
  w->cv.notify_all();
  return LOAM_B200_OK;
}

static void async_shutdown(loam_b200_ctx* c) {
  AsyncWorker* w = c->worker;
  if (!w) return;
  {
    std::unique_lock<std::mutex> lk(w->m);
    w->cv.wait(lk, [w] { return !w->busy && !w->has_job; });
    w->stop = true;
  }
  w->cv.notify_all();
  w->th.join();
  delete w;
  c->worker = nullptr;
}

extern "C" {

const char* loam_b200_strerror(int status) {
  switch (status) {
    case LOAM_B200_OK: return "ok";
    case LOAM_B200_ERR_ARG: return "invalid argument";
    case LOAM_B200_ERR_CUDA: return "CUDA error";
    case LOAM_B200_ERR_NO_DEVICE: return "no usable CUDA device (libloam_b200 has no CPU fallback)";
    case LOAM_B200_ERR_STATE: return "invalid call sequence";
    case LOAM_B200_ERR_CAPACITY: return "output capacity too small";
    case LOAM_B200_ERR_COMM: return "NCCL error";
  }
  return "unknown status";
}

const char* loam_b200_last_error(const loam_b200_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }
int loam_b200_version(void) { return 100; }

int loam_b200_create(loam_b200_ctx** out, int device) {
  if (!out || device < 0) return LOAM_B200_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device >= n) {
    cudaGetLastError();
    return LOAM_B200_ERR_NO_DEVICE;
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    cudaGetLastError();
    return LOAM_B200_ERR_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    cudaGetLastError();
    return LOAM_B200_ERR_NO_DEVICE;
  }
  if (prop.major != 10) return LOAM_B200_ERR_NO_DEVICE;  // kernels are built for sm_100a only
  loam_b200_ctx* c = new loam_b200_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_xfer, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_table, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_loop_done, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_update, cudaEventDisableTiming) != cudaSuccess) {
    cudaGetLastError();
    delete c;
    return LOAM_B200_ERR_CUDA;
  }
  c->main_stream = c->stream;
  bool lanes_ok = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess;
  for (auto& l : c->lanes)
    lanes_ok = lanes_ok && cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking) == cudaSuccess &&
               cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming) == cudaSuccess;
  if (!lanes_ok) {
    cudaGetLastError();
    delete c;
    return LOAM_B200_ERR_CUDA;
  }
  cudaFuncSetAttribute(feature_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (CS_CL > 8) {  // non-portable cluster size: opt in per kernel
    cudaFuncSetAttribute(voxel_filter_cluster_kernel<true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaFuncSetAttribute(voxel_filter_cluster_kernel<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaFuncSetAttribute(bvh_build_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaFuncSetAttribute(cluster_sort_pairs_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaFuncSetAttribute(store_front_cluster_kernel<true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaFuncSetAttribute(store_front_cluster_kernel<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  }
  c->split_map_update = getenv("LOAM_B200_SPLIT_MAP_UPDATE") != nullptr;
  c->cluster_ok = !getenv("LOAM_B200_NO_CLUSTER") &&
                  cudaFuncSetAttribute(voxel_filter_cluster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(ClusterSortSmem)) == cudaSuccess &&
                  cudaFuncSetAttribute(voxel_filter_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(ClusterSortSmem)) == cudaSuccess &&
                  cudaFuncSetAttribute(bvh_build_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(ClusterSortSmem)) == cudaSuccess &&
                  cudaFuncSetAttribute(cluster_sort_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(ClusterSortSmem)) == cudaSuccess &&
                  cudaFuncSetAttribute(store_front_cluster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(ClusterSortSmem)) == cudaSuccess &&
                  cudaFuncSetAttribute(store_front_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(ClusterSortSmem)) == cudaSuccess;
  cudaGetLastError();
  if (c->partials.reserve(4096 * NEQ) != cudaSuccess || c->result.reserve(NEQ) != cudaSuccess ||
      c->ticket.reserve(4) != cudaSuccess || c->result_host.reserve(NEQ) != cudaSuccess ||
      c->result_mailbox.reserve(64) != cudaSuccess || c->int_mailbox.reserve(512) != cudaSuccess) {
    cudaGetLastError();
    delete c;
    return LOAM_B200_ERR_CUDA;
  }
  cudaMemsetAsync(c->ticket.p, 0, 4 * sizeof(unsigned), c->stream);
  cudaStreamSynchronize(c->stream);
  *out = c;
  return LOAM_B200_OK;
}

int loam_b200_destroy(loam_b200_ctx* c) {
  if (!c) return LOAM_B200_ERR_ARG;
  if (c->aux) {
    loam_b200_destroy(c->aux);
    c->aux = nullptr;
  }
  async_shutdown(c);
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  c->reg_pts.release(); c->reg_ring_start.release(); c->reg_ring_end.release(); c->reg_picks.release();
  c->reg_counts.release(); c->reg_label.release(); c->reg_lessflat.release(); c->stage.release(); c->stage2.release();
  for (auto& t : c->tree) {
    t.pts.release(); t.sorted.release(); t.nodes.release(); t.leaf_key.release(); t.parent.release();
    t.flags.release(); t.box_lo.release(); t.box_hi.release();
  }
  c->sort.keys_a.release(); c->sort.keys_b.release(); c->sort.vals_a.release(); c->sort.vals_b.release();
  c->sort.hist.release();
  c->bbox.release(); c->knn_q.release(); c->knn_idx.release(); c->knn_d2.release();
  c->map_q.release(); c->partials.release(); c->result.release(); c->ticket.release(); c->walk_totals.release();
  for (auto& cl : c->cloud) cl.release();
  for (auto& g : c->grid) { g.table.release(); g.sorted.release(); g.meta.release(); }
  c->pool_cls[0].release(); c->pool_cls[1].release(); c->rank_of_cube.release(); c->pool_tmp.release();
  c->pool_tmp_cls.release(); c->cmp_pos.release(); c->cmp_bsum.release(); c->dcount.release(); c->hcount.release(); c->cube_table_host.release();
  for (auto& l : c->lanes) {
    if (l.stream) cudaStreamSynchronize(l.stream);
    l.sort.keys_a.release(); l.sort.keys_b.release(); l.sort.vals_a.release(); l.sort.vals_b.release(); l.sort.hist.release();
    l.bbox.release(); l.vox_key.release(); l.cmp_pos.release(); l.cmp_bsum.release();
    l.tmp_pts.release(); l.tmp_pts2.release(); l.pool_tmp.release();
    if (l.done) cudaEventDestroy(l.done);
    if (l.stream) cudaStreamDestroy(l.stream);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_xfer) cudaEventDestroy(c->ev_xfer);
  if (c->ev_table) cudaEventDestroy(c->ev_table);
  if (c->ev_loop_done) cudaEventDestroy(c->ev_loop_done);
  if (c->ev_update) cudaEventDestroy(c->ev_update);
  c->stack_alt[0].release(); c->stack_alt[1].release(); c->rank_of_cube_alt.release();
  for (auto& st : c->store) {
    st.keys.release(); st.keys_alt.release(); st.state.release(); st.state_alt.release(); st.pts_alt.release();
    st.table.release(); st.cube_stats.release(); st.valid_by_slot.release(); st.s_pts.release(); st.e_pts.release();
    st.e_state.release(); st.e_keys.release(); st.e_vals.release();
  }
  c->odom_loop.destroy();
  c->map_loop.destroy();
  c->seq_features.destroy(); c->seq_begin_sweep.destroy(); c->seq_end_sweep.destroy(); c->seq_rebuild.destroy();
  for (int p = 0; p < 8; p++)
    if (c->peer_mapped[p] && c->peer_is_ipc[p]) cudaIpcCloseMemHandle(c->peer_mapped[p]);
  if (c->peer_inbox) cudaFree(c->peer_inbox);
  if (c->comm) loam_b200_comm_destroy(c); c->dbg_coeff.release();
  c->dbg_sel.release(); c->result_host.release(); c->lm_state.release(); c->bin_xyz.release(); c->od_ring_off[0].release(); c->result_mailbox.release(); c->int_mailbox.release(); c->ring_table_host.release(); c->od_q.release(); c->od_ind.release(); c->tmp_pts.release();
  c->tmp_pts2.release(); c->vox_key.release(); c->vox_val.release(); c->vox_scalars.release();
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return LOAM_B200_OK;
}

int loam_b200_set_priority(loam_b200_ctx* c, int level) {
  CHECK_CTX(c);
  int least = 0, greatest = 0;  // numerically: greatest priority <= least priority
  LB_CUDA(c, cudaDeviceGetStreamPriorityRange(&least, &greatest));
  const int mid = (least + greatest) / 2;
  const int prio = level > 0 ? greatest : (level < 0 ? least : mid);
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaStream_t s = nullptr;
  LB_CUDA(c, cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, prio));
  cudaStreamDestroy(c->stream);
  c->stream = s;
  c->main_stream = s;
  // side lanes carry work nobody waits for immediately (tree rebuilds, the corner half of the map update): lowest
  for (auto& l : c->lanes) {
    cudaStream_t ls = nullptr;
    LB_CUDA(c, cudaStreamCreateWithPriority(&ls, cudaStreamNonBlocking, least));
    if (l.stream) { cudaStreamSynchronize(l.stream); cudaStreamDestroy(l.stream); }
    l.stream = ls;
  }
  return LOAM_B200_OK;
}

int loam_b200_allow_async_capture(loam_b200_ctx* c, int on) {
  CHECK_CTX(c);
  c->async_capture_ok = on != 0;
  return LOAM_B200_OK;
}

int loam_b200_bind_thread(int device) {
  if (device < 0 || cudaSetDevice(device) != cudaSuccess) {
    cudaGetLastError();
    return LOAM_B200_ERR_NO_DEVICE;
  }
  return LOAM_B200_OK;
}

int loam_b200_sync(loam_b200_ctx* c) {
  CHECK_CTX(c);
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  for (auto& l : c->lanes)
    if (l.stream) LB_CUDA(c, cudaStreamSynchronize(l.stream));
  if (c->aux) return loam_b200_sync(c->aux);  // asynchronous surround cloud
  return LOAM_B200_OK;
}

void* loam_b200_stream(loam_b200_ctx* c) { return c ? (void*)c->stream : nullptr; }

// ------------------------------------------------------------------------------------------------ features
// Shared by the host-buffer entry point and the device-resident stage: points are in d_pts (n), ring ranges on the
// host.  Results: dense index lists behind the per-ring slots of reg_picks, gathered feature clouds + less-flat DS in
// the REG_* cloud slots, labels in reg_label, totals in c->reg_totals (host, after one sync).
static int run_features(loam_b200_ctx* c, const float4* d_pts, int n, const int32_t* ring_start, const int32_t* ring_end,
                        int n_rings, const loam_b200_reg_params* prm) {
  if (prm->curvatureRegion < 1 || prm->curvatureRegion > 15 || prm->nFeatureRegions < 1 || prm->nFeatureRegions > 4095 ||
      prm->maxCornerSharp < 0 ||
      prm->maxCornerLessSharp < prm->maxCornerSharp || prm->maxSurfaceFlat < 0 || !(prm->lessFlatFilterSize > 0.f))
    return LOAM_B200_ERR_ARG;
  int max_ring = 0;
  for (int r = 0; r < n_rings; r++) {
    const long long s = ring_start[r], e = ring_end[r];
    if (s < 0 || e >= n || e < s - 1) {
      if (!(n == 0 && s == 0 && e == 0)) return LOAM_B200_ERR_ARG;
    }
    if (e >= s) max_ring = std::max(max_ring, (int)(e - s + 1));
  }
  for (int k = 0; k < 4; k++) c->reg_totals[k] = 0;
  c->reg_n = n;
  c->reg_n_rings = n_rings;
  c->cloud_n[LOAM_B200_C_REG_SHARP] = c->cloud_n[LOAM_B200_C_REG_LESS_SHARP] = 0;
  c->cloud_n[LOAM_B200_C_REG_FLAT] = c->cloud_n[LOAM_B200_C_REG_LESS_FLAT] = 0;
  if (n == 0) return LOAM_B200_OK;
  FeatParams fp;
  fp.nFeatureRegions = prm->nFeatureRegions;
  fp.curvatureRegion = prm->curvatureRegion;
  fp.maxCornerSharp = prm->maxCornerSharp;
  fp.maxCornerLessSharp = prm->maxCornerLessSharp;
  fp.maxSurfaceFlat = prm->maxSurfaceFlat;
  fp.lessFlatFilterSize = prm->lessFlatFilterSize;
  fp.surfaceCurvatureThreshold = prm->surfaceCurvatureThreshold;
  fp.cap_sharp = prm->nFeatureRegions * prm->maxCornerSharp;
  fp.cap_less = prm->nFeatureRegions * prm->maxCornerLessSharp;
  fp.cap_flat = prm->nFeatureRegions * prm->maxSurfaceFlat;
  c->reg_slots.cap_sharp = fp.cap_sharp;
  c->reg_slots.cap_less = fp.cap_less;
  c->reg_slots.cap_flat = fp.cap_flat;
  const int slots = fp.cap_sharp + fp.cap_less + fp.cap_flat;

  int ncap = (max_ring + 31) & ~31;
  if (ncap < 32) ncap = 32;
  int n2cap = 1;
  while (n2cap < ncap) n2cap <<= 1;
  const size_t smem = (size_t)ncap * (16 + 4 + 4 + 2) + (size_t)n2cap * 8;
  if (smem > 200 * 1024) return LOAM_B200_ERR_CAPACITY;  // ring longer than 5344 points (4096 < n: 8 B x 8192 sort keys)

  LB_CUDA(c, c->reg_ring_start.reserve(n_rings));
  LB_CUDA(c, c->reg_ring_end.reserve(n_rings));
  LB_CUDA(c, c->reg_picks.reserve((size_t)n_rings * slots * 2 + 16));
  LB_CUDA(c, c->reg_counts.reserve((size_t)n_rings * 4 + 8));
  LB_CUDA(c, c->reg_label.reserve(n));
  LB_CUDA(c, c->reg_lessflat.reserve(n));
  LB_CUDA(c, c->cloud[LOAM_B200_C_REG_SHARP].reserve((size_t)n_rings * fp.cap_sharp + 1));
  LB_CUDA(c, c->cloud[LOAM_B200_C_REG_LESS_SHARP].reserve((size_t)n_rings * fp.cap_less + 1));
  LB_CUDA(c, c->cloud[LOAM_B200_C_REG_FLAT].reserve((size_t)n_rings * fp.cap_flat + 1));
  LB_CUDA(c, c->cloud[LOAM_B200_C_REG_LESS_FLAT].reserve(n));
  // ring table through a context-owned pinned buffer (the previous use finished: every run ends with a result fetch)
  LB_CUDA(c, c->ring_table_host.reserve(2 * (size_t)n_rings));
  memcpy(c->ring_table_host.p, ring_start, (size_t)n_rings * 4);
  memcpy(c->ring_table_host.p + n_rings, ring_end, (size_t)n_rings * 4);
  int* dense = c->reg_picks.p + (size_t)n_rings * slots;
  int* totals = c->reg_counts.p + (size_t)n_rings * 4;
  prof_begin(c, LOAM_B200_K_FEATURES);
  {
    const int rcs = run_captured(c, c->seq_features, [&]() -> int {
      LB_CUDA(c, cudaMemcpyAsync(c->reg_ring_start.p, c->ring_table_host.p, n_rings * 4, cudaMemcpyHostToDevice, c->stream));
      LB_CUDA(c, cudaMemcpyAsync(c->reg_ring_end.p, c->ring_table_host.p + n_rings, n_rings * 4, cudaMemcpyHostToDevice, c->stream));
      feature_ring_kernel<<<n_rings, FEAT_THREADS, smem, c->stream>>>(d_pts, c->reg_ring_start.p, c->reg_ring_end.p, fp,
                                                                      ncap, n2cap, c->reg_picks.p, c->reg_counts.p,
                                                                      c->reg_label.p, c->reg_lessflat.p);
      LB_LAUNCH_CHECK(c);
      feature_pack_kernel<<<n_rings, 256, 0, c->stream>>>(
          c->reg_counts.p, c->reg_picks.p, c->reg_ring_start.p, d_pts, c->reg_lessflat.p, n_rings, fp, dense,
          dense + (size_t)n_rings * fp.cap_sharp, dense + (size_t)n_rings * (fp.cap_sharp + fp.cap_less),
          c->cloud[LOAM_B200_C_REG_SHARP].p, c->cloud[LOAM_B200_C_REG_LESS_SHARP].p, c->cloud[LOAM_B200_C_REG_FLAT].p,
          c->cloud[LOAM_B200_C_REG_LESS_FLAT].p, totals);
      LB_LAUNCH_CHECK(c);
      return LOAM_B200_OK;
    });
    if (rcs) return rcs;
  }
  prof_end(c);
  {
    const int rcf = fetch_ints(c, totals, 4, c->reg_totals);
    if (rcf) return rcf;
  }
  c->cloud_n[LOAM_B200_C_REG_SHARP] = c->reg_totals[0];
  c->cloud_n[LOAM_B200_C_REG_LESS_SHARP] = c->reg_totals[1];
  c->cloud_n[LOAM_B200_C_REG_FLAT] = c->reg_totals[2];
  c->cloud_n[LOAM_B200_C_REG_LESS_FLAT] = c->reg_totals[3];
  return LOAM_B200_OK;
}

static const int* reg_dense_list(loam_b200_ctx* c, int which) {
  const int slots = c->reg_slots.cap_sharp + c->reg_slots.cap_less + c->reg_slots.cap_flat;
  const int* dense = c->reg_picks.p + (size_t)c->reg_n_rings * slots;
  if (which == 1) return dense;
  if (which == 2) return dense + (size_t)c->reg_n_rings * c->reg_slots.cap_sharp;
  return dense + (size_t)c->reg_n_rings * (c->reg_slots.cap_sharp + c->reg_slots.cap_less);
}

int loam_b200_extract_features(loam_b200_ctx* c, const float* pts, int n, const int32_t* ring_start,
                               const int32_t* ring_end, int n_rings, const loam_b200_reg_params* prm,
                               loam_b200_features* out) {
  CHECK_CTX(c);
  if (!pts || n < 0 || !ring_start || !ring_end || n_rings <= 0 || n_rings > 256 || !prm || !out)
    return LOAM_B200_ERR_ARG;
  out->n_sharp = out->n_less_sharp = out->n_flat = out->n_less_flat = 0;
  if (n > 0) {
    LB_CUDA(c, c->reg_pts.reserve(n));
    LB_CUDA(c, cudaMemcpyAsync(c->reg_pts.p, pts, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
  }
  int rc = run_features(c, c->reg_pts.p, n, ring_start, ring_end, n_rings, prm);
  if (rc) return rc;
  if (n == 0) return LOAM_B200_OK;
  const int* h_tot = c->reg_totals;
  out->n_sharp = h_tot[0];
  out->n_less_sharp = h_tot[1];
  out->n_flat = h_tot[2];
  out->n_less_flat = h_tot[3];
  if ((out->sharp_idx && h_tot[0] > out->sharp_cap) || (out->less_sharp_idx && h_tot[1] > out->less_sharp_cap) ||
      (out->flat_idx && h_tot[2] > out->flat_cap) || (out->less_flat_ds && h_tot[3] > out->less_flat_cap))
    return LOAM_B200_ERR_CAPACITY;
  if (out->sharp_idx && h_tot[0])
    LB_CUDA(c, cudaMemcpyAsync(out->sharp_idx, reg_dense_list(c, 1), h_tot[0] * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out->less_sharp_idx && h_tot[1])
    LB_CUDA(c, cudaMemcpyAsync(out->less_sharp_idx, reg_dense_list(c, 2), h_tot[1] * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out->flat_idx && h_tot[2])
    LB_CUDA(c, cudaMemcpyAsync(out->flat_idx, reg_dense_list(c, 3), h_tot[2] * 4, cudaMemcpyDeviceToHost, c->stream));
  if (out->label) LB_CUDA(c, cudaMemcpyAsync(out->label, c->reg_label.p, n, cudaMemcpyDeviceToHost, c->stream));
  if (out->less_flat_ds && h_tot[3])
    LB_CUDA(c, cudaMemcpyAsync(out->less_flat_ds, c->cloud[LOAM_B200_C_REG_LESS_FLAT].p, (size_t)h_tot[3] * 16,
                               cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  return LOAM_B200_OK;
}

// ------------------------------------------------------------------------------------------------ trees
int loam_b200_tree_build(loam_b200_ctx* c, int slot, const float* pts, int m) {
  CHECK_CTX(c);
  if (slot < 0 || slot >= LOAM_B200_NUM_TREES || m < 0 || (m > 0 && !pts)) return LOAM_B200_ERR_ARG;
  Tree& t = c->tree[slot];
  t.ext_pts = nullptr;
  int rc = upload_points(c, t.pts, pts, m);
  if (rc) return rc;
  prof_begin(c, LOAM_B200_K_TREE_BUILD);
  rc = tree_build_device(c, t, m);
  if (rc == LOAM_B200_OK && slot < LOAM_B200_TREE_MAP_CORNER) rc = odom_ring_offsets(c, slot, t.points(), m);
  // the scan-to-map kernels search the two map slots through the 1 m grid
  if (rc == LOAM_B200_OK && slot >= LOAM_B200_TREE_MAP_CORNER) {
    rc = grid_build_device(c, c->grid[slot - LOAM_B200_TREE_MAP_CORNER], t.points(), m);
    c->map_use_store = false;  // kernel-level API: the scan-to-map search uses this grid, not the persistent store
  }
  prof_end(c);
  if (rc) return rc;
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  return LOAM_B200_OK;
}

int loam_b200_tree_size(loam_b200_ctx* c, int slot) {
  if (!c || slot < 0 || slot >= LOAM_B200_NUM_TREES) return LOAM_B200_ERR_ARG;
  return c->tree[slot].m;
}

int loam_b200_tree_knn(loam_b200_ctx* c, int slot, const float* queries, int nq, int k, float max_d2,
                       int32_t* idx_out, float* d2_out) {
  CHECK_CTX(c);
  if (slot < 0 || slot >= LOAM_B200_NUM_TREES || nq < 0 || (nq > 0 && (!queries || !idx_out || !d2_out)) || k < 1 ||
      k > KNN_MAX)
    return LOAM_B200_ERR_ARG;
  if (nq == 0) return LOAM_B200_OK;
  int rc = upload_points(c, c->knn_q, queries, nq);
  if (rc) return rc;
  LB_CUDA(c, c->knn_idx.reserve((size_t)nq * k));
  LB_CUDA(c, c->knn_d2.reserve((size_t)nq * k));
  const TreeView tv = view_of(c->tree[slot]);
  const int bs = 128, nb = blocks_for(nq, bs);
  prof_begin(c, LOAM_B200_K_KNN);
  switch (k) {
#define KNN_CASE(K)                                                                                              \
  case K:                                                                                                        \
    knn_kernel<K><<<nb, bs, 0, c->stream>>>(tv, c->knn_q.p, nq, max_d2, c->knn_idx.p, c->knn_d2.p);              \
    break;
    KNN_CASE(1) KNN_CASE(2) KNN_CASE(3) KNN_CASE(4) KNN_CASE(5) KNN_CASE(6) KNN_CASE(7) KNN_CASE(8)
#undef KNN_CASE
  }
  LB_LAUNCH_CHECK(c);
  prof_end(c);
  LB_CUDA(c, cudaMemcpyAsync(idx_out, c->knn_idx.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaMemcpyAsync(d2_out, c->knn_d2.p, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  return LOAM_B200_OK;
}

// ------------------------------------------------------------------------------------------------ mapping
int loam_b200_map_set_queries(loam_b200_ctx* c, const float* corner, int n_corner, const float* surf, int n_surf) {
  CHECK_CTX(c);
  if (n_corner < 0 || n_surf < 0 || (n_corner > 0 && !corner) || (n_surf > 0 && !surf)) return LOAM_B200_ERR_ARG;
  LB_CUDA(c, c->map_q.reserve((size_t)n_corner + n_surf + 1));
  if (n_corner)
    LB_CUDA(c, cudaMemcpyAsync(c->map_q.p, corner, (size_t)n_corner * 16, cudaMemcpyHostToDevice, c->stream));
  if (n_surf)
    LB_CUDA(c, cudaMemcpyAsync(c->map_q.p + n_corner, surf, (size_t)n_surf * 16, cudaMemcpyHostToDevice, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  c->map_nc = n_corner;
  c->map_ns = n_surf;
  c->map_q_corner = c->map_q.p;
  c->map_q_surf = c->map_q.p + n_corner;
  return LOAM_B200_OK;
}

// map_iterate_v2_kernel: candidate capacity per query (points staged in shared memory) and the persistent grid.
// Sparse maps (the 0.2 / 0.4 m voxel lattice of a LOAM map holds ~63 candidates per query at 1 M points) take the small
// capacity = 4 CTAs per SM; maps beyond a few million points (~200 candidates per query) the large one.
static int map_v2_cap_index(const loam_b200_ctx* c) {
  const long long pts = (long long)c->cloud_n[LOAM_B200_C_MAP_CORNER_POOL] + c->cloud_n[LOAM_B200_C_MAP_SURF_POOL] +
                        (c->map_use_store ? 0 : (long long)c->grid[0].m + c->grid[1].m);
  return pts > 4000000 ? 1 : 0;
}
static const int MAP_V2_CAP[2] = {96, 224};
extern "C++" {
template <typename K>
static int map_v2_grid_of(loam_b200_ctx* c, K kernel, int& cached, int cap) {
  if (cached > 0) return cached;
  const size_t smem = (size_t)MAP_Q_PER_BLOCK * cap * sizeof(float4);
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, MAPV2_THREADS, smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    return 0;
  }
  cached = per_sm * c->sm_count;
  return cached;
}
}  // extern "C++"

static int map_iterate_impl(loam_b200_ctx* c, const loam_b200_pose* pose, loam_b200_normal_eq* out, float* coeff,
                            int8_t* selected, unsigned long long* walk_totals_host = nullptr) {
  CHECK_CTX(c);
  if (!pose || !out) return LOAM_B200_ERR_ARG;
  const int nc = c->map_nc, ns = c->map_ns;
  memset(out, 0, sizeof *out);
  if (nc + ns == 0) return LOAM_B200_OK;
  MapIterArgs a;
  fill_map_args(pose, a);
  // this rank's contiguous slice of each query kind (everything when not sharded, and with the cube-sharded map, where
  // every rank looks at every query and evaluates those whose transformed position falls into a cell it owns)
  const int W = c->shard_slab > 0 ? 1 : c->shard_world, R = c->shard_slab > 0 ? 0 : c->shard_rank;
  const int c0 = (int)((long long)nc * R / W), c1 = (int)((long long)nc * (R + 1) / W);
  const int s0 = (int)((long long)ns * R / W), s1 = (int)((long long)ns * (R + 1) / W);
  const int lc = c1 - c0, ls = s1 - s0;
  const int cb = blocks_for(lc, MAP_Q_PER_BLOCK), sb = blocks_for(ls, MAP_Q_PER_BLOCK);
  const int nb = std::max(cb + sb, 1);
  LB_CUDA(c, c->partials.reserve((size_t)nb * NEQ));
  const bool dbg = coeff != nullptr;
  const ShardSpec sh = shard_spec_of(c);
  const PeerReduce pr = peer_view_of(c);
  const bool use_mailbox = !c->comm && (c->shard_world == 1 || c->peer_ready) && !c->prof_on && !walk_totals_host &&
                           !getenv_no_mailbox();
  ResultMailbox mb{nullptr, 0};
  if (dbg) {
    LB_CUDA(c, c->dbg_coeff.reserve(nc + ns));
    LB_CUDA(c, c->dbg_sel.reserve(nc + ns));
    if (c->shard_world > 1) {
      LB_CUDA(c, cudaMemsetAsync(c->dbg_coeff.p, 0, (size_t)(nc + ns) * 16, c->stream));
      LB_CUDA(c, cudaMemsetAsync(c->dbg_sel.p, 0, (size_t)(nc + ns), c->stream));
    }
  }
  if (walk_totals_host) {
    LB_CUDA(c, c->walk_totals.reserve(2));
    LB_CUDA(c, cudaMemsetAsync(c->walk_totals.p, 0, 2 * sizeof(unsigned long long), c->stream));
    if (c->map_use_store)
      map_iterate_kernel<true><<<nb, MAP_THREADS, 0, c->stream>>>(
          store_lookup_of(c, 0), store_lookup_of(c, 1), c->map_q_corner, c->map_q_surf, nc, c0, lc, s0, ls, cb, a, c->partials.p, c->result.p,
          c->ticket.p, nullptr, nullptr, c->walk_totals.p);
    else
      map_iterate_kernel<true><<<nb, MAP_THREADS, 0, c->stream>>>(
          GridCellLookup{grid_view_of(c->grid[0])}, GridCellLookup{grid_view_of(c->grid[1])}, c->map_q_corner, c->map_q_surf, nc, c0, lc, s0, ls,
          cb, a, c->partials.p, c->result.p, c->ticket.p, nullptr, nullptr, c->walk_totals.p);
    LB_LAUNCH_CHECK(c);
    LB_CUDA(c, cudaMemcpyAsync(walk_totals_host, c->walk_totals.p, 2 * sizeof(unsigned long long),
                               cudaMemcpyDeviceToHost, c->stream));
  } else {
    // single GPU: the folding CTA posts the sums straight into mapped host memory (no memcpy + synchronise); with a
    // shard / communicator the all-reduce has to run first, so the result is fetched the classic way
    if (use_mailbox) mb = next_mailbox(c);
    // v2 (persistent, warp-specialised, cp.async.bulk staging) is kept as a measured alternative: on B200 it runs 42.9 us
    // against 29.7 us for the phase-split kernel at config 3 (profiles/r2_map_iterate_v2.md) -- 27 bulk copies of ~100 B per
    // query cost more than the loads they replace.  LOAM_B200_MAP_V2=1 selects it.
    static const bool use_v2 = getenv("LOAM_B200_MAP_V2") != nullptr;
    const int ci = map_v2_cap_index(c), cap = MAP_V2_CAP[ci];
    int grid_v2 = 0;
    if (use_v2 && !c->map_v2_off)
      grid_v2 = c->map_use_store ? map_v2_grid_of(c, map_iterate_v2_kernel<MapCellLookup, false>, c->map_v2_grid[1][0][ci], cap)
                                 : map_v2_grid_of(c, map_iterate_v2_kernel<GridCellLookup, false>, c->map_v2_grid[0][0][ci], cap);
    prof_begin(c, LOAM_B200_K_MAP_ITER);
    if (grid_v2 > 0) {
      const size_t smem = (size_t)MAP_Q_PER_BLOCK * cap * sizeof(float4);
      // balanced persistent grid: every CTA gets the same number of 32-query blocks (+-1)
      const int per_cta = (nb + grid_v2 - 1) / grid_v2;
      const int grid = (nb + per_cta - 1) / per_cta;
      if (c->map_use_store)
        map_iterate_v2_kernel<MapCellLookup, false><<<grid, MAPV2_THREADS, smem, c->stream>>>(
            store_lookup_of(c, 0), store_lookup_of(c, 1), c->map_q_corner, c->map_q_surf, nc, c0, lc, s0, ls, cb, nb, a, c->partials.p, c->result.p,
            c->ticket.p, dbg ? c->dbg_coeff.p : nullptr, dbg ? c->dbg_sel.p : nullptr, nullptr, mb, sh, pr, cap);
      else
        map_iterate_v2_kernel<GridCellLookup, false><<<grid, MAPV2_THREADS, smem, c->stream>>>(
            GridCellLookup{grid_view_of(c->grid[0])}, GridCellLookup{grid_view_of(c->grid[1])}, c->map_q_corner, c->map_q_surf, nc, c0, lc, s0, ls, cb,
            nb, a, c->partials.p, c->result.p, c->ticket.p, dbg ? c->dbg_coeff.p : nullptr, dbg ? c->dbg_sel.p : nullptr, nullptr,
            mb, sh, pr, cap);
    }
    else if (c->map_use_store)
      map_iterate_kernel<false><<<nb, MAP_THREADS, 0, c->stream>>>(
          store_lookup_of(c, 0), store_lookup_of(c, 1), c->map_q_corner, c->map_q_surf, nc, c0, lc, s0, ls, cb, a, c->partials.p, c->result.p,
          c->ticket.p, dbg ? c->dbg_coeff.p : nullptr, dbg ? c->dbg_sel.p : nullptr, nullptr, nullptr, mb, sh, pr);
    else
      map_iterate_kernel<false><<<nb, MAP_THREADS, 0, c->stream>>>(
          GridCellLookup{grid_view_of(c->grid[0])}, GridCellLookup{grid_view_of(c->grid[1])}, c->map_q_corner, c->map_q_surf, nc, c0, lc, s0, ls,
          cb, a, c->partials.p, c->result.p, c->ticket.p, dbg ? c->dbg_coeff.p : nullptr, dbg ? c->dbg_sel.p : nullptr,
          nullptr, nullptr, mb, sh, pr);
    LB_LAUNCH_CHECK(c);
    prof_end(c);
  }
  {
    const int rcc = allreduce_result(c);  // no-op without a communicator
    if (rcc) return rcc;
  }
  int rc = mb.host ? fetch_normal_eq_mailbox(c, out) : fetch_normal_eq(c, out);
  if (rc) return rc;
  if (c->peer_ready && c->shard_world > 1 && !std::isfinite(out->AtB[0] + out->AtA[0])) {
    // the fused all-reduce gives up (NaN sums) when a peer's contribution does not arrive within ~2 s
    c->last_error = "peer all-reduce timed out: a rank of the cube-sharded map did not run this iteration";
    return LOAM_B200_ERR_COMM;
  }
  if (dbg) {
    LB_CUDA(c, cudaMemcpyAsync(coeff, c->dbg_coeff.p, (size_t)(nc + ns) * 16, cudaMemcpyDeviceToHost, c->stream));
    if (selected)
      LB_CUDA(c, cudaMemcpyAsync(selected, c->dbg_sel.p, (size_t)(nc + ns), cudaMemcpyDeviceToHost, c->stream));
    LB_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return LOAM_B200_OK;
}

int loam_b200_map_iterate(loam_b200_ctx* c, const loam_b200_pose* pose, loam_b200_normal_eq* out) {
  return map_iterate_impl(c, pose, out, nullptr, nullptr);
}
int loam_b200_map_iterate_debug(loam_b200_ctx* c, const loam_b200_pose* pose, loam_b200_normal_eq* out, float* coeff,
                                int8_t* selected) {
  if (!coeff) return LOAM_B200_ERR_ARG;
  return map_iterate_impl(c, pose, out, coeff, selected);
}
int loam_b200_map_iterate_stats(loam_b200_ctx* c, const loam_b200_pose* pose, loam_b200_normal_eq* out,
                                unsigned long long* nodes_visited, unsigned long long* leaves_visited) {
  if (!nodes_visited || !leaves_visited) return LOAM_B200_ERR_ARG;
  unsigned long long tot[2] = {0, 0};
  int rc = map_iterate_impl(c, pose, out, nullptr, nullptr, tot);
  *nodes_visited = tot[0];
  *leaves_visited = tot[1];
  return rc;
}

// ------------------------------------------------------------------------------------------------ odometry
int loam_b200_odom_set_last(loam_b200_ctx* c, const float* corner, int n_corner, const float* surf, int n_surf) {
  CHECK_CTX(c);
  int rc = loam_b200_tree_build(c, LOAM_B200_TREE_ODOM_CORNER, corner, n_corner);
  if (rc) return rc;
  rc = loam_b200_tree_build(c, LOAM_B200_TREE_ODOM_SURF, surf, n_surf);
  if (rc) return rc;
  c->od_last_set = true;
  return LOAM_B200_OK;
}

int loam_b200_odom_set_current(loam_b200_ctx* c, const float* sharp, int n_sharp, const float* flat, int n_flat) {
  CHECK_CTX(c);
  if (n_sharp < 0 || n_flat < 0 || (n_sharp > 0 && !sharp) || (n_flat > 0 && !flat)) return LOAM_B200_ERR_ARG;
  LB_CUDA(c, c->od_q.reserve((size_t)n_sharp + n_flat + 1));
  LB_CUDA(c, c->od_ind.reserve(((size_t)n_sharp + n_flat + 1) * 3));
  if (n_sharp) LB_CUDA(c, cudaMemcpyAsync(c->od_q.p, sharp, (size_t)n_sharp * 16, cudaMemcpyHostToDevice, c->stream));
  if (n_flat)
    LB_CUDA(c, cudaMemcpyAsync(c->od_q.p + n_sharp, flat, (size_t)n_flat * 16, cudaMemcpyHostToDevice, c->stream));
  LB_CUDA(c, cudaMemsetAsync(c->od_ind.p, 0xff, ((size_t)n_sharp + n_flat + 1) * 3 * sizeof(int), c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  c->od_nsharp = n_sharp;
  c->od_nflat = n_flat;
  return LOAM_B200_OK;
}

static int odom_iterate_impl(loam_b200_ctx* c, const loam_b200_odom_pose* pose, loam_b200_normal_eq* out,
                             float* coeff, int8_t* selected, int32_t* ind) {
  CHECK_CTX(c);
  if (!pose || !out) return LOAM_B200_ERR_ARG;
  if (!c->od_last_set) return LOAM_B200_ERR_STATE;
  LB_CUDA(c, odom_join_rebuild(c));
  const int nsh = c->od_nsharp, nfl = c->od_nflat;
  memset(out, 0, sizeof *out);
  if (nsh + nfl == 0) return LOAM_B200_OK;
  OdomIterArgs a;
  fill_odom_args(pose, a);
  const Tree& tc = c->tree[LOAM_B200_TREE_ODOM_CORNER];
  const Tree& ts = c->tree[LOAM_B200_TREE_ODOM_SURF];
  a.n_last_corner = tc.m;
  a.n_last_surf = ts.m;
  const int cb = blocks_for(nsh, LM_THREADS), sb = blocks_for(nfl, LM_THREADS);
  const int nb = cb + sb;
  LB_CUDA(c, c->partials.reserve((size_t)nb * NEQ));
  const bool dbg = coeff != nullptr;
  if (dbg) {
    LB_CUDA(c, c->dbg_coeff.reserve(nsh + nfl));
    LB_CUDA(c, c->dbg_sel.reserve(nsh + nfl));
  }
  prof_begin(c, LOAM_B200_K_ODOM_ITER);
  if (pose->iter % 5 == 0) {
    const int warps = nsh + nfl;
    odom_search_kernel<false><<<blocks_for((long long)warps * 32, LM_THREADS), LM_THREADS, 0, c->stream>>>(
        view_of(tc), view_of(ts), tc.points(), ts.points(), c->od_q.p, nsh, nfl, a, c->od_ind.p, nullptr,
        ring_off_ptr(c, 0), ring_off_ptr(c, 1));
    LB_LAUNCH_CHECK(c);
  }
  ResultMailbox mb{nullptr, 0};
  if (!c->prof_on && !getenv_no_mailbox()) mb = next_mailbox(c);
  odom_iterate_kernel<false><<<nb, LM_THREADS, 0, c->stream>>>(view_of(tc), view_of(ts), tc.points(), ts.points(), c->od_q.p, nsh,
                                                        nfl, cb, a, c->od_ind.p, c->partials.p, c->result.p,
                                                        c->ticket.p, dbg ? c->dbg_coeff.p : nullptr,
                                                        dbg ? c->dbg_sel.p : nullptr, nullptr, mb);
  LB_LAUNCH_CHECK(c);
  prof_end(c);
  int rc = mb.host ? fetch_normal_eq_mailbox(c, out) : fetch_normal_eq(c, out);
  if (rc) return rc;
  if (dbg) {
    LB_CUDA(c, cudaMemcpyAsync(coeff, c->dbg_coeff.p, (size_t)(nsh + nfl) * 16, cudaMemcpyDeviceToHost, c->stream));
    if (selected)
      LB_CUDA(c, cudaMemcpyAsync(selected, c->dbg_sel.p, (size_t)(nsh + nfl), cudaMemcpyDeviceToHost, c->stream));
    if (ind)
      LB_CUDA(c, cudaMemcpyAsync(ind, c->od_ind.p, (size_t)(nsh + nfl) * 3 * 4, cudaMemcpyDeviceToHost, c->stream));
    LB_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return LOAM_B200_OK;
}

int loam_b200_odom_iterate(loam_b200_ctx* c, const loam_b200_odom_pose* pose, loam_b200_normal_eq* out) {
  return odom_iterate_impl(c, pose, out, nullptr, nullptr, nullptr);
}
int loam_b200_odom_iterate_debug(loam_b200_ctx* c, const loam_b200_odom_pose* pose, loam_b200_normal_eq* out,
                                 float* coeff, int8_t* selected, int32_t* ind) {
  if (!coeff) return LOAM_B200_ERR_ARG;
  return odom_iterate_impl(c, pose, out, coeff, selected, ind);
}

// ------------------------------------------------------------------------------------------------ device-resident loops
// Whole Gauss-Newton loops with the pose kept on the device (lmstep.cuh).  The loop is ONE launch of a pre-instantiated
// CUDA graph: a gate kernel, then a WHILE conditional node whose body holds the iteration kernels and the one-warp step
// kernel; the step kernel clears the condition when the loop has converged (cudaGraphSetConditional) and posts the final
// pose into the mapped host mailbox, so the host pays one round trip per loop instead of one per iteration
// (tools/probes/loop_overheads.cu: 2.3 us per WHILE iteration + 1.2 us per kernel node on B200, against ~12 us per host
// round trip).  What a sweep changes (clouds, counts, pose) is written into the state block by the init kernel, so the
// graph is only rebuilt when a capacity or a baked buffer address changes.  With a communicator the all-reduce sits
// between iteration kernel and step: that mode keeps stream launches in chunks (map_solve_chunked).
static int lm_read_header(loam_b200_ctx* c, const void* d_state, LmHeader* h) {
  LB_CUDA(c, c->result_host.reserve(NEQ));
  LB_CUDA(c, cudaMemcpyAsync(c->result_host.p, d_state, sizeof(LmHeader), cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  memcpy(h, c->result_host.p, sizeof(LmHeader));
  return LOAM_B200_OK;
}

// wait for the loop's final header in the mailbox (see fetch_normal_eq_mailbox)
static int lm_wait_mailbox(loam_b200_ctx* c, LmHeader* h) {
  volatile int* box = reinterpret_cast<volatile int*>(c->result_mailbox.p);
  const auto t0 = std::chrono::steady_clock::now();
  long long spins = 0;
  while (box[32] != c->result_seq) {
    if ((++spins & 0xfff) == 0 && std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 2.0) {
      LB_CUDA(c, cudaStreamSynchronize(c->stream));
      if (box[32] != c->result_seq) return LOAM_B200_ERR_CUDA;
      break;
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  int* w = reinterpret_cast<int*>(h);
  for (int i = 0; i < 9; i++) w[i] = box[i];
  return LOAM_B200_OK;
}

static int round_cap(int n) { return ((n + n / 4 + 255) / 256) * 256; }  // 25 % head room, multiples of 256 queries

// (re)build a loop graph: `launch_gate` and `launch_body` enqueue their kernels on c->stream (captured, not run)
extern "C++" {
template <typename GATE, typename BODY>
static int loop_graph_build(loam_b200_ctx* c, LoopGraph& lg, GATE launch_gate, BODY launch_body) {
  lg.destroy();
  LB_CUDA(c, cudaGraphCreate(&lg.graph, 0));
  cudaGraphConditionalHandle handle;
  LB_CUDA(c, cudaGraphConditionalHandleCreate(&handle, lg.graph, 1, cudaGraphCondAssignDefault));
  lg.handle = (unsigned long long)handle;
  LB_CUDA(c, cudaStreamBeginCaptureToGraph(c->stream, lg.graph, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
  launch_gate();
  cudaGraph_t same = nullptr;
  LB_CUDA(c, cudaStreamEndCapture(c->stream, &same));
  cudaGraphNode_t gate_node = nullptr;
  size_t n_nodes = 1;
  LB_CUDA(c, cudaGraphGetNodes(lg.graph, &gate_node, &n_nodes));
  cudaGraphNodeParams wp = {};
  wp.type = cudaGraphNodeTypeConditional;
  wp.conditional.handle = handle;
  wp.conditional.type = cudaGraphCondTypeWhile;
  wp.conditional.size = 1;
  cudaGraphNode_t while_node = nullptr;
  LB_CUDA(c, cudaGraphAddNode(&while_node, lg.graph, &gate_node, 1, &wp));
  cudaGraph_t body = wp.conditional.phGraph_out[0];
  LB_CUDA(c, cudaStreamBeginCaptureToGraph(c->stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
  launch_body();
  LB_CUDA(c, cudaStreamEndCapture(c->stream, &same));
  LB_CUDA(c, cudaGraphInstantiate(&lg.exec, lg.graph, 0));
  lg.builds++;
  return LOAM_B200_OK;
}
}  // extern "C++"

static bool loop_graphs_enabled() {
  static const bool off = getenv("LOAM_B200_NO_LOOP_GRAPH") != nullptr;
  return !off;
}

int loam_b200_odom_solve(loam_b200_ctx* c, const float rot[3], const float pos[3], float inv_scan_period, int max_iterations,
                         float delta_t_abort, float delta_r_abort, loam_b200_lm_result* out) {
  CHECK_CTX(c);
  if (!rot || !pos || !out || max_iterations < 0) return LOAM_B200_ERR_ARG;
  if (!c->od_last_set) return LOAM_B200_ERR_STATE;
  LB_CUDA(c, odom_join_rebuild(c));
  const int nsh = c->od_nsharp, nfl = c->od_nflat;
  memset(out, 0, sizeof *out);
  for (int i = 0; i < 3; i++) { out->rot[i] = rot[i]; out->pos[i] = pos[i]; }
  if (nsh + nfl == 0 || max_iterations == 0) return LOAM_B200_OK;
  const Tree& tc = c->tree[LOAM_B200_TREE_ODOM_CORNER];
  const Tree& ts = c->tree[LOAM_B200_TREE_ODOM_SURF];
  const bool use_graph = loop_graphs_enabled();
  LoopGraph& lg = c->odom_loop;
  const int cap_sh = use_graph ? std::max(lg.cap_a, nsh > lg.cap_a ? round_cap(nsh) : 0) : nsh;
  const int cap_fl = use_graph ? std::max(lg.cap_b, nfl > lg.cap_b ? round_cap(nfl) : 0) : nfl;
  const int cb = blocks_for(nsh, LM_THREADS), sb = blocks_for(nfl, LM_THREADS);
  const int nb = cb + sb;
  const int nb_cap = blocks_for(cap_sh, LM_THREADS) + blocks_for(cap_fl, LM_THREADS);
  LB_CUDA(c, c->partials.reserve((size_t)std::max(nb, nb_cap) * NEQ));
  LB_CUDA(c, c->lm_state.reserve(sizeof(OdomLmState) + sizeof(MapLmState)));
  OdomLmState* st = reinterpret_cast<OdomLmState*>(c->lm_state.p);
  const bool use_mailbox = !c->prof_on && !getenv_no_mailbox() && c->result_mailbox.reserve(64) == cudaSuccess;
  int seq = 0;
  if (use_mailbox) seq = next_mailbox(c).seq;
  OdomLoopIo io;
  io.corner_tree = view_of(tc); io.surf_tree = view_of(ts);
  io.last_corner = tc.points(); io.last_surf = ts.points(); io.queries = c->od_q.p; io.ind = c->od_ind.p;
  io.ring_off_corner = ring_off_ptr(c, 0); io.ring_off_surf = ring_off_ptr(c, 1);
  io.n_sharp = nsh; io.n_flat = nfl; io.sharp_blocks = cb; io.n_blocks = nb;
  odom_lm_init_kernel<<<1, 32, 0, c->stream>>>(st, rot[0], rot[1], rot[2], pos[0], pos[1], pos[2], inv_scan_period,
                                               delta_t_abort, delta_r_abort, max_iterations, tc.m, ts.m, io, seq);
  LB_LAUNCH_CHECK(c);
  const OdomIterArgs unused{};
  const TreeView tv0{};
  LmHeader h{};
  prof_begin(c, LOAM_B200_K_ODOM_ITER);
  if (use_graph) {
    const void* baked[4] = {st, c->partials.p, c->result.p, use_mailbox ? (void*)c->result_mailbox.p : nullptr};
    if (!lg.exec || lg.cap_a != cap_sh || lg.cap_b != cap_fl || memcmp(lg.baked, baked, sizeof baked) != 0) {
      float* mbp = use_mailbox ? c->result_mailbox.p : nullptr;
      unsigned long long* hp = &lg.handle;
      const int rc = loop_graph_build(
          c, lg, [&] { lm_gate_kernel<<<1, 32, 0, c->stream>>>(&st->h, *hp, mbp); },
          [&] {
            odom_search_kernel<true><<<blocks_for((long long)(cap_sh + cap_fl) * 32, LM_THREADS), LM_THREADS, 0, c->stream>>>(
                tv0, tv0, nullptr, nullptr, nullptr, 0, 0, unused, nullptr, st, nullptr, nullptr);
            odom_iterate_kernel<true><<<nb_cap, LM_THREADS, 0, c->stream>>>(tv0, tv0, nullptr, nullptr, nullptr, 0, 0, 0, unused,
                                                                         nullptr, c->partials.p, c->result.p, c->ticket.p,
                                                                         nullptr, nullptr, st);
            odom_lm_step_kernel<<<1, 32, 0, c->stream>>>(st, c->result.p, *hp, mbp);
          });
      if (rc) return rc;
      lg.cap_a = cap_sh; lg.cap_b = cap_fl;
      memcpy(lg.baked, baked, sizeof baked);
    }
    LB_CUDA(c, cudaGraphLaunch(lg.exec, c->stream));
    const int rc = use_mailbox ? lm_wait_mailbox(c, &h) : lm_read_header(c, st, &h);
    if (rc) return rc;
    // gate + per executed iteration: search (a no-op except every 5th), iterate, step -- launched by the WHILE node
    c->launches += 1 + 3 * h.iters_run;
    g_total_launches.fetch_add(1 + 3 * h.iters_run, std::memory_order_relaxed);
  } else {
    for (int it = 0; it < max_iterations;) {
      const int chunk_end = std::min(max_iterations, it + 5);  // one correspondence search per chunk
      for (; it < chunk_end; it++) {
        if (it % 5 == 0) {
          odom_search_kernel<true><<<blocks_for((long long)(nsh + nfl) * 32, LM_THREADS), LM_THREADS, 0, c->stream>>>(
              tv0, tv0, nullptr, nullptr, nullptr, 0, 0, unused, nullptr, st, nullptr, nullptr);
          LB_LAUNCH_CHECK(c);
        }
        odom_iterate_kernel<true><<<nb, LM_THREADS, 0, c->stream>>>(tv0, tv0, nullptr, nullptr, nullptr, 0, 0, 0, unused, nullptr,
                                                                  c->partials.p, c->result.p, c->ticket.p, nullptr, nullptr, st);
        LB_LAUNCH_CHECK(c);
        odom_lm_step_kernel<<<1, 32, 0, c->stream>>>(st, c->result.p);
        LB_LAUNCH_CHECK(c);
      }
      const int rc = lm_read_header(c, st, &h);
      if (rc) return rc;
      if (h.done) break;
    }
  }
  prof_end(c);
  for (int i = 0; i < 3; i++) { out->rot[i] = h.rot[i]; out->pos[i] = h.pos[i]; }
  out->iterations = h.iters_run;
  out->converged = h.done ? 1 : 0;
  return LOAM_B200_OK;
}

int loam_b200_map_solve(loam_b200_ctx* c, const float rot[3], const float pos[3], int max_iterations, float delta_t_abort,
                        float delta_r_abort, loam_b200_lm_result* out) {
  CHECK_CTX(c);
  if (!rot || !pos || !out || max_iterations < 0) return LOAM_B200_ERR_ARG;
  // a query slice without a communicator only yields partials; the cube-sharded map runs the per-iteration form (its
  // all-reduce is fused into the iteration kernel)
  if (c->shard_world > 1 && !c->comm) return LOAM_B200_ERR_STATE;
  const int nc = c->map_nc, ns = c->map_ns;
  memset(out, 0, sizeof *out);
  for (int i = 0; i < 3; i++) { out->rot[i] = rot[i]; out->pos[i] = pos[i]; }
  if (nc + ns == 0 || max_iterations == 0) return LOAM_B200_OK;
  // this rank's contiguous slice of each query kind (everything when not sharded)
  const int W = c->shard_world, R = c->shard_rank;
  const int c0 = (int)((long long)nc * R / W), c1 = (int)((long long)nc * (R + 1) / W);
  const int s0 = (int)((long long)ns * R / W), s1 = (int)((long long)ns * (R + 1) / W);
  const int lc = c1 - c0, ls = s1 - s0;
  const int cb = blocks_for(lc, MAP_Q_PER_BLOCK), sb = blocks_for(ls, MAP_Q_PER_BLOCK);
  const int nb = std::max(cb + sb, 1);
  const bool use_graph = loop_graphs_enabled() && !c->comm;
  LoopGraph& lg = c->map_loop;
  const int cap_c = use_graph ? std::max(lg.cap_a, lc > lg.cap_a ? round_cap(lc) : 0) : lc;
  const int cap_s = use_graph ? std::max(lg.cap_b, ls > lg.cap_b ? round_cap(ls) : 0) : ls;
  const int nb_cap = std::max(blocks_for(cap_c, MAP_Q_PER_BLOCK) + blocks_for(cap_s, MAP_Q_PER_BLOCK), 1);
  LB_CUDA(c, c->partials.reserve((size_t)std::max(nb, nb_cap) * NEQ));
  LB_CUDA(c, c->lm_state.reserve(sizeof(OdomLmState) + sizeof(MapLmState)));
  MapLmState* st = reinterpret_cast<MapLmState*>(c->lm_state.p + sizeof(OdomLmState));
  const bool use_mailbox = use_graph && !c->prof_on && !getenv_no_mailbox() && c->result_mailbox.reserve(64) == cudaSuccess;
  int seq = 0;
  if (use_mailbox) seq = next_mailbox(c).seq;
  MapLoopIo io;
  memset(&io, 0, sizeof io);
  if (c->map_use_store) {
    const MapCellLookup l0 = store_lookup_of(c, 0), l1 = store_lookup_of(c, 1);
    memcpy(io.lookup[0], &l0, sizeof l0);
    memcpy(io.lookup[1], &l1, sizeof l1);
  } else {
    const GridCellLookup l0{grid_view_of(c->grid[0])}, l1{grid_view_of(c->grid[1])};
    memcpy(io.lookup[0], &l0, sizeof l0);
    memcpy(io.lookup[1], &l1, sizeof l1);
  }
  io.queries = c->map_q_corner; io.queries_surf = c->map_q_surf; io.n_corner_total = nc; io.c0 = c0; io.n_corner = lc; io.s0 = s0; io.n_surf = ls;
  io.corner_blocks = cb; io.n_blocks = nb;
  map_lm_init_kernel<<<1, 128, 0, c->stream>>>(st, rot[0], rot[1], rot[2], pos[0], pos[1], pos[2], delta_t_abort,
                                               delta_r_abort, max_iterations, io, seq);
  LB_LAUNCH_CHECK(c);
  const MapIterArgs unused{};
  LmHeader h{};
  prof_begin(c, LOAM_B200_K_MAP_ITER);
  auto launch_iterate = [&](int grid) {
    if (c->map_use_store)
      map_iterate_kernel<false, MapCellLookup, true><<<grid, MAP_THREADS, 0, c->stream>>>(
          MapCellLookup{}, MapCellLookup{}, nullptr, nullptr, 0, 0, 0, 0, 0, 0, unused, c->partials.p, c->result.p, c->ticket.p, nullptr,
          nullptr, nullptr, st);
    else
      map_iterate_kernel<false, GridCellLookup, true><<<grid, MAP_THREADS, 0, c->stream>>>(
          GridCellLookup{}, GridCellLookup{}, nullptr, nullptr, 0, 0, 0, 0, 0, 0, unused, c->partials.p, c->result.p, c->ticket.p, nullptr,
          nullptr, nullptr, st);
  };
  if (use_graph) {
    const int variant = c->map_use_store ? 1 : 0;
    const void* baked[4] = {st, c->partials.p, c->result.p, use_mailbox ? (void*)c->result_mailbox.p : nullptr};
    if (!lg.exec || lg.cap_a != cap_c || lg.cap_b != cap_s || lg.variant != variant || memcmp(lg.baked, baked, sizeof baked) != 0) {
      float* mbp = use_mailbox ? c->result_mailbox.p : nullptr;
      unsigned long long* hp = &lg.handle;
      const int rc = loop_graph_build(
          c, lg, [&] { lm_gate_kernel<<<1, 32, 0, c->stream>>>(&st->h, *hp, mbp); },
          [&] {
            launch_iterate(nb_cap);
            map_lm_step_kernel<<<1, 32, 0, c->stream>>>(st, c->result.p, *hp, mbp);
          });
      if (rc) return rc;
      lg.cap_a = cap_c; lg.cap_b = cap_s; lg.variant = variant;
      memcpy(lg.baked, baked, sizeof baked);
    }
    LB_CUDA(c, cudaGraphLaunch(lg.exec, c->stream));
    const int rc = use_mailbox ? lm_wait_mailbox(c, &h) : lm_read_header(c, st, &h);
    if (rc) return rc;
    c->launches += 1 + 2 * h.iters_run;  // gate + (iterate, step) per executed iteration
    g_total_launches.fetch_add(1 + 2 * h.iters_run, std::memory_order_relaxed);
  } else {
    for (int it = 0; it < max_iterations;) {
      const int chunk_end = std::min(max_iterations, it + 3);  // 2-3 iterations is the usual case
      for (; it < chunk_end; it++) {
        launch_iterate(nb);
        LB_LAUNCH_CHECK(c);
        {
          const int rcc = allreduce_result(c);  // no-op without a communicator; every rank then takes the same step
          if (rcc) return rcc;
        }
        map_lm_step_kernel<<<1, 32, 0, c->stream>>>(st, c->result.p);
        LB_LAUNCH_CHECK(c);
      }
      const int rc = lm_read_header(c, st, &h);
      if (rc) return rc;
      if (h.done) break;
    }
  }
  prof_end(c);
  for (int i = 0; i < 3; i++) { out->rot[i] = h.rot[i]; out->pos[i] = h.pos[i]; }
  out->iterations = h.iters_run;
  out->converged = h.done ? 1 : 0;
  return LOAM_B200_OK;
}

// The warp-parallel 6 x 6 step of the device-resident loops on caller-supplied normal equations (parity tests: it must
// equal loam_b200_host_gn_solve, the serial host form of the same arithmetic, bit for bit).
namespace loamb {
__global__ void gn_solve_debug_kernel(const float* __restrict__ ata_atb, int n, int first, float eig_thr, GnState* g,
                                      float* __restrict__ x_out, int* __restrict__ deg_out) {
  __shared__ float s_r[NEQ];
  const int lane = threadIdx.x;
  for (int m = 0; m < n; m++) {
    if (lane == 0) g->degenerate = 0;
    const float* src = ata_atb + (size_t)m * 42;
    // 21 upper-triangle entries + 6 right-hand sides, as the iteration kernels leave them
    if (lane < 21) {
      int k = 0, r = 0, c2 = 0;
      for (int i = 0; i < 6; i++)
        for (int j = i; j < 6; j++) {
          if (k == lane) { r = i; c2 = j; }
          k++;
        }
      s_r[lane] = src[r * 6 + c2];
    } else if (lane < 27) {
      s_r[lane] = src[36 + lane - 21];
    } else {
      s_r[lane] = 0.f;
    }
    __syncwarp();
    float x[6];
    gn_solve_warp(s_r, first != 0, eig_thr, g, x);
    if (lane == 0) {
      for (int i = 0; i < 6; i++) x_out[(size_t)m * 6 + i] = x[i];
      deg_out[m] = g->degenerate;
    }
    __syncwarp();
  }
}
}  // namespace loamb

int loam_b200_debug_gn_solve(loam_b200_ctx* c, const float* ata_atb, int n, int first_iteration, float eigen_threshold,
                             float* x_out, int* degenerate_out) {
  CHECK_CTX(c);
  if (!ata_atb || n <= 0 || !x_out || !degenerate_out) return LOAM_B200_ERR_ARG;
  LB_CUDA(c, c->tmp_pts.reserve((size_t)n * 11 + 16));  // 42 floats per system
  LB_CUDA(c, c->tmp_pts2.reserve((size_t)n * 2 + 16));   // x (6 floats) + flag per system
  LB_CUDA(c, c->lm_state.reserve(sizeof(OdomLmState) + sizeof(MapLmState)));
  float* d_in = reinterpret_cast<float*>(c->tmp_pts.p);
  float* d_x = reinterpret_cast<float*>(c->tmp_pts2.p);
  int* d_deg = reinterpret_cast<int*>(d_x + (size_t)n * 6);
  GnState* g = &reinterpret_cast<OdomLmState*>(c->lm_state.p)->gn;
  LB_CUDA(c, cudaMemcpyAsync(d_in, ata_atb, (size_t)n * 42 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  gn_solve_debug_kernel<<<1, 32, 0, c->stream>>>(d_in, n, first_iteration, eigen_threshold, g, d_x, d_deg);
  LB_LAUNCH_CHECK(c);
  LB_CUDA(c, cudaMemcpyAsync(x_out, d_x, (size_t)n * 6 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaMemcpyAsync(degenerate_out, d_deg, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  return LOAM_B200_OK;
}

// ------------------------------------------------------------------------------------------------ bulk transforms
int loam_b200_transform_to_end(loam_b200_ctx* c, float* pts, int n, const loam_b200_odom_pose* p) {
  CHECK_CTX(c);
  if (n < 0 || (n > 0 && !pts) || !p) return LOAM_B200_ERR_ARG;
  if (n == 0) return LOAM_B200_OK;
  int rc = upload_points(c, c->tmp_pts2, pts, n);
  if (rc) return rc;
  ToEndArgs a;
  a.rx = p->rot[0]; a.ry = p->rot[1]; a.rz = p->rot[2];
  a.tx = p->pos[0]; a.ty = p->pos[1]; a.tz = p->pos[2];
  a.inv_sp = p->inv_scan_period;
  a.srx = p->sin_[0]; a.crx = p->cos_[0]; a.sry = p->sin_[1]; a.cry = p->cos_[1]; a.srz = p->sin_[2]; a.crz = p->cos_[2];
  prof_begin(c, LOAM_B200_K_TRANSFORM);
  transform_to_end_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(c->tmp_pts2.p, n, a);
  LB_LAUNCH_CHECK(c);
  prof_end(c);
  LB_CUDA(c, cudaMemcpyAsync(pts, c->tmp_pts2.p, (size_t)n * 16, cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  return LOAM_B200_OK;
}

int loam_b200_transform_to_map(loam_b200_ctx* c, float* pts, int n, const loam_b200_pose* p) {
  CHECK_CTX(c);
  if (n < 0 || (n > 0 && !pts) || !p) return LOAM_B200_ERR_ARG;
  if (n == 0) return LOAM_B200_OK;
  int rc = upload_points(c, c->tmp_pts2, pts, n);
  if (rc) return rc;
  MapIterArgs a;
  fill_map_args(p, a);
  prof_begin(c, LOAM_B200_K_TRANSFORM);
  transform_to_map_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(c->tmp_pts2.p, n, a);
  LB_LAUNCH_CHECK(c);
  prof_end(c);
  LB_CUDA(c, cudaMemcpyAsync(pts, c->tmp_pts2.p, (size_t)n * 16, cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  return LOAM_B200_OK;
}

// ------------------------------------------------------------------------------------------------ voxel grid
int loam_b200_voxel_grid(loam_b200_ctx* c, const float* pts, int n, float leaf, float* out, int cap, int* n_out) {
  CHECK_CTX(c);
  if (n < 0 || (n > 0 && (!pts || !out)) || !n_out || !(leaf > 0.f)) return LOAM_B200_ERR_ARG;
  *n_out = 0;
  if (n == 0) return LOAM_B200_OK;
  int rc = upload_points(c, c->tmp_pts, pts, n);
  if (rc) return rc;
  LB_CUDA(c, c->tmp_pts2.reserve(n));
  int count = 0;
  prof_begin(c, LOAM_B200_K_VOXEL);
  rc = voxel_grid_device(c, c->tmp_pts.p, n, leaf, c->tmp_pts2.p, &count);
  prof_end(c);
  if (rc) return rc;
  if (count > cap) return LOAM_B200_ERR_CAPACITY;
  LB_CUDA(c, cudaMemcpyAsync(out, c->tmp_pts2.p, (size_t)count * 16, cudaMemcpyDeviceToHost, c->stream));
  LB_CUDA(c, cudaStreamSynchronize(c->stream));
  *n_out = count;
  return LOAM_B200_OK;
}

// ------------------------------------------------------------------------------------------------ profiling
int loam_b200_profile_enable(loam_b200_ctx* c, int on) {
  CHECK_CTX(c);
  c->prof_on = on != 0;
  return LOAM_B200_OK;
}
int loam_b200_profile_reset(loam_b200_ctx* c) {
  CHECK_CTX(c);
  for (int i = 0; i < LOAM_B200_NUM_KERNEL_FAMILIES; i++) { c->prof_ms[i] = 0; c->prof_launches[i] = 0; }
  return LOAM_B200_OK;
}
int loam_b200_profile_get(loam_b200_ctx* c, int family, double* gpu_ms, long long* launches) {
  CHECK_CTX(c);
  if (family < 0 || family >= LOAM_B200_NUM_KERNEL_FAMILIES) return LOAM_B200_ERR_ARG;
  if (gpu_ms) *gpu_ms = c->prof_ms[family];
  if (launches) *launches = c->prof_launches[family];
  return LOAM_B200_OK;
}
long long loam_b200_launch_count(loam_b200_ctx* c) { return c ? c->launches : 0; }
long long loam_b200_total_launch_count(void) { return loamb::g_total_launches; }

}  // extern "C"

#include "stages.inc"
