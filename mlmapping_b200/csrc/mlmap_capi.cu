// C ABI of the B200-native MLMapping hot path (include/mlmap_b200.h).  Host logic only:
// table construction (reference init_map functions), the per-frame launch sequence, the
// libstdc++ bucket-count chain, and buffer management.  All map arithmetic runs in the
// kernels of frame_kernels.cuh / order_kernels.cuh / query_kernels.cuh; there is no CPU
// fallback — without a CUDA device mlm_create fails with MLM_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <chrono>
#include <string>
#include <utility>
#include <vector>

#include "../../include/mlmap_b200.h"
#include "frame_kernels.cuh"
#include "order_kernels.cuh"
#include "explore_kernels.cuh"
#include "query_kernels.cuh"
#include "shard_kernels.cuh"
#include "ray_kernels.cuh"
#include "esdf_kernels.cuh"
#include "frontier_kernels.cuh"
#include "view_kernels.cuh"
#include "reach_kernels.cuh"

using namespace mlm;

namespace {

thread_local std::string g_last_error;

// also clears the failure from the thread's last error, so that a later call's cudaGetLastError() does not report it
#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      cudaGetLastError();                                                                     \
      g_last_error = std::string(#expr) + ": " + cudaGetErrorString(_e);                      \
      return MLM_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

// A temporary of a host-pointer entry point: one stream-ordered allocation, released on its stream when the owner goes
// out of scope (or by reset()), so that an error return gives it back to the pool as the success path does.
template <typename T>
class StreamTemp {
 public:
  explicit StreamTemp(cudaStream_t s) : s_(s) {}
  StreamTemp(StreamTemp &&o) noexcept : p_(o.p_), s_(o.s_) { o.p_ = nullptr; }
  ~StreamTemp() { reset(); }
  cudaError_t alloc(size_t count) {
    reset();
    const cudaError_t e = cudaMallocAsync((void **)&p_, count * sizeof(T), s_);
    if (e != cudaSuccess) p_ = nullptr;
    return e;
  }
  void reset() {
    if (p_) cudaFreeAsync(p_, s_);
    p_ = nullptr;
  }
  operator T *() const { return p_; }

 private:
  T *p_ = nullptr;
  cudaStream_t s_;
};

// Scratch that a handle keeps and grows: (buffer, bytes) pairs, allocated all together or not at all.
using ScratchList = std::vector<std::pair<void **, size_t>>;
void scratch_free(const ScratchList &bufs) {
  for (const auto &b : bufs) {
    if (*b.first) cudaFree(*b.first);
    *b.first = nullptr;
  }
}
int scratch_alloc(const ScratchList &bufs, const char *what) {
  for (const auto &b : bufs) {
    const cudaError_t e = cudaMalloc(b.first, b.second);
    if (e == cudaSuccess) continue;
    *b.first = nullptr;
    scratch_free(bufs);
    cudaGetLastError();
    g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return MLM_ERR_CUDA;
  }
  return MLM_OK;
}

// libstdc++ _Prime_rehash_policy growth chain from an empty table with max_load_factor 1:
// first insert -> 13, then next_bkt(2*B) from the sparse __prime_list (SURVEY Appendix B;
// verified against this toolchain's unordered_set in tests/test_host_logic.py).
const uint32_t kBucketChain[] = {1,      13,     29,     59,      127,     257,     541,     1109,
                                 2357,   5087,   10273,  20753,   42043,   85229,   172933,  351061,
                                 712697, 1447153, 2938679, 5967347, 12117689, 24607243, 49969847, 101473717};
constexpr int kBucketChainLen = sizeof(kBucketChain) / sizeof(kBucketChain[0]);
uint32_t chain_next(uint32_t B) {
  for (int i = 0; i + 1 < kBucketChainLen; i++)
    if (kBucketChain[i] == B) return kBucketChain[i + 1];
  return 0;
}
uint32_t chain_cover(uint32_t n) {  // smallest chain value >= n
  for (int i = 0; i < kBucketChainLen; i++)
    if (kBucketChain[i] >= n) return kBucketChain[i];
  return 0;
}
// bucket count of a table with B buckets after a frame put n distinct keys in it (clear() keeps the bucket array): the
// first insert into an empty table allocates 13 buckets, then the chain grows until the keys fit
uint32_t bucket_growth(uint32_t B, int n) {
  if (n > 0 && B == 1) B = 13;
  while ((uint32_t)n > B) {
    const uint32_t nb = chain_next(B);
    if (nb == 0) break;
    B = nb;
  }
  return B;
}

// glibc rand() == random_r() TYPE_3 (x^31 + x^3 + 1 additive feedback), stdlib/random_r.c: the reference
// samples pixels with rand() (src/mlmap.cpp:324-325) and never calls srand(), i.e. seed 1.  Own state per
// handle so the product does not share libc's global generator with anybody.
struct GlibcRand {
  int32_t r[31];
  int f = 3, b = 0;
  GlibcRand() { seed(1); }
  void seed(unsigned s) {
    if (s == 0) s = 1;
    r[0] = (int32_t)s;
    int32_t word = (int32_t)s;
    for (int i = 1; i < 31; i++) {
      long hi = word / 127773, lo = word % 127773;
      long w = 16807 * lo - 2836 * hi;
      if (w < 0) w += 2147483647;
      word = (int32_t)w;
      r[i] = word;
    }
    f = 3;
    b = 0;
    for (int i = 0; i < 310; i++) next();
  }
  int next() {
    uint32_t v = (uint32_t)r[f] + (uint32_t)r[b];
    r[f] = (int32_t)v;
    int res = (int)((v >> 1) & 0x7fffffff);
    if (++f >= 31) f = 0;
    if (++b >= 31) b = 0;
    return res;
  }
};

// x / d == umulhi(x, mul) >> shift for every x < 2^31 (round-up method, checked in tests/test_host_logic.py); d == 1 -> mul 0
void make_div_magic(uint32_t d, uint32_t *mul, int *shift) {
  if (d < 2) {
    *mul = 0;
    *shift = 0;
    return;
  }
  int sh = 0;
  while ((2u << sh) <= d - 1) sh++;  // floor(log2(d - 1))
  *shift = sh;
  *mul = (uint32_t)(((1ull << (32 + sh)) / (uint64_t)d) + 1);
}
// 2^64 mod B (see libstdcxx_bucket_fast)
uint32_t pow64_mod(uint32_t B) { return (uint32_t)((((unsigned __int128)1) << 64) % (unsigned __int128)B); }

int next_pow2(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}
int host_floor_div(int a, int b) {
  int q = a / b, r = a - q * b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}

}  // namespace

struct mlm_map {
  mlm_config cfg;
  MapParams P;
  DeviceBuffers D;
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  FrameParams *h_fp = nullptr;    // pinned
  FrameCounters *h_fc = nullptr;  // pinned
  int64_t cum_ram_expand = 0, cum_obs = 0, n_submaps = 0;  // cumulative counters (reference ram_expand_cnt / obs_cnt)
  uint32_t frame_idx = 0;
  int last_parity = 0;
  GlibcRand rng;  // project_depth's rand() stream (sampled mode)
  // sharded operation (one logical map over several ranks, exchange over peer memory)
  uint32_t *d_key_stamp = nullptr;   // [cells] global ordering stamp per hit key of a rehash scan
  int *d_shard_cursor = nullptr;     // [kMaxWorld] records sent per destination this scan; [kMaxWorld] skip flag; [kMaxWorld + 1] push ticket
  ShardState *d_shard_state = nullptr, *h_shard_state = nullptr;  // device copy / pinned host copy
  int *d_keys_all = nullptr;         // [sort_cap] gathered keys, contiguous (rehash path)
  uint32_t *d_stamps_all = nullptr, *d_bucket_all = nullptr;
  void *shard_arena = nullptr;       // this rank's exchange arena (exported to the peers)
  size_t shard_arena_bytes = 0;
  ShardPeers shard_peers;            // every rank's arena as mapped here
  void *shard_mapped[kMaxWorld] = {};  // cudaIpcOpenMemHandle results to close
  bool shard_open = false, shard_connected = false, shard_pending = false;
  // two-call layer interface / asynchronous frames
  int stage_call = 0;          // run_frame stops after the awareness layer (project + column)
  bool staged = false;         // an awareness-layer update waits for mlm_local_input_pc_pose_direct
  int staged_slow = 0;
  uint32_t staged_order_B = 1;
  int async_call = 0;          // run_frame returns after enqueueing; mlm_frame_finish completes the frame
  bool frame_pending = false;
  int pending_mode = 0;
  int frame_sms = 0;           // CTAs of k_frame when the handle shares the GPU with other maps (0: one per SM)
  bool poisoned = false;       // a frame failed after it had staged its sets: the staging was never consumed
  uint32_t frame_seq = 0;
  int *d_sample_info = nullptr;  // sampled projection of a device image: {points, tries used}
  uint2 *d_sample_tries = nullptr;
  cudaEvent_t sev[MLM_NUM_SHARD_KERNELS + 1] = {};
  float skms[MLM_NUM_SHARD_KERNELS] = {};
  bool shard_shares_device = false;  // another rank of this process runs on the same GPU (single-GPU tests)
  uint32_t shard_epoch = 0;
  unsigned long long shard_timeout_ns = 10ull * 1000 * 1000 * 1000;
  // replicated map over peer memory (mlm_replica_*)
  ReplicaPeers replica_peers = {};
  void *replica_arena = nullptr;
  void *replica_mapped[kMaxWorld] = {};
  bool replica_open = false, replica_connected = false;
  uint32_t replica_epoch = 0;
  int *d_replica_state = nullptr;   // source: {ticket, error}; replica: {new blocks, error, ticket, records}
  int replica_last_blocks = 0;
  int shard_world = 1, shard_rank = 0;
  bool shard_stage_pending = false;
  cudaGraphExec_t graph_exec[3] = {nullptr, nullptr, nullptr};  // by input mode: points, depth image, sampled pixels
  cudaGraph_t graph[3] = {nullptr, nullptr, nullptr};
  cudaGraphNode_t graph_nodes[3][3] = {};
  int col_grid = 1;        // CTAs of the persistent k_column: one per SM, at most one per work column
  int use_fused = 0;       // frames run as one cooperative k_frame launch
  int frame_grid = 1;      // CTAs of k_frame (all co-resident)
  cudaGraph_t fgraph[3] = {nullptr, nullptr, nullptr};
  cudaGraphExec_t fgraph_exec[3] = {nullptr, nullptr, nullptr};
  cudaGraphNode_t fgraph_node[3] = {nullptr, nullptr, nullptr};
  void *h_stage = nullptr;        // pinned input staging
  size_t stage_bytes = 0;
  void *d_input = nullptr;
  size_t input_bytes = 0;
  // slow-path ordering scratch
  uint64_t *d_sort_a = nullptr, *d_sort_b = nullptr;
  int *d_seq_a = nullptr, *d_seq_b = nullptr;
  int sort_cap = 0;
  uint32_t act_cap = 0;
  uint32_t act_miss_cap = 0;
  uint32_t bucket_count_miss = 1;  // emulated miss_idx_set.bucket_count() (exploration mode)
  uint32_t bucket_count = 1;  // emulated hit_idx_odds_hashmap.bucket_count()
  uint32_t last_order_B = 1;  // bucket count the last frame's stamps refer to
  int last_n_hit = 0;
  int col_smem_bytes = 0;
  std::vector<void *> allocs;
  int64_t launches = 0;
  HPose T_bs;
  void *l2_buf = nullptr;
  size_t l2_bytes = 0;
  int sm_count = 148;
  int profiling = 0;
  cudaEvent_t kev[MLM_NUM_FRAME_KERNELS + 1] = {};
  float kms[MLM_NUM_FRAME_KERNELS] = {};
  // signed distance field (mlm_esdf_*): buffers of esdf_cap cells, grown by a larger box; esdf_a holds the cell values
  // (double) after a build, esdf_grid the box of the last one
  uint8_t *esdf_blk = nullptr;
  int2 *esdf_a = nullptr, *esdf_b = nullptr, *esdf_stk = nullptr;
  size_t esdf_cap = 0;
  bool esdf_built = false;
  EsdfGrid esdf_grid = {};
  // frontier clustering (mlm_frontier_clusters*): per-word buffers allocated by the first call, per-cell buffers of
  // fc_cap_cells entries grown by a larger frontier
  FcScratch fc = {};
  size_t fc_cap_cells = 0;
  // candidate-view gain (mlm_view_gain*): per-view setup and tile counts for view_cap views, grown by a larger batch
  ViewSetup *view_setup = nullptr;
  unsigned long long *view_tiles = nullptr;
  size_t view_cap = 0;
  // reachability field (mlm_reach_*): class bytes and costs of reach_cap_cells cells, worklists of reach_cap_tiles tiles,
  // grown by a larger box; reach_grid is the box of the last build
  uint8_t *reach_cls = nullptr;
  int *reach_cost = nullptr, *reach_mark = nullptr, *reach_list = nullptr, *reach_ctl = nullptr;
  size_t reach_cap_cells = 0, reach_cap_tiles = 0;
  bool reach_built = false;
  ReachGrid reach_grid = {};
  // path-cost matrix (mlm_reach_matrix), apart from the field above: class bytes of mat_cap_cells cells; per field of a
  // batch the costs (mat_cap_fcells cells in all), the queue marks and two worklists (mat_cap_items items in all) and the
  // source cell (mat_cap_rows); the three queue counts and the barrier
  uint8_t *mat_cls = nullptr;
  int *mat_cost = nullptr, *mat_mark = nullptr, *mat_list = nullptr, *mat_src = nullptr, *mat_ctl = nullptr;
  size_t mat_cap_cells = 0, mat_cap_fcells = 0, mat_cap_items = 0, mat_cap_rows = 0;
};

namespace {

template <typename T>
int dev_alloc(mlm_map *h, T **p, size_t count) {
  void *q = nullptr;
  CUDA_TRY(cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
  h->allocs.push_back(q);
  *p = reinterpret_cast<T *>(q);
  return MLM_OK;
}

// ---- awareness tables, reference src/map_awareness.cpp:19-82,119-132; include/map_awareness.h:120-146
struct AwarenessTables {
  std::vector<float> odds;  // [21][nRho]
  std::vector<int> k_reach;
  std::vector<double2> centre_xy;
  std::vector<double> centre_z;
  std::vector<double> rate;   // [nZ][nRho]
  std::vector<short2> dz;     // [nZ][nRho][maxK]
  double dPhi, z_border_min;
  int nPhi, nZ;
};
float host_sigma_in_dr(double coe, double dRho, size_t x) {
  float dis = (x * dRho);
  return coe * dis * dis / dRho;
}
float host_standard_ND(float x) {
  double a1 = 0.254829592, a2 = -0.284496736, a3 = 1.421413741, a4 = -1.453152027, a5 = 1.061405429;
  double p = 0.3275911;
  int sign = 1;
  if (x < 0) sign = -1;
  x = fabsf(x) / sqrt(2.0);
  double t = 1.0 / (1.0 + p * x);
  // the reference's exp(-x * x) has a float argument and `using namespace std`: std::exp(float) == expf
  double y = 1.0 - (((((a5 * t + a4) * t) + a3) * t + a2) * t + a1) * t * expf(-x * x);
  return 0.5 * (1.0 + sign * y);
}
float host_get_odds(double coe, double dRho, int diff, size_t r) {
  if (r == 0) r = 1;
  float up = host_standard_ND(static_cast<float>(diff + 0.5) / host_sigma_in_dr(coe, dRho, r));
  float down = host_standard_ND(static_cast<float>(diff - 0.5) / host_sigma_in_dr(coe, dRho, r));
  float res = up - down < 0.001 ? 0.001 : up - down;
  res = res >= 0.999 ? 0.999 : res;
  return res;
}
// K(rho): the last diff_r of update_hits' loop, diff_r < 3 * sigma_in_dr(rho)   (int -> float compare)
int host_k_reach(const mlm_config &c, int r) {
  int K = 0;
  for (int d = 1; d < 3 * host_sigma_in_dr(c.depth_noise_coe, c.am_d_rho, r); d++) {
    K = d;
    if (d > 4 * kDiffRange) break;
  }
  return K;
}
// Half-column split: records below the sensor row (z_idx < n_below) and at/above it never feed the same hit
// cell when every neighbour step stays on its side of the row, i.e. z - n_below and
// round(z -/+ d*rate) - n_below = round((z - n_below) * (1 -/+ d/rho)) have the same sign: 2*K(rho) < rho.
// Their ray walks share only the row n_below itself (arbitrated through the global miss bitmap).  In the
// exploration mode the first-insert stamps of that row's miss cells come from both halves: they are settled after
// all columns (miss_finalize_body).
int half_column_split(const mlm_config &c, const std::vector<int> &k_reach, int nPhi) {
  const int nZ = c.am_n_z_below + c.am_n_z_over + 1;
  for (int r = 0; r < c.am_n_rho; r++)
    if (k_reach[r] > 0 && 2 * k_reach[r] >= r) return 0;
  if (c.am_n_z_below < 1 || c.am_n_z_below >= nZ - 1 || c.am_n_rho >= 4096 || 2 * nPhi > kMaxPhi) return 0;
  return 1;
}
// frame-local voxel grid: the awareness range in voxels plus a margin of a subbox and a cell on every side
void lvg_dims(const mlm_config &c, double *dim_xy, double *dim_z) {
  const int nZ = c.am_n_z_below + c.am_n_z_over + 1;
  const double R = c.am_n_rho * c.am_d_rho, margin = c.subbox_n + 1;
  *dim_xy = ceil(2 * R / c.subbox_d_xyz) + 2 * margin + 2;
  *dim_z = ceil(nZ * c.am_d_z / c.subbox_d_xyz) + 2 * margin + 2;
}

int build_awareness_tables(const mlm_config &c, AwarenessTables &T) {
  const int nRho = c.am_n_rho;
  T.dPhi = c.am_d_phi_deg * M_PI / 180;
  T.nPhi = static_cast<int>(360 / c.am_d_phi_deg);
  T.nZ = c.am_n_z_below + c.am_n_z_over + 1;
  T.z_border_min = -(c.am_n_z_below * c.am_d_z) - 0.5 * c.am_d_z;
  T.odds.resize((size_t)kOddsRows * nRho);
  for (int diff = -kDiffRange; diff < kDiffRange + 1; diff++)
    for (int r = 0; r < nRho; r++)
      T.odds[(size_t)(diff + kDiffRange) * nRho + r] = host_get_odds(c.depth_noise_coe, c.am_d_rho, diff, r);
  T.k_reach.resize(nRho);
  for (int r = 0; r < nRho; r++) T.k_reach[r] = host_k_reach(c, r);
  T.centre_z.resize(T.nZ);
  for (int z = 0; z < T.nZ; z++) T.centre_z[z] = T.z_border_min + (c.am_d_z / 2) + (z * c.am_d_z);
  T.centre_xy.resize((size_t)T.nPhi * nRho);
  for (int phi = 0; phi < T.nPhi; phi++)
    for (int rho = 0; rho < nRho; rho++) {
      double center_rho = c.am_d_rho / 2 + (rho * c.am_d_rho);
      double center_phi = T.dPhi / 2 + (phi * T.dPhi);
      T.centre_xy[(size_t)phi * nRho + rho] = make_double2(center_rho * cos(center_phi), center_rho * sin(center_phi));
    }
  return MLM_OK;
}

int validate_config(const mlm_config &c, std::string &why) {
  auto bad = [&](const char *m) {
    why = m;
    return MLM_ERR_INVALID_CONFIG;
  };
  if (!(c.am_d_rho > 0) || !(c.am_d_phi_deg > 0) || !(c.am_d_z > 0)) return bad("awareness resolutions must be > 0");
  if (c.am_n_rho < 2 || c.am_n_z_below < 0 || c.am_n_z_over < 0) return bad("awareness extents");
  if (c.am_n_rho >= 4096) return bad("n_Rho must be < 4096");
  if (!(c.subbox_d_xyz > 0) || c.subbox_n < 1 || c.subbox_n > 64) return bad("subbox size");
  // the reference marks a collapsed subbox by a one-element cell vector (map_local.h:215-231): with one cell per subbox
  // every subbox looks collapsed once it exists, so later frames and queries skip it
  if (c.subbox_n == 1) return bad("subbox_n must be >= 2: a one-cell subbox is indistinguishable from a collapsed one");
  if (!(c.depth_noise_coe >= 0)) return bad("depth_noise_coe");
  if (c.max_points < 1 || c.max_points > (1 << 26)) return bad("max_points must be in [1, 2^26]");
  if (c.pool_submaps < 1) return bad("pool_submaps");
  int nPhi = static_cast<int>(360 / c.am_d_phi_deg);
  if (nPhi < 1 || nPhi > kMaxPhi) return bad("n_Phi out of supported range [1,4096]");
  int nZ = c.am_n_z_below + c.am_n_z_over + 1;
  if ((long long)nZ * c.am_n_rho >= (1ll << kCellBits)) return bad("n_Z*n_Rho must be < 2^20");
  if ((long long)nZ * c.am_n_rho * nPhi >= (1ll << 31)) return bad("awareness cell count must be < 2^31");
  // preconditions of update_hits (SURVEY §8a a3): table row index diff_r+10 <= 20 and rho-diff_r >= 0
  std::vector<int> K(c.am_n_rho);
  for (int r = 0; r < c.am_n_rho; r++) {
    K[r] = host_k_reach(c, r);
    if (K[r] > kDiffRange || K[r] > r)
      return bad("depth_noise_coe too large: 3*sigma_in_dr(rho) reaches outside the odds table / below rho 0");
  }
  double lvg_xy, lvg_z;
  lvg_dims(c, &lvg_xy, &lvg_z);
  if (!(lvg_xy * lvg_xy * lvg_z < 2147483648.0)) return bad("frame-local voxel grid too large (awareness range / voxel size)");
  // shared memory per block of the frame kernels on sm_100 (227 KB opt-in, 1 KB reserved); mlm_create checks the
  // device's own limit again.  The projection keeps a histogram per work column; the column item keeps two column
  // bitmaps, the odds table and at least a 32 KB sort buffer.
  const int nCol = nPhi * (half_column_split(c, K, nPhi) ? 2 : 1);
  const long long smem = kSmemOptinSm100 - 1024;
  if ((long long)project_smem_bytes(nCol, kProjThreads) > smem) return bad("n_Phi too large for the projection's shared-memory histogram");
  if (smem - (long long)col_smem_prefix_bytes(nZ * ((c.am_n_rho + 31) / 32), c.am_n_rho, nCol) < 32 * 1024)
    return bad("awareness column (n_Z*n_Rho bits) does not fit shared memory");
  return MLM_OK;
}

int map_device_error(int e) {
  switch (e) {
    case 0: return MLM_OK;
    case kErrRange: return MLM_ERR_INVALID_ARG;
    case kErrPool: return MLM_ERR_POOL_EXHAUSTED;
    case kErrCapacity: return MLM_ERR_CAPACITY;
    default: return MLM_ERR_CUDA;
  }
}

inline int grid_for(size_t n, int threads) { return (int)std::max<size_t>(1, (n + threads - 1) / threads); }

// the frame kernels of each input mode: 0 = points, 1 = full depth image, 2 = sampled depth pixels
using FrameKernel = void (*)(MapParams, DeviceBuffers, FrameParams);
const FrameKernel kProjectKernels[3] = {k_project<0>, k_project<1>, k_project<2>};
const FrameKernel kFrameKernels[3] = {k_frame<0>, k_frame<1>, k_frame<2>};
const FrameKernel kFrameExploreKernels[3] = {k_frame_explore<0>, k_frame_explore<1>, k_frame_explore<2>};

// full bitonic sort of keys[0..n_pad) ascending on the handle's stream
void device_sort(mlm_map *h, uint64_t *keys, int n_pad) {
  if (n_pad <= 1) return;
  const int chunk = std::min(kSortChunk, n_pad);
  const int nchunks = n_pad / chunk;
  k_bitonic_local<<<nchunks, kSortThreads, 0, h->stream>>>(keys, n_pad, 2, chunk);
  h->launches++;
  for (int k = chunk << 1; k <= n_pad; k <<= 1) {
    for (int j = k >> 1; j >= chunk; j >>= 1) {
      k_bitonic_global<<<grid_for(n_pad >> 1, 256), 256, 0, h->stream>>>(keys, n_pad, j, k);
      h->launches++;
    }
    k_bitonic_local<<<nchunks, kSortThreads, 0, h->stream>>>(keys, n_pad, k, k);
    h->launches++;
  }
}

// Re-sequences a set whose n distinct keys (O) exceed its emulated bucket count B_start, so that libstdc++ would rehash
// mid-frame (possibly several times).  Produces virtual positions in O.stamp and bucket activations in act for the
// final bucket count, which it returns in *B_final.
int resequence(mlm_map *h, const OrderArrays &O, int n, uint32_t *act, uint32_t act_cap, uint32_t B_start,
               uint32_t *B_final) {
  cudaStream_t s = h->stream;
  const int T = 256;
  int n_pad = next_pow2(n);
  k_order_seed<<<grid_for(n_pad, T), T, 0, s>>>(O, h->d_sort_a, n, n_pad);
  device_sort(h, h->d_sort_a, n_pad);
  k_order_take_seq<<<grid_for(n, T), T, 0, s>>>(h->d_sort_a, h->d_seq_a, n);
  h->launches += 2;
  uint32_t B = B_start;
  while ((uint32_t)n > B) {
    int m = (int)std::min<uint32_t>(B, (uint32_t)n);
    if (m > 1) {
      int m_pad = next_pow2(m);
      k_fill_u32<<<grid_for(B, T), T, 0, s>>>(act, 0xffffffffu, (int)B);
      k_stage_act<<<grid_for(m, T), T, 0, s>>>(h->P, O, act, h->d_seq_a, m, B);
      k_stage_keys<<<grid_for(m_pad, T), T, 0, s>>>(h->P, O, act, h->d_seq_a, h->d_sort_b, m, m_pad, B);
      device_sort(h, h->d_sort_b, m_pad);
      k_stage_apply<<<grid_for(m, T), T, 0, s>>>(h->d_sort_b, h->d_seq_a, h->d_seq_b, m);
      k_copy_i32<<<grid_for(m, T), T, 0, s>>>(h->d_seq_a, h->d_seq_b, m);
      h->launches += 5;
    }
    uint32_t nb = chain_next(B);
    if (nb == 0 || nb > act_cap) {
      g_last_error = "bucket chain of the emulated container exceeded";
      return MLM_ERR_CAPACITY;
    }
    B = nb;
  }
  k_fill_u32<<<grid_for(B, T), T, 0, s>>>(act, 0xffffffffu, (int)B);
  k_order_final<<<grid_for(n, T), T, 0, s>>>(h->P, O, act, h->d_seq_a, n, B);
  h->launches += 2;
  *B_final = B;
  return MLM_OK;
}

// Slow ordering path of the frame's own sets.  kind 0: the hit map (hit_key / hit_t / hit_bucket, act[parity]);
// kind 1: the miss set of exploration mode
int order_slow_path(mlm_map *h, int n, int kind, uint32_t B_start, uint32_t *B_final_out) {
  OrderArrays O;
  O.key = kind == 0 ? h->D.hit_key : h->D.miss_idx;
  O.stamp = kind == 0 ? h->D.hit_t : h->D.miss_t;
  O.bucket = kind == 0 ? h->D.hit_bucket : h->D.miss_bucket;
  O.kind = kind;
  uint32_t *act = kind == 0 ? h->D.act[h->last_parity] : h->D.act_miss[h->last_parity];
  return resequence(h, O, n, act, kind == 0 ? h->act_cap : h->act_miss_cap, B_start, B_final_out);
}

// The ordering of a frame whose staged sets cross a rehash: re-sequences the hit map (n_hit keys) and, in the
// exploration mode, the miss set (n_miss keys; 0 otherwise) when they outgrow their emulated bucket counts, and gives
// the frame's parameters the final counts.  Sets *slow and *order_B (the hit map's final count) when it re-sequences.
int settle_rehash(mlm_map *h, int n_hit, int n_miss, int *slow, uint32_t *order_B) {
  if (n_hit > h->sort_cap || n_miss > h->sort_cap) {
    g_last_error = "hit / miss count exceeds ordering scratch";
    return MLM_ERR_CAPACITY;
  }
  FrameParams &F = *h->h_fp;
  if ((uint32_t)n_hit > h->bucket_count) {
    *slow = 1;
    const int rc = order_slow_path(h, n_hit, 0, h->bucket_count, order_B);
    if (rc != MLM_OK) return rc;
    F.bucket_count = *order_B;
    F.bucket_c64 = pow64_mod(F.bucket_count);
  }
  if ((uint32_t)n_miss > h->bucket_count_miss) {
    *slow = 1;
    const int rc = order_slow_path(h, n_miss, 1, h->bucket_count_miss, &F.bucket_count_miss);
    if (rc != MLM_OK) return rc;
  }
  return MLM_OK;
}

int finish_frame(mlm_map *h, int slow, uint32_t order_B, mlm_frame_stats *stats);
int run_frame_complete(mlm_map *h, mlm_frame_stats *stats);

// Exploration mode (use_exploration_frontiers): the frame needs the neighbours' state between the hit and
// the miss pass, and the miss-set iteration order, so it runs as direct launches with one host check of the
// container sizes in the middle (rehash detection for both emulated containers).
int run_frame_explore_direct(mlm_map *h, int slow, uint32_t order_B, mlm_frame_stats *stats);
int run_frame_explore(mlm_map *h, int mode, int N, mlm_frame_stats *stats) {
  const MapParams &P = h->P;
  cudaStream_t s = h->stream;
  FrameParams &F = *h->h_fp;
  const int parity = F.parity;
  const int proj_grid = grid_for((size_t)std::max(N, 1), kProjThreads * 2);
  F.order_mode = 1;  // rehash detection happens on the host below, not inside k_fuse
  kProjectKernels[mode]<<<proj_grid, kProjThreads, project_smem_bytes(P.nCol, kProjThreads), s>>>(P, h->D, F);
  k_column<<<h->col_grid, kColThreads, h->col_smem_bytes, s>>>(P, h->D, F);
  if (P.split) {
    k_miss_finalize<<<h->sm_count * 4, 256, 0, s>>>(P, h->D, F);
    h->launches++;
  }
  FrameCounters mid;
  CUDA_TRY(cudaMemcpyAsync(&mid, h->D.fc[parity], sizeof(mid), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  h->launches += 2;
  int slow = 0;
  uint32_t order_B = h->bucket_count;
  if (mid.error == 0) {
    const int rc = settle_rehash(h, mid.n_hit, mid.n_miss_list, &slow, &order_B);
    if (rc != MLM_OK) {
      h->poisoned = true;  // the frame's staging stays unconsumed
      return rc;
    }
  }
  if (h->stage_call) {  // awareness layer only: the local layer follows with mlm_local_input_pc_pose_direct
    *h->h_fc = mid;
    h->staged = true;
    h->staged_slow = slow;
    h->staged_order_B = order_B;
    h->last_order_B = order_B;
    h->last_n_hit = mid.n_hit;
    return MLM_OK;
  }
  return run_frame_explore_direct(h, slow, order_B, stats);
}
int run_frame_explore_direct(mlm_map *h, int slow, uint32_t order_B, mlm_frame_stats *stats) {
  const MapParams &P = h->P;
  cudaStream_t s = h->stream;
  FrameParams &F = *h->h_fp;
  const int parity = F.parity;
  const int g4 = h->sm_count * 4;
  k_fuse<1><<<g4, 256, 0, s>>>(P, h->D, F);
  k_miss_tkey<<<g4, 256, 0, s>>>(P, h->D, F);
  k_explore_a<<<g4, 256, 0, s>>>(P, h->D, F);
  k_explore_b<<<g4, 256, 0, s>>>(P, h->D, F);
  k_fuse<2><<<g4, 256, 0, s>>>(P, h->D, F);
  k_release<<<h->sm_count, 256, 0, s>>>(P, h->D, F);
  h->launches += 6;
  CUDA_TRY(cudaMemcpyAsync(h->h_fc, h->D.fc[parity], sizeof(FrameCounters), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  h->bucket_count_miss = bucket_growth(h->bucket_count_miss, h->h_fc->n_miss_list);
  return finish_frame(h, slow, order_B, stats);
}
// the rest of a normal frame whose sets are staged and ordered: the fusion pass as a stand-alone kernel
int run_frame_fuse_direct(mlm_map *h, int slow, uint32_t order_B, mlm_frame_stats *stats) {
  cudaStream_t s = h->stream;
  k_fuse<0><<<h->sm_count * 4, 256, 0, s>>>(h->P, h->D, *h->h_fp);
  h->launches++;
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return finish_frame(h, slow, order_B, stats);
}

// mode: 0 = points, 1 = full depth image, 2 = sampled depth pixels (d_in = uint2 {pixel, raw} x n_points)
int run_frame(mlm_map *h, int mode, const void *d_in, int rows, int cols, int n_points, const double T_wb[7],
              mlm_frame_stats *stats) {
  if (h->poisoned) {
    g_last_error = "an earlier frame failed after staging its sets (capacity); the handle refuses further frames: restore a "
                   "checkpoint into a fresh handle";
    return MLM_ERR_CAPACITY;
  }
  if (h->staged || h->frame_pending) {
    g_last_error = h->staged ? "an awareness-layer update is waiting for mlm_local_input_pc_pose_direct"
                             : "a submitted frame is waiting for mlm_frame_finish";
    return MLM_ERR_INVALID_ARG;
  }
  const bool depth = mode == 1;
  const MapParams &P = h->P;
  cudaStream_t s = h->stream;
  const int N = depth ? rows * cols : n_points;  // sampled mode: n_points sampled pixels of a rows x cols image
  if (N < 0 || N > P.max_points) {
    g_last_error = "frame has more points than cfg.max_points";
    return MLM_ERR_CAPACITY;
  }
  // input_pc_pose prologue, src/map_awareness.cpp:184-186
  HPose Twb = h_pose_from7(T_wb);
  HPose Twa;
  Twa.q = h_normalized(HQuat{1, 0, 0, 0});
  Twa.t[0] = Twb.t[0];
  Twa.t[1] = Twb.t[1];
  Twa.t[2] = Twb.t[2];
  HPose Tws = h_compose(Twb, h->T_bs);
  HPose Tls = h_compose(h_inverse(Twa), Tws);
  FrameParams &F = *h->h_fp;
  F.q_ls[0] = Tls.q.w;
  F.q_ls[1] = Tls.q.x;
  F.q_ls[2] = Tls.q.y;
  F.q_ls[3] = Tls.q.z;
  for (int i = 0; i < 3; i++) {
    F.t_ls[i] = Tls.t[i];
    F.t_wa[i] = Twa.t[i];
  }
  F.input = d_in;
  F.rows = rows;
  F.cols = cols;
  F.cols_shift = 0;
  while ((2 << F.cols_shift) <= std::max(cols - 1, 1)) F.cols_shift++;  // floor(log2(cols - 1))
  F.cols_magic = cols >= 2 ? (uint32_t)(((1ull << (32 + F.cols_shift)) / (uint64_t)cols) + 1) : 0u;  // 0: plain division
  F.n_points = n_points;
  F.n_total = N;
  F.bucket_count = h->bucket_count;
  F.bucket_c64 = pow64_mod(F.bucket_count);
  F.bucket_count_miss = h->bucket_count_miss;
  const int parity = (int)(h->frame_idx & 1);
  h->frame_idx++;
  h->last_parity = parity;
  F.parity = parity;
  F.order_mode = 0;
  F.shard_rank = 0;
  F.shard_world = 1;
  F.stage_only = 0;
  F.inline_resolve = 0;
  F.skip_flag = nullptr;
  F.frame_seq = 0;
  F.tbits = 1;
  while ((1ll << F.tbits) < (long long)std::max(N, 2)) F.tbits++;
  F.tile_pts = kProjThreads * 2;  // stand-alone k_project: 512 threads x 2 rounds per warp
  // frame-local voxel grid origin: awareness bounding box around t_wa plus a margin
  const double R = P.nRho * P.dRho;
  F.lvg_base[0] = (int)floor((Twa.t[0] - R) / P.d_sub) - P.lvg_margin;
  F.lvg_base[1] = (int)floor((Twa.t[1] - R) / P.d_sub) - P.lvg_margin;
  F.lvg_base[2] = (int)floor((Twa.t[2] + P.z_border_min) / P.d_sub) - P.lvg_margin;
  for (int i = 0; i < 3; i++) F.lsg_base[i] = host_floor_div(F.lvg_base[i], P.n) - 1;

  if (h->shard_world > 0 && h->shard_stage_pending) {
    // sharded staging: project + column only; records are emitted and fused by the mlm_shard_* calls
    F.shard_rank = h->shard_rank;
    F.shard_world = h->shard_world;
    F.stage_only = 1;
    F.inline_resolve = 1;  // voxels of subboxes this rank owns are staged as on one GPU: the first toucher resolves the subbox
    F.order_mode = 1;
    const int pg = grid_for((size_t)std::max(N, 1), kProjThreads * 2);
    if (F.bucket_count == 1) F.bucket_count = 13, F.bucket_c64 = pow64_mod(13);  // the first insert of an empty table allocates 13 buckets before anything is ordered
    k_project<0><<<pg, kProjThreads, project_smem_bytes(P.nCol, kProjThreads), s>>>(P, h->D, F);
    if (h->profiling && h->sev[2]) cudaEventRecord(h->sev[2], s);
    k_column<<<h->col_grid, kColThreads, h->col_smem_bytes, s>>>(P, h->D, F);
    h->launches += 2;
    return MLM_OK;  // no host sync: the exchange and the owner-side kernels follow on the stream (mlm_shard_submit_*)
  }
  // exploration mode: one cooperative launch like a normal frame; the stand-alone passes serve the two-call interface,
  // profiling runs and devices / configurations without the cooperative launch
  if (P.explore && (h->stage_call || h->profiling || !h->use_fused)) return run_frame_explore(h, mode, N, stats);
  if (h->stage_call) {
    // awareness layer only (awareness_map_cylindrical::input_pc_pose): hit map + miss set of the frame, staged in the
    // frame-local voxel grid; the ordering of a rehash frame is settled here so that the frame's sets can be read
    const int pg = grid_for((size_t)std::max(N, 1), kProjThreads * 2);
    kProjectKernels[mode]<<<pg, kProjThreads, project_smem_bytes(P.nCol, kProjThreads), s>>>(P, h->D, F);
    k_column<<<h->col_grid, kColThreads, h->col_smem_bytes, s>>>(P, h->D, F);
    h->launches += 2;
    CUDA_TRY(cudaMemcpyAsync(h->h_fc, h->D.fc[parity], sizeof(FrameCounters), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
    int slow = 0;
    uint32_t order_B = h->bucket_count;
    const int n = h->h_fc->n_hit;
    if (h->h_fc->error == 0 && (uint32_t)n > h->bucket_count) {
      const int rc = settle_rehash(h, n, 0, &slow, &order_B);
      if (rc != MLM_OK) return rc;
      F.order_mode = 1;
      CUDA_TRY(cudaStreamSynchronize(s));
    }
    h->staged = true;
    h->staged_slow = slow;
    h->staged_order_B = order_B;
    h->last_order_B = order_B;
    h->last_n_hit = n;
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->n_points = h->h_fc->n_points;
      stats->n_inside = h->h_fc->n_inside;
      stats->n_cast = h->h_fc->n_cast;
      stats->n_hit_cells = h->h_fc->n_hit;
      stats->n_miss_cells = h->h_fc->n_miss;
      stats->ordering_slow_path = slow;
      stats->status = map_device_error(h->h_fc->error);
    }
    return h->h_fc->error ? map_device_error(h->h_fc->error) : MLM_OK;
  }
  const bool prof = h->profiling != 0;
  const int full_grid = grid_for((size_t)P.max_points, kProjThreads * 2);
  const int proj_grid = grid_for((size_t)std::max(N, 1), kProjThreads * 2);
  MapParams Pk = P;
  DeviceBuffers Dk = h->D;
  FrameParams Fk = F;
  void *kargs[3] = {&Pk, &Dk, &Fk};
  if (prof) {
    cudaEventRecord(h->kev[0], s);
    kProjectKernels[mode]<<<proj_grid, kProjThreads, project_smem_bytes(P.nCol, kProjThreads), s>>>(Pk, Dk, Fk);
    cudaEventRecord(h->kev[1], s);
    k_column<<<h->col_grid, kColThreads, h->col_smem_bytes, s>>>(Pk, Dk, Fk);
    cudaEventRecord(h->kev[2], s);
    k_fuse<0><<<h->sm_count * 4, 256, 0, s>>>(Pk, Dk, Fk);
    cudaEventRecord(h->kev[3], s);
  } else if (h->use_fused) {
    // the whole frame is ONE cooperative kernel (k_frame), replayed as a single-node graph
    const int G = h->frame_sms > 0 ? std::min(h->frame_sms, h->frame_grid) : h->frame_grid;
    // one tile per CTA when the frame allows it: N points dealt evenly, in 32-point rounds, at most 128 per warp
    Fk.tile_pts = std::min(kProjMaxPts * kColThreads, std::max(32, (((N + G - 1) / G) + 31) & ~31));
    F.tile_pts = Fk.tile_pts;
    if (!h->async_call) {
      Fk.frame_seq = F.frame_seq = ++h->frame_seq ? h->frame_seq : ++h->frame_seq;
      h->h_fc->seq = 0;
    }
    Fk.inline_resolve = F.inline_resolve = 1;
    const int gi = mode;
    cudaKernelNodeParams np = {};
    np.func = (void *)(P.explore ? kFrameExploreKernels : kFrameKernels)[mode];
    np.gridDim = dim3(G);
    np.blockDim = dim3(kColThreads);
    np.sharedMemBytes = (unsigned)h->col_smem_bytes;
    np.kernelParams = kargs;
    if (!h->fgraph_exec[gi]) {
      CUDA_TRY(cudaGraphCreate(&h->fgraph[gi], 0));
      CUDA_TRY(cudaGraphAddKernelNode(&h->fgraph_node[gi], h->fgraph[gi], nullptr, 0, &np));
      cudaKernelNodeAttrValue av = {};
      av.cooperative = 1;
      CUDA_TRY(cudaGraphKernelNodeSetAttribute(h->fgraph_node[gi], cudaKernelNodeAttributeCooperative, &av));
      CUDA_TRY(cudaGraphInstantiate(&h->fgraph_exec[gi], h->fgraph[gi], 0));
    } else {
      CUDA_TRY(cudaGraphExecKernelNodeSetParams(h->fgraph_exec[gi], h->fgraph_node[gi], &np));
    }
    CUDA_TRY(cudaGraphLaunch(h->fgraph_exec[gi], s));
  } else {
    // the whole frame is one launch of a 3-kernel graph; the per-frame values travel as kernel arguments
    const int gi = mode;
    cudaKernelNodeParams np[3] = {};
    np[0].func = (void *)kProjectKernels[mode];
    np[0].gridDim = dim3(full_grid);  // fixed grid: CTAs beyond this frame's point count return at once
    np[0].blockDim = dim3(kProjThreads);
    np[0].sharedMemBytes = (unsigned)(project_smem_bytes(P.nCol, kProjThreads));
    np[1].func = (void *)k_column;
    np[1].gridDim = dim3(h->col_grid);
    np[1].blockDim = dim3(kColThreads);
    np[1].sharedMemBytes = (unsigned)h->col_smem_bytes;
    np[2].func = (void *)k_fuse<0>;
    np[2].gridDim = dim3(h->sm_count * 4);
    np[2].blockDim = dim3(256);
    np[2].sharedMemBytes = 0;
    for (int i = 0; i < 3; i++) np[i].kernelParams = kargs;
    if (!h->graph_exec[gi]) {
      CUDA_TRY(cudaGraphCreate(&h->graph[gi], 0));
      for (int i = 0; i < 3; i++)
        CUDA_TRY(cudaGraphAddKernelNode(&h->graph_nodes[gi][i], h->graph[gi], i ? &h->graph_nodes[gi][i - 1] : nullptr,
                                        i ? 1 : 0, &np[i]));
      CUDA_TRY(cudaGraphInstantiate(&h->graph_exec[gi], h->graph[gi], 0));
    } else {
      for (int i = 0; i < 3; i++) CUDA_TRY(cudaGraphExecKernelNodeSetParams(h->graph_exec[gi], h->graph_nodes[gi][i], &np[i]));
    }
    CUDA_TRY(cudaGraphLaunch(h->graph_exec[gi], s));
  }
  h->launches += (prof || !h->use_fused) ? 3 : 1;
  if (h->async_call) {  // mlm_frame_finish waits, settles a rehash frame and returns the counters
    h->frame_pending = true;
    h->pending_mode = mode;
    return MLM_OK;
  }
  return run_frame_complete(h, stats);
}

// second half of a frame: wait for the launch, run the rehash path when the frame needs it, counters
int run_frame_complete(mlm_map *h, mlm_frame_stats *stats) {
  const MapParams &P = h->P;
  cudaStream_t s = h->stream;
  FrameParams &F = *h->h_fp;
  const bool prof = h->profiling != 0;
  bool polled = false;
  if (F.frame_seq) {
    // the frame kernel stores the counters, then its sequence number, in mapped host memory before it rearms the next
    // frame's scratch: poll that word (a PCIe write away) instead of waiting for the stream to drain; what follows on
    // the stream is ordered behind the kernel anyway.  Falls back to the stream after 2 ms (a frame that takes that long
    // is on the rehash path or in trouble).
    volatile uint32_t *seq = &h->h_fc->seq;
    const auto t0 = std::chrono::steady_clock::now();
    for (int spin = 0;; spin++) {
      if (*seq == F.frame_seq) {
        polled = true;
        break;
      }
      if ((spin & 1023) == 1023 && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(2)) break;
      __builtin_ia32_pause();
    }
    std::atomic_thread_fence(std::memory_order_acquire);
  }
  if (!polled) {
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaGetLastError());
  }

  if (prof)
    for (int i = 0; i < MLM_NUM_FRAME_KERNELS; i++) cudaEventElapsedTime(&h->kms[i], h->kev[i], h->kev[i + 1]);
  int slow = 0;
  uint32_t order_B = h->bucket_count;
  if (h->h_fc->error == 0 && h->h_fc->overflow) {
    // the frame crosses a rehash of the hit map (exploration mode: or of the miss set) and the kernel returned after
    // staging: re-sequence what needs it and run the rest of the frame as stand-alone kernels
    F.order_mode = 1;
    const int rc = settle_rehash(h, h->h_fc->n_hit, P.explore ? h->h_fc->n_miss_list : 0, &slow, &order_B);
    if (rc != MLM_OK) {
      h->poisoned = true;  // the frame's staging stays unconsumed
      return rc;
    }
    return P.explore ? run_frame_explore_direct(h, slow, order_B, stats) : run_frame_fuse_direct(h, slow, order_B, stats);
  }
  if (P.explore) h->bucket_count_miss = bucket_growth(h->bucket_count_miss, h->h_fc->n_miss_list);
  return finish_frame(h, slow, order_B, stats);
}

int finish_frame(mlm_map *h, int slow, uint32_t order_B, mlm_frame_stats *stats) {
  const FrameCounters &C = *h->h_fc;
  if (C.fused) {
    h->cum_ram_expand += C.n_new_blocks;
    h->cum_obs += C.obs_delta;
    h->n_submaps += C.n_new_blocks;
  }
  h->bucket_count = bucket_growth(h->bucket_count, C.n_hit);  // hit_idx_odds_hashmap
  h->last_order_B = order_B;
  h->last_n_hit = C.n_hit;
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_points = C.n_points;
    stats->n_inside = C.n_inside;
    stats->n_cast = C.n_cast;
    stats->n_hit_cells = C.n_hit;
    stats->n_miss_cells = C.n_miss;
    stats->n_touched_voxels = C.n_touched_voxels;
    stats->n_new_submaps = C.n_new_blocks;
    stats->hit_bucket_count = (int32_t)h->bucket_count;
    stats->ordering_slow_path = slow;
    stats->status = map_device_error(C.error);
    stats->ram_expand_cnt = h->cum_ram_expand;
    stats->obs_cnt = h->cum_obs;
  }
  if (C.error) {
    g_last_error = "device raised error code " + std::to_string(C.error);
    return map_device_error(C.error);
  }
  return MLM_OK;
}

// input staging (device buffer + pinned host mirror).  `bytes` is what this frame needs, `capacity` what the
// handle can ever need for this input kind: allocated once at capacity so frames of varying size never re-allocate
int ensure_input(mlm_map *h, size_t bytes, size_t capacity = 0) {
  if (bytes <= h->input_bytes) return MLM_OK;
  bytes = std::max(bytes, capacity);
  if (h->d_input) cudaFree(h->d_input);
  if (h->h_stage) cudaFreeHost(h->h_stage);
  h->d_input = nullptr;
  h->h_stage = nullptr;
  CUDA_TRY(cudaMalloc(&h->d_input, bytes));
  CUDA_TRY(cudaMallocHost(&h->h_stage, bytes));
  h->input_bytes = h->stage_bytes = bytes;
  return MLM_OK;
}

// host variant of a point query: the device variant's launch, with points and results staged through temporaries
template <typename OutT, typename... Args>
int host_query(mlm_handle h, const double *pos, size_t n, OutT *out, size_t out_per,
               void (*launch)(mlm_handle, const double *, size_t, OutT *, Args...), Args... args) {
  if (!h || (!pos && n) || (!out && n)) return MLM_ERR_INVALID_ARG;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  {
    StreamTemp<double> d_pos(h->stream);
    StreamTemp<OutT> d_out(h->stream);
    CUDA_TRY(d_pos.alloc(n * 3));
    CUDA_TRY(d_out.alloc(n * out_per));
    CUDA_TRY(cudaMemcpyAsync(d_pos, pos, n * 24, cudaMemcpyHostToDevice, h->stream));
    launch(h, d_pos, n, d_out, args...);
    CUDA_TRY(cudaMemcpyAsync(out, d_out, n * out_per * sizeof(OutT), cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
}  // namespace

extern "C" {

// depth_odom_input_callback's pose forwarding, src/mlmap.cpp:470-498: host-side, once per frame, no device work.
// SO3::log / SO3::exp as in 3rdPartLib/Sophus/sophus/so3.cpp:127-199 (SMALL_EPS 1e-10, so3.h:35), rot_og.matrix()
// as Eigen's Quaternion::toRotationMatrix.
int mlm_compensate_pose(const double odom_pos[3], const double odom_quat_wxyz[4], const double odom_lin_vel[3],
                        const double imu_ang_vel[3], double gap_odom_s, double gap_imu_s, double camera2odom_latency_s,
                        double T_wb_out[7]) {
  if (!odom_pos || !odom_quat_wxyz || !odom_lin_vel || !imu_ang_vel || !T_wb_out) return MLM_ERR_INVALID_ARG;
  const double time_gap = gap_imu_s - camera2odom_latency_s;
  const HQuat q = h_normalized(HQuat{odom_quat_wxyz[0], odom_quat_wxyz[1], odom_quat_wxyz[2], odom_quat_wxyz[3]});
  // rot_dot = rot_og.matrix() * angular velocity
  const double tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
  const double twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const double txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const double tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  const double m[3][3] = {{1 - (tyy + tzz), txy - twz, txz + twy}, {txy + twz, 1 - (txx + tzz), tyz - twx}, {txz - twy, tyz + twx, 1 - (txx + tyy)}};
  double rot_dot[3];
  // Matrix3d * Vector3d as Eigen's coefficient-based product evaluates it: rows 0-1 are one packet accumulated in
  // order, the odd last row is a scalar dot product reduced as a halving tree
  for (int i = 0; i < 2; i++) rot_dot[i] = (imu_ang_vel[0] * m[i][0] + imu_ang_vel[1] * m[i][1]) + imu_ang_vel[2] * m[i][2];
  rot_dot[2] = m[2][0] * imu_ang_vel[0] + (m[2][1] * imu_ang_vel[1] + m[2][2] * imu_ang_vel[2]);
  // rot_cp = rot_og.log() + time_gap * rot_dot
  const double n = sqrt(q.x * q.x + q.y * q.y + q.z * q.z);
  const double w = q.w, squared_w = w * w;
  double k;
  if (n < 1e-10)
    k = 2. / w - 2. * (n * n) / (w * squared_w);
  else
    k = 2 * atan(n / w) / n;  // the reference's |w| < SMALL_EPS branch is overwritten by this statement (so3.cpp:152-165)
  const double lg[3] = {k * q.x, k * q.y, k * q.z};
  double rc[3];
  for (int i = 0; i < 3; i++) rc[i] = lg[i] + rot_dot[i] * time_gap;
  // SO3::exp(rot_cp)
  const double theta = sqrt(rc[0] * rc[0] + rc[1] * rc[1] + rc[2] * rc[2]);
  const double half_theta = 0.5 * theta;
  const double real_factor = cos(half_theta);
  double imag_factor;
  if (theta < 1e-10) {
    const double theta_sq = theta * theta, theta_po4 = theta_sq * theta_sq;
    imag_factor = 0.5 - 0.0208333 * theta_sq + 0.000260417 * theta_po4;
  } else {
    imag_factor = sin(half_theta) / theta;
  }
  const HQuat e = h_normalized(HQuat{real_factor, imag_factor * rc[0], imag_factor * rc[1], imag_factor * rc[2]});
  const double dt = gap_odom_s - camera2odom_latency_s;
  for (int i = 0; i < 3; i++) T_wb_out[i] = odom_pos[i] + odom_lin_vel[i] * dt;
  T_wb_out[3] = e.w;
  T_wb_out[4] = e.x;
  T_wb_out[5] = e.y;
  T_wb_out[6] = e.z;
  return MLM_OK;
}

int mlm_abi_version(void) { return MLM_ABI_VERSION; }
size_t mlm_sizeof_config(void) { return sizeof(mlm_config); }
size_t mlm_sizeof_frame_stats(void) { return sizeof(mlm_frame_stats); }
const char *mlm_last_error(void) { return g_last_error.c_str(); }

int mlm_default_config(mlm_config *c) {
  if (!c) return MLM_ERR_INVALID_ARG;
  memset(c, 0, sizeof(*c));
  // reference launch/config/config_sim.yaml:8-55
  c->am_d_rho = 0.20;
  c->am_d_phi_deg = 5;
  c->am_d_z = 0.20;
  c->am_n_rho = 40;
  c->am_n_z_below = 20;
  c->am_n_z_over = 20;
  c->use_raycasting = 1;
  c->depth_noise_coe = 0.000001;
  c->subbox_d_xyz = 0.2;
  c->subbox_n = 10;
  c->log_odds_min = -2.0f;
  c->log_odds_max = 4.2f;
  c->log_odds_hit = 0.7f;
  c->log_odds_miss = -0.9f;
  c->log_odds_occupied_sh = 3.0f;
  c->use_exploration_frontiers = 0;
  c->cam_cx = 320.0f;
  c->cam_cy = 180.0f;
  c->cam_fx = 347.99755859375f;
  c->cam_fy = 347.99755859375f;
  // T_B_S rotation [[0,0,1],[-1,0,0],[0,-1,0]] as a unit quaternion, translation (0.12,0,0)
  c->T_bs[0] = 0.12;
  c->T_bs[1] = 0.0;
  c->T_bs[2] = 0.0;
  c->T_bs[3] = 0.5;
  c->T_bs[4] = -0.5;
  c->T_bs[5] = 0.5;
  c->T_bs[6] = -0.5;
  c->inflate_n = 2;
  c->inflate_global_n = 2;
  c->apply_inflate = 1;
  c->inflate_height = 0.1;
  c->sample_cnt = 500;  // mlmapping_sample_cnt (config_sim.yaml:37); 0 selects the full-frame mode of the north star
  c->max_points = 640 * 480;
  c->pool_submaps = 32768;
  return MLM_OK;
}

int mlm_create(const mlm_config *cfg, int device, mlm_handle *out) {
  if (!cfg || !out) return MLM_ERR_INVALID_ARG;
  *out = nullptr;
  std::string why;
  int rc = validate_config(*cfg, why);
  if (rc != MLM_OK) {
    g_last_error = why;
    return rc;
  }
  if (cfg->sample_cnt < 0 || cfg->sample_cnt > cfg->max_points) {
    g_last_error = "sample_cnt must be in [0, max_points]";
    return MLM_ERR_INVALID_CONFIG;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
    cudaGetLastError();
    g_last_error = "no CUDA device available: the mlmap_b200 hot path has no CPU fallback";
    return MLM_ERR_NO_DEVICE;
  }
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    g_last_error = "kernels are built for sm_100a only; found sm_" + std::to_string(prop.major * 10 + prop.minor);
    return MLM_ERR_NO_DEVICE;
  }

  AwarenessTables T;
  build_awareness_tables(*cfg, T);
  int maxK = 0;  // validate_config has checked update_hits' preconditions
  for (int r = 0; r < cfg->am_n_rho; r++) maxK = std::max(maxK, T.k_reach[r]);
  // test hooks: force the paths that other devices and configurations take.  MLM_NO_FUSED: the three-kernel graph of
  // devices without the cooperative launch; MLM_DEBUG_NO_SPLIT: whole phi columns as work items; MLM_DEBUG_SORT_CAP /
  // MLM_DEBUG_MAP_CAP: smaller shared-memory capacities, i.e. the global-memory fallback paths
  const auto env_flag = [](const char *name) {
    const char *e = getenv(name);
    return e && atoi(e) != 0;
  };
  const bool no_fused = env_flag("MLM_NO_FUSED"), no_split = env_flag("MLM_DEBUG_NO_SPLIT");
  const char *sort_cap_env = getenv("MLM_DEBUG_SORT_CAP"), *map_cap_env = getenv("MLM_DEBUG_MAP_CAP");

  mlm_map *h = new mlm_map();
  h->cfg = *cfg;
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->T_bs = h_pose_from7(cfg->T_bs);
  MapParams &P = h->P;
  memset(&P, 0, sizeof(P));
  P.dRho = cfg->am_d_rho;
  P.dPhi = T.dPhi;
  P.dZ = cfg->am_d_z;
  P.z_border_min = T.z_border_min;
  P.nRho = cfg->am_n_rho;
  P.nPhi = T.nPhi;
  P.nZ = T.nZ;
  P.n_below = cfg->am_n_z_below;
  P.visibility_check = cfg->use_raycasting != 0;
  P.maxK = maxK;
  P.words_per_row = (P.nRho + 31) / 32;
  P.col_words = P.nZ * P.words_per_row;
  P.cell_bits = 1;
  while ((1 << P.cell_bits) < P.nZ * P.nRho) P.cell_bits++;
  P.nRho_magic = (uint32_t)(((1ull << 32) + (uint64_t)P.nRho - 1) / (uint64_t)P.nRho);
  P.split = no_split ? 0 : half_column_split(*cfg, T.k_reach, P.nPhi);
  P.nCol = P.nPhi * (P.split ? 2 : 1);
  // per end cell: the ray's slope and the z rows of its neighbour contributions, with the reference's arithmetic
  // (rate = (z - n_below) / (rho * 1.0); (int)round(z +/- d * rate)), src/map_awareness.cpp:64-71,151,161
  T.rate.resize((size_t)P.nZ * P.nRho);
  T.dz.resize((size_t)P.nZ * P.nRho * std::max(maxK, 1));
  for (int z = 0; z < P.nZ; z++)
    for (int rho = 0; rho < P.nRho; rho++) {
      const double rate = rho > 0 ? (double)(z - P.n_below) / ((double)rho * 1.0) : 0.0;
      T.rate[(size_t)z * P.nRho + rho] = rate;
      for (int d = 1; d <= maxK; d++) {
        const double vp = round((double)z + (double)d * rate), vm = round((double)z - (double)d * rate);
        short2 e;
        e.x = (vp >= 0 && vp < P.nZ) ? (short)vp : (short)-1;
        e.y = (vm >= 0 && vm < P.nZ) ? (short)vm : (short)-1;
        T.dz[((size_t)z * P.nRho + rho) * maxK + (d - 1)] = e;
      }
    }
  // local_map_cartesian::init_map, src/map_local.cpp:56-62
  P.d_sub = cfg->subbox_d_xyz;
  P.d_sub_half = P.d_sub * 0.5;
  P.n = cfg->subbox_n;
  P.d_glb = P.d_sub * P.n;
  P.cells = P.n * P.n * P.n;
  P.inv_d_sub = 1.0 / P.d_sub;
  P.inv_d_glb = 1.0 / P.d_glb;
  P.inv_dRho = 1.0 / P.dRho;
  P.inv_dPhi = 1.0 / P.dPhi;
  P.inv_dZ = 1.0 / P.dZ;
  P.cell_stride = (P.cells + 15) & ~15;
  P.lo_min = cfg->log_odds_min;
  P.lo_max = cfg->log_odds_max;
  P.lo_miss = cfg->log_odds_miss;
  P.lo_sh = cfg->log_odds_occupied_sh;
  P.explore = cfg->use_exploration_frontiers != 0;
  P.front_words = (P.cells + 31) / 32;
  {
    const double bd[6] = {-30, 30, -30, 30, 0, 5};  // global_bd, hard-coded at src/map_local.cpp:124
    for (int i = 0; i < 6; i++) P.bd[i] = bd[i];
  }
  P.cx = cfg->cam_cx;
  P.cy = cfg->cam_cy;
  P.fx = cfg->cam_fx;
  P.fy = cfg->cam_fy;
  P.inv_factor = 1.0 / 1000.0;  // src/mlmap.h:85-86
  P.inv_fx = 1.0 / (double)cfg->cam_fx;
  P.inv_fy = 1.0 / (double)cfg->cam_fy;
  P.fast_inv_dRho = (float)(1.0 / P.dRho);
  P.fast_inv_dZ = (float)(1.0 / P.dZ);
  P.fast_deg2cell = (float)((M_PI / 180) / P.dPhi);
  // glibc dispatches __logf to its FMA build when FMA and AVX2 are usable (ifunc-fma.h)
  P.log10f_fma = (__builtin_cpu_supports("fma") && __builtin_cpu_supports("avx2")) ? 1 : 0;
  P.lvg_margin = P.n + 1;
  {
    double xy, z;  // below 2^31 cells (validate_config)
    lvg_dims(*cfg, &xy, &z);
    P.lvg_dim_xy = (int)xy;
    P.lvg_dim_z = (int)z;
  }
  make_div_magic((uint32_t)P.lvg_dim_xy, &P.dxy_mul, &P.dxy_shift);
  make_div_magic((uint32_t)P.lvg_dim_xy * (uint32_t)P.lvg_dim_xy, &P.dxy2_mul, &P.dxy2_shift);
  make_div_magic((uint32_t)P.n, &P.n_mul, &P.n_shift);
  P.lsg_dim_xy = P.lvg_dim_xy / P.n + 3;
  P.lsg_dim_z = P.lvg_dim_z / P.n + 3;
  const long long n_cells = (long long)P.nZ * P.nPhi * P.nRho;
  const long long lvg_cells = (long long)P.lvg_dim_xy * P.lvg_dim_xy * P.lvg_dim_z;
  const long long lsg_cells = (long long)P.lsg_dim_xy * P.lsg_dim_xy * P.lsg_dim_z;
  P.max_points = cfg->max_points;
  P.contrib_per_point = 1 + 2 * maxK;
  P.max_hits = (int)std::min<long long>(n_cells, (long long)P.max_points * P.contrib_per_point);
  P.max_touched = (int)std::min<long long>(2 * lvg_cells, 2 * n_cells);
  P.pool_blocks = cfg->pool_submaps;
  uint32_t ht_cap = 1;
  while (ht_cap < 2u * (uint32_t)P.pool_blocks) ht_cap <<= 1;
  P.ht_mask = ht_cap - 1;

  // column kernel shared memory: two column bitmaps + the largest power-of-two sort buffer that fits
  int max_optin = 0;
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  const size_t bm_bytes = col_smem_prefix_bytes(P.col_words, P.nRho, P.nCol);
  long long avail = (long long)max_optin - 1024 - (long long)bm_bytes;
  if (avail < 32 * 1024) {
    delete h;
    g_last_error = "awareness column (n_Z*n_Rho bits) does not fit shared memory";
    return MLM_ERR_INVALID_CONFIG;
  }
  // two key buffers (radix ping-pong) of sort_cap_smem 64-bit keys each
  int cap = (int)(avail / 16) & ~127;
  P.sort_cap_smem = cap;
  P.map_cap = kMapCap;
  if (sort_cap_env) P.sort_cap_smem = std::max(128, std::min(cap, atoi(sort_cap_env)) & ~127);
  if (map_cap_env) P.map_cap = std::max(1, std::min(kMapCap, atoi(map_cap_env)));
  h->col_smem_bytes = (int)(bm_bytes + (size_t)cap * 16);
  h->col_grid = std::max(1, std::min(P.nCol, h->sm_count));

#define TRY(x)            \
  do {                    \
    rc = (x);             \
    if (rc != MLM_OK) {   \
      mlm_destroy(h);     \
      return rc;          \
    }                     \
  } while (0)
#define CUDA_TRY_H(expr)                                                   \
  do {                                                                     \
    cudaError_t _e = (expr);                                               \
    if (_e != cudaSuccess) {                                               \
      g_last_error = std::string(#expr) + ": " + cudaGetErrorString(_e);   \
      mlm_destroy(h);                                                      \
      return MLM_ERR_CUDA;                                                 \
    }                                                                      \
  } while (0)

  CUDA_TRY_H(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CUDA_TRY_H(cudaEventCreate(&h->ev0));
  CUDA_TRY_H(cudaEventCreate(&h->ev1));
  CUDA_TRY_H(cudaMallocHost((void **)&h->h_fp, sizeof(FrameParams)));
  CUDA_TRY_H(cudaHostAlloc((void **)&h->h_fc, sizeof(FrameCounters), cudaHostAllocMapped));
  memset(h->h_fc, 0, sizeof(FrameCounters));
  // cudaFuncAttributeMaxDynamicSharedMemorySize is a property of the FUNCTION, shared by every handle of the process: it
  // is set to one configuration-independent ceiling, so that a later handle with a smaller column never lowers the limit
  // under a live handle with a larger one (two configurations in one process, e.g. a depth map next to a LiDAR map)
  const int smem_ceiling = max_optin - 1024;
  CUDA_TRY_H(cudaFuncSetAttribute(k_column, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_ceiling));
  for (const FrameKernel *table : {kProjectKernels, kFrameKernels, kFrameExploreKernels})
    for (int mode = 0; mode < 3; mode++)
      CUDA_TRY_H(cudaFuncSetAttribute(table[mode], cudaFuncAttributeMaxDynamicSharedMemorySize, smem_ceiling));
  if ((long long)project_smem_bytes(P.nCol, kProjThreads) > (long long)max_optin - 1024) {
    mlm_destroy(h);
    g_last_error = "n_Phi too large for the projection's shared-memory histogram";
    return MLM_ERR_INVALID_CONFIG;
  }
  // one cooperative launch per frame when every phase fits the resident CTA (exploration mode: k_frame_explore, with
  // its ordered passes behind further device-wide barriers)
  {
    int per_sm = 0, coop = 0;
    const FrameKernel k_frame_depth = (P.explore ? kFrameExploreKernels : kFrameKernels)[1];
    CUDA_TRY_H(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_frame_depth, kColThreads, h->col_smem_bytes));
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
    h->frame_grid = h->sm_count * std::min(per_sm, 1);
    h->use_fused = coop && per_sm >= 1 && project_smem_bytes(P.nCol, kColThreads) <= (size_t)h->col_smem_bytes && !no_fused;
  }

  DeviceBuffers &D = h->D;
  memset(&D, 0, sizeof(D));
  float *d_odds;
  int *d_k;
  double2 *d_cxy;
  double *d_cz;
  TRY(dev_alloc(h, &d_odds, T.odds.size()));
  TRY(dev_alloc(h, &d_k, T.k_reach.size()));
  TRY(dev_alloc(h, &d_cxy, T.centre_xy.size()));
  TRY(dev_alloc(h, &d_cz, T.centre_z.size()));
  CUDA_TRY_H(cudaMemcpy(d_odds, T.odds.data(), T.odds.size() * sizeof(float), cudaMemcpyHostToDevice));
  CUDA_TRY_H(cudaMemcpy(d_k, T.k_reach.data(), T.k_reach.size() * sizeof(int), cudaMemcpyHostToDevice));
  CUDA_TRY_H(cudaMemcpy(d_cxy, T.centre_xy.data(), T.centre_xy.size() * sizeof(double2), cudaMemcpyHostToDevice));
  CUDA_TRY_H(cudaMemcpy(d_cz, T.centre_z.data(), T.centre_z.size() * sizeof(double), cudaMemcpyHostToDevice));
  double *d_rate;
  short2 *d_dz;
  TRY(dev_alloc(h, &d_rate, T.rate.size()));
  TRY(dev_alloc(h, &d_dz, T.dz.size()));
  CUDA_TRY_H(cudaMemcpy(d_rate, T.rate.data(), T.rate.size() * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY_H(cudaMemcpy(d_dz, T.dz.data(), T.dz.size() * sizeof(short2), cudaMemcpyHostToDevice));
  P.rate_table = d_rate;
  P.dz_table = d_dz;
  P.odds_table = d_odds;
  P.k_reach = d_k;
  P.centre_xy = d_cxy;
  P.centre_z = d_cz;

  TRY(dev_alloc(h, &D.fuse_ticket, 1));
  CUDA_TRY_H(cudaMemset(D.fuse_ticket, 0, sizeof(int)));
  CUDA_TRY_H(cudaHostGetDevicePointer((void **)&D.host_fc, h->h_fc, 0));
  TRY(dev_alloc(h, &D.fc[0], 2));
  D.fc[1] = D.fc[0] + 1;
  TRY(dev_alloc(h, &D.col_ticket, 1));
  TRY(dev_alloc(h, &D.col_queue, 1));
  TRY(dev_alloc(h, &D.grid_bar, 1));
  TRY(dev_alloc(h, &D.rec_lin, (size_t)P.max_points));
  TRY(dev_alloc(h, &D.rec_col, (size_t)P.max_points));
  TRY(dev_alloc(h, &D.rec_dir, (size_t)(std::max((P.max_points + 1023) / 1024, 2 * h->sm_count + 2)) * P.nCol));
  TRY(dev_alloc(h, &D.phi_hist, (size_t)P.nCol));
  TRY(dev_alloc(h, &D.phi_bound, (size_t)P.nCol));
  TRY(dev_alloc(h, &D.col_scratch, (size_t)2 * P.max_points * P.contrib_per_point));
  TRY(dev_alloc(h, &D.hit_key, (size_t)P.max_hits));
  TRY(dev_alloc(h, &D.hit_p, (size_t)P.max_hits));
  TRY(dev_alloc(h, &D.hit_t, (size_t)P.max_hits));
  TRY(dev_alloc(h, &D.hit_next, (size_t)P.max_hits));
  TRY(dev_alloc(h, &D.hit_bucket, (size_t)P.max_hits));
  TRY(dev_alloc(h, &D.miss_bitmap, (size_t)P.nPhi * P.col_words));
  h->act_cap = chain_cover((uint32_t)P.max_hits);
  if (h->act_cap == 0) {
    g_last_error = "max hit cells exceed the bucket chain table";
    mlm_destroy(h);
    return MLM_ERR_INVALID_CONFIG;
  }
  TRY(dev_alloc(h, &D.act[0], (size_t)h->act_cap));
  TRY(dev_alloc(h, &D.act[1], (size_t)h->act_cap));
  TRY(dev_alloc(h, &D.lvg, (size_t)lvg_cells));
  TRY(dev_alloc(h, &D.touched, (size_t)P.max_touched));
  TRY(dev_alloc(h, &D.lsg_flag, (size_t)lsg_cells));
  TRY(dev_alloc(h, &D.lsg_block, (size_t)lsg_cells));
  TRY(dev_alloc(h, &D.touched_sub, (size_t)lsg_cells));
  TRY(dev_alloc(h, &D.ht_key, (size_t)ht_cap));
  TRY(dev_alloc(h, &D.ht_val, (size_t)ht_cap));
  TRY(dev_alloc(h, &D.free_stack, (size_t)P.pool_blocks));
  TRY(dev_alloc(h, &D.free_top, 1));
  TRY(dev_alloc(h, &D.pool_lo, (size_t)P.pool_blocks * P.cell_stride));
  TRY(dev_alloc(h, &D.pool_occ, (size_t)P.pool_blocks * P.cell_stride));
  TRY(dev_alloc(h, &D.pool_inf, (size_t)P.pool_blocks * P.cell_stride));
  if (P.explore) {
    if ((long long)P.max_points * P.nRho >= (1ll << 31)) {
      g_last_error = "exploration mode needs max_points * n_Rho < 2^31 (miss-cell insert stamps)";
      mlm_destroy(h);
      return MLM_ERR_INVALID_CONFIG;
    }
    TRY(dev_alloc(h, &D.pool_front, (size_t)P.pool_blocks * P.front_words));
    TRY(dev_alloc(h, &D.col_occ, (size_t)ht_cap));
    TRY(dev_alloc(h, &D.col_inf, (size_t)ht_cap));
    TRY(dev_alloc(h, &D.col_lo, (size_t)ht_cap));
    TRY(dev_alloc(h, &D.end_t, (size_t)n_cells));
    TRY(dev_alloc(h, &D.miss_stamp, (size_t)n_cells));
    CUDA_TRY_H(cudaMemset(D.miss_stamp, 0xff, (size_t)n_cells * 4));  // (split layouts rely on the sensor row being reset between frames)
    h->act_miss_cap = chain_cover((uint32_t)n_cells);
    if (h->act_miss_cap == 0) {
      g_last_error = "awareness cell count exceeds the bucket chain table";
      mlm_destroy(h);
      return MLM_ERR_INVALID_CONFIG;
    }
    TRY(dev_alloc(h, &D.act_miss[0], (size_t)h->act_miss_cap));
    TRY(dev_alloc(h, &D.act_miss[1], (size_t)h->act_miss_cap));
    TRY(dev_alloc(h, &D.miss_idx, (size_t)n_cells));
    TRY(dev_alloc(h, &D.miss_lv, (size_t)n_cells));
    TRY(dev_alloc(h, &D.miss_t, (size_t)n_cells));
    TRY(dev_alloc(h, &D.miss_bucket, (size_t)n_cells));
    TRY(dev_alloc(h, &D.miss_choice, (size_t)n_cells));
    TRY(dev_alloc(h, &D.lvg_tkey, (size_t)lvg_cells));
    TRY(dev_alloc(h, &D.obs_flag, (size_t)lsg_cells));
    TRY(dev_alloc(h, &D.obs_list, (size_t)lsg_cells));
    CUDA_TRY_H(cudaMemset(D.pool_front, 0, (size_t)P.pool_blocks * P.front_words * 4));
    CUDA_TRY_H(cudaMemset(D.act_miss[0], 0xff, (size_t)h->act_miss_cap * 4));
    CUDA_TRY_H(cudaMemset(D.act_miss[1], 0xff, (size_t)h->act_miss_cap * 4));
    CUDA_TRY_H(cudaMemset(D.lvg_tkey, 0, (size_t)lvg_cells * 8));
    CUDA_TRY_H(cudaMemset(D.obs_flag, 0, (size_t)lsg_cells * 4));
  }
  TRY(dev_alloc(h, &D.cum, 4));
  TRY(dev_alloc(h, &D.debug_cycles, (size_t)(P.nCol + 256) * 16));
  CUDA_TRY_H(cudaMemset(D.debug_cycles, 0, (size_t)(P.nCol + 256) * 16 * sizeof(long long)));
  h->sort_cap = P.explore ? (int)n_cells : P.max_hits;
  const size_t sort_pad = (size_t)next_pow2(h->sort_cap);
  TRY(dev_alloc(h, &h->d_sort_a, sort_pad));
  TRY(dev_alloc(h, &h->d_sort_b, sort_pad));
  TRY(dev_alloc(h, &h->d_seq_a, (size_t)h->sort_cap));
  TRY(dev_alloc(h, &h->d_seq_b, (size_t)h->sort_cap));

  // initial state
  {
    std::vector<int2> init((size_t)lvg_cells, make_int2(kLvgEmpty, 0));
    CUDA_TRY_H(cudaMemcpy(D.lvg, init.data(), init.size() * sizeof(int2), cudaMemcpyHostToDevice));
  }
  CUDA_TRY_H(cudaMemset(D.lsg_flag, 0, (size_t)lsg_cells * 4));
  CUDA_TRY_H(cudaMemset(D.lsg_block, 0xff, (size_t)lsg_cells * 4));
  CUDA_TRY_H(cudaMemset(D.ht_key, 0xff, (size_t)ht_cap * 8));
  CUDA_TRY_H(cudaMemset(D.ht_val, 0xff, (size_t)ht_cap * 4));
  CUDA_TRY_H(cudaMemset(D.cum, 0, 4 * sizeof(int64_t)));
  CUDA_TRY_H(cudaMemset(D.col_ticket, 0, sizeof(int)));
  CUDA_TRY_H(cudaMemset(D.col_queue, 0, sizeof(int)));
  CUDA_TRY_H(cudaMemset(D.grid_bar, 0, sizeof(int)));
  CUDA_TRY_H(cudaMemset(D.fc[0], 0, 2 * sizeof(FrameCounters)));
  CUDA_TRY_H(cudaMemset(D.act[0], 0xff, (size_t)h->act_cap * 4));
  CUDA_TRY_H(cudaMemset(D.act[1], 0xff, (size_t)h->act_cap * 4));
  CUDA_TRY_H(cudaMemset(D.phi_hist, 0, (size_t)P.nCol * 4));
  CUDA_TRY_H(cudaMemset(D.phi_bound, 0, (size_t)P.nCol * 4));
  // every block on the free stack is in the initial state of allocate_ram: 'u', 'u', 0.f
  CUDA_TRY_H(cudaMemset(D.pool_lo, 0, (size_t)P.pool_blocks * P.cell_stride * 4));
  CUDA_TRY_H(cudaMemset(D.pool_occ, 'u', (size_t)P.pool_blocks * P.cell_stride));
  CUDA_TRY_H(cudaMemset(D.pool_inf, 'u', (size_t)P.pool_blocks * P.cell_stride));
  CUDA_TRY_H(cudaMemset(D.miss_bitmap, 0, (size_t)P.nPhi * P.col_words * 4));
  {
    std::vector<int> stack(P.pool_blocks);
    for (int i = 0; i < P.pool_blocks; i++) stack[i] = P.pool_blocks - 1 - i;  // block 0 popped first
    CUDA_TRY_H(cudaMemcpy(D.free_stack, stack.data(), stack.size() * sizeof(int), cudaMemcpyHostToDevice));
    int top = P.pool_blocks;
    CUDA_TRY_H(cudaMemcpy(D.free_top, &top, sizeof(int), cudaMemcpyHostToDevice));
  }
  CUDA_TRY_H(cudaDeviceSynchronize());
#undef TRY
#undef CUDA_TRY_H
  *out = h;
  return MLM_OK;
}

static void esdf_free(mlm_handle h);
static void frontier_free(mlm_handle h);
static void view_free(mlm_handle h);
static void reach_free(mlm_handle h);
static void reach_matrix_free(mlm_handle h);

int mlm_destroy(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (int i = 0; i < 3; i++) {
    if (h->graph_exec[i]) cudaGraphExecDestroy(h->graph_exec[i]);
    if (h->graph[i]) cudaGraphDestroy(h->graph[i]);
    if (h->fgraph_exec[i]) cudaGraphExecDestroy(h->fgraph_exec[i]);
    if (h->fgraph[i]) cudaGraphDestroy(h->fgraph[i]);
  }
  mlm_shard_close(h);
  if (h->h_shard_state) cudaFreeHost(h->h_shard_state);
  for (void *p : h->allocs) cudaFree(p);
  esdf_free(h);
  frontier_free(h);
  view_free(h);
  reach_free(h);
  reach_matrix_free(h);
  if (h->d_input) cudaFree(h->d_input);
  if (h->h_stage) cudaFreeHost(h->h_stage);
  if (h->l2_buf) cudaFree(h->l2_buf);
  if (h->h_fp) cudaFreeHost(h->h_fp);
  if (h->h_fc) cudaFreeHost(h->h_fc);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (int i = 0; i <= MLM_NUM_FRAME_KERNELS; i++)
    if (h->kev[i]) cudaEventDestroy(h->kev[i]);
  for (int i = 0; i <= MLM_NUM_SHARD_KERNELS; i++)
    if (h->sev[i]) cudaEventDestroy(h->sev[i]);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return MLM_OK;
}

int mlm_integrate_depth_u16(mlm_handle h, const uint16_t *img, int rows, int cols, size_t stride_bytes,
                            const double T_wb[7], mlm_frame_stats *stats) {
  if (!h || !img || !T_wb || rows <= 0 || cols <= 0 || stride_bytes < (size_t)cols * 2) return MLM_ERR_INVALID_ARG;
  if ((long long)rows * cols > h->P.max_points) {
    g_last_error = "image larger than cfg.max_points";
    return MLM_ERR_CAPACITY;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  if (h->cfg.sample_cnt > 0) {
    // mlmap::project_depth as written (src/mlmap.cpp:321-346): up to sample_cnt valid pixels out of at most
    // 2*sample_cnt rand() draws; only the sampled (pixel, depth) pairs travel to the device
    const size_t cnt_max = (size_t)h->cfg.sample_cnt;
    int rc2 = ensure_input(h, cnt_max * sizeof(uint2), cnt_max * sizeof(uint2));
    if (rc2 != MLM_OK) return rc2;
    uint2 *pairs = reinterpret_cast<uint2 *>(h->h_stage);
    size_t n_pts = 0;
    int cnt = 0;
    const int max_iter = 2 * (int)cnt_max;
    while (n_pts < cnt_max && cnt < max_iter) {
      cnt++;
      const size_t v = (size_t)(h->rng.next() % rows);
      const size_t u = (size_t)(h->rng.next() % cols);
      const uint16_t raw = *reinterpret_cast<const uint16_t *>(reinterpret_cast<const char *>(img) + v * stride_bytes + u * 2);
      if (raw == 0) continue;
      pairs[n_pts++] = make_uint2((unsigned)(v * cols + u), raw);
    }
    if (n_pts) CUDA_TRY(cudaMemcpyAsync(h->d_input, pairs, n_pts * sizeof(uint2), cudaMemcpyHostToDevice, h->stream));
    return run_frame(h, 2, h->d_input, rows, cols, (int)n_pts, T_wb, stats);
  }
  const size_t bytes = (size_t)rows * cols * 2;
  int rc = ensure_input(h, bytes, (size_t)h->P.max_points * 2);
  if (rc != MLM_OK) return rc;
  // Page-locked caller memory (mlm_host_alloc / cudaHostRegister) with dense rows is copied
  // straight from the caller's buffer; anything else is packed into the pinned staging buffer first.
  cudaPointerAttributes attr;
  const bool pinned = stride_bytes == (size_t)cols * 2 && cudaPointerGetAttributes(&attr, img) == cudaSuccess &&
                      attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  const void *src = img;
  if (!pinned) {
    if (stride_bytes == (size_t)cols * 2) {
      memcpy(h->h_stage, img, bytes);
    } else {
      for (int v = 0; v < rows; v++)
        memcpy((char *)h->h_stage + (size_t)v * cols * 2, (const char *)img + (size_t)v * stride_bytes, (size_t)cols * 2);
    }
    src = h->h_stage;
  }
  // Overlapping the transfer with the projection was measured twice on B200 and lost both times against this one DMA
  // (102.7 us per frame end to end): a second DMA for the lower half of the rows with a ready word the tiles wait for
  // (+6 us: the extra copies cost more than the overlap returns), and reading that half in place over PCIe (+2 to +7 us).
  CUDA_TRY(cudaMemcpyAsync(h->d_input, src, bytes, cudaMemcpyHostToDevice, h->stream));
  return run_frame(h, 1, h->d_input, rows, cols, 0, T_wb, stats);
}

int mlm_integrate_depth_u16_device(mlm_handle h, const uint16_t *d_img, int rows, int cols, const double T_wb[7],
                                   mlm_frame_stats *stats) {
  if (!h || !d_img || !T_wb || rows <= 0 || cols <= 0) return MLM_ERR_INVALID_ARG;
  if ((long long)rows * cols > h->P.max_points) {
    g_last_error = "image larger than cfg.max_points";
    return MLM_ERR_CAPACITY;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  if (h->cfg.sample_cnt > 0) {
    // mlmap::project_depth (src/mlmap.cpp:321-346) on a device image: the rand() draws of all 2*sample_cnt possible tries
    // are made up front on a COPY of the stream (two per try whatever the pixel holds); a kernel looks the pixels up,
    // keeps the tries the reference's loop would have executed (it stops after sample_cnt valid pixels) and reports how
    // many that were, and the handle's stream then advances by exactly that many tries
    const int cnt_max = h->cfg.sample_cnt, max_iter = 2 * cnt_max;
    cudaStream_t s = h->stream;
    if (!h->d_sample_tries) {
      CUDA_TRY(cudaMalloc((void **)&h->d_sample_tries, (size_t)max_iter * sizeof(uint2) * 2));
      h->allocs.push_back(h->d_sample_tries);
      CUDA_TRY(cudaMalloc((void **)&h->d_sample_info, 2 * sizeof(int)));
      h->allocs.push_back(h->d_sample_info);
    }
    int rc2 = ensure_input(h, (size_t)max_iter * sizeof(uint2), (size_t)max_iter * sizeof(uint2));
    if (rc2 != MLM_OK) return rc2;
    GlibcRand ahead = h->rng;
    uint2 *tries = reinterpret_cast<uint2 *>(h->h_stage);
    for (int t = 0; t < max_iter; t++) {
      const unsigned v = (unsigned)(ahead.next() % rows);
      const unsigned u = (unsigned)(ahead.next() % cols);
      tries[t] = make_uint2(v * (unsigned)cols + u, 0u);
    }
    CUDA_TRY(cudaMemcpyAsync(h->d_sample_tries, tries, (size_t)max_iter * sizeof(uint2), cudaMemcpyHostToDevice, s));
    uint2 *d_pairs = h->d_sample_tries + max_iter;
    k_sample_gather<<<1, 1024, 0, s>>>(d_img, h->d_sample_tries, max_iter, cnt_max, d_pairs, h->d_sample_info);
    h->launches++;
    int info[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(info, h->d_sample_info, sizeof(info), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    for (int t = 0; t < info[1]; t++) {  // the tries the reference's loop executes: two draws each
      h->rng.next();
      h->rng.next();
    }
    return run_frame(h, 2, d_pairs, rows, cols, info[0], T_wb, stats);
  }
  return run_frame(h, 1, d_img, rows, cols, 0, T_wb, stats);
}

int mlm_integrate_points_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7], mlm_frame_stats *stats) {
  if (!h || (!xyz && n > 0) || !T_wb || n < 0) return MLM_ERR_INVALID_ARG;
  if (n > h->P.max_points) {
    g_last_error = "more points than cfg.max_points";
    return MLM_ERR_CAPACITY;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t bytes = (size_t)std::max(n, 1) * 24;
  int rc = ensure_input(h, bytes, (size_t)h->P.max_points * 24);
  if (rc != MLM_OK) return rc;
  if (n > 0) {
    // page-locked caller memory (mlm_host_alloc / cudaHostRegister) is copied straight from the caller's buffer
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, xyz) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const void *src = xyz;
    if (!pinned) {
      memcpy(h->h_stage, xyz, (size_t)n * 24);
      src = h->h_stage;
    }
    CUDA_TRY(cudaMemcpyAsync(h->d_input, src, (size_t)n * 24, cudaMemcpyHostToDevice, h->stream));
  }
  return run_frame(h, 0, h->d_input, 0, 0, n, T_wb, stats);
}

int mlm_integrate_points_f64_device(mlm_handle h, const double *d_xyz, int n, const double T_wb[7],
                                    mlm_frame_stats *stats) {
  if (!h || (!d_xyz && n > 0) || !T_wb || n < 0) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  return run_frame(h, 0, d_xyz, 0, 0, n, T_wb, stats);
}

// ---- the two layer entry points mlmap::update_map calls one after the other (src/mlmap.cpp:382-386) -----------------
int mlm_awareness_input_pc_pose_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7], mlm_frame_stats *stats) {
  if (!h) return MLM_ERR_INVALID_ARG;
  h->stage_call = 1;
  const int rc = mlm_integrate_points_f64(h, xyz, n, T_wb, stats);
  h->stage_call = 0;
  return rc;
}
int mlm_awareness_input_depth_u16(mlm_handle h, const uint16_t *img, int rows, int cols, size_t stride_bytes, const double T_wb[7],
                                  mlm_frame_stats *stats) {
  if (!h) return MLM_ERR_INVALID_ARG;
  h->stage_call = 1;
  const int rc = mlm_integrate_depth_u16(h, img, rows, cols, stride_bytes, T_wb, stats);
  h->stage_call = 0;
  return rc;
}
int mlm_local_input_pc_pose_direct(mlm_handle h, mlm_frame_stats *stats) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!h->staged) {
    g_last_error = "no awareness-layer update is staged (mlm_awareness_input_* comes first)";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  h->staged = false;
  return h->P.explore ? run_frame_explore_direct(h, h->staged_slow, h->staged_order_B, stats)
                      : run_frame_fuse_direct(h, h->staged_slow, h->staged_order_B, stats);
}

// ---- asynchronous frames: several maps of one process share a GPU (CFG-D: 8 agent maps) -------------------------------
int mlm_set_sm_budget(mlm_handle h, int n_sms) {
  if (!h || n_sms < 0) return MLM_ERR_INVALID_ARG;
  h->frame_sms = n_sms;
  return MLM_OK;
}
int mlm_frame_submit_depth_u16_device(mlm_handle h, const uint16_t *d_img, int rows, int cols, const double T_wb[7]) {
  if (!h || !d_img || !T_wb || rows <= 0 || cols <= 0) return MLM_ERR_INVALID_ARG;
  if (h->cfg.sample_cnt > 0 || h->P.explore) {
    g_last_error = "asynchronous frames: full-frame projection without the exploration mode only";
    return MLM_ERR_UNSUPPORTED;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  h->async_call = 1;
  const int rc = run_frame(h, 1, d_img, rows, cols, 0, T_wb, nullptr);
  h->async_call = 0;
  return rc;
}
int mlm_frame_submit_points_f64_device(mlm_handle h, const double *d_xyz, int n, const double T_wb[7]) {
  if (!h || (!d_xyz && n > 0) || !T_wb || n < 0) return MLM_ERR_INVALID_ARG;
  if (h->P.explore) {
    g_last_error = "asynchronous frames: not in the exploration mode";
    return MLM_ERR_UNSUPPORTED;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  h->async_call = 1;
  const int rc = run_frame(h, 0, d_xyz, 0, 0, n, T_wb, nullptr);
  h->async_call = 0;
  return rc;
}
int mlm_frame_finish(mlm_handle h, mlm_frame_stats *stats) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!h->frame_pending) {
    g_last_error = "no submitted frame";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  h->frame_pending = false;
  return run_frame_complete(h, stats);
}

// getOdd(const Vec3I &glb_id, size_t subbox_id), include/mlmap.h:128,227-235
static void odd_at_launch(mlm_handle h, const int32_t *d_glb3, const int32_t *d_sub, size_t n, float *d_out) {
  k_get_odd_at<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_glb3, d_sub, n, d_out);
  h->launches++;
}
int mlm_get_odd_at_device(mlm_handle h, const int32_t *d_glb3, const int32_t *d_sub, size_t n, float *d_out) {
  if (!h || ((!d_glb3 || !d_sub || !d_out) && n)) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  odd_at_launch(h, d_glb3, d_sub, n, d_out);
  return MLM_OK;
}
int mlm_get_odd_at(mlm_handle h, const int32_t *glb3, const int32_t *sub, size_t n, float *out) {
  if (!h || ((!glb3 || !sub || !out) && n)) return MLM_ERR_INVALID_ARG;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<int32_t> d_in(s);  // glb3, sub
    StreamTemp<float> d_o(s);
    CUDA_TRY(d_in.alloc(n * 4));
    CUDA_TRY(d_o.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_in, glb3, n * 12, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_in + 3 * n, sub, n * 4, cudaMemcpyHostToDevice, s));
    odd_at_launch(h, d_in, d_in + 3 * n, n, d_o);
    CUDA_TRY(cudaMemcpyAsync(out, d_o, n * 4, cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

int mlm_set_free_in_bound(mlm_handle h, const double box_min[3], const double box_max[3]) {
  if (!h || !box_min || !box_max) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  // coordinates by repeated "+=" in double, like the reference loops (src/mlmap.cpp:392-396)
  std::vector<double> ax[3];
  for (int a = 0; a < 3; a++) {
    for (double v = box_min[a]; v <= box_max[a]; v += h->P.d_sub) {
      ax[a].push_back(v);
      if (ax[a].size() > (size_t)1 << 24) return MLM_ERR_INVALID_ARG;
    }
    if (ax[a].empty()) return MLM_OK;
  }
  size_t total = ax[0].size() * ax[1].size() * ax[2].size();
  size_t ncoord = ax[0].size() + ax[1].size() + ax[2].size();
  std::vector<double> flat;
  flat.reserve(ncoord);
  for (int a = 0; a < 3; a++) flat.insert(flat.end(), ax[a].begin(), ax[a].end());
  {
    StreamTemp<double> d_c(h->stream);
    CUDA_TRY(d_c.alloc(ncoord));
    CUDA_TRY(cudaMemcpyAsync(d_c, flat.data(), ncoord * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    k_set_free<<<grid_for(total, 256), 256, 0, h->stream>>>(h->P, h->D, d_c, (int)ax[0].size(), d_c + ax[0].size(),
                                                             (int)ax[1].size(), d_c + ax[0].size() + ax[1].size(),
                                                             (int)ax[2].size());
    h->launches++;
  }
  CUDA_TRY(cudaStreamSynchronize(h->stream));  // flat must outlive the copy
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

int mlm_inflate_map(mlm_handle h, const double ct_pos[3]) {
  if (!h || !ct_pos) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  const MapParams &P = h->P;
  if (h->cfg.inflate_n < 0 || h->cfg.inflate_global_n < 0 || h->cfg.inflate_global_n > 16) return MLM_ERR_INVALID_CONFIG;
  InflateArgs A;
  // local_map->get_global_idx(ct_pos, ct_glb, subbox_id): floor(p / d_glb) per axis (include/map_local.h:150)
  for (int a = 0; a < 3; a++) A.ct_g[a] = (int)floor(ct_pos[a] / P.d_glb);
  A.N = h->cfg.inflate_global_n;
  A.r = h->cfg.inflate_n;
  A.height = h->cfg.inflate_height;
  const int W = 2 * A.N + 1, nwin = W * W * W;
  cudaStream_t s = h->stream;
  int cnt[2] = {0, 0};
  {
    StreamTemp<int> d_win(s), d_cnt(s);
    CUDA_TRY(d_win.alloc(nwin));
    CUDA_TRY(d_cnt.alloc(2));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(int), s));
    k_inflate_reset<<<nwin, 256, 0, s>>>(P, h->D, A, d_win);
    k_inflate_sources<false><<<nwin, 256, 0, s>>>(P, h->D, A, d_win, d_cnt);
    k_inflate_sources<true><<<nwin, 256, 0, s>>>(P, h->D, A, d_win, d_cnt);
    h->launches += 3;
    CUDA_TRY(cudaMemcpyAsync(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  h->cum_ram_expand += cnt[0];  // allocate_ram from inflate_atpos also counts (include/map_local.h:223)
  h->n_submaps += cnt[0];
  if (cnt[1]) {
    g_last_error = "inflate_map: device raised error code " + std::to_string(cnt[1]);
    return map_device_error(cnt[1]);
  }
  return MLM_OK;
}

// point queries: one launch each, called on the caller's buffers by the _device variants and through host_query
static void occupancy_launch(mlm_handle h, const double *d_pos, size_t n, int32_t *d_out) {
  k_get_occupancy<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_pos, n, d_out);
  h->launches++;
}
static void occupancy_inflate_launch(mlm_handle h, const double *d_pos, size_t n, int32_t *d_out, float inflate) {
  k_get_occupancy_inflate<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_pos, n, inflate, d_out);
  h->launches++;
}
static void inflate_occupancy_launch(mlm_handle h, const double *d_pos, size_t n, int32_t *d_out) {
  k_get_inflate_occupancy<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_pos, n, d_out);
  h->launches++;
}
static void odd_launch(mlm_handle h, const double *d_pos, size_t n, float *d_out) {
  k_get_odd<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_pos, n, d_out);
  h->launches++;
}
static void odd_grad_launch(mlm_handle h, const double *d_pos, size_t n, double *d_out3n, size_t max_iter) {
  k_get_odd_grad<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_pos, n, (int)max_iter, d_out3n);
  h->launches++;
}
int mlm_get_occupancy(mlm_handle h, const double *pos, size_t n, int32_t *out) {
  return host_query(h, pos, n, out, 1, occupancy_launch);
}
int mlm_get_occupancy_inflate(mlm_handle h, const double *pos, size_t n, float inflate, int32_t *out) {
  return host_query(h, pos, n, out, 1, occupancy_inflate_launch, inflate);
}
int mlm_get_inflate_occupancy(mlm_handle h, const double *pos, size_t n, int32_t *out) {
  return host_query(h, pos, n, out, 1, inflate_occupancy_launch);
}
int mlm_get_odd(mlm_handle h, const double *pos, size_t n, float *out) {
  return host_query(h, pos, n, out, 1, odd_launch);
}
int mlm_get_odd_grad(mlm_handle h, const double *pos, size_t n, size_t max_iter, double *out3n) {
  return host_query(h, pos, n, out3n, 3, odd_grad_launch, max_iter);
}
int mlm_get_occupancy_device(mlm_handle h, const double *d_pos, size_t n, int32_t *d_out) {
  if (!h || (!d_pos && n) || (!d_out && n)) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  occupancy_launch(h, d_pos, n, d_out);
  return MLM_OK;
}
int mlm_get_odd_device(mlm_handle h, const double *d_pos, size_t n, float *d_out) {
  if (!h || (!d_pos && n) || (!d_out && n)) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  odd_launch(h, d_pos, n, d_out);
  return MLM_OK;
}
int mlm_get_odd_grad_device(mlm_handle h, const double *d_pos, size_t n, size_t max_iter, double *d_out3n) {
  if (!h || (!d_pos && n) || (!d_out3n && n)) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  odd_grad_launch(h, d_pos, n, d_out3n, max_iter);
  return MLM_OK;
}

// rays, the distance field and frontier clustering read the whole map
static int refuse_sharded(mlm_handle h, const char *fn) {
  if (h->shard_world <= 1) return MLM_OK;
  g_last_error = std::string(fn) + ": a rank of a sharded map holds only the subboxes it owns";
  return MLM_ERR_UNSUPPORTED;
}
// rule 1 of the ray spec along one axis of a box: cells floor(p / d_sub) of the IEEE quotient, |p / d_sub| < 2^30
static int box_axis_cells(mlm_handle h, double a, double b, const char *fn, int *lo, int *hi) {
  const double qa = a / h->P.d_sub, qb = b / h->P.d_sub;
  if (!(std::fabs(qa) < 1073741824.0) || !(std::fabs(qb) < 1073741824.0) || !(a <= b)) {
    g_last_error = std::string(fn) + ": a box corner is not finite, |p / d_sub| >= 2^30, or box_min > box_max";
    return MLM_ERR_INVALID_ARG;
  }
  *lo = (int)std::floor(qa);
  *hi = (int)std::floor(qb);
  return MLM_OK;
}

// ---- batched ray casting (ray_kernels.cuh) --------------------------------------------------------------------
size_t mlm_sizeof_ray_hit(void) { return sizeof(mlm_ray_hit); }
static_assert(sizeof(mlm_ray_hit) == sizeof(RayHit), "mlm_ray_hit / RayHit layouts differ");

static int cast_rays_check(mlm_handle h, const void *from, const void *to, size_t n, int flags, const void *out) {
  if (!h || ((!from || !to || !out) && n) || (flags != 0 && flags != MLM_RAY_INFLATED)) return MLM_ERR_INVALID_ARG;
  return refuse_sharded(h, "mlm_cast_rays");
}
static void cast_rays_launch(mlm_handle h, const double *d_from, const double *d_to, size_t n, int flags, mlm_ray_hit *d_out) {
  RayHit *o = reinterpret_cast<RayHit *>(d_out);
  if (flags & MLM_RAY_INFLATED) k_cast_rays<true><<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_from, d_to, n, o);
  else k_cast_rays<false><<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->D, d_from, d_to, n, o);
  h->launches++;
}
int mlm_cast_rays_device(mlm_handle h, const double *d_from, const double *d_to, size_t n, int flags, mlm_ray_hit *d_out) {
  const int rc = cast_rays_check(h, d_from, d_to, n, flags, d_out);
  if (rc != MLM_OK) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  cast_rays_launch(h, d_from, d_to, n, flags, d_out);
  return MLM_OK;
}
// the host variant stages both endpoint arrays and the records through the handle's stream (like host_query)
int mlm_cast_rays(mlm_handle h, const double *from, const double *to, size_t n, int flags, mlm_ray_hit *out) {
  const int rc = cast_rays_check(h, from, to, n, flags, out);
  if (rc != MLM_OK) return rc;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<double> d_ft(s);  // from, to
    StreamTemp<mlm_ray_hit> d_o(s);
    CUDA_TRY(d_ft.alloc(n * 6));
    CUDA_TRY(d_o.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_ft, from, n * 24, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_ft + 3 * n, to, n * 24, cudaMemcpyHostToDevice, s));
    cast_rays_launch(h, d_ft, d_ft + 3 * n, n, flags, d_o);
    CUDA_TRY(cudaMemcpyAsync(out, d_o, n * sizeof(mlm_ray_hit), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// ---- signed distance field (esdf_kernels.cuh) ------------------------------------------------------------------
// a field is there to query / export
static int esdf_ready(mlm_handle h, const char *fn) {
  const int rc = refuse_sharded(h, fn);
  if (rc != MLM_OK) return rc;
  if (!h->esdf_built) {
    g_last_error = std::string(fn) + ": no signed distance field has been built (mlm_esdf_build first)";
    return MLM_ERR_INVALID_ARG;
  }
  return MLM_OK;
}
// the grid buffers for c cells: blocking bytes, two int2 grids (the first ends as the values), two stacks
static ScratchList esdf_scratch(mlm_handle h, size_t c) {
  return {{(void **)&h->esdf_blk, c}, {(void **)&h->esdf_a, c * sizeof(int2)}, {(void **)&h->esdf_b, c * sizeof(int2)},
          {(void **)&h->esdf_stk, 2 * c * sizeof(int2)}};
}
static void esdf_free(mlm_handle h) {
  scratch_free(esdf_scratch(h, 0));
  h->esdf_cap = 0;
  h->esdf_built = false;
}

// rule 1 of the distance-field spec and its limits (the reachability field shares them): the box's cells, the subboxes
// meeting it and d_sub into G, the number of cells into `cells`
static int esdf_box(mlm_handle h, const double box_min[3], const double box_max[3], const char *fn, EsdfGrid &G,
                    long long &cells) {
  const int n = h->P.n;
  cells = 1;
  for (int k = 0; k < 3; k++) {
    int lo, hi;
    const int rc = box_axis_cells(h, box_min[k], box_max[k], fn, &lo, &hi);
    if (rc != MLM_OK) return rc;
    const long long nk = (long long)hi - lo + 1;
    if (nk > kEsdfMaxAxis) {
      g_last_error = std::string(fn) + ": more than 4096 cells along an axis";
      return MLM_ERR_CAPACITY;
    }
    cells *= nk;
    G.lo[k] = lo;
    G.dims[k] = (int)nk;
    G.glo[k] = host_floor_div(lo, n);
    G.gdims[k] = host_floor_div(hi, n) - G.glo[k] + 1;
  }
  if (cells > kEsdfMaxCells) {
    g_last_error = std::string(fn) + ": more than 2^28 cells in the box";
    return MLM_ERR_CAPACITY;
  }
  G.d = h->P.d_sub;
  return MLM_OK;
}

int mlm_esdf_build(mlm_handle h, const double box_min[3], const double box_max[3], double max_dist, int flags) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!box_min || !box_max || (flags != 0 && flags != MLM_ESDF_INFLATED) || !std::isfinite(max_dist) || !(max_dist > 0)) {
    g_last_error = "mlm_esdf_build: null box, flags other than 0 / MLM_ESDF_INFLATED, or max_dist not finite and > 0";
    return MLM_ERR_INVALID_ARG;
  }
  int rc = refuse_sharded(h, "mlm_esdf_build");
  if (rc != MLM_OK) return rc;
  EsdfGrid G = {};
  long long cells = 0;
  rc = esdf_box(h, box_min, box_max, "mlm_esdf_build", G, cells);
  if (rc != MLM_OK) return rc;
  G.max_dist = max_dist;
  CUDA_TRY(cudaSetDevice(h->device));
  if ((size_t)cells > h->esdf_cap) {
    esdf_free(h);
    rc = scratch_alloc(esdf_scratch(h, (size_t)cells), "mlm_esdf_build: grid buffers");
    if (rc != MLM_OK) return rc;
    h->esdf_cap = (size_t)cells;
  }
  cudaStream_t s = h->stream;
  const int subs = G.gdims[0] * G.gdims[1] * G.gdims[2];
  if (flags & MLM_ESDF_INFLATED) k_esdf_gather<true><<<subs, 256, 0, s>>>(h->P, h->D, G, h->esdf_blk);
  else k_esdf_gather<false><<<subs, 256, 0, s>>>(h->P, h->D, G, h->esdf_blk);
  k_esdf_x<<<G.dims[1] * G.dims[2], 256, 0, s>>>(G, h->esdf_blk, h->esdf_a);
  const int gx = (G.dims[0] + kEsdfLineThreads - 1) / kEsdfLineThreads;
  k_esdf_y<<<dim3(gx, G.dims[2]), kEsdfLineThreads, 0, s>>>(G, h->esdf_a, h->esdf_b, h->esdf_stk);
  k_esdf_z<<<dim3(gx, G.dims[1]), kEsdfLineThreads, 0, s>>>(G, h->esdf_b, reinterpret_cast<double *>(h->esdf_a),
                                                            h->esdf_stk);
  h->launches += 4;
  CUDA_TRY(cudaGetLastError());
  h->esdf_grid = G;
  h->esdf_built = true;
  return MLM_OK;
}

static void esdf_distance_launch(mlm_handle h, const double *d_pos, size_t n, double *d_dist, double *d_grad3n) {
  k_esdf_query<<<grid_for(n, 256), 256, 0, h->stream>>>(h->esdf_grid, reinterpret_cast<const double *>(h->esdf_a),
                                                        d_pos, n, d_dist, d_grad3n);
  h->launches++;
}
int mlm_esdf_distance_device(mlm_handle h, const double *d_pos, size_t n, double *d_dist, double *d_grad3n) {
  if (!h || ((!d_pos || !d_dist) && n)) return MLM_ERR_INVALID_ARG;
  const int rc = esdf_ready(h, "mlm_esdf_distance");
  if (rc != MLM_OK) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  esdf_distance_launch(h, d_pos, n, d_dist, d_grad3n);
  return MLM_OK;
}
// the host variant stages the points, distances and gradients through the handle's stream (like mlm_cast_rays)
int mlm_esdf_distance(mlm_handle h, const double *pos, size_t n, double *dist, double *grad3n) {
  if (!h || ((!pos || !dist) && n)) return MLM_ERR_INVALID_ARG;
  const int rc = esdf_ready(h, "mlm_esdf_distance");
  if (rc != MLM_OK) return rc;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<double> d_buf(s);  // points, distances, gradients
    CUDA_TRY(d_buf.alloc(n * (grad3n ? 7 : 4)));
    double *d_pos = d_buf, *d_dist = d_pos + 3 * n, *d_grad = grad3n ? d_pos + 4 * n : nullptr;
    CUDA_TRY(cudaMemcpyAsync(d_pos, pos, n * 24, cudaMemcpyHostToDevice, s));
    esdf_distance_launch(h, d_pos, n, d_dist, d_grad);
    CUDA_TRY(cudaMemcpyAsync(dist, d_dist, n * 8, cudaMemcpyDeviceToHost, s));
    if (grad3n) CUDA_TRY(cudaMemcpyAsync(grad3n, d_grad, n * 24, cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// lo3 / dims3 always; the grid when out has room for it (out == NULL with cap 0 asks for the size only)
static int esdf_export_check(mlm_handle h, const float *out, size_t cap, int32_t lo3[3], int32_t dims3[3], size_t &cells) {
  if (!h || !lo3 || !dims3) return MLM_ERR_INVALID_ARG;
  const int rc = esdf_ready(h, "mlm_esdf_export");
  if (rc != MLM_OK) return rc;
  const EsdfGrid &G = h->esdf_grid;
  for (int k = 0; k < 3; k++) {
    lo3[k] = G.lo[k];
    dims3[k] = G.dims[k];
  }
  cells = (size_t)G.dims[0] * G.dims[1] * G.dims[2];
  if (!out && cap == 0) return MLM_OK;
  if (!out) return MLM_ERR_INVALID_ARG;
  if (cap < cells) {
    g_last_error = "mlm_esdf_export: cap is smaller than N_x * N_y * N_z";
    return MLM_ERR_CAPACITY;
  }
  return MLM_OK;
}
static void esdf_export_launch(mlm_handle h, size_t cells, float *d_out) {
  k_esdf_export<<<grid_for(cells, 256), 256, 0, h->stream>>>(reinterpret_cast<const double *>(h->esdf_a), cells, d_out);
  h->launches++;
}
int mlm_esdf_export_device(mlm_handle h, float *d_out, size_t cap, int32_t lo3[3], int32_t dims3[3]) {
  size_t cells = 0;
  const int rc = esdf_export_check(h, d_out, cap, lo3, dims3, cells);
  if (rc != MLM_OK || !d_out) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  esdf_export_launch(h, cells, d_out);
  return MLM_OK;
}
int mlm_esdf_export(mlm_handle h, float *out, size_t cap, int32_t lo3[3], int32_t dims3[3]) {
  size_t cells = 0;
  const int rc = esdf_export_check(h, out, cap, lo3, dims3, cells);
  if (rc != MLM_OK || !out) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  {
    StreamTemp<float> d_out(h->stream);
    CUDA_TRY(d_out.alloc(cells));
    esdf_export_launch(h, cells, d_out);
    CUDA_TRY(cudaMemcpyAsync(out, d_out, cells * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// ---- reachability field (reach_kernels.cuh) ------------------------------------------------------------------
// a field is there to query / export
static int reach_ready(mlm_handle h, const char *fn) {
  const int rc = refuse_sharded(h, fn);
  if (rc != MLM_OK) return rc;
  if (!h->reach_built) {
    g_last_error = std::string(fn) + ": no reachability field has been built (mlm_reach_build first)";
    return MLM_ERR_INVALID_ARG;
  }
  return MLM_OK;
}
// class bytes and costs per cell; per tile the queue marks and two worklists; the three queue counts and the barrier
static ScratchList reach_scratch(mlm_handle h, size_t cells, size_t tiles) {
  return {{(void **)&h->reach_cls, cells}, {(void **)&h->reach_cost, cells * sizeof(int)},
          {(void **)&h->reach_mark, tiles * sizeof(int)}, {(void **)&h->reach_list, 2 * tiles * sizeof(int)},
          {(void **)&h->reach_ctl, 4 * sizeof(int)}};
}
static void reach_free(mlm_handle h) {
  scratch_free(reach_scratch(h, 0, 0));
  h->reach_cap_cells = h->reach_cap_tiles = 0;
  h->reach_built = false;
}

// rules 1 and 5 for a build or a matrix: the box, its tiles, the budget and the flags into R, the box's cells into `cells`
static int reach_grid_of(mlm_handle h, const double box_min[3], const double box_max[3], double max_dist, int flags,
                         const char *fn, ReachGrid &R, long long &cells) {
  R = {};
  const int rc = esdf_box(h, box_min, box_max, fn, R.box, cells);
  if (rc != MLM_OK) return rc;
  const double K = std::floor((max_dist / h->P.d_sub) * 1000.0);  // rule 5's budget
  if (!(K <= (double)kReachMaxBudget)) {
    g_last_error = std::string(fn) + ": the cost budget floor(max_dist / d_sub * 1000) exceeds 2^30";
    return MLM_ERR_CAPACITY;
  }
  R.budget = (int)K;
  R.flags = flags;
  for (int k = 0; k < 3; k++) R.tiles[k] = (R.box.dims[k] + kReachTile - 1) / kReachTile;
  return MLM_OK;
}

int mlm_reach_build(mlm_handle h, const double box_min[3], const double box_max[3], const double *starts,
                    size_t n_starts, double max_dist, int flags, int32_t *n_sources) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!box_min || !box_max || !starts || n_starts == 0 || (flags & ~(MLM_REACH_INFLATED | MLM_REACH_UNKNOWN)) ||
      !std::isfinite(max_dist) || !(max_dist > 0)) {
    g_last_error = "mlm_reach_build: null box or starts, n_starts == 0, flags other than MLM_REACH_INFLATED | "
                   "MLM_REACH_UNKNOWN, or max_dist not finite and > 0";
    return MLM_ERR_INVALID_ARG;
  }
  int rc = refuse_sharded(h, "mlm_reach_build");
  if (rc != MLM_OK) return rc;
  ReachGrid R;
  long long cells = 0;
  rc = reach_grid_of(h, box_min, box_max, max_dist, flags, "mlm_reach_build", R, cells);
  if (rc != MLM_OK) return rc;
  const double d = h->P.d_sub;
  const size_t tiles = (size_t)R.tiles[0] * R.tiles[1] * R.tiles[2];
  // rule 3: the distinct source cells, as box-linear indices, found on the host
  std::vector<int> src;
  src.reserve(n_starts);
  for (size_t i = 0; i < n_starts; i++) {
    bool in = true;
    int c[3] = {0, 0, 0};
    for (int k = 0; k < 3 && in; k++) {
      const double q = starts[3 * i + k] / d;
      in = std::fabs(q) < 1073741824.0;
      if (in) c[k] = (int)std::floor(q) - R.box.lo[k];
      in = in && c[k] >= 0 && c[k] < R.box.dims[k];
    }
    if (in) src.push_back((c[2] * R.box.dims[1] + c[1]) * R.box.dims[0] + c[0]);
  }
  std::sort(src.begin(), src.end());
  src.erase(std::unique(src.begin(), src.end()), src.end());
  CUDA_TRY(cudaSetDevice(h->device));
  // from here on the buffers change: a build that fails part way leaves no field rather than a mix of two builds
  h->reach_built = false;
  if ((size_t)cells > h->reach_cap_cells || tiles > h->reach_cap_tiles) {
    const size_t cc = std::max((size_t)cells, h->reach_cap_cells), ct = std::max(tiles, h->reach_cap_tiles);
    reach_free(h);
    rc = scratch_alloc(reach_scratch(h, cc, ct), "mlm_reach_build: field buffers");
    if (rc != MLM_OK) return rc;
    h->reach_cap_cells = cc;
    h->reach_cap_tiles = ct;
  }
  cudaStream_t s = h->stream;
  const int subs = R.box.gdims[0] * R.box.gdims[1] * R.box.gdims[2];
  if (flags & MLM_REACH_INFLATED) k_esdf_gather<true><<<subs, 256, 0, s>>>(h->P, h->D, R.box, h->reach_cls);
  else k_esdf_gather<false><<<subs, 256, 0, s>>>(h->P, h->D, R.box, h->reach_cls);
  h->launches++;
  CUDA_TRY(cudaMemsetAsync(h->reach_cost, 0x7f, (size_t)cells * sizeof(int), s));  // kReachInf
  CUDA_TRY(cudaMemsetAsync(h->reach_mark, 0, tiles * sizeof(int), s));
  CUDA_TRY(cudaMemsetAsync(h->reach_ctl, 0, 4 * sizeof(int), s));
  ReachWork W = {h->reach_mark, h->reach_list, h->reach_list + tiles, h->reach_ctl,
                 reinterpret_cast<unsigned *>(h->reach_ctl + 3)};
  if (!src.empty()) {
    {
      StreamTemp<int> d_src(s);
      CUDA_TRY(d_src.alloc(src.size()));
      CUDA_TRY(cudaMemcpyAsync(d_src, src.data(), src.size() * sizeof(int), cudaMemcpyHostToDevice, s));
      k_reach_seed<<<grid_for(src.size(), 256), 256, 0, s>>>(R, d_src, (int)src.size(), h->reach_cls, h->reach_cost, W);
    }
    // as many CTAs as are resident at once, at most one per tile
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_reach_solve, kReachThreads, 0));
    const int G = (int)std::min<size_t>((size_t)h->sm_count * std::max(per_sm, 1), tiles);
    const uint8_t *cls = h->reach_cls;
    int *cost = h->reach_cost;
    void *args[] = {&R, &cls, &cost, &W};
    CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_reach_solve, dim3(G), dim3(kReachThreads), args, 0, s));
    h->launches += 2;
  }
  CUDA_TRY(cudaGetLastError());
  h->reach_grid = R;
  h->reach_built = true;
  if (n_sources) *n_sources = (int32_t)src.size();
  return MLM_OK;
}

static void reach_cost_launch(mlm_handle h, const double *d_pos, size_t n, double *d_out) {
  k_reach_cost<<<grid_for(n, 256), 256, 0, h->stream>>>(h->reach_grid, h->reach_cost, d_pos, n, d_out);
  h->launches++;
}
int mlm_reach_cost_device(mlm_handle h, const double *d_pos, size_t n, double *d_out) {
  if (!h || ((!d_pos || !d_out) && n)) return MLM_ERR_INVALID_ARG;
  const int rc = reach_ready(h, "mlm_reach_cost");
  if (rc != MLM_OK) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  reach_cost_launch(h, d_pos, n, d_out);
  return MLM_OK;
}
// the host variant stages the points and costs through the handle's stream (like mlm_esdf_distance)
int mlm_reach_cost(mlm_handle h, const double *pos, size_t n, double *out) {
  if (!h || ((!pos || !out) && n)) return MLM_ERR_INVALID_ARG;
  const int rc = reach_ready(h, "mlm_reach_cost");
  if (rc != MLM_OK) return rc;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<double> d_buf(s);  // points, costs
    CUDA_TRY(d_buf.alloc(n * 4));
    CUDA_TRY(cudaMemcpyAsync(d_buf, pos, n * 24, cudaMemcpyHostToDevice, s));
    reach_cost_launch(h, d_buf, n, d_buf + 3 * n);
    CUDA_TRY(cudaMemcpyAsync(out, d_buf + 3 * n, n * 8, cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

static int reach_paths_check(mlm_handle h, const void *goals, size_t n, size_t max_cells, const void *cells3,
                             const void *len) {
  if (!h || ((!goals || !len) && n) || (!cells3 && n && max_cells)) return MLM_ERR_INVALID_ARG;
  if (n && max_cells > ((size_t)1 << 62) / 12 / n) {
    g_last_error = "mlm_reach_paths: n * max_cells * 3 cells overflow";
    return MLM_ERR_INVALID_ARG;
  }
  return reach_ready(h, "mlm_reach_paths");
}
static void reach_paths_launch(mlm_handle h, const double *d_goals, size_t n, size_t max_cells, int32_t *d_cells3,
                               int32_t *d_len) {
  k_reach_paths<<<grid_for(n * 32, 256), 256, 0, h->stream>>>(h->reach_grid, h->reach_cls, h->reach_cost, d_goals, n,
                                                             max_cells, d_cells3, d_len);
  h->launches++;
}
int mlm_reach_paths_device(mlm_handle h, const double *d_goals, size_t n, size_t max_cells, int32_t *d_cells3,
                           int32_t *d_len) {
  const int rc = reach_paths_check(h, d_goals, n, max_cells, d_cells3, d_len);
  if (rc != MLM_OK) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  reach_paths_launch(h, d_goals, n, max_cells, d_cells3, d_len);
  return MLM_OK;
}
int mlm_reach_paths(mlm_handle h, const double *goals, size_t n, size_t max_cells, int32_t *cells3, int32_t *len) {
  const int rc = reach_paths_check(h, goals, n, max_cells, cells3, len);
  if (rc != MLM_OK) return rc;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<double> d_g(s);
    StreamTemp<int32_t> d_o(s);  // lengths, cells
    CUDA_TRY(d_g.alloc(n * 3));
    CUDA_TRY(d_o.alloc(n + n * max_cells * 3));
    CUDA_TRY(cudaMemcpyAsync(d_g, goals, n * 24, cudaMemcpyHostToDevice, s));
    reach_paths_launch(h, d_g, n, max_cells, d_o + n, d_o);
    CUDA_TRY(cudaMemcpyAsync(len, d_o, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (max_cells)
      CUDA_TRY(cudaMemcpyAsync(cells3, d_o + n, n * max_cells * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// lo3 / dims3 always; the field when out has room for it (out == NULL with cap 0 asks for the size only)
static int reach_export_check(mlm_handle h, const int32_t *out, size_t cap, int32_t lo3[3], int32_t dims3[3],
                              size_t &cells) {
  if (!h || !lo3 || !dims3) return MLM_ERR_INVALID_ARG;
  const int rc = reach_ready(h, "mlm_reach_export");
  if (rc != MLM_OK) return rc;
  const EsdfGrid &G = h->reach_grid.box;
  for (int k = 0; k < 3; k++) {
    lo3[k] = G.lo[k];
    dims3[k] = G.dims[k];
  }
  cells = (size_t)G.dims[0] * G.dims[1] * G.dims[2];
  if (!out && cap == 0) return MLM_OK;
  if (!out) return MLM_ERR_INVALID_ARG;
  if (cap < cells) {
    g_last_error = "mlm_reach_export: cap is smaller than N_x * N_y * N_z";
    return MLM_ERR_CAPACITY;
  }
  return MLM_OK;
}
static void reach_export_launch(mlm_handle h, size_t cells, int32_t *d_out) {
  k_reach_export<<<grid_for(cells, 256), 256, 0, h->stream>>>(h->reach_cost, cells, d_out);
  h->launches++;
}
int mlm_reach_export_device(mlm_handle h, int32_t *d_out, size_t cap, int32_t lo3[3], int32_t dims3[3]) {
  size_t cells = 0;
  const int rc = reach_export_check(h, d_out, cap, lo3, dims3, cells);
  if (rc != MLM_OK || !d_out) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  reach_export_launch(h, cells, d_out);
  return MLM_OK;
}
int mlm_reach_export(mlm_handle h, int32_t *out, size_t cap, int32_t lo3[3], int32_t dims3[3]) {
  size_t cells = 0;
  const int rc = reach_export_check(h, out, cap, lo3, dims3, cells);
  if (rc != MLM_OK || !out) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  {
    StreamTemp<int32_t> d_out(h->stream);
    CUDA_TRY(d_out.alloc(cells));
    reach_export_launch(h, cells, d_out);
    CUDA_TRY(cudaMemcpyAsync(out, d_out, cells * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// ---- path-cost matrix (reach_kernels.cuh) --------------------------------------------------------------------------
// at most this many field cells per solve launch (1 GiB of int32 costs), and at least one field
constexpr long long kReachMatrixCells = 1ll << 28;

static ScratchList reach_matrix_scratch(mlm_handle h, size_t cells, size_t fcells, size_t items, size_t rows) {
  return {{(void **)&h->mat_cls, cells}, {(void **)&h->mat_cost, fcells * sizeof(int)},
          {(void **)&h->mat_mark, items * sizeof(int)}, {(void **)&h->mat_list, 2 * items * sizeof(int)},
          {(void **)&h->mat_src, rows * sizeof(int)}, {(void **)&h->mat_ctl, 4 * sizeof(int)}};
}
static void reach_matrix_free(mlm_handle h) {
  scratch_free(reach_matrix_scratch(h, 0, 0, 0, 0));
  h->mat_cap_cells = h->mat_cap_fcells = h->mat_cap_items = h->mat_cap_rows = 0;
}

// the arguments of both variants; R and cells describe the box when the call has work to do
static int reach_matrix_check(mlm_handle h, const double box_min[3], const double box_max[3], const void *starts,
                              size_t n_starts, const void *goals, size_t n_goals, double max_dist, int flags,
                              const void *out, ReachGrid &R, long long &cells) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!box_min || !box_max || (!starts && n_starts) || (!goals && n_goals) || (!out && n_starts && n_goals) ||
      (flags & ~(MLM_REACH_INFLATED | MLM_REACH_UNKNOWN)) || !std::isfinite(max_dist) || !(max_dist > 0)) {
    g_last_error = "mlm_reach_matrix: null box, a null pointer with a non-zero count, flags other than "
                   "MLM_REACH_INFLATED | MLM_REACH_UNKNOWN, or max_dist not finite and > 0";
    return MLM_ERR_INVALID_ARG;
  }
  if (n_starts && n_goals > SIZE_MAX / sizeof(double) / n_starts) {
    g_last_error = "mlm_reach_matrix: n_starts * n_goals entries overflow";
    return MLM_ERR_INVALID_ARG;
  }
  const int rc = refuse_sharded(h, "mlm_reach_matrix");
  if (rc != MLM_OK) return rc;
  return reach_grid_of(h, box_min, box_max, max_dist, flags, "mlm_reach_matrix", R, cells);
}

// one class gather, then per batch of fields: reset, seed, one cooperative solve, the batch's rows of the matrix
static int reach_matrix_enqueue(mlm_handle h, const ReachGrid &R, long long cells, const double *d_starts,
                                size_t n_starts, const double *d_goals, size_t n_goals, double *d_out) {
  const size_t tiles = (size_t)R.tiles[0] * R.tiles[1] * R.tiles[2];
  const size_t batch = std::min<size_t>(n_starts, (size_t)std::max<long long>(1, kReachMatrixCells / cells));
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t need[4] = {(size_t)cells, batch * cells, batch * tiles, batch};
  size_t *cap[4] = {&h->mat_cap_cells, &h->mat_cap_fcells, &h->mat_cap_items, &h->mat_cap_rows};
  if (need[0] > *cap[0] || need[1] > *cap[1] || need[2] > *cap[2] || need[3] > *cap[3]) {
    size_t grown[4];
    for (int k = 0; k < 4; k++) grown[k] = std::max(need[k], *cap[k]);
    reach_matrix_free(h);
    const int rc = scratch_alloc(reach_matrix_scratch(h, grown[0], grown[1], grown[2], grown[3]),
                                 "mlm_reach_matrix: scratch buffers");
    if (rc != MLM_OK) return rc;
    for (int k = 0; k < 4; k++) *cap[k] = grown[k];
  }
  cudaStream_t s = h->stream;
  const int subs = R.box.gdims[0] * R.box.gdims[1] * R.box.gdims[2];
  if (R.flags & MLM_REACH_INFLATED) k_esdf_gather<true><<<subs, 256, 0, s>>>(h->P, h->D, R.box, h->mat_cls);
  else k_esdf_gather<false><<<subs, 256, 0, s>>>(h->P, h->D, R.box, h->mat_cls);
  h->launches++;
  int per_sm = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_reach_matrix_solve, kReachThreads, 0));
  for (size_t row0 = 0; row0 < n_starts; row0 += batch) {
    const size_t nb = std::min(batch, n_starts - row0);
    CUDA_TRY(cudaMemsetAsync(h->mat_cost, 0x7f, nb * cells * sizeof(int), s));  // kReachInf
    CUDA_TRY(cudaMemsetAsync(h->mat_mark, 0, nb * tiles * sizeof(int), s));
    CUDA_TRY(cudaMemsetAsync(h->mat_ctl, 0, 4 * sizeof(int), s));
    ReachWork W = {h->mat_mark, h->mat_list, h->mat_list + nb * tiles, h->mat_ctl,
                   reinterpret_cast<unsigned *>(h->mat_ctl + 3)};
    k_reach_matrix_seed<<<grid_for(nb, 256), 256, 0, s>>>(R, d_starts + 3 * row0, (int)nb, (size_t)cells, (int)tiles,
                                                          h->mat_src, h->mat_cost, W);
    // as many CTAs as are resident at once, at most one per work item
    const int G = (int)std::min<size_t>((size_t)h->sm_count * std::max(per_sm, 1), nb * tiles);
    ReachGrid Rs = R;
    const uint8_t *cls = h->mat_cls;
    int *cost = h->mat_cost;
    const int *src = h->mat_src;
    size_t fc = (size_t)cells;
    int nt = (int)tiles;
    void *args[] = {&Rs, &cls, &cost, &W, &src, &fc, &nt};
    CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_reach_matrix_solve, dim3(G), dim3(kReachThreads), args, 0, s));
    k_reach_matrix_gather<<<grid_for(nb * n_goals, 256), 256, 0, s>>>(R, h->mat_cost, (size_t)cells, d_goals, n_goals,
                                                                      nb * n_goals, d_out + row0 * n_goals);
    h->launches += 3;
  }
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

int mlm_reach_matrix_device(mlm_handle h, const double box_min[3], const double box_max[3], const double *d_starts,
                            size_t n_starts, const double *d_goals, size_t n_goals, double max_dist, int flags,
                            double *d_out) {
  ReachGrid R;
  long long cells = 0;
  const int rc = reach_matrix_check(h, box_min, box_max, d_starts, n_starts, d_goals, n_goals, max_dist, flags, d_out,
                                    R, cells);
  if (rc != MLM_OK || n_starts == 0 || n_goals == 0) return rc;
  return reach_matrix_enqueue(h, R, cells, d_starts, n_starts, d_goals, n_goals, d_out);
}
// the host variant stages the starts, goals and matrix through the handle's stream
int mlm_reach_matrix(mlm_handle h, const double box_min[3], const double box_max[3], const double *starts,
                     size_t n_starts, const double *goals, size_t n_goals, double max_dist, int flags, double *out) {
  ReachGrid R;
  long long cells = 0;
  int rc = reach_matrix_check(h, box_min, box_max, starts, n_starts, goals, n_goals, max_dist, flags, out, R, cells);
  if (rc != MLM_OK || n_starts == 0 || n_goals == 0) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t n = n_starts * n_goals;
  {
    StreamTemp<double> d_buf(s);  // starts, goals, matrix
    CUDA_TRY(d_buf.alloc(3 * n_starts + 3 * n_goals + n));
    double *d_s = d_buf, *d_g = d_s + 3 * n_starts, *d_o = d_g + 3 * n_goals;
    CUDA_TRY(cudaMemcpyAsync(d_s, starts, n_starts * 24, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_g, goals, n_goals * 24, cudaMemcpyHostToDevice, s));
    rc = reach_matrix_enqueue(h, R, cells, d_s, n_starts, d_g, n_goals, d_o);
    if (rc != MLM_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, d_o, n * sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// ---- frontier clustering (frontier_kernels.cuh) ------------------------------------------------------------------
size_t mlm_sizeof_frontier_cluster(void) { return sizeof(mlm_frontier_cluster); }
static_assert(sizeof(mlm_frontier_cluster) == sizeof(FrontierCluster), "mlm_frontier_cluster / FrontierCluster layouts differ");

// per-word buffers, allocated by the first call
static ScratchList frontier_word_scratch(mlm_handle h) {
  FcScratch &S = h->fc;
  const size_t words = (size_t)h->P.pool_blocks * h->P.front_words, slots = (size_t)h->P.ht_mask + 1;
  return {{(void **)&S.mword, words * 4}, {(void **)&S.wbase, words * 4}, {(void **)&S.slot_cnt, (slots + 1) * 4},
          {(void **)&S.counters, 16 * 4}};
}
// per-cell buffers for c frontier cells, grown by a larger frontier
static ScratchList frontier_cell_scratch(mlm_handle h, size_t c) {
  FcScratch &S = h->fc;
  return {{(void **)&S.parent, c * 4},     {(void **)&S.acc_n, c * 4},      {(void **)&S.map, c * 4},
          {(void **)&S.sv[0], c * 4},      {(void **)&S.sv[1], c * 4},      {(void **)&S.acc_lo, 3 * c * 4},
          {(void **)&S.acc_hi, 3 * c * 4}, {(void **)&S.acc_s, 3 * c * 8},  {(void **)&S.acc_key, c * 8},
          {(void **)&S.sk[0], c * 8},      {(void **)&S.sk[1], c * 8}};
}
static void frontier_free(mlm_handle h) {
  scratch_free(frontier_cell_scratch(h, 0));
  scratch_free(frontier_word_scratch(h));
  h->fc_cap_cells = 0;
}

static int frontier_clusters(mlm_handle h, const double box_min[3], const double box_max[3], int32_t min_cells, int flags,
                             mlm_frontier_cluster *out, size_t cap, size_t *n_out, int32_t *cells3, int32_t *cluster_of,
                             size_t cell_cap, size_t *n_cells_out, bool device_out) {
  if (!h || !n_out) return MLM_ERR_INVALID_ARG;
  if ((!box_min) != (!box_max) || min_cells < 1 || (flags & ~MLM_FRONTIER_CONN6) || (!out && cap) ||
      ((!cells3 || !cluster_of) && cell_cap)) {
    g_last_error = "mlm_frontier_clusters: one box pointer without the other, min_cells < 1, unknown flags, or a null "
                   "output with a non-zero cap";
    return MLM_ERR_INVALID_ARG;
  }
  FcBox B = {{INT_MIN, INT_MIN, INT_MIN}, {INT_MAX, INT_MAX, INT_MAX}, box_min ? 0 : 1};
  for (int k = 0; box_min && k < 3; k++) {
    const int rc = box_axis_cells(h, box_min[k], box_max[k], "mlm_frontier_clusters", &B.lo[k], &B.hi[k]);
    if (rc != MLM_OK) return rc;
  }
  if (!h->P.explore) {
    g_last_error = "mlm_frontier_clusters: the handle was created without use_exploration_frontiers";
    return MLM_ERR_UNSUPPORTED;
  }
  int rc = refuse_sharded(h, "mlm_frontier_clusters");
  if (rc != MLM_OK) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const MapParams &P = h->P;
  FcScratch &S = h->fc;
  const int slots = (int)P.ht_mask + 1;
  if (!S.mword) {
    rc = scratch_alloc(frontier_word_scratch(h), "mlm_frontier_clusters: scratch");
    if (rc != MLM_OK) return rc;
  }
  const int wgrid = h->sm_count * 8;  // warp-per-slot kernels: one full wave of 256-thread CTAs, grid-stride over the slots
  k_fc_count<<<wgrid, 256, 0, s>>>(P, h->D, B, S);
  k_fc_scan<<<1, kFcScanThreads, 0, s>>>(S.slot_cnt, slots);
  h->launches += 2;
  int total = 0;
  CUDA_TRY(cudaMemcpyAsync(&total, S.slot_cnt + slots, sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));  // the number of frontier cells sizes the per-cell buffers
  if ((size_t)total > h->fc_cap_cells) {
    scratch_free(frontier_cell_scratch(h, 0));
    h->fc_cap_cells = 0;
    rc = scratch_alloc(frontier_cell_scratch(h, (size_t)total), "mlm_frontier_clusters: per-cell buffers");
    if (rc != MLM_OK) return rc;
    h->fc_cap_cells = (size_t)total;
  }
  int counts[2] = {0, 0};  // clusters kept, cells of kept clusters
  if (total > 0) {
    const int cgrid = std::min(grid_for((size_t)total, 256), wgrid);
    const int init[9] = {0, 0, INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN, 0};
    k_fc_index<<<wgrid, 256, 0, s>>>(P, h->D, S);
    if (flags & MLM_FRONTIER_CONN6) k_fc_hook<true><<<wgrid, 256, 0, s>>>(P, h->D, B, S);
    else k_fc_hook<false><<<wgrid, 256, 0, s>>>(P, h->D, B, S);
    k_fc_compress<<<cgrid, 256, 0, s>>>(S, total);
    k_fc_reduce<0><<<wgrid, 256, 0, s>>>(P, h->D, S);
    k_fc_reduce<1><<<wgrid, 256, 0, s>>>(P, h->D, S);
    CUDA_TRY(cudaMemcpyAsync(S.counters, init, sizeof(init), cudaMemcpyHostToDevice, s));
    k_fc_select<<<cgrid, 256, 0, s>>>(S, total, min_cells);
    k_fc_sort<<<1, kFcSortThreads, 0, s>>>(S);
    h->launches += 7;
    const size_t rec_n = std::min(cap, (size_t)total), lab_n = std::min(cell_cap, (size_t)total);
    StreamTemp<FrontierCluster> t_out(s);
    StreamTemp<int32_t> t_cells(s);  // cells, then labels
    if (!device_out && rec_n) CUDA_TRY(t_out.alloc(rec_n));
    if (!device_out && lab_n) CUDA_TRY(t_cells.alloc(lab_n * 4));
    FrontierCluster *d_out = device_out ? reinterpret_cast<FrontierCluster *>(out) : t_out;
    int32_t *d_cells = device_out ? cells3 : t_cells, *d_of = device_out ? cluster_of : t_cells + 3 * lab_n;
    k_fc_records<<<cgrid, 256, 0, s>>>(S, P.d_sub, d_out, rec_n);
    h->launches++;
    if (lab_n) {
      k_fc_labels<false><<<wgrid, 256, 0, s>>>(P, h->D, S, nullptr, nullptr, 0);
      k_fc_scan<<<1, kFcScanThreads, 0, s>>>(S.slot_cnt, slots);
      k_fc_labels<true><<<wgrid, 256, 0, s>>>(P, h->D, S, d_cells, d_of, lab_n);
      h->launches += 3;
    }
    CUDA_TRY(cudaMemcpyAsync(counts, S.counters, sizeof(counts), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));  // the counts
    if (!device_out) {
      const size_t nr = std::min(rec_n, (size_t)counts[0]), nl = std::min(lab_n, (size_t)counts[1]);
      if (nr) CUDA_TRY(cudaMemcpyAsync(out, d_out, nr * sizeof(FrontierCluster), cudaMemcpyDeviceToHost, s));
      if (nl) CUDA_TRY(cudaMemcpyAsync(cells3, d_cells, nl * 12, cudaMemcpyDeviceToHost, s));
      if (nl) CUDA_TRY(cudaMemcpyAsync(cluster_of, d_of, nl * 4, cudaMemcpyDeviceToHost, s));
      t_out.reset();
      t_cells.reset();
      CUDA_TRY(cudaStreamSynchronize(s));
    }
  }
  CUDA_TRY(cudaGetLastError());
  *n_out = (size_t)counts[0];
  if (n_cells_out) *n_cells_out = (size_t)counts[1];
  return MLM_OK;
}

int mlm_frontier_clusters(mlm_handle h, const double box_min[3], const double box_max[3], int32_t min_cells, int flags,
                          mlm_frontier_cluster *out, size_t cap, size_t *n_out, int32_t *cells3, int32_t *cluster_of,
                          size_t cell_cap, size_t *n_cells_out) {
  return frontier_clusters(h, box_min, box_max, min_cells, flags, out, cap, n_out, cells3, cluster_of, cell_cap,
                           n_cells_out, false);
}
int mlm_frontier_clusters_device(mlm_handle h, const double box_min[3], const double box_max[3], int32_t min_cells,
                                 int flags, mlm_frontier_cluster *d_out, size_t cap, size_t *n_out, int32_t *d_cells3,
                                 int32_t *d_cluster_of, size_t cell_cap, size_t *n_cells_out) {
  return frontier_clusters(h, box_min, box_max, min_cells, flags, d_out, cap, n_out, d_cells3, d_cluster_of, cell_cap,
                           n_cells_out, true);
}

// ---- candidate-view gain (view_kernels.cuh) -----------------------------------------------------------------------
size_t mlm_sizeof_view_gain(void) { return sizeof(mlm_view_gain_record); }
static_assert(sizeof(mlm_view_gain_record) == sizeof(ViewGain), "mlm_view_gain_record / ViewGain layouts differ");
static_assert(sizeof(mlm_view_sensor) == sizeof(ViewSensor), "mlm_view_sensor / ViewSensor layouts differ");

static ScratchList view_scratch(mlm_handle h, size_t n) {
  return {{(void **)&h->view_setup, n * sizeof(ViewSetup)}, {(void **)&h->view_tiles, n * sizeof(unsigned long long)}};
}
static void view_free(mlm_handle h) {
  scratch_free(view_scratch(h, 0));
  h->view_cap = 0;
}

static int view_gain_check(mlm_handle h, const void *poses, size_t n, const mlm_view_sensor *S, int flags, const void *out) {
  if (!h || !S || !out || (!poses && n) || (flags & ~(MLM_VIEW_FRONTIER | MLM_VIEW_INFLATED))) return MLM_ERR_INVALID_ARG;
  const double f[6] = {S->fx, S->fy, S->cx, S->cy, S->min_depth, S->max_depth};
  for (double v : f)
    if (!std::isfinite(v)) return MLM_ERR_INVALID_ARG;
  if (!(S->fx > 0) || !(S->fy > 0) || S->cols < 1 || S->rows < 1 || !(0 <= S->min_depth && S->min_depth < S->max_depth)) {
    g_last_error = "mlm_view_gain: fx or fy <= 0, cols or rows < 1, or not 0 <= min_depth < max_depth";
    return MLM_ERR_INVALID_ARG;
  }
  const double lim = kViewMaxCells * h->P.d_sub;
  const double hx = std::max(std::fabs((-0.5 - S->cx) / S->fx), std::fabs(((double)S->cols - 0.5 - S->cx) / S->fx));
  const double hy = std::max(std::fabs((-0.5 - S->cy) / S->fy), std::fabs(((double)S->rows - 0.5 - S->cy) / S->fy));
  if (S->max_depth > lim || hx * S->max_depth > lim || hy * S->max_depth > lim) {
    g_last_error = "mlm_view_gain: max_depth, or a far corner's offset from the optical axis, exceeds 256 * d_sub";
    return MLM_ERR_CAPACITY;
  }
  if ((flags & MLM_VIEW_FRONTIER) && !h->P.explore) {
    g_last_error = "mlm_view_gain: MLM_VIEW_FRONTIER on a handle created without use_exploration_frontiers";
    return MLM_ERR_UNSUPPORTED;
  }
  return refuse_sharded(h, "mlm_view_gain");
}
using ViewTilesKernel = void (*)(MapParams, DeviceBuffers, ViewSensor, const ViewSetup *, const unsigned long long *,
                                 size_t, ViewGain *);
static ViewTilesKernel view_tiles_kernel(int flags) {
  switch (flags & (MLM_VIEW_FRONTIER | MLM_VIEW_INFLATED)) {
    case 0: return k_view_tiles<false, false>;
    case MLM_VIEW_INFLATED: return k_view_tiles<false, true>;
    case MLM_VIEW_FRONTIER: return k_view_tiles<true, false>;
    default: return k_view_tiles<true, true>;
  }
}
static int view_gain_launch(mlm_handle h, const double *d_T_wb, size_t n, const mlm_view_sensor *sensor,
                            const int32_t *d_boxes, int flags, mlm_view_gain_record *d_out) {
  if (n > h->view_cap) {
    view_free(h);
    const int rc = scratch_alloc(view_scratch(h, n), "mlm_view_gain: per-view scratch");
    if (rc != MLM_OK) return rc;
    h->view_cap = n;
  }
  ViewSensor S;
  memcpy(&S, sensor, sizeof(S));
  ViewGain *o = reinterpret_cast<ViewGain *>(d_out);
  k_view_setup<<<grid_for(n, 256), 256, 0, h->stream>>>(h->P, h->T_bs, S, d_T_wb, d_boxes, n, h->view_setup,
                                                         h->view_tiles, o);
  k_view_scan<<<1, kViewScanThreads, 0, h->stream>>>(h->view_tiles, n);
  // a persistent grid over the (view, tile) items: as many CTAs as fit on the GPU at once
  const ViewTilesKernel k = view_tiles_kernel(flags);
  int per_sm = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kViewTileThreads, 0));
  k<<<h->sm_count * std::max(per_sm, 1), kViewTileThreads, 0, h->stream>>>(h->P, h->D, S, h->view_setup, h->view_tiles, n, o);
  h->launches += 3;
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
int mlm_view_gain_device(mlm_handle h, const double *d_T_wb, size_t n, const mlm_view_sensor *sensor,
                         const int32_t *d_boxes, int flags, mlm_view_gain_record *d_out) {
  const int rc = view_gain_check(h, d_T_wb, n, sensor, flags, d_out);
  if (rc != MLM_OK) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n == 0) return MLM_OK;
  return view_gain_launch(h, d_T_wb, n, sensor, d_boxes, flags, d_out);
}
// the host variant stages the poses, boxes and records through the handle's stream (like mlm_cast_rays)
int mlm_view_gain(mlm_handle h, const double *T_wb, size_t n, const mlm_view_sensor *sensor, const int32_t *boxes,
                  int flags, mlm_view_gain_record *out) {
  int rc = view_gain_check(h, T_wb, n, sensor, flags, out);
  if (rc != MLM_OK) return rc;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<double> d_p(s);
    StreamTemp<int32_t> d_b(s);
    StreamTemp<mlm_view_gain_record> d_o(s);
    CUDA_TRY(d_p.alloc(n * 7));
    CUDA_TRY(d_o.alloc(n));
    CUDA_TRY(cudaMemcpyAsync(d_p, T_wb, n * 56, cudaMemcpyHostToDevice, s));
    if (boxes) {
      CUDA_TRY(d_b.alloc(n * 6));
      CUDA_TRY(cudaMemcpyAsync(d_b, boxes, n * 24, cudaMemcpyHostToDevice, s));
    }
    rc = view_gain_launch(h, d_p, n, sensor, d_b, flags, d_o);
    if (rc != MLM_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, d_o, n * sizeof(mlm_view_gain_record), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

// ---- stream control ----------------------------------------------------------------------------------
int mlm_sync(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
int mlm_timer_start(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
  return MLM_OK;
}
int mlm_timer_stop_ms(mlm_handle h, float *ms) {
  if (!h || !ms) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
  CUDA_TRY(cudaEventSynchronize(h->ev1));
  CUDA_TRY(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return MLM_OK;
}
int mlm_device_alloc(mlm_handle h, size_t bytes, void **d_ptr) {
  if (!h || !d_ptr) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMalloc(d_ptr, bytes));
  return MLM_OK;
}
int mlm_device_free(mlm_handle h, void *d_ptr) {
  if (!h) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaFree(d_ptr));
  return MLM_OK;
}
int mlm_host_alloc(mlm_handle h, size_t bytes, void **ptr) {
  if (!h || !ptr) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMallocHost(ptr, bytes));
  return MLM_OK;
}
int mlm_host_free(mlm_handle h, void *ptr) {
  if (!h) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaFreeHost(ptr));
  return MLM_OK;
}
int mlm_copy_to_device(mlm_handle h, void *d_dst, const void *src, size_t bytes) {
  if (!h || !d_dst || !src) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(d_dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return MLM_OK;
}
int mlm_copy_to_host(mlm_handle h, void *dst, const void *d_src, size_t bytes) {
  if (!h || !dst || !d_src) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(dst, d_src, bytes, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return MLM_OK;
}
int mlm_flush_l2(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->l2_buf) {
    h->l2_bytes = (size_t)256 << 20;  // > 126 MB L2
    CUDA_TRY(cudaMalloc(&h->l2_buf, h->l2_bytes));
  }
  static uint32_t v = 1;
  k_l2_flush<<<h->sm_count * 8, 256, 0, h->stream>>>((uint4 *)h->l2_buf, h->l2_bytes / 16, v++);
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return MLM_OK;
}
int mlm_set_profiling(mlm_handle h, int enable) {
  if (!h) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (enable && !h->kev[0])
    for (int i = 0; i <= MLM_NUM_FRAME_KERNELS; i++) CUDA_TRY(cudaEventCreate(&h->kev[i]));
  h->profiling = enable != 0;
  return MLM_OK;
}
int mlm_last_frame_kernel_ms(mlm_handle h, float ms[MLM_NUM_FRAME_KERNELS]) {
  if (!h || !ms) return MLM_ERR_INVALID_ARG;
  for (int i = 0; i < MLM_NUM_FRAME_KERNELS; i++) ms[i] = h->kms[i];
  return MLM_OK;
}
int mlm_debug_phase_cycles(mlm_handle h, long long *out, size_t cap) {
  if (!h || !out) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  size_t n = std::min(cap, (size_t)(h->P.nCol + 256) * 16);
  CUDA_TRY(cudaMemcpy(out, h->D.debug_cycles, n * sizeof(long long), cudaMemcpyDeviceToHost));
  return MLM_OK;
}
int mlm_srand(mlm_handle h, unsigned seed) {
  if (!h) return MLM_ERR_INVALID_ARG;
  h->rng.seed(seed);
  return MLM_OK;
}
int mlm_debug_rand(mlm_handle h, int32_t *out, size_t n) {
  if (!out && n) return MLM_ERR_INVALID_ARG;
  GlibcRand local;
  GlibcRand &g = h ? h->rng : local;
  for (size_t i = 0; i < n; i++) out[i] = g.next();
  return MLM_OK;
}
int mlm_kernel_launch_count(mlm_handle h, int64_t *count) {
  if (!h || !count) return MLM_ERR_INVALID_ARG;
  *count = h->launches;
  return MLM_OK;
}

// ---- parity / debug exports --------------------------------------------------------------------------
int mlm_last_frame_hits(mlm_handle h, int32_t *keys3, float *p, size_t cap, size_t *n_out) {
  if (!h || !n_out) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  const int n = h->last_n_hit;
  *n_out = (size_t)n;
  if (n == 0 || cap < (size_t)n || !keys3 || !p) return MLM_OK;
  cudaStream_t s = h->stream;
  const int T = 256, n_pad = next_pow2(n);
  {
    OrderArrays O;
    O.key = h->D.hit_key;
    O.stamp = h->D.hit_t;
    O.bucket = h->D.hit_bucket;
    O.kind = 0;
    k_order_seed<<<grid_for(n_pad, T), T, 0, s>>>(O, h->d_sort_a, n, n_pad);
  }
  device_sort(h, h->d_sort_a, n_pad);
  k_export_hit_keys<<<grid_for(n_pad, T), T, 0, s>>>(h->P, h->D, h->D.act[h->last_parity], h->d_sort_b, n, n_pad,
                                                      h->last_order_B);
  device_sort(h, h->d_sort_b, n_pad);
  {
    StreamTemp<int> d_k3(s);
    StreamTemp<float> d_p(s);
    CUDA_TRY(d_k3.alloc((size_t)n * 3));
    CUDA_TRY(d_p.alloc((size_t)n));
    k_export_hit_gather<<<grid_for(n, T), T, 0, s>>>(h->P, h->D, h->d_sort_a, h->d_sort_b, n, d_k3, d_p);
    h->launches += 3;
    CUDA_TRY(cudaMemcpyAsync(keys3, d_k3, (size_t)n * 12, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(p, d_p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

int mlm_last_frame_misses(mlm_handle h, uint64_t *idx, size_t cap, size_t *n_out) {
  if (!h || !n_out) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const size_t words = (size_t)h->P.nPhi * h->P.col_words;
  {
    StreamTemp<int> d_cnt(s);
    StreamTemp<unsigned long long> d_out(s);
    CUDA_TRY(d_cnt.alloc(1));
    CUDA_TRY(d_out.alloc(std::max<size_t>(cap, 1)));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(int), s));
    k_export_miss<<<grid_for(words, 256), 256, 0, s>>>(h->P, h->D, d_out, d_cnt, (int)std::min<size_t>(cap, 0x7fffffff));
    h->launches++;
    int cnt = 0;
    CUDA_TRY(cudaMemcpyAsync(&cnt, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_out = (size_t)cnt;
    if (idx && cap >= (size_t)cnt && cnt > 0) {
      CUDA_TRY(cudaMemcpyAsync(idx, d_out, (size_t)cnt * 8, cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaStreamSynchronize(s));
      std::sort(idx, idx + cnt);  // export formatting only: ascending cell index
    }
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

int mlm_export_map_count(mlm_handle h, size_t *n_submaps) {
  if (!h || !n_submaps) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  *n_submaps = (size_t)h->n_submaps;
  return MLM_OK;
}

namespace {
// shared by mlm_export_map / mlm_export_frontier: front == nullptr skips the frontier bitmasks
int export_common(mlm_handle h, size_t cap_submaps, int32_t *glb3, uint8_t *collapsed, char *occupancy,
                  char *inflate_occupancy, float *log_odds, uint32_t *front, size_t *n_out) {
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const MapParams &P = h->P;
  const size_t cap = std::max<size_t>(cap_submaps, 1);
  {
    StreamTemp<int> d_cnt(s), d_glb(s), d_blk(s);
    CUDA_TRY(d_cnt.alloc(1));
    CUDA_TRY(d_glb.alloc(cap * 3));
    CUDA_TRY(d_blk.alloc(cap));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(int), s));
    k_export_list<<<grid_for((size_t)P.ht_mask + 1, 256), 256, 0, s>>>(P, h->D, d_glb, d_blk, d_cnt, (int)cap_submaps);
    int cnt = 0;
    CUDA_TRY(cudaMemcpyAsync(&cnt, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_out = (size_t)cnt;
    if (cnt > 0 && (size_t)cnt <= cap_submaps) {
      const size_t cells = (size_t)cnt * P.cells;
      StreamTemp<char> d_occ(s), d_inf(s);
      StreamTemp<float> d_lo(s);
      StreamTemp<unsigned char> d_col(s);
      StreamTemp<uint32_t> d_front(s);
      CUDA_TRY(d_occ.alloc(cells));
      CUDA_TRY(d_inf.alloc(cells));
      CUDA_TRY(d_lo.alloc(cells));
      CUDA_TRY(d_col.alloc((size_t)cnt));
      if (front) CUDA_TRY(d_front.alloc((size_t)cnt * P.front_words));
      k_export_blocks<<<cnt, 256, 0, s>>>(P, h->D, d_blk, cnt, d_occ, d_inf, d_lo, d_col, d_front);
      CUDA_TRY(cudaMemcpyAsync(glb3, d_glb, (size_t)cnt * 12, cudaMemcpyDeviceToHost, s));
      if (collapsed) CUDA_TRY(cudaMemcpyAsync(collapsed, d_col, (size_t)cnt, cudaMemcpyDeviceToHost, s));
      if (occupancy) CUDA_TRY(cudaMemcpyAsync(occupancy, d_occ, cells, cudaMemcpyDeviceToHost, s));
      if (inflate_occupancy) CUDA_TRY(cudaMemcpyAsync(inflate_occupancy, d_inf, cells, cudaMemcpyDeviceToHost, s));
      if (log_odds) CUDA_TRY(cudaMemcpyAsync(log_odds, d_lo, cells * 4, cudaMemcpyDeviceToHost, s));
      if (front) CUDA_TRY(cudaMemcpyAsync(front, d_front, (size_t)cnt * P.front_words * 4, cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaStreamSynchronize(s));
      h->launches += 2;
    }
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
}  // namespace

int mlm_export_map(mlm_handle h, size_t cap_submaps, int32_t *glb3, uint8_t *collapsed, char *occupancy,
                   char *inflate_occupancy, float *log_odds, size_t *n_out) {
  if (!h || !n_out || !glb3 || !collapsed || !occupancy || !inflate_occupancy || !log_odds) return MLM_ERR_INVALID_ARG;
  return export_common(h, cap_submaps, glb3, collapsed, occupancy, inflate_occupancy, log_odds, nullptr, n_out);
}

int mlm_export_frontier(mlm_handle h, size_t cap_submaps, int32_t *glb3, uint32_t *frontier_words, size_t *n_out) {
  if (!h || !n_out || !glb3 || !frontier_words) return MLM_ERR_INVALID_ARG;
  return export_common(h, cap_submaps, glb3, nullptr, nullptr, nullptr, nullptr, frontier_words, n_out);
}

// ---- sharded map: stage / order / emit / ingest (SURVEY §8e); collectives are the caller's (NCCL via torch.distributed)
namespace {
// kind >= 0: k_export_cloud, kind < 0: odds slice at `height`; device_out: xyzw is device memory
int export_points(mlm_handle h, int kind, double height, float *xyzw, size_t cap, size_t *n_out, bool device_out) {
  if (!h || !n_out || (cap && !xyzw) || kind > MLM_CLOUD_FRONTIER) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  {
    StreamTemp<unsigned long long> d_cnt(s);
    StreamTemp<float4> t_out(s);
    CUDA_TRY(d_cnt.alloc(1));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), s));
    if (!device_out && cap) CUDA_TRY(t_out.alloc(cap));
    float4 *d_out = device_out ? reinterpret_cast<float4 *>(xyzw) : t_out;
    const int grid = h->sm_count * 8;  // 8 resident CTAs of 256 threads per SM: one full wave, grid-stride over the slots
    if (kind >= 0)
      k_export_cloud<<<grid, 256, 0, s>>>(h->P, h->D, kind, d_out, d_cnt, (unsigned long long)cap);
    else
      k_export_odds_slice<<<grid, 256, 0, s>>>(h->P, h->D, height, d_out, d_cnt, (unsigned long long)cap);
    h->launches++;
    unsigned long long cnt = 0;
    CUDA_TRY(cudaMemcpyAsync(&cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_out = (size_t)cnt;
    const size_t n_copy = std::min<size_t>((size_t)cnt, cap);
    if (!device_out && n_copy) CUDA_TRY(cudaMemcpyAsync(xyzw, d_out, n_copy * sizeof(float4), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
}  // namespace

int mlm_export_cloud(mlm_handle h, int kind, float *xyzw, size_t cap, size_t *n_out) {
  if (kind < 0) return MLM_ERR_INVALID_ARG;
  return export_points(h, kind, 0.0, xyzw, cap, n_out, false);
}
int mlm_export_cloud_device(mlm_handle h, int kind, float *d_xyzw, size_t cap, size_t *n_out) {
  if (kind < 0) return MLM_ERR_INVALID_ARG;
  return export_points(h, kind, 0.0, d_xyzw, cap, n_out, true);
}
int mlm_export_odds_slice(mlm_handle h, double height, float *xyzw, size_t cap, size_t *n_out) {
  return export_points(h, -1, height, xyzw, cap, n_out, false);
}

namespace {
struct CkptFileHeader {
  char magic[8];            // "MLMCKPT1"
  uint32_t version, header_bytes;
  mlm_config cfg;           // configuration of the saving handle (the map-defining fields must match on restore)
  int32_t cells, front_words, explore, rec_bytes;
  uint64_t n_records;
  uint32_t bucket_count, bucket_count_miss;
  int64_t cum_ram_expand, cum_obs, n_submaps;
  int32_t rng_r[31];
  int32_t rng_f, rng_b;
  uint64_t checksum;        // FNV-1a 64 over the record bytes
};
uint64_t fnv1a64(const unsigned char *p, size_t n) {
  uint64_t hsh = 0xcbf29ce484222325ull;
  // 8 bytes per step (the images are tens of MB); the tail byte-wise
  size_t i = 0;
  for (; i + 8 <= n; i += 8) {
    uint64_t w;
    memcpy(&w, p + i, 8);
    hsh = (hsh ^ w) * 0x100000001b3ull;
  }
  for (; i < n; i++) hsh = (hsh ^ p[i]) * 0x100000001b3ull;
  return hsh;
}
bool on_bucket_chain(uint32_t B) {
  for (int i = 0; i < kBucketChainLen; i++)
    if (kBucketChain[i] == B) return true;
  return false;
}
const char kCkptMagic[8] = {'M', 'L', 'M', 'C', 'K', 'P', 'T', '1'};
bool same_map_config(const mlm_config &a, const mlm_config &b) {
  return a.am_d_rho == b.am_d_rho && a.am_d_phi_deg == b.am_d_phi_deg && a.am_d_z == b.am_d_z && a.am_n_rho == b.am_n_rho &&
         a.am_n_z_below == b.am_n_z_below && a.am_n_z_over == b.am_n_z_over && a.use_raycasting == b.use_raycasting &&
         a.depth_noise_coe == b.depth_noise_coe && a.subbox_d_xyz == b.subbox_d_xyz && a.subbox_n == b.subbox_n &&
         a.log_odds_min == b.log_odds_min && a.log_odds_max == b.log_odds_max && a.log_odds_miss == b.log_odds_miss &&
         a.log_odds_occupied_sh == b.log_odds_occupied_sh && a.use_exploration_frontiers == b.use_exploration_frontiers;
}
int count_submaps(mlm_handle h, size_t *n) {
  size_t cnt = 0;
  int rc = mlm_export_map_count(h, &cnt);
  *n = cnt;
  return rc;
}
}  // namespace

int mlm_checkpoint_size(mlm_handle h, size_t *bytes) {
  if (!h || !bytes) return MLM_ERR_INVALID_ARG;
  size_t n = 0;
  int rc = count_submaps(h, &n);
  if (rc != MLM_OK) return rc;
  *bytes = sizeof(CkptFileHeader) + n * ckpt_record_bytes(h->P.cells, h->P.front_words, h->P.explore);
  return MLM_OK;
}

int mlm_checkpoint_save(mlm_handle h, void *buf, size_t cap, size_t *written) {
  if (!h || !buf || !written) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const MapParams &P = h->P;
  size_t n = 0;
  int rc = count_submaps(h, &n);
  if (rc != MLM_OK) return rc;
  const size_t rb = ckpt_record_bytes(P.cells, P.front_words, P.explore);
  const size_t need = sizeof(CkptFileHeader) + n * rb;
  *written = need;
  if (cap < need) {
    g_last_error = "checkpoint buffer too small";
    return MLM_ERR_CAPACITY;
  }
  CkptFileHeader hd;
  memset(&hd, 0, sizeof(hd));
  memcpy(hd.magic, kCkptMagic, 8);
  hd.version = 2;
  hd.header_bytes = (uint32_t)sizeof(hd);
  hd.cfg = h->cfg;
  hd.cells = P.cells;
  hd.front_words = P.front_words;
  hd.explore = P.explore;
  hd.rec_bytes = (int32_t)rb;
  hd.n_records = n;
  hd.bucket_count = h->bucket_count;
  hd.bucket_count_miss = h->bucket_count_miss;
  hd.cum_ram_expand = h->cum_ram_expand;
  hd.cum_obs = h->cum_obs;
  hd.n_submaps = h->n_submaps;
  memcpy(hd.rng_r, h->rng.r, sizeof(hd.rng_r));
  hd.rng_f = h->rng.f;
  hd.rng_b = h->rng.b;
  hd.checksum = fnv1a64(nullptr, 0);
  memcpy(buf, &hd, sizeof(hd));
  if (n == 0) return MLM_OK;
  const size_t batch = std::max<size_t>(1, std::min<size_t>(n, ((size_t)256 << 20) / rb));
  unsigned char *dst = reinterpret_cast<unsigned char *>(buf) + sizeof(hd);
  {
    StreamTemp<int> d_cnt(s), d_glb(s), d_blk(s);
    StreamTemp<unsigned char> d_rec(s);
    CUDA_TRY(d_cnt.alloc(1));
    CUDA_TRY(d_glb.alloc(n * 3));
    CUDA_TRY(d_blk.alloc(n));
    CUDA_TRY(d_rec.alloc(batch * rb));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(int), s));
    k_export_list<<<grid_for((size_t)P.ht_mask + 1, 256), 256, 0, s>>>(P, h->D, d_glb, d_blk, d_cnt, (int)n);
    for (size_t first = 0; first < n; first += batch) {
      const size_t m = std::min(batch, n - first);
      k_ckpt_pack<<<(unsigned)m, 256, 0, s>>>(P, h->D, d_glb, d_blk, (int)first, (int)m, d_rec);
      CUDA_TRY(cudaMemcpyAsync(dst + first * rb, d_rec, m * rb, cudaMemcpyDeviceToHost, s));
      CUDA_TRY(cudaStreamSynchronize(s));
      h->launches++;
    }
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  hd.checksum = fnv1a64(dst, n * rb);
  memcpy(buf, &hd, sizeof(hd));
  return MLM_OK;
}

int mlm_checkpoint_restore(mlm_handle h, const void *buf, size_t bytes) {
  if (!h || !buf || bytes < sizeof(CkptFileHeader)) return MLM_ERR_INVALID_ARG;
  CkptFileHeader hd;
  memcpy(&hd, buf, sizeof(hd));
  const MapParams &P = h->P;
  const size_t rb = ckpt_record_bytes(P.cells, P.front_words, P.explore);
  if (memcmp(hd.magic, kCkptMagic, 8) != 0 || hd.version != 2 || hd.header_bytes != sizeof(hd)) {
    g_last_error = "not a mlmap_b200 checkpoint (magic / version)";
    return MLM_ERR_INVALID_ARG;
  }
  if (!same_map_config(hd.cfg, h->cfg) || hd.cells != P.cells || hd.explore != P.explore || (size_t)hd.rec_bytes != rb) {
    g_last_error = "checkpoint was taken with a different map configuration";
    return MLM_ERR_INVALID_CONFIG;
  }
  if (bytes < sizeof(hd) + hd.n_records * rb) {
    g_last_error = "truncated checkpoint";
    return MLM_ERR_INVALID_ARG;
  }
  if (hd.n_records > (uint64_t)P.pool_blocks + (uint64_t)(P.explore ? P.ht_mask / 2 : 0)) {
    g_last_error = "checkpoint holds more subboxes than this handle's pool";
    return MLM_ERR_POOL_EXHAUSTED;
  }
  // Everything below is checked BEFORE the live map is touched: a refused image leaves the handle as it was.
  // (1) the emulated bucket counts index this handle's activation arrays: they must be members of the growth chain and
  //     fit the arrays (max_points is not part of the map configuration, so the saving handle may have had larger ones)
  if (!on_bucket_chain(hd.bucket_count) || hd.bucket_count > h->act_cap ||
      (P.explore && (!on_bucket_chain(hd.bucket_count_miss) || hd.bucket_count_miss > h->act_miss_cap))) {
    g_last_error = "checkpoint bucket counts are not on the libstdc++ growth chain or exceed this handle's capacity (max_points)";
    return MLM_ERR_CAPACITY;
  }
  // (2) the records are the bytes that were saved
  const unsigned char *recs = reinterpret_cast<const unsigned char *>(buf) + sizeof(hd);
  if (fnv1a64(recs, (size_t)hd.n_records * rb) != hd.checksum) {
    g_last_error = "checkpoint checksum mismatch (corrupt image)";
    return MLM_ERR_INVALID_ARG;
  }
  // (3) every record header is sane: flags, subbox index range, no duplicates, full blocks fit the pool
  {
    std::vector<uint64_t> keys;
    keys.reserve((size_t)hd.n_records);
    uint64_t full_blocks = 0;
    const int lim = 1 << 20;
    for (uint64_t i = 0; i < hd.n_records; i++) {
      CkptRecHeader rh;
      memcpy(&rh, recs + i * rb, sizeof(rh));
      const bool collapsed = rh.flags == 1;
      bool ok = (rh.flags == 0 || (collapsed && P.explore));
      for (int a = 0; a < 3; a++) ok = ok && rh.g[a] >= -lim && rh.g[a] < lim;
      if (!ok) {
        g_last_error = "checkpoint record " + std::to_string(i) + " is malformed";
        return MLM_ERR_INVALID_ARG;
      }
      if (!collapsed) full_blocks++;
      keys.push_back(((uint64_t)(uint32_t)(rh.g[0] + lim) << 42) | ((uint64_t)(uint32_t)(rh.g[1] + lim) << 21) | (uint64_t)(uint32_t)(rh.g[2] + lim));
    }
    std::sort(keys.begin(), keys.end());
    if (std::adjacent_find(keys.begin(), keys.end()) != keys.end()) {
      g_last_error = "checkpoint holds a subbox twice";
      return MLM_ERR_INVALID_ARG;
    }
    if (full_blocks > (uint64_t)P.pool_blocks) {
      g_last_error = "checkpoint holds more subboxes than this handle's pool";
      return MLM_ERR_POOL_EXHAUSTED;
    }
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  CUDA_TRY(cudaStreamSynchronize(s));
  DeviceBuffers &D = h->D;
  const size_t ht_cap = (size_t)P.ht_mask + 1;
  // back to the state mlm_create leaves: empty hash table, full free stack, every block 'u','u',0.f
  CUDA_TRY(cudaMemsetAsync(D.ht_key, 0xff, ht_cap * 8, s));
  CUDA_TRY(cudaMemsetAsync(D.ht_val, 0xff, ht_cap * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.pool_lo, 0, (size_t)P.pool_blocks * P.cell_stride * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.pool_occ, 'u', (size_t)P.pool_blocks * P.cell_stride, s));
  CUDA_TRY(cudaMemsetAsync(D.pool_inf, 'u', (size_t)P.pool_blocks * P.cell_stride, s));
  if (P.explore) {
    CUDA_TRY(cudaMemsetAsync(D.pool_front, 0, (size_t)P.pool_blocks * P.front_words * 4, s));
    CUDA_TRY(cudaMemsetAsync(D.act_miss[0], 0xff, (size_t)h->act_miss_cap * 4, s));
    CUDA_TRY(cudaMemsetAsync(D.act_miss[1], 0xff, (size_t)h->act_miss_cap * 4, s));
  }
  {
    std::vector<int> stack(P.pool_blocks);
    for (int i = 0; i < P.pool_blocks; i++) stack[i] = P.pool_blocks - 1 - i;
    CUDA_TRY(cudaMemcpyAsync(D.free_stack, stack.data(), stack.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    const int top = P.pool_blocks;
    CUDA_TRY(cudaMemcpyAsync(D.free_top, &top, sizeof(int), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));  // `stack` and `top` are read by the copies above
  }
  const size_t lsg_cells = (size_t)P.lsg_dim_xy * P.lsg_dim_xy * P.lsg_dim_z;
  CUDA_TRY(cudaMemsetAsync(D.lsg_flag, 0, lsg_cells * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.lsg_block, 0xff, lsg_cells * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.fc[0], 0, 2 * sizeof(FrameCounters), s));
  CUDA_TRY(cudaMemsetAsync(D.act[0], 0xff, (size_t)h->act_cap * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.act[1], 0xff, (size_t)h->act_cap * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.phi_hist, 0, (size_t)P.nCol * 4, s));
  CUDA_TRY(cudaMemsetAsync(D.phi_bound, 0, (size_t)P.nCol * 4, s));
  memset(h->h_fc, 0, sizeof(FrameCounters));
  int rc = MLM_OK;
  if (hd.n_records) {
    const size_t n = (size_t)hd.n_records;
    const size_t batch = std::max<size_t>(1, std::min<size_t>(n, ((size_t)256 << 20) / rb));
    StreamTemp<int> d_status(s);
    StreamTemp<unsigned char> d_rec(s);
    CUDA_TRY(d_status.alloc(1));
    if (d_rec.alloc(batch * rb) != cudaSuccess) {
      cudaGetLastError();
      g_last_error = "checkpoint restore: out of device memory for the staging buffer";
      return MLM_ERR_CUDA;
    }
    int status = 0;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), s));
    const unsigned char *src = reinterpret_cast<const unsigned char *>(buf) + sizeof(hd);
    for (size_t first = 0; first < n; first += batch) {
      const size_t m = std::min(batch, n - first);
      CUDA_TRY(cudaMemcpyAsync(d_rec, src + first * rb, m * rb, cudaMemcpyHostToDevice, s));
      k_ckpt_unpack<<<(unsigned)m, 256, 0, s>>>(P, D, (int)m, d_rec, d_status);
      h->launches++;
      CUDA_TRY(cudaStreamSynchronize(s));
    }
    CUDA_TRY(cudaMemcpyAsync(&status, d_status, sizeof(int), cudaMemcpyDeviceToHost, s));
    d_status.reset();
    d_rec.reset();
    CUDA_TRY(cudaStreamSynchronize(s));
    if (status) {
      g_last_error = "checkpoint restore: device raised error code " + std::to_string(status);
      rc = map_device_error(status);
    }
  }
  CUDA_TRY(cudaGetLastError());
  h->frame_idx = 0;
  h->last_parity = 0;
  h->bucket_count = hd.bucket_count;
  h->bucket_count_miss = hd.bucket_count_miss;
  h->last_order_B = hd.bucket_count;
  h->last_n_hit = 0;
  h->cum_ram_expand = hd.cum_ram_expand;
  h->cum_obs = hd.cum_obs;
  h->n_submaps = (int64_t)hd.n_records;  // the records actually inserted, not a number taken from the image
  memcpy(h->rng.r, hd.rng_r, sizeof(hd.rng_r));
  h->rng.f = hd.rng_f;
  h->rng.b = hd.rng_b;
  return rc;
}

// ---- one logical map sharded over `world` ranks; the exchanges run over NVLink peer memory (shard_kernels.cuh) ------
namespace {
struct ShardBlob {  // what a rank publishes so that its peers can map its exchange arena (fits MLM_SHARD_BLOB_BYTES)
  uint32_t magic;
  int32_t rank, world, device;
  int32_t hit_cap, rec_cap;
  int32_t max_points, reserved;
  int64_t pid;
  uint64_t ptr;  // arena address in the exporting process (used directly by handles of the same process)
  cudaIpcMemHandle_t ipc;
};
static_assert(sizeof(ShardBlob) <= MLM_SHARD_BLOB_BYTES, "blob must fit the ABI constant");
constexpr uint32_t kShardMagic = 0x4d4c5342u;  // "MLSB"

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
// carve the arena of one rank: flags | mailboxes | cursors | gathered keys | gathered stamps | inboxes
ShardArena carve_arena(void *base, int world, int hit_cap, int rec_cap, int max_points, size_t *total) {
  unsigned char *p = reinterpret_cast<unsigned char *>(base);
  size_t off = 0;
  ShardArena a;
  a.flags = reinterpret_cast<uint32_t *>(p + off);
  off = align256(off + kMaxWorld * sizeof(uint32_t));
  a.mbox = reinterpret_cast<int2 *>(p + off);
  off = align256(off + 2 * kMaxWorld * sizeof(int2));
  a.cursor = reinterpret_cast<int *>(p + off);
  off = align256(off + 2 * sizeof(int));
  a.gather_key = reinterpret_cast<int *>(p + off);
  off = align256(off + (size_t)2 * world * hit_cap * sizeof(int));
  a.gather_stamp = reinterpret_cast<uint32_t *>(p + off);
  off = align256(off + (size_t)2 * world * hit_cap * sizeof(uint32_t));
  a.inbox = reinterpret_cast<ShardRecord *>(p + off);
  off = align256(off + (size_t)2 * rec_cap * sizeof(ShardRecord));
  a.pflags = reinterpret_cast<uint32_t *>(p + off);
  off = align256(off + kMaxWorld * sizeof(uint32_t));
  a.points = reinterpret_cast<double *>(p + off);
  off = align256(off + (size_t)2 * 3 * max_points * sizeof(double));
  if (total) *total = off;
  return a;
}

int shard_check(mlm_handle h, bool need_connected) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!h->shard_open || (need_connected && !h->shard_connected)) {
    g_last_error = "mlm_shard_open / mlm_shard_connect must come first";
    return MLM_ERR_INVALID_ARG;
  }
  return MLM_OK;
}

// everything of one scan after the input is on the device: stage the rank's columns, push keys and records to the
// owners, signal, wait for every source, then the owner-side kernels; no host synchronisation
int shard_enqueue(mlm_handle h, const double *d_xyz, int n, const double T_wb[7], const void *h2d_src = nullptr) {
  cudaStream_t s = h->stream;
  const ShardPeers &X = h->shard_peers;
  const uint32_t epoch = ++h->shard_epoch;
  const int par = (int)(epoch & 1);
  const int parity_next = (int)(h->frame_idx & 1);
  const bool prof = h->profiling != 0;
  if (prof && !h->sev[0])
    for (int i = 0; i <= MLM_NUM_SHARD_KERNELS; i++) CUDA_TRY(cudaEventCreate(&h->sev[i]));
#define MLM_SMARK(i) do { if (prof) cudaEventRecord(h->sev[i], s); } while (0)
  MLM_SMARK(0);
  if (h2d_src && n > 0) CUDA_TRY(cudaMemcpyAsync(h->d_input, h2d_src, (size_t)n * 24, cudaMemcpyHostToDevice, s));
  // resets of the scan in one launch (only the buckets in use: the count can at most step up the growth chain on a rehash
  // scan, which refills the array itself)
  const uint32_t B_now = std::min<uint32_t>(h->bucket_count == 1 ? 13u : h->bucket_count, h->act_cap);
  k_shard_begin<<<std::min(h->sm_count * 2, grid_for(B_now, 256)), 256, 0, s>>>(h->D.act[parity_next], B_now, h->d_shard_cursor, kMaxWorld + 2,
                                                                            X.a[X.rank].cursor + (par ^ 1));
  h->launches++;
  MLM_SMARK(1);
  h->shard_stage_pending = true;
  int rc = run_frame(h, 0, d_xyz, 0, 0, n, T_wb, nullptr);
  h->shard_stage_pending = false;
  if (rc != MLM_OK) return rc;
  MLM_SMARK(3);
  FrameParams F = *h->h_fp;  // as the staging kernels saw it (bucket_count already lifted from 1 to 13)
  int *skip = h->d_shard_cursor + kMaxWorld;
  // latency-bound list walks; one reservation (a same-address atomic per destination) per 1024 list entries
  // from here on the owner-side view of the frame: the first record of a subbox (or, in the push kernel, the first voxel
  // that stays on this rank) resolves / allocates it (k_fuse's tail rearms the flags)
  F.stage_only = 0;
  F.order_mode = 1;  // stamps are complete: first-insert stamps travel in the records, activations come from the gathered keys
  F.shard_world = 1;
  F.inline_resolve = 1;
  k_shard_push<<<h->sm_count * 2, kPushThreads, 0, s>>>(X, h->P, h->D, F, par, h->d_shard_cursor, epoch);
  MLM_SMARK(4);
  // (all of the following returns at once when the wait at the head of k_shard_act_ingest found a rehash scan or an error)
  F.skip_flag = skip;
  // its CTAs spin at the head until every source has signalled: when several ranks share one GPU (tests) they must leave
  // most SMs to the other ranks' staging kernels
  k_shard_act_ingest<<<h->shard_shares_device ? 32 : h->sm_count * 8, 256, 0, s>>>(X, h->P, h->D, F, par, epoch, h->d_shard_state, skip,
                                                                                  h->shard_timeout_ns, h->D.act[F.parity]);
  MLM_SMARK(5);
  k_fuse<0><<<h->sm_count * 5, 256, 0, s>>>(h->P, h->D, F);
  MLM_SMARK(6);
#undef MLM_SMARK
  h->launches += 3;
  CUDA_TRY(cudaMemcpyAsync(h->h_shard_state, h->d_shard_state, sizeof(ShardState), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaMemcpyAsync(h->h_fc, h->D.fc[F.parity], sizeof(FrameCounters), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaGetLastError());
  h->shard_pending = true;
  return MLM_OK;
}

// a scan whose distinct hit keys (over all ranks) exceed the emulated bucket count: libstdc++ would rehash mid-frame.
// Every rank holds the full gathered (key, stamp) list, so each re-sequences it on its own (same result everywhere),
// then ingests its records with the virtual positions and fuses.  Host-driven like order_slow_path; only the first
// scans of a map take this path (the bucket array keeps its size across clear()).
int shard_rehash_path(mlm_handle h, const ShardState &st) {
  cudaStream_t s = h->stream;
  const ShardPeers &X = h->shard_peers;
  const int par = (int)(h->shard_epoch & 1);
  const int n_total = st.n_total;
  if (n_total > h->sort_cap) {
    g_last_error = "hit count exceeds ordering scratch";
    return MLM_ERR_CAPACITY;
  }
  const ShardArena &A = X.a[X.rank];
  int off = 0;
  for (int r = 0; r < X.world; r++) {
    const size_t region = ((size_t)par * X.world + r) * X.hit_cap;
    if (st.cnt_hits[r] > 0) {
      CUDA_TRY(cudaMemcpyAsync(h->d_keys_all + off, A.gather_key + region, (size_t)st.cnt_hits[r] * 4, cudaMemcpyDeviceToDevice, s));
      CUDA_TRY(cudaMemcpyAsync(h->d_stamps_all + off, A.gather_stamp + region, (size_t)st.cnt_hits[r] * 4, cudaMemcpyDeviceToDevice, s));
    }
    off += st.cnt_hits[r];
  }
  const int T = 256;
  FrameParams F = *h->h_fp;  // as the staging kernels saw it (bucket_count already lifted from 1 to 13)
  OrderArrays O;
  O.key = h->d_keys_all;
  O.stamp = h->d_stamps_all;
  O.bucket = h->d_bucket_all;
  O.kind = 0;
  uint32_t Bs = 0;
  const int rc = resequence(h, O, n_total, h->D.act[F.parity], h->act_cap, F.bucket_count, &Bs);
  if (rc != MLM_OK) return rc;
  k_shard_scatter_stamps<<<grid_for(n_total, T), T, 0, s>>>(h->d_keys_all, h->d_stamps_all, n_total, h->d_key_stamp);
  if (st.hit_base > 0) {
    k_shard_restamp<<<grid_for(st.hit_base, T), T, 0, s>>>(h->P, h->D, st.hit_base, h->d_key_stamp, Bs);
    h->launches++;
  }
  F.stage_only = 0;
  F.order_mode = 1;
  F.shard_world = 1;
  F.skip_flag = nullptr;
  F.inline_resolve = 1;
  F.bucket_count = Bs;
  F.bucket_c64 = pow64_mod(F.bucket_count);
  const int G = h->sm_count * 2;
  k_shard_ingest<<<G * 2, 256, 0, s>>>(X, h->P, h->D, F, par, h->d_shard_state, h->d_key_stamp);
  k_fuse<0><<<h->sm_count * 4, 256, 0, s>>>(h->P, h->D, F);
  h->launches += 3;
  CUDA_TRY(cudaMemcpyAsync(h->h_fc, h->D.fc[F.parity], sizeof(FrameCounters), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
}  // namespace

int mlm_shard_open(mlm_handle h, int rank, int world, void *blob_out) {
  if (!h || !blob_out || world < 1 || world > kMaxWorld || rank < 0 || rank >= world) return MLM_ERR_INVALID_ARG;
  if (h->P.explore) return MLM_ERR_UNSUPPORTED;
  if (h->shard_open) {
    g_last_error = "handle is already part of a sharded map";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const MapParams &P = h->P;
  const int hit_cap = P.max_hits;
  // records an owner can receive in a scan: one per hit key plus one per voxel with misses; a ray frees at most n_Rho
  // cells and the voxels lie inside the frame-local grid.  MLM_SHARD_REC_CAP overrides (overflow -> MLM_ERR_CAPACITY)
  const long long lvg_cells = (long long)P.lvg_dim_xy * P.lvg_dim_xy * P.lvg_dim_z;
  long long rc_ll = std::min<long long>(lvg_cells, (long long)P.max_points * P.nRho) + P.max_hits;
  if (const char *e = getenv("MLM_SHARD_REC_CAP")) rc_ll = std::max(1ll, atoll(e));
  const int rec_cap = (int)std::min<long long>(rc_ll, (1ll << 30));
  size_t bytes = 0;
  carve_arena(nullptr, world, hit_cap, rec_cap, P.max_points, &bytes);
  CUDA_TRY(cudaMalloc(&h->shard_arena, bytes));
  h->allocs.push_back(h->shard_arena);
  h->shard_arena_bytes = bytes;
  CUDA_TRY(cudaMemset(h->shard_arena, 0, align256(kMaxWorld * 4) + align256(2 * kMaxWorld * sizeof(int2)) + align256(8)));
  if (!h->D.touched_remote) {
    CUDA_TRY(cudaMalloc((void **)&h->D.touched_remote, (size_t)P.max_touched * sizeof(uint32_t)));
    h->allocs.push_back(h->D.touched_remote);
  }
  if (!h->d_key_stamp) {
    const size_t cells = (size_t)P.nZ * P.nPhi * P.nRho;
    CUDA_TRY(cudaMalloc((void **)&h->d_key_stamp, cells * sizeof(uint32_t)));
    h->allocs.push_back(h->d_key_stamp);
    // [0, kMaxWorld) push cursors, [kMaxWorld] skip flag, [+1] push ticket (k_shard_begin rearms those), [+2, +3] the
    // rank's own entry counts, [+4] ticket of the point scatter (rearmed by its last CTA)
    CUDA_TRY(cudaMalloc((void **)&h->d_shard_cursor, (kMaxWorld + 8) * sizeof(int)));
    h->allocs.push_back(h->d_shard_cursor);
    CUDA_TRY(cudaMemset(h->d_shard_cursor, 0, (kMaxWorld + 8) * sizeof(int)));
    CUDA_TRY(cudaMalloc((void **)&h->d_shard_state, sizeof(ShardState)));
    h->allocs.push_back(h->d_shard_state);
    CUDA_TRY(cudaMemset(h->d_shard_state, 0, sizeof(ShardState)));
    CUDA_TRY(cudaMallocHost((void **)&h->h_shard_state, sizeof(ShardState)));
    memset(h->h_shard_state, 0, sizeof(ShardState));
    CUDA_TRY(cudaMalloc((void **)&h->d_keys_all, (size_t)std::max(h->sort_cap, 1) * 4));
    h->allocs.push_back(h->d_keys_all);
    CUDA_TRY(cudaMalloc((void **)&h->d_stamps_all, (size_t)std::max(h->sort_cap, 1) * 4));
    h->allocs.push_back(h->d_stamps_all);
    CUDA_TRY(cudaMalloc((void **)&h->d_bucket_all, (size_t)std::max(h->sort_cap, 1) * 4));
    h->allocs.push_back(h->d_bucket_all);
  }
  if (const char *e = getenv("MLM_SHARD_TIMEOUT_MS")) h->shard_timeout_ns = (unsigned long long)std::max(1, atoi(e)) * 1000000ull;
  memset(&h->shard_peers, 0, sizeof(h->shard_peers));
  h->shard_peers.rank = rank;
  h->shard_peers.world = world;
  h->shard_peers.hit_cap = hit_cap;
  h->shard_peers.rec_cap = rec_cap;
  h->shard_peers.a[rank] = carve_arena(h->shard_arena, world, hit_cap, rec_cap, P.max_points, nullptr);
  h->shard_peers.max_points = P.max_points;
  CUDA_TRY(cudaMemset(h->shard_peers.a[rank].pflags, 0, kMaxWorld * sizeof(uint32_t)));
  h->shard_rank = rank;
  h->shard_world = world;
  h->shard_epoch = 0;
  ShardBlob b;
  memset(&b, 0, sizeof(b));
  b.magic = kShardMagic;
  b.rank = rank;
  b.world = world;
  b.device = h->device;
  b.hit_cap = hit_cap;
  b.rec_cap = rec_cap;
  b.max_points = P.max_points;
  b.pid = (int64_t)getpid();
  b.ptr = (uint64_t)(uintptr_t)h->shard_arena;
  if (world > 1) CUDA_TRY(cudaIpcGetMemHandle(&b.ipc, h->shard_arena));
  memset(blob_out, 0, MLM_SHARD_BLOB_BYTES);
  memcpy(blob_out, &b, sizeof(b));
  h->shard_open = true;
  h->shard_connected = world == 1;
  return MLM_OK;
}

int mlm_shard_connect(mlm_handle h, const void *blobs) {
  int rc = shard_check(h, false);
  if (rc != MLM_OK) return rc;
  if (!blobs) return MLM_ERR_INVALID_ARG;
  if (h->shard_connected) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  ShardPeers &X = h->shard_peers;
  for (int r = 0; r < X.world; r++) {
    ShardBlob b;
    memcpy(&b, reinterpret_cast<const unsigned char *>(blobs) + (size_t)r * MLM_SHARD_BLOB_BYTES, sizeof(b));
    if (b.magic != kShardMagic || b.rank != r || b.world != X.world || b.hit_cap != X.hit_cap || b.rec_cap != X.rec_cap ||
        b.max_points != X.max_points) {
      g_last_error = "shard blob " + std::to_string(r) + " does not describe a rank of this sharded map (same configuration on every rank?)";
      return MLM_ERR_INVALID_ARG;
    }
    if (r == X.rank) continue;
    void *base = nullptr;
    if (b.pid == (int64_t)getpid()) {
      // a handle of this process (several GPUs driven by one process, or several ranks on one GPU in the tests)
      base = reinterpret_cast<void *>((uintptr_t)b.ptr);
      if (b.device == h->device) h->shard_shares_device = true;
      if (b.device != h->device) {
        int can = 0;
        CUDA_TRY(cudaDeviceCanAccessPeer(&can, h->device, b.device));
        if (!can) {
          g_last_error = "no peer access between devices " + std::to_string(h->device) + " and " + std::to_string(b.device);
          return MLM_ERR_UNSUPPORTED;
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CUDA_TRY(e);
        cudaGetLastError();
      }
    } else {
      CUDA_TRY(cudaIpcOpenMemHandle(&base, b.ipc, cudaIpcMemLazyEnablePeerAccess));
      h->shard_mapped[r] = base;
    }
    X.a[r] = carve_arena(base, X.world, X.hit_cap, X.rec_cap, X.max_points, nullptr);
  }
  h->shard_connected = true;
  return MLM_OK;
}

int mlm_shard_close(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!h->shard_open) return MLM_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (int r = 0; r < kMaxWorld; r++)
    if (h->shard_mapped[r]) {
      cudaIpcCloseMemHandle(h->shard_mapped[r]);
      h->shard_mapped[r] = nullptr;
    }
  cudaGetLastError();
  h->shard_connected = false;  // the arena itself is released by mlm_destroy (peers must have closed by then)
  return MLM_OK;
}

int mlm_shard_submit_points_f64_device(mlm_handle h, const double *d_xyz, int n, const double T_wb[7]) {
  int rc = shard_check(h, true);
  if (rc != MLM_OK) return rc;
  if ((!d_xyz && n > 0) || !T_wb || n < 0) return MLM_ERR_INVALID_ARG;
  if (n > h->P.max_points) return MLM_ERR_CAPACITY;
  if (h->shard_pending) {
    g_last_error = "mlm_shard_finish of the previous scan is missing";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  return shard_enqueue(h, d_xyz, n, T_wb);
}

int mlm_shard_submit_points_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7]) {
  int rc = shard_check(h, true);
  if (rc != MLM_OK) return rc;
  if ((!xyz && n > 0) || !T_wb || n < 0) return MLM_ERR_INVALID_ARG;
  if (n > h->P.max_points) return MLM_ERR_CAPACITY;
  if (h->shard_pending) {
    g_last_error = "mlm_shard_finish of the previous scan is missing";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t bytes = (size_t)std::max(n, 1) * 24;
  rc = ensure_input(h, bytes, (size_t)h->P.max_points * 24);
  if (rc != MLM_OK) return rc;
  const void *src = nullptr;
  if (n > 0) {
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, xyz) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    src = xyz;
    if (!pinned) {
      memcpy(h->h_stage, xyz, (size_t)n * 24);
      src = h->h_stage;
    }
  }
  return shard_enqueue(h, reinterpret_cast<const double *>(h->d_input), n, T_wb, src);
}

// every rank passes ITS slice [first, first + n_slice) of the same scan of n_total points (the slices partition the
// scan): 1/world of the H2D traffic per rank, the slices reach the other ranks over NVLink peer memory
int mlm_shard_submit_points_slice_f64(mlm_handle h, const double *xyz_slice, int first, int n_slice, int n_total, const double T_wb[7]) {
  int rc = shard_check(h, true);
  if (rc != MLM_OK) return rc;
  if ((!xyz_slice && n_slice > 0) || !T_wb || first < 0 || n_slice < 0 || n_total < 0 || (long long)first + n_slice > n_total) return MLM_ERR_INVALID_ARG;
  if (n_total > h->P.max_points) return MLM_ERR_CAPACITY;
  if (h->shard_pending) {
    g_last_error = "mlm_shard_finish of the previous scan is missing";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t s = h->stream;
  const ShardPeers &X = h->shard_peers;
  const uint32_t epoch = h->shard_epoch + 1;   // shard_enqueue advances it
  const int par = (int)(epoch & 1);
  double *mine = X.a[X.rank].points + (size_t)par * 3 * X.max_points;
  if (n_slice > 0) {
    const void *src = xyz_slice;
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, xyz_slice) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (!pinned) {
      rc = ensure_input(h, (size_t)n_slice * 24, (size_t)h->P.max_points * 24);   // (allocates the pinned staging buffer too)
      if (rc != MLM_OK) return rc;
      memcpy(h->h_stage, xyz_slice, (size_t)n_slice * 24);
      src = h->h_stage;
    }
    CUDA_TRY(cudaMemcpyAsync(mine + 3 * (size_t)first, src, (size_t)n_slice * 24, cudaMemcpyHostToDevice, s));
  }
  if (X.world > 1) {
    const int g = std::max(1, std::min(h->sm_count * 2, (int)((3ll * n_slice + 255) / 256)));
    k_shard_scatter_points<<<g, 256, 0, s>>>(X, par, first, n_slice, epoch, h->d_shard_cursor + kMaxWorld + 4);
    k_shard_wait_points<<<1, 32, 0, s>>>(X, epoch, h->shard_timeout_ns, h->D.fc[h->frame_idx & 1]);
    h->launches += 2;
  }
  return shard_enqueue(h, mine, n_total, T_wb);
}

int mlm_shard_finish(mlm_handle h, mlm_frame_stats *stats) {
  int rc = shard_check(h, true);
  if (rc != MLM_OK) return rc;
  if (!h->shard_pending) {
    g_last_error = "no submitted scan";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  h->shard_pending = false;
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  if (h->profiling && h->sev[0])
    for (int i = 0; i < MLM_NUM_SHARD_KERNELS; i++) cudaEventElapsedTime(&h->skms[i], h->sev[i], h->sev[i + 1]);
  const ShardState st = *h->h_shard_state;
  if (st.error) {
    g_last_error = st.error == kErrPeer ? "sharded scan: a peer rank failed or did not signal within the timeout"
                                        : "device raised error code " + std::to_string(st.error);
    return st.error == kErrPeer ? MLM_ERR_CUDA : map_device_error(st.error);
  }
  const uint32_t B = bucket_growth(h->bucket_count, st.n_total);
  if (st.rehash) {
    rc = shard_rehash_path(h, st);
    if (rc != MLM_OK) return rc;
  }
  rc = finish_frame(h, st.rehash, B, stats);
  h->bucket_count = B;  // finish_frame grows it from the LOCAL record count; the gathered count decides
  h->last_order_B = B;
  if (stats) {
    stats->n_hit_cells = st.n_total;  // distinct hit keys of the whole scan (identical on every rank)
    stats->hit_bucket_count = (int32_t)B;
  }
  return rc;
}

int mlm_shard_integrate_points_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7], mlm_frame_stats *stats) {
  int rc = mlm_shard_submit_points_f64(h, xyz, n, T_wb);
  if (rc != MLM_OK) return rc;
  return mlm_shard_finish(h, stats);
}

int mlm_shard_last_kernel_ms(mlm_handle h, float ms[MLM_NUM_SHARD_KERNELS]) {
  if (!h || !ms) return MLM_ERR_INVALID_ARG;
  for (int i = 0; i < MLM_NUM_SHARD_KERNELS; i++) ms[i] = h->skms[i];
  return MLM_OK;
}

int mlm_shard_last_exchange(mlm_handle h, mlm_shard_exchange *out) {
  if (!h || !out || !h->h_shard_state) return MLM_ERR_INVALID_ARG;
  const ShardState &st = *h->h_shard_state;
  memset(out, 0, sizeof(*out));
  out->n_hit_total = st.n_total;
  out->n_hit_local = st.cnt_hits[h->shard_rank];
  out->records_received = st.n_rec_total;
  out->records_from_self = -1;  // not tracked: sources reserve straight in the owner's inbox
  out->rehash_path = st.rehash;
  out->wait_ns = (int64_t)st.wait_ns;
  out->world = h->shard_world;
  out->arena_bytes = (int64_t)h->shard_arena_bytes;
  return MLM_OK;
}

// ---- replicated map: ship the subbox blocks touched by the last frame --------------------------------------
int mlm_dirty_count(mlm_handle h, int32_t *n_blocks, size_t *record_bytes) {
  if (!h || !n_blocks || !record_bytes) return MLM_ERR_INVALID_ARG;
  if (h->P.explore) {
    g_last_error = "mlm_dirty_count: dirty-block shipping does not carry frontier sets or collapses (exploration mode)";
    return MLM_ERR_UNSUPPORTED;
  }
  *n_blocks = h->h_fc->n_touched_sub;
  *record_bytes = dirty_record_bytes(h->P.cells);
  return MLM_OK;
}
int mlm_dirty_export(mlm_handle h, void *d_out, int32_t n_blocks) {
  if (!h || (n_blocks && !d_out) || n_blocks < 0 || n_blocks > h->h_fc->n_touched_sub) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (n_blocks) k_dirty_export<<<n_blocks, 256, 0, h->stream>>>(h->P, h->D, *h->h_fp, n_blocks, (unsigned char *)d_out);
  h->launches++;
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}
int mlm_dirty_import(mlm_handle h, const void *d_in, int32_t n_blocks) {
  if (!h || (n_blocks && !d_in) || n_blocks < 0) return MLM_ERR_INVALID_ARG;
  CUDA_TRY(cudaSetDevice(h->device));
  if (h->P.explore) return MLM_ERR_UNSUPPORTED;
  cudaStream_t s = h->stream;
  int cnt[2] = {0, 0};
  {
    StreamTemp<int> d_cnt(s);
    CUDA_TRY(d_cnt.alloc(2));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(int), s));
    if (n_blocks) k_dirty_import<<<n_blocks, 256, 0, s>>>(h->P, h->D, n_blocks, (const unsigned char *)d_in, d_cnt);
    h->launches++;
    CUDA_TRY(cudaMemcpyAsync(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  h->cum_ram_expand += cnt[0];
  h->n_submaps += cnt[0];
  return cnt[1] ? map_device_error(cnt[1]) : MLM_OK;
}

// ---- replicated map over NVLink peer memory (SURVEY 8e, query streams split over GPUs) -------------------------------
namespace {
constexpr uint32_t kReplicaMagic = 0x4d4c5250u;  // "MLRP"
ReplicaArena carve_replica(void *base, size_t half_bytes, size_t *total) {
  unsigned char *p = reinterpret_cast<unsigned char *>(base);
  size_t off = 0;
  ReplicaArena a;
  a.flags = reinterpret_cast<uint32_t *>(p + off);
  off = align256(off + 2 * sizeof(uint32_t));
  a.count = reinterpret_cast<int *>(p + off);
  off = align256(off + 2 * sizeof(int));
  a.ack = reinterpret_cast<uint32_t *>(p + off);
  off = align256(off + kMaxWorld * sizeof(uint32_t));
  a.inbox = p + off;
  off = align256(off + 2 * half_bytes);
  if (total) *total = off;
  return a;
}
int replica_check(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!h->replica_open || !h->replica_connected) {
    g_last_error = "mlm_replica_open / mlm_replica_connect must come first";
    return MLM_ERR_INVALID_ARG;
  }
  return MLM_OK;
}
}  // namespace

int mlm_replica_open(mlm_handle h, int rank, int world, int src, void *blob_out) {
  if (!h || !blob_out || world < 1 || world > kMaxWorld || rank < 0 || rank >= world || src < 0 || src >= world) return MLM_ERR_INVALID_ARG;
  if (h->P.explore) return MLM_ERR_UNSUPPORTED;
  if (h->replica_open) {
    g_last_error = "handle is already part of a replicated map";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const MapParams &P = h->P;
  // dirty blocks of one frame: at most the subboxes of the frame-local subbox grid (MLM_REPLICA_MAX_BLOCKS overrides)
  long long cap = std::min<long long>((long long)P.lsg_dim_xy * P.lsg_dim_xy * P.lsg_dim_z, 32768);
  if (const char *e = getenv("MLM_REPLICA_MAX_BLOCKS")) cap = std::max(1ll, atoll(e));
  const size_t half = (size_t)cap * dirty_record_bytes(P.cells);
  size_t bytes = 0;
  carve_replica(nullptr, half, &bytes);
  CUDA_TRY(cudaMalloc(&h->replica_arena, bytes));
  h->allocs.push_back(h->replica_arena);
  CUDA_TRY(cudaMemset(h->replica_arena, 0, 3 * 256));
  CUDA_TRY(cudaMalloc((void **)&h->d_replica_state, 4 * sizeof(int)));
  h->allocs.push_back(h->d_replica_state);
  CUDA_TRY(cudaMemset(h->d_replica_state, 0, 4 * sizeof(int)));
  if (const char *e = getenv("MLM_SHARD_TIMEOUT_MS")) h->shard_timeout_ns = (unsigned long long)std::max(1, atoi(e)) * 1000000ull;
  ReplicaPeers &X = h->replica_peers;
  memset(&X, 0, sizeof(X));
  X.rank = rank;
  X.world = world;
  X.src = src;
  X.cap_blocks = (int)cap;
  X.half_bytes = half;
  X.a[rank] = carve_replica(h->replica_arena, half, nullptr);
  h->replica_epoch = 0;
  ShardBlob b;
  memset(&b, 0, sizeof(b));
  b.magic = kReplicaMagic;
  b.rank = rank;
  b.world = world;
  b.device = h->device;
  b.hit_cap = src;
  b.rec_cap = (int)cap;
  b.pid = (int64_t)getpid();
  b.ptr = (uint64_t)(uintptr_t)h->replica_arena;
  if (world > 1) CUDA_TRY(cudaIpcGetMemHandle(&b.ipc, h->replica_arena));
  memset(blob_out, 0, MLM_SHARD_BLOB_BYTES);
  memcpy(blob_out, &b, sizeof(b));
  h->replica_open = true;
  h->replica_connected = world == 1;
  return MLM_OK;
}

int mlm_replica_connect(mlm_handle h, const void *blobs) {
  if (!h || !blobs) return MLM_ERR_INVALID_ARG;
  if (!h->replica_open) {
    g_last_error = "mlm_replica_open must come first";
    return MLM_ERR_INVALID_ARG;
  }
  if (h->replica_connected) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  ReplicaPeers &X = h->replica_peers;
  for (int r = 0; r < X.world; r++) {
    ShardBlob b;
    memcpy(&b, reinterpret_cast<const unsigned char *>(blobs) + (size_t)r * MLM_SHARD_BLOB_BYTES, sizeof(b));
    if (b.magic != kReplicaMagic || b.rank != r || b.world != X.world || b.hit_cap != X.src || b.rec_cap != X.cap_blocks) {
      g_last_error = "replica blob " + std::to_string(r) + " does not describe a rank of this replicated map (same configuration on every rank?)";
      return MLM_ERR_INVALID_ARG;
    }
    if (r == X.rank) continue;
    // the source stores into every replica; a replica only into the source (its acknowledgements)
    if (X.rank != X.src && r != X.src) continue;
    void *base = nullptr;
    if (b.pid == (int64_t)getpid()) {
      base = reinterpret_cast<void *>((uintptr_t)b.ptr);
      if (b.device != h->device) {
        int can = 0;
        CUDA_TRY(cudaDeviceCanAccessPeer(&can, h->device, b.device));
        if (!can) {
          g_last_error = "no peer access between devices " + std::to_string(h->device) + " and " + std::to_string(b.device);
          return MLM_ERR_UNSUPPORTED;
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CUDA_TRY(e);
        cudaGetLastError();
      }
    } else {
      CUDA_TRY(cudaIpcOpenMemHandle(&base, b.ipc, cudaIpcMemLazyEnablePeerAccess));
      h->replica_mapped[r] = base;
    }
    X.a[r] = carve_replica(base, X.half_bytes, nullptr);
  }
  h->replica_connected = true;
  return MLM_OK;
}

int mlm_replica_publish(mlm_handle h, int32_t *n_blocks_out) {
  int rc = replica_check(h);
  if (rc != MLM_OK) return rc;
  ReplicaPeers &X = h->replica_peers;
  if (X.rank != X.src) {
    g_last_error = "only the source rank publishes";
    return MLM_ERR_INVALID_ARG;
  }
  if (h->frame_pending || h->staged) {
    g_last_error = "the frame whose blocks are to be published is not complete (mlm_frame_finish / mlm_local_input_pc_pose_direct first)";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const int n = h->h_fc->n_touched_sub;
  if (n > X.cap_blocks) {
    g_last_error = "frame touched more subboxes than the replicas' inboxes hold (MLM_REPLICA_MAX_BLOCKS)";
    return MLM_ERR_CAPACITY;
  }
  const uint32_t epoch = ++h->replica_epoch;
  cudaStream_t s = h->stream;
  k_replica_push<<<std::max(n, 1), 256, 0, s>>>(X, h->P, h->D, *h->h_fp, n, epoch, h->d_replica_state, h->shard_timeout_ns);
  h->launches++;
  int st[2] = {0, 0};
  CUDA_TRY(cudaMemcpyAsync(st, h->d_replica_state, sizeof(st), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  h->replica_last_blocks = n;
  if (n_blocks_out) *n_blocks_out = n;
  if (st[1]) {
    g_last_error = "a replica did not acknowledge an earlier frame in time (MLM_SHARD_TIMEOUT_MS)";
    return MLM_ERR_CUDA;
  }
  return MLM_OK;
}

int mlm_replica_apply(mlm_handle h, int32_t *n_blocks_out) {
  int rc = replica_check(h);
  if (rc != MLM_OK) return rc;
  ReplicaPeers &X = h->replica_peers;
  if (X.rank == X.src) {
    g_last_error = "the source rank has nothing to apply";
    return MLM_ERR_INVALID_ARG;
  }
  CUDA_TRY(cudaSetDevice(h->device));
  const uint32_t epoch = ++h->replica_epoch;
  cudaStream_t s = h->stream;
  CUDA_TRY(cudaMemsetAsync(h->d_replica_state, 0, 4 * sizeof(int), s));
  k_replica_pull<<<h->sm_count * 2, 256, 0, s>>>(X, h->P, h->D, epoch, h->d_replica_state, h->shard_timeout_ns);
  h->launches++;
  int cnt[4] = {0, 0, 0, 0};
  CUDA_TRY(cudaMemcpyAsync(cnt, h->d_replica_state, sizeof(cnt), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  CUDA_TRY(cudaGetLastError());
  h->cum_ram_expand += cnt[0];
  h->n_submaps += cnt[0];
  h->replica_last_blocks = cnt[3];
  if (n_blocks_out) *n_blocks_out = cnt[3];
  if (cnt[1] == kErrPeer) {
    g_last_error = "the source did not publish the frame in time (MLM_SHARD_TIMEOUT_MS) or reported a failure";
    return MLM_ERR_CUDA;
  }
  return cnt[1] ? map_device_error(cnt[1]) : MLM_OK;
}

int mlm_replica_close(mlm_handle h) {
  if (!h) return MLM_ERR_INVALID_ARG;
  if (!h->replica_open) return MLM_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (int r = 0; r < kMaxWorld; r++)
    if (h->replica_mapped[r]) {
      cudaIpcCloseMemHandle(h->replica_mapped[r]);
      h->replica_mapped[r] = nullptr;
    }
  cudaGetLastError();
  h->replica_connected = false;  // the arena itself is released by mlm_destroy (peers must have closed by then)
  return MLM_OK;
}

int mlm_debug_log10f(mlm_handle h, const float *x, size_t n, float *out) {
  if (!h || (!x && n) || (!out && n)) return MLM_ERR_INVALID_ARG;
  if (n == 0) return MLM_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  {
    StreamTemp<float> d_buf(h->stream);  // x, out
    CUDA_TRY(d_buf.alloc(n * 2));
    CUDA_TRY(cudaMemcpyAsync(d_buf, x, n * 4, cudaMemcpyHostToDevice, h->stream));
    k_debug_log10f<<<grid_for(n, 256), 256, 0, h->stream>>>(d_buf, n, d_buf + n, h->P.log10f_fma);
    h->launches++;
    CUDA_TRY(cudaMemcpyAsync(out, d_buf + n, n * 4, cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaGetLastError());
  return MLM_OK;
}

}  // extern "C"
