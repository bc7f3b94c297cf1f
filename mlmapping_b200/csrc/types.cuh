// Device-visible state of one map handle.  Names follow the reference's domain:
// awareness cells (rho,phi,z), subboxes/submaps, cells, log-odds, hit map / miss set.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mlm {

constexpr int kDiffRange = 10;          // awareness_map_cylindrical::diff_range (map_awareness.cpp:36)
constexpr int kOddsRows = 2 * kDiffRange + 1;
constexpr int kMaxPhi = 4096;           // upper bound on nPhi for the shared-memory histogram
constexpr uint64_t kEmptyKey = ~0ull;   // empty slot of the submap hash table
constexpr int kBlockPending = -1;
constexpr int kBlockCollapsed = -2;     // ht_val of a subbox collapsed by the release pass (map_local.cpp:208-232)
constexpr int kBlockUnusable = -3;      // pool exhausted when the subbox was created
constexpr int kLvgEmpty = -1;
constexpr int kLvgClaimed = -2;
// device-raised error codes (mapped to MLM_ERR_* by the host)
constexpr int kErrRange = 1, kErrPool = 4, kErrCapacity = 5, kErrInternal = 100;
constexpr uint32_t kTouchedHitTag = 0x80000000u;

// record of one castable point after projection (K1 output)
struct __align__(16) RayRecord {
  int rho;        // rho_idx as the reference computes it (may be >= nRho)
  int z;          // z_idx (may be out of range)
  uint32_t phi_flags;  // phi_idx | run length << 16 | inside << 30
  uint32_t t;     // point order stamp = index of the point in input_pc_pose's loop
};
constexpr uint32_t kRecInside = 1u << 30;
constexpr uint32_t kRecPhiMask = (1u << 16) - 1;
constexpr int kRecCountShift = 16;          // run length (1..32) of identical consecutive points
constexpr uint32_t kRecCountMask = 0x3f;

// constants of a handle (mlmap::init_map), immutable after mlm_create
struct MapParams {
  // awareness_map_cylindrical members (include/map_awareness.h:16-30,61-65)
  double dRho, dPhi, dZ, z_border_min;
  int nRho, nPhi, nZ, n_below;
  int visibility_check;
  int maxK;               // max over rho of the neighbour reach K(rho)
  int words_per_row;      // ceil(nRho / 32): bitmap words per (phi,z) row
  int col_words;          // nZ * words_per_row
  int cell_bits;          // bits of a cell id inside a column: ceil(log2(nZ*nRho))
  int split;              // 1: every phi column is worked as two half columns (records below / at-or-above the sensor row n_below)
  int unused0;            // unused: holds the offsets below, without it k_view_tiles (frontier targets) measured ~0.3% slower
  int nCol;               // work columns of k_column: nPhi * (split ? 2 : 1)
  uint32_t nRho_magic;    // ceil(2^32 / nRho): cell / nRho by multiply-high (cells < 2^20, nRho < 2^12)
  // local_map_cartesian members (include/map_local.h:66-78)
  double d_sub, d_glb, d_sub_half;
  double inv_d_sub, inv_d_glb, inv_dRho, inv_dPhi, inv_dZ;  // fl(1/d): fast path of floor_quot_exact only
  int n;                  // subbox_nxyz
  int cells;              // cell_num_subbox
  int cell_stride;        // cells rounded up to 16: per-block stride of the pool arrays
  float lo_min, lo_max, lo_miss, lo_sh;
  int explore;            // apply_explored_area (use_exploration_frontiers)
  int front_words;        // 32-bit words of a subbox's frontier bitmask: ceil(cells/32)
  double bd[6];           // global_bd = {-30,30,-30,30,0,5} (src/map_local.cpp:124)
  // camera (include/mlmap.h:85-86,92)
  float cx, cy, fx, fy;
  double inv_factor;
  double inv_fx, inv_fy;  // fl(1/fx), fl(1/fy): approximate projection of the guarded fast path only
  float fast_inv_dRho, fast_inv_dZ, fast_deg2cell;  // float scale factors of the guarded fast path (cells per metre / per degree)
  int log10f_fma;         // which glibc __logf variant the host CPU dispatches to
  // local voxel grid (frame-local staging) geometry
  int lvg_dim_xy, lvg_dim_z;   // cells per axis
  int lvg_margin;              // cells between awareness bounding box and grid border
  int lsg_dim_xy, lsg_dim_z;   // local submap grid dims
  // division by the grid dimensions / subbox size by multiply-high (x / d == umulhi(x, mul) >> shift for x < 2^31; mul 0: d == 1)
  uint32_t dxy_mul, dxy2_mul, n_mul;
  int dxy_shift, dxy2_shift, n_shift;
  // capacities
  int max_points;
  int max_hits;           // capacity of the per-frame hit list
  int max_touched;
  int pool_blocks;
  uint32_t ht_mask;       // hash table capacity - 1 (power of two)
  int sort_cap_smem;      // 64-bit keys the column kernel can sort in shared memory
  int map_cap;            // records per column addressed through the shared-memory index map (<= kMapCap)
  int contrib_per_point;  // 1 + 2*maxK
  // tables (device pointers)
  const float *odds_table;    // [21][nRho]   get_odds_table (map_awareness.cpp:36-46)
  const int *k_reach;         // [nRho]       number of diff_r >= 1 with diff_r < 3*sigma_in_dr(rho)
  const double2 *centre_xy;   // [nPhi*nRho]  cell centre x,y (map_awareness.cpp:58-61)
  const double *centre_z;     // [nZ]
  const double *rate_table;   // [nZ*nRho]    raycasting_z_over_rho of cell (z,rho) (map_awareness.cpp:64-71)
  const short2 *dz_table;     // [nZ*nRho*maxK] z row of the d-th outer / inner neighbour of an end cell (update_hits :151,:161), -1 = outside
};

// values that change every frame; lives in device memory so a captured graph can be replayed
struct FrameParams {
  double q_ls[4];   // T_ls rotation (w,x,y,z)
  double t_ls[3];   // T_ls translation
  double t_wa[3];   // T_wa translation (= t_wb)
  const void *input; // device pointer: uint16 depth image (rows*cols) or xyz doubles (n_points*3)
  int rows, cols;
  uint32_t cols_magic;  // pixel index / cols == umulhi(index, cols_magic) >> cols_shift for index < 2^31
  int cols_shift;
  int n_points;     // point-cloud input
  int n_total;      // rows*cols or n_points: number of input slots this frame
  uint32_t bucket_count;  // emulated hit_idx_odds_hashmap.bucket_count() at frame start
  uint32_t bucket_c64;    // 2^64 mod bucket_count: libstdc++'s bucket of a NEGATIVE int hash (sign-extended to size_t) without a 64-bit modulo
  int lvg_base[3];  // global cell coordinate of local voxel grid origin
  int lsg_base[3];  // global subbox coordinate of local submap grid origin
  int tbits;        // bits needed for a point stamp this frame (ceil(log2(#points)))
  int tile_pts;     // points per projection tile (multiple of 32, <= 128 per warp of the projecting CTA) = slots of its rec_lin window
  uint32_t bucket_count_miss;  // emulated miss_idx_set.bucket_count() at frame start (exploration mode)
  int shard_rank, shard_world;  // sharded staging: this rank casts the columns phi % world == rank
  int stage_only;   // 1: k_column stages into the voxel grid only (no subbox resolve; records go to the owners)
  int inline_resolve; // 1 (k_frame): the first thread to touch a subbox resolves / allocates it right away
  int parity;       // frame & 1: selects the double-buffered counters / activation stamps
  int order_mode;   // 0: stamps are (bucket activation, first-insert time); 1: virtual sequence positions
  uint32_t frame_seq;        // published to the host counters last: the host may poll it instead of waiting for the stream
  const int *skip_flag;  // sharded scans: when non-null and *skip_flag != 0 the owner-side kernels (resolve, fuse) return at
                         // once; set on device when the gathered hit count calls for the rehash path (the host re-launches)
};

// per-frame counters + error word, reset by k_frame_begin
struct FrameCounters {
  int n_points, n_inside, n_cast;
  int n_hit, n_miss;
  int n_touched, n_touched_sub, n_new_blocks;
  int n_touched_voxels;   // distinct voxels actually fused
  int error;              // MLM_ERR_* raised on device
  int overflow;           // 1: n_hit > bucket_count -> fuse skipped, slow ordering path needed
  int obs_delta;          // occupancy 'o' transitions this frame
  int fused;              // set by k_fuse when it ran to completion
  int n_miss_list;        // exploration mode: entries of the per-frame miss list
  int n_obs;              // exploration mode: subboxes handed to the release pass (observed_subboxes)
  int n_released;         // subboxes collapsed by the release pass this frame
  int n_touched_remote;   // sharded staging: entries of the list of voxels owned by OTHER ranks
  uint32_t seq;           // host copy only: frame_seq of the frame these counters belong to, stored after everything else
};

struct DeviceBuffers {
  FrameCounters *host_fc;  // mapped pinned host memory: the last k_fuse block publishes the frame counters here
  int *fuse_ticket;        // completion ticket of k_fuse
  FrameCounters *fc[2];   // double-buffered: frame f uses fc[f&1], k_fuse clears the other one
  // K1/K1b
  RayRecord *rec_lin;     // [max_points] per projection tile: a tile_pts-slot window, records grouped by column
  uint32_t *rec_dir;      // [tiles][nCol] directory of those windows: offset << 16 | count
  RayRecord *rec_col;     // [max_points] gathered by k_column: contiguous per phi column
  int *phi_hist;          // [nCol] records per work column
  int *phi_bound;         // [nCol] upper bound of hit contributions per work column
  uint64_t *col_scratch;  // [max_points*contrib_per_point] sort spill for oversized columns
  // per-frame hit map / miss set
  int *hit_key;           // [max_hits] awareness linear index (mapIdx)
  float *hit_p;           // [max_hits]
  uint32_t *hit_t;        // [max_hits] first-insert stamp (t*32+substep) or virtual position
  int *hit_next;          // [max_hits] next hit in the same voxel's list
  uint32_t *hit_bucket;   // [max_hits] libstdc++ bucket of the key at this frame's bucket count
  uint32_t *miss_bitmap;  // [nPhi*col_words]
  uint32_t *act[2];       // [bucket capacity] bucket activation stamps, double-buffered like fc
  int *col_ticket;        // completion ticket of k_column (last CTA resolves the touched subboxes)
  int *col_queue;         // next item of k_column's work queue (rearmed by the last CTA)
  int *grid_bar;          // arrival counter of k_frame's device-wide barriers (rearmed by the last CTA)
  // local voxel / submap grids
  int2 *lvg;              // [lvg cells] .x head of this frame's hit list (-1 empty), .y number of miss cells
  uint32_t *touched;      // [max_touched] local voxel index (| kTouchedHitTag)
  uint32_t *touched_remote; // [max_touched] sharded maps only: the same for voxels whose subbox another rank owns
  int *lsg_flag;          // [lsg cells]
  int *lsg_block;         // [lsg cells] pool block of that subbox this frame
  int *touched_sub;       // [lsg cells]
  // submap pool + spatial hash
  uint64_t *ht_key;       // [ht cap]
  int *ht_val;            // [ht cap] pool block index
  int *free_stack;        // [pool_blocks]
  int *free_top;          // scalar: number of free blocks on the stack
  float *pool_lo;         // [pool_blocks*cells]
  char *pool_occ;         // [pool_blocks*cells]
  char *pool_inf;         // [pool_blocks*cells]
  int64_t *cum;           // [0]=ram_expand_cnt [1]=obs_cnt [2]=n_submaps
  // ---- exploration-frontier mode (use_exploration_frontiers), allocated only when enabled ----
  uint32_t *pool_front;   // [pool_blocks*front_words] frontier set of every subbox as a bitmask
  char *col_occ, *col_inf; // [ht cap] element 0 of a collapsed subbox, by hash slot
  float *col_lo;          // [ht cap]
  uint32_t *end_t;        // [nPhi*nZ*nRho] earliest point stamp per inside end cell
  uint32_t *miss_stamp;   // [nPhi*nZ*nRho] first-insert stamp of every miss cell (t*nRho + step)
  uint32_t *act_miss[2];  // [bucket capacity] bucket activation stamps of miss_idx_set
  int *miss_idx;          // [cells] per-frame miss list: awareness cell index
  int *miss_lv;           // [cells]   its local voxel
  uint32_t *miss_t;       // [cells]   its first-insert stamp (or virtual position)
  uint32_t *miss_bucket;  // [cells]   its libstdc++ bucket
  signed char *miss_choice; // [cells] neighbour picked by update_observation (-1 none)
  unsigned long long *lvg_tkey; // [lvg cells] (bucket activation, stamp) of the voxel's first miss cell in iteration order
  int *obs_flag;          // [lsg cells]
  int *obs_list;          // [lsg cells]
  long long *debug_cycles; // [nPhi*16] per-column phase clocks (MLM_PHASE_TIMING builds only)
};

}  // namespace mlm
