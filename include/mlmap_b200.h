/*
 * mlmap_b200.h — C ABI of the B200-native MLMapping hot path (the drop-in boundary).
 *
 * The reference has no FFI layer: its boundary is the C++ class `mlmap`
 * (reference include/mlmap.h:105-139).  A maintainer binds these entry points
 * from that class (see INTEGRATION.md); every function below cites the
 * reference method it replaces.  Plain pointers and sizes only; no C++/torch
 * types cross this boundary; nothing throws.
 *
 * Threading contract (SURVEY §8b): one handle owns one CUDA stream.  Calls on a
 * handle are stream-ordered and must be externally serialised; distinct handles
 * are independent.  Queries observe every previously submitted update.
 *
 * Pose layout everywhere: double[7] = { tx, ty, tz, qw, qx, qy, qz }.  The
 * quaternion is normalised on entry exactly as Sophus::SO3(Quaterniond) does
 * (reference 3rdPartLib/Sophus/sophus/so3.cpp:42-47).
 */
#ifndef MLMAP_B200_H
#define MLMAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define MLM_ABI_VERSION 1

/* status codes returned by every entry point */
enum {
  MLM_OK = 0,
  MLM_ERR_INVALID_ARG = 1,    /* null pointer, bad size, bad handle */
  MLM_ERR_INVALID_CONFIG = 2, /* violates a precondition of the reference's tables (SURVEY §8a a3) */
  MLM_ERR_CUDA = 3,           /* a CUDA runtime call failed; see mlm_last_error() */
  MLM_ERR_POOL_EXHAUSTED = 4, /* submap pool or hash table full */
  MLM_ERR_CAPACITY = 5,       /* more points/records in one frame than the handle was sized for */
  MLM_ERR_UNSUPPORTED = 6,    /* option not implemented on the GPU path (never a silent CPU fallback) */
  MLM_ERR_NO_DEVICE = 7       /* no CUDA device / wrong architecture */
};

/* occupancy codes, reference include/mlmap.h:109-114 */
enum { MLM_FREE = 1, MLM_OCCUPIED = 0, MLM_UNKNOWN = -1 };

/*
 * Configuration = the YAML keys mlmap::init_map reads (reference src/mlmap.cpp:10-33,37-53,75-85)
 * as a plain struct (yamlRead.h is out of scope).
 */
typedef struct mlm_config {
  /* awareness_map_cylindrical::init_map arguments (reference src/map_awareness.cpp:19) */
  double am_d_rho;      /* mlmapping_am_d_Rho      */
  double am_d_phi_deg;  /* mlmapping_am_d_Phi_deg  */
  double am_d_z;        /* mlmapping_am_d_Z        */
  int32_t am_n_rho;     /* mlmapping_am_n_Rho      */
  int32_t am_n_z_below; /* mlmapping_am_n_Z_below  */
  int32_t am_n_z_over;  /* mlmapping_am_n_Z_over   */
  int32_t use_raycasting; /* mlmapping_use_raycasting */
  int32_t _pad0;
  double depth_noise_coe; /* mlmapping_depth_noise_coe */

  /* local_map_cartesian::init_map arguments (reference src/map_local.cpp:46-53) */
  double subbox_d_xyz;  /* mlmapping_subbox_d_xyz */
  int32_t subbox_n;     /* mlmapping_subbox_n     */
  float log_odds_min;   /* mlmapping_lm_log_odds_min */
  float log_odds_max;   /* mlmapping_lm_log_odds_max */
  float log_odds_hit;   /* mlmapping_lm_measurement_hit (read, stored, never used: map_local.cpp:128) */
  float log_odds_miss;  /* mlmapping_lm_measurement_miss */
  float log_odds_occupied_sh; /* mlmapping_lm_occupied_sh */
  int32_t use_exploration_frontiers; /* use_exploration_frontiers */
  int32_t _pad1;

  /* camera intrinsics, float members in the reference (include/mlmap.h:92) */
  float cam_cx, cam_cy, cam_fx, cam_fy;

  /* T_B_S (sensor in body) as pose[7]; reference src/mlmap.cpp:22-25 */
  double T_bs[7];

  /* inflation layer (reference src/mlmap.cpp:10,84-85; include/map_local.h:63-65) */
  int32_t inflate_n;
  int32_t inflate_global_n;
  int32_t apply_inflate;
  int32_t _pad2;
  double inflate_height; /* local_map_cartesian::flate_height, default 0.1 */

  /* project_depth: 0 = full-frame mode (every non-zero pixel, row-major);
   * >0 = mlmapping_sample_cnt random pixels via glibc rand() (reference src/mlmap.cpp:321-326) */
  int32_t sample_cnt;

  /* capacities of the GPU-resident structures (no reference equivalent: the reference mallocs) */
  int32_t max_points;     /* max points (pixels) per frame */
  int32_t pool_submaps;   /* capacity of the submap block pool */
  int32_t _pad3;
} mlm_config;

typedef struct mlm_map *mlm_handle;

/* per-frame counters (reference public counters ram_expand_cnt/obs_cnt, include/map_local.h:79-80) */
typedef struct mlm_frame_stats {
  int32_t n_points;        /* points fed to input_pc_pose */
  int32_t n_inside;        /* points inside the awareness range (update_hits calls) */
  int32_t n_cast;          /* rays cast (can_do_cast && visibility_check) */
  int32_t n_hit_cells;     /* distinct keys of hit_idx_odds_hashmap */
  int32_t n_miss_cells;    /* distinct entries of miss_idx_set */
  int32_t n_touched_voxels;/* distinct local-map cells receiving any update */
  int32_t n_new_submaps;   /* allocate_ram() insertions this frame */
  int32_t hit_bucket_count;/* emulated libstdc++ bucket count of the hit map after this frame */
  int32_t ordering_slow_path; /* 1 if the frame crossed a libstdc++ rehash (SURVEY Appendix B) */
  int32_t status;          /* MLM_OK or the error raised on device */
  int64_t ram_expand_cnt;  /* cumulative */
  int64_t obs_cnt;         /* cumulative */
} mlm_frame_stats;

/* ---- lifetime ------------------------------------------------------------------------------- */

/* Fill cfg with the live reference configuration (launch/config/config_sim.yaml) */
int mlm_default_config(mlm_config *cfg);

/* mlmap::init_map (reference src/mlmap.cpp:3-149) minus ROS: builds the awareness tables
 * (map_awareness.cpp:19-82) and local-map tables (map_local.cpp:46-139), allocates device state. */
int mlm_create(const mlm_config *cfg, int device, mlm_handle *out);
int mlm_destroy(mlm_handle h);
const char *mlm_last_error(void);
int mlm_abi_version(void);
/* sizeof(mlm_config) / sizeof(mlm_frame_stats) as compiled, for binding self-checks */
size_t mlm_sizeof_config(void);
size_t mlm_sizeof_frame_stats(void);

/* ---- per-frame update (the north-star path) --------------------------------------------------- */

/* project_depth() + update_map() (reference src/mlmap.cpp:311-349,382-386) on a HOST depth image
 * (uint16 millimetres, row stride in bytes).  H2D copy, all kernels and the stats read-back are
 * inside the call. */
int mlm_integrate_depth_u16(mlm_handle h, const uint16_t *img, int rows, int cols, size_t stride_bytes,
                            const double T_wb[7], mlm_frame_stats *stats /* may be NULL */);
/* same with the image already resident in device memory (dense rows) */
int mlm_integrate_depth_u16_device(mlm_handle h, const uint16_t *d_img, int rows, int cols,
                                   const double T_wb[7], mlm_frame_stats *stats);

/* awareness_map_cylindrical::input_pc_pose + local_map_cartesian::input_pc_pose_direct
 * (reference src/map_awareness.cpp:173, src/map_local.cpp:143) on sensor-frame points, xyz doubles. */
int mlm_integrate_points_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7],
                             mlm_frame_stats *stats);
int mlm_integrate_points_f64_device(mlm_handle h, const double *d_xyz, int n, const double T_wb[7],
                                    mlm_frame_stats *stats);

/* The two layer entry points behind mlmap's public `awareness_map` / `local_map` pointers, which mlmap::update_map calls
 * one after the other (reference src/mlmap.cpp:382-386, include/mlmap.h:107-108):
 *   mlm_awareness_input_*            awareness_map_cylindrical::input_pc_pose (include/map_awareness.h:74,
 *                                    src/map_awareness.cpp:173-282): the frame's hit map and miss set, readable with
 *                                    mlm_last_frame_hits / mlm_last_frame_misses; the depth variant runs project_depth first
 *   mlm_local_input_pc_pose_direct   local_map_cartesian::input_pc_pose_direct(awareness_map) (include/map_local.h:114,
 *                                    src/map_local.cpp:143-237): fuses the staged sets into the local / global map
 * One difference is visible between the two calls: the subboxes the frame touches are allocated by the first call already
 * (all-unknown cells, so every query still answers like the reference; only mlm_export_map_count is ahead).
 * mlm_integrate_* = both calls as ONE cooperative launch. */
int mlm_awareness_input_pc_pose_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7], mlm_frame_stats *stats);
int mlm_awareness_input_depth_u16(mlm_handle h, const uint16_t *img, int rows, int cols, size_t stride_bytes,
                                  const double T_wb[7], mlm_frame_stats *stats);
int mlm_local_input_pc_pose_direct(mlm_handle h, mlm_frame_stats *stats);

/* Asynchronous frames, for several maps of one process on one GPU (BASELINE config 5: 8 agent maps): submit enqueues the
 * frame on the handle's stream and returns; mlm_frame_finish waits for it, settles a rehash frame and returns the
 * counters.  mlm_set_sm_budget(h, n) makes the handle's frame kernel use n CTAs instead of one per SM (0 restores that),
 * so that the cooperative launches of several handles are co-resident and overlap. */
int mlm_set_sm_budget(mlm_handle h, int n_sms);
int mlm_frame_submit_depth_u16_device(mlm_handle h, const uint16_t *d_img, int rows, int cols, const double T_wb[7]);
int mlm_frame_submit_points_f64_device(mlm_handle h, const double *d_xyz, int n, const double T_wb[7]);
int mlm_frame_finish(mlm_handle h, mlm_frame_stats *stats /* may be NULL */);

/* mlmap::setFree_map_in_bound (reference src/mlmap.cpp:388-407) */
int mlm_set_free_in_bound(mlm_handle h, const double box_min[3], const double box_max[3]);

/* mlmap::inflate_map (reference src/mlmap.cpp:286-309) around centre position ct_pos */
int mlm_inflate_map(mlm_handle h, const double ct_pos[3]);

/* ---- batched queries (reference include/mlmap.h:142-295); pos = n x 3 doubles ------------------ */

int mlm_get_occupancy(mlm_handle h, const double *pos, size_t n, int32_t *out);
int mlm_get_occupancy_inflate(mlm_handle h, const double *pos, size_t n, float inflate, int32_t *out);
int mlm_get_inflate_occupancy(mlm_handle h, const double *pos, size_t n, int32_t *out);
int mlm_get_odd(mlm_handle h, const double *pos, size_t n, float *out);
int mlm_get_odd_grad(mlm_handle h, const double *pos, size_t n, size_t max_iter, double *out3n);
/* getOdd(const Vec3I &glb_id, size_t subbox_id) (include/mlmap.h:128,227-235): glb3 = n x 3 subbox indices, sub = n cell ids */
int mlm_get_odd_at(mlm_handle h, const int32_t *glb3, const int32_t *sub, size_t n, float *out);
int mlm_get_odd_at_device(mlm_handle h, const int32_t *d_glb3, const int32_t *d_sub, size_t n, float *d_out);
/* device-resident variants: pos/out are device pointers, the call only enqueues on the handle's stream */
int mlm_get_occupancy_device(mlm_handle h, const double *d_pos, size_t n, int32_t *d_out);
int mlm_get_odd_device(mlm_handle h, const double *d_pos, size_t n, float *d_out);
int mlm_get_odd_grad_device(mlm_handle h, const double *d_pos, size_t n, size_t max_iter, double *d_out3n);

/* Batched ray casting (no reference counterpart; the query octomap::OcTree::castRay users know): for each segment
 * from[i] -> to[i] (n x 3 doubles, world frame) the cells it crosses, up to the first blocking one.
 *  1. Cell of a point: c_k = (int)floor(p_k / d_sub) per axis, d_sub = subbox_d_xyz, IEEE division (get_subbox_id's
 *     floor(pt / d_sub), reference include/map_local.h:167-173).  This is the canonical cell: the id-0 quirk that
 *     getOccupancy inherits from unordered_map::operator[] applies to point queries only.
 *  2. Traversal, a 6-connected DDA bounded by integer steps: c = cell(from), e = cell(to), rem_k = |e_k - c_k|,
 *     s_k = sign(e_k - c_k), v_k = to_k - from_k.  For each axis with rem_k > 0, inv_k = 1.0 / v_k once, and the next
 *     boundary t_k = ((double)(c_k + (s_k > 0)) * d_sub - from_k) * inv_k, recomputed from the integer cell after every
 *     step.  A step takes, among the axes with rem_k > 0, the one with the smallest t_k (ties: x, then y, then z; an
 *     axis replaces an earlier one only when its t_k compares strictly smaller), sets c_k += s_k, rem_k -= 1 and
 *     t_enter = t_k.  The walk visits |e - c|_1 + 1 cells and ends in e; rounding can only reorder axis steps.  All
 *     arithmetic is IEEE double without fused multiply-add.
 *  3. State of a cell: what getOccupancy returns for it: subbox absent -> UNKNOWN, collapsed -> its element 0, else
 *     occupancy[cell].  A cell blocks when its state is OCCUPIED; with MLM_RAY_INFLATED also when getInflateOccupancy
 *     of it is OCCUPIED (inflate_occupancy[cell] == 'o'; a collapsed subbox never blocks by inflation, reference
 *     include/mlmap.h:195-211).
 *  4. Output: one record per segment.  The walk stops at the first blocking cell, which may be the start cell;
 *     from == to is one cell.
 * mlm_cast_rays stages through the handle's stream and returns when the records are in `out`; mlm_cast_rays_device
 * takes device pointers and only enqueues.  flags is 0 or MLM_RAY_INFLATED.  A rank of a sharded map with world > 1
 * returns MLM_ERR_UNSUPPORTED: a segment crosses subboxes of several owners (replica handles and world-1 shards hold
 * the whole map and answer). */
#define MLM_RAY_INFLATED 1
#define MLM_RAY_INVALID (-2)
typedef struct mlm_ray_hit {
  int32_t status;    /* MLM_OCCUPIED: stopped at a blocking cell; MLM_FREE: reached cell(to) without one;
                        MLM_RAY_INVALID: a non-finite endpoint, |p / d_sub| >= 2^30, or |e - c|_1 > 2^20 cells */
  int32_t cell[3];   /* the stop cell: the first blocking cell, or cell(to); {0,0,0} when INVALID */
  int32_t n_free;    /* non-blocking cells visited whose state is FREE (the end cell included when status is FREE) */
  int32_t n_unknown; /* non-blocking cells visited whose state is UNKNOWN */
  double t;          /* t_enter of the stop cell clamped to [0, 1] (NaN -> 0); 0 for the start cell */
} mlm_ray_hit;
int mlm_cast_rays(mlm_handle h, const double *from, const double *to, size_t n, int flags, mlm_ray_hit *out);
int mlm_cast_rays_device(mlm_handle h, const double *d_from, const double *d_to, size_t n, int flags, mlm_ray_hit *d_out);
size_t mlm_sizeof_ray_hit(void);

/* Signed distance field over a box of the map (no reference counterpart; the ESDF gradient-based planners expect):
 * an exact Euclidean distance transform of the box's blocking cells, queried with trilinear interpolation.
 *  1. Box: lo_k = cell(box_min_k), hi_k = cell(box_max_k) with the ray spec's rule 1 (which fails for a non-finite value
 *     or |p / d_sub| >= 2^30), N_k = hi_k - lo_k + 1.  The grid holds the cells lo <= c <= hi.
 *  2. Blocking set B: the cells of the box that block under the ray spec's rule 3, MLM_ESDF_INFLATED playing the part of
 *     MLM_RAY_INFLATED (absent subbox: UNKNOWN, not blocking; collapsed: its element 0, never blocking by inflation;
 *     else occupancy[cell] == 'o', or inflate_occupancy[cell] == 'o' with the flag).  With max_dist >= d_sub a cell
 *     blocks a ray exactly when its value below is <= 0.  Unknown cells do not block.
 *  3. Squared distances in cell units, exact integers over the cells of the box only:
 *     D+(c) = min over b in B of |c - b|^2, D-(c) = min over f in box \ B of |c - f|^2; an empty set gives +inf.
 *     Obstacles outside the box are not seen: pad the box by max_dist where they matter.
 *  4. Cell value (double, metres): c not in B: v = min(sqrt((double)D+) * d_sub, max_dist); c in B:
 *     v = d_sub - min(sqrt((double)D-) * d_sub, max_dist), where sqrt(+inf) * d_sub counts as above max_dist.  Free
 *     cells are >= d_sub, surface obstacle cells 0, interior cells negative; an empty B gives max_dist everywhere, a
 *     box without a free cell d_sub - max_dist.  IEEE sqrt, multiply and subtract, each correctly rounded.
 *  5. Query at p (IEEE double, no fused multiply-add, in this order).  If cell(p) fails or lies outside the box:
 *     dist = NaN (the quiet NaN 0x7ff8000000000000), grad = {0, 0, 0}.  Otherwise per axis q_k = p_k / d_sub - 0.5,
 *     i_k = (int)floor(q_k), w_k = q_k - (double)i_k, u_k = 1.0 - w_k, and the corner indices
 *     clamp(i_k - lo_k, 0, N_k - 1) and clamp(i_k - lo_k + 1, 0, N_k - 1) (the clamp acts in the box's outer half
 *     cell only).  With v_xyz the corner values (x, y, z in {0, 1}) and g_yz = v_1yz - v_0yz:
 *       e_yz = v_0yz * u_x + v_1yz * w_x;  f_z = e_0z * u_y + e_1z * w_y;  dist = f_0 * u_z + f_1 * w_z;
 *       grad_z = (f_1 - f_0) / d_sub;  grad_y = ((e_10 - e_00) * u_z + (e_11 - e_01) * w_z) / d_sub;
 *       grad_x = ((((g_00 * u_y) * u_z + (g_01 * u_y) * w_z) + (g_10 * w_y) * u_z) + (g_11 * w_y) * w_z) / d_sub.
 *  6. Lifetime: the field is a snapshot of the map at mlm_esdf_build, in stream order; later frames, inflate_map,
 *     set_free_in_bound or a checkpoint restore leave it as it is until the next build.  Querying or exporting before
 *     any build returns MLM_ERR_INVALID_ARG.
 * mlm_esdf_build and the _device calls only enqueue on the handle's stream; the host variants stage through it and
 * return when the data is in place.  MLM_ERR_INVALID_ARG: null handle, null pointer with n > 0, flags other than 0 /
 * MLM_ESDF_INFLATED, max_dist not finite or <= 0, a box corner that fails rule 1, box_min > box_max on an axis.
 * MLM_ERR_CAPACITY: N_k > 4096 on an axis or N_x * N_y * N_z > 2^28 (keeps D+- below 2^26).  A rank of a sharded map
 * with world > 1 returns MLM_ERR_UNSUPPORTED like mlm_cast_rays.  The grid buffers belong to the handle: allocated by
 * the first build, grown for a larger box, freed by mlm_destroy.
 * mlm_esdf_export writes the grid as float32 (float)v(c), x fastest: index (z * N_y + y) * N_x + x, x = c_x - lo_x...;
 * lo3 and dims3 are always filled; out may be NULL with cap 0 to ask for the size; cap < N_x * N_y * N_z returns
 * MLM_ERR_CAPACITY. */
#define MLM_ESDF_INFLATED 1
int mlm_esdf_build(mlm_handle h, const double box_min[3], const double box_max[3], double max_dist, int flags);
int mlm_esdf_distance(mlm_handle h, const double *pos, size_t n, double *dist, double *grad3n /* may be NULL */);
int mlm_esdf_distance_device(mlm_handle h, const double *d_pos, size_t n, double *d_dist, double *d_grad3n /* may be NULL */);
int mlm_esdf_export(mlm_handle h, float *out, size_t cap, int32_t lo3[3], int32_t dims3[3]);
int mlm_esdf_export_device(mlm_handle h, float *d_out, size_t cap, int32_t lo3[3], int32_t dims3[3]);

/* Frontier clustering (no reference counterpart; the first step of a frontier-based explorer's planning cycle):
 * connected components of the exploration frontier sets, one record per cluster.
 *  1. Frontier set F: a cell c = glb * subbox_n + local is in F when its bit is set in its subbox's frontier bitmask
 *     (bit c of the little-endian words, cell ids < subbox_n^3 only): the cells mlm_export_frontier and
 *     MLM_CLOUD_FRONTIER report.  Cell state is not looked at (a cell that mlm_set_free_in_bound made free keeps its
 *     bit, as in the reference).  Absent and collapsed subboxes hold no frontier cells.  With a box, F is intersected
 *     with cell(box_min) <= c <= cell(box_max) per axis, cell() being the ray spec's rule 1.
 *  2. Clusters are the connected components of F.  Two cells a, b are adjacent when max_k |a_k - b_k| == 1
 *     (26-connectivity, the default) or, with MLM_FRONTIER_CONN6, when sum_k |a_k - b_k| == 1.  Cells outside the box
 *     connect nothing: a cluster the box cuts is split.
 *  3. Record of a cluster: n_cells; key = its member smallest in (z, y, x) lexicographic order; lo / hi = the per-axis
 *     minimum / maximum of its members; centroid_k = (((double)S_k / (double)n_cells) + 0.5) * d_sub with S_k the exact
 *     int64 sum of the members' c_k, each operation IEEE double, correctly rounded, without fused multiply-add.
 *  4. Output: the clusters with n_cells >= min_cells, sorted by key in (z, y, x) order; the cluster index is the position
 *     in that list.  *n_out = the number of clusters kept, which may exceed cap (then only the first cap records are
 *     written), as for mlm_export_cloud.
 *  5. Per-cell labels (optional): every cell of a kept cluster as cells3[3 i .. 3 i + 2] with its cluster index in
 *     cluster_of[i]; at most cell_cap of them are written, in unspecified (but repeatable) order; *n_cells_out (may be
 *     NULL) = their total.
 *  6. MLM_ERR_INVALID_ARG: null handle or n_out; only one of box_min / box_max given; a box corner that fails rule 1;
 *     box_min > box_max on an axis; min_cells < 1; flags other than 0 / MLM_FRONTIER_CONN6; a null output pointer with a
 *     non-zero cap (cells3 and cluster_of both for cell_cap).  MLM_ERR_UNSUPPORTED: a handle created without
 *     use_exploration_frontiers, or a rank of a sharded map with world > 1 (a cluster crosses owners; as mlm_cast_rays).
 *  7. The call is a snapshot of the map in stream order.  mlm_frontier_clusters returns once the records are in `out`;
 *     mlm_frontier_clusters_device takes device pointers for out / cells3 / cluster_of.  Both synchronise the handle's
 *     stream twice: for the number of frontier cells (which sizes the handle's scratch) and for the counts.  The scratch
 *     buffers belong to the handle: allocated by the first call, grown for a larger frontier, freed by mlm_destroy. */
#define MLM_FRONTIER_CONN6 1
typedef struct mlm_frontier_cluster {
  int32_t n_cells;
  int32_t key[3];       /* smallest member cell in (z, y, x) lexicographic order */
  int32_t lo[3], hi[3]; /* inclusive cell AABB of the members */
  double centroid[3];   /* metres */
} mlm_frontier_cluster; /* 64 bytes */
size_t mlm_sizeof_frontier_cluster(void);
int mlm_frontier_clusters(mlm_handle h, const double box_min[3], const double box_max[3] /* both NULL: whole map */,
                          int32_t min_cells, int flags, mlm_frontier_cluster *out, size_t cap, size_t *n_out,
                          int32_t *cells3 /* may be NULL */, int32_t *cluster_of /* may be NULL */, size_t cell_cap,
                          size_t *n_cells_out /* may be NULL */);
int mlm_frontier_clusters_device(mlm_handle h, const double box_min[3], const double box_max[3], int32_t min_cells,
                                 int flags, mlm_frontier_cluster *d_out, size_t cap, size_t *n_out, int32_t *d_cells3,
                                 int32_t *d_cluster_of, size_t cell_cap, size_t *n_cells_out);

/* Candidate-view gain (no reference counterpart; the second step of a frontier-based explorer's planning cycle, which
 * scores candidate viewpoints by what a depth camera there would see): per pose T_wb[i] (pose[7], the body pose as the
 * frames take it), the target cells in the frustum of a pinhole sensor and how many of them it sees through free space.
 * All arithmetic is IEEE double, correctly rounded, without fused multiply-add, in the order written.
 *  1. Pose: T_ws = T_wb * T_bs with T_bs from the handle's config and T_sw = T_ws.inverse(), both formed as the frames
 *     form theirs (Sophus SE3 from pose[7] normalising the quaternion, SE3::operator*, SE3::inverse); the origin is
 *     o = T_ws.t.  A view is MLM_VIEW_INVALID (and reports 0 / 0) when a pose component is not finite, when the
 *     quaternion's squared norm (qx^2 + qz^2) + (qy^2 + qw^2) is not > 0 or not finite, when cell(o) fails the ray spec's
 *     rule 1, or, with boxes, when lo > hi on an axis.  These are statuses per view, not call errors.
 *  2. Cells: the centre of cell c is x_k = ((double)c_k + 0.5) * d_sub (cell(x) == c), its sensor coordinates
 *     p = rotate(T_sw.q, x) + T_sw.t (Eigen's _transformVector, then the sum per axis).
 *  3. Frustum: c is in view when min_depth <= p_z <= max_depth, u = (p_x / p_z) * fx + cx and v = (p_y / p_z) * fy + cy
 *     satisfy -0.5 <= u < (double)cols - 0.5 and -0.5 <= v < (double)rows - 0.5 (the pixel centres of project_depth:
 *     pixel u back-projects through (u - cx) / fx), and, with boxes, lo_k <= c_k <= hi_k (boxes[6 i .. 6 i + 5] =
 *     inclusive cells lo[3], hi[3]).
 *  4. Targets: by default the cells whose state under the ray spec's rule 3 is UNKNOWN (neither free nor occupied; an
 *     absent subbox is unknown, a collapsed one its element 0).  With MLM_VIEW_FRONTIER the cells whose bit is set in the
 *     frontier sets (the frontier-clustering spec's rule 1), whatever their state.  n_target counts the targets in view,
 *     occluded or not.
 *  5. Line of sight: the walk of the ray spec's rule 2 from o to x, which ends in c.  The target is visible when every cell
 *     the walk visits before c is FREE and, with MLM_VIEW_INFLATED, does not block by inflation (as with MLM_RAY_INFLATED).
 *     The start cell counts when it is not c, so a view whose origin cell is not free sees nothing beyond it; the
 *     target's own state and inflation are not looked at.  n_visible counts the visible targets.
 *  6. MLM_ERR_INVALID_ARG: null handle, sensor or out; null poses with n > 0; flags other than MLM_VIEW_FRONTIER |
 *     MLM_VIEW_INFLATED; a sensor field that is not finite; fx or fy <= 0; cols or rows < 1; not 0 <= min_depth <
 *     max_depth.  MLM_ERR_CAPACITY: max_depth > 256 * d_sub, or a far corner off the optical axis by more than that,
 *     max(|(-0.5 - cx) / fx|, |((double)cols - 0.5 - cx) / fx|) * max_depth > 256 * d_sub (likewise with fy, cy and
 *     rows); this bounds a view's cells and walks.  MLM_ERR_UNSUPPORTED: MLM_VIEW_FRONTIER on a handle created without
 *     use_exploration_frontiers, or a rank of a sharded map with world > 1 (as mlm_cast_rays).
 *  7. The result is a snapshot of the map in stream order.  mlm_view_gain stages through the handle's stream and returns
 *     when the records are in `out`; mlm_view_gain_device takes device pointers for the poses, boxes and records and only
 *     enqueues (no host synchronisation).  The per-view scratch belongs to the handle: allocated by the first call, grown
 *     for a larger batch, freed by mlm_destroy. */
#define MLM_VIEW_FRONTIER 1 /* targets: the frontier-set cells (exploration handles only); default: the UNKNOWN cells */
#define MLM_VIEW_INFLATED 2 /* the inflation layer blocks the line of sight, as with MLM_RAY_INFLATED */
#define MLM_VIEW_INVALID (-2)
typedef struct mlm_view_sensor { /* pinhole depth sensor, the project_depth model */
  double fx, fy, cx, cy;         /* pixels */
  int32_t cols, rows;
  double min_depth, max_depth;   /* metres, along the optical axis */
} mlm_view_sensor;
typedef struct mlm_view_gain_record {
  int32_t status;    /* 0, or MLM_VIEW_INVALID */
  int32_t n_target;  /* target cells in the frustum (and the view's box), occluded or not */
  int32_t n_visible; /* ... of which the line of sight is clear */
  int32_t _pad;
} mlm_view_gain_record; /* 16 bytes */
size_t mlm_sizeof_view_gain(void);
int mlm_view_gain(mlm_handle h, const double *T_wb /* n x 7 */, size_t n, const mlm_view_sensor *sensor,
                  const int32_t *boxes /* n x 6, may be NULL */, int flags, mlm_view_gain_record *out);
int mlm_view_gain_device(mlm_handle h, const double *d_T_wb, size_t n, const mlm_view_sensor *sensor,
                         const int32_t *d_boxes /* may be NULL */, int flags, mlm_view_gain_record *d_out);

/* ---- stream control / timing (CUDA events on the handle's own stream) ------------------------- */

int mlm_sync(mlm_handle h);
int mlm_timer_start(mlm_handle h);
int mlm_timer_stop_ms(mlm_handle h, float *ms); /* records + synchronises; ms since mlm_timer_start */
/* device scratch helpers for harnesses that keep inputs resident */
int mlm_device_alloc(mlm_handle h, size_t bytes, void **d_ptr);
int mlm_device_free(mlm_handle h, void *d_ptr);
/* page-locked host buffers: images / point arrays placed here are DMA'd without the staging copy */
int mlm_host_alloc(mlm_handle h, size_t bytes, void **ptr);
int mlm_host_free(mlm_handle h, void *ptr);
int mlm_copy_to_device(mlm_handle h, void *d_dst, const void *src, size_t bytes);
int mlm_copy_to_host(mlm_handle h, void *dst, const void *d_src, size_t bytes);
int mlm_flush_l2(mlm_handle h); /* writes a buffer larger than L2 (bench hygiene) */
/* per-kernel timing of the frame pipeline (CUDA events between launches on the handle's stream).
 * enable=1 records events in every following frame; mlm_last_frame_kernel_ms returns the durations
 * of the MLM_NUM_FRAME_KERNELS stages of the last frame in launch order:
 * 0 k_project, 1 k_column, 2 k_fuse */
#define MLM_NUM_FRAME_KERNELS 3
int mlm_set_profiling(mlm_handle h, int enable);
int mlm_last_frame_kernel_ms(mlm_handle h, float ms[MLM_NUM_FRAME_KERNELS]);
/* per-column phase clocks of the last k_column launch (only filled by -DMLM_PHASE_TIMING builds) */
int mlm_debug_phase_cycles(mlm_handle h, long long *out, size_t cap);
/* sampled project_depth (cfg.sample_cnt > 0) draws pixels from the handle's own glibc-compatible rand() stream
 * (seed 1 like a process that never calls srand); mlm_srand reseeds it, mlm_debug_rand draws from it
 * (h == NULL: from a fresh seed-1 stream) so tests can compare with libc's rand() */
int mlm_srand(mlm_handle h, unsigned seed);
int mlm_debug_rand(mlm_handle h, int32_t *out, size_t n);
/* number of kernels launched by this handle since creation */
int mlm_kernel_launch_count(mlm_handle h, int64_t *count);

/* ---- parity / debug exports ------------------------------------------------------------------- */

/* Last frame's hit_idx_odds_hashmap in the reference's iteration order: keys = n x 3 ints
 * (rho,phi,z), p = n floats.  Returns the number of entries through *n_out (cap = array capacity). */
int mlm_last_frame_hits(mlm_handle h, int32_t *keys3, float *p, size_t cap, size_t *n_out);
/* Last frame's miss_idx_set (awareness cell indices, ascending). */
int mlm_last_frame_misses(mlm_handle h, uint64_t *idx, size_t cap, size_t *n_out);

/* Whole-map export.  mlm_export_map_count gives the number of submaps; mlm_export_map fills
 * glb3 (n x 3 int32), collapsed (n bytes), and per submap cells = subbox_n^3 entries of
 * occupancy chars ('u','f','o'), inflate chars and float log-odds (collapsed submaps: entry 0 valid). */
int mlm_export_map_count(mlm_handle h, size_t *n_submaps);
int mlm_export_map(mlm_handle h, size_t cap_submaps, int32_t *glb3, uint8_t *collapsed,
                   char *occupancy, char *inflate_occupancy, float *log_odds, size_t *n_out);

/* Exploration mode: frontier set of every subbox (reference struct subbox::frontier, include/map_local.h:58) as a
 * bitmask of ceil(subbox_n^3 / 32) 32-bit words per subbox (bit c = cell id c), with its own glb3 list. */
int mlm_export_frontier(mlm_handle h, size_t cap_submaps, int32_t *glb3, uint32_t *frontier_words, size_t *n_out);

/* ---- pose forwarding of the ROS callback (SURVEY 8f-3), host-only, no handle ---------------------------------------
 * mlmap::depth_odom_input_callback (src/mlmap.cpp:470-498) forwards the odometry pose to the image stamp with a linear
 * model before the update:  time_gap = gap_imu - latency;  rot_cp = log(R) + time_gap * (R * omega);
 * T_wb = (exp(rot_cp), p + (gap_odom - latency) * v), with Sophus' SO3::log / SO3::exp (so3.cpp:127-199).
 * gap_* = image stamp - odometry / IMU stamp in seconds; quaternion order w,x,y,z; T_wb_out = {x,y,z,qw,qx,qy,qz},
 * ready for mlm_integrate_*. */
int mlm_compensate_pose(const double odom_pos[3], const double odom_quat_wxyz[4], const double odom_lin_vel[3],
                        const double imu_ang_vel[3], double gap_odom_s, double gap_imu_s, double camera2odom_latency_s,
                        double T_wb_out[7]);

/* ---- map clouds for consumers (SURVEY 8f-2) ---------------------------------------------------------------------
 * Whole-map compaction on the device into float4 points {x, y, z, w} (16-byte stride = pcl::PointXYZ, the wire format
 * of the reference's PointCloud2 topics, include/common.h:53):
 *   MLM_CLOUD_INFLATED  cells with inflate_occupancy == 'o'  (rviz_vis::pub_global_local_map, src/rviz_vis.cpp:296-327)
 *   MLM_CLOUD_OCCUPIED  cells with occupancy == 'o'
 *   MLM_CLOUD_FRONTIER  the frontier sets                     (rviz_vis::pub_frontier, src/rviz_vis.cpp:267-294)
 * w is 1.0f.  mlm_export_odds_slice writes the cells whose centre height is within 1e-3 of `height` as
 * {x, y, z, odd}, odd = logit_inv(log_odds)  (mlmap::visualize_odds, src/mlmap.cpp:200-284).
 * `xyzw` holds `cap` points (host memory for the plain calls, device memory for *_device); *n_out is the number of
 * points the map has, which may exceed cap (then only cap points were written).  Point order is unspecified. */
#define MLM_CLOUD_INFLATED 0
#define MLM_CLOUD_OCCUPIED 1
#define MLM_CLOUD_FRONTIER 2
int mlm_export_cloud(mlm_handle h, int kind, float *xyzw, size_t cap, size_t *n_out);
int mlm_export_cloud_device(mlm_handle h, int kind, float *d_xyzw, size_t cap, size_t *n_out);
int mlm_export_odds_slice(mlm_handle h, double height, float *xyzw, size_t cap, size_t *n_out);

/* ---- checkpoint / restore of the map (SURVEY 8f-4; the reference keeps its map in process memory only) ------------
 * A checkpoint is a self-describing byte image: a header (format version, the map-defining configuration fields,
 * the cumulative counters, the emulated bucket counts of the per-frame containers and the rand() stream of the
 * sampled projection) followed by one fixed-size record per subbox (index, collapsed flag, log_odds, occupancy,
 * inflate_occupancy and, in exploration mode, the frontier set).  Restoring it into a handle created with the same
 * map-defining configuration (any pool size that holds the subboxes) replaces that handle's map; frames integrated
 * afterwards give bit for bit what the original handle would have produced.
 *   mlm_checkpoint_size     bytes mlm_checkpoint_save will write for the current map
 *   mlm_checkpoint_save     writes at most `cap` bytes into host memory `buf`; MLM_ERR_CAPACITY if cap is too small
 *   mlm_checkpoint_restore  MLM_ERR_INVALID_ARG for a foreign / truncated image, MLM_ERR_INVALID_CONFIG when the image
 *                           was taken with a different map configuration, MLM_ERR_POOL_EXHAUSTED if the pool is too small */
int mlm_checkpoint_size(mlm_handle h, size_t *bytes);
int mlm_checkpoint_save(mlm_handle h, void *buf, size_t cap, size_t *written);
int mlm_checkpoint_restore(mlm_handle h, const void *buf, size_t bytes);

/* ---- one logical map sharded over `world` ranks (SURVEY 8e: large LiDAR scans) -------------------------------------
 * The sharded form of awareness_map_cylindrical::input_pc_pose + local_map_cartesian::input_pc_pose_direct
 * (reference src/map_awareness.cpp:173-282, src/map_local.cpp:143-207) for scans too large / too frequent for one GPU:
 * every rank gets the SAME points and pose, casts the phi columns `phi % world == rank`, and owns the subboxes whose
 * index hashes to it.  Between the two stages the library itself exchanges (a) every rank's distinct hit keys with
 * their first-insert stamps (all-gather, so that all ranks derive the same unordered_map iteration order) and (b) one
 * 24-byte update record per touched voxel and hit key, sent to the voxel's owner (all-to-all).  Both exchanges are
 * plain stores into the destination's exchange arena over NVLink peer memory followed by a system-scope flag; the
 * owner waits on device.  There is no host synchronisation between mlm_shard_submit_* and mlm_shard_finish and no
 * collective-library call on the path.  The union of the ranks' subboxes equals the single-GPU map bit for bit.
 *
 * Setup (once):  mlm_shard_open on every rank -> exchange the MLM_SHARD_BLOB_BYTES blobs by any means (MPI_Allgather,
 * torch.distributed.all_gather, a file) -> mlm_shard_connect with all `world` blobs in rank order.  Ranks may be
 * processes (one GPU each; arenas mapped with CUDA IPC) or handles of one process (peer access / same device).
 * Per scan:  mlm_shard_submit_points_f64[_device] enqueues the whole scan on the handle's stream and returns;
 * mlm_shard_finish waits for it, runs the rare rehash path (a scan whose distinct hit keys exceed the emulated bucket
 * count: each rank re-sequences the gathered list on its own) and returns the counters.  One process driving several
 * handles must submit on ALL of them before finishing any.  mlm_shard_integrate_points_f64 = submit + finish.
 * A peer that fails or does not signal within MLM_SHARD_TIMEOUT_MS (default 10000) makes finish return MLM_ERR_CUDA. */
#define MLM_SHARD_BLOB_BYTES 128
#define MLM_SHARD_MAX_WORLD 16
typedef struct mlm_shard_exchange {
  int32_t world;
  int32_t n_hit_total;      /* distinct hit keys of the scan over all ranks */
  int32_t n_hit_local;      /* ... cast by this rank */
  int32_t records_received; /* update records this rank ingested (all sources) */
  int32_t records_from_self; /* -1: not tracked (sources reserve straight in the owner's inbox) */
  int32_t rehash_path;      /* 1: the scan took the rehash path */
  int64_t wait_ns;          /* time this rank's wait kernel spun for its peers */
  int64_t arena_bytes;      /* size of this rank's exchange arena */
} mlm_shard_exchange;
int mlm_shard_open(mlm_handle h, int rank, int world, void *blob_out /* MLM_SHARD_BLOB_BYTES */);
int mlm_shard_connect(mlm_handle h, const void *blobs /* world * MLM_SHARD_BLOB_BYTES, rank order */);
int mlm_shard_submit_points_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7]);
int mlm_shard_submit_points_f64_device(mlm_handle h, const double *d_xyz, int n, const double T_wb[7]);
/* the same scan handed over in slices: rank r passes points [first, first + n_slice) of the n_total points (the ranks'
 * slices partition the scan; xyz_slice is host memory, page-locked for a direct copy).  Every rank copies only its
 * slice from the host; the slices reach the other ranks' arenas over NVLink peer memory and every rank waits on the
 * device until the scan is complete. */
int mlm_shard_submit_points_slice_f64(mlm_handle h, const double *xyz_slice, int first, int n_slice, int n_total, const double T_wb[7]);
int mlm_shard_finish(mlm_handle h, mlm_frame_stats *stats /* may be NULL */);
int mlm_shard_integrate_points_f64(mlm_handle h, const double *xyz, int n, const double T_wb[7], mlm_frame_stats *stats);
int mlm_shard_last_exchange(mlm_handle h, mlm_shard_exchange *out);
/* with mlm_set_profiling(h, 1): durations of the stages of the last scan between CUDA events on the handle's stream:
 * 0 resets (+ H2D copy), 1 k_project, 2 k_column (the rank's phi columns), 3 k_shard_push (keys + records to the owners, signal),
 * 4 k_shard_act_ingest (wait for the sources, activation stamps, staging of the received records), 5 k_fuse */
#define MLM_NUM_SHARD_KERNELS 6
int mlm_shard_last_kernel_ms(mlm_handle h, float ms[MLM_NUM_SHARD_KERNELS]);
int mlm_shard_close(mlm_handle h); /* unmaps the peers' arenas; call on every rank before any rank is destroyed */

/* ---- replicated map for split query streams (SURVEY 8e): after a frame the updating rank exports the subbox
 * blocks that frame touched (mlm_dirty_count gives their number and the record size), the caller broadcasts the
 * buffer (NCCL), replicas apply it with mlm_dirty_import; queries on a replica then equal the owner's. */
int mlm_dirty_count(mlm_handle h, int32_t *n_blocks, size_t *record_bytes);
int mlm_dirty_export(mlm_handle h, void *d_out, int32_t n_blocks);
int mlm_dirty_import(mlm_handle h, const void *d_in, int32_t n_blocks);

/* The same replication without a collective of the caller: every rank opens an inbox arena (mlm_replica_open fills
 * a MLM_SHARD_BLOB_BYTES setup blob), the `world` blobs are exchanged once (any transport) and handed to
 * mlm_replica_connect in rank order.  After each frame the source rank calls mlm_replica_publish: one kernel packs the
 * frame's dirty blocks straight into every replica's inbox over NVLink peer memory (CUDA IPC between processes) and
 * raises the frame's flag; every replica calls mlm_replica_apply: one kernel waits for the flag (bounded device-side
 * spin, MLM_SHARD_TIMEOUT_MS), applies the records and acknowledges to the source.  Inboxes are double-buffered by
 * frame parity: the source may be two frames ahead of the slowest replica.  Calls come in lock step, one publish and
 * one apply per frame.  n_blocks_out (may be NULL) receives the number of blocks shipped / applied. */
int mlm_replica_open(mlm_handle h, int rank, int world, int src_rank, void *blob_out /* MLM_SHARD_BLOB_BYTES */);
int mlm_replica_connect(mlm_handle h, const void *blobs /* world * MLM_SHARD_BLOB_BYTES, rank order */);
int mlm_replica_publish(mlm_handle h, int32_t *n_blocks_out);
int mlm_replica_apply(mlm_handle h, int32_t *n_blocks_out);
int mlm_replica_close(mlm_handle h); /* unmaps the peers' arenas; call on every rank before any rank is destroyed */

/* glibc-2.39 log10f as evaluated on device (parity test hook, SURVEY §7 hard part 3) */
int mlm_debug_log10f(mlm_handle h, const float *x, size_t n, float *out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* MLMAP_B200_H */
