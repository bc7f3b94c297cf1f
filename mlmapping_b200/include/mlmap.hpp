// mlmap.hpp — C++ host-side mirror of the reference's `class mlmap` (reference include/mlmap.h:42-140)
// over the C ABI of the B200 library (include/mlmap_b200.h).  Same method names, argument meaning and
// sentinel returns; ROS types are gone: init_map takes the plain config struct, the depth/odom callback
// becomes depth_odom_input().  Header-only; link against libmlmap_b200.so.  No map arithmetic happens
// here: every call is a stream-ordered submission to the CUDA library (no CPU fallback).
#ifndef MLMAP_B200_MLMAP_HPP
#define MLMAP_B200_MLMAP_HPP

#include <cstddef>
#include <cstdint>
#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/mlmap_b200.h"

namespace mlmap_b200 {

// layout-compatible with Eigen::Matrix<double,3,1> / Eigen::Matrix<int,3,1> (reference include/common.h:22-23)
struct Vec3 {
  double v[3];
  Vec3() : v{0, 0, 0} {}
  Vec3(double x, double y, double z) : v{x, y, z} {}
  double &operator()(int i) { return v[i]; }
  double operator()(int i) const { return v[i]; }
  double &operator[](int i) { return v[i]; }
  double operator[](int i) const { return v[i]; }
};
static_assert(sizeof(Vec3) == 3 * sizeof(double), "Vec3 must be 3 contiguous doubles");
// layout-compatible stand-in for Eigen::Matrix<int,3,1> (reference include/common.h:23)
struct Vec3I {
  int32_t v[3];
  Vec3I() : v{0, 0, 0} {}
  Vec3I(int x, int y, int z) : v{x, y, z} {}
  int32_t &operator[](int i) { return v[i]; }
  int32_t operator[](int i) const { return v[i]; }
};

// pose[7] = tx,ty,tz,qw,qx,qy,qz — what Sophus::SE3(SO3(Quaterniond), Vector3d) is built from
struct SE3 {
  double p[7];
  SE3() : p{0, 0, 0, 1, 0, 0, 0} {}
  SE3(double qw, double qx, double qy, double qz, const Vec3 &t) : p{t[0], t[1], t[2], qw, qx, qy, qz} {}
};

class mlmap {
 public:
  enum { FREE = MLM_FREE, OCCUPIED = MLM_OCCUPIED, UNKNOWN = MLM_UNKNOWN };  // include/mlmap.h:109-114
  bool has_data = false;     // include/mlmap.h:115
  bool map_updated = false;  // include/mlmap.h:116

  mlmap() = default;
  mlmap(const mlmap &) = delete;
  mlmap &operator=(const mlmap &) = delete;
  ~mlmap() {
    if (h_) mlm_destroy(h_);
  }

  // mlmap::init_map(ros::NodeHandle&) (src/mlmap.cpp:3-149) with the YAML keys as a struct
  void init_map(const mlm_config &cfg, int device = 0) {
    if (h_) mlm_destroy(h_), h_ = nullptr;
    check(mlm_create(&cfg, device, &h_), "mlm_create");
    cfg_ = cfg;
  }
  static mlm_config default_config() {  // launch/config/config_sim.yaml
    mlm_config c;
    mlm_default_config(&c);
    return c;
  }

  // depth_odom_input_callback (src/mlmap.cpp:463-532) without the ROS message plumbing: the caller
  // provides the 16UC1 image and the (already latency-compensated) body pose.
  const mlm_frame_stats &depth_odom_input(const uint16_t *img, int rows, int cols, size_t stride_bytes, const SE3 &T_wb) {
    set_depth_image(img, rows, cols, stride_bytes);
    T_wb_ = T_wb;
    has_data = true;
    project_depth();
    update_map();
    map_updated = true;
    return stats_;
  }
  void set_depth_image(const uint16_t *img, int rows, int cols, size_t stride_bytes) {
    img_ = img, rows_ = rows, cols_ = cols, stride_ = stride_bytes;
  }
  void set_pose(const SE3 &T_wb) { T_wb_ = T_wb; }

  // the callback's linear pose forwarding to the image stamp (src/mlmap.cpp:470-498); gaps in seconds
  static SE3 compensate_pose(const Vec3 &pos, double qw, double qx, double qy, double qz, const Vec3 &lin_vel,
                             const Vec3 &ang_vel, double gap_odom, double gap_imu, double camera2odom_latency) {
    const double q[4] = {qw, qx, qy, qz};
    SE3 T;
    if (mlm_compensate_pose(pos.v, q, lin_vel.v, ang_vel.v, gap_odom, gap_imu, camera2odom_latency, T.p) != MLM_OK)
      throw std::runtime_error("mlm_compensate_pose failed");
    return T;
  }

  // project_depth() + update_map() (src/mlmap.cpp:311-349,382-386).  Back-projection runs inside the
  // same device pass as the awareness/local update, so project_depth() only arms the frame.
  void project_depth() { projected_ = img_ != nullptr; }
  void update_map() {
    if (!projected_) throw std::logic_error("update_map() without project_depth()");
    check(mlm_integrate_depth_u16(h_, img_, rows_, cols_, stride_, T_wb_.p, &stats_), "mlm_integrate_depth_u16");
    projected_ = false;
  }
  // awareness_map->input_pc_pose(PC_s, T_wb) + local_map->input_pc_pose_direct() for sensor-frame points
  const mlm_frame_stats &input_pc_pose(const std::vector<Vec3> &PC_s, const SE3 &T_wb) {
    check(mlm_integrate_points_f64(h_, PC_s.empty() ? nullptr : PC_s[0].v, (int)PC_s.size(), T_wb.p, &stats_),
          "mlm_integrate_points_f64");
    has_data = map_updated = true;
    return stats_;
  }

  // The reference exposes its two layers as public members and update_map() calls them one after the other
  // (include/mlmap.h:107-108, src/mlmap.cpp:382-386):
  //     awareness_map->input_pc_pose(pc_eigen, T_wb);    local_map->input_pc_pose_direct(awareness_map);
  // the same two calls here, for callers that drive the layers themselves (frame sets readable in between)
  struct awareness_layer {
    mlmap *owner;
    const mlm_frame_stats &input_pc_pose(const std::vector<Vec3> &PC_s, const SE3 &T_wb) {  // include/map_awareness.h:74
      owner->check(mlm_awareness_input_pc_pose_f64(owner->h_, PC_s.empty() ? nullptr : PC_s[0].v, (int)PC_s.size(), T_wb.p,
                                                   &owner->stats_), "mlm_awareness_input_pc_pose_f64");
      return owner->stats_;
    }
  };
  struct local_layer {
    mlmap *owner;
    const mlm_frame_stats &input_pc_pose_direct(awareness_layer *) {  // include/map_local.h:114
      owner->check(mlm_local_input_pc_pose_direct(owner->h_, &owner->stats_), "mlm_local_input_pc_pose_direct");
      owner->has_data = owner->map_updated = true;
      return owner->stats_;
    }
  };
  awareness_layer awareness_map_{this};
  local_layer local_map_{this};
  awareness_layer *awareness_map = &awareness_map_;
  local_layer *local_map = &local_map_;

  void setFree_map_in_bound(Vec3 box_min, Vec3 box_max) {  // src/mlmap.cpp:388-407
    check(mlm_set_free_in_bound(h_, box_min.v, box_max.v), "mlm_set_free_in_bound");
  }
  void inflate_map(const Vec3 &ct_pos) { check(mlm_inflate_map(h_, ct_pos.v), "mlm_inflate_map"); }  // src/mlmap.cpp:286

  // point queries, include/mlmap.h:142-295 (single-point forms: one-element batches)
  int getOccupancy(const Vec3 &pos_w) {
    int32_t r;
    check(mlm_get_occupancy(h_, pos_w.v, 1, &r), "mlm_get_occupancy");
    return r;
  }
  int getOccupancy(const Vec3 &pos_w, float inflate) {
    int32_t r;
    check(mlm_get_occupancy_inflate(h_, pos_w.v, 1, inflate, &r), "mlm_get_occupancy_inflate");
    return r;
  }
  int getInflateOccupancy(const Vec3 &pos_w) {
    int32_t r;
    check(mlm_get_inflate_occupancy(h_, pos_w.v, 1, &r), "mlm_get_inflate_occupancy");
    return r;
  }
  float getOdd(const Vec3 &pos_w) {
    float r;
    check(mlm_get_odd(h_, pos_w.v, 1, &r), "mlm_get_odd");
    return r;
  }
  float getOdd(const Vec3I &glb_id, size_t subbox_id) {  // include/mlmap.h:128,227-235
    float r;
    const int32_t sub = (int32_t)subbox_id;
    check(mlm_get_odd_at(h_, glb_id.v, &sub, 1, &r), "mlm_get_odd_at");
    return r;
  }
  Vec3 getOddGrad(const Vec3 &pos_w, size_t max_iter = 5) {
    Vec3 g;
    check(mlm_get_odd_grad(h_, pos_w.v, 1, max_iter, g.v), "mlm_get_odd_grad");
    return g;
  }
  // batched forms for trajectory optimisers: n positions, one kernel
  void getOccupancy(const Vec3 *pos_w, size_t n, int32_t *out) { check(mlm_get_occupancy(h_, pos_w->v, n, out), "mlm_get_occupancy"); }
  void getOdd(const Vec3 *pos_w, size_t n, float *out) { check(mlm_get_odd(h_, pos_w->v, n, out), "mlm_get_odd"); }
  void getOddGrad(const Vec3 *pos_w, size_t n, Vec3 *out, size_t max_iter = 5) {
    check(mlm_get_odd_grad(h_, pos_w->v, n, max_iter, out->v), "mlm_get_odd_grad");
  }
  // segment traversal up to the first blocking cell (no reference counterpart; spec at mlm_cast_rays): status
  // OCCUPIED / FREE / MLM_RAY_INVALID, stop cell, free and unknown cells crossed, t of the stop cell
  mlm_ray_hit castRay(const Vec3 &from, const Vec3 &to, bool inflated = false) {
    mlm_ray_hit r;
    check(mlm_cast_rays(h_, from.v, to.v, 1, inflated ? MLM_RAY_INFLATED : 0, &r), "mlm_cast_rays");
    return r;
  }
  void castRays(const Vec3 *from, const Vec3 *to, size_t n, mlm_ray_hit *out, bool inflated = false) {
    check(mlm_cast_rays(h_, n ? from->v : nullptr, n ? to->v : nullptr, n, inflated ? MLM_RAY_INFLATED : 0, out),
          "mlm_cast_rays");
  }
  // signed distance field over a box (no reference counterpart; spec at mlm_esdf_build): a snapshot of the map until
  // the next build; getEsdf is NaN with a zero gradient outside the box
  void buildEsdf(const Vec3 &min, const Vec3 &max, double max_dist, bool inflated = false) {
    check(mlm_esdf_build(h_, min.v, max.v, max_dist, inflated ? MLM_ESDF_INFLATED : 0), "mlm_esdf_build");
  }
  double getEsdf(const Vec3 &pos, Vec3 *grad = nullptr) {
    double d;
    check(mlm_esdf_distance(h_, pos.v, 1, &d, grad ? grad->v : nullptr), "mlm_esdf_distance");
    return d;
  }
  void getEsdfs(const Vec3 *pos, size_t n, double *dist, Vec3 *grad = nullptr) {
    check(mlm_esdf_distance(h_, n ? pos->v : nullptr, n, dist, grad ? grad->v : nullptr), "mlm_esdf_distance");
  }

  // frontier clustering (no reference counterpart; spec at mlm_frontier_clusters): the clusters with >= min_cells cells
  // sorted by key (z, y, x); box_min / box_max both null for the whole map; cells3 / cluster_of (optional) receive every
  // cell of a kept cluster with its cluster index
  std::vector<mlm_frontier_cluster> frontierClusters(const Vec3 *box_min = nullptr, const Vec3 *box_max = nullptr,
                                                     int min_cells = 1, bool conn6 = false,
                                                     std::vector<int32_t> *cells3 = nullptr,
                                                     std::vector<int32_t> *cluster_of = nullptr) {
    const double *a = box_min ? box_min->v : nullptr, *b = box_max ? box_max->v : nullptr;
    const int flags = conn6 ? MLM_FRONTIER_CONN6 : 0;
    size_t n = 0, m = 0;
    check(mlm_frontier_clusters(h_, a, b, min_cells, flags, nullptr, 0, &n, nullptr, nullptr, 0, &m),
          "mlm_frontier_clusters");
    std::vector<mlm_frontier_cluster> out(n);
    const bool lab = cells3 && cluster_of;
    if (lab) {
      cells3->resize(3 * m);
      cluster_of->resize(m);
    }
    check(mlm_frontier_clusters(h_, a, b, min_cells, flags, out.data(), n, &n, lab ? cells3->data() : nullptr,
                                lab ? cluster_of->data() : nullptr, lab ? m : 0, &m),
          "mlm_frontier_clusters");
    return out;
  }

  // candidate-view gain (no reference counterpart; spec at mlm_view_gain): per body pose (pose[7] each) the target
  // cells (unknown, or frontier) in the sensor's frustum and how many of them it sees through free cells; boxes
  // (n x 6 inclusive cells lo, hi) may be null
  std::vector<mlm_view_gain_record> viewGain(const double *T_wb, size_t n, const mlm_view_sensor &sensor,
                                             const int32_t *boxes = nullptr, bool frontier = false,
                                             bool inflated = false) {
    std::vector<mlm_view_gain_record> out(n);
    if (n == 0) return out;
    const int flags = (frontier ? MLM_VIEW_FRONTIER : 0) | (inflated ? MLM_VIEW_INFLATED : 0);
    check(mlm_view_gain(h_, T_wb, n, &sensor, boxes, flags, out.data()), "mlm_view_gain");
    return out;
  }

  // map clouds for consumers: what rviz_vis::pub_global_local_map / pub_frontier put on the wire
  // (src/rviz_vis.cpp:267-327) and mlmap::visualize_odds' slice (src/mlmap.cpp:200-284), compacted on the device.
  // Points are {x, y, z, w} floats, the layout of pcl::PointXYZ.
  struct PointXYZW { float x, y, z, w; };
  std::vector<PointXYZW> map_cloud(int kind = MLM_CLOUD_INFLATED) {
    size_t n = 0;
    check(mlm_export_cloud(h_, kind, nullptr, 0, &n), "mlm_export_cloud");
    std::vector<PointXYZW> pts(n);
    if (n) check(mlm_export_cloud(h_, kind, &pts[0].x, n, &n), "mlm_export_cloud");
    pts.resize(std::min(n, pts.size()));
    return pts;
  }
  std::vector<PointXYZW> frontier_cloud() { return map_cloud(MLM_CLOUD_FRONTIER); }
  std::vector<PointXYZW> odds_slice(double height = 0.7) {  // w = logit_inv(log_odds) of the cell
    size_t n = 0;
    check(mlm_export_odds_slice(h_, height, nullptr, 0, &n), "mlm_export_odds_slice");
    std::vector<PointXYZW> pts(n);
    if (n) check(mlm_export_odds_slice(h_, height, &pts[0].x, n, &n), "mlm_export_odds_slice");
    pts.resize(std::min(n, pts.size()));
    return pts;
  }
  // checkpoint / restore of the whole map (no counterpart in the reference, which keeps its map in process memory)
  std::vector<unsigned char> checkpoint() {
    size_t n = 0;
    check(mlm_checkpoint_size(h_, &n), "mlm_checkpoint_size");
    std::vector<unsigned char> image(n);
    check(mlm_checkpoint_save(h_, image.data(), image.size(), &n), "mlm_checkpoint_save");
    image.resize(n);
    return image;
  }
  void restore(const std::vector<unsigned char> &image) {
    check(mlm_checkpoint_restore(h_, image.data(), image.size()), "mlm_checkpoint_restore");
  }

  const mlm_frame_stats &last_stats() const { return stats_; }
  mlm_handle handle() const { return h_; }

 private:
  void check(int rc, const char *what) {
    if (rc != MLM_OK) throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + mlm_last_error());
  }
  mlm_handle h_ = nullptr;
  mlm_config cfg_{};
  mlm_frame_stats stats_{};
  const uint16_t *img_ = nullptr;
  int rows_ = 0, cols_ = 0;
  size_t stride_ = 0;
  SE3 T_wb_;
  bool projected_ = false;
};

}  // namespace mlmap_b200
#endif
