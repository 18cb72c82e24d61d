// nodes.hpp — ROS-free host side of the two reference nodes, above the C ABI.
//
// Same class names, member names (including the reference's spelling), defaults, and
// cloud_handler behaviour as GroundRemover (src/ground_removal.cpp:16-90) and ConeDetector
// (src/cone_detection.cpp:19-364); the PCL hot path inside the handlers is replaced by calls
// into libconesgpu (include/conesgpu.h).  What stays on the host, exactly as in the reference:
// the radial extension (:276-278), the temporal gate / points buffer (:282-320), the colour
// routing (:287-333, through a callback that stands for the ROS service) and the publish
// quirks (:177-186: header and fields copied from the input message, Q6).
#pragma once
#include <cmath>
#include <cstring>
#include <cstdio>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "pointcloud2.hpp"

namespace cones_host {

// include/perception_handling/color.hpp:8-15
enum Color { kUnknownColor = 0, kYellow = 1, kBlue = 2, kOrange = 3, kNumberOfColors = 4 };

// src/perception_handling/utils.cpp:32-34
inline float euclidan_dist(float x1, float y1, float z1, float x2, float y2, float z2) {
  return static_cast<float>(std::sqrt(std::pow(static_cast<double>(x1 - x2), 2) + std::pow(static_cast<double>(y1 - y2), 2) +
                                      std::pow(static_cast<double>(z1 - z2), 2)));
}

class GpuError : public std::runtime_error {
 public:
  GpuError(cp_status s, const std::string& detail)
      : std::runtime_error(std::string(cp_strerror(s)) + ": " + detail), status(s) {}
  cp_status status;
};

// Not in the reference (PARITY UNPINNED, cp_plane_params in include/conesgpu.h): the ground model of a node, node
// parameter ~ground_model: "sectors" (the reference's per-sector minima, the default) or "plane" (a seeded RANSAC plane
// per frame, for a pitching or rolling sensor), with the plane model's ~plane_* parameters.
struct GroundModelParams {
  std::string ground_model = "sectors";
  int plane_seed = 0;
  int plane_hypotheses = 64;
  double plane_inlier_distance = 0.1;
  double plane_ground_height = 0.1;
  double plane_max_tilt_deg = 15.0;

 protected:
  // selects the model on the handle before a call with ground removal
  void apply_ground_model(cp_handle* h) const {
    cp_status st;
    if (ground_model == "sectors") {
      st = cp_set_ground_plane(h, nullptr);
    } else if (ground_model == "plane") {
      const cp_plane_params p{static_cast<uint64_t>(static_cast<uint32_t>(plane_seed)),
                              plane_hypotheses > 0 ? static_cast<uint32_t>(plane_hypotheses) : 0u,
                              static_cast<float>(plane_inlier_distance), static_cast<float>(plane_ground_height),
                              static_cast<float>(plane_max_tilt_deg)};
      st = cp_set_ground_plane(h, &p);
    } else {
      throw GpuError(CP_E_PARAM, "ground_model must be \"sectors\" or \"plane\", not \"" + ground_model + "\"");
    }
    if (st != CP_OK) throw GpuError(st, cp_last_error(h));
  }
};

class GroundRemover : public GroundModelParams {
 public:
  // members, src/ground_removal.cpp:18-27 (set them before the first cloud_handler call; the
  // reference reads them once in its constructor, :31-39)
  int num_of_sectors = 16;
  float default_lowest_point = -0.1f;
  std::string input_cloud_topic = "/cloud";
  std::string groundless_cloud_topic = "groundless_cloud";

  // max_frames > 1 only matters for replay(): messages per device batch (max_points bounds their points)
  explicit GroundRemover(uint64_t max_points = 4u << 20, int device = 0, uint32_t max_point_step = 64,
                         uint32_t max_frames = 1) {
    cp_config cfg{};
    cfg.device = device;
    cfg.max_points = max_points;
    cfg.max_frames = max_frames;
    cfg.max_point_step = max_point_step;
    cp_status st = cp_create(&gpu_, &cfg);
    if (st != CP_OK) throw GpuError(st, cp_create_error());
    max_points_ = max_points;
    max_frames_ = max_frames;
  }
  ~GroundRemover() { cp_destroy(gpu_); }
  GroundRemover(const GroundRemover&) = delete;
  GroundRemover& operator=(const GroundRemover&) = delete;

  // src/ground_removal.cpp:50-89; returns what the node publishes on groundless_cloud
  PointCloud2 cloud_handler(const PointCloud2& cloud_msg) {
    cp_cloud_view in = make_view(cloud_msg, /*fake_missing_intensity=*/false);
    cp_ground_params g{num_of_sectors, default_lowest_point};
    apply_ground_model(gpu_);
    PointCloud2 out = published_shell(cloud_msg);
    cp_status st = cp_ground_remove(gpu_, &in, &g, out.data.data(), &last_kept_, nullptr);
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    return out;
  }

  // cloud_handler for a series of messages, in device batches of up to max_frames messages and max_points points
  // (cp_batch_ground_remove).  Returns, per message, the message cloud_handler would publish.  The node keeps no
  // state between messages, so replay and cloud_handler may be mixed on one object.
  std::vector<PointCloud2> replay(const std::vector<PointCloud2>& msgs) {
    std::vector<PointCloud2> out;
    out.reserve(msgs.size());
    cp_ground_params g{num_of_sectors, default_lowest_point};
    apply_ground_model(gpu_);
    size_t i = 0;
    while (i < msgs.size()) {
      std::vector<cp_cloud_view> views;
      uint64_t pts = 0;
      for (; i < msgs.size() && views.size() < max_frames_; ++i) {
        const uint64_t n = static_cast<uint64_t>(msgs[i].width) * msgs[i].height;
        if (!views.empty() && pts + n > max_points_) break;
        views.push_back(make_view(msgs[i], /*fake_missing_intensity=*/false));
        pts += n;
      }
      const size_t first = i - views.size();
      const uint32_t F = static_cast<uint32_t>(views.size());
      cp_status st = cp_batch_set_host_input(gpu_, views.data(), F);
      if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
      batch_buf_.resize(static_cast<size_t>(pts) * 32);
      std::vector<uint32_t> kept(F);
      st = cp_batch_ground_remove(gpu_, &g, batch_buf_.data(), pts, kept.data(), nullptr);
      if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
      size_t at = 0;
      for (uint32_t f = 0; f < F; ++f) {
        PointCloud2 m = published_shell(msgs[first + f]);
        if (!m.data.empty()) std::memcpy(m.data.data(), batch_buf_.data() + at, m.data.size());
        at += m.data.size();
        out.push_back(std::move(m));
      }
      last_kept_ = kept[F - 1];
    }
    return out;
  }
  uint32_t last_kept() const { return last_kept_; }

 private:
  // the published message around the data: toROSMsg (:86) overwrites the header/fields assigned at :83-84: PCL
  // layout, and the stamp survives the ROS -> PCL -> ROS round trip at microsecond resolution (Q5)
  static PointCloud2 published_shell(const PointCloud2& cloud_msg) {
    PointCloud2 out;
    out.header = cloud_msg.header;
    out.header.stamp_nsec = cloud_msg.header.stamp_nsec / 1000u * 1000u;
    out.height = cloud_msg.height;
    out.width = cloud_msg.width;
    out.fields = pcl_xyzi_fields();
    out.is_bigendian = false;
    out.point_step = 32;
    out.row_step = 32 * out.width;
    out.is_dense = cloud_msg.is_dense;
    out.data.resize(static_cast<size_t>(out.row_step) * out.height);
    return out;
  }
  cp_handle* gpu_ = nullptr;
  uint64_t max_points_ = 0;
  uint32_t max_frames_ = 1;
  uint32_t last_kept_ = 0;
  std::vector<uint8_t> batch_buf_;
};

// the stateful tail of get_centroid_clouds (src/cone_detection.cpp:276-340), separated so it
// can be tested without a GPU
class ConeTracker {
 public:
  bool classify_colors = false;
  bool use_points_buffer = false;
  double cones_matching_dist_theshold = 0.5;
  double cone_position_extension_length = 0.05;
  float CONE_WIDTH = 0.228f;
  // stands for the color_classifier ROS service (src/cone_detection.cpp:342-363): receives the
  // reconstructed raw-point crops (:222-238), returns one Color per crop
  std::function<std::vector<Color>(const std::vector<std::vector<Point>>&)> get_colors;
  // optional: all crops of a frame at once (the GPU box gather, cp_cone_crops).  A crop depends only on
  // its centre and the raw cloud, so gathering them after the loop equals the per-cone calls at :309.
  std::function<std::vector<std::vector<Point>>(const std::vector<Point>&)> reconstruct_cones;
  // optional: classify straight from the centres (the GPU crops + range images, cp_cone_images);
  // replaces reconstruct + get_colors when set
  std::function<std::vector<Color>(const std::vector<Point>&)> classify_centers;

  // centroids: cluster means (x, y) in the order the detector emitted them.
  // whole_cloud: the raw input cloud (only read when classify_colors, :309).
  // Returns the four colour clouds of this frame.
  std::vector<std::vector<Point>> update(const std::vector<std::pair<float, float>>& centroids,
                                         const std::vector<Point>* whole_cloud) {
    std::vector<std::vector<Point>> centroid_clouds(kNumberOfColors);
    auto currently_detected_cones = std::make_shared<std::vector<Point>>();
    std::vector<std::vector<Point>> cones_clouds_for_color_classification;
    std::vector<Point> centroid_cloud_for_color_classification;
    for (const auto& c : centroids) {
      Point p;
      p.x = c.first;
      p.y = c.second;
      p.z = 0.0;
      // :276-278 move centroid further back, closer to the middle of the cone
      float vector_len = euclidan_dist(p.x, p.y, p.z, 0, 0, 0);
      p.x = p.x + p.x / vector_len * cone_position_extension_length;
      p.y = p.y + p.y / vector_len * cone_position_extension_length;
      currently_detected_cones->push_back(p);
      if (prev_detected_cones_) {  // :282
        for (const Point& prev : *prev_detected_cones_) {
          if (!use_points_buffer ||
              euclidan_dist(p.x, p.y, p.z, prev.x, prev.y, prev.z) < cones_matching_dist_theshold) {  // :286
            if (classify_colors) {
              bool need_color = true;
              for (int i = kUnknownColor + 1; i < kNumberOfColors; i++) {  // :291-306
                if (prev_centroid_clouds_[i]) {
                  for (const Point& q : *prev_centroid_clouds_[i]) {
                    if (euclidan_dist(p.x, p.y, p.z, q.x, q.y, q.z) < cones_matching_dist_theshold) {
                      need_color = false;
                      centroid_clouds[i].push_back(p);
                      break;
                    }
                  }
                  if (!need_color) break;
                }
              }
              if (need_color) centroid_cloud_for_color_classification.push_back(p);  // :308-312, crops below
            } else {
              centroid_clouds[kUnknownColor].push_back(p);  // :315
            }
            break;  // :317
          }
        }
      }
    }
    if (classify_colors) {  // :326-333
      const std::vector<Point>& need = centroid_cloud_for_color_classification;
      std::vector<Color> colors(need.size(), kUnknownColor);
      std::vector<Color> got;
      if (classify_centers && !need.empty()) {
        got = classify_centers(need);
      } else if (!need.empty()) {
        if (reconstruct_cones) {
          cones_clouds_for_color_classification = reconstruct_cones(need);
        } else {
          for (const Point& p : need)  // :309
            cones_clouds_for_color_classification.push_back(
                whole_cloud ? get_reconstructed_cone(p, *whole_cloud) : std::vector<Point>());
        }
        if (get_colors) got = get_colors(cones_clouds_for_color_classification);
      }
      // :352-353 std::transform over the response: a service that answers fewer colours than crops
      // (it skips empty crops) fills the front of the vector only
      for (size_t i = 0; i < got.size() && i < colors.size(); ++i) colors[i] = got[i];
      for (size_t i = 0; i < colors.size(); i++) centroid_clouds[colors[i]].push_back(centroid_cloud_for_color_classification[i]);
    }
    for (int i = 0; i < kNumberOfColors; i++)  // :335-337
      prev_centroid_clouds_[i] = std::make_shared<std::vector<Point>>(centroid_clouds[i]);
    prev_detected_cones_ = currently_detected_cones;  // :339
    return centroid_clouds;
  }

  // src/cone_detection.cpp:222-238
  std::vector<Point> get_reconstructed_cone(const Point& cone_center, const std::vector<Point>& cloud) const {
    std::vector<Point> out;
    for (const Point& it : cloud) {
      if ((cone_center.x + (CONE_WIDTH / 1.5) >= it.x && cone_center.x - (CONE_WIDTH / 1.5) <= it.x) &&
          (cone_center.y + (CONE_WIDTH / 1.5) >= it.y && cone_center.y - (CONE_WIDTH / 1.5) <= it.y)) {
        Point p;
        p.x = it.x;
        p.y = it.y;
        p.z = it.z;
        p.intensity = it.intensity;
        out.push_back(p);
      }
    }
    return out;
  }

  void reset() {
    prev_detected_cones_.reset();
    for (auto& p : prev_centroid_clouds_) p.reset();
  }

 private:
  std::shared_ptr<std::vector<Point>> prev_detected_cones_;  // NULL until the first frame (:62)
  std::shared_ptr<std::vector<Point>> prev_centroid_clouds_[kNumberOfColors];
};

class ConeDetector : public GroundModelParams {
 public:
  // members, src/cone_detection.cpp:22-51, same names / types / defaults
  const float CONE_WIDTH = 0.228f;
  const float CONE_HEIGHT = 0.325f;
  double distance_treshold_max = 7.0;
  double distance_treshold_min = 0.7;
  double level_threshold = -0.5;
  double angle_threshold = 90.0;
  int min_cluster_size = 3;
  int max_cluster_size = 50;
  bool classify_colors = true;
  bool use_points_buffer = false;
  double cones_matching_dist_theshold = 0.5;
  double cone_position_extension_length = 0.05;
  double voxel_filter_leaf_size_x = 0.04;
  double voxel_filter_leaf_size_y = 0.04;
  double voxel_filter_leaf_size_z = 0.04;
  std::string cones_frame_id = "cloud";
  std::string input_cloud_topic = "/cloud";
  std::string cones_topics[kNumberOfColors] = {"cones_cloud_unknowns", "cones_cloud_yellows", "cones_cloud_blues",
                                               "cones_cloud_oranges"};
  // not in the reference: fuse the ground_removal node in front (one process, one H2D copy).  The cluster records
  // equal those of the two nodes chained through the groundless_cloud topic; the colour crops equal the chain's only
  // with groundless_color_crops (otherwise they are cut from the raw cloud, ground returns included).  The fused
  // node uses the ground model of GroundModelParams (ground_model = "plane": groundless_color_crops is refused)
  bool fused_ground_removal = false;
  // not in the reference: with fused_ground_removal, cut the colour crops from the ground node's message, as the
  // chained detector does (cp_set_color_cloud(CP_COLOR_CLOUD_GROUNDLESS)); clouds are then staged as the ground node
  // reads them (intensity 0 without an intensity field).  No effect without fused_ground_removal.  kHostCrops holds
  // no groundless cloud on the host and refuses it.
  bool groundless_color_crops = false;
  int num_of_sectors = 16;
  float default_lowest_point = -0.1f;
  std::function<std::vector<Color>(const std::vector<std::vector<Point>>&)> get_colors;
  // not in the reference: where the colour-path inputs are produced.
  //   kHostCrops  the reference's host loop over the whole cloud per cone (:222-238)
  //   kGpuCrops   cp_cone_crops on the cloud the detection call already staged; get_colors sees the same crops
  //   kGpuImages  cp_cone_images: crops and ColorClassifier.to_image both on the device; the classifier
  //               hook get_colors_from_images receives 15x12 uint8 images + CP_CONE_* flags (180 B per cone)
  //   kGpuColors  cp_cone_colors: crops, images and the classifier network (models/dam_net) all on the device; one
  //               byte per cone comes back and no colour service is called.  Needs load_color_model().
  enum ColorInputs { kHostCrops = 0, kGpuCrops = 1, kGpuImages = 2, kGpuColors = 3 };
  ColorInputs color_inputs = kGpuCrops;
  std::function<std::vector<Color>(const std::vector<uint8_t>& images, const std::vector<uint32_t>& flags)>
      get_colors_from_images;

  // max_frames > 1 only matters for replay(): messages per device batch (max_points bounds their points)
  explicit ConeDetector(uint64_t max_points = 4u << 20, int device = 0, uint32_t max_point_step = 64,
                        uint32_t max_frames = 1) {
    cp_config cfg{};
    cfg.device = device;
    cfg.max_points = max_points;
    cfg.max_frames = max_frames;
    cfg.max_point_step = max_point_step;
    cp_status st = cp_create(&gpu_, &cfg);
    if (st != CP_OK) throw GpuError(st, cp_create_error());
    max_points_ = max_points;
    max_frames_ = max_frames;
  }
  ~ConeDetector() { cp_destroy(gpu_); }
  // Loads the classifier the reference's service reads from its ~model_path parameter (a .tflite file,
  // scripts/color_classifier_server.py:44-66) into the library and routes the colour path through it.
  void load_color_model(const std::string& path, float threshold = 0.8f) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw GpuError(CP_E_PARAM, "cannot open colour model " + path);
    std::vector<uint8_t> bytes;
    uint8_t buf[4096];
    size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0) bytes.insert(bytes.end(), buf, buf + n);
    fclose(f);
    load_color_model(bytes.data(), bytes.size(), threshold);
  }
  void load_color_model(const void* data, size_t size, float threshold = 0.8f) {
    cp_status st = cp_color_net_load_tflite(gpu_, data, size, threshold);
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    color_inputs = kGpuColors;
  }
  ConeDetector(const ConeDetector&) = delete;
  ConeDetector& operator=(const ConeDetector&) = delete;

  // src/cone_detection.cpp:130-187; returns the four clouds the node publishes
  // (cones_cloud_unknowns, _yellows, _blues, _oranges)
  std::vector<PointCloud2> cloud_handler(const PointCloud2& cloud_msg) {
    use_entry(kPerMessage);
    if (!intensity_in_cloud_checked_) {  // :131-136
      if (!cones_host::intensity_in_cloud(cloud_msg)) intensity_in_cloud_ = false;
      intensity_in_cloud_checked_ = true;
    }
    cp_detect_params d{distance_treshold_max, distance_treshold_min, level_threshold, angle_threshold,
                       voxel_filter_leaf_size_x, voxel_filter_leaf_size_y, voxel_filter_leaf_size_z,
                       min_cluster_size, max_cluster_size, CONE_WIDTH, CONE_HEIGHT};
    cp_ground_params g{num_of_sectors, default_lowest_point};
    if (fused_ground_removal) apply_ground_model(gpu_);
    set_color_cloud();
    cp_cloud_view in = make_view(cloud_msg, !intensity_in_cloud_ && !groundless());
    clusters_.resize(4096);
    uint32_t n = 0;
    cp_status st = cp_detect(gpu_, &in, &d, fused_ground_removal ? &g : nullptr, clusters_.data(),
                             static_cast<uint32_t>(clusters_.size()), &n, &counters_);
    if (st == CP_E_CAPACITY && counters_.n_clusters > clusters_.size()) {
      clusters_.resize(counters_.n_clusters);
      st = cp_detect(gpu_, &in, &d, fused_ground_removal ? &g : nullptr, clusters_.data(),
                     static_cast<uint32_t>(clusters_.size()), &n, &counters_);
    }
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    std::vector<std::pair<float, float>> centroids(n);
    for (uint32_t k = 0; k < n; ++k) centroids[k] = {clusters_[k].x, clusters_[k].y};
    tracker_.classify_colors = classify_colors;
    tracker_.use_points_buffer = use_points_buffer;
    tracker_.cones_matching_dist_theshold = cones_matching_dist_theshold;
    tracker_.cone_position_extension_length = cone_position_extension_length;
    tracker_.get_colors = get_colors;
    tracker_.reconstruct_cones = nullptr;
    tracker_.classify_centers = nullptr;
    std::vector<Point> whole;
    if (classify_colors && color_inputs == kHostCrops) {
      whole = from_msg(cloud_msg, in);  // :158 copyPointCloud, colour path only
    } else if (classify_colors && color_inputs == kGpuCrops) {
      tracker_.reconstruct_cones = [this](const std::vector<Point>& need) { return gpu_crops(need); };
    } else if (classify_colors && color_inputs == kGpuColors) {
      tracker_.classify_centers = [this](const std::vector<Point>& need) { return gpu_colors(need); };
    } else if (classify_colors) {
      tracker_.classify_centers = [this](const std::vector<Point>& need) { return gpu_classify(need); };
    }
    std::vector<std::vector<Point>> clouds =
        tracker_.update(centroids, classify_colors && color_inputs == kHostCrops ? &whole : nullptr);
    std::vector<PointCloud2> out(kNumberOfColors);
    for (int i = 0; i < kNumberOfColors; i++) {  // :177-186
      out[i] = to_msg(clouds[i]);
      out[i].header = cloud_msg.header;
      out[i].fields = cloud_msg.fields;  // Q6: the input's field list over 32-byte PCL points
    }
    return out;
  }

  // cloud_handler for a series of consecutive messages to this node, in device batches of up to max_frames messages:
  // cp_detect_batch, then cp_batch_track continues the node's state on the device (the gate, the colour carry-over
  // and the publish order of ConeTracker::update).  Returns, per message, the four clouds cloud_handler would publish.
  // Colours: classify_colors = false, or the device net (load_color_model); the external-service colour modes
  // stay on cloud_handler.  One object serves either cloud_handler or replay: the state of one is not the other's.
  std::vector<std::vector<PointCloud2>> replay(const std::vector<PointCloud2>& msgs) {
    use_entry(kReplay);
    if (classify_colors && color_inputs != kGpuColors)
      throw GpuError(CP_E_PARAM, "replay classifies colours with the device net only (load_color_model)");
    set_color_cloud();
    std::vector<std::vector<PointCloud2>> out;
    out.reserve(msgs.size());
    size_t i = 0;
    while (i < msgs.size()) {
      if (!intensity_in_cloud_checked_) {  // :131-136
        if (!cones_host::intensity_in_cloud(msgs[i])) intensity_in_cloud_ = false;
        intensity_in_cloud_checked_ = true;
      }
      std::vector<cp_cloud_view> views;
      uint64_t pts = 0;
      for (; i < msgs.size() && views.size() < max_frames_; ++i) {
        const uint64_t n = static_cast<uint64_t>(msgs[i].width) * msgs[i].height;
        if (!views.empty() && pts + n > max_points_) break;
        views.push_back(make_view(msgs[i], !intensity_in_cloud_ && !groundless()));
        pts += n;
      }
      replay_batch(msgs, i - views.size(), views, &out);
    }
    return out;
  }
  const cp_frame_counters& last_counters() const { return counters_; }
  const std::vector<cp_cluster>& last_clusters() const { return clusters_; }

 private:
  bool groundless() const { return fused_ground_removal && groundless_color_crops; }
  void set_color_cloud() {
    if (groundless() && classify_colors && color_inputs == kHostCrops)
      throw GpuError(CP_E_PARAM, "groundless_color_crops needs the device crops (kGpuCrops, kGpuImages, kGpuColors): "
                                 "kHostCrops has no groundless cloud on the host");
    cp_status st = cp_set_color_cloud(gpu_, groundless() ? CP_COLOR_CLOUD_GROUNDLESS : CP_COLOR_CLOUD_STAGED);
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
  }
  static std::vector<Point> from_msg(const PointCloud2& m, const cp_cloud_view& v) {
    std::vector<Point> out(static_cast<size_t>(m.width) * m.height);
    for (uint32_t r = 0; r < m.height; ++r)
      for (uint32_t c = 0; c < m.width; ++c) {
        const uint8_t* src = m.data.data() + static_cast<size_t>(r) * m.row_step + static_cast<size_t>(c) * m.point_step;
        Point& p = out[static_cast<size_t>(r) * m.width + c];
        if (v.off_x >= 0) std::memcpy(&p.x, src + v.off_x, 4);
        if (v.off_y >= 0) std::memcpy(&p.y, src + v.off_y, 4);
        if (v.off_z >= 0) std::memcpy(&p.z, src + v.off_z, 4);
        if (v.off_intensity >= 0) std::memcpy(&p.intensity, src + v.off_intensity, 4);
      }
    return out;
  }
  static std::vector<cp_cone_center> centers_of(const std::vector<Point>& need) {
    std::vector<cp_cone_center> c(need.size());
    for (size_t i = 0; i < need.size(); ++i) c[i] = {need[i].x, need[i].y};
    return c;
  }
  // get_reconstructed_cone for every cone that needs a colour, on the cloud cp_detect left on the device
  std::vector<std::vector<Point>> gpu_crops(const std::vector<Point>& need) {
    const std::vector<cp_cone_center> c = centers_of(need);
    std::vector<uint32_t> off(c.size() + 1);
    cp_status st = cp_cone_crops(gpu_, nullptr, 0, c.data(), static_cast<uint32_t>(c.size()), CONE_WIDTH, off.data(),
                                 crop_buf_.data(), static_cast<uint32_t>(crop_buf_.size() / 4));
    if (st == CP_E_CAPACITY) {  // offsets are complete: size the buffer and fetch again
      crop_buf_.resize(static_cast<size_t>(off.back()) * 4);
      st = cp_cone_crops(gpu_, nullptr, 0, c.data(), static_cast<uint32_t>(c.size()), CONE_WIDTH, off.data(),
                         crop_buf_.data(), static_cast<uint32_t>(crop_buf_.size() / 4));
    }
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    std::vector<std::vector<Point>> crops(c.size());
    for (size_t k = 0; k < c.size(); ++k) {
      crops[k].resize(off[k + 1] - off[k]);
      for (uint32_t i = off[k]; i < off[k + 1]; ++i) {
        Point& p = crops[k][i - off[k]];  // `Point p;` then four fields (:224-233)
        p.x = crop_buf_[4 * i];
        p.y = crop_buf_[4 * i + 1];
        p.z = crop_buf_[4 * i + 2];
        p.intensity = crop_buf_[4 * i + 3];
      }
    }
    return crops;
  }
  std::vector<Color> gpu_classify(const std::vector<Point>& need) {
    const std::vector<cp_cone_center> c = centers_of(need);
    std::vector<uint8_t> images(c.size() * CP_CONE_IMG_ROWS * CP_CONE_IMG_COLS);
    std::vector<uint32_t> flags(c.size());
    cp_status st = cp_cone_images(gpu_, nullptr, 0, c.data(), static_cast<uint32_t>(c.size()), CONE_WIDTH,
                                  images.data(), nullptr, flags.data());
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    return get_colors_from_images ? get_colors_from_images(images, flags) : std::vector<Color>();
  }
  // The whole service on the device.  Response semantics of handle_classify_color (color_classifier_server.py:
  // 78-126): an empty crop is skipped, so the response is shorter and later colours move up (:83-84); if to_image
  // would raise for any cone the call fails and the node keeps every cone unknown (src/cone_detection.cpp:356-361).
  std::vector<Color> gpu_colors(const std::vector<Point>& need) {
    const std::vector<cp_cone_center> c = centers_of(need);
    std::vector<uint8_t> colors(c.size());
    std::vector<uint32_t> flags(c.size());
    cp_status st = cp_cone_colors(gpu_, nullptr, 0, c.data(), static_cast<uint32_t>(c.size()), CONE_WIDTH, colors.data(),
                                  nullptr, flags.data());
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    std::vector<Color> out;
    for (size_t i = 0; i < c.size(); ++i) {
      if (flags[i] & (CP_CONE_BAD_INDEX | CP_CONE_BAD_INTENSITY)) return std::vector<Color>();
      if (flags[i] & CP_CONE_EMPTY) continue;
      out.push_back(static_cast<Color>(colors[i] < kNumberOfColors ? colors[i] : 0));
    }
    return out;
  }
  enum Entry { kUnused, kPerMessage, kReplay };
  void use_entry(Entry e) {
    if (entry_ != kUnused && entry_ != e)
      throw GpuError(CP_E_STATE, "cloud_handler and replay keep separate node states: use one per ConeDetector");
    entry_ = e;
  }
  void replay_batch(const std::vector<PointCloud2>& msgs, size_t first, const std::vector<cp_cloud_view>& views,
                    std::vector<std::vector<PointCloud2>>* out) {
    cp_detect_params d{distance_treshold_max, distance_treshold_min, level_threshold, angle_threshold,
                       voxel_filter_leaf_size_x, voxel_filter_leaf_size_y, voxel_filter_leaf_size_z,
                       min_cluster_size, max_cluster_size, CONE_WIDTH, CONE_HEIGHT};
    cp_ground_params g{num_of_sectors, default_lowest_point};
    if (fused_ground_removal) apply_ground_model(gpu_);
    const uint32_t F = static_cast<uint32_t>(views.size());
    std::vector<uint32_t> k_off(F + 1);
    uint64_t K = 0;
    cp_status st = cp_detect_batch(gpu_, views.data(), F, &d, fused_ground_removal ? &g : nullptr, nullptr,
                                   k_off.data(), nullptr, 0, &K);
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    cp_track_params t{classify_colors ? 1 : 0, use_points_buffer ? 1 : 0, cones_matching_dist_theshold,
                      cone_position_extension_length, CONE_WIDTH};
    std::vector<cp_tracked_cone> cones(K);
    std::vector<uint32_t> coff(4 * static_cast<size_t>(F) + 1);
    uint64_t n = 0;
    st = cp_batch_track(gpu_, &t, nullptr, 1, cones.data(), coff.data(), K, &n);
    if (st != CP_OK) throw GpuError(st, cp_last_error(gpu_));
    for (uint32_t f = 0; f < F; ++f) {
      std::vector<PointCloud2> clouds(kNumberOfColors);
      for (int c = 0; c < kNumberOfColors; ++c) {
        std::vector<Point> pts;
        for (uint32_t j = coff[4 * f + c]; j < coff[4 * f + c + 1]; ++j) {
          Point p;
          p.x = cones[j].x;
          p.y = cones[j].y;
          p.z = 0.0;
          pts.push_back(p);
        }
        clouds[c] = to_msg(pts);  // :177-186
        clouds[c].header = msgs[first + f].header;
        clouds[c].fields = msgs[first + f].fields;  // Q6
      }
      out->push_back(std::move(clouds));
    }
  }
  cp_handle* gpu_ = nullptr;
  Entry entry_ = kUnused;
  uint64_t max_points_ = 0;
  uint32_t max_frames_ = 1;
  bool intensity_in_cloud_checked_ = false, intensity_in_cloud_ = true;
  std::vector<float> crop_buf_ = std::vector<float>(4 * 16384);
  std::vector<cp_cluster> clusters_;
  cp_frame_counters counters_{};
  ConeTracker tracker_;
};

}  // namespace cones_host
