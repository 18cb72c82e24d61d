// host_c_api.cpp — a small C surface over the C++ host classes (nodes.hpp) so that pytest can
// drive them through ctypes.  Not part of the drop-in boundary (that is include/conesgpu.h).
#include <cstdio>
#include <map>
#include <string>

#include "nodes.hpp"

using namespace cones_host;

namespace {
std::string g_err;

PointCloud2 make_msg(const float* xyzi, uint32_t n, int with_intensity_field, uint32_t sec, uint32_t nsec) {
  PointCloud2 m;
  m.header.seq = 7;
  m.header.stamp_sec = sec;
  m.header.stamp_nsec = nsec;
  m.header.frame_id = "cloud";
  m.height = 1;
  m.width = n;
  m.point_step = 16;
  m.row_step = 16 * n;
  m.fields.resize(with_intensity_field ? 4 : 3);
  const char* names[4] = {"x", "y", "z", "intensity"};
  for (size_t i = 0; i < m.fields.size(); ++i) {
    m.fields[i].name = names[i];
    m.fields[i].offset = static_cast<uint32_t>(4 * i);
  }
  m.data.resize(static_cast<size_t>(n) * 16);
  if (n) std::memcpy(m.data.data(), xyzi, static_cast<size_t>(n) * 16);
  return m;
}

// messages 0..n_msgs-1 of a series: compact xyzi, frame_n[i] points each, stamps 100 + i s, 123456789 + i ns
std::vector<PointCloud2> make_msgs(const float* xyzi, const uint32_t* frame_n, uint32_t n_msgs, int with_intensity_field) {
  std::vector<PointCloud2> msgs;
  size_t at = 0;
  for (uint32_t i = 0; i < n_msgs; ++i) {
    msgs.push_back(make_msg(xyzi + 4 * at, frame_n[i], with_intensity_field, 100 + i, 123456789 + i));
    at += frame_n[i];
  }
  return msgs;
}

// a published message, serialised field by field: header, layout, fields, data
void serialise(const PointCloud2& m, std::vector<uint8_t>* b) {
  auto put = [b](const void* p, size_t n) { b->insert(b->end(), static_cast<const uint8_t*>(p), static_cast<const uint8_t*>(p) + n); };
  put(&m.header.seq, 4); put(&m.header.stamp_sec, 4); put(&m.header.stamp_nsec, 4);
  put(m.header.frame_id.data(), m.header.frame_id.size());
  put(&m.height, 4); put(&m.width, 4);
  for (const PointField& f : m.fields) {
    put(f.name.data(), f.name.size()); put(&f.offset, 4); put(&f.datatype, 1); put(&f.count, 4);
  }
  put(&m.is_bigendian, 1); put(&m.point_step, 4); put(&m.row_step, 4);
  put(m.data.data(), m.data.size()); put(&m.is_dense, 1);
}

int copy_out(const std::vector<uint8_t>& b, uint8_t* out, uint64_t cap, uint64_t* used) {
  *used = b.size();
  if (b.size() > cap) return 3;
  if (!b.empty()) std::memcpy(out, b.data(), b.size());
  return 0;
}
}  // namespace

extern "C" {

const char* ch_last_error(void) { return g_err.c_str(); }

// ---- ConeTracker (no GPU needed) ---------------------------------------------------------
void* ch_tracker_create(int classify_colors, int use_points_buffer, double match_dist, double extension) {
  auto* t = new ConeTracker();
  t->classify_colors = classify_colors != 0;
  t->use_points_buffer = use_points_buffer != 0;
  t->cones_matching_dist_theshold = match_dist;
  t->cone_position_extension_length = extension;
  return t;
}
void ch_tracker_destroy(void* t) { delete static_cast<ConeTracker*>(t); }

// forced_color >= 0: the colour "service" answers with that colour for every crop
int ch_tracker_update(void* tp, const float* xy, uint32_t n, int forced_color, float* out_xy, uint32_t* counts,
                      uint32_t cap) {
  auto* t = static_cast<ConeTracker*>(tp);
  std::vector<std::pair<float, float>> c(n);
  for (uint32_t i = 0; i < n; ++i) c[i] = {xy[2 * i], xy[2 * i + 1]};
  if (forced_color >= 0)
    t->get_colors = [forced_color](const std::vector<std::vector<Point>>& crops) {
      return std::vector<Color>(crops.size(), static_cast<Color>(forced_color));
    };
  std::vector<Point> whole;
  auto clouds = t->update(c, &whole);
  for (int k = 0; k < kNumberOfColors; ++k) {
    counts[k] = static_cast<uint32_t>(clouds[k].size());
    if (clouds[k].size() > cap) return 3;
    for (size_t i = 0; i < clouds[k].size(); ++i) {
      out_xy[(static_cast<size_t>(k) * cap + i) * 2] = clouds[k][i].x;
      out_xy[(static_cast<size_t>(k) * cap + i) * 2 + 1] = clouds[k][i].y;
    }
  }
  return 0;
}

// colour mode with per-record service answers (cp_batch_cone_colors output for this frame's n records): the need list
// is mapped back to records by the exact bits of their extended centres, then the response rules of
// ConeDetector::gpu_colors apply (a bad crop: no answer at all; empty crops skipped)
int ch_tracker_update_answers(void* tp, const float* xy, uint32_t n, const uint8_t* colors, const uint32_t* flags,
                              float* out_xy, uint32_t* counts, uint32_t cap) {
  auto* t = static_cast<ConeTracker*>(tp);
  std::vector<std::pair<float, float>> c(n);
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> index;
  for (uint32_t i = 0; i < n; ++i) {
    c[i] = {xy[2 * i], xy[2 * i + 1]};
    Point p;
    p.x = c[i].first;
    p.y = c[i].second;
    float vector_len = euclidan_dist(p.x, p.y, p.z, 0, 0, 0);  // as ConeTracker::update
    p.x = p.x + p.x / vector_len * t->cone_position_extension_length;
    p.y = p.y + p.y / vector_len * t->cone_position_extension_length;
    uint32_t bx, by;
    std::memcpy(&bx, &p.x, 4);
    std::memcpy(&by, &p.y, 4);
    index.emplace(std::make_pair(bx, by), i);
  }
  t->classify_centers = [&](const std::vector<Point>& need) {
    std::vector<Color> out;
    for (const Point& p : need) {
      uint32_t bx, by;
      std::memcpy(&bx, &p.x, 4);
      std::memcpy(&by, &p.y, 4);
      const uint32_t k = index.at({bx, by});
      if (flags[k] & (CP_CONE_BAD_INDEX | CP_CONE_BAD_INTENSITY)) return std::vector<Color>();
      if (flags[k] & CP_CONE_EMPTY) continue;
      out.push_back(static_cast<Color>(colors[k] < kNumberOfColors ? colors[k] : 0));
    }
    return out;
  };
  auto clouds = t->update(c, nullptr);
  t->classify_centers = nullptr;
  for (int k = 0; k < kNumberOfColors; ++k) {
    counts[k] = static_cast<uint32_t>(clouds[k].size());
    if (clouds[k].size() > cap) return 3;
    for (size_t i = 0; i < clouds[k].size(); ++i) {
      out_xy[(static_cast<size_t>(k) * cap + i) * 2] = clouds[k][i].x;
      out_xy[(static_cast<size_t>(k) * cap + i) * 2 + 1] = clouds[k][i].y;
    }
  }
  return 0;
}

// ---- ConeDetector / GroundRemover (GPU) -----------------------------------------------------
}  // extern "C"
namespace {
// A deterministic stand-in for the color_classifier service, so the three colour-input modes can be
// compared: colour = 1 + fnv1a(bytes) % 3; empty crops are skipped like the service does
// (scripts/color_classifier_server.py:83-84), which shortens the answer.
uint64_t fnv1a(const void* data, size_t n, uint64_t h = 1469598103934665603ull) {
  const uint8_t* b = static_cast<const uint8_t*>(data);
  for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}
struct ColorProbe {
  uint64_t n_inputs = 0, n_points = 0, digest = 1469598103934665603ull;
};
std::vector<Color> probe_crops(ColorProbe* pr, const std::vector<std::vector<Point>>& crops) {
  std::vector<Color> out;
  for (const auto& c : crops) {
    pr->n_inputs++;
    if (c.empty()) continue;
    uint64_t h = 1469598103934665603ull;
    for (const Point& p : c) {
      const float v[4] = {p.x, p.y, p.z, p.intensity};
      h = fnv1a(v, sizeof(v), h);
    }
    pr->n_points += c.size();
    pr->digest = fnv1a(&h, sizeof(h), pr->digest);
    out.push_back(static_cast<Color>(1 + h % 3));
  }
  return out;
}
std::vector<Color> probe_images(ColorProbe* pr, const std::vector<uint8_t>& images, const std::vector<uint32_t>& flags) {
  std::vector<Color> out;
  for (size_t i = 0; i < flags.size(); ++i) {
    pr->n_inputs++;
    if (flags[i] & CP_CONE_EMPTY) continue;
    const uint64_t h = fnv1a(images.data() + i * 180, 180);
    pr->digest = fnv1a(&h, sizeof(h), pr->digest);
    out.push_back(static_cast<Color>(1 + h % 3));
  }
  return out;
}
std::map<void*, ColorProbe> g_probes;
}  // namespace
extern "C" {

// mode: ConeDetector::ColorInputs (0 host crops, 1 GPU crops, 2 GPU crops + range images)
void ch_detector_set_color_inputs(void* dp, int mode) {
  auto* det = static_cast<ConeDetector*>(dp);
  det->color_inputs = static_cast<ConeDetector::ColorInputs>(mode);
  ColorProbe* pr = &g_probes[dp];
  det->get_colors = [pr](const std::vector<std::vector<Point>>& crops) { return probe_crops(pr, crops); };
  det->get_colors_from_images = [pr](const std::vector<uint8_t>& im, const std::vector<uint32_t>& fl) {
    return probe_images(pr, im, fl);
  };
}
// the classifier network on the device (ConeDetector::kGpuColors): model = bytes of the .tflite file
int ch_detector_load_color_model(void* dp, const void* model, uint64_t bytes) {
  try {
    static_cast<ConeDetector*>(dp)->load_color_model(model, static_cast<size_t>(bytes));
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 4;
  }
}
// ConeDetector::groundless_color_crops
void ch_detector_set_groundless_color_crops(void* dp, int on) {
  static_cast<ConeDetector*>(dp)->groundless_color_crops = on != 0;
}
void ch_detector_color_probe(void* dp, uint64_t* n_inputs, uint64_t* n_points, uint64_t* digest) {
  const ColorProbe& pr = g_probes[dp];
  *n_inputs = pr.n_inputs;
  *n_points = pr.n_points;
  *digest = pr.digest;
}

}  // extern "C"
namespace {
void* create_detector(uint64_t max_points, uint32_t max_frames, int device, const cp_detect_params* d,
                      int classify_colors, int use_points_buffer, int fused_ground) {
  try {
    auto* det = new ConeDetector(max_points, device, 32, max_frames);
    det->distance_treshold_max = d->distance_treshold_max;
    det->distance_treshold_min = d->distance_treshold_min;
    det->level_threshold = d->level_threshold;
    det->angle_threshold = d->angle_threshold;
    det->voxel_filter_leaf_size_x = d->voxel_filter_leaf_size_x;
    det->voxel_filter_leaf_size_y = d->voxel_filter_leaf_size_y;
    det->voxel_filter_leaf_size_z = d->voxel_filter_leaf_size_z;
    det->min_cluster_size = d->min_cluster_size;
    det->max_cluster_size = d->max_cluster_size;
    det->classify_colors = classify_colors != 0;
    det->use_points_buffer = use_points_buffer != 0;
    det->fused_ground_removal = fused_ground != 0;
    return det;
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}
}  // namespace
extern "C" {

void* ch_detector_create(uint64_t max_points, int device, const cp_detect_params* d, int classify_colors,
                         int use_points_buffer, int fused_ground) {
  return create_detector(max_points, 1, device, d, classify_colors, use_points_buffer, fused_ground);
}
void ch_detector_destroy(void* d) {
  g_probes.erase(d);
  delete static_cast<ConeDetector*>(d);
}

// one callback: compact xyzi cloud in, the four published clouds out (x, y per cone) plus the
// layout facts of the published messages
int ch_detector_handle(void* dp, const float* xyzi, uint32_t n, int with_intensity_field, float* out_xy,
                       uint32_t* counts, uint32_t cap, uint32_t* out_point_step, uint32_t* out_n_fields,
                       uint32_t* out_stamp_nsec) {
  try {
    auto* det = static_cast<ConeDetector*>(dp);
    PointCloud2 msg = make_msg(xyzi, n, with_intensity_field, 100, 123456789);
    auto clouds = det->cloud_handler(msg);
    for (int k = 0; k < kNumberOfColors; ++k) {
      counts[k] = clouds[k].width;
      if (clouds[k].width > cap) return 3;
      for (uint32_t i = 0; i < clouds[k].width; ++i) {
        float xy[2];
        std::memcpy(xy, clouds[k].data.data() + static_cast<size_t>(i) * clouds[k].point_step, 8);
        out_xy[(static_cast<size_t>(k) * cap + i) * 2] = xy[0];
        out_xy[(static_cast<size_t>(k) * cap + i) * 2 + 1] = xy[1];
      }
    }
    *out_point_step = clouds[0].point_step;
    *out_n_fields = static_cast<uint32_t>(clouds[0].fields.size());
    *out_stamp_nsec = clouds[0].header.stamp_nsec;
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 4;
  }
}

// ConeDetector::replay: messages 0..n_msgs-1 (compact xyzi, frame_n[i] points each) in device batches of up to
// max_frames.  ch_detector_publish: the same messages through replay (replay != 0) or through cloud_handler, one call
// per message; out receives every published message serialised (header, layout, fields, data), 4 per input message.
void* ch_detector_create_replay(uint64_t max_points, uint32_t max_frames, int device, const cp_detect_params* d,
                                int classify_colors, int use_points_buffer, int fused_ground) {
  return create_detector(max_points, max_frames, device, d, classify_colors, use_points_buffer, fused_ground);
}

int ch_detector_publish(void* dp, const float* xyzi, const uint32_t* frame_n, uint32_t n_msgs, int with_intensity_field,
                        int replay, uint8_t* out, uint64_t cap, uint64_t* used) {
  try {
    auto* det = static_cast<ConeDetector*>(dp);
    std::vector<PointCloud2> msgs = make_msgs(xyzi, frame_n, n_msgs, with_intensity_field);
    std::vector<std::vector<PointCloud2>> pub;
    if (replay) {
      pub = det->replay(msgs);
    } else {
      for (const PointCloud2& m : msgs) pub.push_back(det->cloud_handler(m));
    }
    std::vector<uint8_t> b;
    for (const auto& clouds : pub)
      for (const PointCloud2& m : clouds) serialise(m, &b);
    return copy_out(b, out, cap, used);
  } catch (const std::exception& e) {
    g_err = e.what();
    return 4;
  }
}

void* ch_ground_create(uint64_t max_points, int device) {
  try {
    return new GroundRemover(max_points, device, 32);
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}
void ch_ground_destroy(void* g) { delete static_cast<GroundRemover*>(g); }

// GroundRemover::replay in device batches of up to max_frames messages.  ch_ground_publish: messages 0..n_msgs-1
// (compact xyzi, frame_n[i] points each) through replay (replay != 0) or through cloud_handler, one call per
// message; out receives every published message serialised as ch_detector_publish does, one per input message.
void* ch_ground_create_replay(uint64_t max_points, uint32_t max_frames, int device) {
  try {
    return new GroundRemover(max_points, device, 32, max_frames);
  } catch (const std::exception& e) {
    g_err = e.what();
    return nullptr;
  }
}

int ch_ground_publish(void* gp, const float* xyzi, const uint32_t* frame_n, uint32_t n_msgs, int with_intensity_field,
                      int replay, uint8_t* out, uint64_t cap, uint64_t* used) {
  try {
    auto* gr = static_cast<GroundRemover*>(gp);
    std::vector<PointCloud2> msgs = make_msgs(xyzi, frame_n, n_msgs, with_intensity_field);
    std::vector<PointCloud2> pub;
    if (replay) {
      pub = gr->replay(msgs);
    } else {
      for (const PointCloud2& m : msgs) pub.push_back(gr->cloud_handler(m));
    }
    std::vector<uint8_t> b;
    for (const PointCloud2& m : pub) serialise(m, &b);
    return copy_out(b, out, cap, used);
  } catch (const std::exception& e) {
    g_err = e.what();
    return 4;
  }
}

// the node parameters ~ground_model (plane != 0: "plane", else "sectors") and ~plane_* of either node (nodes.hpp
// GroundModelParams); read at the next message
namespace {
void set_ground_model(GroundModelParams* m, int plane, int seed, int hypotheses, double inlier_distance,
                      double ground_height, double max_tilt_deg) {
  m->ground_model = plane ? "plane" : "sectors";
  m->plane_seed = seed;
  m->plane_hypotheses = hypotheses;
  m->plane_inlier_distance = inlier_distance;
  m->plane_ground_height = ground_height;
  m->plane_max_tilt_deg = max_tilt_deg;
}
}  // namespace
void ch_ground_set_ground_model(void* gp, int plane, int seed, int hypotheses, double inlier_distance,
                                double ground_height, double max_tilt_deg) {
  set_ground_model(static_cast<GroundRemover*>(gp), plane, seed, hypotheses, inlier_distance, ground_height,
                   max_tilt_deg);
}
void ch_detector_set_ground_model(void* dp, int plane, int seed, int hypotheses, double inlier_distance,
                                  double ground_height, double max_tilt_deg) {
  set_ground_model(static_cast<ConeDetector*>(dp), plane, seed, hypotheses, inlier_distance, ground_height,
                   max_tilt_deg);
}

int ch_ground_handle(void* gp, const float* xyzi, uint32_t n, int with_intensity_field, void* out32,
                     uint32_t* kept, uint32_t* out_point_step, uint32_t* out_stamp_nsec, uint32_t* out_n_fields) {
  try {
    auto* gr = static_cast<GroundRemover*>(gp);
    PointCloud2 msg = make_msg(xyzi, n, with_intensity_field, 100, 123456789);
    PointCloud2 out = gr->cloud_handler(msg);
    std::memcpy(out32, out.data.data(), out.data.size());
    *kept = gr->last_kept();
    *out_point_step = out.point_step;
    *out_stamp_nsec = out.header.stamp_nsec;
    *out_n_fields = static_cast<uint32_t>(out.fields.size());
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 4;
  }
}

}  // extern "C"
