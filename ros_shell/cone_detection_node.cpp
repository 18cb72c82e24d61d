// cone_detection_node.cpp — drop-in for the reference's `cone_detection` executable
// (src/cone_detection.cpp): same node name, subscriber (queue 2), four publishers (queue 1),
// private parameter names (typos included) and colour service; crop -> VoxelGrid -> clustering
// -> centroid mean run on the GPU through cones_host::ConeDetector -> cp_detect.
// Build on a ROS Noetic box (see INTEGRATION.md).  In the build container (no ROS) it is compiled against the
// stand-in ROS surface of oracle/ref_shim and run next to the reference's own node (ros_shell/shim_harness.cpp).
#include "cones_perception/ClassifyColorSrv.h"
#include "ros_bridge.hpp"

class ConeDetectorNode {
 public:
  ConeDetectorNode() : nh_() {
    using cones_ros::private_param;
    private_param("cones_frame_id", core_.cones_frame_id);                                   // src/cone_detection.cpp:66
    private_param("classify_colors", core_.classify_colors);                                 // :69
    private_param("use_points_buffer", core_.use_points_buffer);                             // :72
    private_param("color_classifier_srv_name", color_classifier_srv_name_);                  // :75
    private_param("distance_treshold_max", core_.distance_treshold_max);                     // :78
    private_param("distance_treshold_min", core_.distance_treshold_min);                     // :81
    private_param("level_threshold", core_.level_threshold);                                 // :84
    private_param("angle_threshold", core_.angle_threshold);                                 // :87
    private_param("min_cluster_size", core_.min_cluster_size);                               // :90
    private_param("max_cluster_size", core_.max_cluster_size);                               // :93
    private_param("cones_matching_dist_theshold", core_.cones_matching_dist_theshold);       // :96
    private_param("cone_position_extension_length", core_.cone_position_extension_length);   // :99
    private_param("voxel_filter_leaf_size_x", core_.voxel_filter_leaf_size_x);               // :102
    private_param("voxel_filter_leaf_size_y", core_.voxel_filter_leaf_size_y);               // :105
    private_param("voxel_filter_leaf_size_z", core_.voxel_filter_leaf_size_z);               // :108
    // extension (off by default): run the ground_removal node's filter inside this process
    private_param("fused_ground_removal", core_.fused_ground_removal);
    private_param("num_of_sectors", core_.num_of_sectors);
    private_param("default_lowest_point", core_.default_lowest_point);
    // extension (default "sectors", the reference's model): with fused_ground_removal, "plane" removes the ground by a
    // seeded RANSAC plane per frame
    private_param("ground_model", core_.ground_model);
    private_param("plane_seed", core_.plane_seed);
    private_param("plane_hypotheses", core_.plane_hypotheses);
    private_param("plane_inlier_distance", core_.plane_inlier_distance);
    private_param("plane_ground_height", core_.plane_ground_height);
    private_param("plane_max_tilt_deg", core_.plane_max_tilt_deg);
    // extension (off by default): with fused_ground_removal, colour crops from the ground node's message, as the
    // detector of the two-node launch cuts them
    private_param("groundless_color_crops", core_.groundless_color_crops);
    // extension (off by default): the classifier network on the device instead of the color_classifier service;
    // the value is what the reference's launch file passes to the Python service as ~model_path
    std::string color_model_path;
    private_param("color_model_path", color_model_path);
    if (core_.classify_colors && !color_model_path.empty()) {
      core_.load_color_model(color_model_path);
      use_color_service_ = false;
    }
    sub_ = nh_.subscribe<sensor_msgs::PointCloud2>(core_.input_cloud_topic, 2, &ConeDetectorNode::cloud_handler, this);  // :112
    for (int i = 0; i < cones_host::kNumberOfColors; i++)
      pubs_[i] = nh_.advertise<sensor_msgs::PointCloud2>(core_.cones_topics[i], 1);          // :113-115
    if (core_.classify_colors && use_color_service_) {
      color_srv_client_ = nh_.serviceClient<cones_perception::ClassifyColorSrv>(color_classifier_srv_name_);  // :118
      core_.get_colors = [this](const std::vector<std::vector<cones_host::Point>>& crops) { return get_colors(crops); };
    }
  }
  void run() {
    if (core_.classify_colors && use_color_service_) color_srv_client_.waitForExistence();  // :123-125
    ROS_INFO("Ready to detect cones.");
    ros::spin();
  }

 private:
  void cloud_handler(const sensor_msgs::PointCloud2ConstPtr& cloud_msg) {
    try {
      auto clouds = core_.cloud_handler(cones_ros::from_ros(*cloud_msg));
      for (int i = 0; i < cones_host::kNumberOfColors; i++) pubs_[i].publish(cones_ros::to_ros(clouds[i]));
    } catch (const cones_host::GpuError& e) {
      ROS_ERROR("conesgpu: %s", e.what());
    }
  }
  // src/cone_detection.cpp:342-363
  std::vector<cones_host::Color> get_colors(const std::vector<std::vector<cones_host::Point>>& crops) {
    cones_perception::ClassifyColorSrv srv;
    for (const auto& crop : crops) {
      sensor_msgs::PointCloud2 m = cones_ros::to_ros(cones_host::to_msg(crop));
      m.header.frame_id = core_.cones_frame_id;
      srv.request.cones_clouds.push_back(m);
    }
    std::vector<cones_host::Color> colors(crops.size(), cones_host::kUnknownColor);
    if (color_srv_client_.call(srv)) {
      for (size_t i = 0; i < colors.size() && i < srv.response.colors.size(); ++i)
        colors[i] = static_cast<cones_host::Color>(srv.response.colors[i]);
    } else {
      ROS_ERROR("Failed to call service");
    }
    return colors;
  }
  ros::NodeHandle nh_;
  ros::Subscriber sub_;
  ros::Publisher pubs_[cones_host::kNumberOfColors];
  ros::ServiceClient color_srv_client_;
  std::string color_classifier_srv_name_ = "color_classifier";
  bool use_color_service_ = true;
  cones_host::ConeDetector core_;
};

int main(int argc, char* argv[]) {
  ros::init(argc, argv, "cone_detector");
  ConeDetectorNode node;
  node.run();
  return 0;
}
