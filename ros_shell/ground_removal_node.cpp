// ground_removal_node.cpp — drop-in for the reference's `ground_removal` executable
// (src/ground_removal.cpp): same node name, topics, queue sizes and private parameters; the
// handler body runs on the GPU through cones_host::GroundRemover -> cp_ground_remove.
// Build on a ROS Noetic box (see INTEGRATION.md).  In the build container (no ROS) it is compiled against the
// stand-in ROS surface of oracle/ref_shim and run next to the reference's own node (ros_shell/shim_harness.cpp).
#include "ros_bridge.hpp"

class GroundRemoverNode {
 public:
  GroundRemoverNode() : nh_() {
    std::string out_topic = core_.groundless_cloud_topic;
    cones_ros::private_param("output_cloud_topic", out_topic);               // src/ground_removal.cpp:31
    cones_ros::private_param("num_of_sectors", core_.num_of_sectors);        // :34
    cones_ros::private_param("default_lowest_point", core_.default_lowest_point);  // :37
    // extension (default "sectors", the reference's model): "plane", a seeded RANSAC plane per frame
    cones_ros::private_param("ground_model", core_.ground_model);
    cones_ros::private_param("plane_seed", core_.plane_seed);
    cones_ros::private_param("plane_hypotheses", core_.plane_hypotheses);
    cones_ros::private_param("plane_inlier_distance", core_.plane_inlier_distance);
    cones_ros::private_param("plane_ground_height", core_.plane_ground_height);
    cones_ros::private_param("plane_max_tilt_deg", core_.plane_max_tilt_deg);
    sub_ = nh_.subscribe<sensor_msgs::PointCloud2>(core_.input_cloud_topic, 2, &GroundRemoverNode::cloud_handler, this);  // :41
    pub_ = nh_.advertise<sensor_msgs::PointCloud2>(out_topic, 1);            // :42
  }
  void run() {
    ROS_INFO("Ready to remove ground.");
    ros::spin();  // single-threaded: one thread uses the cp_handle
  }

 private:
  void cloud_handler(const sensor_msgs::PointCloud2ConstPtr& cloud_msg) {
    try {
      pub_.publish(cones_ros::to_ros(core_.cloud_handler(cones_ros::from_ros(*cloud_msg))));
    } catch (const cones_host::GpuError& e) {
      ROS_ERROR("conesgpu: %s", e.what());
    }
  }
  ros::NodeHandle nh_;
  ros::Subscriber sub_;
  ros::Publisher pub_;
  cones_host::GroundRemover core_;
};

int main(int argc, char* argv[]) {
  ros::init(argc, argv, "ground_remover");
  GroundRemoverNode node;
  node.run();
  return 0;
}
