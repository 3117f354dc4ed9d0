// mov_e.cpp — the ROS node of the reference (`mov_e`, src/external_sync_test.cpp:7-41) over the B200-native class.
//
// Same wiring as the reference node: ApproximateTime(queue 10) over the point cloud and odometry topics, the callback
// converts the message (pcl_conversions::toPCL), calls pushRawCloudAndPose + filterCloud and publishes `output`
// (external_sync_test.cpp:11-18), printing the milliseconds of the pair (:9, :20). Differences, all deliberate:
//   * topics, frame ids and the config path come from MOR_config.txt / argv instead of being hard-coded
//     (external_sync_test.cpp:31-32, :37 point at the author's home directory);
//   * the VISUALIZE side outputs (IncludeAll.h:32) - the debug cloud the reference publishes from inside
//     pushRawCloudAndPose (cpp:553-558) and the CUBE bounding-box markers it publishes from inside filterCloud
//     (cpp:640-642, mark_cluster cpp:7-58: lifetime 2 s, alpha 0.5, zero extents widened to 0.1) - are published here,
//     by the node, from clusterCollection() / movingMarkers(); the library never touches the caller's input cloud;
//   * `--keep-fields` publishes the filtered cloud in the input's own layout (ring, time ... kept: setKeepInputFields)
//     instead of pcl::PointXYZI, for deskewing consumers downstream.
// Build: only with ROS (catkin; -DMOR_WITH_ROS). Offline this file is type-checked against ros/stubs/ (tests/test_cpp_headers.py).
#ifdef MOR_WITH_ROS
#include <boost/bind.hpp>
#include <boost/shared_ptr.hpp>
#include <message_filters/subscriber.h>
#include <message_filters/sync_policies/approximate_time.h>
#include <message_filters/synchronizer.h>
#include <nav_msgs/Odometry.h>
#include <pcl_conversions/pcl_conversions.h>
#include <ros/ros.h>
#include <sensor_msgs/PointCloud2.h>
#include <visualization_msgs/Marker.h>

#include <chrono>
#include <iostream>

#include "MOR/MovingObjectRemoval.h"

static ros::Publisher pub, debug_pub, marker_pub;
static boost::shared_ptr<MovingObjectRemoval> mor;
static bool visualize = true;  // the reference defines VISUALIZE by default (IncludeAll.h:32)

// mark_cluster (cpp:7-58) from the per-cluster statistics the hot path keeps on the device
static visualization_msgs::Marker to_ros_marker(const mor_marker& m, const std::string& f_id) {
    visualization_msgs::Marker marker;
    marker.header.frame_id = f_id;
    marker.header.stamp = ros::Time::now();
    marker.ns = "bounding_box";
    marker.id = m.id;
    marker.type = visualization_msgs::Marker::CUBE;
    marker.action = visualization_msgs::Marker::ADD;
    marker.pose.position.x = m.position[0]; marker.pose.position.y = m.position[1]; marker.pose.position.z = m.position[2];
    marker.pose.orientation.x = 0.0; marker.pose.orientation.y = 0.0; marker.pose.orientation.z = 0.0; marker.pose.orientation.w = 1.0;
    marker.scale.x = m.scale[0]; marker.scale.y = m.scale[1]; marker.scale.z = m.scale[2];
    marker.color.r = m.color[0]; marker.color.g = m.color[1]; marker.color.b = m.color[2]; marker.color.a = m.color[3];
    marker.lifetime = ros::Duration(2);
    return marker;
}

void moving_object_test(const sensor_msgs::PointCloud2ConstPtr& input, const nav_msgs::OdometryConstPtr& odm) {
    const auto t0 = std::chrono::steady_clock::now();
    std::cout << "-----------------------------------------------------\n";
    pcl::PCLPointCloud2 cloud;
    pcl_conversions::toPCL(*input, cloud);

    mor->pushRawCloudAndPose(cloud, odm->pose.pose);
    if (visualize) {  // cpp:553-558
        pcl::PCLPointCloud2 debug_cloud;
        sensor_msgs::PointCloud2 debug_msg;
        if (mor->clusterCollection(debug_cloud)) {
            pcl_conversions::fromPCL(debug_cloud, debug_msg);
            debug_msg.header.frame_id = mor->config().debug_fid;
            debug_pub.publish(debug_msg);
        }
    }
    if (mor->filterCloud(cloud, mor->config().output_fid)) {
        pub.publish(mor->output);
        if (visualize) {  // cpp:640-642
            std::vector<mor_marker> markers;
            if (mor->movingMarkers(markers))
                for (const mor_marker& m : markers) marker_pub.publish(to_ros_marker(m, mor->config().debug_fid));
        }
    }
    std::cout << std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() << std::endl;
    std::cout << "-----------------------------------------------------\n";
}

int main(int argc, char** argv) {
    ros::init(argc, argv, "test_moving_object");
    ros::NodeHandle nh;
    std::string config_path = "config/MOR_config.txt";
    bool keep_fields = false;
    for (int i = 1; i < argc; i++) {
        if (std::string(argv[i]) == "--keep-fields") keep_fields = true;
        else config_path = argv[i];
    }
    mor.reset(new MovingObjectRemoval(nh, config_path, 4, 3));  // n_bad = 4, n_good = 3 as in external_sync_test.cpp:37
    if (keep_fields && !mor->setKeepInputFields(true)) { ROS_ERROR("setKeepInputFields: %s", mor_status_string(mor->lastStatus())); return 1; }
    const mor_config& cfg = mor->config();
    pub = nh.advertise<sensor_msgs::PointCloud2>(cfg.output_topic, 10);
    debug_pub = nh.advertise<sensor_msgs::PointCloud2>(cfg.debug_topic, 10);
    marker_pub = nh.advertise<visualization_msgs::Marker>(cfg.marker_topic, 10);

    message_filters::Subscriber<sensor_msgs::PointCloud2> pc_sub(nh, cfg.input_pointcloud_topic, 1);
    message_filters::Subscriber<nav_msgs::Odometry> odom_sub(nh, cfg.input_odometry_topic, 1);
    typedef message_filters::sync_policies::ApproximateTime<sensor_msgs::PointCloud2, nav_msgs::Odometry> MySyncPolicy;
    message_filters::Synchronizer<MySyncPolicy> sync(MySyncPolicy(10), pc_sub, odom_sub);
    sync.registerCallback(boost::bind(&moving_object_test, _1, _2));
    ros::spin();
    return 0;
}
#else
int main() { return 0; }  // built without ROS: see harness/mov_harness.cpp for the ROS-free equivalent
#endif
