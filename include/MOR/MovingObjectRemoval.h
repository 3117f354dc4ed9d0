// MOR/MovingObjectRemoval.h — drop-in C++ surface of the B200-native MOR hot path.
//
// Mirrors the reference class (prabinrath/dynamicslamtool include/MOR/MovingObjectRemoval.h:96-168):
//   MovingObjectRemoval(ros::NodeHandle, std::string config_path, int n_bad, int n_good)     .h:160
//   void pushRawCloudAndPose(pcl::PCLPointCloud2& cloud, geometry_msgs::Pose pose)           .h:163
//   bool filterCloud(pcl::PCLPointCloud2& cloud, std::string f_id)                           .h:166
//   sensor_msgs::PointCloud2 output                                                          .h:159
// Same names, argument order and call protocol (push, then filter, once per frame; README.md:16-29 and
// src/external_sync_test.cpp:11-18 of the reference). All work is done by the CUDA kernels behind the C ABI of
// include/mor_b200.h; the per-frame state the reference keeps in `ca`, `cb`, `mo_vec`, `corrs_vec`, `res_vec`
// (.h:109-128) lives in device memory inside the handle.
//
// ROS / PCL types: with -DMOR_WITH_ROS the real headers are used. Without it (this repository builds offline,
// ROS and PCL are not installed) field-compatible stand-ins are declared below, so the ROS-free harness and a
// real node compile against the same class.
//
// Differences from the reference, all on error paths (SURVEY.md §8b):
//   * a bad config throws std::runtime_error instead of calling exit(0) (cpp:703-707, :856-860);
//   * filterCloud returns false if the device reported an error or if the preceding pushRawCloudAndPose was rejected
//     (missing x/y/z field, frame larger than the handle's capacity ...): a node that publishes `output` whenever
//     filterCloud returns true (external_sync_test.cpp:15-18) then skips the frame instead of re-publishing the previous
//     one (the reference always returns true, cpp:695);
//   * the VISUALIZE side effects (debug cloud published and copied over the caller's input cloud at cpp:553-558,
//     bounding-box markers published at cpp:640-642) are not performed behind the caller's back: the same data is
//     available on request (clusterCollection, movingMarkers) for the node to publish; the input cloud is never
//     modified by pushRawCloudAndPose.
#ifndef MOR_MOVING_OBJECT_REMOVAL_H
#define MOR_MOVING_OBJECT_REMOVAL_H

#include <cstdint>
#include <string>
#include <vector>

#include "../mor_b200.h"

#ifdef MOR_WITH_ROS
#include <geometry_msgs/Pose.h>
#include <pcl/PCLPointCloud2.h>
#include <ros/ros.h>
#include <sensor_msgs/PointCloud2.h>
#else
namespace pcl {
struct PCLHeader { uint32_t seq = 0; uint64_t stamp = 0; std::string frame_id; };
struct PCLPointField {
    std::string name; uint32_t offset = 0; uint8_t datatype = 0; uint32_t count = 0;
    enum PointFieldTypes { INT8 = 1, UINT8 = 2, INT16 = 3, UINT16 = 4, INT32 = 5, UINT32 = 6, FLOAT32 = 7, FLOAT64 = 8 };
};
struct PCLPointCloud2 {
    PCLHeader header; uint32_t height = 0, width = 0; std::vector<PCLPointField> fields;
    uint8_t is_bigendian = 0; uint32_t point_step = 0, row_step = 0; std::vector<uint8_t> data; uint8_t is_dense = 0;
};
}  // namespace pcl
namespace geometry_msgs {
struct Point { double x = 0, y = 0, z = 0; };
struct Quaternion { double x = 0, y = 0, z = 0, w = 1; };
struct Pose { Point position; Quaternion orientation; };
}  // namespace geometry_msgs
namespace std_msgs { struct Header { uint32_t seq = 0; double stamp = 0; std::string frame_id; }; }
namespace sensor_msgs {
struct PointField { std::string name; uint32_t offset = 0; uint8_t datatype = 0; uint32_t count = 0; };
struct PointCloud2 {
    std_msgs::Header header; uint32_t height = 0, width = 0; std::vector<PointField> fields;
    uint8_t is_bigendian = 0; uint32_t point_step = 0, row_step = 0; std::vector<uint8_t> data; uint8_t is_dense = 0;
};
}  // namespace sensor_msgs
namespace ros { struct NodeHandle {}; }
#endif

class MovingObjectRemoval {
public:
    sensor_msgs::PointCloud2 output;  // the point cloud after the moving objects were removed (.h:159)

    // config_path: MOR_config.txt (same 23 keys as the reference); n_bad = moving_confidence, n_good = static_confidence
    MovingObjectRemoval(ros::NodeHandle nh, std::string config_path, int n_bad, int n_good);
    // extra: choose the CUDA device and the capacities (one object per sensor stream, one stream per object)
    MovingObjectRemoval(ros::NodeHandle nh, std::string config_path, int n_bad, int n_good, int device, const mor_limits* limits);
    ~MovingObjectRemoval();
    MovingObjectRemoval(const MovingObjectRemoval&) = delete;
    MovingObjectRemoval& operator=(const MovingObjectRemoval&) = delete;

    // Input: push the synchronised cloud + odometry pose (cpp:516-611). Asynchronous: returns once the H2D copy and
    // the kernels are enqueued. `cloud` is read-only here and must stay alive until filterCloud returns.
    void pushRawCloudAndPose(pcl::PCLPointCloud2& cloud, geometry_msgs::Pose pose);

    // Output: the filtered cloud (cloud minus confirmed moving clusters, plus the ground points) is written to `cloud`
    // and to `output` with header.frame_id = f_id (cpp:613-696).
    bool filterCloud(pcl::PCLPointCloud2& cloud, std::string f_id);

    // Off by default (PointXYZI output, cpp:690). On: from the next pushRawCloudAndPose, filterCloud publishes the kept
    // points as copies of their input records, with the pushed cloud's fields, point_step and is_bigendian (ring, time
    // and every other field kept; mor_set_output_records). Returns false (lastStatus()) while that cannot be changed.
    bool setKeepInputFields(bool keep);

    // The reference's VISUALIZE outputs, on request (nothing is computed unless these are called):
    // cb->cluster_collection as published on the debug topic (cpp:553-558), valid after pushRawCloudAndPose ...
    bool clusterCollection(pcl::PCLPointCloud2& debug_cloud);
    // ... and the bounding-box markers of the clusters the last filterCloud matched to mo_vec (cpp:640-642).
    bool movingMarkers(std::vector<mor_marker>& markers);

    mor_handle* handle() { return h_; }       // for the parity taps / device-resident calls of mor_b200.h
    const mor_config& config() const { return cfg_; }
    int lastStatus() const { return status_; }

private:
    mor_handle* h_ = nullptr;
    mor_config cfg_{};
    int status_ = MOR_OK;
    uint32_t n_in_ = 0;
    bool push_failed_ = false;    // the last pushRawCloudAndPose did not reach the device: filterCloud must not publish the frame before it
    bool keep_fields_ = false;    // setKeepInputFields
    // layout of the frame pushed last when it was pushed with keep_fields_ on (rec_step_ == 0: PointXYZI output)
    uint32_t rec_step_ = 0; uint8_t rec_bigendian_ = 0; std::vector<pcl::PCLPointField> rec_fields_;
    void* pinned_out_ = nullptr;  // page-locked staging (clusterCollection)
    size_t pinned_cap_ = 0;
    void* registered_ = nullptr;  // storage of output.data, page-locked in place: the D2H copy of filterCloud lands in the message itself
    void pin_output();
    void init(const std::string& path, int n_bad, int n_good, int device, const mor_limits* limits);
};

#endif  // MOR_MOVING_OBJECT_REMOVAL_H
