// MovingObjectRemoval.cpp — host C++ class over the C ABI (see include/MOR/MovingObjectRemoval.h).
#include "../../include/MOR/MovingObjectRemoval.h"

#include <cstring>
#include <stdexcept>

namespace {

// pcl::fromPCLPointCloud2 maps fields by name (reference cpp:523, SURVEY A3); FLOAT32 only, like PointXYZI.
uint32_t find_field(const pcl::PCLPointCloud2& c, const char* name) {
    for (const auto& f : c.fields)
        if (f.name == name && f.datatype == 7 /*FLOAT32*/) return f.offset;
    return UINT32_MAX;
}

}  // namespace

void MovingObjectRemoval::init(const std::string& path, int n_bad, int n_good, int device, const mor_limits* limits) {
    status_ = mor_create_ex(path.c_str(), n_bad, n_good, device, limits, &h_);
    if (status_ != MOR_OK) throw std::runtime_error(std::string("MovingObjectRemoval: ") + mor_status_string(status_) + " (" + path + ")");
    mor_get_config(h_, &cfg_);
    // one pinned staging buffer for the largest frame the handle accepts: re-pinning when a larger frame shows
    // up costs tens of milliseconds
    mor_limits lim;
    mor_get_limits(h_, &lim);
    pinned_cap_ = (size_t)lim.max_points * 32;
    if (mor_alloc_pinned(pinned_cap_, &pinned_out_) != MOR_OK) {
        mor_destroy(h_); h_ = nullptr;
        throw std::runtime_error("MovingObjectRemoval: cannot pin the output staging buffer");
    }
    // `output` keeps one allocation for the largest frame, page-locked in place: filterCloud's D2H copy lands in the
    // message itself (no staging copy), and the vector never reallocates while it stays within this capacity
    output.data.reserve(pinned_cap_);
    pin_output();
}

void MovingObjectRemoval::pin_output() {
    if (registered_ == (void*)output.data.data()) return;
    if (registered_) mor_host_unregister(registered_);
    registered_ = nullptr;
    if (output.data.capacity() && mor_host_register(output.data.data(), output.data.capacity()) == MOR_OK) registered_ = output.data.data();
}

MovingObjectRemoval::MovingObjectRemoval(ros::NodeHandle, std::string config_path, int n_bad, int n_good) { init(config_path, n_bad, n_good, 0, nullptr); }
MovingObjectRemoval::MovingObjectRemoval(ros::NodeHandle, std::string config_path, int n_bad, int n_good, int device, const mor_limits* limits) {
    init(config_path, n_bad, n_good, device, limits);
}

MovingObjectRemoval::~MovingObjectRemoval() {
    if (registered_) mor_host_unregister(registered_);
    if (pinned_out_) mor_free_pinned(pinned_out_);
    mor_destroy(h_);
}

void MovingObjectRemoval::pushRawCloudAndPose(pcl::PCLPointCloud2& cloud, geometry_msgs::Pose pose) {
    const uint32_t ox = find_field(cloud, "x"), oy = find_field(cloud, "y"), oz = find_field(cloud, "z"), oi = find_field(cloud, "intensity");
    push_failed_ = true;
    if (ox == UINT32_MAX || oy == UINT32_MAX || oz == UINT32_MAX) { status_ = MOR_ERR_ARG; return; }  // PCL: "Failed to find match for field"
    const uint32_t n = cloud.width * cloud.height;
    const double p7[7] = {pose.position.x, pose.position.y, pose.position.z, pose.orientation.x, pose.orientation.y, pose.orientation.z, pose.orientation.w};
    n_in_ = n;
    status_ = mor_push_raw_cloud_and_pose(h_, cloud.data.data(), n, cloud.point_step, ox, oy, oz, oi, p7);
    push_failed_ = status_ != MOR_OK;
    rec_step_ = keep_fields_ ? cloud.point_step : 0;
    if (keep_fields_) { rec_fields_ = cloud.fields; rec_bigendian_ = cloud.is_bigendian; }
}

bool MovingObjectRemoval::setKeepInputFields(bool keep) {
    status_ = mor_set_output_records(h_, keep ? 1 : 0);
    if (status_ != MOR_OK) return false;
    keep_fields_ = keep;
    return true;
}

bool MovingObjectRemoval::filterCloud(pcl::PCLPointCloud2& out_cloud, std::string f_id) {
    if (push_failed_) return false;  // status_ keeps the reason; the frame before this one must not be published again
    // the records go straight into `output.data` (page-locked in place); the vector is sized to its capacity for the
    // copy and cut back to the frame's size afterwards (no reallocation, no zero fill beyond the first frame)
    if (output.data.capacity() < pinned_cap_) { output.data.reserve(pinned_cap_); }
    pin_output();
    if (output.data.size() < pinned_cap_) output.data.resize(pinned_cap_);
    uint32_t n_out = 0;
    status_ = mor_filter_cloud(h_, output.data.data(), (uint32_t)(pinned_cap_ / (rec_step_ ? rec_step_ : 32)), &n_out);
    if (status_ != MOR_OK) return false;
    output.header.seq = 0; output.header.frame_id = f_id;
    if (rec_step_) {  // the input records: the pushed cloud's layout
        const uint32_t st = rec_step_;
        output.height = 1; output.width = n_out; output.is_bigendian = rec_bigendian_; output.point_step = st; output.row_step = st * n_out; output.is_dense = 1;
        output.fields.resize(rec_fields_.size());
        for (size_t i = 0; i < rec_fields_.size(); i++) {
            output.fields[i].name = rec_fields_[i].name; output.fields[i].offset = rec_fields_[i].offset;
            output.fields[i].datatype = rec_fields_[i].datatype; output.fields[i].count = rec_fields_[i].count;
        }
        output.data.resize((size_t)n_out * st);
        out_cloud.header = pcl::PCLHeader();
        out_cloud.height = 1; out_cloud.width = n_out; out_cloud.is_bigendian = rec_bigendian_; out_cloud.point_step = st; out_cloud.row_step = st * n_out; out_cloud.is_dense = 1;
        out_cloud.fields = rec_fields_;
        out_cloud.data.assign(output.data.begin(), output.data.end());
        return true;
    }
    // pcl::toPCLPointCloud2 of a pcl::PointCloud<PointXYZI> (cpp:690): 32-byte records, fields x@0 y@4 z@8 intensity@16
    static const char* const names[4] = {"x", "y", "z", "intensity"};
    static const uint32_t offs[4] = {0, 4, 8, 16};
    // pcl_conversions::fromPCL(out_cloud, output); output.header.frame_id = f_id (cpp:691-692)
    output.height = 1; output.width = n_out; output.is_bigendian = 0; output.point_step = 32; output.row_step = 32 * n_out; output.is_dense = 1;
    output.fields.resize(4);
    for (int i = 0; i < 4; i++) { output.fields[i].name = names[i]; output.fields[i].offset = offs[i]; output.fields[i].datatype = 7; output.fields[i].count = 1; }
    output.data.resize((size_t)n_out * 32);  // shrinks: the storage (and its registration) stays
    out_cloud.header = pcl::PCLHeader();
    out_cloud.height = 1; out_cloud.width = n_out; out_cloud.is_bigendian = 0; out_cloud.point_step = 32; out_cloud.row_step = 32 * n_out; out_cloud.is_dense = 1;
    out_cloud.fields.resize(4);
    for (int i = 0; i < 4; i++) { out_cloud.fields[i].name = names[i]; out_cloud.fields[i].offset = offs[i]; out_cloud.fields[i].datatype = 7; out_cloud.fields[i].count = 1; }
    out_cloud.data.assign(output.data.begin(), output.data.end());  // the caller's cloud (cpp:690): the one host copy left
    return true;
}

bool MovingObjectRemoval::clusterCollection(pcl::PCLPointCloud2& debug_cloud) {
    uint32_t n = 0;
    status_ = mor_get_cluster_collection(h_, pinned_out_, (uint32_t)(pinned_cap_ / 32), &n);
    if (status_ != MOR_OK) return false;
    static const char* const names[4] = {"x", "y", "z", "intensity"};
    static const uint32_t offs[4] = {0, 4, 8, 16};
    debug_cloud.header = pcl::PCLHeader();
    debug_cloud.height = 1; debug_cloud.width = n; debug_cloud.is_bigendian = 0; debug_cloud.point_step = 32; debug_cloud.row_step = 32 * n; debug_cloud.is_dense = 1;
    debug_cloud.fields.resize(4);
    for (int i = 0; i < 4; i++) { debug_cloud.fields[i].name = names[i]; debug_cloud.fields[i].offset = offs[i]; debug_cloud.fields[i].datatype = 7; debug_cloud.fields[i].count = 1; }
    const uint8_t* rec = (const uint8_t*)pinned_out_;
    debug_cloud.data.assign(rec, rec + (size_t)n * 32);
    return true;
}

bool MovingObjectRemoval::movingMarkers(std::vector<mor_marker>& markers) {
    uint32_t n = 0;
    status_ = mor_get_moving_markers(h_, nullptr, 0, &n);
    if (status_ != MOR_OK) return false;
    markers.resize(n);
    if (n) status_ = mor_get_moving_markers(h_, markers.data(), n, &n);
    return status_ == MOR_OK;
}
