// mov_harness.cpp — ROS-free stand-in for the reference node `mov_e` (src/external_sync_test.cpp:7-41).
//
// The reference callback converts the incoming message, calls pushRawCloudAndPose + filterCloud, publishes
// `output` and prints the milliseconds the pair took (external_sync_test.cpp:9-20). This harness does the same
// with frames from the seeded synthetic generator instead of ROS topics, and adds a CRC of every output cloud so
// runs can be compared across implementations.
//
//   mov_harness <MOR_config.txt> <scenario 1..4> <seed> <frames> [n_bad=4] [n_good=3] [--quiet]
//   mov_harness <MOR_config.txt> --replay <dir> [frames] [n_bad=4] [n_good=3] [--quiet] [--out <dir>] [--keep-fields]
//       (either form: --stream replays through mor_submit_frame / mor_collect_frame with pipelined launches: full rate, results three frames late)
//       (either form: --debug also fetches the VISUALIZE debug cloud and bounding-box markers of every frame)
//       recorded data: KITTI-style .bin clouds + poses.txt (+ calib.txt), see replay_io.h; --out writes the filtered clouds
//       unsynchronised recording: <dir>/times.txt (one stamp in seconds per cloud) + <dir>/odometry.txt (t tx ty tz qx qy qz qw,
//       its own stamps and rate) instead of poses.txt: cloud and odometry are paired like the reference node pairs its two
//       topics, message_filters ApproximateTime with queue 10 (src/external_sync_test.cpp:31-35; approx_time.h)
//   mov_harness --inspect <dir>                 the frames and poses --replay would feed (host only)
//   mov_harness --pair <stamps A> <stamps B> [queue=10]   the pairs ApproximateTime selects for two stamp files (host only)
//   mov_harness --pose-of <12 numbers>          the pose7 the replay front end derives from a 3x4 matrix (host only)
#include <malloc.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../dynamicslamtool_b200/csrc/mor_synth.h"
#include "../include/MOR/MovingObjectRemoval.h"
#include "approx_time.h"
#include "replay_io.h"

static uint32_t crc32_buf(const uint8_t* p, size_t n) {
    static uint32_t table[256];
    static bool init = false;
    if (!init) {
        for (uint32_t i = 0; i < 256; i++) { uint32_t c = i; for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1; table[i] = c; }
        init = true;
    }
    uint32_t c = 0xFFFFFFFFu;
    for (size_t i = 0; i < n; i++) c = table[(c ^ p[i]) & 0xFF] ^ (c >> 8);
    return c ^ 0xFFFFFFFFu;
}

// Where the frames come from: the seeded generator or a directory of recorded clouds + poses.
struct FrameSource {
    mor_synth* syn = nullptr;
    std::vector<std::string> bins;
    std::vector<std::array<double, 7>> poses;
    uint32_t max_points = 0;
    std::vector<float> buf;

    bool open_synth(int scenario, uint64_t seed) {
        if (mor_synth_create(scenario, seed, &syn)) return false;
        mor_synth_info(syn, &max_points, nullptr, nullptr);
        buf.resize((size_t)max_points * 4);
        return true;
    }
    bool open_replay(const std::string& dir, std::string& err) {
        bins = replay::list_bins(dir);
        if (bins.empty()) bins = replay::list_bins(dir + "/velodyne");
        if (bins.empty()) { err = "no .bin clouds in " + dir; return false; }
        replay::Mat34 tr;
        const bool have_calib = replay::read_calib(dir + "/calib.txt", tr);
        std::vector<double> cloud_t, odom_t;
        if (replay::read_stamps(dir + "/times.txt", 0, cloud_t) && replay::read_stamps(dir + "/odometry.txt", 8, odom_t)) {
            // independently stamped streams: pair them like the reference node does (ApproximateTime, queue 10)
            std::vector<std::array<double, 7>> odom;
            if (!replay::read_poses(dir + "/odometry.txt", nullptr, odom, err)) return false;
            if (cloud_t.size() < bins.size()) bins.resize(cloud_t.size());
            std::vector<std::string> paired_bins;
            replay::ApproximateTime<2> sync(10, [&](const replay::ApproximateTime<2>::Msg (&m)[2]) {
                paired_bins.push_back(bins[m[0].index]);
                poses.push_back(odom[m[1].index]);
            });
            replay::feed_in_arrival_order(sync, cloud_t, bins.size(), odom_t, odom.size());
            bins.swap(paired_bins);
        } else {
            if (!replay::read_poses(dir + "/poses.txt", have_calib ? &tr : nullptr, poses, err)) return false;
            if (poses.size() < bins.size()) bins.resize(poses.size());  // a cloud without a pose cannot be processed
        }
        for (const std::string& b : bins) {
            FILE* f = std::fopen(b.c_str(), "rb");
            if (!f) { err = "cannot open " + b; return false; }
            std::fseek(f, 0, SEEK_END);
            max_points = std::max<uint32_t>(max_points, (uint32_t)(std::ftell(f) / 16));
            std::fclose(f);
        }
        return true;
    }
    size_t frames() const { return syn ? SIZE_MAX : bins.size(); }
    // fills cloud.data / width / row_step and p7
    bool frame(uint32_t f, pcl::PCLPointCloud2& cloud, double p7[7]) {
        uint32_t n = 0;
        if (syn) {
            if (mor_synth_frame(syn, f, buf.data(), max_points, &n, p7, 8)) return false;
            cloud.data.assign((const uint8_t*)buf.data(), (const uint8_t*)buf.data() + (size_t)n * 16);
        } else {
            const long got = replay::read_bin(bins[f], cloud.data);
            if (got < 0) return false;
            n = (uint32_t)got;
            std::copy(poses[f].begin(), poses[f].end(), p7);
        }
        cloud.width = n; cloud.row_step = 16 * n;
        return true;
    }
    ~FrameSource() { if (syn) mor_synth_destroy(syn); }
};

int main(int argc, char** argv) {
    if (argc >= 14 && !std::strcmp(argv[1], "--pose-of")) {
        replay::Mat34 m;
        for (int i = 0; i < 12; i++) m.m[i] = std::atof(argv[2 + i]);
        double p7[7];
        replay::to_pose7(m, p7);
        std::printf("%.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", p7[0], p7[1], p7[2], p7[3], p7[4], p7[5], p7[6]);
        return 0;
    }
    if (argc >= 4 && !std::strcmp(argv[1], "--pair")) {
        std::vector<double> ta, tb;
        if (!replay::read_stamps(argv[2], 0, ta) || !replay::read_stamps(argv[3], 0, tb)) { std::fprintf(stderr, "cannot read the stamp files\n"); return 2; }
        replay::ApproximateTime<2> sync(argc > 4 ? (uint32_t)std::atoi(argv[4]) : 10u, [&](const replay::ApproximateTime<2>::Msg (&m)[2]) {
            std::printf("pair %d %d\n", m[0].index, m[1].index);
        });
        replay::feed_in_arrival_order(sync, ta, ta.size(), tb, tb.size());
        return 0;
    }
    if (argc >= 3 && !std::strcmp(argv[1], "--inspect")) {  // what --replay would feed, without touching a GPU
        FrameSource src;
        std::string err;
        if (!src.open_replay(argv[2], err)) { std::fprintf(stderr, "%s\n", err.c_str()); return 2; }
        std::printf("frames %zu max_points %u\n", src.frames(), src.max_points);
        pcl::PCLPointCloud2 cloud;
        for (size_t f = 0; f < src.frames(); f++) {
            double p7[7];
            if (!src.frame((uint32_t)f, cloud, p7)) { std::fprintf(stderr, "frame %zu: cannot read the cloud\n", f); return 1; }
            std::printf("frame %zu points %u pose %.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", f, cloud.width, p7[0], p7[1], p7[2], p7[3], p7[4], p7[5], p7[6]);
        }
        return 0;
    }
    if (argc < 4) { std::fprintf(stderr, "usage: %s <config> <scenario> <seed> <frames> [n_bad] [n_good] [--quiet]\n       %s <config> --replay <dir> [frames] [n_bad] [n_good] [--quiet] [--out <dir>] [--keep-fields]\n", argv[0], argv[0]); return 2; }
    const std::string cfg = argv[1];
    const bool replay_mode = !std::strcmp(argv[2], "--replay");
    bool quiet = false, debug = false, stream = false, keep_fields = false;  // --debug: also fetch the VISUALIZE outputs (debug cloud, markers) every frame
    std::string out_dir;
    std::vector<std::string> pos;  // positional arguments after the source
    for (int i = replay_mode ? 4 : 2; i < argc; i++) {
        if (!std::strcmp(argv[i], "--quiet")) quiet = true;
        else if (!std::strcmp(argv[i], "--debug")) debug = true;
        else if (!std::strcmp(argv[i], "--stream")) stream = true;  // replay through the pipelined calls (results arrive three frames late)
        else if (!std::strcmp(argv[i], "--out") && i + 1 < argc) out_dir = argv[++i];
        else if (!std::strcmp(argv[i], "--keep-fields")) keep_fields = true;  // output = the input records (mor_set_output_records)
        else pos.push_back(argv[i]);
    }
    FrameSource src;
    int frames = 0;
    size_t next = 0;
    if (replay_mode) {
        std::string err;
        if (!src.open_replay(argv[3], err)) { std::fprintf(stderr, "%s\n", err.c_str()); return 2; }
        frames = (int)src.frames();
        if (pos.size() > next) frames = std::min(frames, std::atoi(pos[next++].c_str()));
    } else {
        if (pos.size() < 3) { std::fprintf(stderr, "scenario, seed and frame count expected\n"); return 2; }
        if (!src.open_synth(std::atoi(pos[0].c_str()), std::strtoull(pos[1].c_str(), nullptr, 10))) { std::fprintf(stderr, "bad scenario\n"); return 2; }
        frames = std::atoi(pos[2].c_str());
        next = 3;
    }
    const int n_bad = pos.size() > next ? std::atoi(pos[next].c_str()) : 4, n_good = pos.size() > next + 1 ? std::atoi(pos[next + 1].c_str()) : 3;

    // The callback allocates and frees ~6 MB of cloud buffers per frame (its local PCLPointCloud2, as in the
    // reference). With glibc's defaults those are mapped and unmapped every time (0.25 ms of page faults per MB on
    // the bench host); keep them in the heap instead.
    mallopt(M_MMAP_THRESHOLD, 32 << 20);
    mallopt(M_TRIM_THRESHOLD, 512 << 20);

    mor_limits lim{};
    lim.max_points = std::max<uint32_t>(src.max_points, 1);
    ros::NodeHandle nh;
    MovingObjectRemoval mor(nh, cfg, n_bad, n_good, 0, &lim);  // mor.reset(new MovingObjectRemoval(nh, "...MOR_config.txt", 4, 3))

    if (stream) {
        // Replay at full rate (mor_b200.h, "pipelined streaming"): the frames go through mor_submit_frame / mor_collect_frame on
        // the class's handle with pipelined launches; four pinned input and output buffers; frame f is collected - and would
        // be published - when frame f+3 has been submitted. Same per-frame lines as the callback loop below.
        mor_handle* h = mor.handle();
        if (mor_set_pipelining(h, 1) != MOR_OK) { std::fprintf(stderr, "mor_set_pipelining: %s\n", mor_last_error(h)); return 1; }
        if (keep_fields && mor_set_output_records(h, 1) != MOR_OK) { std::fprintf(stderr, "mor_set_output_records: %s\n", mor_last_error(h)); return 1; }
        const size_t rec_bytes = keep_fields ? 16 : 32;  // bytes per output point
        const size_t cap = lim.max_points;
        void* in[MOR_STREAM_DEPTH]; void* out[MOR_STREAM_DEPTH]; uint32_t n_of[MOR_STREAM_DEPTH];
        for (int q = 0; q < MOR_STREAM_DEPTH; q++)
            if (mor_alloc_pinned(cap * 16, &in[q]) != MOR_OK || mor_alloc_pinned(cap * 32, &out[q]) != MOR_OK) { std::fprintf(stderr, "pinned allocation failed\n"); return 1; }
        pcl::PCLPointCloud2 c16;
        c16.height = 1; c16.point_step = 16; c16.is_dense = 1;
        const auto t_begin = std::chrono::steady_clock::now();
        int collected = 0;
        auto collect_one = [&]() -> bool {
            uint32_t n_out = 0;
            const int st = mor_collect_frame(h, &n_out);
            if (st != MOR_OK) { std::fprintf(stderr, "frame %d: %s %s\n", collected, mor_status_string(st), mor_last_error(h)); return false; }
            const int q = collected % MOR_STREAM_DEPTH;
            if (!out_dir.empty()) {
                char name[32];
                std::snprintf(name, sizeof name, "/%06d.bin", collected);
                const bool ok = keep_fields ? replay::write_records(out_dir + name, (const uint8_t*)out[q], (size_t)n_out * rec_bytes)
                                            : replay::write_bin(out_dir + name, (const uint8_t*)out[q], n_out);
                if (!ok) { std::fprintf(stderr, "cannot write %s%s\n", out_dir.c_str(), name); return false; }
            }
            if (!quiet) std::printf("frame %d in %u out %u crc %08x ms 0\n", collected, n_of[q], n_out, crc32_buf((const uint8_t*)out[q], (size_t)n_out * rec_bytes));
            collected++;
            return true;
        };
        for (int f = 0; f < frames; f++) {
            double p7[7];
            if (!src.frame((uint32_t)f, c16, p7)) { std::fprintf(stderr, "frame %d: cannot read the cloud\n", f); return 1; }
            const int q = f % MOR_STREAM_DEPTH;
            if (f - collected >= MOR_STREAM_DEPTH && !collect_one()) return 1;  // the slot's previous frame must be out first
            n_of[q] = c16.width;
            std::memcpy(in[q], c16.data.data(), (size_t)c16.width * 16);
            const int st = mor_submit_frame(h, in[q], c16.width, 16, 0, 4, 8, 12, p7, out[q], (uint32_t)cap);
            if (st != MOR_OK) { std::fprintf(stderr, "frame %d: %s %s\n", f, mor_status_string(st), mor_last_error(h)); return 1; }
        }
        while (collected < frames) if (!collect_one()) return 1;
        const double total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        std::printf("summary frames %d mean_ms %.3f fps %.1f (streamed: wall clock incl. reading / generating the frames)\n", frames, total_ms / std::max(frames, 1), 1e3 * frames / total_ms);
        for (int q = 0; q < MOR_STREAM_DEPTH; q++) { mor_free_pinned(in[q]); mor_free_pinned(out[q]); }
        return 0;
    }

    pcl::PCLPointCloud2 cloud;  // what pcl_conversions::toPCL(*input, cloud) would hand over: 16-byte x,y,z,intensity records
    cloud.height = 1; cloud.point_step = 16; cloud.is_dense = 1;
    const char* names[4] = {"x", "y", "z", "intensity"};
    for (int i = 0; i < 4; i++) { pcl::PCLPointField f; f.name = names[i]; f.offset = 4 * i; f.datatype = 7; f.count = 1; cloud.fields.push_back(f); }
    if (keep_fields && !mor.setKeepInputFields(true)) { std::fprintf(stderr, "setKeepInputFields: %s\n", mor_status_string(mor.lastStatus())); return 1; }
    std::vector<double> ms;
    double stage_ms[3] = {0, 0, 0};  // callback copy, pushRawCloudAndPose, filterCloud (frames after the fifth)
    for (int f = 0; f < frames; f++) {
        double p7[7];
        if (!src.frame((uint32_t)f, cloud, p7)) { std::fprintf(stderr, "frame %d: cannot read the cloud\n", f); return 1; }
        const uint32_t n = cloud.width;
        geometry_msgs::Pose pose;
        pose.position.x = p7[0]; pose.position.y = p7[1]; pose.position.z = p7[2];
        pose.orientation.x = p7[3]; pose.orientation.y = p7[4]; pose.orientation.z = p7[5]; pose.orientation.w = p7[6];

        const auto t0 = std::chrono::steady_clock::now();
        pcl::PCLPointCloud2 work = cloud;  // the callback's own copy (external_sync_test.cpp:11-12)
        const auto t1 = std::chrono::steady_clock::now();
        mor.pushRawCloudAndPose(work, pose);
        const auto t2 = std::chrono::steady_clock::now();
        pcl::PCLPointCloud2 debug_cloud;
        if (debug && !mor.clusterCollection(debug_cloud)) { std::fprintf(stderr, "frame %d: %s\n", f, mor_status_string(mor.lastStatus())); return 1; }  // cpp:553-558
        const bool ok = mor.filterCloud(work, "/filtered");
        const auto t3 = std::chrono::steady_clock::now();
        const double dt = std::chrono::duration<double, std::milli>(t3 - t0).count();
        if (f >= 5) {
            stage_ms[0] += std::chrono::duration<double, std::milli>(t1 - t0).count();
            stage_ms[1] += std::chrono::duration<double, std::milli>(t2 - t1).count();
            stage_ms[2] += std::chrono::duration<double, std::milli>(t3 - t2).count();
        }
        if (!ok) { std::fprintf(stderr, "frame %d: %s\n", f, mor_status_string(mor.lastStatus())); return 1; }
        ms.push_back(dt);
        if (!out_dir.empty()) {
            char name[32];
            std::snprintf(name, sizeof name, "/%06d.bin", f);
            const bool ok = keep_fields ? replay::write_records(out_dir + name, mor.output.data.data(), mor.output.data.size())
                                        : replay::write_bin(out_dir + name, mor.output.data.data(), mor.output.width);
            if (!ok) { std::fprintf(stderr, "cannot write %s%s\n", out_dir.c_str(), name); return 1; }
        }
        if (debug) {
            std::vector<mor_marker> markers;
            if (!mor.movingMarkers(markers)) { std::fprintf(stderr, "frame %d: %s\n", f, mor_status_string(mor.lastStatus())); return 1; }
            std::printf("debug %d clustered %u crc %08x markers %zu", f, debug_cloud.width, crc32_buf(debug_cloud.data.data(), debug_cloud.data.size()), markers.size());
            for (const mor_marker& m : markers) std::printf(" [cluster %d scale %.9g %.9g %.9g]", m.cluster, m.scale[0], m.scale[1], m.scale[2]);
            std::printf("\n");
        }
        if (!quiet) std::printf("frame %d in %u out %u crc %08x ms %.3f\n", f, n, mor.output.width, crc32_buf(mor.output.data.data(), mor.output.data.size()), dt);
    }
    if (ms.size() > 5) {
        std::vector<double> s(ms.begin() + 5, ms.end());
        std::sort(s.begin(), s.end());
        double sum = 0;
        for (double v : s) sum += v;
        std::printf("summary frames %zu mean_ms %.3f p50_ms %.3f p99_ms %.3f fps %.1f\n", s.size(), sum / s.size(), s[s.size() / 2], s[(size_t)(s.size() * 0.99)], 1e3 * s.size() / sum);
        std::printf("stages copy_ms %.3f push_ms %.3f filter_ms %.3f\n", stage_ms[0] / s.size(), stage_ms[1] / s.size(), stage_ms[2] / s.size());
    }
    return 0;
}
