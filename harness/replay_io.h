// replay_io.h — recorded-data front end of the ROS-free harness (host only).
//
// The reference node receives `sensor_msgs::PointCloud2` + `nav_msgs::Odometry` pairs from a bag
// (src/external_sync_test.cpp:24-41). Offline the same pairs usually exist as a KITTI-style directory:
//
//   <dir>/000000.bin, 000001.bin, ...   (or <dir>/velodyne/*.bin) float32 x,y,z,reflectance records, 16 B each;
//                                        the blob goes to pushRawCloudAndPose as it is (fields x@0 y@4 z@8
//                                        intensity@12, point_step 16) - no conversion pass on the host
//   <dir>/poses.txt                      one line per frame, any of
//                                          7 numbers  tx ty tz qx qy qz qw            (geometry_msgs::Pose order)
//                                          8 numbers  t tx ty tz qx qy qz qw          (TUM trajectory)
//                                          12 numbers r00 r01 r02 tx r10 ... r22 tz   (KITTI odometry, row-major 3x4)
//   <dir>/calib.txt (optional)           a line "Tr: <12 numbers>" (KITTI: velodyne -> camera). KITTI poses are poses
//                                        of the camera; the sensor pose is then Tr^-1 * P * Tr.
#pragma once
#include <dirent.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

namespace replay {

struct Mat34 { double m[12]; };  // row-major [R | t]

inline Mat34 mul(const Mat34& a, const Mat34& b) {
    Mat34 c;
    for (int r = 0; r < 3; r++) {
        for (int k = 0; k < 3; k++) c.m[4 * r + k] = a.m[4 * r] * b.m[k] + a.m[4 * r + 1] * b.m[4 + k] + a.m[4 * r + 2] * b.m[8 + k];
        c.m[4 * r + 3] = a.m[4 * r] * b.m[3] + a.m[4 * r + 1] * b.m[7] + a.m[4 * r + 2] * b.m[11] + a.m[4 * r + 3];
    }
    return c;
}

inline Mat34 inverse_rigid(const Mat34& a) {
    Mat34 c;
    for (int r = 0; r < 3; r++)
        for (int k = 0; k < 3; k++) c.m[4 * r + k] = a.m[4 * k + r];
    for (int r = 0; r < 3; r++) c.m[4 * r + 3] = -(c.m[4 * r] * a.m[3] + c.m[4 * r + 1] * a.m[7] + c.m[4 * r + 2] * a.m[11]);
    return c;
}

// Rotation matrix -> unit quaternion, largest-component branch (numerically stable for every rotation).
inline void to_pose7(const Mat34& a, double p7[7]) {
    const double r00 = a.m[0], r01 = a.m[1], r02 = a.m[2], r10 = a.m[4], r11 = a.m[5], r12 = a.m[6], r20 = a.m[8], r21 = a.m[9], r22 = a.m[10];
    double x, y, z, w;
    const double tr = r00 + r11 + r22;
    if (tr > 0) {
        const double s = std::sqrt(tr + 1.0) * 2;
        w = 0.25 * s; x = (r21 - r12) / s; y = (r02 - r20) / s; z = (r10 - r01) / s;
    } else if (r00 > r11 && r00 > r22) {
        const double s = std::sqrt(1.0 + r00 - r11 - r22) * 2;
        w = (r21 - r12) / s; x = 0.25 * s; y = (r01 + r10) / s; z = (r02 + r20) / s;
    } else if (r11 > r22) {
        const double s = std::sqrt(1.0 + r11 - r00 - r22) * 2;
        w = (r02 - r20) / s; x = (r01 + r10) / s; y = 0.25 * s; z = (r12 + r21) / s;
    } else {
        const double s = std::sqrt(1.0 + r22 - r00 - r11) * 2;
        w = (r10 - r01) / s; x = (r02 + r20) / s; y = (r12 + r21) / s; z = 0.25 * s;
    }
    p7[0] = a.m[3]; p7[1] = a.m[7]; p7[2] = a.m[11];
    p7[3] = x; p7[4] = y; p7[5] = z; p7[6] = w;
}

inline std::vector<double> numbers_of(const std::string& line) {
    std::vector<double> v;
    std::istringstream ss(line);
    std::string tok;
    while (ss >> tok) {
        char* end = nullptr;
        const double d = std::strtod(tok.c_str(), &end);
        if (end == tok.c_str() || *end) { v.clear(); return v; }  // not a numeric line
        v.push_back(d);
    }
    return v;
}

// One pose7 per line of poses.txt; `calib` (may be null) is Tr of calib.txt. Returns false on a malformed line.
inline bool read_poses(const std::string& path, const Mat34* calib, std::vector<std::array<double, 7>>& out, std::string& err) {
    std::ifstream f(path);
    if (!f) { err = "cannot open " + path; return false; }
    Mat34 tr_inv{};
    if (calib) tr_inv = inverse_rigid(*calib);
    std::string line;
    int ln = 0;
    while (std::getline(f, line)) {
        ln++;
        if (line.empty() || line[0] == '#') continue;
        const std::vector<double> v = numbers_of(line);
        std::array<double, 7> p{};
        if (v.size() == 7) std::copy(v.begin(), v.end(), p.begin());
        else if (v.size() == 8) std::copy(v.begin() + 1, v.end(), p.begin());
        else if (v.size() == 12) {
            Mat34 m;
            std::copy(v.begin(), v.end(), m.m);
            if (calib) m = mul(mul(tr_inv, m), *calib);
            to_pose7(m, p.data());
        } else { err = path + ":" + std::to_string(ln) + ": expected 7, 8 or 12 numbers"; return false; }
        out.push_back(p);
    }
    return true;
}

// First number of every data line (seconds); with `columns` > 0 only lines of exactly that many numbers count.
inline bool read_stamps(const std::string& path, size_t columns, std::vector<double>& out) {
    std::ifstream f(path);
    if (!f) return false;
    std::string line;
    while (std::getline(f, line)) {
        if (line.empty() || line[0] == '#') continue;
        const std::vector<double> v = numbers_of(line);
        if (v.empty() || (columns && v.size() != columns)) return false;
        out.push_back(v[0]);
    }
    return !out.empty();
}

// Feeds two stamped streams to a synchroniser in the order a bag player would deliver them (by stamp; topic 0 first on ties).
template <class Sync>
inline void feed_in_arrival_order(Sync& sync, const std::vector<double>& ta, size_t na, const std::vector<double>& tb, size_t nb) {
    size_t i = 0, j = 0;
    auto ns = [](double t) { return (int64_t)std::llround(t * 1e9); };
    while (i < na || j < nb) {
        if (j >= nb || (i < na && ta[i] <= tb[j])) { sync.add(0, ns(ta[i]), (int)i); i++; }
        else { sync.add(1, ns(tb[j]), (int)j); j++; }
    }
}

inline bool read_calib(const std::string& path, Mat34& tr) {
    std::ifstream f(path);
    std::string line;
    while (f && std::getline(f, line)) {
        if (line.rfind("Tr:", 0) == 0 || line.rfind("Tr ", 0) == 0) {
            const std::vector<double> v = numbers_of(line.substr(3));
            if (v.size() == 12) { std::copy(v.begin(), v.end(), tr.m); return true; }
        }
    }
    return false;
}

inline std::vector<std::string> list_bins(const std::string& dir) {
    std::vector<std::string> names;
    if (DIR* d = opendir(dir.c_str())) {
        while (dirent* e = readdir(d)) {
            const std::string n = e->d_name;
            if (n.size() > 4 && n.compare(n.size() - 4, 4, ".bin") == 0) names.push_back(dir + "/" + n);
        }
        closedir(d);
    }
    std::sort(names.begin(), names.end());
    return names;
}

// Reads a whole .bin into `blob` (bytes, a multiple of 16); returns the number of points or -1.
inline long read_bin(const std::string& path, std::vector<uint8_t>& blob) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) return -1;
    std::fseek(f, 0, SEEK_END);
    const long bytes = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    if (bytes < 0 || bytes % 16) { std::fclose(f); return -1; }
    blob.resize((size_t)bytes);
    const size_t got = bytes ? std::fread(blob.data(), 1, (size_t)bytes, f) : 0;
    std::fclose(f);
    return got == (size_t)bytes ? bytes / 16 : -1;
}

inline bool write_bin(const std::string& path, const uint8_t* records32, uint32_t n) {
    // PointXYZI records (32 B: x y z _ intensity _ _ _) back to the 16-byte x,y,z,intensity wire format
    std::vector<float> out((size_t)n * 4);
    for (uint32_t i = 0; i < n; i++) {
        const float* r = reinterpret_cast<const float*>(records32 + (size_t)i * 32);
        out[4 * i] = r[0]; out[4 * i + 1] = r[1]; out[4 * i + 2] = r[2]; out[4 * i + 3] = r[4];
    }
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = std::fwrite(out.data(), 16, n, f) == n;
    std::fclose(f);
    return ok;
}

// Output records in the input's own layout (--keep-fields): written as they are.
inline bool write_records(const std::string& path, const uint8_t* records, size_t bytes) {
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = std::fwrite(records, 1, bytes, f) == bytes;
    std::fclose(f);
    return ok;
}

}  // namespace replay
