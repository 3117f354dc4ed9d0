/*
 * mor_b200.h — C ABI of the B200-native MOR (Moving Object Removal) per-frame filtering hot path.
 *
 * This is the drop-in boundary between host code (the C++ `MovingObjectRemoval` class in
 * include/MOR/MovingObjectRemoval.h, a ROS callback, a ctypes/cffi binding ...) and the
 * hand-written sm_100a kernels. Plain pointers and sizes only; every function returns an int
 * status (mor_status); nothing here ever calls exit().
 *
 * Each entry point cites the reference interface it replaces (paths relative to the upstream
 * prabinrath/dynamicslamtool tree):
 *
 *   mor_create                    <- MovingObjectRemoval::MovingObjectRemoval(nh, config_path, n_bad, n_good)
 *                                    include/MOR/MovingObjectRemoval.h:160, src/MovingObjectRemoval.cpp:368-391
 *                                    + setVariables, src/MovingObjectRemoval.cpp:698-864
 *   mor_push_raw_cloud_and_pose   <- MovingObjectRemoval::pushRawCloudAndPose(pcl::PCLPointCloud2&, geometry_msgs::Pose)
 *                                    include/MOR/MovingObjectRemoval.h:163, src/MovingObjectRemoval.cpp:516-611
 *   mor_filter_cloud              <- MovingObjectRemoval::filterCloud(pcl::PCLPointCloud2&, std::string f_id) + `output`
 *                                    include/MOR/MovingObjectRemoval.h:159,166, src/MovingObjectRemoval.cpp:613-696
 *   mor_destroy                   <- ~MovingObjectRemoval (implicit)
 *
 * The *_device variants take/return device pointers (point data stays resident in HBM); the
 * mor_tap / mor_get_* functions expose every per-frame intermediate for the parity tests.
 *
 * The CPU oracle (oracle/mor_oracle.cpp, test infrastructure only) exports the same functions with
 * the prefix `oracle_` instead of `mor_` and identical signatures, so tests drive both through one
 * binding.
 */
#ifndef MOR_B200_H
#define MOR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mor_handle mor_handle;

typedef enum mor_status {
    MOR_OK = 0,
    MOR_ERR_CONFIG_OPEN = 1,    /* reference: "Couldnt open the file" + exit(0), cpp:703-707 */
    MOR_ERR_CONFIG_KEY = 2,     /* reference: "Invalid parameter found in config file" + exit(0), cpp:856-860 */
    MOR_ERR_CONFIG_VALUE = 3,   /* reference: std::stof/stol/stoi throws (uncaught) */
    MOR_ERR_CONFIG_MISSING = 4, /* reference: member left uninitialised (UB); here a defined error */
    MOR_ERR_ARG = 5,
    MOR_ERR_CAPACITY = 6,       /* frame larger than the handle's device buffers / grid too large */
    MOR_ERR_CUDA = 7,
    MOR_ERR_STATE = 8           /* e.g. filter before any push */
} mor_status;

/* Ground-removal mode. The reference hard-codes mode 0 (cpp:526); mode 1 is its commented-out,
 * crashing voxel-covariance path (cpp:527, cpp:90-200) with the repairs listed in DESIGN.md;
 * mode 2 is the eigen-normal generalisation (no reference behaviour). Selected with the optional
 * config key `ground_mode` (absent => 0). */
enum { MOR_GROUND_CROP = 0, MOR_GROUND_VOXEL_COV = 1, MOR_GROUND_VOXEL_EIGEN = 2 };

/* Optional capacities; zero fields take defaults. */
typedef struct mor_limits {
    uint32_t max_points;    /* largest frame accepted (default 300000) */
    uint32_t max_clusters;  /* largest number of size-valid clusters per frame (default 8192, at most 16384) */
    uint32_t max_moving;    /* capacity of the confirmed-moving list mo_vec (default 1024) */
    uint32_t max_cells;     /* voxel ground modes only (ground_mode 1/2): largest dense voxel / ball-query table over the
                               bounding box of a frame's raw cloud (default 2^24 cells; a frame that needs more is
                               MOR_ERR_CAPACITY). The clustering grid is a sparse hash grid with no such limit: neither
                               the crop box nor the radius enters its size */
    uint32_t reserved[4];
} mor_limits;

/* The 23 MOR_config.txt keys (config/MOR_config.txt:1-39) + extension keys, as parsed. */
typedef struct mor_config {
    float gp_limit, gp_leaf, bin_gap, volume_constraint, pde_lb, pde_ub, leave_off_distance,
        catch_up_distance, trim_x, trim_y, trim_z, ec_distance_threshold, pde_distance_threshold;
    int64_t min_cluster_size, max_cluster_size;
    int32_t method_choice, opc_normalization_factor;
    int32_t ground_mode;       /* extension, default 0 */
    float gp_planarity;        /* extension (mode 2), default 0.01 */
    float gp_bin_width;        /* extension (mode 2), default = gp_leaf */
    int32_t n_bad, n_good;     /* ctor args: moving_confidence, static_confidence */
    char output_topic[64], debug_topic[64], marker_topic[64], input_pointcloud_topic[64],
        input_odometry_topic[64], output_fid[64], debug_fid[64];
} mor_config;

/* ---- lifecycle ------------------------------------------------------------------------- */
int mor_create(const char* config_path, int n_bad, int n_good, int device, mor_handle** out);
int mor_create_ex(const char* config_path, int n_bad, int n_good, int device,
                  const mor_limits* limits, mor_handle** out);
int mor_destroy(mor_handle* h);
/* Back to the state of a freshly created handle (no frames seen, nothing tracked): what destroying the reference
 * object and constructing a new one does (cpp:368-391), without re-allocating. For replaying several sequences. */
int mor_reset(mor_handle* h);
int mor_get_config(const mor_handle* h, mor_config* out);
int mor_get_limits(const mor_handle* h, mor_limits* out); /* the capacities in effect (defaults filled in) */
const char* mor_status_string(int status);
const char* mor_last_error(const mor_handle* h);

/* Parse a MOR_config.txt without creating a handle (host only; same grammar as cpp:698-864). */
int mor_parse_config(const char* config_path, mor_config* out);

/* ---- per-frame hot path, host buffers --------------------------------------------------- */
/* `data` = n points, point i at data + i*point_step; float32 fields at the given byte offsets
 * (the PCLPointCloud2 fields named x, y, z, intensity: pcl::fromPCLPointCloud2, cpp:523).
 * off_i == UINT32_MAX => no intensity field (intensity 0, as PCL does).
 * pose7 = position x,y,z then orientation x,y,z,w (geometry_msgs::Pose), doubles.
 * n <= mor_limits.max_points, and n * point_step <= 32 B x max_points (the device staging buffer; records wider than
 * 32 bytes need a proportionally larger max_points), else MOR_ERR_CAPACITY.
 * Asynchronous: returns after enqueueing the H2D copy and the kernels on the handle's stream. */
int mor_push_raw_cloud_and_pose(mor_handle* h, const void* data, uint32_t n, uint32_t point_step,
                                uint32_t off_x, uint32_t off_y, uint32_t off_z, uint32_t off_i,
                                const double pose7[7]);

/* Writes the filtered cloud as pcl::PointXYZI wire records (32 B/point: x@0 y@4 z@8 1.0f@12
 * intensity@16, zero pad; pcl::toPCLPointCloud2, cpp:690) into `out` (capacity cap_points) and
 * the count into *n_out. Synchronous (the D2H copy completes before return).
 * Returns MOR_ERR_CAPACITY (and the needed count in *n_out) if cap_points is too small. */
int mor_filter_cloud(mor_handle* h, void* out, uint32_t cap_points, uint32_t* n_out);

/* ---- per-frame hot path, device-resident ------------------------------------------------ */
/* Same as above but `d_data` / `d_out` are device pointers on the handle's device; no PCIe
 * traffic except the 7 pose doubles. mor_filter_cloud_device with n_out == NULL does not
 * synchronise (read the count later with mor_sync + mor_tap(MOR_TAP_COUNTS)). */
int mor_push_raw_cloud_and_pose_device(mor_handle* h, const void* d_data, uint32_t n,
                                       uint32_t point_step, uint32_t off_x, uint32_t off_y,
                                       uint32_t off_z, uint32_t off_i, const double pose7[7]);
int mor_filter_cloud_device(mor_handle* h, void* d_out, uint32_t cap_points, uint32_t* n_out);
/* Zero-copy: mor_filter_cloud_device(h, NULL, 0, n_out or NULL) leaves the records in the handle's own device buffer;
 * this returns its address (valid until the next push on the handle). */
int mor_get_output_device(mor_handle* h, const void** d_records);
int mor_sync(mor_handle* h);

/* Batched device-resident step (BASELINE config 5: many independent sequences per GPU): one pushRawCloudAndPose +
 * filterCloud for S sequences in ONE launch of the frame kernel (a group of CTAs per sequence). With the voxel ground
 * modes (ground_mode 1 / 2) the ground stage of all S frames runs first, as 9 launches whatever S (S <= 65535). All
 * handles must live on the same device with the same config (ground_mode included), limits and frame count.
 * d_data[s] / d_out[s] are device pointers (d_out[s] must hold n[s] records), poses7 = S x 7 doubles. Asynchronous on
 * hs[0]'s stream; mor_sync / mor_tap on any of the handles waits for it. */
int mor_batch_step_device(mor_handle* const* hs, uint32_t S, const void* const* d_data, const uint32_t* n,
                          uint32_t point_step, uint32_t off_x, uint32_t off_y, uint32_t off_z, uint32_t off_i,
                          const double* poses7, void* const* d_out);

/* ---- pipelined streaming, host buffers (replay of recorded data / throughput) ------------- */
/* One frame of the callback body of the reference's node (external_sync_test.cpp:9-21: pushRawCloudAndPose, then
 * filterCloud, then publish `output`) as two calls that do not wait for the device in between:
 *   mor_submit_frame  enqueues the frame's H2D copy, its frame kernel and the D2H copy of the filtered cloud, each on a
 *                     stream of its own (copies of frame f+1 and f-1 overlap the kernel of frame f), and returns;
 *   mor_collect_frame waits for the OLDEST submitted frame and delivers its count: `out` of that frame then holds the
 *                     records mor_filter_cloud would have written.
 * At most MOR_STREAM_DEPTH (4) frames may be in flight; a fifth mor_submit_frame returns MOR_ERR_STATE. `data` must stay
 * untouched until the frame is collected and `out` (capacity cap_points records, >= n to be safe) until it has been
 * read; both should be pinned (mor_alloc_pinned / mor_host_register), else the copies do not overlap anything.
 * Every submitted frame is committed like push + one filterCloud (the tracker update of cpp:630-671 is applied once).
 * The synchronous calls above may be mixed in only while no frame is in flight (MOR_ERR_STATE otherwise).
 * mor_collect_frame returns MOR_ERR_STATE if nothing is in flight, MOR_ERR_CAPACITY (count in *n_out) if cap_points was
 * too small or a device-side capacity was exceeded (mor_last_error tells which). */
#define MOR_STREAM_DEPTH 4
int mor_submit_frame(mor_handle* h, const void* data, uint32_t n, uint32_t point_step, uint32_t off_x, uint32_t off_y,
                     uint32_t off_z, uint32_t off_i, const double pose7[7], void* out, uint32_t cap_points);
int mor_collect_frame(mor_handle* h, uint32_t* n_out);
/* Throughput mode for callers that hand frames over ahead of needing their results (replay; the device-resident calls with
 * n_out == NULL; the streaming calls above): clustering a frame needs nothing of the frame before it, so the back half of
 * frame f (pose transform, correspondences, moving test, chain, filterCloud's part) is launched together with the front
 * half of frame f+1 (ingest ... cluster statistics), in ONE kernel on disjoint groups of SMs, instead of one after the
 * other. Results are identical; a call that needs a frame's results (count, taps, host output) runs its back half at
 * once. Applies to method_choice 2 with the crop ground mode; ignored otherwise. Off by default. */
int mor_set_pipelining(mor_handle* h, int enabled);
/* Frames submitted and not yet collected (0..MOR_STREAM_DEPTH). */
int mor_frames_in_flight(const mor_handle* h, uint32_t* out);

/* cudaMallocHost / cudaFreeHost passthroughs so callers can stage frames in pinned memory. */
int mor_alloc_pinned(size_t bytes, void** out);
int mor_free_pinned(void* p);
/* cudaHostRegister / cudaHostUnregister passthroughs: page-lock memory the caller already owns (e.g. the storage of the
 * message a ROS node publishes), so that mor_filter_cloud copies straight into it at full PCIe rate. */
int mor_host_register(void* p, size_t bytes);
int mor_host_unregister(void* p);
/* Plain device buffer helpers for harnesses that keep frames resident (cudaMalloc/Memcpy/Free). */
int mor_device_alloc(int device, size_t bytes, void** out);
int mor_device_free(int device, void* p);
int mor_device_upload(int device, void* d_dst, const void* src, size_t bytes);
int mor_device_download(int device, void* dst, const void* d_src, size_t bytes);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches), and device time
 * (ms, CUDA events on the handle's stream) of the last push / filter call. */
int mor_get_launch_count(const mor_handle* h, uint64_t* out);
int mor_get_last_device_ms(mor_handle* h, float* push_ms, float* filter_ms);
/* Enable per-call CUDA-event timing (adds two event records per call). */
int mor_set_timing(mor_handle* h, int enabled);

/* Event slots (0..7) recorded on the handle's stream, so callers can time a region of calls on the
 * device: mor_event_record(h, 0); ...calls...; mor_event_record(h, 1); mor_event_elapsed_ms(h, 0, 1, &ms). */
int mor_event_record(mor_handle* h, int slot);
int mor_event_elapsed_ms(mor_handle* h, int slot_a, int slot_b, float* ms);
/* Per-kernel profiling: every launch of the hot path is bracketed by CUDA events; totals are read
 * back with mor_get_kernel_profile(h, index, ...) for index = 0.. until it returns MOR_ERR_ARG.
 * Forces a stream synchronisation per frame; never enable it inside a throughput measurement. */
int mor_set_kernel_profiling(mor_handle* h, int enabled);
int mor_get_kernel_profile(mor_handle* h, int index, char name[32], double* total_ms, uint64_t* launches);
/* The frame kernel's own timeline (always recorded: one %globaltimer store per phase): microseconds the last frame spent
 * in each of its phases, group barrier included. *n_phases receives the number of phases; names by mor_phase_name. */
int mor_get_phase_times(mor_handle* h, float* us, int cap, int* n_phases);
const char* mor_phase_name(int index);

/* ---- the reference's VISUALIZE outputs (IncludeAll.h:32), on request ---------------------- */
/* cb->cluster_collection as published on the debug topic (cpp:226-229, :553-558): the points of all size-valid
 * clusters, cluster after cluster in cluster order, ascending cloud index inside a cluster; 32-byte pcl::PointXYZI
 * records like mor_filter_cloud. Valid after mor_push_raw_cloud_and_pose. out == NULL: only the count. */
int mor_get_cluster_collection(mor_handle* h, void* out, uint32_t cap_points, uint32_t* n_out);
/* One bounding-box marker per mo_vec entry the last mor_filter_cloud looked up, in mo_vec order (marker_pub,
 * cpp:640-642; mark_cluster, cpp:7-58), from the per-cluster statistics kept on the device. `position` is the
 * cluster centroid of the hot path (double sums rounded to float; the reference's marker uses a float-accumulated
 * centroid, equal to ~1e-6 relative), `scale` the exact bounding-box extents with 0 replaced by 0.1. */
typedef struct mor_marker {
    float position[3];
    float scale[3];
    float color[4];  /* 0.8, 0.1, 0.4, alpha 0.5 */
    int32_t id;      /* 1, 2, 3, ... in mo_vec order: the reference's counter starts at 1 (cpp:622) and advances per entry (cpp:669) */
    int32_t cluster; /* index into this frame's cluster list */
} mor_marker;
int mor_get_moving_markers(mor_handle* h, mor_marker* out, uint32_t cap, uint32_t* n_out);

/* Diagnostic, on request: the number of point pairs of the current frame's `cloud` whose squared distance lies within
 * `ulps` units in the last place of the squared clustering radius (float)((double)tol*tol) - the pairs on which an
 * implementation that rounds the distance differently, or prunes its tree search (FLANN, SURVEY A8), could decide the
 * other way than EuclideanClusterExtraction's strict `<` (cpp:213-218). Brute force over all pairs, ~1 ms. */
int mor_count_radius_ties(mor_handle* h, int ulps, uint64_t* pairs);

/* ---- parity taps ------------------------------------------------------------------------ */
typedef enum mor_tap_id {
    MOR_TAP_COUNTS = 0,          /* int32[MOR_NCOUNTS], see below */
    MOR_TAP_POINT_CLASS = 1,     /* uint8[N]: 0 trimmed (cpp:66-74), 1 `cloud`, 2 gp_indices (cpp:78-86) */
    MOR_TAP_LABELS = 2,          /* int32[N_c]: min `cloud` index of the point's radius-component */
    MOR_TAP_CLUSTER_ID = 3,      /* int32[N_c]: index into cluster_indices (cpp:218) or -1 */
    MOR_TAP_CLUSTER_ROOT = 4,    /* int32[K]: min `cloud` index of cluster k */
    MOR_TAP_CLUSTER_SIZE = 5,    /* int32[K] */
    MOR_TAP_CENTROIDS = 6,       /* float[K*3]: centroid_collection (cpp:239-243) */
    MOR_TAP_TRANSFORM = 7,       /* float[12]: row-major 3x4 of the Affine3f of cpp:536-551 */
    MOR_TAP_PREV_CENTROIDS_T = 8,/* float[K'*3]: ca->centroid_collection after cpp:541 */
    MOR_TAP_PREV_POINTS_T = 9,   /* float[N_c'*3]: ca cluster points after cpp:550, in ca `cloud` order; NaN if not in a cluster */
    MOR_TAP_MATCH_QUERY = 10,    /* int32[M]: index_query (prev cluster) after volumeConstraint (cpp:297-306) */
    MOR_TAP_MATCH_MATCH = 11,    /* int32[M]: index_match (current cluster) */
    MOR_TAP_MATCH_DIST = 12,     /* float[M]: squared centroid distance */
    MOR_TAP_MATCH_SCORE = 13,    /* double[M]: param_vec (cpp:568-576) */
    MOR_TAP_FLAGS = 14,          /* uint8[K]: cb->detection_results (cpp:580-606) */
    MOR_TAP_MO_CENTROIDS = 15,   /* float[n_mo*3]: mo_vec centroids (state after the last call) */
    MOR_TAP_MO_CONF = 16,        /* int32[n_mo] */
    MOR_TAP_REMOVED_MASK = 17,   /* uint8[N] after filter: 0 TRIMMED, 1 KEPT, 2 REMOVED */
    MOR_TAP_CLUSTER_REMOVED = 18,/* uint8[K] after filter: cluster selected at cpp:644-648 */
    MOR_TAP_RECIP_QUERY = 19,    /* int32[Mu]: reciprocal correspondences before the volume test (cpp:294) */
    MOR_TAP_RECIP_MATCH = 20,    /* int32[Mu] */
    MOR_TAP_GROUND_VOXELS = 21,  /* float[V*8] (ground modes 1/2): centroid xyz, accepted, bin key, normal xyz */
    MOR_TAP_CLUSTER_BBOX = 22,   /* float[K*6]: min xyz, max xyz of cluster k (getMinMax3D, cpp:274) */
    MOR_TAP_PREV_BBOX_T = 23,    /* float[K'*6]: bbox of the transformed prev clusters (cpp:272) */
    MOR_TAP__COUNT
} mor_tap_id;

enum {
    MOR_CNT_N = 0,        /* input points */
    MOR_CNT_NT = 1,       /* raw_cloud after x/y trim */
    MOR_CNT_NC = 2,       /* cloud (clustering domain) */
    MOR_CNT_NG = 3,       /* gp_indices */
    MOR_CNT_K = 4,        /* clusters in current frame */
    MOR_CNT_KPREV = 5,
    MOR_CNT_M = 6,        /* matches after volume constraint */
    MOR_CNT_NMO = 7,      /* mo_vec size */
    MOR_CNT_NOUT = 8,     /* output points (valid after filter) */
    MOR_CNT_NKPREV = 9,   /* points in prev clusters (transformed) */
    MOR_CNT_P1 = 10,      /* points of matched prev clusters */
    MOR_CNT_P2 = 11,      /* points of matched current clusters */
    MOR_CNT_TWO_FRAMES = 12,
    MOR_CNT_EXTRACT_OVERFLOW = 13, /* A18: moving index list longer than cloud => empty extract */
    MOR_CNT_MU = 14,      /* reciprocal correspondences before volume constraint */
    MOR_CNT_NCPREV = 15,  /* prev frame cloud size */
    MOR_CNT_NK = 16,      /* points in current clusters */
    MOR_CNT_NVOX = 17,    /* ground voxels (modes 1/2) */
    MOR_CNT_FRAME = 18,   /* frames pushed so far */
    MOR_CNT_ERRFLAGS = 19,/* device-side error bits (capacity overflows) */
    MOR_NCOUNTS = 24
};

/* Copies tap `tap` into dst (host). *n_bytes receives the tap's size; if cap_bytes is smaller
 * nothing is copied and MOR_ERR_CAPACITY is returned. Synchronises the handle's stream. */
int mor_tap(mor_handle* h, int tap, void* dst, size_t cap_bytes, size_t* n_bytes);

/* Named wrappers (SURVEY §8b). n = capacity in elements of the destination. */
int mor_get_counts(mor_handle* h, int32_t* counts, size_t n);
int mor_get_trim_mask(mor_handle* h, uint8_t* point_class, size_t n);
int mor_get_ground_mask(mor_handle* h, uint8_t* point_class, size_t n);
int mor_get_labels(mor_handle* h, int32_t* labels, size_t n);
int mor_get_cluster_order(mor_handle* h, int32_t* roots, size_t n);
int mor_get_centroids(mor_handle* h, float* xyz, size_t n);
int mor_get_transform(mor_handle* h, float* m12, size_t n);
int mor_get_transformed_xyz(mor_handle* h, float* xyz, size_t n);
int mor_get_matches(mor_handle* h, int32_t* query, int32_t* match, size_t n);
int mor_get_scores(mor_handle* h, double* scores, size_t n);
int mor_get_flags(mor_handle* h, uint8_t* flags, size_t n);
int mor_get_mo_vec(mor_handle* h, float* xyz, int32_t* conf, size_t n);
int mor_get_removed_mask(mor_handle* h, uint8_t* mask, size_t n);

#ifdef __cplusplus
}
#endif
#endif /* MOR_B200_H */
