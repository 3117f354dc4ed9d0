// mor_b200.cu — handle, launch sequence and C ABI (include/mor_b200.h) of the B200-native MOR hot path.
//
// One handle = one CUDA device + one compute stream (+ two copy streams for the streaming calls) + device-resident SoA
// frame state that persists across frames (previous frame's clusters, mo_vec, the corrs_vec / res_vec ring buffers). A
// frame is pushRawCloudAndPose (reference cpp:516-611) = one H2D copy + ONE cooperative kernel launch (k_frame: all phases
// of the frame incl. the filter phase, no host synchronisation), then filterCloud (cpp:613-696) = commit of the filter
// phase's result + the D2H copy of the output cloud.
// Throughput paths on top of that: mor_submit_frame / mor_collect_frame (copies of neighbouring frames on their own
// streams, up to four frames in flight) and mor_set_pipelining (k_frame_pipe: the back half of frame f in one launch with
// the front half of frame f+1; the frame products are triple-buffered for it, see fill_frame / launch_pipe).
// There is no CPU fallback: every entry point that computes needs the device.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mor_kernels.cuh"
#include "mor_ground.cuh"
#include "mor_debug.cuh"

using namespace mor;

#define MOR_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            h->last_error = std::string(#call) + ": " + cudaGetErrorString(e__);                    \
            return MOR_ERR_CUDA;                                                                    \
        }                                                                                           \
    } while (0)

namespace {

// ---- host-side pose delta (double, tf semantics A11) and the Eigen float affine (A12) -------------
struct Tf { double m[3][3]; double o[3]; };

// tf::Transform(tf::Quaternion(x,y,z,w), tf::Vector3) via Matrix3x3::setRotation; q is NOT normalised
// (tf::poseMsgToTF, reference cpp:524).
Tf tf_from_pose(const double p[7]) {
    Tf t;
    const double qx = p[3], qy = p[4], qz = p[5], qw = p[6];
    const double s = 2.0 / (qx * qx + qy * qy + qz * qz + qw * qw);
    const double xs = qx * s, ys = qy * s, zs = qz * s;
    const double wx = qw * xs, wy = qw * ys, wz = qw * zs, xx = qx * xs, xy = qx * ys, xz = qx * zs, yy = qy * ys, yz = qy * zs, zz = qz * zs;
    t.m[0][0] = 1.0 - (yy + zz); t.m[0][1] = xy - wz; t.m[0][2] = xz + wy;
    t.m[1][0] = xy + wz; t.m[1][1] = 1.0 - (xx + zz); t.m[1][2] = yz - wx;
    t.m[2][0] = xz - wy; t.m[2][1] = yz + wx; t.m[2][2] = 1.0 - (xx + yy);
    t.o[0] = p[0]; t.o[1] = p[1]; t.o[2] = p[2];
    return t;
}

// cb.ps.inverseTimes(ca.ps) (cpp:536): basis cur^T * prev, origin cur^T * (prev.o - cur.o).
// Then tf getRotation (double) -> Eigen::Quaternionf -> Translation3f * q (pcl_ros::transformPointCloud).
void pose_delta_affine(const double prev7[7], const double cur7[7], float M[12]) {
    const Tf a = tf_from_pose(cur7), b = tf_from_pose(prev7);
    double R[3][3], o[3];
    const double v[3] = {b.o[0] - a.o[0], b.o[1] - a.o[1], b.o[2] - a.o[2]};
    for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) R[i][j] = a.m[0][i] * b.m[0][j] + a.m[1][i] * b.m[1][j] + a.m[2][i] * b.m[2][j];
        o[i] = a.m[0][i] * v[0] + a.m[1][i] * v[1] + a.m[2][i] * v[2];
    }
    double q[4];
    const double trace = R[0][0] + R[1][1] + R[2][2];
    if (trace > 0.0) {
        double s = std::sqrt(trace + 1.0);
        q[3] = s * 0.5;
        s = 0.5 / s;
        q[0] = (R[2][1] - R[1][2]) * s; q[1] = (R[0][2] - R[2][0]) * s; q[2] = (R[1][0] - R[0][1]) * s;
    } else {
        const int i = R[0][0] < R[1][1] ? (R[1][1] < R[2][2] ? 2 : 1) : (R[0][0] < R[2][2] ? 2 : 0);
        const int j = (i + 1) % 3, k = (i + 2) % 3;
        double s = std::sqrt(R[i][i] - R[j][j] - R[k][k] + 1.0);
        q[i] = s * 0.5;
        s = 0.5 / s;
        q[3] = (R[k][j] - R[j][k]) * s; q[j] = (R[j][i] + R[i][j]) * s; q[k] = (R[k][i] + R[i][k]) * s;
    }
    const float x = (float)q[0], y = (float)q[1], z = (float)q[2], w = (float)q[3];
    const float tx = 2.0f * x, ty = 2.0f * y, tz = 2.0f * z;
    const float twx = tx * w, twy = ty * w, twz = tz * w, txx = tx * x, txy = ty * x, txz = tz * x, tyy = ty * y, tyz = tz * y, tzz = tz * z;
    M[0] = 1.0f - (tyy + tzz); M[1] = txy - twz; M[2] = txz + twy; M[3] = (float)o[0];
    M[4] = txy + twz; M[5] = 1.0f - (txx + tzz); M[6] = tyz - twx; M[7] = (float)o[1];
    M[8] = txz - twy; M[9] = tyz + twx; M[10] = 1.0f - (txx + tyy); M[11] = (float)o[2];
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

struct mor_handle {
    mor_config cfg;
    int device = 0;
    cudaStream_t stream = nullptr;
    uint32_t spec_out = 0;        // speculative size of the output D2H copy (points), from the previous frame
    cudaStream_t last_stream = nullptr;  // stream that carries this handle's latest work (differs after a batched step)
    // batched stepping (this handle as the leader of a batch): device array of per-sequence arguments + pinned ring; a slot
    // holds S FramePtrs followed by S GroundPtrs (the latter used by the voxel ground modes only)
    uint8_t* d_batch = nullptr; uint8_t* h_batch = nullptr; uint32_t batch_cap = 0; int batch_slot = 0;
    cudaEvent_t batch_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    uint32_t nmax = 0, kmax = 0, momax = 0;
    int ring_depth = 0, pde_ring = 0;
    int max_cells = 0; double cell_h = 0;  // max_cells: dense tables of the voxel ground modes
    int num_sms = 148, frame_ctas = 148;
    size_t frame_smem = 0;
    std::string last_error;

    // one big device arena + carved pointers
    uint8_t* arena = nullptr;
    size_t arena_bytes = 0;
    uint8_t* d_in = nullptr;
    size_t d_in_bytes = 0;
    // pipelined streaming (mor_submit_frame / mor_collect_frame): two slots, each with its own staging buffer, output
    // buffer, pinned counts and events; copies run on two streams of their own beside the frame kernels
    struct StreamSlot {
        uint8_t* d_in = nullptr; float4* d_out = nullptr; int32_t* h_counts = nullptr;
        cudaEvent_t h2d = nullptr, done = nullptr, d2h = nullptr;
        void* out = nullptr; uint32_t cap = 0, spec = 0, n = 0;
        const int* d_counts = nullptr;
        bool used = false, d2h_enqueued = false;
    } slot[MOR_STREAM_DEPTH];
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t ev_join = nullptr;
    int sf_head = 0, inflight = 0;
    float4* out_cur = nullptr;  // output buffer of the frame being enqueued (slot 0's unless a streaming slot says otherwise)
    size_t lattice_cap = 0, table_cap = 0, edge_cap = 0, heavy_cap = 0;
    FramePtrs base;  // pointers that do not change from frame to frame
    int* coll_cursor = nullptr; int* coll_turn = nullptr; float4* coll_out = nullptr;  // mor_get_cluster_collection scratch
    GroundPtrs ground;  // voxel-covariance ground removal state (ground_mode 1/2 only)
    // ping-pong
    // frame products: three in rotation (cur, prev and - in a pipelined launch - the frame whose front half is running)
    float4* pts[3]; float4* spts[3]; int* cid[3]; int* cl_root[3]; int* cl_size[3]; float* cl_centroid[3]; uint8_t* cl_flags[3]; float* cl_bbox[3]; int* counts[3];
    // products of the front half that only the back half of the SAME frame reads: two, by frame parity
    int* scid2[2]; float4* gpts2[2]; int* gsrc2[2]; int* cloud_src2[2]; uint8_t* removed_mask2[2];
    unsigned long long* acc_sum2[2]; unsigned* acc_box2[2];
    int cur = 0, fpar = 0;
    // pipelining (mor_set_pipelining): the back half of the last filtered frame waits to be launched beside the front half
    // of the next frame
    bool pipelining = false, back_pending = false;
    FramePtrs back_frame;
    bool have_cur = false, have_prev = false, filtered = false;
    int mo_parity = 0;
    double cur_pose[7], prev_pose[7];
    float M[12];
    bool two_frames = false;
    uint32_t n_input = 0, n_prev_input = 0;
    uint64_t launches = 0;
    FramePtrs frame;  // arguments of the current frame
    // timing
    bool timing = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int32_t* h_counts = nullptr;  // pinned
    // generic event slots (bench.py brackets its timed regions with these, on the handle's stream)
    cudaEvent_t slot_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // per-phase profiling (off by default): every phase of the frame kernel is launched as its own kernel between events
    bool profiling = false;
    std::vector<cudaEvent_t> prof_pool;
    std::vector<int> prof_ids;  // kernel id of every recorded pair of the current frame
    double prof_ms[40] = {0};
    uint64_t prof_n[40] = {0};
};

namespace {

enum KernelId { KID_PHASE0 = 0, KID_FRAME = PH__COUNT, KID_FILTER_AGAIN,
                KID_G_INGEST, KID_G_KEYS, KID_G_SCAN_CELLS, KID_G_SCAN_VOX, KID_G_SCATTER, KID_G_EVAL, KID_G_MODE, KID_G_MARK, KID_G_PARTITION, KID__COUNT };
const char* const kKernelNames[KID__COUNT] = {"ph_ingest", "ph_cells", "ph_scatter+link", "ph_test", "ph_jump", "ph_cross", "ph_roots", "ph_select+transform", "ph_stats+match",
                                              "ph_moving_test+chain", "ph_filter+cleanup", "k_frame", "k_filter_again",
                                              "k_ingest_raw", "k_ground_keys", "k_scan_cells", "k_scan_voxels", "k_ground_scatter",
                                              "k_voxel_eval", "k_ground_mode", "k_ground_mark", "k_ground_partition"};
static_assert(KID__COUNT <= 40, "profile table too small");

inline void prof_begin(mor_handle* h, int id) {
    if (!h->profiling) return;
    const size_t i = h->prof_ids.size() * 2;
    while (h->prof_pool.size() < i + 2) { cudaEvent_t e; cudaEventCreate(&e); h->prof_pool.push_back(e); }
    cudaEventRecord(h->prof_pool[i], h->stream);
    h->prof_ids.push_back(id);
}
inline void prof_end(mor_handle* h) {
    if (!h->profiling) return;
    cudaEventRecord(h->prof_pool[h->prof_ids.size() * 2 - 1], h->stream);
}
void prof_harvest(mor_handle* h) {  // stream must be idle
    for (size_t i = 0; i < h->prof_ids.size(); i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->prof_pool[2 * i], h->prof_pool[2 * i + 1]) == cudaSuccess) { h->prof_ms[h->prof_ids[i]] += ms; h->prof_n[h->prof_ids[i]]++; }
    }
    h->prof_ids.clear();
}
// Launch with the programmatic-stream-serialisation attribute (see pdl_prologue in mor_device.cuh): the chain of
// short kernels of the voxel ground modes.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}
#define MOR_KLAUNCH(id, kernel, grid, block, smem, ...)                                           \
    do {                                                                                           \
        cudaError_t le__;                                                                          \
        if (h->profiling) { prof_begin(h, id); kernel<<<grid, block, smem, st>>>(__VA_ARGS__); le__ = cudaGetLastError(); prof_end(h); } \
        else le__ = launch_pdl(kernel, dim3(grid), dim3(block), smem, st, __VA_ARGS__);           \
        if (le__ != cudaSuccess) { h->last_error = std::string(#kernel) + ": " + cudaGetErrorString(le__); return MOR_ERR_CUDA; } \
        h->launches++;                                                                             \
    } while (0)

// All CTAs of the frame kernel must be resident at once (they meet at group barriers): cooperative launch.
template <typename K, typename... Args>
cudaError_t launch_coop(K kernel, unsigned grid, size_t smem, cudaStream_t st, Args... args) {
    void* argv[] = {(void*)&args...};
    return cudaLaunchCooperativeKernel((const void*)kernel, dim3(grid), dim3(kT), argv, smem, st);
}

template <typename T>
T* carve(uint8_t*& p, size_t count) {
    T* r = reinterpret_cast<T*>(p);
    p += align_up(count * sizeof(T), 256);
    return r;
}

int build_grid(mor_handle* h) {
    const mor_config& c = h->cfg;
    // A7: r2 = (float)((double)tol * (double)tol); effective radius = sqrt(r2). Cell edge h = r/sqrt(3) shrunk by
    // 2^-10: the diagonal of a cell stays below r even after float rounding of the distance (every two points of
    // a cell are neighbours), and d < r implies a cell offset of at most 2 per axis (r/h = 1.734).
    // The grid is sparse (a hash table of the occupied cells), so neither the crop box nor the extent of a frame
    // enters anywhere: any finite coordinate up to 2^20 cells from the origin is binned.
    const float r2 = (float)((double)c.ec_distance_threshold * (double)c.ec_distance_threshold);
    if (!(r2 > 0.f) || !(c.trim_x > 0.f) || !(c.trim_y > 0.f)) return MOR_ERR_CONFIG_VALUE;
    h->cell_h = std::sqrt((double)r2) / std::sqrt(3.0) * (1.0 - 1.0 / 1024.0);
    if (!(h->cell_h > 0.0) || !std::isfinite(1.0 / h->cell_h)) return MOR_ERR_CONFIG_VALUE;
    h->pde_ring = (int)std::ceil(std::sqrt((double)c.pde_ub) / h->cell_h);
    if (h->pde_ring < 1) h->pde_ring = 1;
    if (h->pde_ring > 64) h->pde_ring = 64;
    return MOR_OK;
}

int allocate(mor_handle* h) {
    const size_t N = h->nmax, K = h->kmax, MO = h->momax, D = (size_t)h->ring_depth;
    const size_t tiles_pts = N / kBlock + 2;
    size_t lat = 1;
    while (lat < 2 * N) lat <<= 1;
    h->lattice_cap = lat;
    size_t tab = 1024;
    while (tab < 2 * N) tab <<= 1;  // load factor <= 1/2 even if every point had a cell of its own
    h->table_cap = tab;
    h->d_in_bytes = N * 32;
    h->edge_cap = 24 * N + 65536; h->heavy_cap = 6 * N + 16384;  // split into per-CTA segments at launch (a cell has at most 62 edges; ~8 is typical)
    const bool ground = h->cfg.ground_mode != MOR_GROUND_CROP;
    // ---- size pass (mirror of the carve pass below)
    auto plan = [&](uint8_t* p0) -> uint8_t* {
        uint8_t* p = p0;
        FramePtrs& b = h->base;
        h->d_in = carve<uint8_t>(p, h->d_in_bytes);
        h->slot[0].d_in = h->d_in;
        for (int q = 1; q < MOR_STREAM_DEPTH; q++) h->slot[q].d_in = carve<uint8_t>(p, h->d_in_bytes);
        b.scratch = carve<Scratch>(p, 1);
        b.st_ingest = carve<unsigned long long>(p, tiles_pts);
        b.st_out = carve<unsigned long long>(p, tiles_pts);
        b.table = carve<Cell>(p, tab);
        b.cell_list = carve<int>(p, N); b.ckey = carve<unsigned long long>(p, N + 1); b.cstart = carve<int>(p, N + 1); b.ccnt = carve<int>(p, N + 1);
        b.pslot = carve<int2>(p, N); b.slead = carve<int>(p, N);
        b.edges = carve<int2>(p, h->edge_cap); b.light = carve<int2>(p, h->edge_cap); b.heavy = carve<int4>(p, h->heavy_cap);
        b.edge_cnt = carve<int>(p, 256);
        b.hook = carve<int>(p, N); b.rsize = carve<int>(p, N); b.rmin = carve<int>(p, N); b.root_list = carve<int>(p, N);
        b.point_class = carve<uint8_t>(p, N); b.removed_mask = carve<uint8_t>(p, N);
        b.cloud_src = carve<int>(p, N); b.gpts = carve<float4>(p, N); b.gsrc = carve<int>(p, N);
        b.label = carve<int>(p, N); b.cid_of_root = carve<int>(p, N); b.cid_of_pos = carve<int>(p, N);
        b.scid = carve<int>(p, N);
        b.acc_sum = carve<unsigned long long>(p, K * 6); b.acc_box = carve<unsigned>(p, K * 6); b.pacc_box = carve<unsigned>(p, K * 6);
        b.tpts = carve<float4>(p, N); b.pct = carve<float>(p, K * 3); b.pbbox = carve<float>(p, K * 6);
        b.recip_q = carve<int>(p, K); b.recip_m = carve<int>(p, K); b.match_q = carve<int>(p, K); b.match_m = carve<int>(p, K);
        b.match_dist = carve<float>(p, K); b.match_score = carve<double>(p, K);
        b.match_of_prev = carve<int>(p, K); b.mid_of_prev = carve<int>(p, K); b.mid_of_cur = carve<int>(p, K);
        b.anchorp = carve<double>(p, K * 3); b.newcount = carve<int>(p, K);
        b.lattice = carve<unsigned long long>(p, lat);
        b.cluster_removed = carve<uint8_t>(p, K); b.found = carve<int>(p, K);
        b.marker_cluster = carve<int>(p, MO); b.phase_ts = carve<unsigned long long>(p, 32); b.cta_trace = carve<unsigned long long>(p, 32 * 256); h->coll_cursor = carve<int>(p, K); h->coll_turn = carve<int>(p, 2);
        b.out = carve<float4>(p, N * 2); h->coll_out = carve<float4>(p, N * 2);
        h->slot[0].d_out = b.out; h->out_cur = b.out;
        for (int q = 1; q < MOR_STREAM_DEPTH; q++) h->slot[q].d_out = carve<float4>(p, N * 2);
        for (int f = 0; f < 2; f++) {
            h->scid2[f] = f ? carve<int>(p, N) : b.scid; h->gpts2[f] = f ? carve<float4>(p, N) : b.gpts; h->gsrc2[f] = f ? carve<int>(p, N) : b.gsrc;
            h->cloud_src2[f] = f ? carve<int>(p, N) : b.cloud_src; h->removed_mask2[f] = f ? carve<uint8_t>(p, N) : b.removed_mask;
            h->acc_sum2[f] = f ? carve<unsigned long long>(p, K * 6) : b.acc_sum; h->acc_box2[f] = f ? carve<unsigned>(p, K * 6) : b.acc_box;
        }
        for (int f = 0; f < 3; f++) {
            h->pts[f] = carve<float4>(p, N); h->spts[f] = carve<float4>(p, N); h->cid[f] = carve<int>(p, N);
            h->cl_root[f] = carve<int>(p, K); h->cl_size[f] = carve<int>(p, K); h->cl_centroid[f] = carve<float>(p, K * 3);
            h->cl_flags[f] = carve<uint8_t>(p, K); h->cl_bbox[f] = carve<float>(p, K * 6); h->counts[f] = carve<int>(p, MOR_NCOUNTS);
        }
        if (ground) {  // dense ball-query grid and pcl::VoxelGrid index space over the bounding box of raw_cloud
            GroundPtrs& g = h->ground;
            const size_t vc = (size_t)h->max_cells;
            b.cell_count = carve<int>(p, vc + 16); b.cell_start = carve<int>(p, vc + 16); b.cell_key = carve<int>(p, N); b.skey = carve<int>(p, N);
            b.dgrid = carve<GridDesc>(p, 1); b.st_cells = carve<unsigned long long>(p, vc / kScanTile + 2);
            g.rpts = carve<float4>(p, N); g.rsrc = carve<int>(p, N); g.is_ground = carve<uint8_t>(p, N); g.vkey = carve<int>(p, N);
            g.vox_count = carve<int>(p, vc + 1); g.vox_ord = carve<int>(p, vc + 1); g.tiles_vox = (int)(vc / kTile + 2);  // k_scan_voxels pulls kTile-voxel tiles
            g.st_vox = carve<unsigned long long>(p, g.tiles_vox);
            g.vox_n = carve<int>(p, N); g.vacc = carve<unsigned long long>(p, N * 6); g.vox_info = carve<float>(p, N * 8);
            g.bin_hist = carve<int>(p, 65536); g.ggrid = carve<GridDesc>(p, 1); g.vdesc = carve<VoxDesc>(p, 1); g.gstate = carve<int>(p, 8);
        }
        b.track = carve<TrackState>(p, 1); b.mo_centroid = carve<float>(p, 2 * MO * 3); b.mo_conf = carve<int>(p, 2 * MO);
        b.res_ring = carve<uint8_t>(p, D * K); b.res_len = carve<int>(p, D); b.corr_ring = carve<int>(p, D * K); b.corr_len = carve<int>(p, D);
        return p;
    };
    h->arena_bytes = (size_t)(plan(nullptr) - (uint8_t*)nullptr) + 256;
    MOR_CUDA(cudaMalloc(&h->arena, h->arena_bytes));
    plan(h->arena);
    MOR_CUDA(cudaMallocHost(&h->h_counts, sizeof(int32_t) * MOR_NCOUNTS));
    for (int i = 0; i < 4; i++) MOR_CUDA(cudaEventCreate(&h->ev[i]));
    // dynamic shared memory of the frame kernel: the link phase's point tile + neighbour lists, or the cluster sort keys
    // of the select phase
    int P = 1;
    while (P < (int)K) P <<= 1;
    h->frame_smem = (size_t)P * sizeof(unsigned long long);
    if (h->frame_smem < kLinkSmem) h->frame_smem = kLinkSmem;
    return MOR_OK;
}

template <int PH>
int set_phase_smem(mor_handle* h) {
    MOR_CUDA(cudaFuncSetAttribute(k_phase<PH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->frame_smem));
    return MOR_OK;
}
int configure_kernels(mor_handle* h) {
    MOR_CUDA(cudaFuncSetAttribute(k_frame, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->frame_smem));
    MOR_CUDA(cudaFuncSetAttribute(k_frame_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->frame_smem));
    MOR_CUDA(cudaFuncSetAttribute(k_frame_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->frame_smem));
    int st = set_phase_smem<PH_SELECT>(h);
    if (st == MOR_OK) st = set_phase_smem<PH_LINK>(h);
    if (st == MOR_OK) st = set_phase_smem<PH_STATS>(h);
    if (st == MOR_OK) st = set_phase_smem<PH_INGEST>(h);
    if (st != MOR_OK) return st;
    int sms = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device) == cudaSuccess && sms > 0) h->num_sms = sms;
    MOR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_frame, kT, h->frame_smem));
    if (per_sm < 1) { h->last_error = "the frame kernel does not fit on an SM of this device"; return MOR_ERR_CUDA; }
    h->frame_ctas = h->num_sms;  // one CTA per SM
    return MOR_OK;
}

void fill_static(mor_handle* h) {
    FramePtrs& b = h->base;
    const mor_config& c = h->cfg;
    b.trim_x = c.trim_x; b.trim_y = c.trim_y; b.trim_z = c.trim_z; b.gp_limit = c.gp_limit;
    b.r2 = (float)((double)c.ec_distance_threshold * (double)c.ec_distance_threshold);
    b.volume_constraint = c.volume_constraint; b.pde_lb = c.pde_lb; b.pde_ub = c.pde_ub; b.pde_thr = c.pde_distance_threshold;
    b.leave_off = c.leave_off_distance; b.catch_up = c.catch_up_distance;
    b.min_cluster = c.min_cluster_size; b.max_cluster = c.max_cluster_size;
    b.method = c.method_choice; b.opc_factor = c.opc_normalization_factor;
    b.moving_confidence = c.n_bad; b.static_confidence = c.n_good;
    b.kmax = (int)h->kmax; b.momax = (int)h->momax; b.ring_depth = h->ring_depth;
    b.cell_h = h->cell_h; b.inv_h = 1.0 / h->cell_h;
    b.skip_ingest = c.ground_mode != MOR_GROUND_CROP ? 1 : 0;
    b.table_mask = (unsigned)(h->table_cap - 1);
    b.lattice_mask = (unsigned)(h->lattice_cap - 1);
    b.pde_ring = h->pde_ring;
    b.lattice_words16 = (unsigned)(h->lattice_cap / 2);
    b.tiles_pts = (int)(h->nmax / kBlock + 2);
    b.frame_smem = (int)h->frame_smem;
    b.max_cells = h->max_cells;
    b.tiles_cells = (int)((size_t)h->max_cells / kScanTile + 2);
    if (c.ground_mode != MOR_GROUND_CROP) {
        GroundPtrs& g = h->ground;
        g.mode = c.ground_mode; g.leaf = c.gp_leaf; g.inv_leaf = 1.0f / c.gp_leaf; g.r2 = (float)((double)c.gp_leaf * (double)c.gp_leaf);
        g.bin_gap = c.bin_gap; g.planarity = c.gp_planarity; g.bin_width = c.gp_bin_width;
        g.ball_cell_h = (double)c.gp_leaf * (1.0 + 1.0 / 1024.0);
    }
}

inline unsigned blocks_for(uint32_t n) { return n ? (n + kBlock - 1) / kBlock : 1; }

// pcl::fromPCLPointCloud2 accepts any record layout (cpp:523): float4 records and 4-byte aligned fields are read with
// vector / word loads, anything else (e.g. the 22-byte velodyne XYZIRT record) byte by byte.
int validate_layout(uint32_t step, uint32_t ox, uint32_t oy, uint32_t oz, uint32_t oi) {
    if (step < 12) return MOR_ERR_ARG;
    if (ox > step - 4 || oy > step - 4 || oz > step - 4 || (oi != 0xFFFFFFFFu && oi > step - 4)) return MOR_ERR_ARG;
    return MOR_OK;
}
int input_mode(const void* d_points, uint32_t step, uint32_t ox, uint32_t oy, uint32_t oz, uint32_t oi) {
    if (step == 16 && ox == 0 && oy == 4 && oz == 8 && oi == 12 && ((uintptr_t)d_points % 16) == 0) return 0;
    if (step % 4 == 0 && ox % 4 == 0 && oy % 4 == 0 && oz % 4 == 0 && (oi == 0xFFFFFFFFu || oi % 4 == 0) && ((uintptr_t)d_points % 4) == 0) return 1;
    return 2;
}

// The link phases write their results into one segment per CTA of the group that runs the frame.
void set_segments(mor_handle* h, FramePtrs& a, int group_ctas) {
    a.edge_seg = (int)(h->edge_cap / (size_t)group_ctas);
    a.light_cap = (int)h->edge_cap; a.heavy_cap = (int)h->heavy_cap;
}

// Arguments of the current frame (everything the kernels read) from the handle's host-side state.
void fill_frame(mor_handle* h, const uint8_t* d_points, uint32_t n, uint32_t step, uint32_t ox, uint32_t oy, uint32_t oz, uint32_t oi) {
    FramePtrs& a = h->frame;
    a = h->base;
    const int cur = h->cur, prev = (cur + 2) % 3;
    a.scid = h->scid2[h->fpar]; a.gpts = h->gpts2[h->fpar]; a.gsrc = h->gsrc2[h->fpar]; a.cloud_src = h->cloud_src2[h->fpar]; a.removed_mask = h->removed_mask2[h->fpar];
    a.acc_sum = h->acc_sum2[h->fpar]; a.acc_box = h->acc_box2[h->fpar];
    a.in = d_points; a.n = n; a.step = step; a.off_x = ox; a.off_y = oy; a.off_z = oz; a.off_i = oi;
    a.in_mode = input_mode(d_points, step, ox, oy, oz, oi);
    a.pts = h->pts[cur]; a.spts = h->spts[cur]; a.cid = h->cid[cur]; a.cl_root = h->cl_root[cur]; a.cl_size = h->cl_size[cur];
    a.cl_centroid = h->cl_centroid[cur]; a.cl_flags = h->cl_flags[cur]; a.cl_bbox = h->cl_bbox[cur]; a.counts = h->counts[cur];
    a.p_pts = h->pts[prev]; a.p_spts = h->spts[prev]; a.p_cid = h->cid[prev]; a.p_cl_root = h->cl_root[prev]; a.p_cl_size = h->cl_size[prev];
    a.p_cl_centroid = h->cl_centroid[prev]; a.p_cl_flags = h->cl_flags[prev]; a.p_counts = h->counts[prev];
    a.two_frames = h->two_frames ? 1 : 0;
    a.mo_parity = h->mo_parity;
    a.out = h->out_cur;
    std::memcpy(a.M.m, h->M, sizeof(h->M));
    set_segments(h, a, h->frame_ctas);
}

template <int PH>
int launch_phase(mor_handle* h, const FramePtrs& a) {
    prof_begin(h, KID_PHASE0 + PH);
    const size_t smem = (PH == PH_INGEST || PH == PH_SELECT || PH == PH_LINK || PH == PH_STATS) ? h->frame_smem : 0;
    cudaError_t e = launch_coop(k_phase<PH>, (unsigned)h->frame_ctas, smem, h->stream, a);
    prof_end(h);
    h->launches++;
    if (e != cudaSuccess) { h->last_error = std::string("k_phase: ") + cudaGetErrorString(e); return MOR_ERR_CUDA; }
    return MOR_OK;
}

// Pipelined launches (k_frame_pipe): the front half of `front` on most CTAs beside the pending back half, or either alone.
int launch_pipe(mor_handle* h, const FramePtrs* front, const FramePtrs* back) {
    const int G = h->frame_ctas;
    // the back half gets 5/32 of the CTAs (23 of 148): measured optimum on C2 (swept 100 ... 140: the front half holds two thirds
    // of a frame's chain of phases and is tile-granular in its first one, the back half is three short phases over the
    // points plus its single-CTA steps)
    int Gf = G, Gb = 0;
    if (front && back && G < 8) {  // too few SMs to share: one half after the other
        int s0 = launch_pipe(h, nullptr, back);
        return s0 != MOR_OK ? s0 : launch_pipe(h, front, nullptr);
    }
    if (front && back) {
        Gb = (G * 5) / 32;
        if (Gb < 4) Gb = 4;
        Gf = G - Gb;
        if (const char* env = std::getenv("MOR_PIPE_GF")) { const int v = std::atoi(env); if (v > 0 && v < G) Gf = v; }  // (tuning)
        Gb = G - Gf;
    } else if (back) { Gf = 0; Gb = G; }
    FramePtrs f = front ? *front : *back, b = back ? *back : *front;
    set_segments(h, f, Gf > 0 ? Gf : G);
    (void)Gb;
    cudaError_t e = launch_coop(k_frame_pipe, (unsigned)G, h->frame_smem, h->stream, f, b, Gf);
    h->launches++;
    if (e != cudaSuccess) { h->last_error = std::string("k_frame_pipe: ") + cudaGetErrorString(e); return MOR_ERR_CUDA; }
    return MOR_OK;
}
// The back half of the last filtered frame, if it is still waiting for a partner: alone.
int flush_back(mor_handle* h) {
    if (!h->back_pending) return MOR_OK;
    h->back_pending = false;
    return launch_pipe(h, nullptr, &h->back_frame);
}

int enqueue_push(mor_handle* h, const uint8_t* d_points, uint32_t n, uint32_t step, uint32_t ox, uint32_t oy, uint32_t oz, uint32_t oi, bool allow_pipe) {
    cudaStream_t st = h->stream;
    fill_frame(h, d_points, n, step, ox, oy, oz, oi);
    FramePtrs& a = h->frame;
    const unsigned gb = blocks_for(n);
    if (h->cfg.ground_mode != MOR_GROUND_CROP) {
        // voxel-covariance ground removal (reference cpp:90-200, repaired): 9 launches, then the frame kernel takes over
        const GroundPtrs& g = h->ground;
        FramePtrs ag = a;
        ag.dgrid = g.ggrid;  // the cell scan of this stage runs over the ball-query grid
        MOR_KLAUNCH(KID_G_INGEST, k_ingest_raw, gb, kBlock, 0, a, g);
        MOR_KLAUNCH(KID_G_KEYS, k_ground_keys, gb, kBlock, 0, a, g);
        MOR_KLAUNCH(KID_G_SCAN_CELLS, k_scan_cells, h->num_sms * 8, kBlock, 0, ag);
        MOR_KLAUNCH(KID_G_SCAN_VOX, k_scan_voxels, h->num_sms * 8, kBlock, 0, a, g);
        MOR_KLAUNCH(KID_G_SCATTER, k_ground_scatter, gb, kBlock, 0, a, g);
        MOR_KLAUNCH(KID_G_EVAL, k_voxel_eval, h->num_sms * 8, kBlock, 0, a, g);  // warps stride over the voxels
        MOR_KLAUNCH(KID_G_MODE, k_ground_mode, 1, 1024, 0, a, g);
        MOR_KLAUNCH(KID_G_MARK, k_ground_mark, h->num_sms * 8, kBlock, 0, a, g);
        MOR_KLAUNCH(KID_G_PARTITION, k_ground_partition, gb, kBlock, 0, a, g);
    }
    if (h->profiling) {  // one launch per phase, each between a pair of events
        int s;
        if ((s = launch_phase<PH_INGEST>(h, a)) || (s = launch_phase<PH_CELLS>(h, a)) || (s = launch_phase<PH_LINK>(h, a)) || (s = launch_phase<PH_TEST>(h, a)) ||
            (s = launch_phase<PH_JUMP>(h, a)) || (s = launch_phase<PH_CROSS>(h, a)) || (s = launch_phase<PH_ROOTS>(h, a)) || (s = launch_phase<PH_SELECT>(h, a)) || (s = launch_phase<PH_STATS>(h, a)) || 
            (s = launch_phase<PH_MOVING>(h, a)) || (s = launch_phase<PH_FILTER>(h, a)))
            return s;
    } else if (allow_pipe && h->pipelining && h->cfg.method_choice == 2 && h->cfg.ground_mode == MOR_GROUND_CROP) {
        // front half of this frame, beside the back half of the frame before if that one has been filtered already
        const bool fused = h->back_pending;
        h->back_pending = false;
        int s = launch_pipe(h, &a, fused ? &h->back_frame : nullptr);
        if (s != MOR_OK) return s;
        h->back_frame = a;  // this frame's back half: beside the next frame's front half, or alone as soon as somebody needs its results
        h->back_pending = true;
    } else {
        cudaError_t e = launch_coop(k_frame, (unsigned)h->frame_ctas, h->frame_smem, st, a);
        h->launches++;
        if (e != cudaSuccess) { h->last_error = std::string("k_frame: ") + cudaGetErrorString(e); return MOR_ERR_CUDA; }
    }
    return MOR_OK;
}

// The voxel ground stage of mor_batch_step_device: the nine kernels of enqueue_push, each launched once for all S
// sequences (blockIdx.y = sequence, arguments P[s] / GP[s]). The point-indexed stages are sized for the largest frame
// of the batch; the strided stages share the num_sms * 8 blocks of one single-handle launch among the sequences (C4 on
// B200: as fast as or faster than 2, 8 or 16 blocks per sequence at S = 1 ... 37).
int enqueue_ground_batch(mor_handle* h, const FramePtrs* P, const GroundPtrs* GP, uint32_t S, uint32_t n_max) {
    cudaStream_t st = h->stream;
    const dim3 pts(blocks_for(n_max), S), strided(((unsigned)h->num_sms * 8 + S - 1) / S, S), single(1, S);
#define MOR_GLAUNCH(kernel, grid, block)                                                                                \
    do {                                                                                                               \
        cudaError_t le__ = launch_pdl(kernel, grid, dim3(block), 0, st, P, GP);                                        \
        if (le__ != cudaSuccess) { h->last_error = std::string(#kernel) + ": " + cudaGetErrorString(le__); return MOR_ERR_CUDA; } \
        h->launches++;                                                                                                 \
    } while (0)
    MOR_GLAUNCH(k_ingest_raw_batch, pts, kBlock);
    MOR_GLAUNCH(k_ground_keys_batch, pts, kBlock);
    MOR_GLAUNCH(k_scan_cells_batch, strided, kBlock);
    MOR_GLAUNCH(k_scan_voxels_batch, strided, kBlock);
    MOR_GLAUNCH(k_ground_scatter_batch, pts, kBlock);
    MOR_GLAUNCH(k_voxel_eval_batch, strided, kBlock);
    MOR_GLAUNCH(k_ground_mode_batch, single, kSingle);
    MOR_GLAUNCH(k_ground_mark_batch, strided, kBlock);
    MOR_GLAUNCH(k_ground_partition_batch, pts, kBlock);
#undef MOR_GLAUNCH
    return MOR_OK;
}

// ca = cb; cb = new frame (cpp:520-521), pose delta cb.ps^-1 * ca.ps (cpp:536)
void advance_frame(mor_handle* h, uint32_t n, const double pose7[7]) {
    if (h->have_cur) { h->cur = (h->cur + 1) % 3; h->fpar ^= 1; std::memcpy(h->prev_pose, h->cur_pose, sizeof(h->cur_pose)); h->have_prev = true; h->n_prev_input = h->n_input; }
    std::memcpy(h->cur_pose, pose7, sizeof(h->cur_pose));
    h->n_input = n;
    h->two_frames = h->have_prev;  // ca->init && cb->init (cpp:534)
    std::memset(h->M, 0, sizeof(h->M));
    if (h->two_frames) pose_delta_affine(h->prev_pose, h->cur_pose, h->M);
    h->have_cur = true;
    h->filtered = false;
}

// Work of a handle may have been enqueued on another handle's stream by mor_batch_step_device.
int join_foreign_stream(mor_handle* h, bool keep_pending_back = false) {
    if (!keep_pending_back) { int fs = flush_back(h); if (fs != MOR_OK) return fs; }
    if (h->last_stream && h->last_stream != h->stream) {
        MOR_CUDA(cudaStreamSynchronize(h->last_stream));
        h->last_stream = h->stream;
    }
    return MOR_OK;
}

int do_push(mor_handle* h, const void* data, bool on_device, uint32_t n, uint32_t step, uint32_t ox, uint32_t oy, uint32_t oz, uint32_t oi, const double pose7[7]) {
    if (!h || (!data && n) || !pose7) return MOR_ERR_ARG;
    if (validate_layout(step, ox, oy, oz, oi) != MOR_OK) { h->last_error = "point_step / field offsets do not describe a record with float32 x, y, z"; return MOR_ERR_ARG; }
    if (n > h->nmax) { h->last_error = "frame larger than mor_limits.max_points"; return MOR_ERR_CAPACITY; }
    if (h->inflight) { h->last_error = "submitted frames are in flight: collect them first"; return MOR_ERR_STATE; }
    h->out_cur = h->slot[0].d_out;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h, on_device && h->pipelining && h->cfg.ground_mode == MOR_GROUND_CROP && !h->profiling); if (js != MOR_OK) return js; }
    if (h->timing) MOR_CUDA(cudaEventRecord(h->ev[0], h->stream));
    if (h->profiling && !h->prof_ids.empty()) { MOR_CUDA(cudaStreamSynchronize(h->stream)); prof_harvest(h); }
    const uint8_t* d_points = (const uint8_t*)data;
    if (!on_device) {
        const size_t bytes = (size_t)n * step;
        if (bytes > h->d_in_bytes) { h->last_error = "n * point_step exceeds the staging buffer (32 B/point)"; return MOR_ERR_CAPACITY; }
        if (bytes) MOR_CUDA(cudaMemcpyAsync(h->d_in, data, bytes, cudaMemcpyHostToDevice, h->stream));
        d_points = h->d_in;
    }
    advance_frame(h, n, pose7);
    int st = enqueue_push(h, d_points, n, step, ox, oy, oz, oi, /*allow_pipe=*/on_device);
    if (st != MOR_OK) return st;
    if (h->timing) MOR_CUDA(cudaEventRecord(h->ev[1], h->stream));
    return MOR_OK;
}

// filterCloud. The frame kernel has already run the filter phase on the frame (tracking update into the spare half of
// the mo_vec double buffer, output cloud into the handle's buffer): the first filterCloud on a frame COMMITS that
// result (flips the double buffer) and delivers the cloud; a frame that is never filtered leaves mo_vec untouched,
// as in the reference. A further filterCloud on the same frame runs the filter phase again (k_filter_again) on the
// updated mo_vec, which is what the reference does when the call is repeated.
int do_filter(mor_handle* h, void* out, bool on_device, uint32_t cap_points, uint32_t* n_out) {
    if (!h) return MOR_ERR_ARG;
    if (!h->have_cur) return MOR_ERR_STATE;
    if (h->inflight) { h->last_error = "submitted frames are in flight: collect them first"; return MOR_ERR_STATE; }
    MOR_CUDA(cudaSetDevice(h->device));
    // (pipelining: a filter call that asks for nothing now leaves the frame's back half waiting for the next frame's front half)
    const bool stays_pending = h->back_pending && on_device && !n_out && !out && !h->profiling && !h->filtered;
    { int js = join_foreign_stream(h, stays_pending); if (js != MOR_OK) return js; }
    cudaStream_t st = h->stream;
    if (h->timing) MOR_CUDA(cudaEventRecord(h->ev[2], st));
    FramePtrs& a = h->frame;
    if (on_device && out && cap_points < h->n_input) { h->last_error = "device output buffer must hold n_input points"; return MOR_ERR_CAPACITY; }
    if (h->filtered) {  // repeated call: the tracking update runs once more
        a.mo_parity = h->mo_parity;
        prof_begin(h, KID_FILTER_AGAIN);
        k_filter_again<<<h->n_input ? (h->n_input + kOutTile - 1) / kOutTile : 1, kT, 0, st>>>(a);
        prof_end(h);
        h->launches++;
        MOR_CUDA(cudaGetLastError());
        h->filtered = false;  // committed below like a first call
    }
    if (h->timing) MOR_CUDA(cudaEventRecord(h->ev[3], st));
    if (on_device && !n_out && !h->profiling) {  // fully asynchronous device-resident mode
        if (out && h->n_input) MOR_CUDA(cudaMemcpyAsync(out, a.out, (size_t)h->n_input * 32, cudaMemcpyDeviceToDevice, st));
        h->mo_parity ^= 1; a.mo_parity = h->mo_parity; h->filtered = true;
        return MOR_OK;
    }
    MOR_CUDA(cudaMemcpyAsync(h->h_counts, a.counts, sizeof(int32_t) * MOR_NCOUNTS, cudaMemcpyDeviceToHost, st));
    // The size of the output is only known on the device. Instead of a second round trip (sync on the count, then
    // copy), the cloud copy is issued speculatively with the previous frame's size plus a margin and topped up in
    // the rare case the frame turned out larger.
    uint32_t spec = 0;
    if (!on_device && out) {
        spec = h->spec_out ? h->spec_out + h->spec_out / 32 + 1024 : h->n_input;
        if (spec > h->n_input) spec = h->n_input;
        if (spec > cap_points) spec = cap_points;
        if (spec) MOR_CUDA(cudaMemcpyAsync(out, a.out, (size_t)spec * 32, cudaMemcpyDeviceToHost, st));
    }
    MOR_CUDA(cudaStreamSynchronize(st));
    if (h->profiling) prof_harvest(h);
    const uint32_t no = (uint32_t)h->h_counts[CNT_SPEC_NOUT];
    if (n_out) *n_out = no;
    h->spec_out = no;
    if (h->h_counts[MOR_CNT_ERRFLAGS]) {  // a device-side capacity was exceeded: the frame's results are not reference-exact
        char msg[200];
        std::snprintf(msg, sizeof msg, "device capacity exceeded (error bits 0x%x: 1=clusters 2=moving 4=lattice range 8=ground grid 16=coordinate beyond the grid's range 32=cell pairs)",
                      h->h_counts[MOR_CNT_ERRFLAGS]);
        h->last_error = msg;
        return MOR_ERR_CAPACITY;
    }
    if (no > cap_points && out) return MOR_ERR_CAPACITY;  // not committed: the call can be repeated with a larger buffer
    if (!on_device && out && no > spec) {
        MOR_CUDA(cudaMemcpyAsync((uint8_t*)out + (size_t)spec * 32, (const uint8_t*)a.out + (size_t)spec * 32, (size_t)(no - spec) * 32, cudaMemcpyDeviceToHost, st));
        MOR_CUDA(cudaStreamSynchronize(st));
    }
    if (on_device && out && no) MOR_CUDA(cudaMemcpyAsync(out, a.out, (size_t)no * 32, cudaMemcpyDeviceToDevice, st));
    h->mo_parity ^= 1; a.mo_parity = h->mo_parity; h->filtered = true;  // commit
    return MOR_OK;
}

// The state of a handle that has seen no frame: all device tables zero, no tracked objects, empty buffers (the
// reference's freshly constructed object, cpp:368-391). Ordered on the handle's stream.
int reset_state(mor_handle* h) {
    if (h->copy_in) MOR_CUDA(cudaStreamSynchronize(h->copy_in));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    if (h->copy_out) MOR_CUDA(cudaStreamSynchronize(h->copy_out));
    h->inflight = 0; h->sf_head = 0; h->out_cur = h->slot[0].d_out;
    MOR_CUDA(cudaMemsetAsync(h->arena, 0, h->arena_bytes, h->stream));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    h->cur = 0; h->fpar = 0; h->back_pending = false; h->have_cur = h->have_prev = h->filtered = h->two_frames = false;
    h->mo_parity = 0; h->n_input = h->n_prev_input = 0; h->spec_out = 0;
    h->last_stream = h->stream;
    return MOR_OK;
}

}  // namespace

// ============================================================================================ C ABI
extern "C" {

int mor_create_ex(const char* config_path, int n_bad, int n_good, int device, const mor_limits* limits, mor_handle** out) {
    if (!out || !config_path) return MOR_ERR_ARG;
    *out = nullptr;
    // moving_confidence / static_confidence are compared as unsigned sizes in the reference (cpp:489; .h:88-93): a
    // negative value never confirms anything there. Rejected here instead of imitated.
    if (n_bad < 0 || n_good < 0) return MOR_ERR_ARG;
    mor_config cfg;
    int st = mor_parse_config(config_path, &cfg);
    if (st != MOR_OK) return st;
    cfg.n_bad = n_bad; cfg.n_good = n_good;
    if (cfg.ground_mode != MOR_GROUND_CROP && !(cfg.gp_leaf > 0.f)) return MOR_ERR_CONFIG_VALUE;
    if (limits && limits->max_points >= (1u << 25)) return MOR_ERR_ARG;  // packed 31-bit partition counters, 2 x N table slots
    mor_handle* h = new mor_handle();
    h->cfg = cfg; h->device = device;
    h->nmax = limits && limits->max_points ? limits->max_points : 300000u;
    h->kmax = limits && limits->max_clusters ? limits->max_clusters : 8192u;
    h->momax = limits && limits->max_moving ? limits->max_moving : 1024u;
    h->max_cells = limits && limits->max_cells ? (int)(limits->max_cells > 0x40000000u ? 0x40000000u : limits->max_cells) : (1 << 24);
    if (h->kmax > 16384u) h->kmax = 16384u;  // the select phase sorts the clusters of a frame in shared memory (128 KB of keys)
    h->ring_depth = (n_bad > 1 ? n_bad : 1) + 2;
    st = build_grid(h);
    if (st != MOR_OK) { delete h; return st; }
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { cudaGetLastError(); mor_destroy(h); return MOR_ERR_CUDA; }  // mor_destroy releases whatever exists
    st = allocate(h);
    if (st == MOR_OK) st = configure_kernels(h);
    if (st != MOR_OK) { cudaGetLastError(); mor_destroy(h); return st; }
    fill_static(h);
    st = reset_state(h);
    if (st != MOR_OK) { mor_destroy(h); return st; }
    *out = h;
    return MOR_OK;
}

int mor_reset(mor_handle* h) {
    if (!h) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    return reset_state(h);
}

int mor_create(const char* config_path, int n_bad, int n_good, int device, mor_handle** out) {
    return mor_create_ex(config_path, n_bad, n_good, device, nullptr, out);
}

int mor_destroy(mor_handle* h) {
    if (!h) return MOR_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto& e : h->ev) if (e) cudaEventDestroy(e);
    for (auto& e : h->slot_ev) if (e) cudaEventDestroy(e);
    for (auto& e : h->prof_pool) cudaEventDestroy(e);
    if (h->h_counts) cudaFreeHost(h->h_counts);
    if (h->copy_in) { cudaStreamSynchronize(h->copy_in); cudaStreamDestroy(h->copy_in); }
    if (h->copy_out) { cudaStreamSynchronize(h->copy_out); cudaStreamDestroy(h->copy_out); }
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (auto& sl : h->slot) {
        if (sl.h_counts) cudaFreeHost(sl.h_counts);
        if (sl.h2d) cudaEventDestroy(sl.h2d);
        if (sl.done) cudaEventDestroy(sl.done);
        if (sl.d2h) cudaEventDestroy(sl.d2h);
    }
    if (h->d_batch) cudaFree(h->d_batch);
    if (h->h_batch) cudaFreeHost(h->h_batch);
    for (auto& e : h->batch_ev) if (e) cudaEventDestroy(e);
    if (h->arena) cudaFree(h->arena);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return MOR_OK;
}

int mor_get_config(const mor_handle* h, mor_config* out) {
    if (!h || !out) return MOR_ERR_ARG;
    *out = h->cfg;
    return MOR_OK;
}

int mor_get_limits(const mor_handle* h, mor_limits* out) {
    if (!h || !out) return MOR_ERR_ARG;
    *out = mor_limits{};
    out->max_points = h->nmax; out->max_clusters = h->kmax; out->max_moving = h->momax; out->max_cells = (uint32_t)h->max_cells;
    return MOR_OK;
}

const char* mor_last_error(const mor_handle* h) { return h ? h->last_error.c_str() : ""; }

int mor_push_raw_cloud_and_pose(mor_handle* h, const void* data, uint32_t n, uint32_t point_step, uint32_t off_x, uint32_t off_y, uint32_t off_z,
                                uint32_t off_i, const double pose7[7]) {
    return do_push(h, data, false, n, point_step, off_x, off_y, off_z, off_i, pose7);
}
int mor_push_raw_cloud_and_pose_device(mor_handle* h, const void* d_data, uint32_t n, uint32_t point_step, uint32_t off_x, uint32_t off_y,
                                       uint32_t off_z, uint32_t off_i, const double pose7[7]) {
    return do_push(h, d_data, true, n, point_step, off_x, off_y, off_z, off_i, pose7);
}
int mor_filter_cloud(mor_handle* h, void* out, uint32_t cap_points, uint32_t* n_out) {
    if (!out && cap_points) return MOR_ERR_ARG;
    return do_filter(h, out, false, cap_points, n_out);
}
int mor_filter_cloud_device(mor_handle* h, void* d_out, uint32_t cap_points, uint32_t* n_out) { return do_filter(h, d_out, true, cap_points, n_out); }

int mor_get_output_device(mor_handle* h, const void** d_records) {
    if (!h || !d_records) return MOR_ERR_ARG;
    if (!h->have_cur || !h->filtered) return MOR_ERR_STATE;
    *d_records = h->frame.out;
    return MOR_OK;
}

// One pushRawCloudAndPose + filterCloud for S independent sequences in one launch (BASELINE config 5).
int mor_batch_step_device(mor_handle* const* hs, uint32_t S, const void* const* d_data, const uint32_t* n, uint32_t point_step, uint32_t off_x,
                          uint32_t off_y, uint32_t off_z, uint32_t off_i, const double* poses7, void* const* d_out) {
    if (!hs || !S || !d_data || !n || !poses7 || !d_out || !hs[0]) return MOR_ERR_ARG;
    mor_handle* h = hs[0];  // leader: owns the stream and the argument array of the batch
    if (validate_layout(point_step, off_x, off_y, off_z, off_i) != MOR_OK) return MOR_ERR_ARG;
    for (uint32_t s = 0; s < S; s++) {
        mor_handle* g = hs[s];
        // same device, limits, frame count and configuration (every key that reaches the kernels)
        if (!g || g->device != h->device || g->nmax != h->nmax || g->kmax != h->kmax || g->momax != h->momax || g->have_prev != h->have_prev ||
            g->have_cur != h->have_cur || g->profiling || g->inflight || std::memcmp(&g->cfg, &h->cfg, offsetof(mor_config, output_topic)) != 0) {
            h->last_error = "batched handles must share device, limits, config and frame count";
            return MOR_ERR_ARG;
        }
        { int fs = flush_back(g); if (fs != MOR_OK) return fs; }
        if (n[s] > g->nmax || (!d_data[s] && n[s]) || !d_out[s]) return n[s] > g->nmax ? MOR_ERR_CAPACITY : MOR_ERR_ARG;
        for (uint32_t t = 0; t < s; t++) if (hs[t] == g) return MOR_ERR_ARG;
    }
    const bool ground = h->cfg.ground_mode != MOR_GROUND_CROP;  // (shared by every handle: part of the config compared above)
    if (ground && S > 65535u) { h->last_error = "the voxel ground modes batch at most 65535 sequences per step"; return MOR_ERR_ARG; }
    MOR_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    static_assert(sizeof(FramePtrs) % alignof(GroundPtrs) == 0, "GroundPtrs follow the FramePtrs of a ring slot");
    const size_t per_seq = sizeof(FramePtrs) + sizeof(GroundPtrs);
    if (S > h->batch_cap) {
        MOR_CUDA(cudaStreamSynchronize(st));
        if (h->d_batch) cudaFree(h->d_batch);
        if (h->h_batch) cudaFreeHost(h->h_batch);
        h->d_batch = nullptr; h->h_batch = nullptr; h->batch_cap = 0;
        MOR_CUDA(cudaMalloc(&h->d_batch, per_seq * S * 4));
        MOR_CUDA(cudaMallocHost(&h->h_batch, per_seq * S * 4));
        for (auto& e : h->batch_ev) if (!e) MOR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->batch_cap = S;
    }
    // ring of 4 argument slots: the H2D copy of a slot runs later on the stream, so a slot is only rewritten once the
    // step that used it four steps ago has consumed it
    const int slot = h->batch_slot;
    h->batch_slot = (slot + 1) & 3;
    MOR_CUDA(cudaEventSynchronize(h->batch_ev[slot]));
    FramePtrs* hp = reinterpret_cast<FramePtrs*>(h->h_batch + (size_t)slot * per_seq * h->batch_cap);
    FramePtrs* dp = reinterpret_cast<FramePtrs*>(h->d_batch + (size_t)slot * per_seq * h->batch_cap);
    GroundPtrs* hg = reinterpret_cast<GroundPtrs*>(hp + S);
    const GroundPtrs* dg = reinterpret_cast<const GroundPtrs*>(dp + S);
    uint32_t n_max = 0;
    // G CTAs per sequence; the groups run side by side, a group that has more than one sequence steps them in turn
    int G = h->frame_ctas / (int)S;
    if (const char* env = std::getenv("MOR_BATCH_G")) { const int v = std::atoi(env); if (v > 0) G = v; }
    if (G < 1) G = 1;
    if (G > h->frame_ctas) G = h->frame_ctas;
    int groups = h->frame_ctas / G;
    if (groups > (int)S) groups = (int)S;
    for (uint32_t s = 0; s < S; s++) {
        mor_handle* g = hs[s];
        if (g->last_stream != st) {  // earlier work of this handle ran elsewhere (its own stream or another batch): wait for it once
            if (g->last_stream) MOR_CUDA(cudaStreamSynchronize(g->last_stream));
            if (g->stream != st) MOR_CUDA(cudaStreamSynchronize(g->stream));
        }
        advance_frame(g, n[s], poses7 + 7 * s);
        g->out_cur = g->slot[0].d_out;
        fill_frame(g, (const uint8_t*)d_data[s], n[s], point_step, off_x, off_y, off_z, off_i);
        g->frame.out = (float4*)d_out[s];
        set_segments(g, g->frame, G);
        hp[s] = g->frame;
        if (ground) { hg[s] = g->ground; n_max = n[s] > n_max ? n[s] : n_max; }
        g->last_stream = st;
    }
    MOR_CUDA(cudaMemcpyAsync(dp, hp, (ground ? per_seq : sizeof(FramePtrs)) * S, cudaMemcpyHostToDevice, st));
    MOR_CUDA(cudaEventRecord(h->batch_ev[slot], st));
    if (ground) {  // voxel-covariance ground removal of all S frames: 9 launches, then the frame kernel takes over
        int gs = enqueue_ground_batch(h, dp, dg, S, n_max);
        if (gs != MOR_OK) return gs;
    }
    {
        cudaError_t e = launch_coop(k_frame_batch, (unsigned)(groups * G), h->frame_smem, st, (const FramePtrs*)dp, (int)S, G);
        h->launches++;
        if (e != cudaSuccess) { h->last_error = std::string("k_frame_batch: ") + cudaGetErrorString(e); return MOR_ERR_CUDA; }
    }
    for (uint32_t s = 0; s < S; s++) {  // push + filter in one call: the frame is committed
        hs[s]->mo_parity ^= 1;
        hs[s]->frame.mo_parity = hs[s]->mo_parity;
        hs[s]->filtered = true;
    }
    return MOR_OK;
}

int mor_sync(mor_handle* h) {
    if (!h) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    if (h->copy_out) MOR_CUDA(cudaStreamSynchronize(h->copy_out));
    return MOR_OK;
}

// ---- pipelined streaming ---------------------------------------------------------------------------
// Frame f lives in slot f mod MOR_STREAM_DEPTH. Three streams: copy_in (H2D of the raw records), the handle's stream
// (frame kernels, in order: the tracker state is a chain through the frames) and copy_out (counts + filtered cloud). A
// slot is reused by frame f + DEPTH, which cannot be submitted before frame f has been collected, i.e. before its D2H
// copy - and with it the kernel that read the slot's staging buffer and wrote its output buffer - has completed. With
// three frames in flight the H2D copy of frame f+1 is issued while the host still waits for frame f-1: the kernels then
// run back to back (with two, every kernel waited ~14 us for its input); with pipelined launches a frame's results come
// one launch later (its back half rides with the next frame's front half), which takes a fourth. The per-frame counts
// rotate through three blocks: the kernel of frame f overwrites the block frame f-3's D2H reads, so it waits for that
// copy (normally long done).
static int ensure_streaming(mor_handle* h) {
    if (h->copy_in) return MOR_OK;
    MOR_CUDA(cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking));
    MOR_CUDA(cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
    MOR_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    for (auto& sl : h->slot) {
        MOR_CUDA(cudaMallocHost(&sl.h_counts, sizeof(int32_t) * MOR_NCOUNTS));
        MOR_CUDA(cudaEventCreateWithFlags(&sl.h2d, cudaEventDisableTiming));
        MOR_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        MOR_CUDA(cudaEventCreateWithFlags(&sl.d2h, cudaEventDisableTiming));
    }
    return MOR_OK;
}

// The frame of a slot is complete on the handle's stream: its counts and its cloud go to the host on copy_out.
static int enqueue_slot_d2h(mor_handle* h, mor_handle::StreamSlot& sl) {
    MOR_CUDA(cudaEventRecord(sl.done, h->stream));
    MOR_CUDA(cudaStreamWaitEvent(h->copy_out, sl.done, 0));
    MOR_CUDA(cudaMemcpyAsync(sl.h_counts, sl.d_counts, sizeof(int32_t) * MOR_NCOUNTS, cudaMemcpyDeviceToHost, h->copy_out));
    // the size of the output is known on the device only: the copy is sized from the last collected frame plus a margin
    // and topped up at collection in the rare case the frame turned out larger
    uint32_t spec = h->spec_out ? h->spec_out + h->spec_out / 32 + 1024 : sl.n;
    if (spec > sl.n) spec = sl.n;
    if (spec > sl.cap) spec = sl.cap;
    if (spec) MOR_CUDA(cudaMemcpyAsync(sl.out, sl.d_out, (size_t)spec * 32, cudaMemcpyDeviceToHost, h->copy_out));
    MOR_CUDA(cudaEventRecord(sl.d2h, h->copy_out));
    sl.spec = spec; sl.d2h_enqueued = true;
    return MOR_OK;
}

int mor_submit_frame(mor_handle* h, const void* data, uint32_t n, uint32_t step, uint32_t ox, uint32_t oy, uint32_t oz, uint32_t oi,
                     const double pose7[7], void* out, uint32_t cap_points) {
    if (!h || (!data && n) || !pose7 || (!out && cap_points)) return MOR_ERR_ARG;
    if (validate_layout(step, ox, oy, oz, oi) != MOR_OK) { h->last_error = "point_step / field offsets do not describe a record with float32 x, y, z"; return MOR_ERR_ARG; }
    if (n > h->nmax) { h->last_error = "frame larger than mor_limits.max_points"; return MOR_ERR_CAPACITY; }
    const size_t bytes = (size_t)n * step;
    if (bytes > h->d_in_bytes) { h->last_error = "n * point_step exceeds the staging buffer (32 B/point)"; return MOR_ERR_CAPACITY; }
    if (h->profiling) { h->last_error = "per-phase profiling serialises every frame: not available while streaming"; return MOR_ERR_STATE; }
    if (h->inflight >= MOR_STREAM_DEPTH) { h->last_error = "MOR_STREAM_DEPTH frames are in flight: collect one first"; return MOR_ERR_STATE; }
    MOR_CUDA(cudaSetDevice(h->device));
    { int st = ensure_streaming(h); if (st != MOR_OK) return st; }
    { int js = join_foreign_stream(h, /*keep_pending_back=*/h->inflight > 0); if (js != MOR_OK) return js; }
    const int si = (h->sf_head + h->inflight) % MOR_STREAM_DEPTH;
    mor_handle::StreamSlot& sl = h->slot[si];
    {   // the count block this frame's kernel writes (three in rotation) was the one of the frame three back: its D2H must be over
        mor_handle::StreamSlot& s3 = h->slot[(si + MOR_STREAM_DEPTH - 3) % MOR_STREAM_DEPTH];
        if (s3.used && s3.d2h_enqueued) MOR_CUDA(cudaStreamWaitEvent(h->stream, s3.d2h, 0));
    }
    if (!h->inflight) {  // the pipeline starts: earlier work of the synchronous calls may still use slot 0's buffers
        MOR_CUDA(cudaEventRecord(h->ev_join, h->stream));
        MOR_CUDA(cudaStreamWaitEvent(h->copy_in, h->ev_join, 0));
    }
    if (bytes) MOR_CUDA(cudaMemcpyAsync(sl.d_in, data, bytes, cudaMemcpyHostToDevice, h->copy_in));
    MOR_CUDA(cudaEventRecord(sl.h2d, h->copy_in));
    MOR_CUDA(cudaStreamWaitEvent(h->stream, sl.h2d, 0));
    advance_frame(h, n, pose7);
    h->out_cur = sl.d_out;
    const bool piped = h->pipelining && h->cfg.method_choice == 2 && h->cfg.ground_mode == MOR_GROUND_CROP;
    int st = enqueue_push(h, sl.d_in, n, step, ox, oy, oz, oi, /*allow_pipe=*/true);
    if (st != MOR_OK) return st;
    sl.out = out; sl.cap = cap_points; sl.n = n; sl.d_counts = h->frame.counts; sl.used = true; sl.d2h_enqueued = false;
    if (piped) {
        // the launch just enqueued carried the back half of the frame before (if one was waiting): that frame is complete now
        if (h->inflight) {
            mor_handle::StreamSlot& sp = h->slot[(si + MOR_STREAM_DEPTH - 1) % MOR_STREAM_DEPTH];
            if (!sp.d2h_enqueued) { int es = enqueue_slot_d2h(h, sp); if (es != MOR_OK) return es; }
        }
    } else {
        int es = enqueue_slot_d2h(h, sl);
        if (es != MOR_OK) return es;
    }
    h->mo_parity ^= 1; h->frame.mo_parity = h->mo_parity; h->filtered = true;  // committed like push + one filterCloud
    h->inflight++;
    return MOR_OK;
}

int mor_collect_frame(mor_handle* h, uint32_t* n_out) {
    if (!h) return MOR_ERR_ARG;
    if (!h->inflight) { h->last_error = "no frame in flight"; return MOR_ERR_STATE; }
    MOR_CUDA(cudaSetDevice(h->device));
    mor_handle::StreamSlot& sl = h->slot[h->sf_head];
    if (!sl.d2h_enqueued) {  // pipelining: its back half is still waiting for a next frame that has not come
        { int fs = flush_back(h); if (fs != MOR_OK) return fs; }
        { int es = enqueue_slot_d2h(h, sl); if (es != MOR_OK) return es; }
    }
    MOR_CUDA(cudaEventSynchronize(sl.d2h));
    h->sf_head = (h->sf_head + 1) % MOR_STREAM_DEPTH; h->inflight--;
    const uint32_t no = (uint32_t)sl.h_counts[CNT_SPEC_NOUT];
    if (n_out) *n_out = no;
    h->spec_out = no;
    if (sl.h_counts[MOR_CNT_ERRFLAGS]) {
        char msg[200];
        std::snprintf(msg, sizeof msg, "device capacity exceeded (error bits 0x%x: 1=clusters 2=moving 4=lattice range 8=ground grid 16=coordinate beyond the grid's range 32=cell pairs)",
                      sl.h_counts[MOR_CNT_ERRFLAGS]);
        h->last_error = msg;
        return MOR_ERR_CAPACITY;
    }
    if (no > sl.cap) { h->last_error = "output buffer of the submitted frame too small"; return MOR_ERR_CAPACITY; }
    if (no > sl.spec) {  // (the slot's device buffer is not rewritten before the frame after next is submitted)
        MOR_CUDA(cudaMemcpyAsync((uint8_t*)sl.out + (size_t)sl.spec * 32, (const uint8_t*)sl.d_out + (size_t)sl.spec * 32, (size_t)(no - sl.spec) * 32,
                                 cudaMemcpyDeviceToHost, h->copy_out));
        MOR_CUDA(cudaStreamSynchronize(h->copy_out));
    }
    return MOR_OK;
}

int mor_set_pipelining(mor_handle* h, int enabled) {
    if (!h) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    if (h->inflight) { h->last_error = "submitted frames are in flight: collect them first"; return MOR_ERR_STATE; }
    h->pipelining = enabled != 0;
    return MOR_OK;
}

int mor_frames_in_flight(const mor_handle* h, uint32_t* out) {
    if (!h || !out) return MOR_ERR_ARG;
    *out = (uint32_t)h->inflight;
    return MOR_OK;
}

int mor_alloc_pinned(size_t bytes, void** out) { return cudaMallocHost(out, bytes) == cudaSuccess ? MOR_OK : MOR_ERR_CUDA; }
int mor_free_pinned(void* p) { return cudaFreeHost(p) == cudaSuccess ? MOR_OK : MOR_ERR_CUDA; }
int mor_host_register(void* p, size_t bytes) {
    if (!p || !bytes) return MOR_ERR_ARG;
    if (cudaHostRegister(p, bytes, cudaHostRegisterDefault) == cudaSuccess) return MOR_OK;
    cudaGetLastError();
    return MOR_ERR_CUDA;
}
int mor_host_unregister(void* p) {
    if (cudaHostUnregister(p) == cudaSuccess) return MOR_OK;
    cudaGetLastError();
    return MOR_ERR_CUDA;
}
int mor_device_alloc(int device, size_t bytes, void** out) {
    if (cudaSetDevice(device) != cudaSuccess) return MOR_ERR_CUDA;
    return cudaMalloc(out, bytes) == cudaSuccess ? MOR_OK : MOR_ERR_CUDA;
}
int mor_device_free(int device, void* p) {
    if (cudaSetDevice(device) != cudaSuccess) return MOR_ERR_CUDA;
    return cudaFree(p) == cudaSuccess ? MOR_OK : MOR_ERR_CUDA;
}
int mor_device_upload(int device, void* d_dst, const void* src, size_t bytes) {
    if (cudaSetDevice(device) != cudaSuccess) return MOR_ERR_CUDA;
    return cudaMemcpy(d_dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess ? MOR_OK : MOR_ERR_CUDA;
}
int mor_device_download(int device, void* dst, const void* d_src, size_t bytes) {
    if (cudaSetDevice(device) != cudaSuccess) return MOR_ERR_CUDA;
    return cudaMemcpy(dst, d_src, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? MOR_OK : MOR_ERR_CUDA;
}

int mor_get_launch_count(const mor_handle* h, uint64_t* out) {
    if (!h || !out) return MOR_ERR_ARG;
    *out = h->launches;
    return MOR_OK;
}
int mor_set_timing(mor_handle* h, int enabled) {
    if (!h) return MOR_ERR_ARG;
    h->timing = enabled != 0;
    return MOR_OK;
}
int mor_get_last_device_ms(mor_handle* h, float* push_ms, float* filter_ms) {
    if (!h || !h->timing) return MOR_ERR_STATE;
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    if (push_ms) MOR_CUDA(cudaEventElapsedTime(push_ms, h->ev[0], h->ev[1]));
    if (filter_ms) MOR_CUDA(cudaEventElapsedTime(filter_ms, h->ev[2], h->ev[3]));
    return MOR_OK;
}

int mor_event_record(mor_handle* h, int slot) {
    if (!h || slot < 0 || slot >= 8) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    if (!h->slot_ev[slot]) MOR_CUDA(cudaEventCreate(&h->slot_ev[slot]));
    MOR_CUDA(cudaEventRecord(h->slot_ev[slot], h->stream));
    return MOR_OK;
}
int mor_event_elapsed_ms(mor_handle* h, int slot_a, int slot_b, float* ms) {
    if (!h || !ms || slot_a < 0 || slot_a >= 8 || slot_b < 0 || slot_b >= 8 || !h->slot_ev[slot_a] || !h->slot_ev[slot_b]) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    MOR_CUDA(cudaEventSynchronize(h->slot_ev[slot_b]));
    MOR_CUDA(cudaEventElapsedTime(ms, h->slot_ev[slot_a], h->slot_ev[slot_b]));
    return MOR_OK;
}
int mor_set_kernel_profiling(mor_handle* h, int enabled) {
    if (!h) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    if (!h->prof_ids.empty()) prof_harvest(h);
    h->profiling = enabled != 0;
    if (enabled) { std::memset(h->prof_ms, 0, sizeof(h->prof_ms)); std::memset(h->prof_n, 0, sizeof(h->prof_n)); }
    return MOR_OK;
}
// The last frame kernel's own timeline: microseconds CTA 0 spent in each phase (barrier included), from %globaltimer.
int mor_get_phase_times(mor_handle* h, float* us, int cap, int* n_phases) {
    if (!h || !us || !n_phases) return MOR_ERR_ARG;
    if (!h->have_cur) return MOR_ERR_STATE;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    unsigned long long ts[PH__COUNT + 1];
    MOR_CUDA(cudaMemcpy(ts, h->base.phase_ts, sizeof ts, cudaMemcpyDeviceToHost));
    *n_phases = PH__COUNT;
    for (int i = 0; i < PH__COUNT && i < cap; i++) us[i] = (float)((double)(ts[i + 1] - ts[i]) * 1e-3);
    return MOR_OK;
}
int mor_debug_phase_ts(mor_handle* h, unsigned long long* out32) {  // raw timeline words incl. the sub-steps some phases record
    if (!h || !out32) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    MOR_CUDA(cudaMemcpy(out32, h->base.phase_ts, sizeof(unsigned long long) * 32, cudaMemcpyDeviceToHost));
    return MOR_OK;
}
int mor_debug_cta_trace(mor_handle* h, unsigned long long* out, int n_words) {  // MOR_CTA_TRACE builds: [phase][cta] arrival times
    if (!h || !out || n_words > 32 * 256) return MOR_ERR_ARG;
    MOR_CUDA(cudaSetDevice(h->device));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    MOR_CUDA(cudaMemcpy(out, h->base.cta_trace, sizeof(unsigned long long) * n_words, cudaMemcpyDeviceToHost));
    return MOR_OK;
}
const char* mor_phase_name(int index) { return index >= 0 && index < PH__COUNT ? kKernelNames[index] : ""; }

int mor_get_kernel_profile(mor_handle* h, int index, char name[32], double* total_ms, uint64_t* launches) {
    if (!h || index < 0 || index >= KID__COUNT || !name || !total_ms || !launches) return MOR_ERR_ARG;
    std::snprintf(name, 32, "%s", kKernelNames[index]);
    *total_ms = h->prof_ms[index];
    *launches = h->prof_n[index];
    return MOR_OK;
}

// ---- parity taps ----------------------------------------------------------------------------------
int mor_tap(mor_handle* h, int tap, void* dst, size_t cap_bytes, size_t* n_bytes) {
    if (!h) return MOR_ERR_ARG;
    if (!h->have_cur) return MOR_ERR_STATE;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    const FramePtrs& a = h->frame;
    int32_t c[MOR_NCOUNTS];
    MOR_CUDA(cudaMemcpy(c, a.counts, sizeof(c), cudaMemcpyDeviceToHost));
    // the filter phase parks its results in spare slots until filterCloud commits the frame (do_filter)
    if (h->filtered) { c[MOR_CNT_NOUT] = c[CNT_SPEC_NOUT]; c[MOR_CNT_NMO] = c[CNT_SPEC_NMO]; c[MOR_CNT_EXTRACT_OVERFLOW] = c[CNT_SPEC_OVERFLOW]; }
    c[CNT_SPEC_NOUT] = c[CNT_SPEC_NMO] = c[CNT_SPEC_OVERFLOW] = 0;
    const void* src = nullptr;
    size_t bytes = 0;
    std::vector<uint8_t> host;  // for taps assembled on the host
    const size_t N = c[MOR_CNT_N], NC = c[MOR_CNT_NC], K = c[MOR_CNT_K], KP = c[MOR_CNT_KPREV], M = c[MOR_CNT_M], MU = c[MOR_CNT_MU], NMO = c[MOR_CNT_NMO],
                 NCP = c[MOR_CNT_NCPREV];
    switch (tap) {
        case MOR_TAP_COUNTS: host.assign((uint8_t*)c, (uint8_t*)c + sizeof(c)); break;  // (after the merge of the filter phase's results below)
        case MOR_TAP_POINT_CLASS: src = a.point_class; bytes = N; break;
        case MOR_TAP_LABELS: src = a.label; bytes = NC * 4; break;
        case MOR_TAP_CLUSTER_ID: src = a.cid; bytes = NC * 4; break;
        case MOR_TAP_CLUSTER_ROOT: src = a.cl_root; bytes = K * 4; break;
        case MOR_TAP_CLUSTER_SIZE: src = a.cl_size; bytes = K * 4; break;
        case MOR_TAP_CENTROIDS: src = a.cl_centroid; bytes = K * 12; break;
        case MOR_TAP_TRANSFORM: host.assign((uint8_t*)h->M, (uint8_t*)h->M + sizeof(h->M)); break;
        case MOR_TAP_PREV_CENTROIDS_T: src = a.pct; bytes = KP * 12; break;
        case MOR_TAP_PREV_POINTS_T: {
            std::vector<float4> t(NCP);
            if (NCP) MOR_CUDA(cudaMemcpy(t.data(), a.tpts, NCP * sizeof(float4), cudaMemcpyDeviceToHost));
            host.resize(NCP * 12);
            float* o = (float*)host.data();
            for (size_t i = 0; i < NCP; i++) {
                int k; std::memcpy(&k, &t[i].w, 4);
                const float nan = std::nanf("");
                o[i * 3] = k >= 0 ? t[i].x : nan; o[i * 3 + 1] = k >= 0 ? t[i].y : nan; o[i * 3 + 2] = k >= 0 ? t[i].z : nan;
            }
        } break;
        case MOR_TAP_MATCH_QUERY: src = a.match_q; bytes = M * 4; break;
        case MOR_TAP_MATCH_MATCH: src = a.match_m; bytes = M * 4; break;
        case MOR_TAP_MATCH_DIST: src = a.match_dist; bytes = M * 4; break;
        case MOR_TAP_MATCH_SCORE: src = a.match_score; bytes = M * 8; break;
        case MOR_TAP_FLAGS: src = a.cl_flags; bytes = K; break;
        case MOR_TAP_MO_CENTROIDS: src = a.mo_centroid + (size_t)h->mo_parity * h->momax * 3; bytes = NMO * 12; break;
        case MOR_TAP_MO_CONF: src = a.mo_conf + (size_t)h->mo_parity * h->momax; bytes = NMO * 4; break;
        case MOR_TAP_REMOVED_MASK: if (!h->filtered) return MOR_ERR_STATE; src = a.removed_mask; bytes = N; break;
        case MOR_TAP_CLUSTER_REMOVED: if (!h->filtered) return MOR_ERR_STATE; src = a.cluster_removed; bytes = K; break;
        case MOR_TAP_RECIP_QUERY: src = a.recip_q; bytes = MU * 4; break;
        case MOR_TAP_RECIP_MATCH: src = a.recip_m; bytes = MU * 4; break;
        case MOR_TAP_GROUND_VOXELS: if (h->cfg.ground_mode != MOR_GROUND_CROP) { src = h->ground.vox_info; bytes = (size_t)c[MOR_CNT_NVOX] * 32; } break;
        case MOR_TAP_CLUSTER_BBOX: src = a.cl_bbox; bytes = K * 24; break;
        case MOR_TAP_PREV_BBOX_T: src = a.pbbox; bytes = KP * 24; break;
        default: return MOR_ERR_ARG;
    }
    if (!host.empty() || tap == MOR_TAP_PREV_POINTS_T) bytes = host.size();
    if (n_bytes) *n_bytes = bytes;
    if (bytes > cap_bytes) return MOR_ERR_CAPACITY;
    if (!bytes) return MOR_OK;
    if (!host.empty()) std::memcpy(dst, host.data(), bytes);
    else MOR_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return MOR_OK;
}

#define MOR_NAMED_TAP(name, tapid, type)                                           \
    int name(mor_handle* h, type* dst, size_t n) { size_t nb = 0; return mor_tap(h, tapid, dst, n * sizeof(type), &nb); }
MOR_NAMED_TAP(mor_get_counts, MOR_TAP_COUNTS, int32_t)
MOR_NAMED_TAP(mor_get_trim_mask, MOR_TAP_POINT_CLASS, uint8_t)
MOR_NAMED_TAP(mor_get_ground_mask, MOR_TAP_POINT_CLASS, uint8_t)
MOR_NAMED_TAP(mor_get_labels, MOR_TAP_LABELS, int32_t)
MOR_NAMED_TAP(mor_get_cluster_order, MOR_TAP_CLUSTER_ROOT, int32_t)
MOR_NAMED_TAP(mor_get_centroids, MOR_TAP_CENTROIDS, float)
MOR_NAMED_TAP(mor_get_transform, MOR_TAP_TRANSFORM, float)
MOR_NAMED_TAP(mor_get_transformed_xyz, MOR_TAP_PREV_POINTS_T, float)
MOR_NAMED_TAP(mor_get_scores, MOR_TAP_MATCH_SCORE, double)
MOR_NAMED_TAP(mor_get_flags, MOR_TAP_FLAGS, uint8_t)
MOR_NAMED_TAP(mor_get_removed_mask, MOR_TAP_REMOVED_MASK, uint8_t)
int mor_get_matches(mor_handle* h, int32_t* query, int32_t* match, size_t n) {
    size_t nb = 0;
    int st = mor_tap(h, MOR_TAP_MATCH_QUERY, query, n * 4, &nb);
    return st != MOR_OK ? st : mor_tap(h, MOR_TAP_MATCH_MATCH, match, n * 4, &nb);
}
int mor_get_mo_vec(mor_handle* h, float* xyz, int32_t* conf, size_t n) {
    size_t nb = 0;
    int st = mor_tap(h, MOR_TAP_MO_CENTROIDS, xyz, n * 12, &nb);
    return st != MOR_OK ? st : mor_tap(h, MOR_TAP_MO_CONF, conf, n * 4, &nb);
}

// ---- VISUALIZE outputs (IncludeAll.h:32), on request
int mor_get_cluster_collection(mor_handle* h, void* out, uint32_t cap_points, uint32_t* n_out) {
    if (!h || !n_out) return MOR_ERR_ARG;
    if (!h->have_cur) return MOR_ERR_STATE;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    const FramePtrs& a = h->frame;
    CollectionPtrs c;
    c.cid = a.cid; c.pts = a.pts; c.cl_size = a.cl_size; c.counts = a.counts; c.cursor = h->coll_cursor; c.turn = h->coll_turn;
    c.out = h->coll_out;  // not base.out: that holds the frame's filtered cloud until filterCloud has delivered it
    k_collection_offsets<<<1, kCollBlock, 0, h->stream>>>(c);
    k_cluster_collection<<<h->n_input ? (h->n_input + kCollBlock - 1) / kCollBlock : 1, kCollBlock, 0, h->stream>>>(c);
    h->launches += 2;
    MOR_CUDA(cudaGetLastError());
    MOR_CUDA(cudaMemcpyAsync(h->h_counts, a.counts, sizeof(int32_t) * MOR_NCOUNTS, cudaMemcpyDeviceToHost, h->stream));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    const uint32_t nk = (uint32_t)h->h_counts[MOR_CNT_NK];
    *n_out = nk;
    if (!out) return MOR_OK;
    if (nk > cap_points) return MOR_ERR_CAPACITY;
    if (nk) MOR_CUDA(cudaMemcpy(out, c.out, (size_t)nk * 32, cudaMemcpyDeviceToHost));
    return MOR_OK;
}

int mor_count_radius_ties(mor_handle* h, int ulps, uint64_t* pairs) {
    if (!h || !pairs || ulps < 0) return MOR_ERR_ARG;
    if (!h->have_cur) return MOR_ERR_STATE;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    const float r2 = (float)((double)h->cfg.ec_distance_threshold * (double)h->cfg.ec_distance_threshold);
    float lo = r2, hi = r2;
    for (int u = 0; u < ulps; u++) { lo = std::nextafterf(lo, 0.f); hi = std::nextafterf(hi, 3.402823466e+38f); }
    unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(h->coll_cursor);  // (scratch of the on-request outputs, 8-byte aligned)
    MOR_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long), h->stream));
    k_radius_ties<<<h->num_sms * 2, 1024, 0, h->stream>>>(h->frame.pts, h->frame.counts, lo, hi, d_cnt);
    h->launches++;
    MOR_CUDA(cudaGetLastError());
    unsigned long long v = 0;
    MOR_CUDA(cudaMemcpyAsync(&v, d_cnt, sizeof v, cudaMemcpyDeviceToHost, h->stream));
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    *pairs = v;
    return MOR_OK;
}

int mor_get_moving_markers(mor_handle* h, mor_marker* out, uint32_t cap, uint32_t* n_out) {
    if (!h || !n_out) return MOR_ERR_ARG;
    if (!h->have_cur || !h->filtered) return MOR_ERR_STATE;
    MOR_CUDA(cudaSetDevice(h->device));
    { int js = join_foreign_stream(h); if (js != MOR_OK) return js; }
    MOR_CUDA(cudaStreamSynchronize(h->stream));
    const FramePtrs& a = h->frame;
    TrackState ts;
    MOR_CUDA(cudaMemcpy(&ts, a.track, sizeof ts, cudaMemcpyDeviceToHost));
    const uint32_t n = (uint32_t)ts.n_markers;
    *n_out = n;
    if (!out || !n) return MOR_OK;
    if (n > cap) return MOR_ERR_CAPACITY;
    MOR_CUDA(cudaMemcpy(h->h_counts, a.counts, sizeof(int32_t) * MOR_NCOUNTS, cudaMemcpyDeviceToHost));
    const size_t K = (size_t)h->h_counts[MOR_CNT_K];
    std::vector<int> which(n);
    std::vector<float> cen(K * 3), box(K * 6);
    MOR_CUDA(cudaMemcpy(which.data(), a.marker_cluster, n * sizeof(int), cudaMemcpyDeviceToHost));
    MOR_CUDA(cudaMemcpy(cen.data(), a.cl_centroid, K * 12, cudaMemcpyDeviceToHost));
    MOR_CUDA(cudaMemcpy(box.data(), a.cl_bbox, K * 24, cudaMemcpyDeviceToHost));
    for (uint32_t i = 0; i < n; i++) {
        const int k = which[i];
        mor_marker& m = out[i];
        for (int q = 0; q < 3; q++) {
            m.position[q] = cen[(size_t)k * 3 + q];
            const float ext = box[(size_t)k * 6 + 3 + q] - box[(size_t)k * 6 + q];
            m.scale[q] = ext == 0.f ? 0.1f : ext;  // cpp:40-47
        }
        m.color[0] = 0.8f; m.color[1] = 0.1f; m.color[2] = 0.4f; m.color[3] = 0.5f;  // cpp:622, :53
        m.id = (int32_t)i + 1;  // cpp:622, :669: filterCloud's counter starts at 1 and advances once per looked-up entry
        m.cluster = k;
    }
    return MOR_OK;
}

}  // extern "C"
